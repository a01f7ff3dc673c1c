"""Document co-occurrence coherence of topics (numpy only; the counts come from LDA.cooccurrence on the GPU)."""
import numpy as np


def coherence_from_counts(counts, num_docs, measure='npmi'):
	"""Coherence of every topic from document frequencies of its top words.

	`counts` is K x n x n (LDA.cooccurrence): counts[k, i, j] = D(w_i, w_j), the number of documents containing both the
	words of ranks i and j of topic k, and counts[k, i, i] = D(w_i).  `num_docs` is the number of documents N.
	Returns K values (float64).

	'npmi' (Bouma 2009; Lau et al. 2014): the mean over the pairs i < j of
	    NPMI(w_i, w_j) = log(P(w_i, w_j) / (P(w_i) P(w_j))) / (-log P(w_i, w_j)),   P = document frequency / N,
	with NPMI = -1 when D(w_i, w_j) = 0 and NPMI = 1 when P(w_i, w_j) = 1.  No smoothing term.

	'umass' (Mimno et al. 2011, Eq. 1 divided by the number of pairs counted): the mean over the pairs i > j (rank order, so
	w_j is the more probable word) of
	    log((D(w_i, w_j) + 1) / D(w_j)),
	skipping the pairs with D(w_j) = 0.  A topic with no pair left gives NaN.  num_docs does not enter.

	With n = 1 there is no pair, and every topic gives NaN."""
	counts = np.asarray(counts)
	if counts.ndim != 3 or counts.shape[1] != counts.shape[2]:
		raise ValueError('counts must be a K x n x n array')
	n = counts.shape[1]
	D = counts.astype(np.float64)
	single = np.diagonal(D, axis1=1, axis2=2)                     # K x n: D(w_i)
	with np.errstate(divide='ignore', invalid='ignore'):
		if measure == 'npmi':
			if not num_docs > 0:
				raise ValueError('num_docs must be positive')
			N = float(num_docs)
			i, j = np.triu_indices(n, 1)
			joint = D[:, i, j]
			p_ij, p_i, p_j = joint / N, single[:, i] / N, single[:, j] / N
			npmi = np.log(p_ij / (p_i * p_j)) / -np.log(p_ij)
			npmi = np.where(joint == 0, -1., np.where(joint == N, 1., npmi))
			return npmi.mean(axis=1) if i.size else np.full(D.shape[0], np.nan)
		if measure == 'umass':
			i, j = np.tril_indices(n, -1)
			joint, d_j = D[:, i, j], single[:, j]
			valid = d_j > 0
			terms = np.where(valid, np.log((joint + 1.) / np.where(valid, d_j, 1.)), 0.)
			return terms.sum(axis=1) / valid.sum(axis=1)
	raise ValueError("measure should be 'npmi' or 'umass'")


def topic_coherence(model, batches, num_words=10, measure='npmi', top_words=None):
	"""Coherence of every topic of `model` (an LDA model) on a reference corpus, as in coherence_from_counts.

	`batches` is an iterable of minibatches, each a list of documents or a (doc_ptr, word_ids, counts) triple, e.g.
	load_documents_csr(path, 4096); pass a single minibatch as [docs].  The top words are taken once, with
	model.top_words(num_words), unless `top_words` (K x n word ids) is given.  The document frequencies of each batch are
	counted on the GPU (model.cooccurrence) and summed in int64, so the result does not depend on how the corpus is cut
	into batches.  Returns K values."""
	if top_words is None:
		top_words, _ = model.top_words(num_words)
	total, num_docs = None, 0
	for docs in batches:
		counts, n = model.cooccurrence(docs, top_words)
		total = counts if total is None else total + counts
		num_docs += n
	if total is None:
		raise ValueError('no batch of documents was given')
	return coherence_from_counts(total, num_docs, measure)
