"""
Synthetic corpora drawn from the LDA generative process, shared by bench.py and the parity tests.

Mirrors what `LDA::sample` does (reference code/trlda/src/lda.cpp:88-115: document length ~ Poisson,
beta_k ~ Dirichlet, theta_d ~ Dirichlet, one (topic, word) draw per token) but is generated with numpy
outside the reference, because `LDA::sample` is not reproducible across thread counts (rand() inside an
OpenMP loop, utils.cpp:273-284).  Tokens are collapsed to unique (word_id, count) pairs sorted by id, the
form `load_documents` produces (python/utils/load_documents.py:41-44).
"""
import numpy as np


def _topic_weights(seed, k, num_words, eta):
	"""unnormalised beta_k ~ Dirichlet(eta 1_V) of topic k of corpus `seed`: standard_gamma(eta, V) from the topic's own
	stream, floored at 1e-300 so that every word has positive probability"""
	topic_rng = np.random.Generator(np.random.PCG64([seed, k]))
	return np.maximum(topic_rng.standard_gamma(eta, size=num_words), 1e-300)


def make_topics(num_words, num_topics, eta=.2, seed=0):
	"""
	The topics make_corpus(..., num_words, num_topics, eta=eta, seed=seed) draws its words from: a num_topics x num_words
	float64 array whose row k is beta_k (sums to 1).  Useful as the lambda of a reference model, e.g. to check with
	topic_distances that training recovers the topics.
	"""
	topics = np.empty((num_topics, num_words))
	for k in range(num_topics):
		beta = _topic_weights(seed, k, num_words, eta)
		topics[k] = beta / beta.sum()
	return topics


def make_corpus(num_docs, num_words, num_topics, alpha=.1, eta=.2, mean_length=150, seed=0, doc_seed=None):
	"""
	Returns the minibatch in CSR form: (doc_ptr[int64, B+1], word_ids[int32, N], counts[int32, N]).

	beta_k ~ Dirichlet(eta 1_V) is drawn as a normalised standard_gamma(eta, V) from a per-topic stream so
	that the K x V matrix never has to be held (cfg-3: 800 MB); theta_d ~ Dirichlet(alpha 1_K);
	length_d ~ Poisson(mean_length).  `seed` fixes the corpus (its topics); `doc_seed` (default: seed) the documents
	drawn from it, so that several processes can draw different documents of ONE corpus.
	"""
	rng = np.random.Generator(np.random.PCG64(seed if doc_seed is None else [seed, 7919, doc_seed]))
	lengths = rng.poisson(mean_length, size=num_docs).astype(np.int64)
	total = int(lengths.sum())
	doc_of_token = np.repeat(np.arange(num_docs, dtype=np.int64), lengths)

	# topic of every token
	theta = rng.standard_gamma(alpha, size=(num_docs, num_topics))
	theta = np.maximum(theta, 1e-300)
	theta_cdf = np.cumsum(theta, axis=1)
	theta_cdf /= theta_cdf[:, -1:]
	u = rng.random(total)
	topics = np.empty(total, dtype=np.int64)
	start = 0
	for d in range(num_docs):
		n = lengths[d]
		topics[start:start + n] = np.searchsorted(theta_cdf[d], u[start:start + n], side='right')
		start += n
	np.minimum(topics, num_topics - 1, out=topics)

	# word of every token, one topic at a time
	words = np.empty(total, dtype=np.int64)
	order = np.argsort(topics, kind='stable')
	sorted_topics = topics[order]
	bounds = np.searchsorted(sorted_topics, np.arange(num_topics + 1))
	v = rng.random(total)
	for k in range(num_topics):
		lo, hi = bounds[k], bounds[k + 1]
		if lo == hi:
			continue
		cdf = np.cumsum(_topic_weights(seed, k, num_words, eta))
		cdf /= cdf[-1]
		idx = order[lo:hi]
		words[idx] = np.minimum(np.searchsorted(cdf, v[idx], side='right'), num_words - 1)

	# collapse tokens to unique (word, count) pairs per document, sorted by word id
	key = doc_of_token * num_words + words
	key.sort()
	unique, counts = np.unique(key, return_counts=True)
	docs = unique // num_words
	word_ids = (unique - docs * num_words).astype(np.int32)
	doc_ptr = np.zeros(num_docs + 1, dtype=np.int64)
	np.add.at(doc_ptr, docs + 1, 1)
	np.cumsum(doc_ptr, out=doc_ptr)
	return doc_ptr, word_ids, counts.astype(np.int32)


def gamma_matrix(rows, cols, seed, shape=100., scale=.01):
	"""iid Gamma(100, 1/100) in column-major order: the law of the reference's initial lambda (lda.cpp:71) and
	initial gamma (lda.cpp:135)."""
	rng = np.random.Generator(np.random.PCG64(seed))
	return np.asfortranarray(rng.gamma(shape, scale, size=(cols, rows)).T)


def to_lists(doc_ptr, word_ids, counts):
	"""CSR -> list of lists of (word_id, count), the reference's Python document format"""
	ids = word_ids.tolist()
	cts = counts.tolist()
	ptr = doc_ptr.tolist()
	return [list(zip(ids[ptr[d]:ptr[d + 1]], cts[ptr[d]:ptr[d + 1]])) for d in range(len(ptr) - 1)]
