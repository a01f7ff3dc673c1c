"""
Host-side helpers of trlda.utils that sit beside the hot path in the reference (utils.cpp:235-287, 294-330), written
with numpy.  LDA::sample itself runs on the device (csrc/sample.cu, trlda_sample).
"""
import numpy as np


def random_select(k, n):
	"""k distinct indices out of range(n) (reference: utils.cpp randomSelect)."""
	if k > n:
		raise Exception('k must be smaller than n.')
	if k < 0 or n < 0:
		raise Exception('n and k must be non-negative.')
	return sorted(int(i) for i in np.random.permutation(n)[:k])


def split_documents(docs, held_out=.2, seed=None):
	"""Splits every document into an observed and a held-out part for document-completion evaluation
	(LDA.predictive_log_likelihood): floor(held_out * n_d) of the n_d token occurrences of document d are drawn without
	replacement.  `docs` is a list of lists of (word_id, count) or a (doc_ptr, word_ids, counts) triple; returns
	(observed, held_out) in the same form, pairs whose count drops to 0 removed and the order of the rest kept."""
	if not 0 <= held_out < 1:
		raise ValueError('held_out should lie in [0, 1).')
	as_lists = not isinstance(docs, tuple)
	if as_lists:
		doc_ptr = np.cumsum([0] + [len(doc) for doc in docs], dtype=np.int64)
		word_ids = np.array([w for doc in docs for w, _ in doc], dtype=np.int32)
		counts = np.array([c for doc in docs for _, c in doc], dtype=np.int64)
	else:
		doc_ptr = np.asarray(docs[0], dtype=np.int64)
		word_ids = np.asarray(docs[1], dtype=np.int32)
		counts = np.asarray(docs[2], dtype=np.int64)
	rng = np.random.default_rng(seed)
	held = np.zeros_like(counts)
	for d in range(doc_ptr.size - 1):
		lo, hi = int(doc_ptr[d]), int(doc_ptr[d + 1])
		k = int(np.floor(held_out * int(counts[lo:hi].sum())))
		if k > 0:
			held[lo:hi] = rng.multivariate_hypergeometric(counts[lo:hi], k)
	parts = []
	for part in (counts - held, held):
		keep = part > 0
		ptr = np.concatenate([[0], np.cumsum(keep)]).astype(np.int64)[doc_ptr]
		ids, cts = word_ids[keep], part[keep].astype(np.int32)
		if as_lists:
			parts.append([list(zip(ids[ptr[d]:ptr[d + 1]].tolist(), cts[ptr[d]:ptr[d + 1]].tolist())) for d in range(ptr.size - 1)])
		else:
			parts.append((ptr, ids, cts))
	return parts[0], parts[1]


def sample_dirichlet(m, n=1, alpha=.1):
	"""m x n array whose columns are draws from a symmetric Dirichlet(alpha) (reference: utils.cpp:252-264)."""
	sample = np.maximum(np.random.standard_gamma(alpha, size=(m, n)), 1e-300)
	return sample / sample.sum(0, keepdims=True)
