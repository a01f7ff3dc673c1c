"""trlda.utils.coherence_from_counts (numpy only) against a direct restatement of the NPMI and UMass definitions."""
import itertools
import math

import numpy as np
import pytest


def counts_from_sets(docs, top):
	"""K x n x n document frequencies from documents given as word sets"""
	K, n = top.shape
	out = np.zeros((K, n, n), dtype=np.int64)
	for words in docs:
		for k in range(K):
			for i, j in itertools.product(range(n), repeat=2):
				out[k, i, j] += top[k, i] in words and top[k, j] in words
	return out


def npmi_direct(counts, N):
	out = []
	for c in counts:
		n = c.shape[0]
		values = []
		for i in range(n):
			for j in range(i + 1, n):
				if c[i, j] == 0:
					values.append(-1.)
				elif c[i, j] == N:
					values.append(1.)
				else:
					p_ij, p_i, p_j = c[i, j] / N, c[i, i] / N, c[j, j] / N
					values.append(math.log(p_ij / (p_i * p_j)) / -math.log(p_ij))
		out.append(sum(values) / len(values))
	return np.array(out)


def umass_direct(counts):
	out = []
	for c in counts:
		n = c.shape[0]
		values = [math.log((c[i, j] + 1) / c[j, j]) for i in range(n) for j in range(i) if c[j, j] > 0]
		out.append(sum(values) / len(values) if values else math.nan)
	return np.array(out)


def hand_made():
	"""6 documents over words 0..7; topic 0 has a word in every document (0) and a pair that never co-occurs (1, 2);
	topic 1 has a word in no document (7)"""
	docs = [{0, 1, 3}, {0, 2, 3}, {0, 1, 4}, {0, 2, 5, 6}, {0, 3, 5}, {0, 4, 5, 6, 1}]
	return docs, np.array([[0, 1, 2, 3], [5, 6, 7, 4]])


def test_npmi_and_umass_match_the_definitions():
	from trlda.utils import coherence_from_counts
	docs, top = hand_made()
	counts = counts_from_sets(docs, top)
	assert counts[0, 1, 2] == 0 and counts[0, 0, 0] == len(docs) and counts[1, 2, 2] == 0
	np.testing.assert_allclose(coherence_from_counts(counts, len(docs), 'npmi'), npmi_direct(counts, len(docs)), rtol=1e-14)
	np.testing.assert_allclose(coherence_from_counts(counts, len(docs), 'umass'), umass_direct(counts), rtol=1e-14)
	assert np.array_equal(coherence_from_counts(counts, len(docs)), coherence_from_counts(counts, len(docs), 'npmi'))


def test_edge_cases():
	from trlda.utils import coherence_from_counts
	N = 10
	# one topic of two words: never together, always together, a word in every document, a word in no document
	never = np.array([[[4, 0], [0, 3]]])
	always = np.array([[[N, N], [N, N]]])
	everywhere = np.array([[[N, 5], [5, 5]]])
	nowhere = np.array([[[6, 0], [0, 0]]])
	assert coherence_from_counts(never, N, 'npmi')[0] == -1.
	assert coherence_from_counts(always, N, 'npmi')[0] == 1.
	assert coherence_from_counts(everywhere, N, 'npmi')[0] == 0.
	assert coherence_from_counts(nowhere, N, 'npmi')[0] == -1.
	assert coherence_from_counts(never, N, 'umass')[0] == pytest.approx(math.log(1 / 4), rel=1e-15)
	assert coherence_from_counts(everywhere, N, 'umass')[0] == pytest.approx(math.log(6 / N), rel=1e-15)
	# UMass skips pairs whose more probable word is in no document; none left: NaN
	assert math.isnan(coherence_from_counts(np.array([[[0, 0], [0, 6]]]), N, 'umass')[0])
	partly = np.zeros((1, 3, 3), dtype=np.int64)
	partly[0] = [[0, 0, 0], [0, 4, 2], [0, 2, 3]]
	assert coherence_from_counts(partly, N, 'umass')[0] == pytest.approx(math.log(3 / 4), rel=1e-15)
	# one word: no pair
	assert np.isnan(coherence_from_counts(np.array([[[3]]]), N, 'npmi')).all()


def test_against_scipy_on_random_corpus():
	from scipy import sparse
	from trlda.utils import coherence_from_counts
	rng = np.random.default_rng(0)
	D, V, K, n = 400, 60, 7, 9
	X = sparse.csr_matrix((rng.random((D, V)) < .15).astype(np.int64))
	top = np.stack([rng.choice(V, n, replace=False) for _ in range(K)])
	counts = np.stack([(X[:, t].T @ X[:, t]).toarray() for t in top])
	np.testing.assert_allclose(coherence_from_counts(counts, D, 'npmi'), npmi_direct(counts, D), rtol=1e-13)
	np.testing.assert_allclose(coherence_from_counts(counts, D, 'umass'), umass_direct(counts), rtol=1e-13)


def test_bad_arguments():
	from trlda.utils import coherence_from_counts
	with pytest.raises(ValueError):
		coherence_from_counts(np.zeros((2, 3, 3)), 5, 'cv')
	with pytest.raises(ValueError):
		coherence_from_counts(np.zeros((2, 3, 2)), 5)
	with pytest.raises(ValueError):
		coherence_from_counts(np.zeros((2, 3, 3)), 0, 'npmi')
