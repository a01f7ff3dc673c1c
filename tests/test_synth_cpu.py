"""
The synthetic corpora: make_corpus stays bitwise what it was (bench.py and the parity tests draw from it), and make_topics
returns the topics it draws from.
"""
import hashlib

import numpy as np
import pytest

from trlda_b200.synth import make_corpus, make_topics


@pytest.mark.parametrize('args,digest', [
	((512, 2000, 20), '634b8daa2307f90b9a833ef38edef65ea622cb3b788386b3aba8b53ef23b48a9'),
	((256, 100000, 1000), '5dbd461f64b6be942e1ac5b6ee6d5370e4b40d60716b5505ae5ea2ec82ec603a'),
])
def test_make_corpus_is_pinned(args, digest):
	h = hashlib.sha256()
	for a in make_corpus(*args, seed=3):
		h.update(a.tobytes())
	assert h.hexdigest() == digest


def test_make_topics_are_the_corpus_topics():
	V, K, seed = 300, 4, 9
	topics = make_topics(V, K, eta=.2, seed=seed)
	assert topics.shape == (K, V) and topics.dtype == np.float64
	assert (topics > 0).all() and np.allclose(topics.sum(axis=1), 1., rtol=0, atol=1e-12)
	assert not np.array_equal(make_topics(V, K, seed=seed + 1), topics)
	assert np.array_equal(make_topics(V, K, eta=.2, seed=seed), topics)
	# topic k does not depend on the number of topics; a one-topic corpus draws every word from row 0
	assert np.array_equal(make_topics(V, 1, eta=.2, seed=seed)[0], topics[0])
	ptr, ids, cts = make_corpus(2000, V, 1, eta=.2, mean_length=200, seed=seed)
	freq = np.bincount(ids, weights=cts, minlength=V) / cts.sum()
	assert float(np.abs(freq - topics[0]).sum()) < .05
