"""trlda.utils.split_documents: the observed / held-out split of document-completion evaluation (no GPU needed)."""
import math
from collections import Counter

import numpy as np
import pytest

from trlda.utils import split_documents


def _docs(seed=3):
	rng = np.random.default_rng(seed)
	docs = []
	for n in [0, 1, 5, 40, 3, 120, 0, 17]:
		ids = rng.permutation(500)[:n]
		docs.append([(int(w), int(1 + rng.integers(6))) for w in ids])
	docs[3].append((docs[3][0][0], 4))        # a duplicated id inside one document
	return docs


def _to_csr(docs):
	ptr = np.cumsum([0] + [len(d) for d in docs]).astype(np.int64)
	ids = np.array([w for d in docs for w, _ in d], dtype=np.int32)
	cts = np.array([c for d in docs for _, c in d], dtype=np.int32)
	return ptr, ids, cts


def _per_doc(doc):
	out = Counter()
	for w, c in doc:
		out[w] += c
	return out


@pytest.mark.parametrize('fraction', [.2, .5, .9])
def test_observed_plus_held_out_is_the_input(fraction):
	docs = _docs()
	observed, held = split_documents(docs, fraction, seed=1)
	assert len(observed) == len(held) == len(docs)
	for doc, o, h in zip(docs, observed, held):
		assert _per_doc(o) + _per_doc(h) == _per_doc(doc)
		assert all(c > 0 for _, c in o + h)
		n = sum(c for _, c in doc)
		assert sum(c for _, c in h) == math.floor(fraction * n)


def test_order_is_kept_and_zero_pairs_are_dropped():
	docs = [[(7, 1), (3, 5), (9, 2), (1, 1)]]
	observed, held = split_documents(docs, .5, seed=4)
	for part in (observed[0], held[0]):
		ids = [w for w, _ in part]
		assert ids == [w for w in (7, 3, 9, 1) if w in ids]
		assert all(c > 0 for _, c in part)
	assert sum(c for _, c in held[0]) == 4


def test_seed_and_form_give_the_same_split():
	docs = _docs()
	a = split_documents(docs, .3, seed=11)
	b = split_documents(docs, .3, seed=11)
	assert a == b
	ptr, ids, cts = split_documents(_to_csr(docs), .3, seed=11)[1]
	assert ptr.dtype == np.int64 and ids.dtype == np.int32 and cts.dtype == np.int32
	assert [list(zip(ids[ptr[d]:ptr[d + 1]].tolist(), cts[ptr[d]:ptr[d + 1]].tolist())) for d in range(len(docs))] == a[1]
	ptr, ids, cts = split_documents(_to_csr(docs), .3, seed=11)[0]
	assert [list(zip(ids[ptr[d]:ptr[d + 1]].tolist(), cts[ptr[d]:ptr[d + 1]].tolist())) for d in range(len(docs))] == a[0]


def test_nothing_held_out_at_zero():
	docs = _docs()
	observed, held = split_documents(docs, 0., seed=2)
	assert held == [[] for _ in docs]
	assert observed == docs
	ptr, ids, cts = split_documents(_to_csr(docs), 0, seed=2)[1]
	assert ptr.tolist() == [0] * (len(docs) + 1) and ids.size == 0 and cts.size == 0


@pytest.mark.parametrize('fraction', [-.1, 1., 1.5])
def test_fraction_out_of_range(fraction):
	with pytest.raises(ValueError):
		split_documents(_docs(), fraction)
