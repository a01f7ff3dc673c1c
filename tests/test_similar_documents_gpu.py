"""
Similar documents on the device: trlda_index_documents / trlda_similar_documents, the nearest indexed documents of every
query under the Hellinger distance of the topic proportions.  Exact answers on dyadic data, agreement with numpy, bitwise
independence of the path (streaming or product), the batch, the order of the index and the precision mode,
self-retrieval, untouched training state and the errors.
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PRECISIONS = ['fp64', 'mixed']
BAD_GAMMA = 'Gamma must be finite and non-negative, with a positive sum in every column.'
N_RANGE = 'Number of neighbors must lie in [1, min(32, number of indexed documents)].'


@pytest.fixture(scope='module')
def capi():
	from trlda_b200 import capi
	capi.lib()        # raises if libtrlda_b200.so is missing
	return capi


def new_model(capi, K, precision='fp64', V=50):
	return capi.Model('online', V, K, 1000, .1, .2, precision=precision)


def gammas(rng, K, D):
	"""positive, tie-free gamma: Gamma(0.3, 1) + 1e-3, column-major"""
	return np.asfortranarray(rng.gamma(.3, 1., size=(K, D)) + 1e-3)


def numpy_affinity(gq, gd):
	tq, td = gq / gq.sum(axis=0), gd / gd.sum(axis=0)
	return np.sqrt(tq).T @ np.sqrt(td)        # Q x D


def check_against_numpy(ids, dist, gq, gd, n):
	c = numpy_affinity(gq, gd)
	Q, D = c.shape
	assert ids.shape == dist.shape == (Q, n) and ids.dtype == np.int64 and dist.dtype == np.float64
	assert (ids >= 0).all() and (ids < D).all()
	rows = np.arange(Q)[:, None]
	# the distance is the square root of 1 - C, C a sum of K products: its rounding error is about K 2^-53
	assert float(np.max(np.abs(dist * dist - np.maximum(0., 1. - c[rows, ids])))) < 1e-12
	# a valid top n under numpy's C: nothing left out is better than the worst one taken, by more than the rounding
	for q in range(Q):
		assert len(set(ids[q].tolist())) == n
		rest = np.delete(c[q], ids[q])
		if rest.size:
			assert rest.max() <= c[q, ids[q]].min() + 1e-12
	# sorted by (distance, id)
	d0, d1, i0, i1 = dist[:, :-1], dist[:, 1:], ids[:, :-1], ids[:, 1:]
	assert ((d0 < d1) | ((d0 == d1) & (i0 < i1))).all()


# ---- 1. known answers, exact -----------------------------------------------------------------------------------------
def dyadic_theta(K):
	"""columns of theta whose square roots are dyadic: one-hot, uniform over 4 or 16 topics, 9/16 + 7 x 1/16"""
	cols = []
	for k in range(0, K, 3):
		cols.append(np.eye(K)[:, k])
	for start in range(0, K - 16, 5):
		u4 = np.zeros(K)
		u4[start:start + 4] = .25
		u16 = np.zeros(K)
		u16[start:start + 16] = 1. / 16
		peak = np.zeros(K)
		peak[start] = 9. / 16
		peak[start + 1:start + 8] = 1. / 16
		cols += [u4, u16, peak]
	return np.array(cols).T


@pytest.mark.parametrize('precision', PRECISIONS)
def test_exact_dyadic(capi, precision):
	K = 40
	theta = dyadic_theta(K)
	theta = np.concatenate([theta, theta[:, ::7]], axis=1)     # duplicates: the tie goes to the smaller id
	D = theta.shape[1]
	scale = 2. ** (np.arange(D) % 13 - 6)                      # gamma = theta times a power of two per column
	gamma = np.asfortranarray(theta * scale)
	# every operation is exact: sqrt(theta) and their products are dyadic, and C = 1 - (a dyadic number)
	c = np.sqrt(theta).T @ np.sqrt(theta)
	want_dist = np.sqrt(np.maximum(0., 1. - c))
	n = 12
	order = np.lexsort((np.broadcast_to(np.arange(D), c.shape), -c), axis=1)[:, :n]
	model = new_model(capi, K, precision)
	model.index_documents(gamma)
	ids, dist = model.similar_documents(gamma, n)
	assert np.array_equal(ids, order)
	assert np.array_equal(dist, np.take_along_axis(want_dist, order, axis=1))
	assert (dist[:, 0] == 0.).all()
	model.close()


@pytest.mark.parametrize('precision', PRECISIONS)
def test_one_topic(capi, precision):
	rng = np.random.default_rng(1)
	model = new_model(capi, 1, precision)
	model.index_documents(rng.gamma(1., 1., size=(1, 300)))
	ids, dist = model.similar_documents(rng.gamma(1., 1., size=(1, 5)), 32)
	assert np.array_equal(ids, np.broadcast_to(np.arange(32), (5, 32)))
	assert (dist == 0.).all()
	model.close()


# ---- 2. against numpy ------------------------------------------------------------------------------------------------
SHAPES = [
	# K, D, Q, n
	(1, 50, 3, 1),
	(33, 1000, 7, 10),
	(33, 777, 300, 32),
	(1000, 3001, 5, 10),
	(1000, 3001, 200, 1),
	(4096, 1500, 70, 32),
	(4096, 300, 1, 32),
]


@pytest.mark.parametrize('K,D,Q,n', SHAPES)
def test_vs_numpy(capi, K, D, Q, n):
	rng = np.random.default_rng(K * 7 + D + Q)
	gd, gq = gammas(rng, K, D), gammas(rng, K, Q)
	gq[:, 0] = gd[:, D // 2] * 3.      # a query equal to an indexed document, up to scale
	model = new_model(capi, K)
	model.index_documents(gd)
	ids, dist = model.similar_documents(gq, n)
	check_against_numpy(ids, dist, gq, gd, n)
	if K > 1:
		assert ids[0, 0] == D // 2
	model.close()


# ---- 3. independence, bitwise ----------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_path_and_batch_independence(capi, precision):
	rng = np.random.default_rng(3)
	for K, D, Q in ((1000, 5000, 1024), (100, 20000, 8192)):
		gd, gq = gammas(rng, K, D), gammas(rng, K, Q)
		model = new_model(capi, K, precision)
		model.index_documents(gd)
		ids, dist = model.similar_documents(gq, 10)           # the product path
		for q in (0, 1, Q // 2, Q - 1):
			one = model.similar_documents(gq[:, q:q + 1], 10)   # the streaming path
			assert np.array_equal(one[0][0], ids[q]) and np.array_equal(one[1][0], dist[q])
		few = model.similar_documents(gq[:, 5:45], 10)         # 40 queries: the streaming path, 5 query groups
		assert np.array_equal(few[0], ids[5:45]) and np.array_equal(few[1], dist[5:45])
		model.close()


def test_index_permutation(capi):
	rng = np.random.default_rng(4)
	K, D, Q = 200, 6000, 150
	gd, gq = gammas(rng, K, D), gammas(rng, K, Q)
	perm = rng.permutation(D)
	model = new_model(capi, K)
	model.index_documents(gd)
	ids, dist = model.similar_documents(gq, 16)
	model.index_documents(gd[:, perm])
	ids_p, dist_p = model.similar_documents(gq, 16)
	assert np.array_equal(perm[ids_p], ids) and np.array_equal(dist_p, dist)
	model.close()


def test_precisions_agree(capi):
	rng = np.random.default_rng(5)
	K, D = 300, 4000
	gd = gammas(rng, K, D)
	out = []
	for precision in PRECISIONS:
		model = new_model(capi, K, precision)
		model.index_documents(gd)
		out.append([model.similar_documents(gammas(np.random.default_rng(Q), K, Q), 10) for Q in (1, 500)])
		model.close()
	for a, b in zip(out[0], out[1]):
		assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


# ---- 4. self-retrieval -----------------------------------------------------------------------------------------------
def test_self_retrieval_random(capi):
	rng = np.random.default_rng(6)
	K, D = 500, 3000
	gd = gammas(rng, K, D)
	model = new_model(capi, K)
	model.index_documents(gd)
	for cols in (np.arange(D), np.arange(0, D, 97)):
		ids, dist = model.similar_documents(gd[:, cols], 5)
		assert np.array_equal(ids[:, 0], cols)
		assert (dist[:, 0] < 1e-6).all()       # the square root of the rounding of C_dd = 1, about K 2^-53
	model.close()


# a model with the true topics, its gamma of the first 60 % of every document indexed and queried with the rest: the right
# document is among the 10 nearest of 0.889 (fp64) / 0.891 (mixed) of the queries on an NVIDIA B200; chance is 10 / 2000
SELF_HIT_BOUND = .5


@pytest.mark.parametrize('precision', PRECISIONS)
def test_self_retrieval_corpus(capi, precision):
	from trlda.utils import split_documents
	from trlda_b200.synth import make_corpus, make_topics
	K, V, B = 50, 3000, 2000
	corpus = make_corpus(B, V, K, .1, .2, mean_length=200, seed=11)
	first, second = split_documents(corpus, .4, seed=2)
	model = capi.Model('online', V, K, 10000, .1, .2, precision=precision)
	model.lambdas = np.asfortranarray(make_topics(V, K, .2, seed=11) * 1e4 + .01)
	gamma_first = model.update_variables(capi.CSR(*first), want_sstats=False)[0]
	gamma_second = model.update_variables(capi.CSR(*second), want_sstats=False)[0]
	model.index_documents(gamma_first)
	ids, _ = model.similar_documents(gamma_second, 10)
	hits = float(np.mean((ids == np.arange(B)[:, None]).any(axis=1)))
	print('self-retrieval hit rate in the top 10:', hits)
	assert hits > SELF_HIT_BOUND
	model.close()


# ---- 5. state and errors ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_training_state_and_index_lifetime(capi, precision):
	from trlda_b200.synth import make_corpus
	rng = np.random.default_rng(7)
	K, V = 64, 2000
	train = capi.CSR(*make_corpus(200, V, K, .1, .2, mean_length=60, seed=3))
	lam0 = np.asfortranarray(rng.gamma(100., .01, size=(K, V)))
	model = capi.Model('online', V, K, 10000, .1, .2, precision=precision)
	model.lambdas = lam0
	model.upload_docs_slot(train, 1)
	gd, gq = gammas(rng, K, 3000), gammas(rng, K, 40)
	before = (model.lambdas, model.alpha, model.eta, model.update_count)
	model.index_documents(gd)
	first = model.similar_documents(gq, 8)
	after = (model.lambdas, model.alpha, model.eta, model.update_count)
	assert all(np.array_equal(a, b) for a, b in zip(before, after))
	# the parked slot is intact: training on it gives what it gives without the calls above
	model.select_docs(1)
	capi.seed(5)
	model.update_parameters_resident(max_iter_tr=2, max_iter_inference=20)
	twin = capi.Model('online', V, K, 10000, .1, .2, precision=precision)
	twin.lambdas = lam0
	twin.upload_docs_slot(train, 1)
	twin.select_docs(1)
	capi.seed(5)
	twin.update_parameters_resident(max_iter_tr=2, max_iter_inference=20)
	assert np.array_equal(model.lambdas, twin.lambdas)
	twin.close()
	# the index survives training, set_lambda and set_precision
	model.update_parameters(train, max_iter_tr=1, max_iter_inference=10)
	model.lambdas = model.lambdas * 2.
	model.precision = 'mixed' if precision == 'fp64' else 'fp64'
	again = model.similar_documents(gq, 8)
	assert np.array_equal(first[0], again[0]) and np.array_equal(first[1], again[1])
	# re-indexing replaces the index
	model.index_documents(gd[:, :100])
	ids, _ = model.similar_documents(gq, 8)
	assert (ids < 100).all()
	model.close()


def test_index_memory_is_freed(capi):
	import torch
	rng = np.random.default_rng(8)
	K, D = 1000, 100000                   # 800 MB of index
	model = new_model(capi, K)
	free0 = torch.cuda.mem_get_info(0)[0]
	model.index_documents(gammas(rng, K, D))
	free1 = torch.cuda.mem_get_info(0)[0]
	assert free0 - free1 >= 8 * K * D * .9
	model.index_documents(np.zeros((K, 0)))
	free2 = torch.cuda.mem_get_info(0)[0]
	assert abs(free2 - free0) < (64 << 20)
	status, message = _raw_similar(capi, model, gammas(rng, K, 2), 1)
	assert (status, message) == (capi.ERR_ARG, 'similar_documents: no documents are indexed.')
	model.close()


def _raw_index(capi, model, gamma, rows=None, cols=None):
	status = model._lib.trlda_index_documents(model.h, capi._dptr(gamma), gamma.shape[0] if rows is None else rows,
		gamma.shape[1] if cols is None else cols)
	return status, model._lib.trlda_last_error(model.h).decode()


def _raw_similar(capi, model, gamma, n, ids=True, dist=True):
	q = gamma.shape[1]
	out_ids = np.full((max(q, 1), max(n, 1)), -1, dtype=np.int64)
	out_dist = np.full((max(q, 1), max(n, 1)), -1.)
	status = model._lib.trlda_similar_documents(model.h, capi._dptr(gamma), gamma.shape[0], q, n,
		out_ids.ctypes.data_as(C.POINTER(C.c_int64)) if ids else None, capi._dptr(out_dist) if dist else None)
	if status != 0:
		assert (out_ids == -1).all() and (out_dist == -1.).all()     # nothing written
	return status, model._lib.trlda_last_error(model.h).decode()


def test_errors(capi):
	rng = np.random.default_rng(9)
	K, D = 20, 40
	model = new_model(capi, K)
	good = gammas(rng, K, D)
	assert _raw_similar(capi, model, good, 1) == (capi.ERR_ARG, 'similar_documents: no documents are indexed.')
	assert _raw_index(capi, model, np.asfortranarray(good[:-1])) == (capi.ERR_ARG, 'Gamma has wrong dimensionality.')
	assert _raw_index(capi, model, good, cols=(1 << 31)) == (capi.ERR_ARG, 'Too many documents to index.')
	bads = []
	for value in (-1e-3, np.nan, np.inf):
		bad = good.copy(order='F')
		bad[3, 7] = value
		bads.append(bad)
	zero = good.copy(order='F')
	zero[:, 11] = 0.
	bads.append(zero)
	for bad in bads:
		assert _raw_index(capi, model, good)[0] == capi.OK
		assert _raw_index(capi, model, bad) == (capi.ERR_ARG, BAD_GAMMA)
		# a failed index leaves none
		assert _raw_similar(capi, model, good, 1) == (capi.ERR_ARG, 'similar_documents: no documents are indexed.')
	assert _raw_index(capi, model, good)[0] == capi.OK
	for bad in bads:
		assert _raw_similar(capi, model, bad, 3) == (capi.ERR_ARG, BAD_GAMMA)
	assert _raw_similar(capi, model, np.asfortranarray(good[:-1]), 3) == (capi.ERR_ARG, 'Gamma has wrong dimensionality.')
	for n in (0, 33, D + 1):
		assert _raw_similar(capi, model, good, n) == (capi.ERR_ARG, N_RANGE)
	assert _raw_similar(capi, model, good, 3, ids=False) == (capi.ERR_ARG, 'similar_documents: no output buffer.')
	# dist_out may be NULL, Q = 0 does nothing, and the model still answers
	assert _raw_similar(capi, model, good, 3, dist=False)[0] == capi.OK
	assert _raw_similar(capi, model, np.zeros((K, 0), order='F'), 3)[0] == capi.OK
	ids, dist = model.similar_documents(good, 32)
	check_against_numpy(ids, dist, good, good, 32)
	model.close()


def test_python_api_all_kinds():
	import trlda.models
	rng = np.random.default_rng(10)
	K, V, D = 30, 500, 700
	gd, gq = gammas(rng, K, D), gammas(rng, K, 9)
	results = []
	for model in (trlda.models.OnlineLDA(V, K, 1000, .1, .2), trlda.models.BatchLDA(V, K, .1, .2),
	              trlda.models.CumulativeLDA(V, K, .1, .2)):
		assert model.index_documents(gd) is None
		ids, dist = model.similar_documents(gq, num_neighbors=7)
		assert ids.dtype == np.int64 and dist.dtype == np.float64 and ids.shape == dist.shape == (9, 7)
		default = model.similar_documents(gq)
		assert default[0].shape == (9, 10)
		check_against_numpy(ids, dist, gq, gd, 7)
		results.append((ids, dist))
		with pytest.raises(RuntimeError, match='Number of neighbors'):
			model.similar_documents(gq, 0)
	for ids, dist in results[1:]:
		assert np.array_equal(ids, results[0][0]) and np.array_equal(dist, results[0][1])
