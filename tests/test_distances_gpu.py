"""
Distances between topics on the device: trlda_topic_distances (Hellinger and Kullback-Leibler, between the topics of one
model or of two), against numpy, its exact properties, topic recovery by training on a corpus with known topics, and its
errors.
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PRECISIONS = ['fp64', 'mixed']
METRICS = ['hellinger', 'kullback_leibler']
# bounds on the diagonal of a self-comparison at V = 100 k.  The device measured 6.2e-8 (Hellinger: the square root of
# |1 - C_ii|, about 4e-15) and 5.2e-14 (KL) on an NVIDIA B200; numpy on the CPU gives |1 - C_ii| = 9e-16 and KL 1.4e-14
HELLINGER_FLOOR = 1e-6
KL_FLOOR = 1e-12


@pytest.fixture(scope='module')
def capi():
	from trlda_b200 import capi
	capi.lib()        # raises if libtrlda_b200.so is missing
	return capi


def random_lambda(rng, K, V, spread):
	"""Gamma(100, 1/100) (the law of the initial lambda: nearly uniform topics) or Gamma(0.3, 1) + 1e-3 (distinct topics)"""
	if spread:
		return np.asfortranarray(rng.gamma(.3, 1., size=(K, V)) + 1e-3)
	return np.asfortranarray(rng.gamma(100., .01, size=(K, V)))


def model_with(capi, lam, precision='fp64'):
	K, V = lam.shape
	model = capi.Model('online', V, K, 1000, .1, .2, precision=precision)
	model.lambdas = lam
	return model


def numpy_product(lam_a, lam_b, metric):
	"""C = f(P_A) g(P_B)^T and the row entropies of P_A"""
	pa = lam_a / lam_a.sum(axis=1, keepdims=True)
	pb = lam_b / lam_b.sum(axis=1, keepdims=True)
	if metric == 'hellinger':
		return np.sqrt(pa) @ np.sqrt(pb).T, None
	return pa @ np.log(pb).T, np.sum(pa * np.log(np.where(pa > 0, pa, 1.)), axis=1)   # 0 log 0 = 0


def check_against_numpy(d, lam_a, lam_b, metric):
	c, h = numpy_product(lam_a, lam_b, metric)
	assert d.shape == (lam_a.shape[0], lam_b.shape[0]) and d.flags.f_contiguous and np.isfinite(d).all()
	if metric == 'hellinger':
		# C is a sum of V positive products of at most 1 in total: its rounding error is about V 2^-53
		assert float(np.max(np.abs(d * d - np.maximum(0., 1. - c)))) < 1e-10
		assert (d >= 0).all() and (d <= 1).all()
	else:
		assert float(np.max(np.abs(d - np.maximum(0., h[:, None] - c)))) < 1e-9
		assert (d >= 0).all()


# ---- 1. against numpy ------------------------------------------------------------------------------------------------
SHAPES = [
	# K_A, K_B, V, other = self, spread-out topics
	(1, 1, 20, True, True),
	(1, 1, 20, False, True),
	(33, 17, 5000, False, True),
	(33, 33, 5000, True, True),
	(1000, 1000, 100000, True, False),
	(1000, 100, 100000, False, False),
	(4096, 50, 3000, False, True),
	(129, 257, 777, False, True),
]


@pytest.mark.parametrize('KA,KB,V,self_,spread', SHAPES)
@pytest.mark.parametrize('metric', METRICS)
def test_vs_numpy(capi, KA, KB, V, self_, spread, metric):
	rng = np.random.default_rng(KA * 31 + KB * 7 + V)
	lam_a = random_lambda(rng, KA, V, spread)
	a = model_with(capi, lam_a)
	if self_:
		d = a.topic_distances(None, metric)
		lam_b = lam_a
	else:
		lam_b = random_lambda(rng, KB, V, spread)
		b = model_with(capi, lam_b)
		d = a.topic_distances(b, metric)
		b.close()
	a.close()
	check_against_numpy(d, lam_a, lam_b, metric)


# ---- 2. exact properties -----------------------------------------------------------------------------------------------
def test_self_comparison_symmetric_with_diagonal_at_floor(capi):
	rng = np.random.default_rng(11)
	lam = random_lambda(rng, 1000, 100000, False)
	model = model_with(capi, lam)
	d = model.topic_distances()
	kl = model.topic_distances(metric='kullback_leibler')
	model.close()
	assert np.array_equal(d, d.T)                       # bitwise
	print('self diagonal: Hellinger max %.3g, KL max %.3g' % (np.diag(d).max(), np.diag(kl).max()))
	assert float(np.diag(d).max()) <= HELLINGER_FLOOR
	assert float(np.diag(kl).max()) <= KL_FLOOR
	off = ~np.eye(1000, dtype=bool)
	assert float(d[off].min()) > 100 * HELLINGER_FLOOR and float(kl[off].min()) > 100 * KL_FLOOR
	assert (kl >= 0).all()


@pytest.mark.parametrize('metric', METRICS)
def test_permutation_is_recovered(capi, metric):
	from scipy.optimize import linear_sum_assignment
	rng = np.random.default_rng(5)
	K, V = 300, 20000
	lam = random_lambda(rng, K, V, True)
	perm = rng.permutation(K)
	a, b = model_with(capi, lam), model_with(capi, np.asfortranarray(lam[perm]))
	d = a.topic_distances(b, metric)                    # topic j of b is topic perm[j] of a
	a.close()
	b.close()
	floor = HELLINGER_FLOOR if metric == 'hellinger' else KL_FLOOR
	assert float(d[perm, np.arange(K)].max()) <= floor
	assert np.array_equal(np.argmin(d, axis=0), perm)
	rows, cols = linear_sum_assignment(d)
	assert np.array_equal(rows, np.arange(K)) and np.array_equal(cols, np.argsort(perm))


@pytest.mark.parametrize('metric', METRICS)
def test_bitwise_across_modes_and_calls(capi, metric):
	rng = np.random.default_rng(8)
	lam_a, lam_b = random_lambda(rng, 300, 30000, True), random_lambda(rng, 200, 30000, True)
	out = {}
	for precision in PRECISIONS:
		a, b = model_with(capi, lam_a, precision), model_with(capi, lam_b, precision)
		out[precision] = [a.topic_distances(b, metric), a.topic_distances(None, metric), a.topic_distances(b, metric)]
		a.close()
		b.close()
	first = out['fp64']
	assert np.array_equal(first[0], first[2])
	for precision in PRECISIONS:
		for got, want in zip(out[precision], first):
			assert np.array_equal(got, want)
	check_against_numpy(first[0], lam_a, lam_b, metric)


def test_launches_count_as_misc(capi):
	lam = random_lambda(np.random.default_rng(1), 64, 3000, True)
	model = model_with(capi, lam)
	model.reset_stats()
	model.topic_distances()
	stats = model.stats()
	model.close()
	assert stats['launches']['misc'] > 0
	assert sum(n for kind, n in stats['launches'].items() if kind not in ('misc', 'rowsum', 'reduce')) == 0


def test_models_on_different_devices(capi):
	import torch
	if torch.cuda.device_count() < 2:
		pytest.skip('needs two GPUs')
	lam = random_lambda(np.random.default_rng(2), 8, 100, True)
	a = model_with(capi, lam)
	b = capi.Model('online', 100, 8, 1000, .1, .2, device=1)
	b.lambdas = lam
	assert _raw(capi, a, b, 0) == (capi.ERR_ARG, 'The two models must be on the same device.')
	a.close()
	b.close()


# ---- 3. recovery of known topics ---------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_training_recovers_the_topics(precision):
	from scipy.optimize import linear_sum_assignment
	import trlda
	import trlda.models
	from trlda_b200.synth import make_corpus, make_topics
	K, V, seed = 20, 2000, 17
	trlda.seed(3)
	truth = trlda.models.BatchLDA(V, K, .1, .2)
	truth.lambdas = make_topics(V, K, seed=seed)
	model = trlda.models.OnlineLDA(V, K, 100000, .1, .2)
	model.precision = precision

	def matched():
		d = model.topic_distances(truth)
		rows, cols = linear_sum_assignment(d)
		return float(d[rows, cols].mean())

	before = matched()
	for step in range(30):
		model.update_parameters(make_corpus(256, V, K, .1, .2, mean_length=100, seed=seed, doc_seed=step), max_iter_tr=2)
	after = matched()
	print('%s: mean matched Hellinger distance to the true topics before %.4f after %.4f' % (precision, before, after))
	# NVIDIA B200: 0.606 before, 0.315 after in fp64
	assert before > .5
	assert after < .4 and after < .65 * before


# ---- 4. training state ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_training_state_untouched(capi, precision):
	from trlda_b200.synth import make_corpus
	K, V = 256, 4000
	train = capi.CSR(*make_corpus(300, V, K, .1, .2, mean_length=60, seed=3))
	lam0 = np.asfortranarray(np.random.default_rng(2).gamma(100., .01, size=(K, V)))
	lam_other = np.asfortranarray(np.random.default_rng(4).gamma(100., .01, size=(50, V)))
	kwargs = dict(max_iter_tr=2, max_iter_inference=20, update_alpha=1, update_eta=1)
	results = []
	for evaluate in (True, False):
		model = capi.Model('online', V, K, 10000, .1, .2, precision=precision)
		model.lambdas = lam0
		model.update_count = 3
		model.upload_docs_slot(train, 1)
		if evaluate:
			other = model_with(capi, lam_other, precision)
			before = (model.lambdas, model.alpha, model.eta, model.update_count)
			for metric in METRICS:
				model.topic_distances(None, metric)
				model.topic_distances(other, metric)
				other.topic_distances(model, metric)
			after = (model.lambdas, model.alpha, model.eta, model.update_count)
			assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
			assert before[2] == after[2] and before[3] == after[3]
			assert np.array_equal(other.lambdas, lam_other)
			other.close()
		model.select_docs(1)
		capi.seed(5)
		model.update_parameters_resident(**kwargs)
		results.append(model.lambdas)
		model.close()
	assert np.array_equal(results[0], results[1])


# ---- 5. errors ---------------------------------------------------------------------------------------------------------
def _raw(capi, model, other, metric, with_out=True):
	k_other = model.K if other is None else other.K
	out = np.zeros(model.K * k_other)
	status = model._lib.trlda_topic_distances(model.h, None if other is None else other.h, metric,
		out.ctypes.data_as(C.POINTER(C.c_double)) if with_out else None)
	return status, model._lib.trlda_last_error(model.h).decode()


def test_errors(capi):
	K, V = 6, 50
	rng = np.random.default_rng(0)
	good = random_lambda(rng, K, V, True)
	a, b = model_with(capi, good), model_with(capi, random_lambda(rng, 4, V, True))
	wide = model_with(capi, random_lambda(rng, K, V + 1, True))
	negative = good.copy()
	negative[2, 7] = -1e-3
	zero = good.copy()
	zero[3, 9] = 0.
	neg_model, zero_model = model_with(capi, negative), model_with(capi, zero)
	negative_msg = 'topic_distances: lambda has a negative entry.'
	zero_msg = 'topic_distances: the Kullback-Leibler distance needs a positive lambda in the second model.'
	cases = [
		(a, b, 2, True, 'Unknown distance metric.'),
		(a, b, -1, True, 'Unknown distance metric.'),
		(a, b, 0, False, 'topic_distances: no output buffer.'),
		(a, wide, 0, True, 'The two models must have the same number of words.'),
		(wide, a, 1, True, 'The two models must have the same number of words.'),
		(neg_model, None, 0, True, negative_msg),
		(neg_model, None, 1, True, negative_msg),
		(a, neg_model, 0, True, negative_msg),
		(neg_model, a, 1, True, negative_msg),
		(a, zero_model, 1, True, zero_msg),
		(zero_model, None, 1, True, zero_msg),
	]
	for m, other, metric, with_out, message in cases:
		assert _raw(capi, m, other, metric, with_out) == (capi.ERR_ARG, message)
		assert np.isfinite(a.topic_distances(b)).all()     # the model still works
	# zeros are fine where no log is taken of them
	for m, other, metric in ((zero_model, None, 0), (zero_model, a, 1), (a, zero_model, 0)):
		assert _raw(capi, m, other, metric)[0] == capi.OK
	check_against_numpy(zero_model.topic_distances(a, 'kullback_leibler'), zero, good, 'kullback_leibler')
	for m in (a, b, wide, neg_model, zero_model):
		m.close()


def test_python_api(capi):
	import trlda.models
	K, V = 12, 300
	rng = np.random.default_rng(3)
	lam_a, lam_b = random_lambda(rng, K, V, True), random_lambda(rng, 5, V, True)
	models = [trlda.models.OnlineLDA(V, K, 1000, .1, .2), trlda.models.BatchLDA(V, K, .1, .2),
		trlda.models.CumulativeLDA(V, K, .1, .2)]
	other = trlda.models.BatchLDA(V, 5, .1, .2)
	other.lambdas = lam_b
	for model in models:
		model.lambdas = lam_a
		d = model.topic_distances()
		assert d.shape == (K, K) and d.flags.f_contiguous and np.array_equal(d, d.T)
		assert np.array_equal(model.topic_distances(metric='hellinger'), d)
		for metric in METRICS:
			d = model.topic_distances(other, metric=metric)
			assert d.shape == (K, 5) and d.flags.f_contiguous
			check_against_numpy(d, lam_a, lam_b, metric)
			assert np.array_equal(d, model.topic_distances(other=other, metric=metric))
		with pytest.raises(TypeError):
			model.topic_distances(lam_b)
		with pytest.raises(TypeError):
			model.topic_distances(capi.Model('batch', V, 5, 0, .1, .2))
		with pytest.raises(ValueError, match='metric'):
			model.topic_distances(metric='jensen_shannon')
		with pytest.raises(RuntimeError, match='same number of words'):
			model.topic_distances(trlda.models.BatchLDA(V + 1, 5, .1, .2))
	# the ctypes view
	a, b = model_with(capi, lam_a), model_with(capi, lam_b)
	assert np.array_equal(a.topic_distances(b), models[0].topic_distances(other))
	a.close()
	b.close()
