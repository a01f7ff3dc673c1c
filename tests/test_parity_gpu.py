"""
GPU parity tests (`-m gpu`): the CUDA path, driven through the C ABI (include/trlda_b200.h) with host buffers,
against the CPU oracle on the same seeded inputs and against the golden fixtures generated from the compiled
reference.  Tolerances are BASELINE.json's: fp64 mode <= 1e-9 relative on gamma / lambda / alpha / eta; mixed
(fp32 tile + fp32 inner products, fp64 accumulation) <= 1e-4 relative and per-document ELBO <= 1e-5 relative, each
measured by common.parity_err (elementwise in fp64 mode, per column in the infinity norm in mixed mode).
"""
import os

import numpy as np
import pytest

from common import (TOL_ELBO_MIXED, TOL_FP64, TOL_MIXED, load_case, mixed_flip_check, parity_err, random_docs, rel_err, rel_err_columns,
	run_batch_case, run_cumulative_case, run_online_case)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def capi():
	from trlda_b200 import capi
	capi.lib()        # raises if libtrlda_b200.so is missing: the GPU tests never fall back to anything else
	return capi


def tol(precision):
	return TOL_FP64 if precision == 'fp64' else TOL_MIXED


# ---- special functions -----------------------------------------------------------------------------------------------
def test_device_special_functions_vs_reference_fixture(capi):
	case = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'special.npz'))
	x = case['x']
	for which, name, bound in ((0, 'digamma', 2e-14), (1, 'trigamma', 2e-14), (2, 'lngamma', 2e-13)):
		got = capi.device_special(which, x)
		scale = np.maximum(np.abs(case[name]), 1e-3)
		assert np.max(np.abs(got - case[name]) / scale) < bound, name


def test_device_digamma_known_answers(capi):
	# python/tests/utils_test.py:35-41 (7 places)
	x = np.array([.1, 1., 120., .01, .1, .4, 11.])
	psi = capi.device_special(0, x[:3])
	assert np.allclose(psi, [-10.423754940411, -0.5772156649015329, 4.7833192891185], rtol=0, atol=5e-8)
	tri = capi.device_special(1, x[3:])
	assert np.allclose(tri, [10001.6212135283, 101.433299150792758, 7.275356590529597, 0.09516633568168575], rtol=1e-10)


def test_device_exp_digamma_variants(capi):
	"""the log-free exp(psi(x)) used by the kernels: the fp64-mode evaluation to a few ulp, the mixed-mode one
	(recurrence to s >= 6, MUFU-seeded reciprocal) far inside the float32 rounding it feeds"""
	case = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'special.npz'))
	x = case['x'][case['x'] > 1e-3]
	want = np.exp(case['digamma'][case['x'] > 1e-3])
	ok = want > 1e-300
	assert np.max(np.abs(capi.device_special(4, x)[ok] - want[ok]) / want[ok]) < 5e-13
	assert np.max(np.abs(capi.device_special(3, x)[ok] - want[ok]) / want[ok]) < 1e-10
	# the branch-free evaluation inside the mixed-mode E-step kernel (Estrin polynomials, degree-9 exp): 2e-11
	assert np.max(np.abs(capi.device_special(5, x)[ok] - want[ok]) / want[ok]) < 1e-10
	dense = np.exp(np.random.default_rng(0).uniform(np.log(1e-3), np.log(1e5), size=20000))
	exact = capi.device_special(4, dense)
	big = exact > 1e-290          # below, the kernel's evaluation flushes to zero (exponent patch); float32 underflows at 1e-45
	assert np.max(np.abs(capi.device_special(5, dense)[big] - exact[big]) / exact[big]) < 1e-10


# ---- E-step ----------------------------------------------------------------------------------------------------------
ESTEP_SHAPES = [
	# K, V, B, max_len, max_iter
	(1, 10, 4, 6, 10),
	(12, 60, 9, 30, 20),
	(33, 45, 7, 40, 50),       # K not a multiple of 32
	(100, 700, 40, 150, 20),   # cfg-1 topic count
	(200, 500, 24, 120, 20),
	(500, 400, 12, 150, 20),   # cfg-4 topic count: cluster of 2-4 CTAs per document
	(1000, 600, 10, 150, 20),  # cfg-3 topic count: cluster of 8 CTAs per document
	(1000, 600, 6, 150, 0),    # max_iter = 0: statistics from the initial gamma
	(2048, 300, 8, 60, 20),    # fp64: cluster kernel, whole tile in shared memory
	(1040, 400, 16, 300, 20),  # mixed: documents of > 192 pairs on the cluster kernel, the rest in tensor memory
	(2560, 300, 6, 100, 10),   # mixed: K beyond the tensor-memory kernel
	(4096, 200, 4, 60, 5),     # the topic limit: cluster of 8 CTAs, 512 rows each
]


@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
@pytest.mark.parametrize('K,V,B,max_len,max_iter', ESTEP_SHAPES)
def test_update_variables_vs_oracle(capi, oracle_built, precision, K, V, B, max_len, max_iter):
	rng = np.random.default_rng(K * 7 + B)
	lists = random_docs(rng, B, V, min(V, max_len), empty=(1,) if B > 2 else (), duplicates=(2,) if B > 3 else ())
	lam0 = np.asfortranarray(rng.gamma(100., .01, size=(V, K)).T)
	g0 = np.asfortranarray(rng.gamma(100., .01, size=(B, K)).T)
	alpha = rng.uniform(.05, .5, size=K)

	port = oracle_built.PortModel('online', V, K, 1000, alpha, .2)
	port.lambdas = lam0
	want_gamma, want_sstats, want_it = port.update_variables(
		oracle_built.CSR.from_lists(lists), g0, max_iter=max_iter, want_iterations=True)

	model = capi.Model('online', V, K, 1000, alpha, .2, precision=precision)
	model.lambdas = lam0
	gamma, sstats = model.update_variables(capi.CSR.from_lists(lists), g0, max_iter=max_iter)
	stats = model.stats()

	assert parity_err(gamma, want_gamma, precision) < tol(precision)
	assert rel_err_columns(sstats, want_sstats) < tol(precision)      # per word: not in the tolerance list, see below
	# sum of the statistics is the token mass of the minibatch regardless of phi
	assert np.sum(sstats) == pytest.approx(sum(c for doc in lists for _, c in doc), rel=1e-6)
	if precision == 'fp64':
		assert stats['estep_doc_iterations'] == int(want_it.sum())    # identical early exits
	assert stats['estep_sweeps'] == stats['estep_doc_iterations'] + B  # every E-step kernel counts its sweeps


def test_update_variables_draws_gamma_when_no_latents(capi):
	capi.seed(123)
	rng = np.random.default_rng(0)
	lists = random_docs(rng, 20, 50, 20)
	model = capi.Model('online', 50, 16, 100, .1, .2)
	gamma, sstats = model.update_variables(capi.CSR.from_lists(lists), max_iter=0)
	# with max_iter = 0 gamma is the initial draw itself: Gamma(100, 1/100), mean 1, std .1 (lda.cpp:135)
	assert gamma.shape == (16, 20) and np.all(gamma > 0)
	assert abs(gamma.mean() - 1.) < .03 and abs(gamma.std() - .1) < .03
	lam = model.lambdas                                               # lda.cpp:71, same law
	assert abs(lam.mean() - 1.) < .02 and abs(lam.std() - .1) < .02


def test_update_variables_long_documents_stream_from_l2(capi, oracle_built):
	"""documents with more distinct words than fit in shared memory: the tail of the tile streams from L2"""
	rng = np.random.default_rng(4)
	K, V, B = 1000, 3000, 3
	lists = [[(int(w), int(1 + rng.integers(5))) for w in rng.permutation(V)[:n]] for n in (2500, 17, 1200)]
	lam0 = np.asfortranarray(rng.gamma(100., .01, size=(V, K)).T)
	g0 = np.asfortranarray(rng.gamma(100., .01, size=(B, K)).T)
	port = oracle_built.PortModel('online', V, K, 1000, .1, .2)
	port.lambdas = lam0
	want_gamma, want_sstats = port.update_variables(oracle_built.CSR.from_lists(lists), g0, max_iter=8)
	for precision in ('fp64', 'mixed'):
		model = capi.Model('online', V, K, 1000, .1, .2, precision=precision)
		model.lambdas = lam0
		gamma, sstats = model.update_variables(capi.CSR.from_lists(lists), g0, max_iter=8)
		assert rel_err_columns(gamma, want_gamma) < tol(precision)
		assert rel_err(sstats, want_sstats) < tol(precision)


def test_wrong_latents_shape_raises_reference_message(capi):
	model = capi.Model('online', 20, 4, 10)
	docs = capi.CSR.from_lists([[(1, 1)], [(2, 2)]])
	with pytest.raises(RuntimeError, match='Initial gamma has wrong dimensionality.'):     # lda.cpp:166
		model.update_variables(docs, np.ones((4, 3)))
	with pytest.raises(RuntimeError, match='Word ID out of range.'):
		model.update_variables(capi.CSR.from_lists([[(20, 1)]]), np.ones((4, 1)))


# ---- golden fixtures from the compiled reference ---------------------------------------------------------------------
@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
@pytest.mark.parametrize('name', ['online_tr.npz', 'online_sgd.npz', 'online_adaptive.npz'])
def test_online_golden(capi, name, precision):
	case = load_case(name)
	model = capi.Model('online', case['V'], case['K'], case['D'], case['alpha0'], case['eta0'], precision=precision)
	out = run_online_case(model, capi.CSR, case)
	t = tol(precision)
	assert rel_err_columns(out['estep_gamma'], case['estep_gamma']) < t
	assert rel_err(out['estep_sstats'], case['estep_sstats']) < t
	assert out['rho'] == pytest.approx(float(case['rho']), rel=1e-14)
	assert parity_err(out['lambda1'], case['lambda1'], precision) < t
	assert parity_err(out['alpha1'], case['alpha1'], precision) < t
	assert out['eta1'] == pytest.approx(float(case['eta1']), rel=t)
	assert out['update_count1'] == int(case['update_count1'])


@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
def test_batch_golden(capi, precision):
	case = load_case('batch.npz')
	model = capi.Model('batch', case['V'], case['K'], 0, case['alpha0'], case['eta0'], precision=precision)
	out = run_batch_case(model, capi.CSR, case)
	t = tol(precision)
	assert out['rho'] == 1.
	assert parity_err(out['lambda1'], case['lambda1'], precision) < t
	assert parity_err(out['alpha1'], case['alpha1'], precision) < t
	assert out['eta1'] == pytest.approx(float(case['eta1']), rel=t)


@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
def test_cumulative_golden(capi, precision):
	case = load_case('cumulative.npz')
	model = capi.Model('cumulative', case['V'], case['K'], 0, case['alpha0'], case['eta0'], precision=precision)
	assert np.all(model.lambdas == case['eta0'])                  # cumulativelda.cpp:30
	out = run_cumulative_case(model, capi.CSR, case)
	t = tol(precision)
	for call in range(2):
		assert parity_err(out['lambda1_%d' % call], case['lambda1_%d' % call], precision) < t
		assert parity_err(out['alpha1_%d' % call], case['alpha1_%d' % call], precision) < t


# ---- update_parameters against the oracle at larger shapes -----------------------------------------------------------
@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
@pytest.mark.parametrize('K,V,B', [(100, 7000, 200), (1000, 2000, 64)])
def test_online_update_parameters_vs_oracle(capi, oracle_built, precision, K, V, B):
	"""cfg-1 (README example) in full and cfg-3's topic count on a reduced vocabulary, T=10, I=20, with the
	empirical-Bayes updates on"""
	from trlda_b200.synth import gamma_matrix, make_corpus
	ptr, ids, cts = make_corpus(B, V, K, .1, .2, seed=1001)
	lam0, g0 = gamma_matrix(K, V, 2001), gamma_matrix(K, B, 3001)
	kwargs = dict(max_iter_tr=10, max_iter_inference=20, kappa=.7, tau=100., update_alpha=1, update_eta=1)

	port = oracle_built.PortModel('online', V, K, 1000000, .1, .2)
	port.lambdas = lam0
	want_rho, want_gamma = port.update_parameters(oracle_built.CSR(ptr, ids, cts), gamma0=g0, want_gamma=True, **kwargs)

	model = capi.Model('online', V, K, 1000000, .1, .2, precision=precision)
	model.lambdas = lam0
	rho = model.update_parameters(capi.CSR(ptr, ids, cts), gamma0=g0, **kwargs)

	t = tol(precision)
	assert rho == pytest.approx(want_rho, rel=1e-14)
	assert parity_err(model.lambdas, port.lambdas, precision) < t
	assert parity_err(model.alpha, port.alpha, precision) < t
	assert model.eta == pytest.approx(port.eta, rel=t)
	assert model.update_count == port.update_count == 1


def test_update_count_and_empty_batch_semantics(capi):
	"""onlinelda_test.py:113-124: update_parameters([]) is a no-op returning 1.0 and does not count"""
	rng = np.random.default_rng(1)
	model = capi.Model('online', 100, 10, 1000)
	before = model.lambdas
	assert model.update_parameters(capi.CSR([0], [], [])) == 1.0
	assert model.update_count == 0
	assert np.array_equal(model.lambdas, before)
	docs = capi.CSR.from_lists(random_docs(rng, 10, 100, 5))
	rho0 = model.update_parameters(docs, max_iter_inference=20)
	rho1 = model.update_parameters(docs, max_iter_inference=20)
	assert model.update_count == 2
	assert rho0 == pytest.approx((100. + 0) ** -.7) and rho1 == pytest.approx((100. + 1) ** -.7)   # onlinelda.cpp:65
	assert np.all(np.isfinite(model.lambdas))


def test_resident_path_equals_host_path(capi):
	"""bench.py's device-only leg (docs already in HBM) computes exactly what the host-buffer call computes"""
	from trlda_b200.synth import gamma_matrix, make_corpus
	K, V, B = 64, 500, 50
	docs = capi.CSR(*make_corpus(B, V, K, .1, .2, seed=3))
	lam0, g0 = gamma_matrix(K, V, 4), gamma_matrix(K, B, 5)
	out = []
	for resident in (False, True):
		model = capi.Model('online', V, K, 10000, .1, .2)
		model.lambdas = lam0
		if resident:
			model.upload_docs(docs)
			model.update_parameters_resident(gamma0=g0, max_iter_inference=20)
		else:
			model.update_parameters(docs, gamma0=g0, max_iter_inference=20)
		out.append(model.lambdas)
	assert np.array_equal(out[0], out[1])


def test_runs_are_bitwise_deterministic(capi):
	from trlda_b200.synth import gamma_matrix, make_corpus
	K, V, B = 200, 800, 96
	docs = capi.CSR(*make_corpus(B, V, K, .1, .2, seed=8))
	lam0, g0 = gamma_matrix(K, V, 9), gamma_matrix(K, B, 10)
	out = []
	for _ in range(2):
		model = capi.Model('online', V, K, 10000, .1, .2, precision='mixed')
		model.lambdas = lam0
		model.update_parameters(docs, gamma0=g0, max_iter_inference=20, max_iter_tr=3)
		out.append(model.lambdas)
	assert np.array_equal(out[0], out[1])


# ---- BASELINE.json shapes against the reference at sizes the CPU finishes in seconds ---------------------------------
_CPU_CACHE = {}


def _cpu_once(key, fn):
	"""the CPU side of a test is the same for both precision parameters: computed once per session"""
	if key not in _CPU_CACHE:
		_CPU_CACHE[key] = fn()
	return _CPU_CACHE[key]


def _cpu_model(oracle_built, kind, V, K, D, alpha, eta):
	"""the unmodified reference core where it was compiled (oracle/_ref), else the plain-C port"""
	if oracle_built.have_ref():
		return oracle_built.RefModel(kind, V, K, D, alpha, eta, fast_init=True)
	return oracle_built.PortModel(kind, V, K, D, alpha, eta)


@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
def test_cfg3_shape_vs_reference(capi, oracle_built, precision):
	"""cfg-3's real shape - K=1000 topics over the full V=100 000 vocabulary - on a minibatch the CPU handles:
	B=256 documents, T=2 trust-region iterations, I=20, injected gamma0 / lambda0 (onlinelda.cpp:53-180)"""
	from trlda_b200.synth import gamma_matrix, make_corpus
	K, V, B, D = 1000, 100000, 256, 1000000
	ptr, ids, cts = make_corpus(B, V, K, .1, .2, seed=1003)
	lam0, g0 = gamma_matrix(K, V, 2003), gamma_matrix(K, B, 3003)
	kwargs = dict(max_iter_tr=2, max_iter_inference=20, kappa=.7, tau=100.)

	def cpu_side():
		cpu = _cpu_model(oracle_built, 'online', V, K, D, .1, .2)
		cpu.lambdas = lam0
		rho = cpu.update_parameters(oracle_built.CSR(ptr, ids, cts), gamma0=g0, **kwargs)
		lam1 = cpu.lambdas
		# and the E-step alone on the updated model (gamma, sufficient statistics; lda.cpp:160-220)
		gamma, sstats = cpu.update_variables(oracle_built.CSR(ptr, ids, cts), g0, max_iter=20)
		return rho, lam1, gamma, sstats

	want_rho, want, want_gamma, want_sstats = _cpu_once('cfg3', cpu_side)
	model = capi.Model('online', V, K, D, .1, .2, precision=precision)
	model.lambdas = lam0
	rho = model.update_parameters(capi.CSR(ptr, ids, cts), gamma0=g0, **kwargs)
	assert rho == pytest.approx(want_rho, rel=1e-14)
	assert parity_err(model.lambdas, want, precision) < tol(precision)
	gamma, sstats = model.update_variables(capi.CSR(ptr, ids, cts), g0, max_iter=20)
	assert parity_err(gamma, want_gamma, precision) < tol(precision)
	# the sufficient statistics are not in BASELINE.json's tolerance list (gamma, lambda, alpha, eta); they carry
	# exp(psi(gamma)), which amplifies a 1e-11 difference of a gamma near alpha a hundredfold: per word, infinity norm
	assert rel_err_columns(sstats, want_sstats) < tol(precision)


@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
def test_cfg4_shape_vs_reference(capi, oracle_built, precision):
	"""cfg-4: OnlineLDA K=500, V=50 000 with the empirical-Bayes Newton steps for alpha and eta (onlinelda.cpp:116-162)"""
	from trlda_b200.synth import gamma_matrix, make_corpus
	K, V, B, D = 500, 50000, 256, 1000000
	ptr, ids, cts = make_corpus(B, V, K, .1, .2, seed=1004)
	lam0, g0 = gamma_matrix(K, V, 2004), gamma_matrix(K, B, 3004)
	kwargs = dict(max_iter_tr=3, max_iter_inference=20, kappa=.7, tau=100., update_alpha=1, update_eta=1)

	def cpu_side():
		cpu = _cpu_model(oracle_built, 'online', V, K, D, .1, .2)
		cpu.lambdas = lam0
		cpu.update_parameters(oracle_built.CSR(ptr, ids, cts), gamma0=g0, **kwargs)
		return cpu.lambdas, np.ravel(cpu.alpha), cpu.eta

	want_lam, want_alpha, want_eta = _cpu_once('cfg4', cpu_side)
	model = capi.Model('online', V, K, D, .1, .2, precision=precision)
	model.lambdas = lam0
	model.update_parameters(capi.CSR(ptr, ids, cts), gamma0=g0, **kwargs)
	t = tol(precision)
	if precision == 'fp64':
		assert parity_err(model.lambdas, want_lam, precision) < t
	else:
		# three E-steps at D/B = 3900: one document flips its convergence test (common.mixed_flip_check)
		q999, worst = mixed_flip_check(model.lambdas, want_lam)
		assert q999 < t and worst < 10 * t
	assert parity_err(model.alpha, want_alpha, precision) < t
	assert model.eta == pytest.approx(want_eta, rel=t)


@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
def test_cfg2_shape_vs_port(capi, oracle_built, precision):
	"""cfg-2: BatchLDA K=100, V=10 000, two epochs over 2000 documents with the line-searched alpha / eta updates
	(batchlda.cpp:43-209); every epoch starts from a fresh gamma, injected on both sides through the port's seam"""
	from trlda_b200.synth import gamma_matrix, make_corpus
	K, V, B = 100, 10000, 2000
	ptr, ids, cts = make_corpus(B, V, K, .1, .2, seed=1002)
	lam0, g0 = gamma_matrix(K, V, 2002), gamma_matrix(K, B, 3002)
	kwargs = dict(max_epochs=2, max_iter_inference=20, update_alpha=1, update_eta=1)
	def cpu_side():
		port = oracle_built.PortModel('batch', V, K, 0, .1, .2)
		port.lambdas = lam0
		port.update_parameters(oracle_built.CSR(ptr, ids, cts), gamma0=g0, **kwargs)
		return port.lambdas, np.array(port.alpha), port.eta

	want_lam, want_alpha, want_eta = _cpu_once('cfg2', cpu_side)
	model = capi.Model('batch', V, K, 0, .1, .2, precision=precision)
	model.lambdas = lam0
	model.update_parameters(capi.CSR(ptr, ids, cts), gamma0=g0, **kwargs)
	t = tol(precision)
	assert parity_err(model.lambdas, want_lam, precision) < t
	assert parity_err(model.alpha, want_alpha, precision) < t
	assert model.eta == pytest.approx(want_eta, rel=t)


@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
def test_cfg5_shape_vs_port(capi, oracle_built, precision):
	"""cfg-5: CumulativeLDA K=200, V=100 000 streamed in two batches, with its cross-call alpha statistics
	(cumulativelda.cpp:49-153); lambda's random restart and the fresh gammas are injected on both sides"""
	from trlda_b200.synth import gamma_matrix, make_corpus
	K, V, B = 200, 100000, 128
	ptr, ids, cts = make_corpus(2 * B, V, K, .1, .2, seed=1005)
	kwargs = dict(max_epochs=1, max_iter_inference=20, update_alpha=1)

	def inputs(call):
		lo, hi = ptr[call * B], ptr[(call + 1) * B]
		batch = (ptr[call * B:(call + 1) * B + 1] - lo, ids[lo:hi], cts[lo:hi])
		return batch, gamma_matrix(K, V, 2005 + call), gamma_matrix(K, B, 3005 + call)

	def cpu_side():
		port = oracle_built.PortModel('cumulative', V, K, 0, .1, .2)
		out = []
		for call in range(2):
			batch, lam_rand, g0 = inputs(call)
			port.update_parameters(oracle_built.CSR(*batch), gamma0=g0, lambda0=lam_rand, **kwargs)
			out.append((port.lambdas, np.array(port.alpha)))
		return out

	want = _cpu_once('cfg5', cpu_side)
	model = capi.Model('cumulative', V, K, 0, .1, .2, precision=precision)
	for call in range(2):
		batch, lam_rand, g0 = inputs(call)
		model.update_parameters(capi.CSR(*batch), gamma0=g0, lambda0=lam_rand, **kwargs)
		t = tol(precision)
		assert parity_err(model.lambdas, want[call][0], precision) < t
		assert parity_err(model.alpha, want[call][1], precision) < t


def test_mixed_mode_stays_finite_when_a_column_underflows(capi, oracle_built):
	"""a word every topic has (almost) no mass on: its float32 expElogbeta column underflows to zero, phi hits the
	1e-100 floor of lda.cpp:183 and the token weight leaves the float32 range; the fp64 reference gets 0 * huge = 0,
	the float32 products must not get 0 * inf = NaN"""
	rng = np.random.default_rng(5)
	K, V, B = 64, 300, 12
	lam0 = np.asfortranarray(rng.gamma(100., .01, size=(V, K)).T)
	lam0[:, 7] = .004                  # exp(psi(.004)) ~ 1e-109: zero in float32
	lists = random_docs(rng, B, V, 40)
	lists[3].append((7, 60))           # held-out word with a large count
	lists[5] = [(7, 45)]               # a document of nothing else
	g0 = np.asfortranarray(rng.gamma(100., .01, size=(B, K)).T)
	port = oracle_built.PortModel('online', V, K, 1000, .1, .01)
	port.lambdas = lam0
	want_gamma, want_sstats = port.update_variables(oracle_built.CSR.from_lists(lists), g0, max_iter=20)
	model = capi.Model('online', V, K, 1000, .1, .01, precision='mixed')
	model.lambdas = lam0
	gamma, sstats = model.update_variables(capi.CSR.from_lists(lists), g0, max_iter=20)
	assert np.all(np.isfinite(gamma)) and np.all(np.isfinite(sstats))
	assert parity_err(gamma, want_gamma, 'mixed') < TOL_MIXED
	rho = model.update_parameters(capi.CSR.from_lists(lists), gamma0=g0, max_iter_tr=3, max_iter_inference=20)
	assert np.isfinite(rho) and np.all(np.isfinite(model.lambdas))


def test_parked_minibatch_survives_other_calls(capi):
	"""trlda_select_docs hands the live buffers to a slot; a call that uploads other documents in between (lower_bound,
	update_variables) must park them first, so that selecting the slot again trains on the original minibatch"""
	from trlda_b200.synth import gamma_matrix, make_corpus
	K, V, B = 64, 500, 50
	docs = capi.CSR(*make_corpus(B, V, K, .1, .2, seed=3))
	other = capi.CSR(*make_corpus(30, V, K, .1, .2, seed=4))
	lam0, g0 = gamma_matrix(K, V, 4), gamma_matrix(K, B, 5)
	host = capi.Model('online', V, K, 10000, .1, .2)
	host.lambdas = lam0
	host.update_parameters(docs, gamma0=g0, max_iter_inference=20)
	model = capi.Model('online', V, K, 10000, .1, .2)
	model.lambdas = lam0
	model.upload_docs_slot(docs, 0)
	model.upload_docs_slot(other, 1)
	model.select_docs(0)
	model.lower_bound(other, gamma_matrix(K, 30, 6), max_iter=5)
	model.select_docs(0)
	model.update_parameters_resident(gamma0=g0, max_iter_inference=20)
	assert np.array_equal(model.lambdas, host.lambdas)


def test_parked_minibatches_survive_slot_growth_and_teardown(capi):
	"""uploads into slots 2, 0 and 5 grow the slot vector and move the minibatches parked before; selecting each slot
	then trains on its own documents.  Closing the model with its slots parked frees every buffer once: a second free
	would leave a CUDA error behind that fails the next call on this thread"""
	from trlda_b200.synth import gamma_matrix, make_corpus
	K, V = 64, 500
	batches = {slot: capi.CSR(*make_corpus(B, V, K, .1, .2, seed=10 + slot)) for slot, B in ((2, 50), (0, 40), (5, 30))}
	g0 = {slot: gamma_matrix(K, docs.num_docs, 20 + slot) for slot, docs in batches.items()}
	lam0 = gamma_matrix(K, V, 4)
	host = capi.Model('online', V, K, 10000, .1, .2)
	host.lambdas = lam0
	model = capi.Model('online', V, K, 10000, .1, .2)
	model.lambdas = lam0
	for slot in (2, 0, 5):
		model.upload_docs_slot(batches[slot], slot)
	for slot in (0, 2, 5):
		host.update_parameters(batches[slot], gamma0=g0[slot], max_iter_inference=20)
		model.select_docs(slot)
		model.update_parameters_resident(gamma0=g0[slot], max_iter_inference=20)
		assert np.array_equal(model.lambdas, host.lambdas)
	model.close()
	again = capi.Model('online', V, K, 10000, .1, .2)
	again.update_parameters(batches[0], max_iter_inference=20)
	assert np.all(np.isfinite(again.lambdas))


def test_csr_input_is_validated(capi):
	model = capi.Model('online', 20, 4, 10)
	with pytest.raises(RuntimeError, match='Word counts should not be negative.'):
		model.update_variables(capi.CSR([0, 2], [1, 2], [3, -1]), np.ones((4, 1)))
	bad = capi.CSR([0, 2], [1, 2], [3, 1])
	bad.doc_ptr[0] = 1
	with pytest.raises(RuntimeError, match='Document offsets must start at zero.'):
		model.update_variables(bad, np.ones((4, 1)))


# ---- lower bound -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
def test_lower_bound_vs_oracle(capi, oracle_built, precision):
	from trlda_b200.synth import gamma_matrix, make_corpus
	K, V, B, D = 50, 900, 80, 5000
	ptr, ids, cts = make_corpus(B, V, K, .1, .2, mean_length=60, seed=21)
	lam0, g0 = gamma_matrix(K, V, 22), gamma_matrix(K, B, 23)
	port = oracle_built.PortModel('online', V, K, D, .1, .2)
	port.lambdas = lam0
	want_total, want_docs = port.lower_bound(oracle_built.CSR(ptr, ids, cts), g0, max_iter=50)
	model = capi.Model('online', V, K, D, .1, .2, precision=precision)
	model.lambdas = lam0
	total, per_doc = model.lower_bound(capi.CSR(ptr, ids, cts), g0, max_iter=50)
	t = 1e-9 if precision == 'fp64' else TOL_ELBO_MIXED
	assert np.max(np.abs(per_doc - want_docs) / np.abs(want_docs)) < t
	assert total == pytest.approx(want_total, rel=t)


# ---- accessors / errors ----------------------------------------------------------------------------------------------
def test_accessors_and_error_messages(capi):
	"""onlinelda_test.py:14-35 through the C ABI"""
	W, D, K = 102, 1010, 11
	model = capi.Model('online', W, K, D, .27, 3.1)
	assert (model.K, model.V, model.num_documents, model.eta) == (K, W, D, 3.1)
	assert np.all(model.alpha == .27)
	with pytest.raises(RuntimeError, match='Alpha has wrong dimensionality.'):
		model.alpha = np.random.rand(K + 1)
	with pytest.raises(RuntimeError, match='Alpha should not be negative.'):
		model.alpha = -np.ones(K)
	with pytest.raises(RuntimeError, match='Eta should not be negative.'):
		model.eta = -1.
	with pytest.raises(RuntimeError, match='Lambda has wrong dimensionality.'):
		model.lambdas = np.ones((K, W + 1))
	alpha = np.random.rand(K, 1)
	model.alpha = alpha
	assert np.max(np.abs(model.alpha - alpha.ravel())) < 1e-20
	lam = np.random.rand(K, W)
	model.lambdas = lam
	assert np.array_equal(model.lambdas, lam) and model.lambdas.flags.f_contiguous
	model.alpha = 2.5                                                # scalar form, lda.h:146
	assert np.all(model.alpha == 2.5)


# ---- full BASELINE size: properties that need no oracle --------------------------------------------------------------
def test_full_size_cfg3_properties(capi):
	"""cfg-3 at full size (K=1000, V=100k, B=8192, T=10, I=20), where the CPU oracle would need minutes per E-step:
	checks size-independent identities of the algorithm instead.
	  * E-step: phi is normalised, so every gamma column sums to sum(alpha) + the document's token count and the
	    sufficient statistics sum to the token mass of the minibatch; row sums of sstats equal those of the
	    per-document statistics;
	  * M-step: the blend is linear in the row sums (onlinelda.cpp:99-100);
	  * both precisions agree, runs are bitwise reproducible, the resident and host-buffer paths agree."""
	from trlda_b200.synth import gamma_matrix, make_corpus
	K, V, B, D = 1000, 100000, 8192, 1000000
	ptr, ids, cts = make_corpus(B, V, K, .1, .2, seed=1003)
	docs = capi.CSR(ptr, ids, cts)
	lam0, g0 = gamma_matrix(K, V, 2003), gamma_matrix(K, B, 3003)
	tokens = np.add.reduceat(cts, ptr[:-1]).astype(np.float64)

	gammas, lams = {}, {}
	for precision in ('fp64', 'mixed'):
		model = capi.Model('online', V, K, D, .1, .2, precision=precision)
		model.lambdas = lam0
		gamma, sstats = model.update_variables(docs, g0, max_iter=20)
		rel = 1e-12 if precision == 'fp64' else 2e-6
		assert np.max(np.abs(gamma.sum(0) - (K * .1 + tokens)) / tokens) < rel
		assert abs(sstats.sum() - cts.sum()) / cts.sum() < rel
		assert np.all(sstats >= 0) and np.all(np.isfinite(gamma))
		gammas[precision] = gamma

		rows0 = lam0.sum(1)
		rho = model.update_parameters(docs, gamma0=g0, max_iter_tr=10, max_iter_inference=20, kappa=.7, tau=100.)
		lam1 = model.lambdas
		assert rho == pytest.approx(100. ** -.7)
		# sum over topics of the row sums: (1-rho) sum(lambda') + rho (K V eta + D/B * token mass)
		want_total = (1 - rho) * rows0.sum() + rho * (K * V * .2 + D / B * cts.sum())
		assert abs(lam1.sum() - want_total) / want_total < (1e-12 if precision == 'fp64' else 1e-6)
		assert np.all(lam1 > 0)
		lams[precision] = lam1

		again = capi.Model('online', V, K, D, .1, .2, precision=precision)
		again.lambdas = lam0
		again.upload_docs(docs)
		again.update_parameters_resident(gamma0=g0, max_iter_tr=10, max_iter_inference=20, kappa=.7, tau=100.)
		assert np.array_equal(again.lambdas, lam1)                  # bitwise: deterministic, resident == host path
		again.close()
		model.close()

	assert rel_err_columns(gammas['mixed'], gammas['fp64']) < TOL_MIXED
	assert rel_err(lams['mixed'], lams['fp64']) < TOL_MIXED


def test_documents_do_not_depend_on_the_schedule(capi):
	"""A document's gamma depends on nothing but the document: the tensor-memory kernel hands documents to teams by a work
	counter (the order depends on timing), and a permuted minibatch puts every document on another team, in another
	tile slot - the per-document results must be bitwise the same."""
	from trlda_b200.synth import gamma_matrix
	rng = np.random.default_rng(77)
	K, V, B = 1000, 6000, 640                      # more than twice the 74 teams: most documents are drawn dynamically
	lam0, g0 = gamma_matrix(K, V, 78), gamma_matrix(K, B, 79)
	lengths = rng.integers(1, 200, size=B)          # every tile shape, a few documents for the streaming kernel
	lengths[:8] = rng.integers(193, 260, size=8)
	lengths[8:12] = 0
	docs = [[(int(w), int(1 + rng.integers(5))) for w in rng.permutation(V)[:n]] for n in lengths]

	def run(order):
		ptr = np.zeros(B + 1, dtype=np.int64)
		ids, cts = [], []
		for i, d in enumerate(order):
			ids += [w for w, _ in docs[d]]
			cts += [c for _, c in docs[d]]
			ptr[i + 1] = len(ids)
		model = capi.Model('online', V, K, 100000, .1, .2, precision='mixed')
		model.lambdas = lam0
		gamma, _ = model.update_variables(capi.CSR(ptr, np.array(ids, dtype=np.int32), np.array(cts, dtype=np.int32)),
			np.asfortranarray(g0[:, order]), max_iter=7)
		model.close()
		out = np.empty_like(gamma)
		out[:, order] = gamma
		return out

	first = run(np.arange(B))
	assert np.all(np.isfinite(first))
	for seed in (1, 2):
		assert np.array_equal(run(np.random.default_rng(seed).permutation(B)), first)
