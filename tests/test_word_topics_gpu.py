"""
Topics of the words of documents (trlda_word_topics): gamma fitted by the E-step exactly as trlda_update_variables fits it,
then for every (word, count) pair j of document d the n most probable topics under
phi_jk = softmax_k(psi(gamma_dk) + psi(lambda_kw) - psi(sum_v lambda_kv)), in fp64 in both precision modes.

Run as a script under torch.distributed.run (`--worker`), this file is also the worker of the two-GPU test.
"""
import argparse
import ctypes as C
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if __name__ == '__main__':
	sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

PRECISIONS = ['fp64', 'mixed']
# probabilities against scipy's digamma and numpy's softmax from the returned gamma: at most 2.2e-14 relative measured
# (NVIDIA B200, all shapes below, both modes); scores within this bound of each other may come out in either order
TOL_PHI = 2e-13


@pytest.fixture(scope='module')
def capi():
	from trlda_b200 import capi
	capi.lib()        # raises if libtrlda_b200.so is missing
	return capi


def make_docs(rng, V, lengths, max_count=5):
	return [[(int(w), int(1 + rng.integers(max_count))) for w in rng.permutation(V)[:n]] for n in lengths]


def lambdas(rng, K, V):
	return np.asfortranarray(rng.gamma(.3, 2., size=(V, K)).T + .05)


def gammas(rng, K, B):
	return np.asfortranarray(rng.gamma(100., .01, size=(B, K)).T)


def scores_numpy(gamma, lam, csr):
	"""s[j, k] = psi(gamma_dk) + psi(lambda_kw) - psi(sum_v lambda_kv) for every pair j (word w, document d)"""
	from scipy.special import digamma
	doc = np.repeat(np.arange(csr.num_docs), np.diff(csr.doc_ptr))
	log_beta = digamma(lam[:, csr.word_ids]) - digamma(lam.sum(axis=1))[:, None]
	return (digamma(gamma)[:, doc] + log_beta).T


def check_against_numpy(topics, probs, s):
	"""returns the largest relative error of the probabilities; asserts the ranking"""
	N, n = topics.shape
	K = s.shape[1]
	top = s.max(axis=1, keepdims=True)
	e = np.exp(s - top)
	phi = e / e.sum(axis=1, keepdims=True)
	order = np.lexsort((np.broadcast_to(np.arange(K), s.shape), -s), axis=1)[:, :n]
	rows = np.arange(N)[:, None]
	# a different topic only where numpy's scores of the two candidates are within the bound
	differ = topics != order
	s_got = s[rows, topics]
	s_want = s[rows, order]
	assert np.all(np.abs(s_got - s_want)[differ] <= TOL_PHI * np.maximum(1., np.abs(s_want[differ])))
	want = phi[rows, topics]
	err = float(np.max(np.abs(probs - want) / want)) if N else 0.
	assert err <= TOL_PHI
	assert np.all(np.diff(probs, axis=1) <= 0.)
	if n == K:
		assert np.all(np.abs(probs.sum(axis=1) - 1.) <= 1e-12)
	return err


# ---- 1 / 2. gamma is the E-step's; the topics against numpy -------------------------------------------------------------
SHAPES = [
	# K, V, document lengths, one more document of this many pairs (the long-document E-step route), n
	(1000, 20000, [80, 150, 300, 60, 1200, 25, 500, 190, 7], 9000, 5),   # the tensor-memory kernel (mixed mode)
	(33, 12000, [40, 200, 90, 700, 15, 350], None, 7),                   # K not a multiple of 32: the generic k_estep
	(4096, 6000, [60, 250, 130, 900, 30], None, 32),                     # the topic limit
	(20, 3000, [30, 5, 120, 64, 1, 300], None, 20),                      # n = K
]


def shape_inputs(capi, K, V, lengths, long_doc):
	rng = np.random.default_rng(K + len(lengths))
	docs = make_docs(rng, V, lengths)
	if long_doc:
		docs.append([(int(w), int(1 + rng.integers(4))) for w in rng.permutation(V)[:long_doc]])
	return capi.CSR.from_lists(docs), lambdas(rng, K, V), gammas(rng, K, len(docs)), rng.uniform(.05, .5, size=K)


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('K,V,lengths,long_doc,n', SHAPES)
def test_gamma_is_the_esteps(capi, precision, K, V, lengths, long_doc, n):
	csr, lam0, g0, alpha = shape_inputs(capi, K, V, lengths, long_doc)
	model = capi.Model('online', V, K, 1000, alpha, .2, precision=precision)
	model.lambdas = lam0
	want, _ = model.update_variables(csr, g0, 40, 1e-4, want_sstats=False)
	_, _, gamma = model.word_topics(csr, n, g0, 40, 1e-4)
	assert np.array_equal(gamma, want)
	capi.seed(31)
	want, _ = model.update_variables(csr, None, 40, 1e-4, want_sstats=False)
	capi.seed(31)
	_, _, gamma = model.word_topics(csr, n, None, 40, 1e-4)
	assert np.array_equal(gamma, want)
	model.close()


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('K,V,lengths,long_doc,n', SHAPES)
def test_against_numpy(capi, precision, K, V, lengths, long_doc, n):
	csr, lam0, g0, alpha = shape_inputs(capi, K, V, lengths, long_doc)
	model = capi.Model('online', V, K, 1000, alpha, .2, precision=precision)
	model.lambdas = lam0
	topics, probs, gamma = model.word_topics(csr, n, g0, 40, 1e-4)
	model.close()
	assert topics.shape == probs.shape == (csr.word_ids.size, n)
	err = check_against_numpy(topics, probs, scores_numpy(gamma, lam0, csr))
	print('word_topics vs numpy K=%d n=%d %s: %.2e' % (K, n, precision, err))


# ---- 3. edge cases ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_one_topic(capi, precision):
	model = capi.Model('batch', 50, 1, 0, .1, .2, precision=precision)
	topics, probs, _ = model.word_topics(capi.CSR.from_lists([[(1, 2), (7, 0)], [], [(3, 1), (3, 4)]]))
	model.close()
	assert np.array_equal(topics, np.zeros((4, 1), dtype=np.int32)) and np.all(probs == 1.)


@pytest.mark.parametrize('precision', PRECISIONS)
def test_edge_cases(capi, precision):
	rng = np.random.default_rng(3)
	K, V = 12, 400
	lam0 = lambdas(rng, K, V)
	lam0[:, 17] = 1e-5                   # exp(E[log beta]) underflows even in fp64 for this word
	lam0[5] = lam0[2]                    # topics 2 and 5 tie exactly
	g0 = gammas(rng, K, 4)
	g0[5] = g0[2]
	docs = [[(4, 3), (9, 0), (4, 1), (17, 2), (30, 1)],   # a repeated word, a count-0 pair, the underflowing word
		[],                                                # an empty document
		[(17, 5)],
		[(int(w), 2) for w in rng.permutation(V)[:40]]]
	csr = capi.CSR.from_lists(docs)
	model = capi.Model('online', V, K, 1000, .1, .2, precision=precision)
	model.lambdas = lam0
	topics, probs, gamma = model.word_topics(csr, K, g0)
	model.close()
	assert topics.shape == (46, K)
	assert np.all(np.isfinite(probs)) and np.all(np.abs(probs.sum(axis=1) - 1.) <= 1e-12)
	assert np.array_equal(np.sort(topics, axis=1), np.broadcast_to(np.arange(K), topics.shape))
	assert np.array_equal(topics[0], topics[2]) and np.array_equal(probs[0], probs[2])   # word 4 twice
	assert np.array_equal(gamma[2], gamma[5])                                             # precondition of the tie
	for row_t, row_p in zip(topics, probs):
		i, i5 = int(np.flatnonzero(row_t == 2)[0]), int(np.flatnonzero(row_t == 5)[0])
		assert i5 == i + 1 and row_p[i] == row_p[i5]
	# the scores of word 17 are about -1e5, so their rounding differs from numpy's by about 1e-11 absolute
	rest = csr.word_ids != 17
	check_against_numpy(topics[rest], probs[rest], scores_numpy(gamma, lam0, csr)[rest])


# ---- 4. known answer ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_disjoint_topics(capi, precision):
	rng = np.random.default_rng(11)
	K, V = 16, 1600
	owner = np.arange(V) % K
	lam0 = np.full((K, V), .01, order='F')
	lam0[owner, np.arange(V)] = 1000.
	docs = []
	for d in range(60):
		chosen = rng.choice(K, size=2 + d % 2, replace=False)
		words = rng.permutation(np.flatnonzero(np.isin(owner, chosen)))[:int(rng.integers(10, 80))]
		docs.append([(int(w), int(1 + rng.integers(3))) for w in words])
	csr = capi.CSR.from_lists(docs)
	model = capi.Model('online', V, K, 1000, .1, .01, precision=precision)
	model.lambdas = lam0
	capi.seed(4)
	topics, probs, _ = model.word_topics(csr)
	model.close()
	assert np.array_equal(topics[:, 0], owner[csr.word_ids]) and np.all(probs[:, 0] > .99)


# ---- 5. the E-step's fixed point -------------------------------------------------------------------------------------------
def test_fixed_point(capi):
	rng = np.random.default_rng(8)
	K, V = 24, 2000
	csr = capi.CSR.from_lists(make_docs(rng, V, [5, 40, 200, 90, 13, 600, 1]))
	alpha = rng.uniform(.05, .5, size=K)
	model = capi.Model('batch', V, K, 0, alpha, .2)
	model.lambdas = lambdas(rng, K, V)
	topics, probs, gamma = model.word_topics(csr, K, gammas(rng, K, csr.num_docs), max_iter=100000, threshold=1e-10)
	model.close()
	phi = np.zeros_like(probs)
	np.put_along_axis(phi, topics.astype(np.int64), probs, axis=1)
	for d in range(csr.num_docs):
		lo, hi = csr.doc_ptr[d], csr.doc_ptr[d + 1]
		update = csr.counts[lo:hi] @ phi[lo:hi] + alpha
		assert np.max(np.abs(update - gamma[:, d])) <= 1e-6 * gamma[:, d].sum()


# ---- 6. determinism --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_bitwise_reproducible(capi, precision):
	rng = np.random.default_rng(5)
	K, V = 1000, 8000
	csr = capi.CSR.from_lists(make_docs(rng, V, [100, 200, 50, 400, 20, 150, 90, 700]))
	lam0, g0 = lambdas(rng, K, V), gammas(rng, K, csr.num_docs)
	model = capi.Model('online', V, K, 1000, .1, .2, precision=precision)
	model.lambdas = lam0
	a = model.word_topics(csr, 4, g0)
	b = model.word_topics(csr, 4, g0)
	assert all(np.array_equal(x, y) for x, y in zip(a, b))
	# a pair's row does not depend on the other documents of the call
	c = model.word_topics(csr.slice(2, 5), 4, np.asfortranarray(g0[:, 2:5]))
	lo, hi = csr.doc_ptr[2], csr.doc_ptr[5]
	assert np.array_equal(c[0], a[0][lo:hi]) and np.array_equal(c[1], a[1][lo:hi])
	model.close()


# ---- 7. training state -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_training_state_untouched(capi, precision):
	from trlda_b200.synth import make_corpus
	K, V = 256, 4000
	train = capi.CSR(*make_corpus(300, V, K, .1, .2, mean_length=60, seed=3))
	evaluation = capi.CSR(*make_corpus(100, V, K, .1, .2, mean_length=60, seed=3, doc_seed=9))
	lam0 = lambdas(np.random.default_rng(2), K, V)
	kwargs = dict(max_iter_tr=2, max_iter_inference=20, update_alpha=1, update_eta=1)
	results = []
	for evaluate in (True, False):
		model = capi.Model('online', V, K, 10000, .1, .2, precision=precision)
		model.lambdas = lam0
		model.update_count = 3
		model.upload_docs_slot(train, 1)
		if evaluate:
			before = (model.lambdas, model.alpha, model.eta, model.update_count)
			capi.seed(77)
			model.word_topics(evaluation, 3)
			after = (model.lambdas, model.alpha, model.eta, model.update_count)
			assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
			assert before[2] == after[2] and before[3] == after[3]
		model.select_docs(1)
		capi.seed(5)
		model.update_parameters_resident(**kwargs)
		results.append(model.lambdas)
		model.close()
	assert np.array_equal(results[0], results[1])


# ---- 8. errors -------------------------------------------------------------------------------------------------------------
def _raw_call(capi, model, csr, n, latents=None, gibbs=False, topics=True):
	params = capi.default_params(inference_method=1 if gibbs else 0)
	rows, cols = (latents.shape if latents is not None else (0, 0))
	out = np.empty((max(csr.word_ids.size, 1), max(n, 1)), dtype=np.int32)
	status = model._lib.trlda_word_topics(model.h, C.byref(csr.c), capi._dptr(latents), rows, cols, C.byref(params), n,
		out.ctypes.data_as(C.POINTER(C.c_int32)) if topics else None, None, None)
	return status, model._lib.trlda_last_error(model.h).decode()


def test_errors(capi):
	K, V = 20, 500
	model = capi.Model('batch', V, K, 0, .1, .2)
	good = capi.CSR.from_lists([[(1, 2), (3, 1)], [(4, 4)]])
	n_range = 'Number of topics per word must lie in [1, min(32, number of topics)].'
	cases = [
		(good, 0, {}, capi.ERR_ARG, n_range),
		(good, 33, {}, capi.ERR_ARG, n_range),
		(good, K + 1, {}, capi.ERR_ARG, n_range),
		(good, 1, dict(topics=False), capi.ERR_ARG, 'word_topics: no output buffer.'),
		(good, 1, dict(latents=np.ones((K, 3), order='F')), capi.ERR_ARG, 'Initial gamma has wrong dimensionality.'),
		(good, 1, dict(gibbs=True), capi.ERR_UNSUPPORTED, "Only variational inference ('VI') is implemented on the device."),
		(capi.CSR.from_lists([[(2, 1)], [(V, 1)]]), 1, {}, capi.ERR_ARG, 'Word ID out of range.'),
		(capi.CSR.from_lists([[(2, -1)], [(7, 3)]]), 1, {}, capi.ERR_ARG, 'Word counts should not be negative.'),
	]
	for csr, n, kwargs, status, message in cases:
		assert _raw_call(capi, model, csr, n, **kwargs) == (status, message)
		topics, probs, gamma = model.word_topics(good, 2)
		assert topics.shape == (3, 2) and np.all(np.isfinite(probs)) and np.all(gamma > 0.)
	model.close()


# ---- 9. Python API ---------------------------------------------------------------------------------------------------------
def test_python_api_list_and_csr_forms():
	import trlda.models
	from trlda_b200.synth import make_corpus, to_lists
	K, V = 100, 3000
	csr = make_corpus(64, V, K, .1, .2, mean_length=80, seed=4)
	lists = to_lists(*csr)
	g0 = gammas(np.random.default_rng(1), K, 64)
	for model in (trlda.models.OnlineLDA(V, K, 1000, .1, .2), trlda.models.BatchLDA(V, K, .1, .2)):
		a = model.word_topics(lists, num_topics=3, latents=g0, max_iter=50)
		b = model.word_topics(csr, 3, g0, 50, .001)
		assert all(np.array_equal(x, y) for x, y in zip(a, b))
		topics, probs, gamma = a
		assert topics.dtype == np.int32 and probs.dtype == np.float64 and gamma.dtype == np.float64
		assert topics.shape == probs.shape == (int(csr[0][-1]), 3) and gamma.shape == (K, 64)
		assert gamma.flags['F_CONTIGUOUS']
		assert np.array_equal(gamma, model.update_variables(csr, g0, max_iter=50)[0])
		one = model.word_topics(lists, latents=g0)
		assert one[0].shape == (int(csr[0][-1]), 1)


# ---- 10. two GPUs ------------------------------------------------------------------------------------------------------------
def _free_port():
	with socket.socket() as s:
		s.bind(('127.0.0.1', 0))
		return s.getsockname()[1]


def test_two_gpus_match_one():
	import torch
	if torch.cuda.device_count() < 2:
		pytest.skip('needs two GPUs')
	cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
		'--master-addr', '127.0.0.1', '--master-port', str(_free_port()), os.path.abspath(__file__), '--worker']
	proc = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
	lines = [l for l in proc.stdout.splitlines() if l.startswith('RESULT')]
	assert proc.returncode == 0 and lines, proc.stdout[-2000:] + proc.stderr[-4000:]
	assert lines[0].split()[1:] == ['True'] * len(PRECISIONS)


def _worker():
	import torch
	import torch.distributed as dist
	from trlda_b200 import capi
	from trlda_b200.distributed import init_comm, shard_bounds

	rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
	local_rank = int(os.environ.get('LOCAL_RANK', rank))
	rng = np.random.default_rng(41)
	K, V = 1000, 10000
	full = capi.CSR.from_lists(make_docs(rng, V, list(rng.integers(1, 400, size=40))))
	lam0, g0 = lambdas(rng, K, V), gammas(rng, K, full.num_docs)
	begin, end = shard_bounds(full.doc_ptr, world)[rank]
	lo, hi = full.doc_ptr[begin], full.doc_ptr[end]

	torch.cuda.set_device(local_rank)
	dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
	equal = []
	for precision in PRECISIONS:
		model = capi.Model('online', V, K, 5000, .1, .2, device=local_rank, precision=precision)
		model.lambdas = lam0
		init_comm(model, dist, torch.device('cuda', local_rank))
		sharded = model.word_topics(full.slice(begin, end), 5, np.asfortranarray(g0[:, begin:end]), max_iter=30)
		model.close()
		model = capi.Model('online', V, K, 5000, .1, .2, device=local_rank, precision=precision)
		model.lambdas = lam0
		single = model.word_topics(full, 5, g0, max_iter=30)
		model.close()
		equal.append(int(np.array_equal(sharded[0], single[0][lo:hi]) and np.array_equal(sharded[1], single[1][lo:hi])
			and np.array_equal(sharded[2], single[2][:, begin:end])))
	flags = torch.tensor(equal, device='cuda')
	dist.all_reduce(flags, op=dist.ReduceOp.MIN)
	if rank == 0:
		print('RESULT', *[bool(f) for f in flags.tolist()], flush=True)
	dist.barrier()
	dist.destroy_process_group()


if __name__ == '__main__':
	ap = argparse.ArgumentParser()
	ap.add_argument('--worker', action='store_true')
	if ap.parse_args().worker:
		_worker()
