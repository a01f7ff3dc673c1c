"""
Document-completion predictive log-likelihood (trlda_predictive_log_likelihood, Hoffman et al. 2013 section 5): gamma
fitted on the observed part with the E-step, each held-out token w of document d scored with
log sum_k E[theta_dk] E[beta_kw].

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
	sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from common import TOL_FP64

pytestmark = pytest.mark.gpu

PRECISIONS = ['fp64', 'mixed']
# mixed mode against the oracle: 1.9e-9 per document measured (K = 4096, NVIDIA B200), well inside the bound
TOL_PREDICTIVE_MIXED = 1e-5


@pytest.fixture(scope='module')
def capi():
	from trlda_b200 import capi
	capi.lib()        # raises if libtrlda_b200.so is missing
	return capi


def make_docs(rng, V, lengths, max_count=5):
	return [[(int(w), int(1 + rng.integers(max_count))) for w in rng.permutation(V)[:n]] for n in lengths]


def to_csr(capi, lists):
	return capi.CSR.from_lists(lists)


def lambdas(rng, K, V):
	"""a lambda with topics of clearly different shapes, so that gamma matters for the score"""
	return np.asfortranarray(rng.gamma(.3, 2., size=(V, K)).T + .05)


def gammas(rng, K, B):
	return np.asfortranarray(rng.gamma(100., .01, size=(B, K)).T)


def predictive_numpy(gamma, lam, held_out):
	"""the formula on the host: per_doc[d] = sum_j c_j log(sum_k E[theta_dk] E[beta_k,w_j])"""
	theta = gamma / gamma.sum(axis=0, keepdims=True)
	beta = lam / lam.sum(axis=1, keepdims=True)
	out = np.zeros(len(held_out))
	for d, doc in enumerate(held_out):
		if doc:
			ids = np.array([w for w, _ in doc])
			cts = np.array([c for _, c in doc], dtype=np.float64)
			out[d] = float(np.sum(cts * np.log(theta[:, d] @ beta[:, ids])))
	return out


def rel_per_doc(got, want):
	nz = want != 0
	assert np.all(got[~nz] == 0.)
	return float(np.max(np.abs(got[nz] - want[nz]) / np.abs(want[nz]))) if nz.any() else 0.


def split_inputs(rng, K, V, lengths, long_observed=None):
	"""observed / held-out pairs with the edge cases: document 0 has an empty observed part, document 1 an empty held-out
	part, document 2 a duplicated held-out id, document 3 held-out words that are absent from its observed part"""
	from trlda.utils import split_documents
	observed, held = split_documents(make_docs(rng, V, lengths), .25, seed=int(rng.integers(1 << 30)))
	observed[0] = []
	held[0] = held[0] or [(5, 2)]
	held[1] = []
	held[2] = held[2] + [held[2][0]] if held[2] else [(9, 1), (9, 3)]
	seen = {w for w, _ in observed[3]}
	held[3] = [(int(w), 2) for w in rng.permutation(V)[:30] if int(w) not in seen]
	if long_observed:
		observed.append([(int(w), int(1 + rng.integers(4))) for w in rng.permutation(V)[:long_observed]])
		held.append([(int(w), 1) for w in rng.permutation(V)[:200]])
	return observed, held


# ---- 1. against the oracle's gamma and the formula on the host -------------------------------------------------------
ORACLE_SHAPES = [
	# K, V, document lengths, length of one more observed document (the long-document E-step route)
	(1000, 20000, [80, 150, 300, 60, 1200, 25, 500, 190, 7], 9000),
	(33, 12000, [40, 200, 90, 700, 15, 350], None),          # K not a multiple of 32: the generic k_estep
	(4096, 6000, [60, 250, 130, 900, 30], None),              # the topic limit
]


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('K,V,lengths,long_observed', ORACLE_SHAPES)
def test_predictive_vs_oracle(capi, oracle_built, precision, K, V, lengths, long_observed):
	rng = np.random.default_rng(K + len(lengths))
	observed, held = split_inputs(rng, K, V, lengths, long_observed)
	B = len(observed)
	lam0, g0 = lambdas(rng, K, V), gammas(rng, K, B)
	alpha = rng.uniform(.05, .5, size=K)
	max_iter, threshold = 40, 1e-4

	port = oracle_built.PortModel('online', V, K, 1000, alpha, .2)
	port.lambdas = lam0
	want_gamma, _ = port.update_variables(oracle_built.CSR.from_lists(observed), g0, max_iter, threshold, want_sstats=False)
	want = predictive_numpy(want_gamma, lam0, held)

	model = capi.Model('online', V, K, 1000, alpha, .2, precision=precision)
	model.lambdas = lam0
	total, tokens, per_doc = model.predictive_log_likelihood(to_csr(capi, observed), to_csr(capi, held), g0, max_iter, threshold)
	model.close()

	assert tokens == int(sum(c for doc in held for _, c in doc))
	err, err_total = rel_per_doc(per_doc, want), abs(total - want.sum()) / abs(want.sum())
	print('predictive vs oracle K=%d %s: per-document %.2e, total %.2e' % (K, precision, err, err_total))
	if precision == 'fp64':
		assert err <= TOL_FP64 and err_total <= TOL_FP64
	else:
		assert err <= TOL_PREDICTIVE_MIXED
	# E[theta] of an empty observed part is alpha / sum(alpha)
	theta0, rows = alpha / alpha.sum(), lam0.sum(axis=1)
	want0 = sum(c * np.log(theta0 @ (lam0[:, v] / rows)) for v, c in held[0])
	assert per_doc[0] == pytest.approx(want0, rel=TOL_FP64 if precision == 'fp64' else TOL_PREDICTIVE_MIXED)


# ---- 2. the kernel alone: the device's own gamma through the formula on the host --------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('K,V', [(1000, 20000), (4096, 6000)])
def test_kernel_against_device_gamma(capi, precision, K, V):
	rng = np.random.default_rng(7 * K)
	observed, held = split_inputs(rng, K, V, [120, 40, 260, 90, 600, 10, 333, 75])
	lam0, g0 = lambdas(rng, K, V), gammas(rng, K, len(observed))
	model = capi.Model('batch', V, K, 0, .1, .2, precision=precision)
	model.lambdas = lam0
	gamma, _ = model.update_variables(to_csr(capi, observed), g0, max_iter=30, want_sstats=False)
	_, _, per_doc = model.predictive_log_likelihood(to_csr(capi, observed), to_csr(capi, held), g0, max_iter=30)
	model.close()
	assert rel_per_doc(per_doc, predictive_numpy(gamma, lam0, held)) <= 1e-12


# ---- 3. determinism ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_bitwise_reproducible(capi, precision):
	rng = np.random.default_rng(5)
	K, V = 1000, 8000
	observed, held = split_inputs(rng, K, V, [100, 200, 50, 400, 20, 150, 90, 700])
	lam0, g0 = lambdas(rng, K, V), gammas(rng, K, len(observed))
	obs, ho = to_csr(capi, observed), to_csr(capi, held)
	model = capi.Model('online', V, K, 1000, .1, .2, precision=precision)
	model.lambdas = lam0
	a = model.predictive_log_likelihood(obs, ho, g0)
	b = model.predictive_log_likelihood(obs, ho, g0)
	assert a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2], b[2])
	capi.seed(123)
	c = model.predictive_log_likelihood(obs, ho)
	capi.seed(123)
	d = model.predictive_log_likelihood(obs, ho)
	assert c[0] == d[0] and np.array_equal(c[2], d[2])
	# a document's value does not depend on the documents that share the launch
	e = model.predictive_log_likelihood(obs.slice(2, 5), ho.slice(2, 5), np.asfortranarray(g0[:, 2:5]))
	assert np.array_equal(e[2], a[2][2:5])
	model.close()


# ---- 4. training state ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_training_state_untouched(capi, precision):
	from trlda_b200.synth import make_corpus
	K, V = 256, 4000
	train = capi.CSR(*make_corpus(300, V, K, .1, .2, mean_length=60, seed=3))
	evaluation = capi.CSR(*make_corpus(100, V, K, .1, .2, mean_length=60, seed=3, doc_seed=9))
	from trlda.utils import split_documents
	obs, ho = (capi.CSR(*p) for p in split_documents((evaluation.doc_ptr, evaluation.word_ids, evaluation.counts), .2, seed=1))
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
			model.predictive_log_likelihood(obs, ho)
			after = (model.lambdas, model.alpha, model.eta, model.update_count)
			assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
			assert before[2] == after[2] and before[3] == after[3]
		model.select_docs(1)
		capi.seed(5)
		model.update_parameters_resident(**kwargs)
		results.append(model.lambdas)
		model.close()
	assert np.array_equal(results[0], results[1])


# ---- 5. errors ---------------------------------------------------------------------------------------------------------
def _raw_call(capi, model, obs, ho, latents=None, gibbs=False):
	params = capi.default_params(inference_method=1 if gibbs else 0)
	rows, cols = (latents.shape if latents is not None else (0, 0))
	total, tokens = C.c_double(0.), C.c_int64(0)
	status = model._lib.trlda_predictive_log_likelihood(model.h, C.byref(obs.c), C.byref(ho.c), capi._dptr(latents), rows, cols,
		C.byref(params), C.byref(total), C.byref(tokens), None)
	return status, model._lib.trlda_last_error(model.h).decode()


def test_errors(capi):
	K, V = 64, 500
	model = capi.Model('batch', V, K, 0, .1, .2)
	obs = capi.CSR.from_lists([[(1, 2), (3, 1)], [(4, 4)]])
	good = capi.CSR.from_lists([[(2, 1)], [(7, 3)]])
	cases = [
		(obs, capi.CSR.from_lists([[(2, 1)]]), None, False, capi.ERR_ARG, 'Observed and held-out documents differ in number.'),
		(obs, capi.CSR.from_lists([[(2, 1)], [(V, 1)]]), None, False, capi.ERR_ARG, 'Word ID out of range.'),
		(obs, capi.CSR.from_lists([[(2, -1)], [(7, 3)]]), None, False, capi.ERR_ARG, 'Word counts should not be negative.'),
		(obs, good, np.ones((K, 3), order='F'), False, capi.ERR_ARG, 'Initial gamma has wrong dimensionality.'),
		(obs, good, None, True, capi.ERR_UNSUPPORTED, "Only variational inference ('VI') is implemented on the device."),
	]
	for o, h, latents, gibbs, status, message in cases:
		assert _raw_call(capi, model, o, h, latents, gibbs) == (status, message)
		total, tokens, per_doc = model.predictive_log_likelihood(obs, good)
		assert tokens == 4 and np.isfinite(total) and total == pytest.approx(per_doc.sum(), rel=1e-15)
	model.close()


# ---- 6. Python API -----------------------------------------------------------------------------------------------------
def test_python_api_list_and_csr_forms():
	import trlda.models
	from trlda.utils import split_documents
	from trlda_b200.synth import make_corpus, to_lists
	K, V = 100, 3000
	csr = make_corpus(64, V, K, .1, .2, mean_length=80, seed=4)
	obs_csr, ho_csr = split_documents(csr, .2, seed=8)
	obs_lists, ho_lists = split_documents(to_lists(*csr), .2, seed=8)
	g0 = gammas(np.random.default_rng(1), K, 64)
	for model in (trlda.models.OnlineLDA(V, K, 1000, .1, .2), trlda.models.BatchLDA(V, K, .1, .2)):
		a = model.predictive_log_likelihood(obs_lists, ho_lists, latents=g0, max_iter=50)
		b = model.predictive_log_likelihood(obs_csr, ho_csr, g0, 50)
		assert a == b
		assert a[1] == int(ho_csr[2].sum()) and a[0] < 0


def test_training_raises_the_predictive_likelihood():
	import trlda
	import trlda.models
	from trlda.utils import split_documents
	from trlda_b200.synth import make_corpus
	K, V, D = 20, 2000, 100000
	trlda.seed(3)
	obs, ho = split_documents(make_corpus(200, V, K, .1, .05, mean_length=100, seed=12, doc_seed=999), .2, seed=4)
	g0 = gammas(np.random.default_rng(2), K, 200)
	model = trlda.models.OnlineLDA(V, K, D, .1, .05)
	total0, tokens = model.predictive_log_likelihood(obs, ho, g0)
	for step in range(20):
		model.update_parameters(make_corpus(256, V, K, .1, .05, mean_length=100, seed=12, doc_seed=step), max_iter_tr=2)
	total1, _ = model.predictive_log_likelihood(obs, ho, g0)
	assert total1 / tokens > total0 / tokens + .1


# ---- 7. two GPUs --------------------------------------------------------------------------------------------------------
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
	out = lines[0].split()[1:]
	for i in range(0, len(out), 3):      # per precision: total relative error, tokens equal, per_doc bitwise on every rank
		assert float(out[i]) <= 1e-12 and out[i + 1] == 'True' and out[i + 2] == 'True'


def _worker():
	import torch
	import torch.distributed as dist
	from trlda_b200 import capi
	from trlda_b200.distributed import init_comm, shard_bounds, shard_documents

	rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
	local_rank = int(os.environ.get('LOCAL_RANK', rank))
	rng = np.random.default_rng(41)
	K, V = 1000, 10000
	observed, held = split_inputs(rng, K, V, list(rng.integers(1, 400, size=40)))
	obs_full, ho_full = capi.CSR.from_lists(observed), capi.CSR.from_lists(held)
	lam0, g0 = lambdas(rng, K, V), gammas(rng, K, len(observed))
	begin, end = shard_bounds(obs_full.doc_ptr, world)[rank]
	obs = capi.CSR(*shard_documents(obs_full.doc_ptr, obs_full.word_ids, obs_full.counts, rank, world))
	ho = ho_full.slice(begin, end)

	torch.cuda.set_device(local_rank)
	dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
	sharded = {}
	for precision in PRECISIONS:
		model = capi.Model('online', V, K, 5000, .1, .2, device=local_rank, precision=precision)
		model.lambdas = lam0
		init_comm(model, dist, torch.device('cuda', local_rank))
		sharded[precision] = model.predictive_log_likelihood(obs, ho, np.asfortranarray(g0[:, begin:end]), max_iter=30)
		model.close()
	single = {}
	for precision in PRECISIONS:
		model = capi.Model('online', V, K, 5000, .1, .2, device=local_rank, precision=precision)
		model.lambdas = lam0
		single[precision] = model.predictive_log_likelihood(obs_full, ho_full, g0, max_iter=30)
		model.close()
	flags = torch.tensor([int(np.array_equal(sharded[p][2], single[p][2][begin:end])) for p in PRECISIONS], device='cuda')
	dist.all_reduce(flags, op=dist.ReduceOp.MIN)
	if rank == 0:
		out = []
		for i, p in enumerate(PRECISIONS):
			out += [abs(sharded[p][0] - single[p][0]) / abs(single[p][0]), sharded[p][1] == single[p][1], bool(flags[i].item())]
		print('RESULT', *out, flush=True)
	dist.barrier()
	dist.destroy_process_group()


if __name__ == '__main__':
	ap = argparse.ArgumentParser()
	ap.add_argument('--worker', action='store_true')
	if ap.parse_args().worker:
		_worker()
