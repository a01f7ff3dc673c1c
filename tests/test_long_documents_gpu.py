"""
Documents longer than the shared memory of the E-step kernels hold (DESIGN.md section 10): they run on the
global-memory variant of k_estep, the other documents of the minibatch keep their kernel and their bits.

Run as a script under torch.distributed.run (`--worker`), this file is also the worker of the two-GPU test.
"""
import argparse
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

from common import TOL_ELBO_MIXED, TOL_FP64, TOL_MIXED, mixed_flip_check, parity_err, rel_err_columns

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def capi():
	from trlda_b200 import capi
	capi.lib()        # raises if libtrlda_b200.so is missing
	return capi


def tol(precision):
	return TOL_FP64 if precision == 'fp64' else TOL_MIXED


def make_docs(rng, V, lengths, max_count=5, distinct=True):
	"""one document per length: distinct word ids (or drawn with repetition) and counts in [1, max_count]"""
	docs = []
	for n in lengths:
		ids = rng.permutation(V)[:n] if distinct else rng.integers(0, V, size=n)
		docs.append([(int(w), int(1 + rng.integers(max_count))) for w in ids])
	return docs


def gammas(rng, K, B):
	return np.asfortranarray(rng.gamma(100., .01, size=(B, K)).T)


def lambdas(rng, K, V):
	return np.asfortranarray(rng.gamma(100., .01, size=(V, K)).T)


# ---- E-step parity with the plain-C oracle ---------------------------------------------------------------------------
def _sample_like(rng, V, n):
	"""the form LDA::sample emits: one pair per token, repeated word ids, count 1"""
	return [(int(w), 1) for w in rng.integers(0, V, size=n)]


PARITY_SHAPES = [
	# K, V, lengths of the documents (the long ones first in the list, not in the minibatch), max_iter, sampled
	(1000, 30000, [150, 8200, 40, 20000, 600, 9], 10, False),     # just over the limit of k_estep, and far over it
	(100, 40000, [300, 30000, 250, 120, 1500, 700], 20, False),  # beyond the streaming kernel too; the rest streams
	(33, 12000, [10000, 20, 300, 7], 20, False),                 # K not a multiple of 32
	(4096, 10240, [40, 9000, 100], 5, False),                    # the topic limit
	(256, 5000, [30, 100000, 200], 20, True),                    # 100 000 tokens: float32 sums over groups of columns
]


@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
@pytest.mark.parametrize('K,V,lengths,max_iter,sampled', PARITY_SHAPES)
def test_long_documents_vs_oracle(capi, oracle_built, precision, K, V, lengths, max_iter, sampled):
	rng = np.random.default_rng(K + len(lengths))
	lists = make_docs(rng, V, lengths)
	if sampled:
		lists = [_sample_like(rng, V, n) if n > 10000 else doc for n, doc in zip(lengths, lists)]
	B = len(lists)
	lam0, g0 = lambdas(rng, K, V), gammas(rng, K, B)
	alpha = rng.uniform(.05, .5, size=K)

	port = oracle_built.PortModel('online', V, K, 1000, alpha, .2)
	port.lambdas = lam0
	want_gamma, want_sstats, want_it = port.update_variables(
		oracle_built.CSR.from_lists(lists), g0, max_iter=max_iter, want_iterations=True)

	model = capi.Model('online', V, K, 1000, alpha, .2, precision=precision)
	model.lambdas = lam0
	gamma, sstats = model.update_variables(capi.CSR.from_lists(lists), g0, max_iter=max_iter)
	stats = model.stats()
	model.close()

	assert parity_err(gamma, want_gamma, precision) < tol(precision)
	assert rel_err_columns(sstats, want_sstats) < tol(precision)
	assert np.sum(sstats) == pytest.approx(sum(c for doc in lists for _, c in doc), rel=1e-6)
	if precision == 'fp64':
		assert stats['estep_doc_iterations'] == int(want_it.sum())
	assert stats['estep_sweeps'] == stats['estep_doc_iterations'] + B


# ---- documents that run without a long document keep their kernel and their bits -------------------------------------
ISOLATION = [
	# K, precision, lengths of the ordinary documents, length of the long one
	(1000, 'mixed', [5, 60, 130, 192, 193, 400, 1200, 2000, 17, 150, 250, 90], 9000),   # tensor memory + streaming
	(1040, 'mixed', [193, 260, 400, 900, 1500, 3000, 70, 10], 9000),                    # length buckets of k_estep
	(2048, 'fp64', [3, 50, 200, 800, 2500, 4000], 9000),                                  # k_estep only
]


@pytest.mark.parametrize('K,precision,lengths,long_len', ISOLATION)
def test_other_documents_keep_their_bits(capi, K, precision, lengths, long_len):
	rng = np.random.default_rng(K)
	V = 6000
	ordinary = make_docs(rng, V, lengths)
	long_doc = make_docs(rng, V, [long_len], distinct=False)[0]
	lam0 = lambdas(rng, K, V)
	g0 = gammas(rng, K, len(ordinary) + 1)
	runs = {}
	for name, lists, g in (('alone', ordinary, g0[:, :-1]), ('with long', ordinary[:3] + [long_doc] + ordinary[3:],
			np.asfortranarray(np.concatenate([g0[:, :3], g0[:, -1:], g0[:, 3:-1]], axis=1)))):
		model = capi.Model('online', V, K, 1000, .1, .2, precision=precision)
		model.lambdas = lam0
		gamma, _ = model.update_variables(capi.CSR.from_lists(lists), np.asfortranarray(g), max_iter=15)
		model.close()
		runs[name] = gamma
	with_long = np.delete(runs['with long'], 3, axis=1)
	assert np.all(np.isfinite(runs['with long']))
	assert np.array_equal(with_long, runs['alone'])


# ---- the calls that run an E-step ------------------------------------------------------------------------------------
def _driver_inputs(seed=11):
	rng = np.random.default_rng(seed)
	K, V = 1000, 12000
	lists = make_docs(rng, V, [120, 300, 8600, 45, 1000, 10, 220, 60])
	return rng, K, V, lists, lambdas(rng, K, V), gammas(rng, K, len(lists))


@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
def test_online_update_parameters_with_a_long_document(capi, oracle_built, precision):
	rng, K, V, lists, lam0, g0 = _driver_inputs()
	kwargs = dict(max_iter_tr=2, max_iter_inference=20, kappa=.7, tau=100., update_alpha=1, update_eta=1)
	port = oracle_built.PortModel('online', V, K, 100000, .1, .2)
	port.lambdas = lam0
	want_rho = port.update_parameters(oracle_built.CSR.from_lists(lists), gamma0=g0, **kwargs)
	model = capi.Model('online', V, K, 100000, .1, .2, precision=precision)
	model.lambdas = lam0
	rho = model.update_parameters(capi.CSR.from_lists(lists), gamma0=g0, **kwargs)
	assert rho == pytest.approx(want_rho, rel=1e-14)
	if precision == 'fp64':
		assert parity_err(model.lambdas, port.lambdas, precision) < TOL_FP64
	else:
		q999, worst = mixed_flip_check(model.lambdas, port.lambdas)
		assert q999 < TOL_MIXED and worst < 10 * TOL_MIXED
	assert parity_err(model.alpha, port.alpha, precision) < tol(precision)
	assert model.eta == pytest.approx(port.eta, rel=tol(precision))
	model.close()


@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
def test_batch_epoch_with_a_long_document(capi, oracle_built, precision):
	rng, K, V, lists, lam0, g0 = _driver_inputs(12)
	kwargs = dict(max_epochs=1, max_iter_inference=20)
	port = oracle_built.PortModel('batch', V, K, 0, .1, .2)
	port.lambdas = lam0
	port.update_parameters(oracle_built.CSR.from_lists(lists), gamma0=g0, **kwargs)
	model = capi.Model('batch', V, K, 0, .1, .2, precision=precision)
	model.lambdas = lam0
	model.update_parameters(capi.CSR.from_lists(lists), gamma0=g0, **kwargs)
	assert parity_err(model.lambdas, port.lambdas, precision) < tol(precision)
	model.close()


@pytest.mark.parametrize('precision', ['fp64', 'mixed'])
def test_lower_bound_with_a_long_document(capi, oracle_built, precision):
	rng, K, V, lists, lam0, g0 = _driver_inputs(13)
	port = oracle_built.PortModel('online', V, K, 5000, .1, .2)
	port.lambdas = lam0
	want_total, want_docs = port.lower_bound(oracle_built.CSR.from_lists(lists), g0, max_iter=30)
	model = capi.Model('online', V, K, 5000, .1, .2, precision=precision)
	model.lambdas = lam0
	total, per_doc = model.lower_bound(capi.CSR.from_lists(lists), g0, max_iter=30)
	t = 1e-9 if precision == 'fp64' else TOL_ELBO_MIXED
	assert np.max(np.abs(per_doc - want_docs) / np.abs(want_docs)) < t
	assert total == pytest.approx(want_total, rel=t)
	model.close()


# ---- end to end through the Python API -------------------------------------------------------------------------------
def test_training_on_a_file_with_a_long_line(tmp_path):
	import trlda.models
	from trlda.utils import load_documents, load_documents_csr
	rng = np.random.default_rng(21)
	V = 20000
	lines = []
	for n in [30, 200, 12000, 80, 5, 400]:
		ids = rng.permutation(V)[:n]
		lines.append('%d %s' % (n, ' '.join('%d:%d' % (w, 1 + rng.integers(4)) for w in ids)))
	path = tmp_path / 'corpus.txt'
	path.write_text('\n'.join(lines) + '\n')

	docs = load_documents(str(path))
	assert max(len(d) for d in docs) == 12000
	csr = load_documents_csr(str(path))
	for batch in (docs, csr):
		model = trlda.models.OnlineLDA(num_words=V, num_topics=1000, num_documents=1000, alpha=.1, eta=.2)
		rho = model.update_parameters(batch, max_iter_tr=2, max_iter_inference=10)
		assert np.isfinite(rho)
		assert np.all(np.isfinite(model.lambdas))


# ---- two GPUs --------------------------------------------------------------------------------------------------------
def _free_port():
	with socket.socket() as s:
		s.bind(('127.0.0.1', 0))
		return s.getsockname()[1]


def test_two_gpus_with_a_long_document_in_one_shard():
	"""the rank that holds the long document does not strand the other in the exchange, and both agree with one GPU"""
	import torch
	if torch.cuda.device_count() < 2:
		pytest.skip('needs two GPUs')
	cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
		'--master-addr', '127.0.0.1', '--master-port', str(_free_port()), os.path.abspath(__file__), '--worker']
	proc = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
	lines = [l for l in proc.stdout.splitlines() if l.startswith('RESULT')]
	assert proc.returncode == 0 and lines, proc.stdout[-2000:] + proc.stderr[-4000:]
	out = [float(x) for x in lines[0].split()[1:]]
	fp64, mixed = out[:5], out[5:]
	assert fp64[0] == 0. and max(fp64[1:]) < 1e-11
	assert mixed[0] == 0. and max(mixed[1:]) < 1e-4


def _worker():
	import torch
	import torch.distributed as dist
	from trlda_b200 import capi
	from trlda_b200.distributed import init_comm, shard_bounds, shard_documents

	rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
	local_rank = int(os.environ.get('LOCAL_RANK', rank))
	rng = np.random.default_rng(31)
	K, V = 1000, 10000
	lengths = list(rng.integers(1, 400, size=40))
	lengths[30] = 8800                                 # in the second shard
	lists = make_docs(rng, V, lengths)
	full = capi.CSR.from_lists(lists)
	ptr, ids, cts = full.doc_ptr, full.word_ids, full.counts
	lam0, g0 = lambdas(rng, K, V), gammas(rng, K, len(lists))
	begin, end = shard_bounds(ptr, world)[rank]
	shard = shard_documents(ptr, ids, cts, rank, world)
	kwargs = dict(max_iter_tr=3, max_iter_inference=20, update_alpha=1, update_eta=1)

	torch.cuda.set_device(local_rank)
	dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
	results = {}
	for precision in ('fp64', 'mixed'):
		model = capi.Model('online', V, K, 5000, .1, .2, device=local_rank, precision=precision)
		model.lambdas = lam0
		init_comm(model, dist, torch.device('cuda', local_rank))
		rho = model.update_parameters(capi.CSR(*shard), gamma0=g0[:, begin:end], **kwargs)
		elbo, _ = model.lower_bound(capi.CSR(*shard), g0[:, begin:end], max_iter=20)
		results[precision] = (rho, model.lambdas, model.alpha, model.eta, elbo)
		model.close()
	dist.barrier()
	if rank == 0:
		out = []
		for precision in ('fp64', 'mixed'):
			single = capi.Model('online', V, K, 5000, .1, .2, device=local_rank, precision=precision)
			single.lambdas = lam0
			rho = single.update_parameters(capi.CSR(ptr, ids, cts), gamma0=g0, **kwargs)
			elbo, _ = single.lower_bound(capi.CSR(ptr, ids, cts), g0, max_iter=20)
			r = results[precision]
			out += [abs(r[0] - rho), float(np.max(np.abs(r[1] - single.lambdas) / single.lambdas)),
				float(np.max(np.abs(r[2] - single.alpha) / single.alpha)), abs(r[3] - single.eta) / single.eta,
				abs(r[4] - elbo) / abs(elbo)]
			single.close()
		print('RESULT', *out, flush=True)
	dist.barrier()
	dist.destroy_process_group()


if __name__ == '__main__':
	ap = argparse.ArgumentParser()
	ap.add_argument('--worker', action='store_true')
	if ap.parse_args().worker:
		_worker()
