"""
Topic inspection and document co-occurrence on the device: trlda_top_words (the n most probable words of every topic)
and trlda_cooccurrence (document frequencies of those words and of their pairs), with the UMass / NPMI coherence built on
them in trlda.utils.

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


@pytest.fixture(scope='module')
def capi():
	from trlda_b200 import capi
	capi.lib()        # raises if libtrlda_b200.so is missing
	return capi


def top_words_numpy(lam, n):
	"""np.lexsort((ids, -lambda_row))[:n] for every row, on the entries at or above the row's n-th largest value"""
	K, V = lam.shape
	nth = np.partition(lam, V - n, axis=1)[:, V - n]
	ids = np.empty((K, n), dtype=np.int32)
	for k in range(K):
		cand = np.nonzero(lam[k] >= nth[k])[0]
		ids[k] = cand[np.lexsort((cand, -lam[k, cand]))][:n]
	return ids


def check_probs(lam, ids, probs, rows):
	"""probs are lambda_kw / rows_k with the row sums the model uses for E[beta] (model.row_sums(), the rowsum kernel of
	prepare_beta), to the last bit; those row sums are within the error bound of their summation order of the exact ones:
	positive terms added in sequence over chunks of 128 words, then the ceil(V / 128) chunk sums in sequence, so at most
	(128 + ceil(V / 128)) units of 2^-53 relative (numpy's pairwise sum adds a few more)"""
	V = lam.shape[1]
	assert np.array_equal(probs, np.take_along_axis(lam, ids.astype(np.int64), axis=1) / rows[:, None])
	bound = (128 + -(-V // 128) + 24) * 2. ** -53
	assert float(np.max(np.abs(rows - lam.sum(axis=1)) / lam.sum(axis=1))) <= bound


def cooccurrence_numpy(doc_ptr, word_ids, counts, top):
	"""counts[k, i, j] from the word set of every document (pairs with a positive count)"""
	K, n = top.shape
	out = np.zeros((K, n, n), dtype=np.int64)
	for d in range(len(doc_ptr) - 1):
		lo, hi = int(doc_ptr[d]), int(doc_ptr[d + 1])
		words = np.unique(word_ids[lo:hi][counts[lo:hi] > 0])
		present = np.isin(top, words)
		rows = np.nonzero(present.any(axis=1))[0]
		p = present[rows].astype(np.int64)
		out[rows] += p[:, :, None] * p[:, None, :]
	return out, len(doc_ptr) - 1


# ---- 1. top words -------------------------------------------------------------------------------------------------------
TOP_SHAPES = [
	# K, V, n
	(1, 20, 20),        # n = V
	(1, 100000, 32),
	(33, 5000, 1),
	(33, 20, 10),
	(1000, 100000, 10),
	(1000, 100000, 32),
	(4096, 20000, 32),
	(4096, 3000, 1),
]


@pytest.mark.parametrize('K,V,n', TOP_SHAPES)
def test_top_words_vs_numpy(capi, K, V, n):
	rng = np.random.default_rng(K * 7 + V + n)
	lam = np.asfortranarray(rng.gamma(100., .01, size=(K, V)))
	out = {}
	for precision in PRECISIONS:
		model = capi.Model('online', V, K, 1000, .1, .2, precision=precision)
		model.lambdas = lam
		out[precision] = model.top_words(n)
		rows = model.row_sums()
		model.close()
	ids, probs = out['fp64']
	assert np.array_equal(ids, top_words_numpy(lam, n))
	check_probs(lam, ids, probs, rows)
	# fp64 lambda in both modes: bitwise the same lists
	assert np.array_equal(out['mixed'][0], ids) and np.array_equal(out['mixed'][1], probs)


@pytest.mark.parametrize('K,V,n', [(33, 20, 20), (1000, 30000, 32), (64, 5000, 10)])
def test_top_words_ties_break_by_smaller_id(capi, K, V, n):
	rng = np.random.default_rng(3)
	lam = np.asfortranarray(rng.integers(1, 4, size=(K, V)).astype(np.float64))   # thousands of exact ties per row
	model = capi.Model('batch', V, K, 0, .1, .2)
	model.lambdas = lam
	ids, probs = model.top_words(n)
	rows = model.row_sums()
	model.close()
	want = np.stack([np.lexsort((np.arange(V), -lam[k]))[:n] for k in range(K)])
	assert np.array_equal(ids, want)
	check_probs(lam, ids, probs, rows)


@pytest.mark.parametrize('precision', PRECISIONS)
def test_top_words_after_training(capi, precision):
	from trlda_b200.synth import make_corpus
	K, V = 100, 5000
	model = capi.Model('online', V, K, 100000, .1, .2, precision=precision)
	for step in range(3):
		model.update_parameters(capi.CSR(*make_corpus(256, V, K, .1, .2, mean_length=80, seed=5, doc_seed=step)), max_iter_tr=2)
	ids, probs = model.top_words(10)
	lam, rows = model.lambdas, model.row_sums()
	model.close()
	assert np.array_equal(ids, top_words_numpy(lam, 10))
	check_probs(lam, ids, probs, rows)


# ---- 2. co-occurrence ---------------------------------------------------------------------------------------------------
def corpus_with_edge_cases(rng, V, K, B, long_pairs=None):
	"""make_corpus documents plus: an empty document, one with duplicate ids, one with zero counts (and a duplicate whose
	other pair has a positive count), and optionally one document of `long_pairs` pairs"""
	from trlda_b200.synth import make_corpus, to_lists
	docs = to_lists(*make_corpus(B, V, K, .1, .2, mean_length=60, seed=int(rng.integers(1 << 30))))
	docs[1] = []
	docs[2] = docs[2] + docs[2][:5]
	docs[3] = [(w, 0) for w, _ in docs[3][:10]] + docs[3][10:] + [(docs[3][-1][0], 0)]
	docs.append([])
	if long_pairs:
		docs.append([(int(w), int(1 + rng.integers(3))) for w in rng.integers(V, size=long_pairs)])
	return docs


def shared_word_ids(rng, K, V, n, word):
	"""user-supplied lists, not the model's top words: random distinct words, with `word` on every topic's list"""
	ids = np.stack([rng.choice(V, n, replace=False) for _ in range(K)]).astype(np.int32)
	for k in range(K):
		if word not in ids[k]:
			ids[k, k % n] = word
	return ids


COOC_SHAPES = [
	# K, V, n, documents, long document, own top words
	(1000, 30000, 10, 400, 20000, True),
	(33, 2000, 32, 300, None, True),
	(100, 3000, 20, 300, None, False),
	(4096, 8000, 32, 120, None, False),
	(1, 20, 20, 50, None, True),
]


@pytest.mark.parametrize('K,V,n,B,long_pairs,own', COOC_SHAPES)
def test_cooccurrence_vs_numpy(capi, K, V, n, B, long_pairs, own):
	rng = np.random.default_rng(K + n + B)
	csr = capi.CSR.from_lists(corpus_with_edge_cases(rng, V, min(K, 200), B, long_pairs))
	model = capi.Model('online', V, K, 1000, .1, .2)
	if own:
		top, _ = model.top_words(n)
	else:
		frequent = int(np.bincount(csr.word_ids, minlength=V).argmax())
		top = shared_word_ids(rng, K, V, n, frequent)
	counts, num_docs = model.cooccurrence(csr, top)
	again, _ = model.cooccurrence(csr, top)
	model.close()
	want, want_docs = cooccurrence_numpy(csr.doc_ptr, csr.word_ids, csr.counts, top)
	assert num_docs == want_docs == csr.num_docs
	assert np.array_equal(counts, want)
	assert np.array_equal(again, counts)
	if K > 1:
		assert (want == 0).any()        # pairs that never co-occur are counted as 0


def test_cooccurrence_empty_batch(capi):
	model = capi.Model('batch', 500, 8, 0, .1, .2)
	top, _ = model.top_words(5)
	counts, num_docs = model.cooccurrence(capi.CSR.from_lists([[], []]), top)
	assert num_docs == 2 and not counts.any()
	counts, num_docs = model.cooccurrence(capi.CSR.from_lists([]), top)
	assert num_docs == 0 and not counts.any()
	model.close()


# ---- 3. coherence through the Python API: streaming equals one shot ---------------------------------------------------
def write_corpus(path, doc_ptr, word_ids, counts):
	with open(path, 'w') as f:
		for d in range(len(doc_ptr) - 1):
			lo, hi = int(doc_ptr[d]), int(doc_ptr[d + 1])
			f.write('%d %s\n' % (hi - lo, ' '.join('%d:%d' % (w, c) for w, c in zip(word_ids[lo:hi], counts[lo:hi]))))


def test_streaming_equals_one_shot(tmp_path):
	import trlda.models
	from trlda.utils import coherence_from_counts, load_documents_csr, topic_coherence
	from trlda_b200.synth import make_corpus, to_lists
	K, V, B = 50, 4000, 1000
	csr = make_corpus(B, V, K, .1, .2, mean_length=70, seed=21)
	path = str(tmp_path / 'corpus.txt')
	write_corpus(path, *csr)
	model = trlda.models.OnlineLDA(V, K, 10000, .1, .2)
	model.update_parameters(make_corpus(256, V, K, .1, .2, mean_length=70, seed=21, doc_seed=5), max_iter_tr=2)
	top, probs = model.top_words(12)
	assert top.shape == (K, 12) and top.dtype == np.int32 and probs.shape == (K, 12)
	want_counts, _ = cooccurrence_numpy(*csr, top)
	for measure in ('npmi', 'umass'):
		one = topic_coherence(model, [csr], num_words=12, measure=measure)
		assert np.array_equal(one, coherence_from_counts(want_counts, B, measure))
		assert np.array_equal(topic_coherence(model, [to_lists(*csr)], num_words=12, measure=measure), one)
		assert np.array_equal(topic_coherence(model, [csr], measure=measure, top_words=top.astype(np.int64)), one)
		for b in (1, 7, 64, 333):
			streamed = topic_coherence(model, load_documents_csr(path, b), num_words=12, measure=measure)
			assert np.array_equal(streamed, one), (measure, b)
	counts, num_docs = model.cooccurrence(to_lists(*csr), top)
	assert num_docs == B and np.array_equal(counts, want_counts)


# ---- 4. training state ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_training_state_untouched(capi, precision):
	from trlda_b200.synth import make_corpus
	K, V = 256, 4000
	train = capi.CSR(*make_corpus(300, V, K, .1, .2, mean_length=60, seed=3))
	reference = capi.CSR(*make_corpus(200, V, K, .1, .2, mean_length=60, seed=3, doc_seed=9))
	lam0 = np.asfortranarray(np.random.default_rng(2).gamma(100., .01, size=(K, V)))
	kwargs = dict(max_iter_tr=2, max_iter_inference=20, update_alpha=1, update_eta=1)
	results = []
	for evaluate in (True, False):
		model = capi.Model('online', V, K, 10000, .1, .2, precision=precision)
		model.lambdas = lam0
		model.update_count = 3
		model.upload_docs_slot(train, 1)
		if evaluate:
			before = (model.lambdas, model.alpha, model.eta, model.update_count)
			top, _ = model.top_words(20)
			model.cooccurrence(reference, top)
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
def _raw_top_words(capi, model, n):
	ids = np.zeros(model.K * max(n, 1), dtype=np.int32)
	status = model._lib.trlda_top_words(model.h, n, ids.ctypes.data_as(C.POINTER(C.c_int32)), None)
	return status, model._lib.trlda_last_error(model.h).decode()


def _raw_cooccurrence(capi, model, docs, ids, n):
	ids = np.ascontiguousarray(ids, dtype=np.int32)
	counts = np.zeros(model.K * max(n, 1) ** 2, dtype=np.int64)
	num_docs = C.c_int64(0)
	status = model._lib.trlda_cooccurrence(model.h, C.byref(docs.c), ids.ctypes.data_as(C.POINTER(C.c_int32)), n,
		counts.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(num_docs))
	return status, model._lib.trlda_last_error(model.h).decode()


def test_errors(capi):
	K, V = 4, 20
	model = capi.Model('batch', V, K, 0, .1, .2)
	n_message = 'Number of top words must lie in [1, min(32, number of words)].'
	for n in (0, 33, V + 1, -1):
		assert _raw_top_words(capi, model, n) == (capi.ERR_ARG, n_message)
	good_docs = capi.CSR.from_lists([[(1, 2), (3, 1)], [(4, 4)]])
	good = np.arange(K * 3, dtype=np.int32).reshape(K, 3)
	bad_range = good.copy()
	bad_range[2, 1] = V
	negative = good.copy()
	negative[0, 0] = -1
	duplicate = good.copy()
	duplicate[3, 2] = duplicate[3, 0]
	cases = [
		(good_docs, np.zeros((K, 1)), 0, n_message),
		(good_docs, np.zeros((K, 33)), 33, n_message),
		(good_docs, bad_range, 3, 'Word ID out of range.'),
		(good_docs, negative, 3, 'Word ID out of range.'),
		(good_docs, duplicate, 3, 'Top words of a topic must be distinct.'),
		(capi.CSR(np.array([0, 2, 1, 3]), np.array([1, 2, 3]), np.array([1, 1, 1])), good, 3,
			'Document offsets must be non-decreasing.'),
		(capi.CSR.from_lists([[(1, 2)], [(V, 1)]]), good, 3, 'Word ID out of range.'),
		(capi.CSR.from_lists([[(1, -2)], [(4, 1)]]), good, 3, 'Word counts should not be negative.'),
	]
	for docs, ids, n, message in cases:
		assert _raw_cooccurrence(capi, model, docs, ids, n) == (capi.ERR_ARG, message)
		counts, num_docs = model.cooccurrence(good_docs, good)     # the model still works
		assert num_docs == 2 and counts[1, 0, 0] == 1
	with pytest.raises(ValueError):
		model.cooccurrence(good_docs, good[:2])
	model.close()

	import trlda.models
	lda = trlda.models.BatchLDA(V, K, .1, .2)
	for n in (0, 33, V + 1):
		with pytest.raises(RuntimeError, match=r'Number of top words must lie'):
			lda.top_words(n)
	with pytest.raises(RuntimeError, match='Top words of a topic must be distinct.'):
		lda.cooccurrence([[(1, 1)]], duplicate)
	with pytest.raises(RuntimeError, match='Word ID out of range.'):
		lda.cooccurrence([[(1, 1)]], np.where(good == 5, np.int64(1) << 40, good.astype(np.int64)))
	with pytest.raises(ValueError):
		lda.cooccurrence([[(1, 1)]], good[:, 0])


# ---- 6. coherence tracks training --------------------------------------------------------------------------------------
def test_training_raises_npmi_on_held_out_documents():
	import trlda
	import trlda.models
	from trlda.utils import topic_coherence
	from trlda_b200.synth import make_corpus
	K, V = 20, 2000
	trlda.seed(3)
	held_out = make_corpus(2000, V, K, .1, .05, mean_length=100, seed=12, doc_seed=999)
	model = trlda.models.OnlineLDA(V, K, 100000, .1, .05)
	before = topic_coherence(model, [held_out], num_words=10)
	for step in range(20):
		model.update_parameters(make_corpus(256, V, K, .1, .05, mean_length=100, seed=12, doc_seed=step), max_iter_tr=2)
	after = topic_coherence(model, [held_out], num_words=10)
	print('mean NPMI before %.4f after %.4f' % (before.mean(), after.mean()))
	assert after.mean() > before.mean() + .1


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
	assert lines[0].split()[1:] == ['True'] * 4


def _worker():
	import torch
	import torch.distributed as dist
	from trlda_b200 import capi
	from trlda_b200.distributed import init_comm, shard_documents

	rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
	local_rank = int(os.environ.get('LOCAL_RANK', rank))
	rng = np.random.default_rng(41)
	K, V = 1000, 10000
	full = capi.CSR.from_lists(corpus_with_edge_cases(rng, V, 200, 500, 12000))
	lam0 = np.asfortranarray(rng.gamma(100., .01, size=(K, V)))
	shard = capi.CSR(*shard_documents(full.doc_ptr, full.word_ids, full.counts, rank, world))

	torch.cuda.set_device(local_rank)
	dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
	model = capi.Model('online', V, K, 5000, .1, .2, device=local_rank)
	model.lambdas = lam0
	init_comm(model, dist, torch.device('cuda', local_rank))
	top, probs = model.top_words(20)
	sharded = model.cooccurrence(shard, top)
	model.close()
	model = capi.Model('online', V, K, 5000, .1, .2, device=local_rank)
	model.lambdas = lam0
	single_top, single_probs = model.top_words(20)
	single = model.cooccurrence(full, top)
	model.close()
	mine = torch.from_numpy(np.concatenate([top.ravel().view(np.uint8), probs.ravel().view(np.uint8)])).cuda()
	theirs = [torch.empty_like(mine) for _ in range(world)]
	dist.all_gather(theirs, mine)
	flags = torch.tensor([int(sharded[1] == single[1] == full.num_docs), int(np.array_equal(sharded[0], single[0])),
		int(np.array_equal(top, single_top) and np.array_equal(probs, single_probs)),
		int(all(torch.equal(t, theirs[0]) for t in theirs))], device='cuda')
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
