"""
Cost of topic inspection and document co-occurrence (trlda_top_words, trlda_cooccurrence; DESIGN.md section 4.2).

Workload: the cfg-3 shape (OnlineLDA K=1000, V=100 000) with lambda ~ Gamma(100, 1/100).  It prints one JSON line per
measurement, after the card's name and power limit:
  * top_words, n = 10, 20, 32: kernel_ms, the two top-word kernels per call (the `misc` kind of the model's kernel timers,
    CUDA events, mean over `--repeat` calls; the call's row-sum kernels count under other kinds), call_ms (host clock
    around calls that end in a device synchronise), algorithmic bytes (K V 8 + the candidate lists written and read
    again, chunks K n 12 each way) and that over kernel_ms against 7.7 TB/s.  lambda (800 MB) does not fit the 126 MB L2,
    so every call reads it from HBM;
  * cooccurrence, n = 10 and 20, on 8192-document make_corpus minibatches: kernel_ms (k_cooccurrence alone) and call_ms
    (upload and checks of the CSR, the inverse map, the kernel, read-back);
  * topic_coherence with n = 10 over `--batches` minibatches of 8192 documents streamed from a text file with the native
    reader (load_documents_csr), in documents/s.  The file is written to a temporary directory and removed.

    python scripts/coherence_probe.py [--repeat 20] [--batches 16]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K, V, B, D = 1000, 100000, 8192, 1000000
HBM_TB_S = 7.7


def card():
	try:
		out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv'],
			capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[-1]
	except (OSError, subprocess.SubprocessError, IndexError) as e:
		out = 'unknown (%s)' % e
	return out


def timed(fn, repeat):
	t0 = time.perf_counter()
	for _ in range(repeat):
		fn()
	return (time.perf_counter() - t0) * 1e3 / repeat


def misc_ms(model, fn, repeat):
	"""device time of the `misc` kernels per call, and their launches per call"""
	model.set_profiling(True)
	model.reset_stats()
	for _ in range(repeat):
		fn()
	stats = model.stats()
	model.set_profiling(False)
	return stats['ms']['misc'] / repeat, stats['launches']['misc'] // repeat


def write_corpus(path, batches):
	with open(path, 'w') as f:
		for doc_ptr, word_ids, counts in batches:
			for d in range(len(doc_ptr) - 1):
				lo, hi = int(doc_ptr[d]), int(doc_ptr[d + 1])
				f.write('%d %s\n' % (hi - lo, ' '.join('%d:%d' % p for p in zip(word_ids[lo:hi].tolist(), counts[lo:hi].tolist()))))


def top_words_chunks(n, sms):
	"""the word chunks of the candidate pass, as top_words_chunks (csrc/topics.cu) picks them on a B200: CTAs of 128
	threads with n * 128 * 12 bytes of lists, 16 CTAs or 228 KB of shared memory (1 KB reserved per CTA) per SM"""
	per_sm = min(16, (228 * 1024) // (n * 128 * 12 + 1024))
	slabs = (K + 127) // 128
	want = max(1, (per_sm * sms + slabs - 1) // slabs)
	chunk = max(256, (V + want - 1) // want)
	return (V + chunk - 1) // chunk


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--repeat', type=int, default=20)
	ap.add_argument('--batches', type=int, default=16)
	args = ap.parse_args()
	import torch
	import trlda.models
	from trlda.utils import load_documents_csr, topic_coherence
	from trlda_b200 import capi
	from trlda_b200.synth import gamma_matrix, make_corpus

	print(json.dumps({'card': card()}), flush=True)
	sms = torch.cuda.get_device_properties(0).multi_processor_count
	lam0 = gamma_matrix(K, V, 2003)
	model = capi.Model('online', V, K, D, .1, .2)
	model.lambdas = lam0
	for n in (10, 20, 32):
		call = lambda: model.top_words(n)
		call()
		call_ms = timed(call, args.repeat)
		kernel_ms, launches = misc_ms(model, call, args.repeat)
		chunks = top_words_chunks(n, sms)
		algorithmic_bytes = K * V * 8 + 2 * chunks * K * n * 12 + K * 8 + K * n * 12
		tb_s = algorithmic_bytes / (kernel_ms * 1e-3) / 1e12
		print(json.dumps({'what': 'top_words', 'n': n, 'kernels_per_call': launches, 'kernel_ms': round(kernel_ms, 4),
			'call_ms': round(call_ms, 3), 'chunks': chunks, 'algorithmic_bytes': algorithmic_bytes, 'tb_s': round(tb_s, 3),
			'hbm_frac': round(tb_s / HBM_TB_S, 3)}), flush=True)

	batches = [make_corpus(B, V, K, .1, .2, seed=1003, doc_seed=5000 + i) for i in range(args.batches)]
	for n in (10, 20):
		top, _ = model.top_words(n)
		docs = capi.CSR(*batches[0])
		call = lambda: model.cooccurrence(docs, top)
		call()
		call_ms = timed(call, args.repeat)
		kernel_ms, _ = misc_ms(model, call, args.repeat)
		print(json.dumps({'what': 'cooccurrence', 'n': n, 'documents': B, 'pairs': docs.num_pairs,
			'kernel_ms': round(kernel_ms, 4), 'call_ms': round(call_ms, 3)}), flush=True)
	model.close()

	lda = trlda.models.OnlineLDA(V, K, D, .1, .2)
	lda.lambdas = lam0
	with tempfile.TemporaryDirectory() as tmp:
		path = os.path.join(tmp, 'corpus.txt')
		write_corpus(path, batches)
		topic_coherence(lda, load_documents_csr(path, B), num_words=10)      # warm-up, and the file in the page cache
		t0 = time.perf_counter()
		values = topic_coherence(lda, load_documents_csr(path, B), num_words=10)
		seconds = time.perf_counter() - t0
	documents = B * args.batches
	print(json.dumps({'what': 'topic_coherence', 'n': 10, 'batches': args.batches, 'documents': documents,
		'seconds': round(seconds, 3), 'documents_per_s': round(documents / seconds), 'mean_npmi': float(values.mean())}), flush=True)


if __name__ == '__main__':
	main()
