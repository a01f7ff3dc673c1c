"""
Cost of the topics of the words of documents (trlda_word_topics, DESIGN.md section 4.2).

Workload: the cfg-3 shape (OnlineLDA K=1000, V=100 000) with a TRAINED lambda (--train update_parameters steps on
make_corpus minibatches of 4096 documents: the cost of psi depends on how many entries of lambda lie below the shift point of
its recurrence), and 8192 documents the model has not seen, in mixed and fp64 precision.  It prints the card's name and
power limit, then one JSON line per (precision, n) with n = 1, 5, 32:
  * call_ms          the whole word_topics call (upload, E-step from the same initial gamma, the new kernels, read-back of
                     topics, probabilities and gamma), host clock around calls that end in a device synchronise, mean over
                     `--repeat` calls;
  * update_vars_ms   update_variables on the same documents and initial gamma without sufficient statistics, timed the
                     same way: call_ms - update_vars_ms is what the topics cost end to end;
  * kernel_ms        the new kernels alone (psi(gamma), the log-beta table and the pair pass: the `misc` kind of the
                     model's kernel timers, CUDA events around every launch, per call; the E-step's own beta preparation
                     has already run, so nothing else of the call counts as `misc`);
  * bytes, tb_s      table: lambda read + table written (U K 16); psi(gamma): B K 16; pairs: the table column and the
                     psi(gamma) column of every pair (N K 16) + 12 N of the list + 12 N n of results, over kernel_ms;
  * fp64_gop_s       exp evaluations (N K) + psi evaluations (U K + B K) over kernel_ms, in 10^9 per second.
Nothing is written to disk.

    python scripts/word_topics_probe.py [--repeat 5] [--warmup 2] [--train 4]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

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


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--repeat', type=int, default=5)
	ap.add_argument('--warmup', type=int, default=2)
	ap.add_argument('--train', type=int, default=4)
	args = ap.parse_args()
	from trlda_b200 import capi
	from trlda_b200.synth import gamma_matrix, make_corpus

	print(json.dumps({'card': card()}), flush=True)
	docs = capi.CSR(*make_corpus(B, V, K, .1, .2, seed=1003, doc_seed=4242))
	N, U = docs.word_ids.size, np.unique(docs.word_ids).size
	g0 = gamma_matrix(K, B, 3003)
	trainer = capi.Model('online', V, K, D, .1, .2, precision='mixed')
	trainer.lambdas = gamma_matrix(K, V, 2003)
	for step in range(args.train):
		trainer.update_parameters(capi.CSR(*make_corpus(4096, V, K, .1, .2, seed=1003, doc_seed=step)), max_iter_tr=2)
	lam = trainer.lambdas
	trainer.close()
	print(json.dumps({'documents': B, 'pairs': N, 'distinct_words': U, 'train_steps': args.train,
		'lambda_below_shift': round(float(np.mean(lam < 10.)), 4)}), flush=True)
	for precision in ('mixed', 'fp64'):
		model = capi.Model('online', V, K, D, .1, .2, precision=precision)
		model.lambdas = lam
		update_vars = lambda: model.update_variables(docs, g0, want_sstats=False)
		for _ in range(args.warmup):
			update_vars()
		update_vars_ms = timed(update_vars, args.repeat)
		for n in (1, 5, 32):
			call = lambda: model.word_topics(docs, n, g0)
			for _ in range(args.warmup):
				call()
			call_ms = timed(call, args.repeat)
			model.set_profiling(True)
			model.reset_stats()
			for _ in range(args.repeat):
				call()
			stats = model.stats()
			model.set_profiling(False)
			kernel_ms = stats['ms']['misc'] / args.repeat
			bytes_ = U * K * 16 + B * K * 16 + N * K * 16 + 12 * N + 12 * N * n
			ops = N * K + U * K + B * K
			print(json.dumps({'precision': precision, 'n': n, 'call_ms': round(call_ms, 3),
				'update_vars_ms': round(update_vars_ms, 3), 'topics_ms_end_to_end': round(call_ms - update_vars_ms, 3),
				'kernel_ms': round(kernel_ms, 3), 'launches': stats['launches']['misc'] // args.repeat,
				'estep_ms': round(stats['ms']['estep'] / args.repeat, 3), 'bytes': bytes_,
				'tb_s': round(bytes_ / (kernel_ms * 1e-3) / 1e12, 3),
				'hbm_frac_if_all_from_hbm': round(bytes_ / (kernel_ms * 1e-3) / 1e12 / HBM_TB_S, 3),
				'fp64_gop_s': round(ops / (kernel_ms * 1e-3) / 1e9, 1)}), flush=True)
		model.close()


if __name__ == '__main__':
	main()
