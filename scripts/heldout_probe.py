"""
Cost of the document-completion predictive log-likelihood (trlda_predictive_log_likelihood, DESIGN.md section 4.2).

Workload: the cfg-3 shape (OnlineLDA K=1000, V=100 000), 8192 documents the model has not seen drawn with make_corpus,
split 80/20 by trlda.utils.split_documents, in mixed and fp64 precision.  For each precision it prints one JSON line with
  * call_ms         the whole predictive_log_likelihood call (upload, E-step from the same initial gamma, scoring,
                    read-back), host clock around calls that end in a device synchronise, mean over `--repeat` calls;
  * lower_bound_ms  lower_bound on the observed part, timed the same way, for comparison;
  * kernel_ms       k_heldout_loglik alone: the `elbo` kind of the model's kernel timers during predictive calls (that
                    call launches no ELBO kernel), mean per launch;
  * tb_s, hbm_frac  algorithmic bytes (N_ho K 8 + B K 8 + 16 N_ho + 8 B) over kernel_ms, and that over 7.7 TB/s;
and, first, the card's name and power limit.  Nothing is written to disk.

    python scripts/heldout_probe.py [--repeat 5] [--warmup 2]
"""
import argparse
import json
import os
import subprocess
import sys
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


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--repeat', type=int, default=5)
	ap.add_argument('--warmup', type=int, default=2)
	args = ap.parse_args()
	from trlda_b200 import capi
	from trlda_b200.synth import gamma_matrix, make_corpus
	from trlda.utils import split_documents

	print(json.dumps({'card': card()}), flush=True)
	observed, held_out = split_documents(make_corpus(B, V, K, .1, .2, seed=1003, doc_seed=4242), .2, seed=5)
	obs, ho = capi.CSR(*observed), capi.CSR(*held_out)
	n_ho = ho.num_pairs
	algorithmic_bytes = n_ho * K * 8 + B * K * 8 + 16 * n_ho + 8 * B
	lam0, g0 = gamma_matrix(K, V, 2003), gamma_matrix(K, B, 3003)
	for precision in ('mixed', 'fp64'):
		model = capi.Model('online', V, K, D, .1, .2, precision=precision)
		model.lambdas = lam0
		predictive = lambda: model.predictive_log_likelihood(obs, ho, g0)
		bound = lambda: model.lower_bound(obs, g0)
		for _ in range(args.warmup):
			predictive()
			bound()
		call_ms = timed(predictive, args.repeat)
		lower_bound_ms = timed(bound, args.repeat)
		model.set_profiling(True)
		model.reset_stats()
		for _ in range(args.repeat):
			total, tokens, _ = predictive()
		stats = model.stats()
		model.set_profiling(False)
		model.close()
		kernel_ms = stats['ms']['elbo'] / stats['launches']['elbo']
		tb_s = algorithmic_bytes / (kernel_ms * 1e-3) / 1e12
		print(json.dumps({'precision': precision, 'documents': B, 'held_out_pairs': n_ho, 'held_out_tokens': tokens,
			'per_word': total / tokens, 'call_ms': round(call_ms, 3), 'lower_bound_ms': round(lower_bound_ms, 3),
			'kernel_ms': round(kernel_ms, 4), 'estep_ms': round(stats['ms']['estep'] / args.repeat, 3),
			'algorithmic_bytes': algorithmic_bytes, 'tb_s': round(tb_s, 3), 'hbm_frac': round(tb_s / HBM_TB_S, 3)}), flush=True)


if __name__ == '__main__':
	main()
