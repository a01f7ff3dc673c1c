"""
Cost of documents too long for the shared memory of the E-step kernels (DESIGN.md sections 4.2 and 10).

Starts from the cfg-3 minibatch (OnlineLDA K=1000, V=100 000, 8192 documents, mixed precision) and adds sets of long
documents of distinct words: none, one of 10 000 pairs, one of 50 000 pairs, four of 20 000 pairs.  For every set it
prints one JSON line with
  * step_ms      mean device-resident update_parameters step (T=10, I=20), CUDA events around `--steps` steps;
  * cold_estep_ms the E-step from a fresh gamma (I=20) alone, from the model's own kernel timers (stats()['ms']);
and, first, the card's name and power limit.  Nothing is written to disk.

    python scripts/long_doc_probe.py [--steps 5] [--warmup 2] [--label NAME]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K, V, B, D = 1000, 100000, 8192, 1000000
SETS = {'none': [], '1x10k': [10000], '1x50k': [50000], '4x20k': [20000] * 4}


def card():
	try:
		out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
			capture_output=True, text=True, timeout=30).stdout.strip()
	except (OSError, subprocess.SubprocessError) as e:
		out = 'unknown (%s)' % e
	return out


def with_long(docs, lengths, seed):
	"""the minibatch with documents of the given lengths (distinct word ids, counts 1-5) appended"""
	ptr, ids, cts = docs
	rng = np.random.default_rng(seed)
	ptr, ids, cts = list(ptr), [ids], [cts]
	for n in lengths:
		ids.append(rng.permutation(V)[:n].astype(np.int32))
		cts.append(rng.integers(1, 6, size=n).astype(np.int32))
		ptr.append(ptr[-1] + n)
	return np.array(ptr, dtype=np.int64), np.concatenate(ids), np.concatenate(cts)


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--steps', type=int, default=5)
	ap.add_argument('--warmup', type=int, default=2)
	ap.add_argument('--label', default='')
	args = ap.parse_args()
	import torch
	from trlda_b200 import capi
	from trlda_b200.synth import gamma_matrix, make_corpus

	print(json.dumps({'card': card(), 'label': args.label}), flush=True)
	base = make_corpus(B, V, K, .1, .2, seed=1003)
	lam0 = gamma_matrix(K, V, 2003)
	params = dict(max_iter_tr=10, max_iter_inference=20, kappa=.7, tau=100.)
	for name, lengths in SETS.items():
		docs = capi.CSR(*with_long(base, lengths, 7))
		nb = docs.doc_ptr.size - 1
		model = capi.Model('online', V, K, D, .1, .2, precision='mixed')
		model.lambdas = lam0
		g0 = gamma_matrix(K, nb, 3003)
		model.update_variables(docs, g0, max_iter=20, want_sstats=False)          # warm-up of every kernel the E-step uses
		model.set_profiling(True)
		model.reset_stats()
		model.update_variables(docs, g0, max_iter=20, want_sstats=False)
		cold = model.stats()['ms']['estep']
		model.set_profiling(False)

		model.upload_docs(docs)
		for _ in range(args.warmup):
			model.update_parameters_resident(**params)
		stream = torch.cuda.ExternalStream(model.stream)
		torch.cuda.synchronize()
		e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
		e0.record(stream)
		for _ in range(args.steps):
			model.update_parameters_resident(**params)
		e1.record(stream)
		torch.cuda.synchronize()
		finite = bool(np.all(np.isfinite(model.row_sums())))
		model.close()
		print(json.dumps({'label': args.label, 'set': name, 'documents': nb, 'long_pairs': lengths,
			'step_ms': round(e0.elapsed_time(e1) / args.steps, 3), 'cold_estep_ms': round(cold, 3), 'finite': finite}), flush=True)


if __name__ == '__main__':
	main()
