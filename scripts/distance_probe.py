"""
Cost of the distances between topics (trlda_topic_distances; DESIGN.md section 4.2).

Workload: the cfg-3 shape (K=1000, V=100 000) with lambda ~ Gamma(100, 1/100) (800 MB, more than the 126 MB L2).  It prints
the card's name and power limit, then one JSON line per case:
  * self-comparison (K_A = K_B = 1000) under Hellinger and under Kullback-Leibler, and K=1000 against a K=100 model under
    both;
  * kernel_ms: the call's distance kernels (prepare, entropy, product, finish: the `misc` kind of the model's kernel timers,
    CUDA events around every launch, mean over `--repeat` calls; the two row-sum kernels count under other kinds);
  * call_ms: host clock around calls, each of which ends in a device synchronise (row sums, kernels, read-back of D);
  * flop = 2 K_A K_B V of the product, achieved fp64 TFLOP/s over kernel_ms and over call_ms, and the share of the data
    sheet's FP64 rate of the HGX B200 (37 TFLOP/s a GPU, dense, at a 1000 W power limit).

    python scripts/distance_probe.py [--repeat 10]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

V = 100000
FP64_TFLOPS = 37.


def card():
	try:
		out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv'],
			capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[-1]
	except (OSError, subprocess.SubprocessError, IndexError) as e:
		out = 'unknown (%s)' % e
	return out


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--repeat', type=int, default=10)
	args = ap.parse_args()
	from trlda_b200 import capi
	from trlda_b200.synth import gamma_matrix

	print('card: %s' % card(), flush=True)
	a = capi.Model('online', V, 1000, 1000000, .1, .2)
	a.lambdas = gamma_matrix(1000, V, 1)
	b = capi.Model('online', V, 100, 1000000, .1, .2)
	b.lambdas = gamma_matrix(100, V, 2)
	for other, kb in ((None, 1000), (b, 100)):
		for metric in ('hellinger', 'kullback_leibler'):
			a.topic_distances(other, metric)           # warm-up: allocations and module load
			a.set_profiling(True)
			a.reset_stats()
			for _ in range(args.repeat):
				a.topic_distances(other, metric)
			stats = a.stats()
			a.set_profiling(False)
			kernel_ms = stats['ms']['misc'] / args.repeat
			t0 = time.perf_counter()
			for _ in range(args.repeat):
				a.topic_distances(other, metric)
			call_ms = (time.perf_counter() - t0) * 1e3 / args.repeat
			flop = 2. * 1000 * kb * V
			print(json.dumps({
				'case': '%s K_A=1000 K_B=%d%s' % (metric, kb, ' (self)' if other is None else ''),
				'kernel_ms': round(kernel_ms, 3), 'launches': stats['launches']['misc'] // args.repeat,
				'call_ms': round(call_ms, 3), 'flop': flop,
				'kernel_tflops': round(flop / kernel_ms * 1e-9, 2), 'call_tflops': round(flop / call_ms * 1e-9, 2),
				'kernel_share_of_fp64_peak': round(flop / kernel_ms * 1e-9 / FP64_TFLOPS, 3),
				'floor_ms_at_peak': round(flop / (FP64_TFLOPS * 1e9), 3)}), flush=True)
	a.close()
	b.close()


if __name__ == '__main__':
	main()
