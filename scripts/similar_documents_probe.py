"""
Cost of the document index and the similar-documents search (trlda_index_documents / trlda_similar_documents; DESIGN.md
section 4.2).

Workload: K = 1000 topics, an index of D = 2^20 documents (2^19 when the host has less than 96 GB of memory; the line
`index` says which) with gamma ~ synth.gamma_matrix (Gamma(100, 1/100)), n = 10 neighbours, Q = 1 ... 8192 queries.  The
index (8.4 GB at D = 2^20) is far larger than the 126 MB L2.  It prints the card's name and power limit, then one JSON line
for the index build and one per (Q, path):
  * call_ms: host clock around whole calls (each ends in a device synchronise: upload of the queries, kernels, read-back);
  * affinity_ms, select_ms, prepare_ms: the call's kernels from torch.profiler (CUDA activities, a run of its own):
    k_similar_stream or k_distance_product; k_top_words_candidates and k_top_words_merge; k_similar_prepare;
  * streaming path: index bytes read per query group (8 K_pad ld bytes) over affinity_ms, and the share of 7.7 TB/s;
  * product path: 2 ld_Q K_pad ld_D flops (the tiles it computes) over affinity_ms, and the share of the 20.9 TFLOP/s
    k_distance_product reaches in topic_distances.
Both paths are run at the Q around the crossover (TRLDA_SIMILAR_STREAM_MAX selects them).

    python scripts/similar_documents_probe.py [--repeat 5] [--out results.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K = 1000
N = 10
HBM_TBS = 7.7
PRODUCT_TFLOPS = 20.9
GROUP = 8          # queries per CTA of the streaming pass


def card():
	try:
		out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv'],
			capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[-1]
	except (OSError, subprocess.SubprocessError, IndexError) as e:
		out = 'unknown (%s)' % e
	return out


def up(x, m):
	return (x + m - 1) // m * m


def kernel_ms(model, gamma, repeat):
	"""per-call kernel time by group, from torch.profiler"""
	import torch
	from torch.profiler import ProfilerActivity, profile
	with profile(activities=[ProfilerActivity.CUDA]) as prof:
		for _ in range(repeat):
			model.similar_documents(gamma, N)
		torch.cuda.synchronize()
	groups = {'affinity': ('k_similar_stream', 'k_distance_product'), 'select': ('k_top_words_candidates', 'k_top_words_merge'),
	          'prepare': ('k_similar_prepare',)}
	out = {g: 0. for g in groups}
	for e in prof.key_averages():
		for g, names in groups.items():
			if any(n in e.key for n in names):
				out[g] += e.device_time_total / 1e3 / repeat
	return out


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--repeat', type=int, default=5)
	ap.add_argument('--out', help='also write the card and the JSON lines to this file')
	args = ap.parse_args()
	import torch
	from trlda_b200 import capi
	from trlda_b200.synth import gamma_matrix

	print('card: %s' % card(), flush=True)
	host_gb = os.sysconf('SC_PAGE_SIZE') * os.sysconf('SC_PHYS_PAGES') / 2 ** 30
	D = 1 << 20 if host_gb >= 96 else 1 << 19
	torch.cuda.init()
	model = capi.Model('online', 100, K, 1000000, .1, .2)
	gamma = gamma_matrix(K, D, 1)
	torch.cuda.synchronize()
	t = time.perf_counter()
	model.index_documents(gamma)
	index_ms = (time.perf_counter() - t) * 1e3
	del gamma
	kp, ld_d = up(K, 8), up(D, 128)
	lines = [dict(case='index', K=K, D=D, host_gb=round(host_gb), index_gb=8 * kp * ld_d / 1e9, call_ms=index_ms)]
	print(json.dumps(lines[-1]), flush=True)

	default_max = 56
	cases = [(q, None) for q in (1, 4, 16, 64, 256, 1024, 8192)] + [(q, 'stream') for q in (128, 256)] + \
		[(q, 'product') for q in (16, 64)]
	for q, force in cases:
		if force == 'stream':
			os.environ['TRLDA_SIMILAR_STREAM_MAX'] = str(q)
		elif force == 'product':
			os.environ['TRLDA_SIMILAR_STREAM_MAX'] = '0'
		else:
			os.environ.pop('TRLDA_SIMILAR_STREAM_MAX', None)
		streaming = q <= int(os.environ.get('TRLDA_SIMILAR_STREAM_MAX', default_max))
		queries = gamma_matrix(K, q, 100 + q)
		model.similar_documents(queries, N)          # warm-up: allocations and module load
		t = time.perf_counter()
		for _ in range(args.repeat):
			model.similar_documents(queries, N)
		call_ms = (time.perf_counter() - t) * 1e3 / args.repeat
		ms = kernel_ms(model, queries, args.repeat)
		line = dict(case='search', Q=q, path='stream' if streaming else 'product', n=N, D=D, call_ms=call_ms,
			affinity_ms=ms['affinity'], select_ms=ms['select'], prepare_ms=ms['prepare'])
		if streaming:
			nbytes = 8. * kp * ld_d * ((q + GROUP - 1) // GROUP)
			line['bytes_per_group'] = 8. * kp * ld_d
			line['TBps'] = nbytes / (ms['affinity'] * 1e-3) / 1e12 if ms['affinity'] else None
			line['share_of_hbm'] = line['TBps'] / HBM_TBS if line['TBps'] else None
		else:
			flop = 2. * up(min(q, 8192), 128) * ((q + 8191) // 8192) * kp * ld_d
			line['flop'] = flop
			line['TFLOPs'] = flop / (ms['affinity'] * 1e-3) / 1e12 if ms['affinity'] else None
			line['share_of_product'] = line['TFLOPs'] / PRODUCT_TFLOPS if line['TFLOPs'] else None
		lines.append(line)
		print(json.dumps(line), flush=True)
	os.environ.pop('TRLDA_SIMILAR_STREAM_MAX', None)
	model.close()
	if args.out:
		with open(args.out, 'w') as f:
			f.write('card: %s\n' % card())
			for line in lines:
				f.write(json.dumps(line) + '\n')


if __name__ == '__main__':
	main()
