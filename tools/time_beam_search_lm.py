"""Time the CTC prefix beam search with a word n-gram LM (cab_ctc_beam_search_lm) against the acoustic-only search.

  python tools/time_beam_search_lm.py [--profile]

Shape C2: B = 80, T = 751, C = 38 (the char labels), W = 100, N = 40, alpha = 0.8, beta = 1.5.  Two seeded synthetic
3-gram ARPA files (tests/beam_lm_oracle.py write_synthetic_arpa), written to a temporary directory: a small one (2 000
words, 20 000 bigrams and trigrams) whose tables fit the 126 MB L2, and a large one (200 000 words, 3 M bigrams, 3 M
trigrams) whose tables do not.  Posteriors: peaked (a sentence of the LM's words planted every 6th frame, scale 6, over
randn) and diffuse (randn log_softmax).  For each LM and each kind the acoustic and the LM search alternate, `iters`
calls each after warm-up, timed with CUDA events: ms per batch and µs per frame.  ARPA parse + table build and upload
times and table bytes are reported per LM.  With --profile (a separate run) the kernels' times come from torch.profiler.
The device name, power limit and max SM clock are printed in the same run.  Needs a CUDA device.
"""
import argparse
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import beam_lm_oracle as LO  # noqa: E402
from convasr_b200 import ops  # noqa: E402
from convasr_b200.lm import NGramLM  # noqa: E402
from time_beam_search import device_line, time_call  # noqa: E402

CHARS = list(LO.RU) + ['*', '.', '2', ' ', '|']


def posteriors(B, C, T, kind, words, seed = 0):
	g = torch.Generator().manual_seed(seed)
	if kind == 'diffuse':
		return torch.randn(B, C, T, generator = g).log_softmax(1).cuda()
	rng = np.random.default_rng(seed)
	cid = {l: c for c, l in enumerate(CHARS)}
	seqs = []
	for _ in range(B):
		text = ''
		while len(text) < T // 6:
			text += ('' if not text else ' ') + words[rng.integers(0, len(words))]
		seqs.append([cid[ch] for ch in text[:T // 6]])
	return LO.planted(B, C, T, seqs, C - 1, g, scale = 6.0).cuda()


def kernel_times(fn, calls = 3):
	"""ms per call of each beam kernel from torch.profiler, averaged over the launches the profiler recorded (a later
	profiling session in one process can drop a call, so the count is read, not assumed)"""
	from torch.profiler import ProfilerActivity, profile
	with profile(activities = [ProfilerActivity.CUDA]) as prof:
		for _ in range(calls):
			fn()
		torch.cuda.synchronize()
	out = {}
	for e in prof.key_averages():
		if 'beam_' in e.key and e.count:
			name = e.key.split('(')[0].split('::')[-1].replace('void ', '')
			out[name] = (getattr(e, 'device_time_total', getattr(e, 'cuda_time_total', 0.0)) / e.count / 1000.0, e.count)
	return out


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--warmup', type = int, default = 3)
	ap.add_argument('--iters', type = int, default = 10)
	ap.add_argument('--profile', action = 'store_true', help = 'kernel times from torch.profiler instead of CUDA-event timing')
	args = ap.parse_args()
	assert torch.cuda.is_available(), 'needs a CUDA device'
	print(device_line(), flush = True)
	B, C, T, W, N, alpha, beta = 80, 38, 751, 100, 40, 0.8, 1.5
	olen = torch.full((B, ), T, device = 'cuda', dtype = torch.int64)
	with tempfile.TemporaryDirectory() as tmp:
		for name, n_words, n_grams in (('small', 2000, 20000), ('large', 200000, 3000000)):
			path = os.path.join(tmp, f'{name}.arpa')
			words = LO.random_words(n_words, seed = 1, lengths = (2, 9))
			t0 = time.perf_counter()
			LO.write_synthetic_arpa(path, words, seed = 2, n_bigrams = n_grams, n_trigrams = n_grams)
			t1 = time.perf_counter()
			lm = NGramLM.from_arpa(path, CHARS)
			t2 = time.perf_counter()
			lm.device_struct(torch.device('cuda'))
			torch.cuda.synchronize()
			t3 = time.perf_counter()
			counts = [int(np.count_nonzero(t['key'])) for t in lm.tables]
			print(f'LM {name}: {n_words} words, n-grams {counts}, trie {len(lm.word)} nodes; tables {lm.nbytes / 2 ** 20:.1f} MiB '
					f'(n-gram {sum(t.nbytes for t in lm.tables) / 2 ** 20:.1f}, trie {(lm.child.nbytes + lm.word.nbytes) / 2 ** 20:.1f}); '
					f'ARPA {os.path.getsize(path) / 2 ** 20:.1f} MiB written in {t1 - t0:.1f} s, parsed + tables built in {t2 - t1:.1f} s, '
					f'uploaded in {t3 - t2:.2f} s', flush = True)
			for kind in ('peaked', 'diffuse'):
				lp = posteriors(B, C, T, kind, words)
				acoustic = lambda: ops.ctc_beam_search(lp, olen, beam_width = W, cutoff_top_n = N)  # noqa: E731
				fused = lambda: ops.ctc_beam_search(lp, olen, beam_width = W, cutoff_top_n = N, lm = lm, alpha = alpha, beta = beta)  # noqa: E731
				if args.profile:
					for label, fn in (('acoustic', acoustic), ('LM', fused)):
						fn()
						k = kernel_times(fn)
						tot = sum(v for v, _ in k.values())
						print(f'  profile {name} {kind:7s} {label:8s}: ' + ', '.join(f'{n} {v:.3f} ms ({100 * v / tot:.1f} %, {c} launches)' for n, (v, c) in sorted(k.items())),
								flush = True)
					continue
				ms = {'acoustic': [], 'LM': []}
				for _ in range(3):  # alternate
					ms['acoustic'].append(time_call(acoustic, args.warmup, args.iters))
					ms['LM'].append(time_call(fused, args.warmup, args.iters))
				for label in ('acoustic', 'LM'):
					v = min(ms[label])
					print(f'  C2 B={B} T={T} C={C} W={W} N={N} {kind:7s} {label:8s} LM={name}: {v:8.3f} ms/batch  {1000 * v / T:7.2f} us/frame  '
							f'(rounds: {", ".join(f"{x:.3f}" for x in ms[label])})', flush = True)
			del lm


if __name__ == '__main__':
	main()
