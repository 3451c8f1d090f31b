"""Time ctc.alignment: the one-CTA kernel (cab_ctc_alignment) against the cluster kernel (cab_ctc_alignment_long), and
the cluster path at long-recording sizes, with the recursion and the back-trace reported separately.

  python tools/time_ctc_align.py            # all shapes
  python tools/time_ctc_align.py --shapes a # the C2 alignment shape only

Shapes: (a) the C2 alignment shape, B = 80, t = 753, L = 169 (old entry; cluster entry forced to 1, 3 and 6 CTAs);
(b) four 10-minute utterances, T = 30 000, L = 8 000; (c) one hour, T = 180 000, L = 45 000.  Random log-probs over
C = 38 classes (the kernels' cost does not depend on the values).  Call times: CUDA events around `iters` calls after
warm-up.  Per-kernel times: torch.profiler over separate calls.  Needs a CUDA device; there is no CPU path.
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from convasr_b200 import ops  # noqa: E402


def device_line():
	q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output = True, text = True)
	return f'device: {torch.cuda.get_device_name(0)} | nvidia-smi: {q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "n/a"}'


def inputs(B, T, L, C = 38, seed = 0):
	g = torch.Generator(device = 'cuda').manual_seed(seed)
	lp = torch.randn(B, C, T, device = 'cuda', generator = g).log_softmax(1).permute(2, 0, 1)  # the model's [B, C, T] view
	y = torch.randint(0, C - 1, (B, L), device = 'cuda', generator = g)
	ylen = torch.full((B, ), L, device = 'cuda', dtype = torch.int64)
	olen = torch.full((B, ), T, device = 'cuda', dtype = torch.int64)
	return lp, y, olen, ylen, C - 1


def time_call(fn, warmup, iters):
	for _ in range(warmup):
		fn()
	torch.cuda.synchronize()
	e0, e1 = torch.cuda.Event(enable_timing = True), torch.cuda.Event(enable_timing = True)
	e0.record()
	for _ in range(iters):
		fn()
	e1.record()
	torch.cuda.synchronize()
	return e0.elapsed_time(e1) / iters


def kernel_times(fn, calls):
	"""mean device time per call of each of our kernels (torch.profiler, a run of its own)"""
	from torch.profiler import ProfilerActivity, profile
	fn()
	torch.cuda.synchronize()
	with profile(activities = [ProfilerActivity.CUDA]) as prof:
		for _ in range(calls):
			fn()
		torch.cuda.synchronize()
	out = {}
	for e in prof.key_averages():
		if 'ctc_align' in e.key:
			us = getattr(e, 'self_device_time_total', None)
			if us is None:
				us = e.self_cuda_time_total
			name = e.key.split('(')[0].replace('void ', '').replace('cab::', '')
			out[name] = us / calls / 1e3
	return out


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--shapes', default = 'abc')
	args = ap.parse_args()
	if not torch.cuda.is_available():
		raise SystemExit('time_ctc_align: needs a CUDA device')
	print(device_line(), flush = True)
	if 'a' in args.shapes:
		B, T, L = 80, 753, 169
		lp, y, olen, ylen, blank = inputs(B, T, L)
		ref = ops.ctc_alignment(lp, y, olen, ylen, blank)
		ms = time_call(lambda: ops.ctc_alignment(lp, y, olen, ylen, blank), 5, 50)
		print(f'(a) B={B} T={T} L={L} one-CTA kernel (cab_ctc_alignment): {ms:.3f} ms/call', flush = True)
		for spc in (0, 128, 64):
			got = ops.ctc_alignment(lp, y, olen, ylen, blank, _states_per_cta = spc)
			fn = lambda: ops.ctc_alignment(lp, y, olen, ylen, blank, _states_per_cta = spc)
			ms = time_call(fn, 5, 50)
			n_cta = 1 if spc == 0 else -(-(2 * L + 1) // spc)
			kt = kernel_times(fn, 10)
			print(f'(a) B={B} T={T} L={L} cluster kernel, {n_cta} CTA(s)/utterance (states_per_cta={spc}): {ms:.3f} ms/call, '
					f'kernels {", ".join(f"{k} {v:.3f} ms" for k, v in kt.items())}, equal to one-CTA: {torch.equal(got, ref)}', flush = True)
		kt = kernel_times(lambda: ops.ctc_alignment(lp, y, olen, ylen, blank), 10)
		print(f'(a) one-CTA kernel alone: {", ".join(f"{k} {v:.3f} ms" for k, v in kt.items())}', flush = True)
	for key, (B, T, L, warm, iters) in (('b', (4, 30000, 8000, 1, 5)), ('c', (1, 180000, 45000, 1, 3))):
		if key not in args.shapes:
			continue
		lp, y, olen, ylen, blank = inputs(B, T, L, seed = 1)
		fn = lambda: ops.ctc_alignment(lp, y, olen, ylen, blank)
		ms = time_call(fn, warm, iters)
		kt = kernel_times(fn, 2)
		ws = B * T * -(-(2 * L + 1) // 4)
		print(f'({key}) B={B} T={T} L={L} cluster kernel (library default split): {ms:.1f} ms/call, packed workspace {ws / 2**20:.0f} MiB, '
				f'kernels {", ".join(f"{k} {v:.2f} ms" for k, v in kt.items())}, recursion {1e3 * kt.get("ctc_align_cluster_kernel<false>", float("nan")) / T:.2f} us/frame',
				flush = True)
		del lp
		torch.cuda.empty_cache()


if __name__ == '__main__':
	main()
