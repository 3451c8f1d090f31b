"""Time the CTC prefix beam search (cab_ctc_beam_search: prune, search and back-trace launches) with CUDA events.

  python tools/time_beam_search.py

Shapes: C2, B = 80, T = 751, C = 38, W = 100, N = 40 through the model's [B, C, T] layout; C4, B = 64, T = 751,
C = 5000 through the class-contiguous [B, C, T] view of the large-vocabulary head, W = 16 and W = 100, N = 40.  Each on
peaked posteriors (a planted label path, scale 6 for C = 38 and 10 for C = 5000) and on diffuse ones (randn log_softmax).
Reports ms per batch (CUDA events around `iters` calls after warm-up; the per-call workspace allocation comes from
torch's caching allocator) and µs per frame (ms per batch / T: the frames of an utterance run in sequence, the
utterances in parallel), and the three kernels' shares from torch.profiler over separate calls.  The device name,
power limit and max SM clock are printed in the same run.  Needs a CUDA device; there is no CPU path.
"""
import argparse
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from convasr_b200 import ops  # noqa: E402


def device_line():
	q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output = True, text = True)
	return f'device: {torch.cuda.get_device_name(0)} | nvidia-smi: {q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "n/a"}'


def posteriors(B, C, T, kind, layout, seed = 0):
	g = torch.Generator(device = 'cuda').manual_seed(seed)
	x = torch.randn(B, C, T, device = 'cuda', generator = g)
	if kind == 'peaked':
		path = torch.full((B, T), C - 1, device = 'cuda')
		pos = torch.arange(0, T, 6, device = 'cuda')
		path[:, pos] = torch.randint(0, C - 1, (B, pos.numel()), device = 'cuda', generator = g)
		x += (6.0 if C < 1000 else 10.0) * F.one_hot(path, C).permute(0, 2, 1)
	lp = x.log_softmax(1)
	if layout == 'btc':  # class-contiguous memory, [B, C, T] view (the large-vocabulary head's log_probs)
		lp = lp.permute(0, 2, 1).contiguous().permute(0, 2, 1)
	return lp


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


def kernel_shares(fn):
	from torch.profiler import ProfilerActivity, profile
	with profile(activities = [ProfilerActivity.CUDA]) as prof:
		for _ in range(3):
			fn()
		torch.cuda.synchronize()
	out = {}
	for e in prof.key_averages():
		if 'beam_' in e.key:
			name = e.key.split('(')[0].split('::')[-1].replace('void ', '')
			out[name] = getattr(e, 'device_time_total', getattr(e, 'cuda_time_total', 0.0)) / 3 / 1000.0
	return out


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--warmup', type = int, default = 3)
	ap.add_argument('--iters', type = int, default = 10)
	args = ap.parse_args()
	assert torch.cuda.is_available(), 'needs a CUDA device'
	print(device_line(), flush = True)
	T = 751
	shapes = [('C2', 80, 38, 100, 'bct'), ('C4', 64, 5000, 16, 'btc'), ('C4', 64, 5000, 100, 'btc')]
	for name, B, C, W, layout in shapes:
		for kind in ('peaked', 'diffuse'):
			lp = posteriors(B, C, T, kind, layout)
			olen = torch.full((B, ), T, device = 'cuda', dtype = torch.int64)
			fn = lambda: ops.ctc_beam_search(lp, olen, beam_width = W, cutoff_top_n = 40, topk = 1)  # noqa: E731
			ms = time_call(fn, args.warmup, args.iters)
			k = kernel_shares(fn)
			ks = ', '.join(f'{n} {v:.3f} ms' for n, v in sorted(k.items()))
			print(f'{name} B={B} T={T} C={C} W={W} N=40 {kind:7s}: {ms:8.3f} ms/batch  {1000 * ms / T:7.2f} us/frame  [{ks}]', flush = True)


if __name__ == '__main__':
	main()
