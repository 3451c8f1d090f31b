"""Time the CTC loss and gradient: the one-CTA kernels (cab_ctc_loss_fwd / cab_ctc_loss_bwd) against the cluster kernel
(cab_ctc_loss_long_fwd / cab_ctc_loss_long_bwd), and the cluster path at long-recording sizes, with the alpha pass and the
beta + gradient pass reported separately.

  python tools/time_ctc_loss.py            # all shapes
  python tools/time_ctc_loss.py --shapes a # the C2 loss shape only

Shapes: (a) the C2 shape, B = 80, t = 753, L = 169, loss + gradient (old entry; cluster entry forced to 1, 3 and 6 CTAs);
(b) four 10-minute utterances, T = 30 000, L = 8 000; (c) one hour, T = 180 000, L = 45 000; (b) and (c) loss only and
loss + gradient.  Random log-probs over C = 38 classes through the model's [B, C, T] view.  Call times: CUDA events around
`iters` calls after warm-up.  Per-kernel times: torch.profiler over separate calls.  Peak memory: torch's peak allocation
of one call above what was allocated before it.  Needs a CUDA device; there is no CPU path.
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
	lp = torch.randn(B, C, T, device = 'cuda', generator = g).log_softmax(1)  # leaf; the kernels see its [T, B, C] view
	y = torch.randint(0, C - 1, (B, L), device = 'cuda', generator = g)
	ylen = torch.full((B, ), L, device = 'cuda', dtype = torch.int64)
	olen = torch.full((B, ), T, device = 'cuda', dtype = torch.int64)
	return lp, y, olen, ylen, C - 1


def loss_fn(lp, y, olen, ylen, blank, spc = None, grad = True):
	def fn():
		if not grad:
			with torch.no_grad():
				return ops.ctc_loss(lp.permute(2, 0, 1), y, olen, ylen, blank, _states_per_cta = spc), None
		x = lp.detach().requires_grad_(True)
		nll = ops.ctc_loss(x.permute(2, 0, 1), y, olen, ylen, blank, _states_per_cta = spc)
		nll.sum().backward()
		return nll.detach(), x.grad
	return fn


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
	"""mean device time per call of each of our CTC kernels in ms (torch.profiler, a run of its own)"""
	from torch.profiler import ProfilerActivity, profile
	fn()
	torch.cuda.synchronize()
	with profile(activities = [ProfilerActivity.CUDA]) as prof:
		for _ in range(calls):
			fn()
		torch.cuda.synchronize()
	out = {}
	for e in prof.key_averages():
		if 'ctc_' in e.key:
			us = getattr(e, 'self_device_time_total', None)
			if us is None:
				us = e.self_cuda_time_total
			name = e.key.split('(')[0].replace('void ', '').replace('cab::', '')
			out[name] = us / calls / 1e3
	return out


def peak_bytes(fn):
	torch.cuda.synchronize()
	base = torch.cuda.memory_allocated()
	torch.cuda.reset_peak_memory_stats()
	out = fn()
	torch.cuda.synchronize()
	peak = torch.cuda.max_memory_allocated() - base
	del out
	return peak


def fmt(kt):
	return ", ".join(f"{k} {v:.3f} ms" for k, v in kt.items())


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--shapes', default = 'abc')
	args = ap.parse_args()
	if not torch.cuda.is_available():
		raise SystemExit('time_ctc_loss: needs a CUDA device')
	print(device_line(), flush = True)
	if 'a' in args.shapes:
		B, T, L = 80, 753, 169
		lp, y, olen, ylen, blank = inputs(B, T, L)
		ref_nll, ref_grad = loss_fn(lp, y, olen, ylen, blank)()
		ms = time_call(loss_fn(lp, y, olen, ylen, blank), 5, 50)
		kt = kernel_times(loss_fn(lp, y, olen, ylen, blank), 10)
		print(f'(a) B={B} T={T} L={L} loss + gradient, one-CTA kernels (cab_ctc_loss_fwd/bwd): {ms:.3f} ms/call, kernels {fmt(kt)}', flush = True)
		for spc in (0, 128, 64):
			fn = loss_fn(lp, y, olen, ylen, blank, spc)
			nll, grad = fn()
			ms = time_call(fn, 5, 50)
			n_cta = 1 if spc == 0 else -(-(2 * L + 1) // spc)
			kt = kernel_times(fn, 10)
			err = float((grad - ref_grad).norm() / ref_grad.norm())
			print(f'(a) B={B} T={T} L={L} loss + gradient, cluster kernel, {n_cta} CTA(s)/utterance (states_per_cta={spc}): {ms:.3f} ms/call, '
					f'kernels {fmt(kt)}, nll equal to one-CTA: {torch.equal(nll, ref_nll)}, gradient rel. diff {err:.1e}', flush = True)
		del lp, ref_grad
		torch.cuda.empty_cache()
	for key, (B, T, L, warm, iters) in (('b', (4, 30000, 8000, 1, 3)), ('c', (1, 180000, 45000, 1, 2))):
		if key not in args.shapes:
			continue
		lp, y, olen, ylen, blank = inputs(B, T, L, seed = 1)
		for grad in (False, True):
			fn = loss_fn(lp, y, olen, ylen, blank, grad = grad)
			ms = time_call(fn, warm, iters)
			peak = peak_bytes(fn)
			kt = kernel_times(fn, 1)
			what = 'loss + gradient' if grad else 'loss only'
			alpha = kt.get('ctc_loss_cluster_kernel<1>' if grad else 'ctc_loss_cluster_kernel<0>', float('nan'))
			line = (f'({key}) B={B} T={T} L={L} {what}: {ms:.1f} ms/call, peak allocation {peak / 2**30:.2f} GiB, kernels {fmt(kt)}; '
					f'alpha pass {1e3 * alpha / T:.2f} us/frame')
			if grad:
				line += f', beta + gradient pass {1e3 * kt.get("ctc_loss_cluster_kernel<2>", float("nan")) / T:.2f} us/frame'
			print(line, flush = True)
			torch.cuda.empty_cache()
		del lp
		torch.cuda.empty_cache()


if __name__ == '__main__':
	main()
