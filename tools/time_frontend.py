"""Times the frontend on a B200 (radix-16 FFT path, instance norm and bf16 pack) and, as a probe, the tensor-pipe cost of
DFT-as-GEMM in the split-bf16 tier (the [frames, 192] x [192, 256] contraction with hi*hi + hi*lo + lo*hi passes, run through
cab_conv1d_fused on a pre-built frame matrix: GEMM time only, no operand construction, no mel / log).  B = 80 x 15 s int16 PCM."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from convasr_b200 import models, ops, _lib

dev = torch.device('cuda:0')
B, T = 80, 120000
g = torch.Generator().manual_seed(0)
sig = (torch.randn(B, T, generator = g) * 3000).round().clamp(-32767, 32767).to(torch.int16).to(dev)
xlen = torch.ones(B, device = dev)
fe = models.LogFilterBankFrontend(64, 8000, .02, .01, 'hann_window').to(dev)
norm = models.MaskedInstanceNorm1d(64, affine = False, eps = 2.0**-14, track_running_stats = False, temporal_mask = True, legacy = True)
flush = torch.empty(256 << 20, dtype = torch.uint8, device = dev)

def timed(fn, n = 20):
	for _ in range(3): fn()
	torch.cuda.synchronize()
	tot = 0.0
	for _ in range(n):
		flush.zero_()
		e0, e1 = torch.cuda.Event(enable_timing = True), torch.cuda.Event(enable_timing = True)
		e0.record(); fn(); e1.record(); torch.cuda.synchronize()
		tot += e0.elapsed_time(e1)
	return tot / n * 1e3

us = timed(lambda: fe.features(sig, xlen, norm, True, 64, False))
with _lib.trace() as tr:
	fe.features(sig, xlen, norm, True, 64, False)
print(f'frontend + instance norm + pack, B = {B} x 15 s: {us:.1f} us (HBM floor for 19.2 MB in + 15.4 MB out: {(19.2e6 + 15.4e6) / 6548e9 * 1e6:.1f} us)')
# DFT-as-GEMM probe: tensor-pipe time of the split-bf16 contraction alone
F = T // 80 + 1
a_hi = torch.randn(B, F, 192, device = dev).to(torch.bfloat16); a_lo = (torch.randn(B, F, 192, device = dev) * 1e-3).to(torch.bfloat16)
w_hi = torch.randn(1, 256, 192, device = dev).to(torch.bfloat16); w_lo = (torch.randn(1, 256, 192, device = dev) * 1e-3).to(torch.bfloat16)
out = torch.empty(B, F, 256, dtype = torch.bfloat16, device = dev)
srcs = [ops.Source(a_hi, w_hi, 192, 1, 1, 0, T_in = F), ops.Source(a_hi, w_lo, 192, 1, 1, 0, T_in = F), ops.Source(a_lo, w_hi, 192, 1, 1, 0, T_in = F)]
us_g = timed(lambda: ops.conv1d_fused(srcs, B, F, 256, out_hi = out))
print(f'[dft-gemm probe] split-bf16 [B*F = {B * F}, 192] x [192, 256] x 3 passes through the tcgen05 conv kernel: {us_g:.1f} us (GEMM only; 16-bit operands bound the error by 2^-16 of the FRAME energy, not of the bin)')
