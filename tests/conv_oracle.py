"""Exact references for the conv GEMM (conv1d_umma_kernel) and the weight-gradient GEMM (wgrad_umma_kernel).

bf16 x bf16 products are exact in fp32.  When every operand is a small integer times a fixed power of two, every partial
sum of a launch is a multiple of the product granularity g; while its magnitude stays below 2^24 * g it is exactly
representable in fp32, so the fp32 accumulator is exact in any summation order (K chunks, sources, batch splits, L2
reductions).  The generators here build such operands and `assert_exact` refuses a case whose worst partial sum could
round.  The references are written on torch tensors in float64, so they run on the device in the GPU tests and on the
CPU in the host tests.
"""
import math

import torch

BF16 = torch.bfloat16
EXACT_LIMIT = 2.0 ** 24


# ------------------------------------------------------------------------------------------ data
def ints(shape, lo, hi, gen, zero_frac = 0.0):
	"""float32 tensor of integers uniform in [lo, hi] (a share `zero_frac` set to zero), drawn from a CPU generator"""
	x = torch.randint(lo, hi + 1, shape, generator = gen).to(torch.float32)
	if zero_frac > 0:
		x = x * (torch.rand(shape, generator = gen) >= zero_frac)
	return x


def split_ints(shape, gen, hi_max, lo_max, lo_exp, zero_frac = 0.0):
	"""(hi, lo) float32 pair: hi integers in [-hi_max, hi_max], lo integers in [-lo_max, lo_max] times 2^lo_exp.  Both parts
	are exact in bf16 while hi_max, lo_max <= 256."""
	assert hi_max <= 256 and lo_max <= 256
	hi = ints(shape, -hi_max, hi_max, gen, zero_frac)
	lo = ints(shape, -lo_max, lo_max, gen, zero_frac) * 2.0 ** lo_exp
	return hi, lo


def to_bf16_exact(x):
	"""bf16 copy of x that must not round (NaN poison stays NaN)"""
	y = x.to(BF16)
	assert torch.equal(y.float().nan_to_num(1e30), x.float().nan_to_num(1e30)), 'operand is not exact in bf16'
	return y


def poison_rows(x, T):
	"""NaN in rows T.. of a [B, T_rows, ld] tensor (in place)"""
	x[:, T:] = float('nan')
	return x


def poison_channels(x, off, n):
	"""NaN in every channel of the last dimension outside [off, off + n) (in place)"""
	x[..., :off] = float('nan')
	x[..., off + n:] = float('nan')
	return x


def assert_exact(abs_bound, granularity, what = ''):
	"""abs_bound: an upper bound of |partial sum| per output element (e.g. conv_acc64 of |a|, |w|); every partial sum is a
	multiple of `granularity`.  Refuses the case if a partial sum could reach 2^24 * granularity, where fp32 rounds."""
	worst = float(abs_bound.abs().max()) if abs_bound.numel() else 0.0
	ratio = worst / granularity
	if not ratio < EXACT_LIMIT:
		raise ValueError(f'{what}: a partial sum can reach {worst} = 2^{math.log2(ratio):.2f} x granularity {granularity}: '
						f'fp32 accumulation would not be exact')
	return ratio


# ------------------------------------------------------------------------------------------ conv GEMM
class Src:
	"""one K segment of a launch, as the kernel reads it: act [B, T_rows, ld] (rows >= T_in and channels outside [ch_off,
	ch_off + C_in) are never read), wgt [taps, w_rows, w_ld] (channels outside [w_ch_off, w_ch_off + C_in) never read)"""

	def __init__(self, act, wgt, C_in, taps, dil, pad_left, T_in = None, ch_off = 0, w_ch_off = 0):
		self.act, self.wgt, self.C_in, self.taps, self.dil, self.pad_left = act, wgt, C_in, taps, dil, pad_left
		self.T_in = act.shape[1] if T_in is None else T_in
		self.ch_off, self.w_ch_off = ch_off, w_ch_off

	def abs(self):
		a, w = self.act.double().abs(), self.wgt.double().abs()
		return Src(a, w, self.C_in, self.taps, self.dil, self.pad_left, self.T_in, self.ch_off, self.w_ch_off)


def conv_acc64(sources, B, T_out):
	"""float64 [B, T_out, max w_rows]: sum over sources and taps of W[tap] . x[t + tap * dil - pad_left], rows outside
	[0, T_in) zero, channel windows respected"""
	dev = sources[0].act.device
	N = max(s.wgt.shape[1] for s in sources)
	acc = torch.zeros(B, T_out, N, dtype = torch.float64, device = dev)
	t = torch.arange(T_out, device = dev)
	for s in sources:
		a = s.act[:B, :, s.ch_off:s.ch_off + s.C_in].double()
		w = s.wgt[:, :, s.w_ch_off:s.w_ch_off + s.C_in].double()
		n = w.shape[1]
		for tap in range(s.taps):
			idx = t + tap * s.dil - s.pad_left
			ok = (idx >= 0) & (idx < s.T_in)
			if not bool(ok.any()):
				continue
			xs = torch.zeros(B, T_out, s.C_in, dtype = torch.float64, device = dev)
			xs[:, ok] = a[:, idx[ok]]
			acc[:, :, :n] += xs @ w[tap].T
	return acc


def conv_bound(sources, B, T_out):
	"""per-element bound of every partial sum: the accumulation of |a| |w|"""
	return conv_acc64([s.abs() for s in sources], B, T_out)


def act_ref(y, act, a = 0.0, b = 0.0):
	"""the kernel's activations on an fp32 tensor (codes of _lib.ACT_*)"""
	if act == 1:
		return torch.clamp(y, min = 0.0)
	if act == 2:
		return torch.minimum(torch.maximum(y, torch.tensor(a, dtype = y.dtype, device = y.device)), torch.tensor(b, dtype = y.dtype, device = y.device))
	if act == 3:
		return torch.where(y > 0, y, y * torch.tensor(a, dtype = y.dtype))
	return y


def frac_lengths(xlen, T):
	"""ceil(fp32(frac) * T): the kernel's frac_len"""
	return (xlen.to(torch.float32) * torch.tensor(float(T), dtype = torch.float32)).ceil().long()


def act_bf16_ref(acc64, C_out, bias = None, act = 0, a = 0.0, b = 0.0, xlen = None, want_lo = False):
	"""ACT_BF16 epilogue: y = act(fp32(acc) + bias) * mask in fp32, hi = bf16_rn(y), lo = bf16_rn(y - hi)"""
	B, T = acc64.shape[:2]
	y = acc64[:, :, :C_out].to(torch.float32)
	if bias is not None:
		y = y + bias[:C_out].to(torch.float32)
	y = act_ref(y, act, a, b)
	if xlen is not None:
		keep = torch.arange(T, device = y.device)[None, :, None] < frac_lengths(xlen, T).to(y.device)[:, None, None]
		y = torch.where(keep, y, torch.zeros((), device = y.device))
	hi = y.to(BF16)
	lo = (y - hi.float()).to(BF16) if want_lo else None
	return hi, lo


def stats_ref(hi, lo = None):
	"""float64 [2, C]: per-channel sum and sum of squares of the stored values (hi + lo in fp32, as the kernel adds them)"""
	x = hi.float() if lo is None else hi.float() + lo.float()
	x = x.double()
	return torch.stack([x.sum(dim = (0, 1)), (x * x).sum(dim = (0, 1))])


def bnr_ref(g_hi, y, ss, C, act, a, b, xlen = None):
	"""folded BatchNorm-backward sums [2, C]: sum(dz) and sum(dz * y), dz = g * act'(y * scale + shift) * (t < len),
	with z = fmaf(y, scale, shift) (exact for the data the tests use)"""
	B, T = g_hi.shape[:2]
	g = g_hi[:, :, :C].double()
	yy = y[:, :, :C].double()
	z = yy * ss[0, :C].double() + ss[1, :C].double()
	if act == 1:
		dz = torch.where(z > 0, g, torch.zeros_like(g))
	elif act == 2:
		dz = torch.where((z > a) & (z < b), g, torch.zeros_like(g))
	elif act == 3:
		dz = torch.where(z > 0, g, g * float(torch.tensor(a, dtype = torch.float32)))
	else:
		dz = g
	if xlen is not None:
		keep = torch.arange(T, device = g.device)[None, :, None] < frac_lengths(xlen, T).to(g.device)[:, None, None]
		dz = dz * keep
	return torch.stack([dz.sum(dim = (0, 1)), (dz * yy).sum(dim = (0, 1))])


def logits_ref(acc64, C, bias = None):
	"""fp32 acc + bias, as LOGSOFTMAX / LOGITS_F32 / LOGITS_ROWS compute it: [B, T, C] fp32"""
	x = acc64[:, :, :C].to(torch.float32)
	return x if bias is None else x + bias[:C].to(torch.float32)


def argmax_lowest(x):
	"""argmax over the last dim, ties going to the lowest index"""
	m = x.max(dim = -1, keepdim = True).values
	idx = torch.arange(x.shape[-1], device = x.device).expand_as(x)
	return torch.where(x == m, idx, x.shape[-1]).min(dim = -1).values


def logsoftmax_ref(x32):
	"""float64 log-softmax and log-sum-exp of fp32 logits [..., C]"""
	x = x32.double()
	lse = torch.logsumexp(x, dim = -1)
	return x - lse[..., None], lse


# ------------------------------------------------------------------------------------------ weight gradient
def wgrad64(a, a_T, M, bx, b_T, N, taps, dil, pad_left, skip = None):
	"""float64 [taps, M, N]: out[tap, m, n] = sum_{b,t} a[b, t, m] * bx[b, t + tap * dil - pad_left, n] over t < a_T, frames of
	bx outside [0, b_T) zero; skip = (frac, T, margin): frames t >= ceil(frac[b] * T) + margin of `a` left out"""
	B = a.shape[0]
	dev = a.device
	A = a[:, :a_T, :M].double()
	if skip is not None:
		lens = (frac_lengths(skip[0], skip[1]).to(dev) + skip[2]).clamp(max = a_T)
		A = A * (torch.arange(a_T, device = dev)[None, :, None] < lens[:, None, None])
	X = bx[:, :b_T, :N].double()
	out = torch.zeros(taps, M, N, dtype = torch.float64, device = dev)
	t = torch.arange(a_T, device = dev)
	for tap in range(taps):
		idx = t + tap * dil - pad_left
		ok = (idx >= 0) & (idx < b_T)
		if not bool(ok.any()):
			continue
		out[tap] = torch.einsum('btm,btn->mn', A[:, ok], X[:, idx[ok]])
	return out


def wgrad_bound(a, a_T, M, bx, b_T, N, taps, dil, pad_left):
	return wgrad64(a.double().abs(), a_T, M, bx.double().abs(), b_T, N, taps, dil, pad_left)
