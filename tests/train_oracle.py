"""References for the training-step kernels of csrc/train.cu and csrc/optim.cu: the streamed and row-walker BatchNorm
passes, the multi-branch forward and its dz pass, weight packing / unpacking, the logits-gradient layout cast and the
multi-tensor optimizer step.

Exact data.  bf16 activations are small integers times a power of two; the scale / shift table `ss` is given by the test
(scale, mean and invstd signed powers of two, shift a small dyadic) and B*T is a power of two, so 1 / n is exact.  Then
z = fmaf(y, scale, shift), the gates, dz, the fp32 partial sums, the fp64 replica sums, the centred second sum, the
apply coefficients and the apply output are all exactly representable, whatever FMA contraction the compiler chose and
in whatever order the partial sums are added.  `bn_bwd_ref(..., check = True)` verifies that premise on the data it is
given: each elementwise result must be an fp32 value, and each sum must stay below 2^24 times the granularity of its
terms (conv_oracle.assert_exact); otherwise it raises ValueError and the case is refused.

The references are written on torch tensors in float64 (fp32 where the kernel's own rounding is the contract: the
dropout scale, the split-bf16 lo part), so they run on the device in the GPU tests and on the CPU in the host tests.
"""
import math

import numpy as np
import torch

from conv_oracle import BF16, assert_exact, frac_lengths

# ------------------------------------------------------------------------------------------ launch geometry
STREAM_UNITS = 4          # kStreamUnits: 16-byte units per thread per chunk
STREAM_MAX_THREADS = 512  # kStreamMaxThreads
STAGE_BUDGET = 48 * 1024
SUM_REPLICAS = 8          # kBnSumReplicas
SM_COUNT = 148
ROW_LANES = 8             # kRowLanes of the row walkers
WALKER_BLOCKS_TARGET = 148 * 8


def stream_geometry(R, ld, n_inputs):
	"""stream_geometry() of train.cu: None when the streamed kernels do not cover the pitch, else the launch geometry.
	n_inputs: 1 forward, 2 forward split / backward, 4 backward split"""
	if ld % 8 != 0 or R <= 0:
		return None
	vectors = ld // 8
	lanes = max(1, 256 // vectors)
	while (vectors * lanes) % 32:
		lanes += 1
	threads = vectors * lanes
	if threads > STREAM_MAX_THREADS:
		return None
	rows_per_chunk = STREAM_UNITS * lanes
	stage_bytes = STREAM_UNITS * threads * 16
	stages = min(8, max(2, STAGE_BUDGET // (n_inputs * stage_bytes)))
	smem = stages * n_inputs * stage_bytes + 8 * stages
	smem = (smem + 15) & ~15
	smem += 4 * ld * 4
	smem = max(smem, threads * 64)
	if smem > 220 * 1024:
		return None
	return dict(ld = ld, vectors = vectors, lanes = lanes, threads = threads, rows_per_chunk = rows_per_chunk, stages = stages,
				stage_bytes = stage_bytes, smem = smem, n_chunks = (R + rows_per_chunk - 1) // rows_per_chunk)


def resident_cta_bound(geo, sms = SM_COUNT):
	"""an upper bound of the persistent grid: no SM holds more than min(2048 / threads, 228 KB / smem, 32) CTAs"""
	return sms * min(2048 // geo['threads'], (228 * 1024) // geo['smem'], 32)


def ring_wraps(geo, sms = SM_COUNT):
	"""a lower bound of how many times every CTA's stage ring wraps (chunks per CTA / stages - 1)"""
	per_cta = geo['n_chunks'] // resident_cta_bound(geo, sms)
	return per_cta // geo['stages'] - 1


def rows_per_block_for(R, ld):
	cols = (ld // 8 + 31) // 32
	rpb = (R * cols + WALKER_BLOCKS_TARGET - 1) // WALKER_BLOCKS_TARGET
	rpb = (rpb + 31) // 32 * 32
	return min(512, max(32, rpb))


# ------------------------------------------------------------------------------------------ dropout
_M64 = (1 << 64) - 1


def dropout_keep(seed, salt, rows, ld, p):
	"""keep mask [rows, ld] of the kernels' dropout_keep: splitmix64 of (seed + salt * 0xD1B54A32D192ED03) + idx * golden, idx =
	row * ld + channel; kept when the top 24 bits >= fp32(p) * 2^24 (compared as integers)"""
	s = np.uint64((seed + salt * 0xD1B54A32D192ED03) & _M64)
	idx = np.arange(rows * ld, dtype = np.uint64)
	with np.errstate(over = 'ignore'):
		z = s + idx * np.uint64(0x9E3779B97F4A7C15)
		z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
		z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
		z ^= z >> np.uint64(31)
	thr = math.ceil(float(np.float32(p)) * 2.0 ** 24)
	return torch.from_numpy((z >> np.uint64(40)).astype(np.int64) >= thr).view(rows, ld)


def inv_keep32(p):
	"""the kernels' 1.f / (1.f - p)"""
	return float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))


def row_mask(B, T, xlen, dev):
	"""bool [B, T, 1]: t < ceil(fp32(frac) * T), all true without xlen"""
	if xlen is None:
		return torch.ones(B, T, 1, dtype = torch.bool, device = dev)
	return (torch.arange(T, device = dev)[None, :] < frac_lengths(xlen.cpu(), T).to(dev)[:, None])[..., None]


# ------------------------------------------------------------------------------------------ exactness
def fp32_exact(x, what):
	"""every element of the float64 tensor x is an fp32 value: one fp32 operation producing it cannot round"""
	x = x.double()
	bad = x.float().double() != x
	if bool(bad.any()):
		raise ValueError(f'{what}: {int(bad.sum())} values are not exact in fp32 (e.g. {float(x[bad][0])!r})')


def grain(x):
	"""largest power of two dividing every nonzero element of a float64 tensor (1.0 for an all-zero tensor)"""
	nz = x[x != 0].double().abs()
	if nz.numel() == 0:
		return 1.0
	m, e = torch.frexp(nz)
	# m in [0.5, 1) has at most 53 significant bits: the lowest set bit of m * 2^53
	mi = (m * 2.0 ** 53).to(torch.int64)
	low = (mi & -mi).double()
	return float((low * torch.pow(2.0, (e - 53).double())).min())


def assert_sum_exact(terms, dims, what):
	"""every partial sum over `dims` of `terms`, in any order, is exact in fp32"""
	assert_exact(terms.abs().sum(dim = dims), grain(terms), what)


# ------------------------------------------------------------------------------------------ exact data
def ints(shape, lo, hi, gen):
	return torch.randint(lo, hi + 1, shape, generator = gen).double()


def pow2_table(C, gen, lo_exp, hi_exp, signed = True):
	e = torch.randint(lo_exp, hi_exp + 1, (C, ), generator = gen).double()
	s = torch.where(torch.rand(C, generator = gen) < 0.5, -1.0, 1.0) if signed else torch.ones(C, dtype = torch.float64)
	return s * torch.pow(2.0, e)


def exact_ss(C, gen):
	"""[4, C] float64: scale = +-2^k (some negative: negative gammas), shift = small dyadic, mean = +-2^k, invstd = 2^k"""
	sc = pow2_table(C, gen, -2, 1)
	sh = ints((C, ), -12, 12, gen) / 4
	mean = pow2_table(C, gen, -2, 1)
	istd = pow2_table(C, gen, -1, 1, signed = False)
	return torch.stack([sc, sh, mean, istd])


def plant_z(y, ss, C, targets, gen):
	"""set some entries of y (float64 [R, ld]) so that z = y * scale + shift lands exactly on each target value; y stays a
	multiple of 1/4 below 16 in magnitude (exact in bf16, and small
	enough that the apply output stays exact)"""
	R = y.shape[0]
	for v in targets:
		rows = torch.randint(0, R, (max(1, R // 32), ), generator = gen)
		cols = torch.randint(0, C, rows.shape, generator = gen)
		yv = (v - ss[1, cols]) / ss[0, cols]
		ok = (yv * 4 == (yv * 4).round()) & (yv.abs() < 16)
		y[rows[ok], cols[ok]] = yv[ok]
	return y


# ------------------------------------------------------------------------------------------ BatchNorm references
def act64(z, act, a, b):
	if act == 1:
		return torch.clamp(z, min = 0.0)
	if act == 2:
		return torch.clamp(z, min = a, max = b)
	if act == 3:
		return torch.where(z > 0, z, z * a)
	return z


def gate64(z, g, act, a, b):
	"""g * act'(z), selected (never multiplied) for the 0 / 1 gates"""
	if act == 1:
		return torch.where(z > 0, g, torch.zeros_like(g))
	if act == 2:
		return torch.where((z > a) & (z < b), g, torch.zeros_like(g))
	if act == 3:
		return torch.where(z > 0, g, g * a)
	return g


def split_store(o32):
	"""(hi, lo) bf16 of an fp32 tensor, as store_split / pack8_lo compute it"""
	hi = o32.to(BF16)
	lo = (o32 - hi.float()).to(BF16)
	return hi, lo


def bn_fwd_ref(y, ss, B, T, C, act, a, b, xlen = None, drop = None):
	"""y: float64 [B*T, ld] (hi + lo in the split tier); ss [4, C]; drop = (p, keep mask [B*T, ld]) or None.
	-> fp32 [B*T, ld] before the bf16 store: act(fmaf(y, scale, shift)) masked, channels >= C zero, dropout scaled in fp32"""
	R, ld = y.shape
	dev = y.device
	z = y[:, :C] * ss[0, :C] + ss[1, :C]
	o = torch.zeros(R, ld, dtype = torch.float64, device = dev)
	o[:, :C] = act64(z, act, a, b)
	o = torch.where(row_mask(B, T, xlen, dev).reshape(R, 1), o, torch.zeros((), dtype = torch.float64, device = dev))
	o = o.float()
	if drop is not None:
		p, keep = drop
		o = torch.where(keep.to(dev), o * torch.tensor(inv_keep32(p), dtype = torch.float32, device = dev), torch.zeros((), device = dev))
	return o


def bn_bwd_ref(y, g, ss, B, T, C, act, a, b, xlen = None, drop = None, frozen = False, check = False):
	"""backward of out = mask(dropout(act(y * scale + shift))) w.r.t. y for a batch-statistics BatchNorm (frozen: running
	statistics, dy = scale * dz).  y, g: float64 [B*T, ld] (g may hold anything on masked rows and channels >= C: it is
	selected away).  -> dict(dz, sums = [sum dz, sum dz * xhat] (float64 [2, C]), raw = [sum dz, sum dz * y], dy (fp32 [B*T, ld]))
	check: raise ValueError unless the kernels' arithmetic is exact on this data."""
	R, ld = y.shape
	dev = y.device
	keep_rows = row_mask(B, T, xlen, dev).reshape(R, 1)
	yc, gc = y[:, :C], g[:, :C]
	if drop is not None:
		p, keep = drop
		gc = torch.where(keep[:, :C].to(dev), gc * inv_keep32(p), torch.zeros((), dtype = torch.float64, device = dev))
	z = yc * ss[0, :C] + ss[1, :C]
	dz = torch.where(keep_rows, gate64(z, gc, act, a, b), torch.zeros((), dtype = torch.float64, device = dev))
	s1 = dz.sum(0)
	s2y = (dz * yc).sum(0)
	mean, istd, sc = ss[2, :C], ss[3, :C], ss[0, :C]
	m2 = istd * (s2y - mean * s1)
	inv_n = 0.0 if frozen else 1.0 / R
	k1 = -sc * (m2 * inv_n) * istd
	k0 = -sc * (s1 * inv_n) - k1 * mean
	dy = torch.zeros(R, ld, dtype = torch.float64, device = dev)
	dy[:, :C] = sc * dz + (k1 * yc + k0)
	if check:
		fp32_exact(z, 'z = y * scale + shift')
		fp32_exact(gc, 'g / (1 - p)')
		assert_sum_exact(dz, 0, 'sum(dz)')
		assert_sum_exact(dz * yc, 0, 'sum(dz * y)')
		assert_sum_exact(istd * (dz * yc - mean * dz), 0, 'row walker: centred partial sums')
		for v, what in ((s1, 'sum(dz)'), (m2, 'centred sum'), (m2 * inv_n, 'm2 / n'), (s1 * inv_n, 'm1 / n'), (k1, 'k1'), (k0, 'k0'),
						(sc * (s1 * inv_n), 'scale * m1 / n'), (k1 * mean, 'k1 * mean'), (k1 * yc, 'k1 * y'), (k1 * yc + k0, 'k1 * y + k0'),
						(sc * dz, 'scale * dz'), (dy, 'dy')):
			fp32_exact(v, what)
	return dict(dz = dz, sums = torch.stack([s1, m2]), raw = torch.stack([s1, s2y]), dy = dy.float())


def batch_stats_ref(y, C, n, gamma, beta, eps, momentum, running_mean = None, running_var = None):
	"""float64 BatchNorm1d training statistics of y [n, >= C]: biased variance for the normalisation, running_var with the
	unbiased one (n / max(n - 1, 1)).  -> (ss [4, C] = scale, shift, mean, invstd; running_mean'; running_var')"""
	x = y[:, :C].double()
	mean = x.mean(0)
	var = (x * x).mean(0) - mean * mean
	istd = 1.0 / torch.sqrt(var.clamp(min = 0) + eps)
	g = gamma.double() if gamma is not None else torch.ones_like(mean)
	bb = beta.double() if beta is not None else torch.zeros_like(mean)
	ss = torch.stack([g * istd, bb - mean * g * istd, mean, istd])
	rm = None if running_mean is None else (1 - momentum) * running_mean.double() + momentum * mean
	rv = None if running_var is None else (1 - momentum) * running_var.double() + momentum * var * (n / max(n - 1, 1))
	return ss, rm, rv


def multi_fwd_ref(branches, B, T, C, act, a, b, xlen = None, drop = None):
	"""branches: [(y float64 [R, ld], ss [4, C] or None)]: z = sum of fmaf(y_i, scale_i, shift_i) (identity: y_i), then as
	bn_fwd_ref.  -> (z float64 [R, C], out fp32 [R, ld])"""
	R, ld = branches[0][0].shape
	dev = branches[0][0].device
	z = torch.zeros(R, C, dtype = torch.float64, device = dev)
	for y, ss in branches:
		z = z + (y[:, :C] * ss[0, :C] + ss[1, :C] if ss is not None else y[:, :C])
	ident = torch.stack([torch.ones(C, dtype = torch.float64, device = dev), torch.zeros(C, dtype = torch.float64, device = dev)])
	zf = torch.zeros(R, ld, dtype = torch.float64, device = dev)
	zf[:, :C] = z
	return z, bn_fwd_ref(zf, ident, B, T, C, act, a, b, xlen, drop)


def dz_stored_gate_ref(out, g, B, T, C, act, a, b, xlen = None, drop = None):
	"""cab_act_mask_bwd_dz: dz = g * gate(v) with v = out * (1 - p) in fp32 (out: the stored fp32 value, hi + lo), then
	dropout; float64 [R, ld] (channels >= C and masked rows zero)"""
	R, ld = out.shape
	dev = out.device
	p = drop[0] if drop is not None else 0.0
	v = (out.float() * torch.tensor(float(np.float32(1.0) - np.float32(p)), dtype = torch.float32, device = dev)).double()
	gate = torch.zeros(R, ld, dtype = torch.float64, device = dev)
	ones = torch.ones_like(v[:, :C])
	gate[:, :C] = gate64(v[:, :C], ones, act, a, b) if act != 3 else torch.where(v[:, :C] > 0, ones, ones * a)
	d = (g.float() * gate.float()).double()
	if drop is not None:
		d = torch.where(drop[1].to(dev), (d.float() * inv_keep32(p)).double(), torch.zeros((), dtype = torch.float64, device = dev))
	d[:, C:] = 0
	return torch.where(row_mask(B, T, xlen, dev).reshape(R, 1), d, torch.zeros((), dtype = torch.float64, device = dev))


def z_gate(z, act, a, b):
	"""autograd's gate act'(z), float64"""
	return gate64(z, torch.ones_like(z), act, a, b)


# ------------------------------------------------------------------------------------------ packing
def taps2(K, pad):
	return (K - 1 - pad) // 2 - (0 - pad) // 2 + 1


def pack_ref(w, ci_ld, co_ld, mode = 0, pad = 0):
	"""float64 packed operands of an fp32 weight [Co, Ci, K] (NaN in the slots the kernel never writes).
	mode 0: fwd [K, Co, ci_ld] = w[co, ci, k], dgrad [K, Ci, co_ld] = w[co, ci, K - 1 - k];
	mode 1: stride-2 pair layout fwd [taps2, Co, 2 * ci_ld]: tap k lands at pair tap floor((k - pad) / 2) - floor(-pad / 2),
	channel block q = (k - pad) mod 2 (engine.pack_taps_stride2); no dgrad operand"""
	Co, Ci, K = w.shape
	w = w.double()
	nan = float('nan')
	if mode == 0:
		fwd = torch.full((K, Co, ci_ld), nan, dtype = torch.float64, device = w.device)
		fwd[:, :, :Ci] = w.permute(2, 0, 1)
		dgr = torch.full((K, Ci, co_ld), nan, dtype = torch.float64, device = w.device)
		dgr[:, :, :Co] = w.flip(2).permute(2, 1, 0)
		return fwd, dgr
	n2 = taps2(K, pad)
	fwd = torch.full((n2, Co, 2 * ci_ld), nan, dtype = torch.float64, device = w.device)
	dp_min = (0 - pad) // 2
	for k in range(K):
		j = k - pad
		dp, q = j // 2, j % 2
		fwd[dp - dp_min, :, q * ci_ld:q * ci_ld + Ci] = w[:, :, k]
	return fwd, None


def unpack_ref(packed, K, Co, Ci, mode, pair_pad = 0, pair_ci_alloc = 0):
	"""float64 [Co, Ci, K] gradient from a packed fp32 gradient: mode 0 [K, Co, ld], mode 1 [K, Ci, ld] (transposed),
	mode 2 the stride-2 pair layout [taps2, Co, ld] with channel block q at q * pair_ci_alloc"""
	p = packed.double()
	if mode == 0:
		return p[:, :Co, :Ci].permute(1, 2, 0).contiguous()
	if mode == 1:
		return p[:, :Ci, :Co].permute(2, 1, 0).contiguous()
	out = torch.empty(Co, Ci, K, dtype = torch.float64, device = p.device)
	dp_min = (0 - pair_pad) // 2
	for k in range(K):
		j = k - pair_pad
		dp, q = j // 2, j % 2
		out[:, :, k] = p[dp - dp_min, :Co, q * pair_ci_alloc:q * pair_ci_alloc + Ci]
	return out


def bct_to_btc_ref(x, ld):
	"""fp32 [B, C, T] -> float64 [B, T, ld] (channels >= C zero) and the per-class sums over (b, t)"""
	B, C, T = x.shape
	out = torch.zeros(B, T, ld, dtype = torch.float64, device = x.device)
	out[:, :, :C] = x.double().permute(0, 2, 1)
	return out, x.double().sum(dim = (0, 2))


# ------------------------------------------------------------------------------------------ optimizers
def clip_coef(grads, max_norm):
	"""float64 global norm over all gradients and torch.nn.utils.clip_grad_norm_'s coefficient"""
	total = math.sqrt(sum(float((g.double() ** 2).sum()) for g in grads))
	return total, (min(max_norm / (total + 1e-6), 1.0) if max_norm else 1.0)


def sgd_step(p, g, buf, lr, momentum, dampening, weight_decay, nesterov, coef = 1.0):
	"""torch.optim.SGD on float64 tensors (buf None on the first step) -> (p', buf')"""
	d = g.double() * coef + weight_decay * p.double()
	buf = d.clone() if buf is None else buf * momentum + (1 - dampening) * d
	step = d + momentum * buf if nesterov else buf
	return p.double() - lr * step, buf


def novograd_step(p, g, buf, ema, lr, beta1, beta2, eps, weight_decay, dampening, coef = 1.0):
	"""the reference's NovoGrad (optimizers.py:72-90) on float64 tensors, per tensor; ema None on the first step
	-> (p', buf', ema')"""
	gc = g.double() * coef
	g2 = float((gc ** 2).sum())
	ema = g2 if ema is None else ema * beta2 + g2 * (1 - beta2)
	d = gc / math.sqrt(ema + eps) + weight_decay * p.double()
	if dampening:
		d = d * (1 - beta1)
	buf = d.clone() if buf is None else buf * beta1 + d
	return p.double() - lr * buf, buf, ema
