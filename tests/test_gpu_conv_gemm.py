"""conv1d_umma_kernel (every forward conv, dgrad and decoder head of the bf16 and split-bf16 tiers) and wgrad_umma_kernel
(every weight gradient), launch by launch against the exact float64 references of tests/conv_oracle.py.

The operands are small integers (split tier: plus lo parts of integers x 2^lo_exp), so the fp32 accumulator is exact in
any order and almost every assertion is torch.equal: accumulator, bf16 hi / lo, statistics, folded BatchNorm-backward
sums, logits, argmax, weight gradients.  Don't-care regions of the inputs hold NaN (rows T_in.. T_rows, channels outside
each window), so a wrong descriptor, swizzle or coordinate turns into NaN, and every output buffer starts as NaN so a
store outside its box or a missing store is visible.  The assertions that carry a tolerance derive it next to them."""
import math

import pytest
import torch

import conv_oracle as CO

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
NAN = float('nan')


@pytest.fixture(scope = 'module')
def dev():
	return torch.device('cuda:0')


# ------------------------------------------------------------------------------------------ operands
class S:
	"""geometry of one operand pair: C_in, taps, dilation, pad_left; T_in (None: T_out), poisoned rows past T_in, channel
	window of the activation (ch_off, ld) and of the weights (w_ch_off, w_ld)"""

	def __init__(self, C_in, taps = 1, dil = 1, pad = 0, T_in = None, extra_rows = 3, ch_off = 0, ld = None, w_ch_off = 0, w_ld = None):
		self.C_in, self.taps, self.dil, self.pad, self.T_in, self.extra_rows = C_in, taps, dil, pad, T_in, extra_rows
		self.ch_off, self.ld = ch_off, (ch_off + C_in if ld is None else ld)
		self.w_ch_off, self.w_ld = w_ch_off, (w_ch_off + C_in if w_ld is None else w_ld)


def build_sources(dev, seed, B, T_out, C_out, specs, split = False, amax = 2, zero_frac = 0.5, lo_exp = -12, lens = None):
	"""-> (kernel sources, reference sources, granularity).  split: every pair becomes the three K segments of the split
	tier, a_hi.w_hi + a_hi.w_lo + a_lo.w_hi (engine._sources; no lo.lo term).  lens: activation rows t >= lens[b] are zero
	(structural zeros of a ragged batch)."""
	from convasr_b200 import ops
	g = torch.Generator().manual_seed(seed)
	kern, ref = [], []
	for sp in specs:
		T_in = sp.T_in or T_out
		a_hi, a_lo = CO.split_ints((B, T_in, sp.C_in), g, amax, 8, lo_exp, zero_frac)
		w_hi, w_lo = CO.split_ints((sp.taps, C_out, sp.C_in), g, amax, 8, lo_exp, zero_frac)
		if lens is not None:
			keep = (torch.arange(T_in)[None, :, None] < torch.as_tensor(lens)[:, None, None])
			a_hi, a_lo = a_hi * keep, a_lo * keep

		def place_a(v):
			t = torch.full((B, T_in + sp.extra_rows, sp.ld), NAN)
			t[:, :T_in, sp.ch_off:sp.ch_off + sp.C_in] = v
			return t.to(dev)

		def place_w(v):
			t = torch.full((sp.taps, C_out, sp.w_ld), NAN)
			t[:, :, sp.w_ch_off:sp.w_ch_off + sp.C_in] = v
			return t.to(dev)

		pairs = [(a_hi, w_hi)] + ([(a_hi, w_lo), (a_lo, w_hi)] if split else [])
		for a, w in pairs:
			A, W = place_a(a), place_w(w)
			ref.append(CO.Src(A, W, sp.C_in, sp.taps, sp.dil, sp.pad, T_in, sp.ch_off, sp.w_ch_off))
			kern.append(ops.Source(CO.to_bf16_exact(A), CO.to_bf16_exact(W), sp.C_in, sp.taps, sp.dil, sp.pad, T_in = T_in, ch_off = sp.ch_off, w_ch_off = sp.w_ch_off))
	gran = 2.0 ** lo_exp if split else 1.0
	return kern, ref, gran


def exact_acc(ref, B, T_out, gran, what):
	acc = CO.conv_acc64(ref, B, T_out)
	CO.assert_exact(CO.conv_bound(ref, B, T_out), gran, what)
	assert float(acc.abs().max()) > 0, f'{what}: degenerate data'
	return acc


def int_bias(C, seed, scale = 3):
	g = torch.Generator().manual_seed(seed)
	return torch.randint(-scale, scale + 1, (C, ), generator = g).to(torch.float32)


def assert_nan_outside(out, T_out, C_out, what):
	assert bool(out[:, T_out:].isnan().all()), f'{what}: a store landed in rows >= T_out'
	assert bool(out[:, :, C_out:].isnan().all()), f'{what}: a store landed in channels >= C_out'


def run_act(dev, what, kern, B, T_out, C_out, out_rows = 5, out_ld = None, want_lo = False, want_stats = False, **kw):
	from convasr_b200 import ops
	ld = out_ld or C_out + 8
	hi = torch.full((B, T_out + out_rows, ld), NAN, dtype = BF16, device = dev)
	lo = torch.full_like(hi, NAN) if want_lo else None
	st = torch.full((2, C_out), NAN, dtype = torch.float64, device = dev) if want_stats else None
	ops.conv1d_fused(kern, B, T_out, C_out, out_hi = hi, out_lo = lo, stats = st, **kw)
	torch.cuda.synchronize()
	assert_nan_outside(hi, T_out, C_out, what)
	if lo is not None:
		assert_nan_outside(lo, T_out, C_out, what + ' lo')
	return hi[:, :T_out, :C_out], None if lo is None else lo[:, :T_out, :C_out], st


def check_act_case(dev, what, seed, B, T_out, C_out, specs, split = False, act = (0, 0.0, 0.0), bias = True, xlen = None, stats = False,
				   block_n = 0, skip = None, lens = None, lo_exp = -12, amax = 2, zero_frac = 0.5):
	kern, ref, gran = build_sources(dev, seed, B, T_out, C_out, specs, split = split, lo_exp = lo_exp, amax = amax, zero_frac = zero_frac, lens = lens)
	acc = exact_acc(ref, B, T_out, gran, what)
	b = int_bias(C_out, seed).to(dev) if bias else None
	xl = None if xlen is None else torch.tensor(xlen, dtype = torch.float32).to(dev)
	sk = None if skip is None else (torch.tensor(skip[0], dtype = torch.float32).to(dev), skip[1], skip[2])
	hi, lo, st = run_act(dev, what, kern, B, T_out, C_out, want_lo = split, want_stats = stats, bias = b, act = act[0], act_a = act[1],
						 act_b = act[2], xlen = xl, block_n = block_n, skip = sk)
	want_hi, want_lo = CO.act_bf16_ref(acc, C_out, b, *act, xlen = xl, want_lo = split)
	assert torch.equal(hi, want_hi), f'{what}: hi differs at {(hi != want_hi).nonzero()[:5].tolist()}'
	if split:
		assert torch.equal(lo, want_lo), f'{what}: lo differs at {(lo != want_lo).nonzero()[:5].tolist()}'
	if stats:
		x = hi.float() if lo is None else hi.float() + lo.float()
		# the kernel sums 32 rows per fp32 partial: exact while 32 max x^2 stays below 2^24 (granularity^2)
		g2 = gran * gran if split else 1.0
		CO.assert_exact(32 * x.double() ** 2, g2, what + ' stats')
		assert torch.equal(st, CO.stats_ref(hi, lo)), f'{what}: stats {st} != {CO.stats_ref(hi, lo)}'
	return hi, lo, acc


# ------------------------------------------------------------------------------------------ canary
def test_canary_single_tile_is_exact(dev):
	"""one 128 x 32 tile, K = 64: the premise of every exact assertion below (tcgen05 kind::f16 accumulates such data
	exactly) -- if this fails, nothing else here means anything"""
	from convasr_b200 import _lib
	kern, ref, _ = build_sources(dev, 1, 1, 128, 32, [S(64)], zero_frac = 0.0)
	acc = exact_acc(ref, 1, 128, 1.0, 'canary')
	logits = torch.full((1, 32, 128), NAN, device = dev)
	from convasr_b200 import ops
	ops.conv1d_fused(kern, 1, 128, 32, logits = logits, epilogue = _lib.EPI_LOGITS_F32, block_n = 32)
	torch.cuda.synchronize()
	assert torch.equal(logits.double(), acc.permute(0, 2, 1))


# ------------------------------------------------------------------------------------------ ACT_BF16 forward / dgrad
ACT_CASES = {
	# T_out edges, one k-step (C_in 64, k 1)
	't1': dict(B = 2, T_out = 1, C_out = 32, specs = [S(64)], act = (1, 0.0, 0.0)),
	't127': dict(B = 2, T_out = 127, C_out = 96, specs = [S(64, 3, 1, 1)], act = (2, -4.0, 5.0)),
	't128': dict(B = 2, T_out = 128, C_out = 96, specs = [S(128, 5, 1, 2)], act = (3, 0.25, 0.0)),
	't129': dict(B = 3, T_out = 129, C_out = 32, specs = [S(64, 11, 1, 5)], act = (1, 0.0, 0.0), stats = True),
	't257_c1024': dict(B = 1, T_out = 257, C_out = 1024, specs = [S(64, 3, 1, 1)], stats = True),
	# hundreds of k-steps: C_in 1024, k 29, dilation 2
	'k29_d2_c1024': dict(B = 2, T_out = 150, C_out = 96, specs = [S(1024, 29, 2, 28)], act = (2, 0.0, 20.0), zero_frac = 0.8, amax = 1),
	# partial last N tile (640 = 3 x 224 in the auto pick) with stats and the implied xlen skip
	'c640_xlen_stats': dict(B = 3, T_out = 300, C_out = 640, specs = [S(128, 3, 1, 1)], act = (1, 0.0, 0.0), xlen = [1.0, 0.5, 0.1], stats = True),
	# persistent schedule: 8 utterances x 8 M tiles x 8 N tiles = 512 tiles on 148 SMs wrap the 4-stage smem ring and both
	# TMEM accumulator stages many times
	'wrap_schedule': dict(B = 8, T_out = 1000, C_out = 1024, specs = [S(128, 3, 1, 1)], block_n = 128, act = (1, 0.0, 0.0)),
	# split tier: three K segments per operand pair, out_lo
	'split_relu': dict(B = 2, T_out = 257, C_out = 96, specs = [S(128, 3, 1, 1)], split = True, act = (1, 0.0, 0.0)),
	'split_hardtanh_t1': dict(B = 3, T_out = 1, C_out = 64, specs = [S(64, 5, 1, 2)], split = True, act = (2, -3.0, 4.0)),
	'split_leaky_c640': dict(B = 2, T_out = 129, C_out = 640, specs = [S(64, 1)], split = True, act = (3, 0.125, 0.0), xlen = [0.7, 1.0]),
	# split tier statistics: lo parts of granularity 2^-4 keep 32 x^2 exact in fp32
	'split_stats': dict(B = 2, T_out = 200, C_out = 64, specs = [S(64, 1)], split = True, stats = True, lo_exp = -4, amax = 2, zero_frac = 0.6,
						bias = False, xlen = [1.0, 0.3]),
	# 18 K segments: mixed taps, dilation, pad_left (negative, 0, > T_in), T_in != T_out, channel windows, poisoned rows
	'18_sources': dict(B = 2, T_out = 140, C_out = 96, act = (3, 0.5, 0.0), zero_frac = 0.85, amax = 1, specs = [
		S(64, 1, 1, 0), S(64, 3, 1, 1, T_in = 100), S(128, 5, 2, 4, ch_off = 64, ld = 256), S(64, 2, 1, -3, T_in = 150),
		S(64, 7, 3, 9, w_ch_off = 64, w_ld = 192), S(64, 1, 1, 145), S(64, 4, 1, -200, T_in = 300), S(64, 1, 1, 0, T_in = 7),
		S(64, 11, 1, 5, ch_off = 128, ld = 192, w_ch_off = 128, w_ld = 256), S(64, 2, 5, 0), S(192, 1, 1, 0), S(64, 3, 1, 2, T_in = 139),
		S(64, 9, 1, 150, T_in = 160), S(64, 1, 1, -1), S(64, 29, 2, 28), S(128, 3, 1, 1, ch_off = 0, ld = 192), S(64, 1, 1, 0, T_in = 141),
		S(64, 6, 1, 3, extra_rows = 60)]),
	# ragged: xlen 0.0 at b = 0 and b = B-1, one 1-frame utterance, exactly 128 and 256 frames, 1.0
	'ragged_xlen': dict(B = 6, T_out = 512, C_out = 64, specs = [S(64, 3, 1, 1)], act = (2, -2.0, 2.0), xlen = [0.0, 1 / 512, 0.25, 0.5, 1.0, 0.0],
						stats = True),
	'ragged_xlen_split': dict(B = 6, T_out = 512, C_out = 32, specs = [S(64, 1)], split = True, xlen = [0.0, 1 / 512, 0.25, 0.5, 1.0, 0.0]),
}


@pytest.mark.parametrize('name', list(ACT_CASES))
def test_act_bf16_epilogue_is_exact(dev, name):
	kw = dict(ACT_CASES[name])
	check_act_case(dev, name, 100 + list(ACT_CASES).index(name), **kw)


def test_explicit_skip_with_margin_on_structural_zeros(dev):
	"""skip = (frac, skip_T, margin) as the training step passes it: (xlen, T of the conv input, the conv's padding).  The
	input is zero from ceil(frac * skip_T); a conv padded by `margin` on the left (7 taps, pad_left 3 = margin, no bias)
	is then non-zero up to row ceil(frac * skip_T) + margin - 1 and zero from the next row on, exactly where the contract
	puts the structural zeros.  skip_T = 700 differs from T_out = 680, and the fractions put a 128-row tile boundary
	inside the margin band (0.18: rows 127..129, 0.365: rows 256..258) and between ceil(frac * T_out) + margin and
	ceil(frac * skip_T) + margin, so a launch that drops the margin or measures the lengths on T_out skips live tiles
	and stores zeros over non-zero rows."""
	B, skip_T, T_out, margin = 4, 700, 680, 3
	frac = [0.18, 0.365, 1.0, 0.0]
	lens = CO.frac_lengths(torch.tensor(frac), skip_T).tolist()
	live = lambda T, m: [min(T_out, l + m) for l in CO.frac_lengths(torch.tensor(frac), T).tolist()]
	tiles = lambda rows: [(r + 127) // 128 for r in rows]
	assert tiles(live(skip_T, margin)) != tiles(live(skip_T, 0)), 'no tile boundary inside the margin band'
	assert tiles(live(skip_T, margin)) != tiles(live(T_out, margin)), 'skip_T and T_out give the same tiles'
	for split in (False, True):
		_, _, acc = check_act_case(dev, f'skip split={split}', 7, B, T_out, 64, [S(64, 2 * margin + 1, 1, margin, T_in = skip_T)], split = split,
								   bias = False, skip = (frac, skip_T, margin), lens = lens)
		for b in range(B):
			end = lens[b] + margin
			if end < T_out:
				assert float(acc[b, end:].abs().max()) == 0, 'data must be zero where the contract puts structural zeros'
			if 0 < lens[b] and end <= T_out:
				assert float(acc[b, end - 1].abs().max()) > 0, 'the last row of the margin band must be non-zero'


def test_every_block_n_gives_the_same_exact_result(dev):
	"""C_out 640: every legal N tile (multiples of 32 up to 256, partial last tiles) and the automatic pick"""
	B, T_out, C_out = 2, 257, 640
	kern, ref, _ = build_sources(dev, 3, B, T_out, C_out, [S(128, 3, 1, 1)])
	acc = exact_acc(ref, B, T_out, 1.0, 'block_n')
	b = int_bias(C_out, 3).to(dev)
	want, _ = CO.act_bf16_ref(acc, C_out, b, 1)
	for bn in [0] + list(range(32, 257, 32)):
		hi, _, _ = run_act(dev, f'block_n={bn}', kern, B, T_out, C_out, bias = b, act = 1, block_n = bn)
		assert torch.equal(hi, want), f'block_n={bn}'


# ------------------------------------------------------------------------------------------ fp32 logits epilogues
def test_logits_f32_every_block_n_with_activation(dev):
	"""LOGITS_F32 stores fp32 act(acc + bias) in [B, C, T]: C = 200 (not a multiple of 16), every multiple of 16"""
	from convasr_b200 import _lib, ops
	B, T_out, C = 2, 129, 200
	kern, ref, _ = build_sources(dev, 4, B, T_out, C, [S(64, 3, 1, 1), S(64, 2, 2, 0, T_in = 100)])
	acc = exact_acc(ref, B, T_out, 1.0, 'logits_f32')
	b = int_bias(C, 4).to(dev) * 0.5
	want = CO.act_ref(CO.logits_ref(acc, C, b), 3, 0.25).permute(0, 2, 1)
	for bn in [0] + list(range(16, 257, 16)):
		out = torch.full((B, C, T_out), NAN, device = dev)
		ops.conv1d_fused(kern, B, T_out, C, bias = b, logits = out, epilogue = _lib.EPI_LOGITS_F32, act = _lib.ACT_LEAKY_RELU, act_a = 0.25, block_n = bn)
		torch.cuda.synchronize()
		assert torch.equal(out, want), f'block_n={bn}'


def lse_tolerance_expf(C, lse):
	"""LOGSOFTMAX: lse = vmax + logf(sum expf(x - vmax)).  expf is within 2 ulp (CUDA programming guide, non-fast-math),
	logf within 1 ulp; each term carries a relative error <= 2 * 2^-23, the fp32 sum of C terms (C - 1) * 2^-24, so the
	sum S >= 1 is off by a relative (4 + C) * 2^-24 and log S by that much absolutely; logf adds 2^-23 |log S|, the two
	final additions 2^-24 |lse| and 2^-24 |log_prob| each."""
	return (4 + C) * 2.0 ** -24 + 2.0 ** -23 * math.log(C + 1) + 2.0 ** -24 * 2 * lse.abs() + 2.0 ** -23


def lse_tolerance_fast_expf(C, lse):
	"""LOGITS_ROWS: __expf(x) is within 2 + floor(1.173 |x|) ulp (CUDA programming guide).  For x <= 0 the absolute error of
	a term e^x is <= 2^-23 (2 + 1.173 |x|) e^x <= 2^-23 (2 e^x + 0.44): summed over C terms and divided by S >= 1, a
	relative 2^-23 (2 + 0.44 C).  Each of the ceil(C / 32) rescales of the running sum by __expf(m_old - m_new) adds at
	most 2.5 * 2^-23 relative, the fp32 sum C * 2^-24; logf and the final addition as for LOGSOFTMAX."""
	rel = 2.0 ** -23 * (2 + 0.44 * C) + 2.5 * 2.0 ** -23 * math.ceil(C / 32) + C * 2.0 ** -24
	return rel + 2.0 ** -23 * math.log(C + 1) + 2.0 ** -24 * 2 * lse.abs() + 2.0 ** -23


@pytest.mark.parametrize('C', [1, 29, 38, 256])
def test_logsoftmax_epilogue(dev, C):
	from convasr_b200 import _lib, ops
	B, T_out = 2, 257
	kern, ref, _ = build_sources(dev, 5 + C, B, T_out, C, [S(128, 3, 1, 1)])
	acc = exact_acc(ref, B, T_out, 1.0, f'logsoftmax C={C}')
	b = int_bias(C, C).to(dev)
	logits = torch.full((B, C, T_out), NAN, device = dev)
	lp = torch.full_like(logits, NAN)
	am = torch.full((B, T_out), -1, dtype = torch.int32, device = dev)
	ops.conv1d_fused(kern, B, T_out, C, bias = b, logits = logits, log_probs = lp, argmax = am, epilogue = _lib.EPI_LOGSOFTMAX)
	torch.cuda.synchronize()
	x = CO.logits_ref(acc, C, b)
	assert torch.equal(logits, x.permute(0, 2, 1))
	assert torch.equal(am.long(), CO.argmax_lowest(x))
	want, lse = CO.logsoftmax_ref(x)
	err = (lp.double() - want.permute(0, 2, 1)).abs()
	assert bool((err <= lse_tolerance_expf(C, lse)[:, None, :]).all()), float(err.max())


def run_logits_rows(dev, kern, B, T_out, C, bias, block_n = 0, ld = None):
	from convasr_b200 import _lib, ops
	ld = ld or (C + 3) // 4 * 4 + 8
	logits = torch.full((B, T_out, ld), NAN, device = dev)
	lse = torch.full((B, T_out), NAN, device = dev)
	am = torch.full((B, T_out), -1, dtype = torch.int32, device = dev)
	ops.conv1d_fused(kern, B, T_out, C, bias = bias, logits = logits, log_probs = lse, argmax = am, epilogue = _lib.EPI_LOGITS_ROWS, block_n = block_n)
	torch.cuda.synchronize()
	assert bool(logits[:, :, C:].isnan().all()), 'a store landed in columns >= C'
	return logits[:, :, :C], lse, am


@pytest.mark.parametrize('C', [1000, 5000])
def test_logits_rows_online_softmax(dev, C):
	from convasr_b200 import ops
	B, T_out = 2, 300
	kern, ref, _ = build_sources(dev, C, B, T_out, C, [S(128, 1)])
	acc = exact_acc(ref, B, T_out, 1.0, f'logits_rows C={C}')
	b = int_bias(C, C + 1).to(dev)
	x = CO.logits_ref(acc, C, b)
	want_lp, want_lse = CO.logsoftmax_ref(x)
	tol = lse_tolerance_fast_expf(C, want_lse)
	for bn in (0, 32, 224, 256):
		logits, lse, am = run_logits_rows(dev, kern, B, T_out, C, b, block_n = bn)
		assert torch.equal(logits, x), f'block_n={bn}'
		assert torch.equal(am.long(), CO.argmax_lowest(x)), f'block_n={bn}'
		assert bool(((lse.double() - want_lse).abs() <= tol).all()), (bn, float((lse.double() - want_lse).abs().max()))
	# the public head: logits and argmax exact, log_probs = logits - lse in fp32 (one more rounding: 2^-24 |log_prob|)
	lg, lp, am = ops.large_vocab_head(kern, B, T_out, C, b)
	torch.cuda.synchronize()
	assert torch.equal(lg.permute(0, 2, 1), x) and torch.equal(am.long(), CO.argmax_lowest(x))
	err = (lp.permute(0, 2, 1).double() - want_lp).abs()
	assert bool((err <= tol[:, :, None] + 2.0 ** -24 * want_lp.abs()).all()), float(err.max())


def tie_sources(dev, B, T_out, C, i, j, seed):
	"""weights with rows i and j identical and bias[i] = bias[j] far above the rest: classes i and j tie exactly at the max
	in every frame"""
	from convasr_b200 import ops
	g = torch.Generator().manual_seed(seed)
	a = CO.ints((B, T_out, 64), -2, 2, g)
	w = CO.ints((1, C, 64), -2, 2, g)
	w[0, j] = w[0, i]
	bias = CO.ints((C, ), -3, 3, g)
	bias[i] = bias[j] = 1000.0
	return [ops.Source(a.to(BF16).to(dev), w.to(BF16).to(dev), 64, 1, 1, 0)], bias.to(dev)


def test_argmax_ties_go_to_the_lowest_class(dev):
	from convasr_b200 import _lib, ops
	B, T_out = 2, 130
	# LOGITS_ROWS, block_n 128: inside a 32-column chunk, across chunks, across N tiles, first against last class
	C = 1000
	for i, j in ((5, 17), (31, 32), (127, 128), (0, C - 1)):
		kern, bias = tie_sources(dev, B, T_out, C, i, j, i * 7 + j)
		_, _, am = run_logits_rows(dev, kern, B, T_out, C, bias, block_n = 128)
		assert bool((am == i).all()), ('logits_rows', i, j, am.unique().tolist())
	# LOGSOFTMAX: one N tile, 16-column loads
	C = 256
	for i, j in ((5, 17), (15, 16), (31, 32), (0, C - 1)):
		kern, bias = tie_sources(dev, B, T_out, C, i, j, i * 5 + j)
		am = torch.full((B, T_out), -1, dtype = torch.int32, device = dev)
		ops.conv1d_fused(kern, B, T_out, C, bias = bias, argmax = am, epilogue = _lib.EPI_LOGSOFTMAX)
		torch.cuda.synchronize()
		assert bool((am == i).all()), ('logsoftmax', i, j, am.unique().tolist())


# ------------------------------------------------------------------------------------------ folded BatchNorm-backward sums
@pytest.mark.parametrize('act', [(0, 0.0, 0.0), (1, 0.0, 0.0), (2, -1.0, 1.0), (3, 0.25, 0.0)])
def test_bn_backward_sums_folded_into_the_epilogue(dev, act):
	"""bnr_partials summed over the replicas equal the float64 sum(dz) and sum(dz y): y integer, scale a power of two and
	shift a multiple of 1/16, so z = fmaf(y, scale, shift), the gate and every fp32 partial are exact"""
	from convasr_b200 import _lib, ops
	B, T, C_out, C, ld = 3, 300, 64, 40, 72
	g = torch.Generator().manual_seed(30 + act[0])
	kern, ref, _ = build_sources(dev, 30 + act[0], B, T, C_out, [S(64, 3, 1, 1)])
	acc = exact_acc(ref, B, T, 1.0, 'bnr')
	y = torch.full((B, T + 4, ld), NAN, dtype = BF16)
	y[:, :T, :C_out] = CO.ints((B, T, C_out), -6, 6, g).to(BF16)
	y = y.to(dev)
	ss = torch.zeros(4, C)
	ss[0] = torch.tensor([-2.0, -0.5, 0.5, 1.0, 2.0, 0.25])[torch.randint(0, 6, (C, ), generator = g)]
	ss[1] = torch.randint(-24, 25, (C, ), generator = g) / 16.0
	ss = ss.to(dev)
	xlen = torch.tensor([1.0, 0.45, 0.01]).to(dev)
	partials = torch.full((_lib.BN_SUM_REPLICAS, 2, C), NAN, dtype = torch.float64, device = dev)
	hi = torch.full((B, T + 4, ld), NAN, dtype = BF16, device = dev)
	ops.conv1d_fused(kern, B, T, C_out, out_hi = hi, bn_reduce = (y, ss, C, act[0], act[1], act[2], xlen, partials))
	torch.cuda.synchronize()
	want_hi, _ = CO.act_bf16_ref(acc, C_out)
	assert torch.equal(hi[:, :T, :C_out], want_hi)
	assert_nan_outside(hi, T, C_out, 'bnr')
	want = CO.bnr_ref(hi[:, :T], y[:, :T], ss, C, act[0], act[1], act[2], xlen)
	g_abs = hi[:, :T, :C].double().abs()
	CO.assert_exact((g_abs * (1 + y[:, :T, :C].double().abs())).sum(dim = (0, 1)), 0.25, 'bnr sums')  # dz, dz * y: multiples of 1/4
	assert torch.equal(partials.sum(dim = 0), want), (partials.sum(dim = 0) - want).abs().max()


# ------------------------------------------------------------------------------------------ precision format
def test_conv_accumulator_precision_on_random_normal_data(dev):
	"""random-normal bf16 operands, raw accumulator through LOGITS_F32 (fp32 acc + bias, no bf16 rounding).  The tensor core
	adds K / 16 partial products of 16 into the fp32 accumulator.  Tensor-core fp32 accumulation truncates instead of
	rounding to nearest (Fasi, Higham, Mikaitis, Pranesh, PeerJ CS 2021, for earlier NVIDIA tensor cores), so each addition
	loses up to 2^-23 of the running magnitude <= sum |a w|; with the 16-term partials no worse than 16 such steps the error
	is <= (K / 16 + 16) 2^-23 sum |a w| <= 2^-15 sum |a w| for K = 3072 (208 < 256 steps), plus 2^-24 |y| for the bias add:
	that per-element bound is derived.  The 1e-5 limit on the relative Frobenius error is a measured limit, not a derived
	one: it measured 2.35e-6 on an NVIDIA B200 (1000 W power limit), and since it scales as 2^(23 - p) for an accumulator
	with a p-bit significand, the limit still fails any accumulator of 20 bits or fewer."""
	from convasr_b200 import _lib, ops
	B, T_out, C, C_in, k = 2, 200, 96, 1024, 3
	g = torch.Generator().manual_seed(40)
	a = torch.randn(B, T_out, C_in, generator = g).to(BF16).to(dev)
	w = (torch.randn(k, C, C_in, generator = g) / (C_in * k) ** 0.5).to(BF16).to(dev)
	b = torch.randn(C, generator = g).to(dev)
	out = torch.full((B, C, T_out), NAN, device = dev)
	ops.conv1d_fused([ops.Source(a, w, C_in, k, 1, 1)], B, T_out, C, bias = b, logits = out, epilogue = _lib.EPI_LOGITS_F32, block_n = 96)
	torch.cuda.synchronize()
	src = [CO.Src(a.double(), w.double(), C_in, k, 1, 1)]
	want = (CO.conv_acc64(src, B, T_out) + b.double()).permute(0, 2, 1)
	absum = CO.conv_bound(src, B, T_out).permute(0, 2, 1)
	err = (out.double() - want).abs()
	frob = float((out.double() - want).norm() / want.norm())
	print(f'\nconv accumulator, K = {C_in * k}: relative Frobenius error {frob:.3e}, max err / sum|a w| {float((err / absum).max()):.3e}')
	assert frob <= 1e-5
	assert bool((err <= 2.0 ** -15 * absum + 2.0 ** -24 * want.abs()).all()), float((err / absum).max())


# ------------------------------------------------------------------------------------------ weight gradient
WGRAD_CASES = {
	# M_total, N_total, taps, dilation, pad_left, B, a_T, b_T
	'm40_n1_t64': (40, 1, 1, 1, 0, 3, 64, 64),
	'm128_n3_k11_t129': (128, 3, 11, 1, 5, 3, 129, 129),
	'm129_n5_k29_d2_t127': (129, 5, 29, 2, 28, 2, 127, 127),
	'm320_n64_aT_ne_bT': (320, 64, 1, 1, 0, 3, 130, 100),
	'm64_n190_swapped': (64, 190, 11, -1, -5, 3, 191, 191),
	'm40_n257_k3': (40, 257, 3, 1, 1, 4, 65, 70),
	'm128_n640_t191': (128, 640, 1, 1, 0, 2, 191, 191),
	# 29 taps x 3 M tiles x 3 N tiles = 261 items: the persistent schedule wraps both rings
	'm320_n640_k29_wrap': (320, 640, 29, 1, 14, 2, 100, 100),
}


def wgrad_operands(dev, seed, M, N, B, a_T, b_T, lens = None):
	g = torch.Generator().manual_seed(seed)
	a_ld, b_ld = (M + 63) // 64 * 64, (N + 63) // 64 * 64
	a = torch.full((B, a_T + 5, a_ld), NAN)
	a[:, :a_T, :M] = CO.ints((B, a_T, M), -2, 2, g, 0.5)
	if lens is not None:
		a[:, :a_T, :M] *= (torch.arange(a_T)[None, :, None] < torch.as_tensor(lens)[:, None, None])
	bx = torch.full((B, b_T + 7, b_ld), NAN)
	bx[:, :b_T, :N] = CO.ints((B, b_T, N), -2, 2, g, 0.5)
	return CO.to_bf16_exact(a.to(dev)), CO.to_bf16_exact(bx.to(dev))


@pytest.mark.parametrize('name', list(WGRAD_CASES))
def test_wgrad_is_exact_for_every_split(dev, name):
	from convasr_b200 import ops
	M, N, taps, dil, pad, B, a_T, b_T = WGRAD_CASES[name]
	a, bx = wgrad_operands(dev, 200 + list(WGRAD_CASES).index(name), M, N, B, a_T, b_T)
	want = CO.wgrad64(a, a_T, M, bx, b_T, N, taps, dil, pad)
	CO.assert_exact(CO.wgrad_bound(a, a_T, M, bx, b_T, N, taps, dil, pad), 1.0, name)
	assert float(want.abs().max()) > 0
	for ns in sorted({0, 1, 2, 3, B} & set(range(B + 1))):
		out = ops.conv1d_wgrad(a, a_T, M, bx, b_T, N, taps, dil, pad, n_splits = ns)
		torch.cuda.synchronize()
		assert torch.equal(out[:, :, :N].double(), want), (name, ns, (out[:, :, :N].double() - want).abs().max())
	# accumulate_into: onto a prefilled integer tensor (padding columns NaN: never written)
	g = torch.Generator().manual_seed(9)
	ld = (N + 3) // 4 * 4
	pre = torch.full((taps, M, ld), NAN)
	pre[:, :, :N] = CO.ints((taps, M, N), -50, 50, g)
	for ns in (1, B):
		out = pre.clone().to(dev)
		ops.conv1d_wgrad(a, a_T, M, bx, b_T, N, taps, dil, pad, n_splits = ns, out = out)
		torch.cuda.synchronize()
		assert torch.equal(out[:, :, :N].double(), want + pre[:, :, :N].double().to(dev)), (name, 'accumulate_into', ns)
		assert bool(out[:, :, N:].isnan().all())


@pytest.mark.parametrize('margin', [0, 5])
def test_wgrad_skip_on_structural_zeros(dev, margin):
	"""frames t >= ceil(frac * T) + margin are left out.  The M-side operand is non-zero up to frame ceil(frac * T) +
	margin - 1 and zero from there, exactly where the contract puts the structural zeros, so the result equals the full
	contraction exactly -- with xlen 0.0 at the first and the last utterance.  frac 0.42 gives 126 frames: with margin 5
	the live frames (131) cross the 64-frame chunk boundary at 128, so a launch that drops the margin leaves out frames
	that carry products."""
	from convasr_b200 import ops
	B, T, M, N = 4, 300, 128, 96
	frac = torch.tensor([0.0, 0.42, 1.0, 0.0])
	lens = CO.frac_lengths(frac, T)
	live = (lens + margin).clamp(max = T).tolist()
	if margin:
		assert [(r + 63) // 64 for r in live] != [(r + 63) // 64 for r in lens.tolist()], 'no chunk boundary inside the margin band'
	for orient in ('dy_on_m', 'swapped'):
		a, bx = wgrad_operands(dev, 50 + margin, M, N, B, T, T, lens = live)
		dil, pad = (1, 5) if orient == 'dy_on_m' else (-1, -5)
		want = CO.wgrad64(a, T, M, bx, T, N, 11, dil, pad)
		if margin:
			assert not torch.equal(want, CO.wgrad64(a, T, M, bx, T, N, 11, dil, pad, skip = (frac.to(dev), T, 0))), 'the margin frames must contribute'
		for ns in (0, 1, 2, B):
			out = ops.conv1d_wgrad(a, T, M, bx, T, N, 11, dil, pad, n_splits = ns, skip = (frac.to(dev), T, margin))
			torch.cuda.synchronize()
			assert torch.equal(out[:, :, :N].double(), want), (orient, ns)


def test_wgrad_precision_on_random_normal_data(dev):
	"""B T = 512 frames: each item accumulates 32 MMAs of K = 16 in fp32 and each split adds one fp32 reduction, so with
	truncating additions (see the conv case) the error is <= (512 / 16 + 16 + n_splits) 2^-23 sum |a b| < 2^-17 sum |a b|
	per element: that bound is derived.  The 1e-6 limit on the relative Frobenius error is a measured limit, not a derived
	one: on an NVIDIA B200 (1000 W power limit) it measured 4.8e-7 with one split and 2.3e-7 with two (32 accumulator
	additions per element, 6 times fewer than the 192 of the conv case)."""
	from convasr_b200 import ops
	B, T, M, N = 2, 256, 128, 64
	g = torch.Generator().manual_seed(60)
	a = torch.randn(B, T, M, generator = g).to(BF16).to(dev)
	bx = torch.randn(B, T, N, generator = g).to(BF16).to(dev)
	want = CO.wgrad64(a, T, M, bx, T, N, 3, 1, 1)
	absum = CO.wgrad_bound(a, T, M, bx, T, N, 3, 1, 1)
	for ns in (1, 2):
		out = ops.conv1d_wgrad(a, T, M, bx, T, N, 3, 1, 1, n_splits = ns)[:, :, :N].double()
		torch.cuda.synchronize()
		frob = float((out - want).norm() / want.norm())
		print(f'\nwgrad, n_splits = {ns}: relative Frobenius error {frob:.3e}')
		assert frob <= 1e-6
		assert bool(((out - want).abs() <= 2.0 ** -17 * absum).all())


# ------------------------------------------------------------------------------------------ refusals
def refused(fn, match):
	"""a refused call returns nonzero before any launch, with cab_last_error naming the argument"""
	from convasr_b200 import _lib
	before = _lib.launch_count()
	with pytest.raises(RuntimeError, match = match):
		fn()
	torch.cuda.synchronize()
	assert _lib.launch_count() == before, match


def test_conv_refusals_launch_nothing(dev):
	from convasr_b200 import _lib, ops
	B, T = 2, 100
	a = torch.zeros(B, T, 64, dtype = BF16, device = dev)
	w = torch.zeros(1, 64, 64, dtype = BF16, device = dev)
	src = [ops.Source(a, w, 64, 1, 1, 0)]
	out = torch.empty(B, T, 64, dtype = BF16, device = dev)
	ops.conv1d_fused(src, B, T, 64, out_hi = out)  # the base call is valid
	refused(lambda: ops.conv1d_fused(src, B, T, 40, out_hi = out), 'C_out=40 must be a multiple of 32')
	refused(lambda: ops.conv1d_fused(src, B, T, 64, out_hi = out, block_n = 48), 'block_n=48 must be a multiple of 32')
	refused(lambda: ops.conv1d_fused(src, B, T, 64, out_hi = out, block_n = 24), r'block_n=24 must be a multiple of 16')
	refused(lambda: ops.conv1d_fused(src, B, T, 64, out_hi = out, block_n = 288), r'block_n=288 must be a multiple of 16 in \[16,256\]')
	lg = torch.empty(B, 300, T, device = dev)
	refused(lambda: ops.conv1d_fused([ops.Source(a, torch.zeros(1, 300, 64, dtype = BF16, device = dev), 64, 1, 1, 0)], B, T, 300, logits = lg,
									 epilogue = _lib.EPI_LOGSOFTMAX, block_n = 256), 'at most 256 classes')
	refused(lambda: ops.conv1d_fused(src, B, T, 38, logits = lg, epilogue = _lib.EPI_LOGSOFTMAX, block_n = 32), 'block_n=32 must cover all 38 classes')
	rows = torch.empty(B, T, 64, device = dev)
	refused(lambda: ops.conv1d_fused(src, B, T, 64, logits = rows, epilogue = _lib.EPI_LOGITS_ROWS, act = _lib.ACT_RELU), 'applies no activation')
	refused(lambda: ops.conv1d_fused(src, B, T, 62, logits = torch.empty(B, T, 62, device = dev), epilogue = _lib.EPI_LOGITS_ROWS), 'multiple of 4 floats')
	refused(lambda: ops.conv1d_fused([ops.Source(a, w, 32, 1, 1, 0)], B, T, 64, out_hi = out), 'C_in=32 must be a multiple of 64')
	refused(lambda: ops.conv1d_fused([], B, T, 64, out_hi = out), r'n_sources=0 out of \[1,18\]')
	refused(lambda: ops.conv1d_fused(src * 19, B, T, 64, out_hi = out), r'n_sources=19 out of \[1,18\]')
	flat = torch.zeros(B * T * 64 + 1, dtype = BF16, device = dev)
	shifted = flat[1:].view(B, T, 64)  # contiguous, 2 bytes off a 16-byte boundary
	refused(lambda: ops.conv1d_fused([ops.Source(shifted, w, 64, 1, 1, 0)], B, T, 64, out_hi = out), 'pointers must be 16-byte aligned')
	refused(lambda: ops.conv1d_fused(src, B, T, 64, out_hi = shifted), 'out_hi must be 16-byte aligned')
	refused(lambda: ops.conv1d_fused(src, B, T, 64, out_hi = out[:, :T - 1].contiguous()), f'out_T_rows={T - 1} < T_out={T}')


def test_wgrad_refusals_launch_nothing(dev):
	from convasr_b200 import _lib, ops
	B, T = 2, 100
	a = torch.zeros(B, T, 64, dtype = BF16, device = dev)
	ops.conv1d_wgrad(a, T, 64, a, T, 64, 1, 1, 0, n_splits = 2)  # valid
	refused(lambda: ops.conv1d_wgrad(a, T, 64, a, T, 64, 1, 1, 0, n_splits = 3), 'n_splits=3 > B=2')
	odd = torch.zeros(B, T, 96, dtype = BF16, device = dev)
	refused(lambda: ops.conv1d_wgrad(odd, T, 96, a, T, 64, 1, 1, 0), 'multiples of 64')
	out = torch.zeros(1, 64, 8, device = dev)
	lib = _lib.load()
	refused(lambda: _lib.check(lib.cab_conv1d_wgrad(ops._p(a), T, T, 64, 64, ops._p(a), T, T, 64, 6, B, 1, 1, 0, ops._p(out), 6, 1, None, 0, 0, 0,
												  ops._stream()), 'cab_conv1d_wgrad'), 'out_ld=6 must be a multiple of 4')
