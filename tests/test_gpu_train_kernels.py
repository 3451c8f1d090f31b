"""Launch-level tests of the training-step kernels of csrc/train.cu and csrc/optim.cu against tests/train_oracle.py.

Where the data makes the arithmetic exact (train_oracle's module docstring) the comparison is `torch.equal`.  Where a
case cannot be exact (1 / n not a power of two, sums too long for 24 bits) the apply output is held to the bound
derived next to `_close_dy`; the case list asserts which geometries are exact.  Output buffers start as NaN, so a
missing store shows up; padded rows of the incoming gradient are NaN, because the kernels select them away and never
multiply them.  Channels [C, ld) of y and g only have to be finite (the apply pass multiplies them by zero
coefficients): they hold a large finite value."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

import conv_oracle as CO
import train_oracle as TO

BF16 = torch.bfloat16
ACTS = [(0, 0.0, 0.0), (1, 0.0, 0.0), (2, 0.0, 20.0), (3, 0.125, 0.0)]
POISON = 4096.0  # finite, exact in bf16
SEED, SALT = 0x1234_5678_9ABC, 5


def _dev():
	return torch.device('cuda:0')


def _p(t):
	return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _lib():
	from convasr_b200 import _lib
	return _lib.load()


def _stream():
	return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check(rc, what):
	from convasr_b200 import _lib
	_lib.check(rc, what)


def _nan(*shape, dtype = BF16):
	return torch.full(shape, float('nan'), dtype = dtype, device = _dev())


def _bf(x64):
	"""exact bf16 copy on the device"""
	return CO.to_bf16_exact(x64.float()).to(_dev())


# ------------------------------------------------------------------------------------------ data
def _data(R, C, ld, gen, split, big):
	"""y, g float64 [R, ld] (hi + lo in the split tier) and their bf16 parts.  `big`: a small value range so that the sums of
	2^20 rows stay exact"""
	lim_y, lim_g = (3, 2) if big else (12, 8)
	y_hi = TO.ints((R, ld), -lim_y, lim_y, gen) / 4
	g_hi = TO.ints((R, ld), -lim_g, lim_g, gen) / 2
	y_lo = TO.ints((R, ld), -3, 3, gen) / 64 if split else None
	g_lo = TO.ints((R, ld), -1, 1, gen) / 16 if split else None
	for t in (y_hi, g_hi):
		t[:, C:] = POISON
	for t in (y_lo, g_lo):
		if t is not None:
			t[:, C:] = 0
	return y_hi, y_lo, g_hi, g_lo


def _bn_data(R, C, ld, gen, split, big, act, a, b):
	y_hi, y_lo, g_hi, g_lo = _data(R, C, ld, gen, split, big)
	ss = TO.exact_ss(C, gen)
	if not big:  # z exactly on 0 (and on the hardtanh bounds) for some elements of every activation
		TO.plant_z(y_hi, ss, C, [0.0, a, b] if act == 2 else [0.0], gen)
	return y_hi, y_lo, g_hi, g_lo, ss


def _pois_rows(g, B, T, xlen):
	"""NaN on the rows the mask removes"""
	keep = TO.row_mask(B, T, xlen, g.device).reshape(-1, 1)
	return torch.where(keep, g, torch.full_like(g, float('nan')))


def _bf16_ulp(x):
	"""spacing of bf16 at |x| (at least the smallest normal spacing)"""
	a = x.abs().double().clamp(min = 2.0 ** -126)
	return torch.pow(2.0, torch.floor(torch.log2(a)) - 7)


def _close_dy(got, ref, terms, what):
	"""dy = fmaf(scale, dz, fmaf(k1, y, k0)) when the data is not exact: k0, k1 and m2 carry a few fp32 roundings (each
	<= 2^-24 relative) of terms whose magnitudes add up to `terms`, so the fp32 value is within 2^-20 * terms of the float64
	one; the bf16 store then adds at most one bf16 ulp (half an ulp of rounding, moved across a midpoint at most once)."""
	d = (got.double() - ref.double()).abs()
	lim = _bf16_ulp(ref) + 2.0 ** -20 * terms
	bad = ~(d <= lim)
	assert not bool(bad.any()), f'{what}: {int(bad.sum())} of {d.numel()} outside the bound (worst excess {float((d - lim)[bad].max())})'
	return float((got.float() != ref.float().to(BF16).float()).double().mean())  # share that differs from the rounded reference


# ------------------------------------------------------------------------------------------ BatchNorm geometry cases
# (name, ld, C, B, T, xlen fractions or None); B*T a power of two where the case must be exact
CASES = [
	('ld64', 64, 64, 8, 32, [1.0, 0.5, 0.25, 0.0, 1 / 32, 0.75, 0.125, 0.9]),
	('ld320', 320, 300, 4, 64, [1.0, 0.3, 0.5, 1 / 64]),
	('ld576', 576, 576, 2, 128, [0.5, 1.0]),
	('ld1024', 1024, 1000, 2, 64, [1.0, 0.75]),
	('ld2048', 2048, 2048, 1, 64, None),
	('C40_ld64', 64, 40, 4, 32, [1.0, 0.5, 0.0, 0.25]),
	('R1', 64, 64, 1, 1, None),
	('R_below_chunk', 320, 320, 1, 16, [0.5]),
	('T1', 64, 64, 64, 1, None),
	('T2', 64, 64, 32, 2, [1.0, 0.5] * 16),
	('T3', 320, 320, 16, 3, [1.0, 0.34, 0.0, 0.67] * 4),
	('chunk_plus1', 64, 64, 1, 3 * 128 + 1, None),
	('chunk_minus1', 64, 64, 1, 5 * 128 - 1, [0.5]),
	('chunk_boundary_xlen', 64, 64, 4, 512, [0.25, 0.5, 1.0, 0.75]),  # lengths 128, 256, 512, 384: chunk boundaries at 128 rows
]
EXACT = {'ld64', 'ld320', 'ld576', 'ld1024', 'ld2048', 'C40_ld64', 'R1', 'R_below_chunk', 'T1', 'T2', 'chunk_boundary_xlen'}


def _xlen(fr, B):
	return torch.tensor(fr[:B], dtype = torch.float32, device = _dev()) if fr is not None else None


def _combos(idx):
	"""(split, act, dropout, frozen) per geometry: every activation in both tiers, dropout and frozen rotating"""
	out = []
	for split in (False, True):
		for i, (act, a, b) in enumerate(ACTS):
			out.append((split, act, a, b, 0.5 if (i + idx + split) % 2 else 0.0, (i + idx) % 4 == 3))
	return out


def _bn_run(name, ld, C, B, T, fr, split, act, a, b, drop_p, frozen, gen, big = False, report = None):
	lib, dev = _lib(), _dev()
	R = B * T
	xlen = _xlen(fr, B)
	y_hi, y_lo, g_hi, g_lo, ss = _bn_data(R, C, ld, gen, split, big, act, a, b)
	y = y_hi + (y_lo if split else 0)
	g = g_hi + (g_lo if split else 0)
	keep = TO.dropout_keep(SEED, SALT, R, ld, drop_p).to(dev) if drop_p else None
	drop = (drop_p, keep) if drop_p else None
	y_d, g_d, ss_d = y.to(dev), _pois_rows(g.to(dev), B, T, xlen), ss.to(dev)
	yh, yl = _bf(y_hi), (_bf(y_lo) if split else None)
	gh = _pois_rows(_bf(g_hi).float(), B, T, xlen).to(BF16)
	gl = _pois_rows(_bf(g_lo).float(), B, T, xlen).to(BF16) if split else None
	ss32 = ss_d.float().contiguous()
	seed = torch.tensor([SEED], dtype = torch.int64, device = dev)
	tag = (name, 'split' if split else 'bf16', act, drop_p, frozen)

	# forward
	out, out_lo = _nan(R, ld), (_nan(R, ld) if split else None)
	_check(lib.cab_bn_act_mask_fwd(_p(yh), _p(yl), _p(ss32), B, T, C, ld, act, a, b, _p(xlen), _p(out), _p(out_lo), drop_p, _p(seed), SALT, _stream()), 'fwd')
	o_ref = TO.bn_fwd_ref(y_d, ss_d, B, T, C, act, a, b, xlen, drop)
	if split:
		hi, lo = TO.split_store(o_ref)
		assert torch.equal(out, hi) and torch.equal(out_lo, lo), tag
	else:
		assert torch.equal(out, o_ref.to(BF16)), tag

	# backward: reference, exact when the data allows it
	try:
		ref = TO.bn_bwd_ref(y_d, g_d.nan_to_num(0.0), ss_d, B, T, C, act, a, b, xlen, drop, frozen = frozen, check = True)
		exact = True
	except ValueError:
		ref = TO.bn_bwd_ref(y_d, g_d.nan_to_num(0.0), ss_d, B, T, C, act, a, b, xlen, drop, frozen = frozen)
		exact = False
	if name in EXACT and not big and not split:
		assert exact, f'{tag}: the case is meant to be exact'  # (split-tier lo parts are finer: some of those cases are not)
	sum_terms = torch.stack([ref['dz'].abs().sum(0), (ref['dz'] * y_d[:, :C]).abs().sum(0)])
	mean, istd, sc = ss_d[2, :C], ss_d[3, :C], ss_d[0, :C]
	inv_n = 0.0 if frozen else 1.0 / R
	m2_terms = istd * (sum_terms[1] + mean.abs() * sum_terms[0])
	# Bounds for data that is not exact.  The channel sums accumulate at most a few thousand terms in fp32 before they reach
	# the fp64 replicas (chunks per CTA x 4 rows + the lane reduction, or a row walker's rows per block): relative error
	# <= 4096 * 2^-24 = 2^-12 of the sum of |terms|.  dy inherits that through k0 / k1, plus a few fp32 roundings of every term.
	dy_terms = torch.zeros(R, ld, dtype = torch.float64, device = dev)
	dy_terms[:, :C] = 2.0 ** 8 * ((sc * m2_terms * inv_n * istd * (y_d[:, :C].abs() + mean.abs())).abs() + (sc * sum_terms[0] * inv_n).abs()) + (sc * ref['dz']).abs()

	def check_dy(dy, dy_lo, what):
		if split:
			got = dy.float() + dy_lo.float()
			if exact:
				hi, lo = TO.split_store(ref['dy'])
				assert torch.equal(dy, hi) and torch.equal(dy_lo, lo), (tag, what)
			else:
				# hi + lo keeps ~16 bits: the fp32 error bound plus 2^-16 relative
				d = (got.double() - ref['dy'].double()).abs()
				assert bool((d <= 2.0 ** -15 * ref['dy'].double().abs() + 2.0 ** -20 * dy_terms + 2.0 ** -126).all()), (tag, what)
		elif exact:
			assert torch.equal(dy, ref['dy'].to(BF16)), (tag, what)
		else:
			share = _close_dy(dy.float(), ref['dy'], dy_terms, str((tag, what)))
			if report is not None:
				report.append((tag, what, share))

	def check_sums(sums, what):
		want = ref['sums'].float()
		if exact:
			assert torch.equal(sums, want), (tag, what)
		else:
			lim = 2.0 ** -12 * torch.stack([sum_terms[0], m2_terms]) + 1e-30
			assert bool(((sums.double() - ref['sums']).abs() <= lim).all()), (tag, what)

	parts = torch.empty(TO.SUM_REPLICAS * 2 * C, dtype = torch.float64, device = dev)
	# streamed reduce + apply (partials given)
	# with partials: the streamed reduce + apply where the pitch is covered; without: the row walkers (bf16 tier only)
	for use_partials in ((True, False) if not split else (True, )):
		sums, dy, dy_lo = _nan(2, C, dtype = torch.float32), _nan(R, ld), (_nan(R, ld) if split else None)
		_check(lib.cab_bn_act_mask_bwd(_p(yh), _p(yl), _p(gh), _p(gl), _p(ss32), B, T, C, ld, act, a, b, _p(xlen), _p(sums), _p(dy), _p(dy_lo), drop_p, _p(seed), SALT,
										int(frozen), _p(parts) if use_partials else None, _stream()), 'bwd')
		what = 'streamed' if use_partials else 'row walker'
		check_sums(sums, what)
		check_dy(dy, dy_lo, what)
	# apply alone, partials planted unevenly over the 8 replicas (a reader that sums fewer replicas misses >= 1/128 of each)
	if TO.stream_geometry(R, ld, 4 if split else 2) is not None:
		w = torch.tensor([2.0 ** -(r + 1) for r in range(TO.SUM_REPLICAS - 1)] + [2.0 ** -(TO.SUM_REPLICAS - 1)], dtype = torch.float64, device = dev)
		planted = (w[:, None, None] * ref['raw'][None]).contiguous()
		assert torch.equal(planted.sum(0), ref['raw'])
		sums, dy, dy_lo = _nan(2, C, dtype = torch.float32), _nan(R, ld), (_nan(R, ld) if split else None)
		_check(lib.cab_bn_act_mask_bwd_apply(_p(yh), _p(yl), _p(gh), _p(gl), _p(ss32), B, T, C, ld, act, a, b, _p(xlen), _p(sums), _p(dy), _p(dy_lo), drop_p, _p(seed), SALT,
											int(frozen), _p(planted), _stream()), 'apply')
		check_sums(sums, 'apply')
		check_dy(dy, dy_lo, 'apply')
	return exact


@pytest.mark.parametrize('case', CASES, ids = [c[0] for c in CASES])
def test_bn_act_mask_kernels_exact(case):
	name, ld, C, B, T, fr = case
	idx = [c[0] for c in CASES].index(name)
	gen = torch.Generator().manual_seed(1000 + idx)
	geo = TO.stream_geometry(B * T, ld, 2)
	print(name, 'stream geometry (bwd, bf16):', geo)
	for split, act, a, b, drop_p, frozen in _combos(idx):
		_bn_run(name, ld, C, B, T, fr, split, act, a, b, drop_p, frozen, gen)


def test_bn_kernels_wrap_the_stage_ring():
	"""2^20 rows at ld = 64: more chunks than (resident-CTA bound) x stages x 3, in every mode and tier, so each CTA's ring
	wraps at least twice (mbarrier parity flips); the sums stay exact"""
	B, T, ld, C = 256, 4096, 64, 64
	for n_in in (1, 2, 4):
		geo = TO.stream_geometry(B * T, ld, n_in)
		print('wrap case n_inputs', n_in, geo, 'CTA bound', TO.resident_cta_bound(geo), 'wraps >=', TO.ring_wraps(geo))
		assert TO.ring_wraps(geo) >= 2, geo
	gen = torch.Generator().manual_seed(99)
	report = []
	fr = [1.0, 0.5, 0.25, 0.75] * 64
	for split, act, a, b, drop_p, frozen in ((False, 2, 0.0, 20.0, 0.0, False), (True, 1, 0.0, 0.0, 0.5, False), (False, 3, 0.125, 0.0, 0.5, True)):
		_bn_run('wrap', ld, C, B, T, fr, split, act, a, b, drop_p, frozen, gen, big = True, report = report)
	print('wrap case: share of bf16 outputs one ulp away from the rounded float64 reference:', report)


def test_uncovered_pitch_row_walker_and_split_refusal():
	"""ld = 1088 (136 channel vectors: no CTA of <= 512 threads is a whole number of warps): the bf16 tier runs the row
	walkers exactly; the split tier is refused and launches nothing"""
	from convasr_b200 import _lib as L
	lib, dev = _lib(), _dev()
	assert TO.stream_geometry(256, 1088, 1) is None and lib.cab_bn_bwd_apply_covers(256, 1088, 1) == 0
	gen = torch.Generator().manual_seed(5)
	for act, a, b in ACTS:
		_bn_run('ld1088', 1088, 1050, 4, 64, [1.0, 0.5, 0.25, 0.0], False, act, a, b, 0.5 if act % 2 else 0.0, act == 3, gen)
	y = torch.zeros(64, 1088, dtype = BF16, device = dev)
	ss = torch.zeros(4, 1088, device = dev)
	before = L.launch_count()
	rc = lib.cab_bn_act_mask_fwd(_p(y), _p(y), _p(ss), 1, 64, 1088, 1088, 1, 0.0, 0.0, None, _p(y.clone()), _p(y.clone()), 0.0, None, 0, _stream())
	assert rc != 0 and b'not covered' in lib.cab_last_error()
	sums = torch.zeros(2, 1088, device = dev)
	parts = torch.zeros(TO.SUM_REPLICAS * 2 * 1088, dtype = torch.float64, device = dev)
	rc = lib.cab_bn_act_mask_bwd(_p(y), _p(y), _p(y), _p(y), _p(ss), 1, 64, 1088, 1088, 1, 0.0, 0.0, None, _p(sums), _p(y.clone()), _p(y.clone()), 0.0, None, 0, 0, _p(parts), _stream())
	assert rc != 0
	assert L.launch_count() == before


# ------------------------------------------------------------------------------------------ statistics
def test_batch_stats_finalize_and_folded_finalize_are_bit_identical():
	"""cab_bn_batch_stats / cab_bn_finalize against float64 (rsqrtf within 2 ulp), and the folded finalize of
	cab_bn_act_mask_fwd_stats bit-identical to cab_bn_finalize: scale / shift table and running statistics"""
	lib, dev = _lib(), _dev()
	gen = torch.Generator().manual_seed(11)
	for B, T, C, ld, sums_ld in ((4, 50, 40, 64, 64), (2, 33, 300, 320, 384), (1, 1, 64, 64, 128), (8, 64, 1000, 1024, 1024)):
		R = B * T
		y = TO.ints((R, ld), -40, 40, gen) / 8
		y[:, C:] = float('nan')  # colstats reads whole vectors; channels >= C never reach the sums
		yd = _bf(y)
		gamma = torch.randn(C, generator = gen).to(dev)
		gamma[::4] *= -1
		beta = torch.randn(C, generator = gen).to(dev)
		rm0, rv0 = torch.randn(C, generator = gen).to(dev), (torch.rand(C, generator = gen) + 0.5).to(dev)
		ws = torch.empty(2, C, dtype = torch.float64, device = dev)
		ss_a, rm_a, rv_a = _nan(4, C, dtype = torch.float32), rm0.clone(), rv0.clone()
		_check(lib.cab_bn_batch_stats(_p(yd), B, T, C, ld, _p(gamma), _p(beta), 1e-5, 0.1, _p(rm_a), _p(rv_a), _p(ws), _p(ss_a), _stream()), 'stats')
		raw = torch.stack([y[:, :C].sum(0), (y[:, :C] ** 2).sum(0)]).to(dev)
		assert torch.equal(ws, raw), (B, T, C)  # integer / 8 data: every partial sum exact
		ref, rm_r, rv_r = TO.batch_stats_ref(y.to(dev), C, R, gamma, beta, 1e-5, 0.1, rm0, rv0)
		# mean: a double product rounded to fp32 (1 ulp); var: a double rounded to fp32, + eps in fp32 (1 ulp each, halved by the
		# square root); invstd = rsqrtf within 2 ulp: 4 ulp in all.  scale = gamma * invstd adds one rounding; shift = beta - mean *
		# scale adds two, relative to the larger of |beta| and |mean * scale|.
		ulp = lambda x: torch.pow(2.0, torch.floor(torch.log2(x.abs().double().clamp(min = 2.0 ** -126))) - 23)
		assert bool(((ss_a[2].double() - ref[2]).abs() <= ulp(ref[2])).all())
		assert bool(((ss_a[3].double() - ref[3]).abs() <= 4 * ulp(ref[3])).all())
		assert bool(((ss_a[0].double() - ref[0]).abs() <= 5 * ulp(ref[0])).all())
		assert bool(((ss_a[1].double() - ref[1]).abs() <= 8 * (ulp(ref[1]) + ulp(ref[2] * ref[0]))).all())
		assert torch.allclose(rm_a.double(), rm_r, rtol = 1e-6, atol = 1e-6) and torch.allclose(rv_a.double(), rv_r, rtol = 1e-5, atol = 1e-6)
		# finalize from padded sums [2][sums_ld]
		padded = torch.full((2, sums_ld), float('nan'), dtype = torch.float64, device = dev)
		padded[:, :C] = raw
		ss_b, rm_b, rv_b = _nan(4, C, dtype = torch.float32), rm0.clone(), rv0.clone()
		_check(lib.cab_bn_finalize(_p(raw.contiguous()), R, C, _p(gamma), _p(beta), 1e-5, 0.1, _p(rm_b), _p(rv_b), _p(ss_b), _stream()), 'finalize')
		assert torch.equal(ss_a, ss_b) and torch.equal(rm_a, rm_b) and torch.equal(rv_a, rv_b)
		for split in (False, True):
			ss_c, rm_c, rv_c = _nan(4, C, dtype = torch.float32), rm0.clone(), rv0.clone()
			out, out_lo = _nan(R, ld), (_nan(R, ld) if split else None)
			ylo = torch.zeros_like(yd) if split else None
			_check(lib.cab_bn_act_mask_fwd_stats(_p(yd), _p(ylo), _p(padded), sums_ld, R, _p(gamma), _p(beta), 1e-5, 0.1, _p(rm_c), _p(rv_c), _p(ss_c), B, T, C, ld,
												2, 0.0, 20.0, None, _p(out), _p(out_lo), 0.0, None, 0, _stream()), 'fwd_stats')
			assert torch.equal(ss_c, ss_b), ('folded finalize differs from cab_bn_finalize', B, T, C, split)
			assert torch.equal(rm_c, rm_b) and torch.equal(rv_c, rv_b), ('running statistics', B, T, C, split)
			o_ref = TO.bn_fwd_ref(y.to(dev), ss_c.double(), B, T, C, 2, 0.0, 20.0)  # z = fmaf(y, scale, shift): one fp32 rounding
			assert torch.equal(out, o_ref.to(BF16)) if not split else torch.equal(out, TO.split_store(o_ref)[0])


# ------------------------------------------------------------------------------------------ multi-branch forward and dz
@pytest.mark.parametrize('split', [False, True], ids = ['bf16', 'split'])
def test_multi_branch_forward_and_stored_output_gate(split):
	from convasr_b200 import _lib as L
	lib, dev = _lib(), _dev()
	gen = torch.Generator().manual_seed(21 + split)
	B, T, C, ld = 4, 50, 40, 64
	R = B * T
	xlen = torch.tensor([1.0, 0.5, 0.02, 0.0], device = dev)
	seed = torch.tensor([SEED], dtype = torch.int64, device = dev)
	band_hits = 0
	for n in range(1, L.MAX_BN_BRANCHES + 1):
		for (act, a, b), drop_p in ((ACTS[n % 4], 0.0), (ACTS[(n + 1) % 4], 0.5), (ACTS[2], 0.0)):
			drop = (drop_p, TO.dropout_keep(SEED, SALT, R, ld, drop_p).to(dev)) if drop_p else None
			keep_alive, branches, structs = [], [], []
			for i in range(n):
				ident = i % 3 == 1
				hi = TO.ints((R, ld), -8, 8, gen) / 4
				lo = TO.ints((R, ld), -3, 3, gen) / 256 if split else None
				hi[:, C:] = POISON
				ss = None if ident else TO.exact_ss(C, gen)
				if n >= 2:
					# plant z = b - 1/32 = 19.96875 on rows 0..7 (bf16 stores 20.0 there): branch 0 contributes -1/32, branch 1
					# (identity) carries 20, every other branch contributes 0
					want = -1 / 32 if i == 0 else (20.0 if i == 1 else 0.0)
					yv0 = torch.full((C, ), want, dtype = torch.float64) if ident else (want - ss[1, :C]) / ss[0, :C]
					ok = yv0.float().to(BF16).double() == yv0
					assert i != 1 or bool(ok.all())
					hi[:8, :C] = torch.where(ok, yv0, hi[:8, :C])
					if lo is not None:
						lo[:8, :C] = 0
				yv = hi + (lo if split else 0)
				branches.append((yv.to(dev), ss.to(dev) if ss is not None else None))
				h, l = _bf(hi), (_bf(lo) if split else None)
				s32 = ss.float().contiguous().to(dev) if ss is not None else None
				keep_alive += [h, l, s32]
				structs.append(L.BnBranch(h.data_ptr(), l.data_ptr() if l is not None else None, s32.data_ptr() if s32 is not None else None))
			arr = (L.BnBranch * n)(*structs)
			out, out_lo = _nan(R, ld), (_nan(R, ld) if split else None)
			_check(lib.cab_bn_multi_act_mask_fwd(arr, n, B, T, C, ld, act, a, b, _p(xlen), _p(out), _p(out_lo), drop_p, _p(seed), SALT, _stream()), 'multi fwd')
			z, o_ref = TO.multi_fwd_ref(branches, B, T, C, act, a, b, xlen, drop)
			TO.fp32_exact(z, 'z')
			if split:
				hi_r, lo_r = TO.split_store(o_ref)
				assert torch.equal(out, hi_r) and torch.equal(out_lo, lo_r), (n, act, drop_p)
			else:
				assert torch.equal(out, o_ref.to(BF16)), (n, act, drop_p)
			# dz from the stored output
			g_hi = TO.ints((R, ld), -8, 8, gen) / 2
			g_lo = TO.ints((R, ld), -1, 1, gen) / 64 if split else None
			g_hi[:, C:] = POISON
			gh, gl = _bf(g_hi), (_bf(g_lo) if split else None)
			gsum = g_hi + (g_lo if split else 0)
			dz, dz_lo = _nan(R, ld), (_nan(R, ld) if split else None)
			_check(lib.cab_act_mask_bwd_dz(_p(out), _p(out_lo), _p(gh), _p(gl), B, T, C, ld, act, a, b, _p(xlen), _p(dz), _p(dz_lo), drop_p, _p(seed), SALT, _stream()), 'dz')
			stored = out.float() + out_lo.float() if split else out.float()
			d_ref = TO.dz_stored_gate_ref(stored, gsum.to(dev), B, T, C, act, a, b, xlen, drop)
			if split:
				hi_r, lo_r = TO.split_store(d_ref.float())
				assert torch.equal(dz, hi_r) and torch.equal(dz_lo, lo_r), (n, act, drop_p)
			else:
				assert torch.equal(dz, d_ref.float().to(BF16)), (n, act, drop_p)
			# against autograd's z-gate: disagreements only inside the band of finding "stored-output gate" (train.cu,
			# act_bwd_dz_kernel): within 2^-8 (bf16) / 2^-16 (split) of |bound| from a hardtanh clamp bound
			zg = torch.zeros(R, ld, dtype = torch.float64, device = dev)
			zg[:, :C] = TO.z_gate(z, act, a, b)
			sg = torch.zeros_like(zg)
			sg[:, :C] = TO.gate64((stored.double() * float(torch.tensor(1.0 - drop_p, dtype = torch.float32)))[:, :C], torch.ones(R, C, dtype = torch.float64, device = dev), act, a, b) if act != 3 else torch.where(stored[:, :C] > 0, 1.0, a).double()
			live = TO.row_mask(B, T, xlen, dev).reshape(R, 1).expand(R, ld).clone()
			live[:, C:] = False
			if drop:
				live &= drop[1]
			dis = live & (zg != sg)
			if act != 2:
				assert not bool(dis.any()), (n, act, drop_p)
			else:
				rel = 2.0 ** -8 if not split else 2.0 ** -16
				zz = torch.zeros(R, ld, dtype = torch.float64, device = dev)
				zz[:, :C] = z
				near = ((zz - a).abs() <= rel * max(abs(a), 1e-30)) | ((zz - b).abs() <= rel * abs(b))
				assert bool(near[dis].all()), (n, drop_p, zz[dis & ~near][:4])
				if not split and drop_p == 0.0 and n >= 2:
					band_hits += int(dis.sum())
	if not split:
		assert band_hits > 0, 'the planted z = b - 1/32 must read as clamped in the bf16 tier'


# ------------------------------------------------------------------------------------------ packing
def _pack_items(specs, split, gen):
	"""NaN-prefilled outputs for each (Co, Ci, K, mode, pad, ci_ld, co_ld, want_dgrad) -> (items, outputs, weights)"""
	from convasr_b200 import _lib as L
	dev = _dev()
	items, outs, ws = [], [], []
	for Co, Ci, K, mode, pad, ci_ld, co_ld, want_dgrad in specs:
		w = torch.randn(Co, Ci, K, generator = gen).to(dev)
		if mode == 1:
			fwd = _nan(TO.taps2(K, pad), Co, 2 * ci_ld)
			dgr = None
		else:
			fwd = _nan(K, Co, ci_ld)
			dgr = _nan(K, Ci, co_ld) if want_dgrad else None
		fwd_lo = torch.full_like(fwd, float('nan')) if split else None
		dgr_lo = torch.full_like(dgr, float('nan')) if split and dgr is not None else None
		items.append(L.PackItem(w.data_ptr(), fwd.data_ptr(), dgr.data_ptr() if dgr is not None else None, fwd_lo.data_ptr() if fwd_lo is not None else None,
								dgr_lo.data_ptr() if dgr_lo is not None else None, Co, Ci, K, 2 * ci_ld if mode == 1 else ci_ld, co_ld, mode, pad))
		outs.append((fwd, dgr, fwd_lo, dgr_lo))
		ws.append(w)
	return items, outs, ws


def _check_packed(w, mode, pad, ci_ld, co_ld, outs, what):
	fwd, dgr, fwd_lo, dgr_lo = outs
	rf, rd = TO.pack_ref(w, ci_ld, co_ld, mode, pad)
	for got, ref, lo in ((fwd, rf, fwd_lo), (dgr, rd, dgr_lo)):
		if got is None:
			continue
		r32 = ref.float()
		hi = r32.to(BF16)
		assert torch.equal(got.float().isnan(), r32.isnan()), (what, 'a slot outside the documented ones changed or was skipped')
		m = ~r32.isnan()
		assert torch.equal(got[m], hi[m]), what
		if lo is not None:
			assert torch.equal(lo.float().isnan(), r32.isnan()), what
			assert torch.equal(lo[m], (r32[m] - hi[m].float()).to(BF16)), what


PACK_SPECS = [
	# (Co, Ci, K, mode, pad, ci_ld, co_ld, want_dgrad)
	(40, 24, 11, 0, 5, 64, 64, True), (17, 33, 1, 0, 0, 40, 24, True), (70, 9, 2, 0, 0, 16, 72, True), (33, 50, 13, 0, 6, 56, 40, False),
	(48, 20, 29, 0, 14, 24, 48, True), (36, 10, 11, 1, 5, 16, 0, False), (20, 7, 13, 1, 6, 8, 0, False), (16, 33, 2, 1, 1, 40, 0, False),
	(5, 3, 11, 1, 4, 4, 0, False), (9, 17, 29, 1, 14, 24, 0, False),
]


@pytest.mark.parametrize('split', [False, True], ids = ['bf16', 'split'])
def test_batched_weight_packing_all_modes_and_chunking(split):
	"""34 items (two batched launches of at most 32, as training._pack_all chunks them): modes 0 and 1, even and odd pads,
	K in {1, 2, 11, 13, 29}, Co / Ci not multiples of 16 / 32; only the documented slots change"""
	from convasr_b200 import _lib as L
	gen = torch.Generator().manual_seed(31)
	specs = (PACK_SPECS * 4)[:34]
	items, outs, ws = _pack_items(specs, split, gen)
	for lo in range(0, len(items), L.PACK_MAX_ITEMS):
		chunk = items[lo:lo + L.PACK_MAX_ITEMS]
		_check(_lib().cab_pack_weights_batched((L.PackItem * len(chunk))(*chunk), len(chunk), _stream()), 'pack batched')
	for s, w, o in zip(specs, ws, outs):
		_check_packed(w, s[3], s[4], s[5], s[6], o, s)
	# training._pack_all over the same specs (two launches): the same values in its zero-filled buffers
	from convasr_b200 import training
	got = training._pack_all([(w, s[5], s[6], s[7], s[3], s[4]) for s, w in zip(specs, ws)], split)
	for s, w, o, g in zip(specs, ws, outs, got):
		for mine, theirs in zip(o, g):
			if mine is not None:
				assert torch.equal(mine.nan_to_num(0.0), theirs), s


def test_per_layer_weight_packing():
	lib = _lib()
	gen = torch.Generator().manual_seed(32)
	for Co, Ci, K, _, _, ci_ld, co_ld, _ in [s for s in PACK_SPECS if s[3] == 0]:
		w = torch.randn(Co, Ci, K, generator = gen).to(_dev())
		fwd, dgr = _nan(K, Co, ci_ld), _nan(K, Ci, co_ld)
		_check(lib.cab_pack_weight(_p(w), Co, Ci, K, _p(fwd), ci_ld, _p(dgr), co_ld, _stream()), 'pack')
		_check_packed(w, 0, 0, ci_ld, co_ld, (fwd, dgr, None, None), (Co, Ci, K))


UNPACK_SPECS = [
	# (K, Co, Ci, mode, pad)
	(11, 40, 24, 0, 0), (2, 17, 33, 1, 0), (13, 36, 10, 2, 6), (1, 70, 9, 0, 0), (4, 33, 50, 2, 1), (29, 9, 17, 1, 0), (12, 5, 3, 2, 5),
	(11, 36, 19, 2, 5),
]


def _packed_grad(K, Co, Ci, mode, pad, gen):
	"""fp32 packed gradient with NaN in every slot the unpack never reads, plus (ld, pair_ci_alloc)"""
	dev = _dev()
	w = torch.randn(Co, Ci, K, generator = gen).double()
	if mode == 2:
		ca = Ci + 3
		p, _ = TO.pack_ref(w, ca, 0, 1, pad)
		return p.float().to(dev), w.to(dev), 2 * ca, ca
	fwd, dgr = TO.pack_ref(w, Ci + 5, Co + 3)
	p = fwd if mode == 0 else dgr.flip(0)
	return p.float().contiguous().to(dev), w.to(dev), p.shape[2], 0


def test_unpack_per_layer_and_batched():
	"""per-layer cab_unpack_wgrad (modes 0, 1, 2, with and without accumulate) and the batched kernel over 36 items in
	training's chunks of 32 (even K, Co * Ci not a multiple of 256)"""
	from convasr_b200 import _lib as L
	lib, dev = _lib(), _dev()
	gen = torch.Generator().manual_seed(41)
	for K, Co, Ci, mode, pad in UNPACK_SPECS:
		packed, w, ld, ca = _packed_grad(K, Co, Ci, mode, pad, gen)
		want = TO.unpack_ref(packed, K, Co, Ci, mode, pad, ca)
		assert torch.equal(want, w.float().double())
		for acc in (0, 1):
			base = torch.randn(Co, Ci, K, generator = gen).to(dev)
			grad = base.clone() if acc else _nan(Co, Ci, K, dtype = torch.float32)
			_check(lib.cab_unpack_wgrad(_p(packed), K, Co, Ci, ld, mode, _p(grad), acc, pad, ca, _stream()), 'unpack')
			assert torch.equal(grad, base + want.float() if acc else want.float()), (K, Co, Ci, mode, acc)
	specs = (UNPACK_SPECS * 5)[:36]
	assert any((Co * Ci) % 256 and K % 2 == 0 for K, Co, Ci, _, _ in specs)
	items, keep, wants = [], [], []
	for K, Co, Ci, mode, pad in specs:
		packed, w, ld, ca = _packed_grad(K, Co, Ci, mode, pad, gen)
		grad = _nan(Co, Ci, K, dtype = torch.float32)
		items.append(L.UnpackItem(packed.data_ptr(), grad.data_ptr(), K, Co, Ci, ld, mode, pad, ca))
		keep += [packed, grad]
		wants.append((grad, TO.unpack_ref(packed, K, Co, Ci, mode, pad, ca).float()))
	for lo in range(0, len(items), 32):
		chunk = items[lo:lo + 32]
		_check(lib.cab_unpack_wgrad_batched((L.UnpackItem * len(chunk))(*chunk), len(chunk), _stream()), 'unpack batched')
	for (grad, want), s in zip(wants, specs):
		assert torch.equal(grad, want), s


# ------------------------------------------------------------------------------------------ logits-gradient layout cast
def test_bct_to_btc():
	lib, dev = _lib(), _dev()
	gen = torch.Generator().manual_seed(51)
	for B, C, T, ld in ((3, 29, 45, 40), (2, 38, 33, 64), (1, 100, 70, 104), (4, 5, 1, 8)):
		for integer in (True, False):
			x = (torch.randint(-50, 51, (B, C, T), generator = gen).float() if integer else torch.randn(B, C, T, generator = gen)).to(dev)
			ref, cs_ref = TO.bct_to_btc_ref(x, ld)
			for want_lo, want_sums in ((False, True), (True, False), (True, True)):
				out, lo = _nan(B, T, ld), (_nan(B, T, ld) if want_lo else None)
				cs = _nan(C, dtype = torch.float32) if want_sums else None
				_check(lib.cab_bct_to_btc(_p(x), B, C, T, ld, _p(out), _p(lo), _p(cs), _stream()), 'bct_to_btc')
				hi, lo_r = TO.split_store(ref.float())
				assert torch.equal(out, hi), (B, C, T, ld)
				if want_lo:
					assert torch.equal(lo, lo_r)
				if want_sums:
					if integer:
						assert torch.equal(cs, cs_ref.float())  # integer data: every order of the sum is exact
					else:
						assert torch.allclose(cs.double(), cs_ref, rtol = 1e-5, atol = 1e-4)


# ------------------------------------------------------------------------------------------ optimizer
def _carve(sizes, offsets, gen, scale = 1.0):
	"""tensors of the given sizes at the given element offsets into flat buffers (offset % 4 != 0: not 16-byte aligned)"""
	out = []
	for n, off in zip(sizes, offsets):
		buf = torch.randn(n + off + 4, generator = gen) * scale
		t = buf.to(_dev())[off:off + n]
		assert (t.data_ptr() % 16 != 0) == (off % 4 != 0)
		out.append(t)
	return out


OPT_SIZES = [1, 3, 4, 5, 65536 - 1, 65536 + 1, 2 * 65536 - 3, 2 * 65536 + 3, 7, 300]
OPT_OFFS = [1, 2, 3, 0, 1, 0, 2, 3, 0, 1]


@pytest.mark.parametrize('kind', ['sgd', 'sgd_nesterov_dampening', 'novograd', 'novograd_dampening'])
def test_optimizer_unaligned_tensors_and_groups(kind):
	"""parameters, gradients and momentum at element offsets 1, 2, 3 of flat buffers, mixed with aligned tensors in one
	launch; numel 1 .. 2 * 65536 + 3 (chunk edges); two parameter groups with the global clip norm against float64"""
	from convasr_b200 import optimizers
	gen = torch.Generator().manual_seed(61)
	ps = _carve(OPT_SIZES, OPT_OFFS, gen)
	assert any(p.data_ptr() % 16 for p in ps)
	params = [torch.nn.Parameter(p) for p in ps]  # a Parameter shares the (unaligned) storage of the view
	assert all(q.data_ptr() == p.data_ptr() for p, q in zip(ps, params))
	ref = [p.detach().double().cpu() for p in ps]
	groups = [dict(params = params[:6]), dict(params = params[6:], lr = 0.02, weight_decay = 1e-2)]
	if kind.startswith('sgd'):
		nest = kind != 'sgd'
		opt = optimizers.SGD(groups, lr = 0.05, momentum = 0.9, dampening = 0.0, weight_decay = 1e-3, nesterov = nest)
		hyper = [(0.05, 1e-3), (0.02, 1e-2)]
	else:
		damp = kind == 'novograd_dampening'
		opt = optimizers.NovoGrad(groups, lr = 0.01, betas = (0.95, 0.98), weight_decay = 1e-3, dampening = damp)
		hyper = [(0.01, 1e-3), (0.02, 1e-2)]
	# momentum buffers at unaligned offsets too: replace the zero buffers with views of fresh flat buffers
	for i, p in enumerate(params):
		st = opt.state[p]
		off = (i + 1) % 4
		mb = torch.zeros(p.numel() + off + 4, device = _dev())[off:off + p.numel()]
		st['momentum_buffer'] = mb
		st['_fresh'] = True
	bufs, emas = [None] * len(ps), [None] * len(ps)
	for step in range(3):
		grads = _carve(OPT_SIZES, [(o + step + 1) % 4 for o in OPT_OFFS], gen, scale = 2.0)
		assert any(g.data_ptr() % 16 for g in grads)
		for p, g in zip(params, grads):
			p.grad = g
		opt.step(max_grad_norm = 5.0)
		total, coef = TO.clip_coef([g.cpu() for g in grads], 5.0)
		assert abs(float(opt.total_grad_norm) - total) <= 1e-5 * total, (step, float(opt.total_grad_norm), total)
		for i, g in enumerate(grads):
			lr, wd = hyper[0] if i < 6 else hyper[1]
			if kind.startswith('sgd'):
				ref[i], bufs[i] = TO.sgd_step(ref[i], g.cpu(), bufs[i], lr, 0.9, 0.0, wd, kind != 'sgd', coef)
			else:
				ref[i], bufs[i], emas[i] = TO.novograd_step(ref[i], g.cpu(), bufs[i], emas[i], lr, 0.95, 0.98, 1e-8, wd, kind == 'novograd_dampening', coef)
			got = params[i].detach().cpu().double()
			assert torch.allclose(got, ref[i], rtol = 2e-5, atol = 2e-6), (kind, step, i, float((got - ref[i]).abs().max()))


def test_optimizer_many_tensors():
	"""more than 256 tensors: mt_prepare_kernel strides over them; aligned and unaligned mixed"""
	from convasr_b200 import optimizers
	gen = torch.Generator().manual_seed(62)
	sizes = [1 + (i * 37) % 300 for i in range(300)]
	ps = _carve(sizes, [i % 4 for i in range(300)], gen)
	params = [torch.nn.Parameter(p) for p in ps]
	ref = [p.detach().double().cpu() for p in ps]
	opt = optimizers.SGD(params, lr = 0.1, momentum = 0.9)
	bufs = [None] * len(ps)
	for step in range(2):
		grads = _carve(sizes, [(i + step) % 4 for i in range(300)], gen)
		for p, g in zip(params, grads):
			p.grad = g
		opt.step(max_grad_norm = 1.0)
		total, coef = TO.clip_coef([g.cpu() for g in grads], 1.0)
		assert abs(float(opt.total_grad_norm) - total) <= 1e-5 * total
		for i, g in enumerate(grads):
			ref[i], bufs[i] = TO.sgd_step(ref[i], g.cpu(), bufs[i], 0.1, 0.9, 0.0, 0.0, False, coef)
		for p, r in zip(params, ref):
			assert torch.allclose(p.detach().cpu().double(), r, rtol = 2e-5, atol = 2e-6), step


# ------------------------------------------------------------------------------------------ end to end
def test_training_step_with_a_batchnorm_width_not_a_multiple_of_4():
	"""Wav2Letter(base_width = 18): BatchNorm widths 36 / 126 / 144, so dgamma of the 126-wide layers is a view 126 floats into
	the flat gradient buffer (not 16-byte aligned).  Two eager steps and two graphed steps with optimizers.SGD and clipping,
	at the bars of test_gpu_training.py"""
	from convasr_b200 import models, optimizers, training
	from oracle import oracle as O
	dev = _dev()
	C = 38

	def make():
		m = models.Wav2Letter(64, [C], base_width = 18, num_blocks = 1, frontend = models.LogFilterBankFrontend(64, 8000, .02, .01, 'hann_window'), dropout = 0., check_time_dim_padded = False)
		shapes = {k: tuple(v.shape) for k, v in m.state_dict().items() if not k.startswith('frontend.')}
		sd = O.synth_state_dict(shapes, seed = 7)
		m.load_state_dict(sd, strict = False)
		m = m.to(dev).train().set_precision('bf16')
		assert training.supported(m)
		return m, sd

	g = torch.Generator().manual_seed(3)
	sig = (torch.randn(4, 12000, generator = g) * 3000).round().clamp(-32767, 32767).to(torch.int16)
	xlen = torch.tensor([1.0, 0.9, 0.66, 0.5])
	y = torch.randint(0, C - 1, (4, 1, 14), generator = g)
	ylen = torch.tensor([[14], [11], [8], [5]])
	m, sd = make()
	assert 126 in {r.conv.C_out for r in training._graph(m)}
	opt = optimizers.SGD(m.parameters(), lr = 1e-3, momentum = 0.9)
	sd_, yd, yl, xl = sig.to(dev), y.to(dev), ylen.to(dev), xlen.to(dev)
	eager = []
	for step in range(2):
		opt.zero_grad(set_to_none = True)
		o = m(sd_, xl, y = yd, ylen = yl)
		loss = (o['loss'] * yl[:, 0]).mean()
		loss.backward()
		if step == 0:
			grads = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}
			print('gradients handed to the optimizer at a 16-byte misaligned address:', sum(p.grad.data_ptr() % 16 != 0 for p in m.parameters() if p.grad is not None))
		opt.step(max_grad_norm = 100.0)
		eager.append(o['loss'].detach().clone())
	# first step against the float64-accumulating oracle (bars of test_training_step_shallow_model_matches_oracle)
	ref_sd = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and 'running' not in k else v.clone()) for k, v in sd.items()}
	_, lp, olen = O.model_forward(ref_sd, sig, xlen, model = 'Wav2Letter', training = True, round_bf16 = True)
	ref_loss = O.ctc_loss_torch(lp[0].permute(2, 0, 1), y[:, 0], olen[0], ylen[:, 0], C - 1).mean()
	ref_loss.backward()
	got_loss = float((eager[0].cpu() * ylen[:, 0]).mean())
	assert abs(got_loss - float(ref_loss)) / abs(float(ref_loss)) < 2e-2
	keys = [k for k, v in ref_sd.items() if v.is_floating_point() and v.requires_grad]
	flat = torch.cat([grads[k].flatten().cpu() for k in keys])
	flat_ref = torch.cat([ref_sd[k].grad.flatten() for k in keys])
	assert float((flat - flat_ref).norm() / flat_ref.norm()) < 0.15
	params_eager = {k: v.detach().cpu().clone() for k, v in m.named_parameters()}
	# graphed: same start, two replays
	m2, _ = make()
	opt2 = optimizers.SGD(m2.parameters(), lr = 1e-3, momentum = 0.9)
	step = training.GraphedTrainStep(m2, opt2, sd_, xl, yd, yl, warmup = 2, max_grad_norm = 100.0)
	m2.load_state_dict(sd, strict = False)
	for st in opt2.state.values():
		st['momentum_buffer'].zero_()
	graphed = [step(sd_, xl, yd, yl) for _ in range(2)]
	assert torch.allclose(eager[0], graphed[0], rtol = 1e-4, atol = 1e-4)
	assert torch.allclose(torch.stack(eager), torch.stack(graphed), rtol = 2e-2, atol = 2e-2)
	for k, v in m2.named_parameters():
		assert bool(torch.isfinite(v).all()), k
		d = float((v.detach().cpu() - params_eager[k]).norm() / params_eager[k].norm().clamp(min = 1e-12))
		assert d < 2e-2, (k, d)
