"""CPU checks of tests/train_oracle.py: the references the training-kernel tests compare with are pinned against
F.batch_norm / F.conv1d / torch.optim under float64 autograd before any GPU run, and the exactness bound refuses data
that could round."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import train_oracle as TO

ACTS = [(0, 0.0, 0.0), (1, 0.0, 0.0), (2, 0.0, 20.0), (3, 0.125, 0.0)]


def _torch_act(z, act, a, b):
	if act == 1:
		return F.relu(z)
	if act == 2:
		return F.hardtanh(z, a, b)
	if act == 3:
		return F.leaky_relu(z, a)
	return z


@pytest.mark.parametrize('act,a,b', ACTS)
@pytest.mark.parametrize('frozen', [False, True])
@pytest.mark.parametrize('dropout', [0.0, 0.5])
def test_bn_references_match_batch_norm_autograd(act, a, b, frozen, dropout):
	"""out = mask(dropout(act(BN(y)))): forward, dy, dbeta = sums[0], dgamma = sums[1] against float64 autograd"""
	gen = torch.Generator().manual_seed(10 + act)
	B, T, C, ld = 3, 11, 12, 16
	R = B * T
	y = torch.randn(R, ld, generator = gen, dtype = torch.float64) * 3 + 1
	g = torch.randn(R, ld, generator = gen, dtype = torch.float64)
	gamma = torch.randn(C, generator = gen, dtype = torch.float64)
	gamma[::3] *= -1
	beta = torch.randn(C, generator = gen, dtype = torch.float64)
	rm, rv = torch.randn(C, generator = gen, dtype = torch.float64), torch.rand(C, generator = gen, dtype = torch.float64) + 0.5
	xlen = torch.tensor([1.0, 0.5, 0.3])
	keep = TO.dropout_keep(5, 3, R, ld, dropout) if dropout else None
	drop = (dropout, keep) if dropout else None
	if frozen:
		istd = 1 / torch.sqrt(rv + 1e-5)
		ss = torch.stack([gamma * istd, beta - rm * gamma * istd, rm, istd])
	else:
		ss, _, _ = TO.batch_stats_ref(y, C, R, gamma, beta, 1e-5, 0.1)
	yl = y[:, :C].clone().reshape(B, T, C).permute(0, 2, 1).requires_grad_(True)
	gl, bl = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
	z = F.batch_norm(yl, rm.clone(), rv.clone(), gl, bl, training = not frozen, momentum = 0.1, eps = 1e-5)
	o = _torch_act(z, act, a, b)
	mask = TO.row_mask(B, T, xlen, 'cpu').reshape(B, T)[:, None, :]
	o = o * mask
	if drop:
		o = o * keep[:, :C].reshape(B, T, C).permute(0, 2, 1) * TO.inv_keep32(dropout)
	gg = g[:, :C].reshape(B, T, C).permute(0, 2, 1)
	(o * gg).sum().backward()
	fwd = TO.bn_fwd_ref(y, ss, B, T, C, act, a, b, xlen, drop)
	assert torch.allclose(fwd[:, :C].double(), o.detach().permute(0, 2, 1).reshape(R, C), rtol = 1e-6, atol = 1e-6)
	assert torch.equal(fwd[:, C:], torch.zeros(R, ld - C))
	ref = TO.bn_bwd_ref(y, g, ss, B, T, C, act, a, b, xlen, drop, frozen = frozen)
	assert torch.allclose(ref['dy'][:, :C].double(), yl.grad.permute(0, 2, 1).reshape(R, C), rtol = 1e-5, atol = 1e-6)
	assert torch.allclose(ref['sums'][0], bl.grad, rtol = 1e-10, atol = 1e-10)  # dbeta
	assert torch.allclose(ref['sums'][1], gl.grad, rtol = 1e-10, atol = 1e-10)  # dgamma
	assert torch.equal(ref['dy'][:, C:], torch.zeros(R, ld - C))


def test_batch_stats_reference_running_statistics():
	gen = torch.Generator().manual_seed(1)
	for n in (1, 2, 37):
		y = torch.randn(n, 8, generator = gen, dtype = torch.float64)
		gamma, beta = torch.randn(5, generator = gen, dtype = torch.float64), torch.randn(5, generator = gen, dtype = torch.float64)
		rm, rv = torch.randn(5, dtype = torch.float64), torch.rand(5, dtype = torch.float64) + 1
		rm_t, rv_t = rm.clone(), rv.clone()
		x = y[:, :5].T[None]
		out = F.batch_norm(x, rm_t, rv_t, gamma, beta, training = True, momentum = 0.1, eps = 1e-5) if n > 1 else None
		ss, rm2, rv2 = TO.batch_stats_ref(y, 5, n, gamma, beta, 1e-5, 0.1, rm, rv)
		if n > 1:  # torch refuses a single-value batch; the kernel uses n / max(n - 1, 1)
			assert torch.allclose(rm2, rm_t) and torch.allclose(rv2, rv_t)
			assert torch.allclose(x[0].T * ss[0] + ss[1], out[0].T)
		else:
			assert torch.allclose(rv2, 0.9 * rv)  # a single row: biased variance 0, running_var gets 0.1 * 0 * 1 / 1


def test_stored_output_gate_reference_matches_z_gate_away_from_bounds():
	"""dz_stored_gate_ref reads the gate off the stored output; with z exact in bf16 and off the clamp bounds it is the
	autograd gate"""
	gen = torch.Generator().manual_seed(2)
	B, T, C, ld = 2, 8, 8, 8
	z = TO.ints((B * T, ld), -40, 40, gen) / 2
	g = TO.ints((B * T, ld), -8, 8, gen)
	for act, a, b in ACTS:
		_, out = TO.multi_fwd_ref([(z, None)], B, T, C, act, a, b)
		out = out.to(torch.bfloat16).float()
		d = TO.dz_stored_gate_ref(out, g, B, T, C, act, a, b)
		ok = (z != a) & (z != b) if act == 2 else torch.ones_like(z, dtype = torch.bool)
		want = g * TO.z_gate(z, act, a, b)
		assert torch.equal(d[ok], want[ok]), act


def test_pair_packing_reference_is_a_stride2_conv():
	"""mode-1 packing: a stride-1 conv over frame pairs with the packed weight == the stride-2 conv (engine.pack_taps_stride2)"""
	gen = torch.Generator().manual_seed(3)
	B, Ci, Co, T = 2, 5, 7, 40
	for K, pad in ((11, 5), (13, 6), (2, 0), (1, 0), (4, 3)):
		w = torch.randn(Co, Ci, K, generator = gen, dtype = torch.float64)
		x = torch.randn(B, Ci, T, generator = gen, dtype = torch.float64)
		ref = F.conv1d(x, w, stride = 2, padding = pad)
		ci_ld = 8
		fwd, _ = TO.pack_ref(w, ci_ld, 0, mode = 1, pad = pad)
		assert fwd.shape[0] == TO.taps2(K, pad)
		wp = torch.nan_to_num(fwd, 0.0).permute(1, 2, 0)  # [Co, 2 * ci_ld, taps2]
		xp = torch.zeros(B, T // 2, 2 * ci_ld, dtype = torch.float64)
		xp.view(B, T // 2, 2, ci_ld)[:, :, :, :Ci] = x.permute(0, 2, 1).reshape(B, T // 2, 2, Ci)
		pad_left = -((0 - pad) // 2)
		n2 = fwd.shape[0]
		xpp = F.pad(xp.permute(0, 2, 1), (pad_left, n2))
		out = F.conv1d(xpp, wp)[:, :, :ref.shape[2]]
		assert torch.allclose(out, ref, atol = 1e-12), (K, pad)


def test_pack_unpack_round_trip():
	gen = torch.Generator().manual_seed(4)
	for Co, Ci, K, pad in ((7, 5, 11, 5), (33, 17, 2, 1), (16, 3, 13, 6), (1, 1, 1, 0)):
		w = torch.randn(Co, Ci, K, generator = gen, dtype = torch.float64)
		fwd, dgr = TO.pack_ref(w, Ci + 3, Co + 5)
		assert torch.equal(TO.unpack_ref(fwd, K, Co, Ci, 0), w)
		assert torch.equal(TO.unpack_ref(dgr.flip(0), K, Co, Ci, 1), w)
		assert bool(fwd[:, :, Ci:].isnan().all()) and bool(dgr[:, :, Co:].isnan().all())
		pf, _ = TO.pack_ref(w, Ci + 3, 0, mode = 1, pad = pad)
		assert torch.equal(TO.unpack_ref(pf, K, Co, Ci, 2, pair_pad = pad, pair_ci_alloc = Ci + 3), w)
		# every original tap lands in its own slot: exactly Co * Ci * K non-NaN values
		assert int((~pf.isnan()).sum()) == Co * Ci * K


def test_bct_to_btc_reference():
	x = torch.arange(2 * 3 * 5, dtype = torch.float32).view(2, 3, 5)
	out, cs = TO.bct_to_btc_ref(x, 8)
	assert torch.equal(out[1, 4, :3], x[1, :, 4].double()) and torch.equal(out[..., 3:], torch.zeros(2, 5, 5, dtype = torch.float64))
	assert torch.equal(cs, x.double().sum(dim = (0, 2)))


def test_stream_geometry_restatement_matches_the_library():
	"""cab_bn_bwd_apply_covers (host only, no device) against the restated geometry for every pitch 8 .. 4096"""
	from convasr_b200 import _lib
	lib = _lib.load()
	for ld in range(8, 4097, 8):
		for split in (0, 1):
			want = TO.stream_geometry(80 * 751, ld, 4 if split else 2) is not None
			assert (lib.cab_bn_bwd_apply_covers(80 * 751, ld, split) == 1) == want, (ld, split)
	assert TO.stream_geometry(1, 1088, 2) is None and TO.stream_geometry(1, 1024, 4) is not None
	geo = TO.stream_geometry(3 * 77, 96, 2)  # the shape of the older single-shape kernel test: no CTA takes a second chunk
	assert (geo['threads'], geo['rows_per_chunk'], geo['n_chunks']) == (288, 96 // 8 * 8, 3)
	assert TO.stream_geometry(1, 320, 1)['lanes'] == 8  # 40 vectors: 6 lanes rounded up to 8 for a whole number of warps
	assert TO.stream_geometry(1, 576, 1)['threads'] == 288


def test_dropout_mask_restatement():
	"""numpy uint64 splitmix64 against Python integers, and the keep rate"""
	seed, salt, rows, ld = 123456789, 7, 3, 40
	m = TO.dropout_keep(seed, salt, rows, ld, 0.3)
	M = (1 << 64) - 1
	for idx in (0, 1, 77, rows * ld - 1):
		z = (seed + salt * 0xD1B54A32D192ED03 + idx * 0x9E3779B97F4A7C15) & M
		z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
		z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
		z ^= z >> 31
		assert bool(m.view(-1)[idx]) == ((z >> 40) * 2.0 ** -24 >= float(np.float32(0.3)))
	big = TO.dropout_keep(1, 2, 512, 512, 0.3)
	assert abs(float(big.float().mean()) - 0.7) < 0.01


def _exact_case(R, C, gen, scale = 1):
	y = TO.ints((R, C), -12, 12, gen) / 4 * scale
	g = TO.ints((R, C), -8, 8, gen) / 8 * scale
	return y, g, TO.exact_ss(C, gen)


def test_exactness_bound_accepts_exact_data_and_refuses_data_that_could_round():
	gen = torch.Generator().manual_seed(6)
	B, T, C = 4, 64, 16
	y, g, ss = _exact_case(B * T, C, gen)
	TO.plant_z(y, ss, C, [0.0, 20.0], gen)
	for act, a, b in ACTS:
		TO.bn_bwd_ref(y, g, ss, B, T, C, act, a, b, check = True)
	# 1 / n not a power of two: m1 / n rounds
	with pytest.raises(ValueError):
		TO.bn_bwd_ref(y[:B * 3 * 7], g[:B * 3 * 7] + 1 / 8, ss, B, 21, C, 0, 0.0, 0.0, check = True)
	# sums that exceed 2^24 x the granularity: the fp32 partials could round
	big_y = y.clone()
	big_y[0, 0] = 2.0 ** 30
	with pytest.raises(ValueError):
		TO.bn_bwd_ref(big_y, g + 1 / 1024, ss, B, T, C, 0, 0.0, 0.0, check = True)
	# a non-dyadic scale makes z round
	ss2 = ss.clone()
	ss2[0, 0] = 0.1
	with pytest.raises(ValueError):
		TO.bn_bwd_ref(y, g, ss2, B, T, C, 0, 0.0, 0.0, check = True)


@pytest.mark.parametrize('nesterov,dampening,wd', [(False, 0.0, 0.0), (True, 0.0, 1e-2), (False, 0.3, 1e-3)])
def test_sgd_reference_matches_torch_sgd(nesterov, dampening, wd):
	gen = torch.Generator().manual_seed(7)
	p = torch.randn(50, generator = gen, dtype = torch.float64)
	q = p.clone().requires_grad_(True)
	opt = torch.optim.SGD([q], lr = 0.1, momentum = 0.9, dampening = dampening, weight_decay = wd, nesterov = nesterov)
	buf = None
	for _ in range(3):
		g = torch.randn(50, generator = gen, dtype = torch.float64)
		q.grad = g.clone()
		opt.step()
		p, buf = TO.sgd_step(p, g, buf, 0.1, 0.9, dampening, wd, nesterov)
		assert torch.allclose(p, q.detach(), rtol = 1e-12, atol = 1e-12)


def test_novograd_reference_matches_the_oracle_restatement():
	from oracle import oracle as O
	gen = torch.Generator().manual_seed(8)
	ps = [torch.randn(s, generator = gen, dtype = torch.float64) for s in (7, 30)]
	ref, state = [p.clone() for p in ps], [dict() for _ in ps]
	bufs, emas = [None, None], [None, None]
	for _ in range(3):
		grads = [torch.randn(p.shape, generator = gen, dtype = torch.float64) for p in ps]
		use, _ = O.clip_grad_norm(grads, 2.0)
		O.novograd_step(ref, [u.double() for u in use], state, lr = 0.01, weight_decay = 1e-3, dampening = True)
		total, coef = TO.clip_coef(grads, 2.0)
		for i in range(2):
			ps[i], bufs[i], emas[i] = TO.novograd_step(ps[i], grads[i], bufs[i], emas[i], 0.01, 0.95, 0.98, 1e-8, 1e-3, True, coef)
		for p, r in zip(ps, ref):
			assert torch.allclose(p, r, rtol = 1e-6, atol = 1e-9)


def test_pair_packing_reference_matches_engine_pack_taps_stride2():
	from convasr_b200 import engine
	gen = torch.Generator().manual_seed(9)
	for K, pad in ((11, 5), (13, 6), (4, 1), (1, 0)):
		w = torch.randn(6, 5, K, generator = gen)
		mine, _ = TO.pack_ref(w, 8, 0, mode = 1, pad = pad)
		theirs, taps, pad_left = engine.pack_taps_stride2(w, pad, 8)
		assert taps == TO.taps2(K, pad) and pad_left == -((0 - pad) // 2)
		assert torch.equal(mine.nan_to_num(0.0).float(), theirs)


def test_fp32_tier_refuses_an_uncovered_batchnorm_pitch_before_any_launch():
	"""Wav2Letter(base_width = 136) has BatchNorm widths 952 and 1088 (row pitches 960 and 1088).  The split-bf16 backward
	streams 4 inputs, and neither pitch fits it: 1088 has no CTA of <= 512 threads that is a whole number of warps, and 960
	needs 240 KB of stages.  The fp32 tier names the first such width and refuses before the step launches anything (the
	input never reaches a device here)"""
	from convasr_b200 import models, training
	m = models.Wav2Letter(64, [38], base_width = 136, num_blocks = 1, dropout = 0.).train().set_precision('fp32')
	assert training.unsupported_reason(m) is None
	assert TO.stream_geometry(1, 960, 4) is None and TO.stream_geometry(1, 1088, 4) is None
	with pytest.raises(NotImplementedError, match = r'not built \(BatchNorm width 952: row pitch 960 has no split-bf16'):
		training.forward_training(m, torch.zeros(1, 64, 32), torch.ones(1))
	ok = models.Wav2Letter(64, [38], base_width = 68, num_blocks = 1, dropout = 0.).train().set_precision('fp32')
	assert {r.conv.co_alloc for r in training._graph(ok)} == {192, 512, 576}
	for r in training._graph(ok):
		assert TO.stream_geometry(1, r.conv.co_alloc, 4) is not None
