"""FP8 inference tier, host side (no GPU): weight quantisation with one alpha shared by all sources of a launch, the
128-channel allocations of the fp8 plan, and the saturating E4M3 conversion."""
import torch

from convasr_b200 import engine, models


def _all_keys(plan):
	return {g.in_key for L in plan.launches() for g in L.gemms} | {L.key for L in plan.launches()}


def test_e4m3_saturates_instead_of_producing_nan():
	x = torch.tensor([500.0, -1000.0, 448.0, 1e30, -1e30, 0.1])
	# torch's own cast is not saturating: this is why engine.e4m3 clamps first
	assert torch.isnan(x.to(torch.float8_e4m3fn).float()[0])
	q = engine.e4m3(x).float()
	assert q.tolist()[:5] == [448.0, -448.0, 448.0, 448.0, -448.0]
	assert torch.isfinite(q).all()


def test_sources_share_one_alpha_and_absorb_their_input_scale():
	g = torch.Generator().manual_seed(0)
	w1 = torch.randn(3, 40, 128, generator = g)
	w2 = torch.randn(1, 40, 256, generator = g) * 5
	w3 = torch.randn(1, 24, 128, generator = g) * 0.01  # fewer rows (a narrower residual)
	w1[:, 7] = 0
	w2[:, 7] = 0  # row 7 is zero in every source it exists in
	w3[:, 7] = 0
	s = [0.02, 0.5, 3.0]
	(q1, q2, q3), alpha = engine.quantize_sources_fp8([w1, w2, w3], s)
	assert alpha.shape == (40, ) and alpha[7] == 1.0
	peak = torch.stack([w1.abs().amax(dim = (0, 2)) * s[0], w2.abs().amax(dim = (0, 2)) * s[1], torch.cat([w3.abs().amax(dim = (0, 2)) * s[2], torch.zeros(16)])]).amax(0)
	live = peak > 0
	assert torch.allclose(alpha[live], peak[live] / 448)
	for q in (q1, q2, q3):
		assert q.dtype == torch.float8_e4m3fn and torch.isfinite(q.float()).all() and float(q.float().abs().max()) <= 448
	# exactly one source reaches +-448 in each live row, and dequantised weights approximate W_j * s_j / alpha
	top = torch.stack([q1.float().abs().amax(dim = (0, 2)), q2.float().abs().amax(dim = (0, 2)), torch.cat([q3.float().abs().amax(dim = (0, 2)), torch.zeros(16)])]).amax(0)
	assert torch.equal(top[live], torch.full_like(top[live], 448.0))
	for w, q, sj in ((w1, q1, s[0]), (w2, q2, s[1]), (w3, q3, s[2])):
		ref = w * sj / alpha[:w.shape[1]].view(1, -1, 1)
		err = (q.float() - ref).abs()
		assert bool((err <= ref.abs() * 2**-4 + 2**-9 + 1e-12).all())  # half an E4M3 step (3 mantissa bits), or subnormal step


def test_fp8_plan_pads_every_contracted_width_to_128():
	for name, kw, nc in (('Wav2Letter', {}, [38]), ('JasperNetSeparable', dict(groups = 8), [38]), ('JasperNetBigNoStride', {}, [38]),
							('JasperNetBig', dict(decoder_type = 'bpe'), [38, 300]), ('Wav2LetterFlat', {}, [38])):
		m = getattr(models, name)(64, nc, base_width = 8, **kw).eval()
		bf = engine.StackPlan(m, False)
		scales = {k: 0.01 * (i + 1) for i, k in enumerate(sorted(_all_keys(bf), key = str))}
		p8 = engine.StackPlan(m, False, fp8_scales = scales)
		assert p8.fp8 and not p8.fp32_tier and bf.align == 64 and p8.align == 128
		# stride-2 prologue: 64-wide features whose frame-pair view is 128 wide; stride 1: 128-wide features
		assert p8.feat_align == (128 if name == 'JasperNetBigNoStride' else 64)
		for L in p8.launches():
			assert L.alpha is not None and L.alpha.dtype == torch.float32 and L.alpha.numel() >= L.C_out
			if L.epilogue == engine._lib.EPI_ACT_BF16:
				assert L.C_alloc % 128 == 0 and L.alpha.numel() == L.C_alloc
				assert L.out_scale == scales[L.key]
			for g in L.gemms:
				assert g.c_in_alloc % 128 == 0, (name, g.c_in_alloc)
				assert g.weights.hi.dtype == torch.float8_e4m3fn and g.weights.hi.shape[2] == g.c_in_alloc
				assert g.weights.f32 is None
		# the bf16 plan is untouched by the tier: 64-channel allocations
		assert all(g.c_in_alloc % 64 == 0 for L in bf.launches() for g in L.gemms)
		assert any(g.c_in_alloc % 128 for L in bf.launches() for g in L.gemms)


def test_fp8_plan_names_a_missing_scale():
	import pytest
	m = models.Wav2Letter(64, [38], base_width = 8).eval()
	with pytest.raises(RuntimeError, match = 'calibrate_fp8'):
		engine.StackPlan(m, False, fp8_scales = {'feat': 1.0})


def test_fp8_tier_refuses_training_and_uncalibrated_use():
	import pytest
	m = models.Wav2Letter(64, [38], base_width = 8).eval().set_precision('fp8')
	with pytest.raises(RuntimeError, match = 'inference only'):
		m.train()
	with pytest.raises(RuntimeError, match = r'calibrate_fp8\(x, xlen\) first'):
		m._get_plan()
	m.set_precision('bf16').train()  # other tiers train as before
	assert m.training
	# scales never enter the checkpoint
	keys = list(m.state_dict())
	m._fp8_calibration = (m._params_sig(), {})
	assert list(m.state_dict()) == keys
