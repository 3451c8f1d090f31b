"""The exact references of tests/conv_oracle.py, pinned in float64 against torch's conv1d and autograd on the CPU: the
GPU tests of the conv GEMM and the weight-gradient GEMM are only as good as these."""
import pytest
import torch
import torch.nn.functional as F

import conv_oracle as CO


def f64(*shape, seed):
	return torch.randn(*shape, generator = torch.Generator().manual_seed(seed), dtype = torch.float64)


def cl(x):
	"""[B, C, T] -> channels-last [B, T, C]"""
	return x.permute(0, 2, 1).contiguous()


@pytest.mark.parametrize('k, dil, pad', [(1, 1, 0), (3, 1, 1), (11, 1, 5), (7, 2, 6), (29, 2, 28), (5, 3, 0), (4, 1, 7)])
def test_conv_acc64_matches_conv1d(k, dil, pad):
	B, Ci, Co, T = 2, 5, 7, 40
	x, w = f64(B, Ci, T, seed = 1), f64(Co, Ci, k, seed = 2)
	want = F.conv1d(x, w, padding = pad, dilation = dil)
	T_out = want.shape[-1]
	got = CO.conv_acc64([CO.Src(cl(x), w.permute(2, 0, 1).contiguous(), Ci, k, dil, pad)], B, T_out)
	torch.testing.assert_close(got.permute(0, 2, 1), want, rtol = 1e-12, atol = 1e-12)


def test_conv_acc64_respects_channel_windows_rows_and_t_in():
	"""NaN outside every window the kernel promises not to read: activation channels, weight channels, rows >= T_in"""
	B, Ci, Co, T_in, T_rows, k, pad = 2, 6, 4, 30, 37, 5, 3
	x, w = f64(B, Ci, T_in, seed = 3), f64(Co, Ci, k, seed = 4)
	want = F.conv1d(x, w, padding = pad)
	act = torch.full((B, T_rows, 16), float('nan'), dtype = torch.float64)
	act[:, :T_in, 9:9 + Ci] = cl(x)
	wgt = torch.full((k, Co, 12), float('nan'), dtype = torch.float64)
	wgt[:, :, 2:2 + Ci] = w.permute(2, 0, 1)
	got = CO.conv_acc64([CO.Src(act, wgt, Ci, k, 1, pad, T_in = T_in, ch_off = 9, w_ch_off = 2)], B, want.shape[-1])
	torch.testing.assert_close(got.permute(0, 2, 1), want, rtol = 1e-12, atol = 1e-12)


def test_conv_acc64_sums_sources_with_their_own_geometry():
	"""two K segments of different taps, dilation, T_in and a negative pad_left (reads ahead), summed into one output"""
	B, T_out = 2, 25
	x1, w1 = f64(B, 3, 25, seed = 5), f64(4, 3, 3, seed = 6)
	x2, w2 = f64(B, 2, 40, seed = 7), f64(4, 2, 2, seed = 8)
	want = F.conv1d(x1, w1, padding = 1)  # pad_left 1
	shifted = x2[:, :, 4:]  # pad_left -4: out[t] reads x2[t + 4 + 3 tap]
	want = want + F.conv1d(shifted, w2, dilation = 3)[:, :, :T_out]
	srcs = [CO.Src(cl(x1), w1.permute(2, 0, 1).contiguous(), 3, 3, 1, 1), CO.Src(cl(x2), w2.permute(2, 0, 1).contiguous(), 2, 2, 3, -4)]
	got = CO.conv_acc64(srcs, B, T_out)
	torch.testing.assert_close(got.permute(0, 2, 1), want, rtol = 1e-12, atol = 1e-12)


@pytest.mark.parametrize('k, pad', [(11, 5), (4, 1), (3, 0)])
def test_stride2_frame_pair_view(k, pad):
	from convasr_b200 import engine
	B, Ci, Co, Fr = 2, 3, 5, 34
	x, w = f64(B, Ci, Fr, seed = 9), f64(Co, Ci, k, seed = 10)
	want = F.conv1d(x, w, stride = 2, padding = pad)
	wp, taps, pad_left = engine.pack_taps_stride2(w.float(), pad, Ci)
	pair = cl(x).reshape(B, Fr // 2, 2 * Ci)
	got = CO.conv_acc64([CO.Src(pair, wp.double(), 2 * Ci, taps, 1, pad_left)], B, want.shape[-1])
	torch.testing.assert_close(got.permute(0, 2, 1), want, rtol = 1e-6, atol = 1e-6)  # the packed weights are fp32


@pytest.mark.parametrize('k, dil, pad', [(1, 1, 0), (11, 1, 5), (29, 2, 28), (6, 1, 2)])
def test_dgrad_form_matches_autograd(k, dil, pad):
	"""grad_input = the forward GEMM over dy with flipped, transposed weights and pad_left = dil (k - 1) - pad"""
	B, Ci, Co, T_in = 2, 4, 6, 70
	x = f64(B, Ci, T_in, seed = 11).requires_grad_(True)
	w = f64(Co, Ci, k, seed = 12)
	y = F.conv1d(x, w, padding = pad, dilation = dil)
	dy = f64(*y.shape, seed = 13)
	y.backward(dy)
	w_dgrad = w.flip(2).permute(2, 1, 0).contiguous()  # [k, Ci, Co]
	got = CO.conv_acc64([CO.Src(cl(dy), w_dgrad, Co, k, dil, dil * (k - 1) - pad, T_in = y.shape[-1])], B, T_in)
	torch.testing.assert_close(got.permute(0, 2, 1), x.grad, rtol = 1e-12, atol = 1e-12)


@pytest.mark.parametrize('k, dil, pad', [(1, 1, 0), (11, 1, 5), (29, 2, 28), (3, 1, 0)])
def test_wgrad64_both_orientations_match_autograd(k, dil, pad):
	B, Ci, Co, T_in = 3, 5, 4, 66
	x = f64(B, Ci, T_in, seed = 14)
	w = f64(Co, Ci, k, seed = 15).requires_grad_(True)
	y = F.conv1d(x, w, padding = pad, dilation = dil)
	dy = f64(*y.shape, seed = 16)
	y.backward(dy)
	T_out = y.shape[-1]
	# dy on the M side: out[tap, co, ci]
	got = CO.wgrad64(cl(dy), T_out, Co, cl(x), T_in, Ci, k, dil, pad)
	torch.testing.assert_close(got, w.grad.permute(2, 0, 1), rtol = 1e-12, atol = 1e-12)
	# swapped: x on the M side, negative dilation and pad_left (the training step's orientation for narrow outputs)
	got = CO.wgrad64(cl(x), T_in, Ci, cl(dy), T_out, Co, k, -dil, -pad)
	torch.testing.assert_close(got, w.grad.permute(2, 1, 0), rtol = 1e-12, atol = 1e-12)


def test_wgrad64_skip_leaves_out_padding_frames():
	B, M, N, T = 3, 4, 5, 50
	a, bx = f64(B, T, M, seed = 17), f64(B, T, N, seed = 18)
	xlen = torch.tensor([1.0, 0.5, 0.0])
	lens = CO.frac_lengths(xlen, T) + 2
	a_cut = a * (torch.arange(T)[None, :, None] < lens[:, None, None])
	want = CO.wgrad64(a_cut, T, M, bx, T, N, 3, 1, 1)
	got = CO.wgrad64(a, T, M, bx, T, N, 3, 1, 1, skip = (xlen, T, 2))
	assert torch.equal(got, want)


def test_act_bf16_reference_split_is_exact():
	"""hi + lo reproduces the fp32 epilogue value to 16 bits; masked rows are zero in both parts"""
	g = torch.Generator().manual_seed(19)
	acc = torch.randn(2, 9, 32, generator = g, dtype = torch.float64) * 100
	bias = torch.randn(32, generator = g)
	hi, lo = CO.act_bf16_ref(acc, 32, bias = bias, act = 3, a = 0.01, xlen = torch.tensor([1.0, 0.5]), want_lo = True)
	assert bool((hi[1, 5:] == 0).all()) and bool((lo[1, 5:] == 0).all())  # ceil(0.5 * 9) = 5 valid rows
	y = acc[0].float() + bias
	y = torch.where(y > 0, y, y * 0.01)
	assert bool(((hi[0].float() + lo[0].float() - y).abs() <= y.abs() * 2 ** -16).all())
	assert not torch.equal(hi[0].float(), y)


def test_argmax_lowest_breaks_ties_to_the_lowest_id():
	x = torch.tensor([[1.0, 3.0, 3.0, 0.0], [5.0, 0.0, 0.0, 5.0], [2.0, 2.0, 2.0, 2.0]])
	assert CO.argmax_lowest(x).tolist() == [1, 0, 0]


def test_exactness_bound_refuses_a_case_that_could_round():
	g = torch.Generator().manual_seed(20)
	# 1024 channels x 29 taps of |a| = |w| = 256: partial sums reach 2^30.9 > 2^24: refused
	a = torch.full((1, 64, 1024), 256.0)
	w = torch.full((29, 32, 1024), 256.0)
	src = [CO.Src(a, w, 1024, 29, 1, 14)]
	with pytest.raises(ValueError, match = 'not be exact'):
		CO.assert_exact(CO.conv_bound(src, 1, 64), 1.0, 'big')
	# the same sums at granularity 2^-12 (hi * lo products) refuse far earlier
	hi, lo = CO.split_ints((1, 64, 256), g, 3, 4, -12)
	wh, wl = CO.split_ints((3, 32, 256), g, 3, 4, -12)
	srcs = [CO.Src(hi, wh, 256, 3, 1, 1), CO.Src(hi, wl, 256, 3, 1, 1), CO.Src(lo, wh, 256, 3, 1, 1)]
	r = CO.assert_exact(CO.conv_bound(srcs, 1, 64), 2.0 ** -12, 'split')
	assert r > 2 ** 22  # close to the limit: the check is what keeps the GPU cases honest
	with pytest.raises(ValueError):
		CO.assert_exact(CO.conv_bound(srcs, 1, 64) * 16, 2.0 ** -12, 'split x16')
	# wgrad: sums over batch and time
	A = torch.full((4, 3000, 8), 64.0)
	with pytest.raises(ValueError):
		CO.assert_exact(CO.wgrad_bound(A, 3000, 8, A, 3000, 8, 1, 1, 0), 1.0, 'wgrad')


def test_generators_are_exact_in_bf16_and_poison_helpers():
	g = torch.Generator().manual_seed(21)
	hi, lo = CO.split_ints((3, 10, 64), g, 256, 256, -12)
	CO.to_bf16_exact(hi)
	CO.to_bf16_exact(lo)
	with pytest.raises(AssertionError):
		CO.to_bf16_exact(torch.tensor([257.0]))
	x = CO.poison_channels(CO.poison_rows(torch.zeros(2, 8, 16), 5), 4, 8)
	assert bool(x[:, 5:].isnan().all()) and bool(x[..., :4].isnan().all()) and bool(x[..., 12:].isnan().all())
	assert not bool(x[:, :5, 4:12].isnan().any())
