"""Thin torch-tensor wrappers over the C ABI (include/convasr_b200.h).

PyTorch is used for device memory and streams only; every function here launches hand-written
sm_100a kernels through ctypes and raises if the tensors are not on a CUDA device.
"""
import ctypes
import math

import torch

from . import _lib

BF16 = torch.bfloat16
FP8 = torch.float8_e4m3fn


def _stream():
	return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
	return None if t is None else ctypes.c_void_p(t.data_ptr())


def _need_cuda(*tensors):
	for t in tensors:
		if t is not None and not t.is_cuda:
			raise RuntimeError('convasr_b200: tensors must live on a CUDA device (there is no CPU fallback)')


def frac_lengths(xlen, T):
	"""ceil(fp32(xlen) * T) as int64 -- models.py:611-614."""
	if xlen is None:
		return None
	return (xlen.to(torch.float32) * T).ceil().long()


# ------------------------------------------------------------------------------------------
# frontend
# ------------------------------------------------------------------------------------------
def make_twiddle(nfft, device):
	k = torch.arange(nfft // 2, dtype = torch.float64)
	ang = 2.0 * math.pi * k / nfft
	return torch.stack([ang.cos(), -ang.sin()], dim = -1).to(torch.float32).contiguous().to(device)


def make_mel_band(mel_fb):
	"""first / one-past-last non-zero bin per filter, int32 [n_mels, 2]"""
	nz = mel_fb != 0
	n_freq = mel_fb.shape[1]
	idx = torch.arange(n_freq, device = mel_fb.device)
	lo = torch.where(nz, idx, n_freq).min(dim = 1).values
	hi = torch.where(nz, idx + 1, 0).max(dim = 1).values
	lo = torch.minimum(lo, hi)
	return torch.stack([lo, hi], dim = 1).to(torch.int32).contiguous()


def frontend_logmel(
	signal, xlen, window, mel_fb, mel_band, twiddle, hop, nfft, preemphasis = 0.97, log_eps = 2.0**-14,
	normalize_signal = True, denom_multiplier = 1.0
):
	_need_cuda(signal, xlen, window, mel_fb, mel_band, twiddle)
	assert signal.ndim == 2
	if signal.dtype == torch.int16:
		is_i16 = 1
	else:
		signal = signal.to(torch.float32)
		is_i16 = 0
	signal = signal.contiguous()
	B, T = signal.shape
	n_mels = mel_fb.shape[0]
	F = T // hop + 1
	out = torch.empty(B, n_mels, F, dtype = torch.float32, device = signal.device)
	ws = torch.empty(B, dtype = torch.float32, device = signal.device)
	xl = None if xlen is None else xlen.to(torch.float32).contiguous()
	if B == 0 or T == 0:
		return out
	lib = _lib.load()
	rc = lib.cab_frontend_logmel(
		_p(signal), is_i16, _p(xl), B, T, window.numel(), hop, nfft, n_mels, _p(window), _p(mel_fb), _p(mel_band),
		_p(twiddle), float(preemphasis), float(log_eps), int(bool(normalize_signal)), float(denom_multiplier), _p(out),
		_p(ws), _stream()
	)
	_lib.check(rc, 'cab_frontend_logmel')
	return out


def frontend_features(signal, xlen, window, mel_fb, mel_band, twiddle, hop, nfft, preemphasis, log_eps, normalize_signal, denom_multiplier,
					normalize_features, norm_masked, norm_eps, F_pad, C_pad, want_lo = False):
	"""signal [B, T] int16 / fp32 -> (bf16 hi [B, F_pad, C_pad], bf16 lo or None, fp32 log-mel [B, n_mels, F]): frontend + masked
	instance norm + layout change (cab_frontend_features)"""
	_need_cuda(signal, xlen, window, mel_fb, mel_band, twiddle)
	assert signal.ndim == 2
	is_i16 = int(signal.dtype == torch.int16)
	if not is_i16:
		signal = signal.to(torch.float32)
	signal = signal.contiguous()
	B, T = signal.shape
	n_mels = mel_fb.shape[0]
	F = T // hop + 1
	dev = signal.device
	logmel = torch.empty(B, n_mels, F, dtype = torch.float32, device = dev)
	hi = torch.empty(B, F_pad, C_pad, dtype = BF16, device = dev)
	lo = torch.empty_like(hi) if want_lo else None
	absmax = torch.empty(2 * B, dtype = torch.float32, device = dev)
	partials = torch.empty(B, (F + 63) // 64 + 1, max(n_mels, 1), 2, dtype = torch.float32, device = dev)
	xl = None if xlen is None else xlen.to(torch.float32).contiguous()
	rc = _lib.load().cab_frontend_features(
		_p(signal), is_i16, _p(xl), B, T, window.numel(), hop, nfft, n_mels, _p(window), _p(mel_fb), _p(mel_band), _p(twiddle), float(preemphasis), float(log_eps),
		int(bool(normalize_signal)), float(denom_multiplier), int(bool(normalize_features)), int(bool(norm_masked)), float(norm_eps), _p(logmel), F_pad, C_pad, _p(hi), _p(lo), None,
		_p(absmax), _p(partials), _stream()
	)
	_lib.check(rc, 'cab_frontend_features')
	return hi, lo, logmel


def instnorm_pack(feat, xlen, eps, F_pad = None, C_pad = None, want_lo = False, want_f32 = False, want_hi = None, normalize = True):
	"""fp32 [B,C,F] -> (bf16 hi [B,F_pad,C_pad], bf16 lo or None, fp32 [B,C,F] or None)"""
	_need_cuda(feat, xlen)
	feat = feat.to(torch.float32).contiguous()
	B, C, F = feat.shape
	F_pad = F if F_pad is None else F_pad
	C_pad = C if C_pad is None else C_pad
	want_hi = (not want_f32 or want_lo) if want_hi is None else want_hi
	hi = torch.empty(B, F_pad, C_pad, dtype = BF16, device = feat.device) if want_hi or want_lo else None
	lo = torch.empty_like(hi) if want_lo else None
	f32 = torch.empty_like(feat) if want_f32 else None
	stats = torch.empty(B, C, 2, dtype = torch.float32, device = feat.device)
	xl = None if xlen is None else xlen.to(torch.float32).contiguous()
	rc = _lib.load().cab_instnorm_pack(
		_p(feat), _p(xl), B, C, F, float(eps), int(bool(normalize)), F_pad, C_pad, _p(hi), _p(lo), _p(f32), _p(stats), _stream()
	)
	_lib.check(rc, 'cab_instnorm_pack')
	return hi, lo, f32


# ------------------------------------------------------------------------------------------
# conv
# ------------------------------------------------------------------------------------------
class Source:
	"""One (activation, packed weight) operand pair of the fused conv GEMM."""

	def __init__(self, act, wgt, C_in, taps, dilation, pad_left, T_in = None, ch_off = 0, w_ch_off = 0):
		# act: bf16 [B, T_rows, ld_ch]; wgt: bf16 [taps, w_rows, w_ld_ch] (both E4M3 for conv1d_fused_fp8)
		assert act.dtype in (BF16, FP8) and wgt.dtype == act.dtype and act.is_contiguous() and wgt.is_contiguous()
		self.act, self.wgt = act, wgt
		self.C_in, self.taps, self.dilation, self.pad_left = C_in, taps, dilation, pad_left
		self.T_in = act.shape[1] if T_in is None else T_in
		self.ch_off, self.w_ch_off = ch_off, w_ch_off

	def to_c(self):
		return _lib.ConvSource(
			self.act.data_ptr(), self.wgt.data_ptr(), self.T_in, self.act.shape[1], self.act.shape[2], self.ch_off,
			self.C_in, self.wgt.shape[1], self.wgt.shape[2], self.w_ch_off, self.taps, self.dilation, self.pad_left
		)


def conv1d_fused(
	sources, B, T_out, C_out, bias = None, act = _lib.ACT_NONE, act_a = 0.0, act_b = 0.0, xlen = None, out_hi = None,
	out_lo = None, logits = None, log_probs = None, argmax = None, epilogue = _lib.EPI_ACT_BF16, block_n = 0, stats = None,
	skip = None, bn_reduce = None
):
	"""skip = (frac [B] fp32, T, margin): output rows t >= ceil(frac[b]*T) + margin are structural zeros (ragged-batch
	padding) -- whole 128-row tiles there are stored as zeros without being computed.
	bn_reduce = (y bf16 [B, T_out, ld] like out_hi, ss fp32 [4, C], C, act, act_a, act_b, xlen or None, partials fp64
	[BN_SUM_REPLICAS, 2, C]): the launch is the dgrad GEMM producing dL/d(out) of a ConvBn1d repeat; its epilogue also
	accumulates that repeat's BatchNorm-backward channel sums (cab_conv_epilogue_t.bnr_*)"""
	_need_cuda(*(s.act for s in sources), bias, xlen, out_hi, out_lo, logits, log_probs, argmax)
	assert all(s.act.dtype == BF16 for s in sources), 'E4M3 sources run on conv1d_fused_fp8'
	n = len(sources)
	arr = (_lib.ConvSource * n)(*[s.to_c() for s in sources])
	ep = _lib.ConvEpilogue()
	ep.B, ep.T_out, ep.C_out, ep.block_n, ep.epilogue, ep.act = B, T_out, C_out, block_n, epilogue, act
	ep.act_a, ep.act_b = float(act_a), float(act_b)
	ep.bias = None if bias is None else bias.data_ptr()
	ep.xlen_frac = None if xlen is None else xlen.data_ptr()
	ep.out_hi = None if out_hi is None else out_hi.data_ptr()
	ep.out_lo = None if out_lo is None else out_lo.data_ptr()
	if out_hi is not None:
		ep.out_T_rows, ep.out_ld_ch = out_hi.shape[1], out_hi.shape[2]
	if epilogue == _lib.EPI_LOGITS_ROWS:  # logits: fp32 [B, T_out, ld] class-contiguous; log_probs slot: fp32 [B, T_out] log-sum-exp
		assert logits is not None and logits.ndim == 3 and logits.is_contiguous() and logits.shape[1] == T_out
		ep.out_T_rows, ep.out_ld_ch = T_out, logits.shape[2]
	ep.logits = None if logits is None else logits.data_ptr()
	ep.log_probs = None if log_probs is None else log_probs.data_ptr()
	ep.argmax = None if argmax is None else argmax.data_ptr()
	ep.stats = None if stats is None else stats.data_ptr()
	if skip is not None:
		_need_cuda(skip[0])
		ep.skip_frac, ep.skip_T, ep.skip_margin = skip[0].data_ptr(), int(skip[1]), int(skip[2])
	if bn_reduce is not None:
		y, ss, C, b_act, b_a, b_b, b_xlen, partials = bn_reduce
		_need_cuda(y, ss, b_xlen, partials)
		assert out_hi is not None and out_lo is None and stats is None and y.shape == out_hi.shape and y.dtype == BF16 and y.is_contiguous()
		assert ss.dtype == torch.float32 and ss.shape == (4, C) and ss.is_contiguous() and partials.dtype == torch.float64 and partials.numel() >= _lib.BN_SUM_REPLICAS * 2 * C
		ep.bnr_y, ep.bnr_ss, ep.bnr_partials = y.data_ptr(), ss.data_ptr(), partials.data_ptr()
		ep.bnr_xlen_frac = None if b_xlen is None else b_xlen.data_ptr()
		ep.bnr_C, ep.bnr_act, ep.bnr_act_a, ep.bnr_act_b = int(C), int(b_act), float(b_a), float(b_b)
	rc = _lib.load().cab_conv1d_fused(arr, n, ctypes.byref(ep), _stream())
	_lib.check(rc, 'cab_conv1d_fused')


def conv1d_fused_fp8(
	sources, B, T_out, C_out, alpha, out_scale_inv = 1.0, bias = None, act = _lib.ACT_NONE, act_a = 0.0, act_b = 0.0, xlen = None,
	out = None, logits = None, log_probs = None, argmax = None, epilogue = _lib.EPI_ACT_BF16, block_n = 0
):
	"""cab_conv1d_fused_fp8: E4M3 sources (weights already carry their source's activation scale over alpha), fp32 alpha
	[C_out] applied to the accumulator before the bias; EPI_ACT_BF16 stores E4M3 `out` [B, T_rows, ld] = act(.) *
	out_scale_inv, the other epilogues write fp32 exactly as in conv1d_fused"""
	_need_cuda(*(s.act for s in sources), alpha, bias, xlen, out, logits, log_probs, argmax)
	assert all(s.act.dtype == FP8 for s in sources) and alpha.dtype == torch.float32 and alpha.is_contiguous() and alpha.numel() >= C_out
	n = len(sources)
	arr = (_lib.ConvSource * n)(*[s.to_c() for s in sources])
	ep = _lib.ConvEpilogue()
	ep.B, ep.T_out, ep.C_out, ep.block_n, ep.epilogue, ep.act = B, T_out, C_out, block_n, epilogue, act
	ep.act_a, ep.act_b = float(act_a), float(act_b)
	ep.bias = None if bias is None else bias.data_ptr()
	ep.xlen_frac = None if xlen is None else xlen.data_ptr()
	if out is not None:
		assert out.dtype == FP8 and out.is_contiguous()
		ep.out_hi = out.data_ptr()
		ep.out_T_rows, ep.out_ld_ch = out.shape[1], out.shape[2]
	if epilogue == _lib.EPI_LOGITS_ROWS:
		assert logits is not None and logits.ndim == 3 and logits.is_contiguous() and logits.shape[1] == T_out
		ep.out_T_rows, ep.out_ld_ch = T_out, logits.shape[2]
	ep.logits = None if logits is None else logits.data_ptr()
	ep.log_probs = None if log_probs is None else log_probs.data_ptr()
	ep.argmax = None if argmax is None else argmax.data_ptr()
	rc = _lib.load().cab_conv1d_fused_fp8(arr, n, ctypes.byref(ep), _p(alpha), float(out_scale_inv), _stream())
	_lib.check(rc, 'cab_conv1d_fused_fp8')


def absmax_bf16(x):
	"""max |x| of a bf16 tensor as a device fp32 [1] (calibration of the FP8 tier)"""
	_need_cuda(x)
	assert x.dtype == BF16 and x.is_contiguous()
	out = torch.empty(1, dtype = torch.float32, device = x.device)
	_lib.check(_lib.load().cab_absmax_bf16(_p(x), x.numel(), _p(out), _stream()), 'cab_absmax_bf16')
	return out


def quantize_e4m3(x, scale):
	"""bf16 -> E4M3 of x / scale, saturating at +-448, same shape"""
	_need_cuda(x)
	assert x.dtype == BF16 and x.is_contiguous()
	out = torch.empty(x.shape, dtype = FP8, device = x.device)
	_lib.check(_lib.load().cab_quantize_e4m3(_p(x), x.numel(), 1.0 / float(scale), _p(out), _stream()), 'cab_quantize_e4m3')
	return out


def conv1d_wgrad(a, a_T, M_total, bx, b_T, N_total, taps, dilation, pad_left, n_splits = 0, skip = None, out = None, alloc = None):
	"""out[tap, m, n] = sum_{b,t} a[b,t,m] * bx[b, t + tap*dilation - pad_left, n]  (fp32 [taps, M, N_ld]);
	skip = (frac [B], T, margin): frames t >= ceil(frac[b]*T) + margin only contribute zeros and are left out;
	out given: the products are ADDED to it (partial products of the split-bf16 tier)"""
	_need_cuda(a, bx)
	assert a.dtype == BF16 and bx.dtype == BF16 and a.is_contiguous() and bx.is_contiguous()
	B = a.shape[0]
	out_ld = (N_total + 3) // 4 * 4
	accumulate = out is not None
	if out is None:
		# alloc: caller-provided allocator (numel -> flat fp32 tensor), e.g. slices of a gradient bucket
		out = alloc(taps * M_total * out_ld).view(taps, M_total, out_ld) if alloc is not None else torch.empty(taps, M_total, out_ld, dtype = torch.float32, device = a.device)
	rc = _lib.load().cab_conv1d_wgrad(
		_p(a), a_T, a.shape[1], a.shape[2], M_total, _p(bx), b_T, bx.shape[1], bx.shape[2], N_total, B, taps, dilation, pad_left,
		_p(out), out_ld, n_splits, _p(skip[0]) if skip is not None else None, int(skip[1]) if skip is not None else 0,
		int(skip[2]) if skip is not None else 0, int(accumulate), _stream()
	)
	_lib.check(rc, 'cab_conv1d_wgrad')
	return out  # [taps, M_total, ld >= N_total]; columns past N_total are padding


def grouped_conv1d(act, T, C_in, wgt, bias, groups, pad_left, ld_out = None, act_lo = None, want_lo = False, relu = True, T_out = None):
	"""grouped conv (+ bias + ReLU): bf16 channels-last [B, T_rows, ld_in] -> [B, T, ld_out]; T frames in and out"""
	_need_cuda(act, act_lo, wgt, bias)
	B, T_rows, ld_in = act.shape
	C_out, _, k = wgt.shape
	assert T_out is None or T_out == T, 'grouped conv keeps the frame count (odd kernel, same padding)'
	out = torch.empty(B, T, ld_out or C_out, dtype = BF16, device = act.device)
	out_lo = torch.empty_like(out) if want_lo else None
	rc = _lib.load().cab_grouped_conv1d(
		_p(act), _p(act_lo if want_lo else None), B, T, T_rows, C_in, ld_in, _p(wgt), _p(bias), C_out, groups, k, pad_left, _p(out), _p(out_lo),
		out.shape[1], out.shape[2], int(bool(relu)), _stream()
	)
	_lib.check(rc, 'cab_grouped_conv1d')
	return out, out_lo


def grouped_conv1d_relu(act, T, C_in, wgt, bias, groups, pad_left, ld_out = None, act_lo = None, want_lo = False):
	return grouped_conv1d(act, T, C_in, wgt, bias, groups, pad_left, ld_out = ld_out, act_lo = act_lo, want_lo = want_lo, relu = True)


def grouped_conv1d_fp8(act, T, C_in, in_scale, wgt, bias, groups, pad_left, ld_out, out_scale):
	"""grouped conv + bias + ReLU of the FP8 tier: E4M3 [B, T_rows, ld_in] (value = q * in_scale) -> E4M3 [B, T, ld_out]
	(value / out_scale, saturating)"""
	_need_cuda(act, wgt, bias)
	assert act.dtype == FP8 and act.is_contiguous()
	B, T_rows, ld_in = act.shape
	C_out, _, k = wgt.shape
	out = torch.empty(B, T, ld_out, dtype = FP8, device = act.device)
	rc = _lib.load().cab_grouped_conv1d_fp8(
		_p(act), B, T, T_rows, C_in, ld_in, float(in_scale), _p(wgt), _p(bias), C_out, groups, k, pad_left, _p(out), out.shape[1], out.shape[2],
		1.0 / float(out_scale), _stream()
	)
	_lib.check(rc, 'cab_grouped_conv1d_fp8')
	return out


def grouped_conv1d_wgrad(dy, T, x, x_T, C_in, C_out, groups, k, pad_left, db = None):
	"""dy, x: engine._Act-like (hi, lo) bf16 channels-last; returns dW fp32 [C_out, C_in / groups, k]; db (fp32 [C_out]) is filled"""
	_need_cuda(dy.hi, x.hi)
	assert T == x_T
	B = dy.hi.shape[0]
	dw = torch.empty(C_out, C_in // groups, k, dtype = torch.float32, device = dy.hi.device)
	rc = _lib.load().cab_grouped_conv1d_wgrad(
		_p(dy.hi), _p(dy.lo), dy.hi.shape[1], dy.hi.shape[2], _p(x.hi), _p(x.lo if dy.lo is not None else None), B, T, x.hi.shape[1], C_in, x.hi.shape[2], C_out, groups, k, pad_left,
		_p(dw), _p(db), _stream()
	)
	_lib.check(rc, 'cab_grouped_conv1d_wgrad')
	return dw


# ------------------------------------------------------------------------------------------
# log_softmax / decode
# ------------------------------------------------------------------------------------------
def log_softmax_argmax(logits, want_log_probs = True, want_argmax = True):
	_need_cuda(logits)
	logits = logits.to(torch.float32).contiguous()
	B, C, T = logits.shape
	lp = torch.empty_like(logits) if want_log_probs else None
	am = torch.empty(B, T, dtype = torch.int32, device = logits.device) if want_argmax else None
	rc = _lib.load().cab_log_softmax_argmax(_p(logits), 0, B, C, T, _p(lp), _p(am), _stream())
	_lib.check(rc, 'cab_log_softmax_argmax')
	return lp, am


def large_vocab_head(sources, B, T_out, C, bias, alpha = None):
	"""Decoder 1x1 conv + log_softmax + argmax for large vocabularies (models.py:26,316; transcript_generators.py:27):
	one GEMM launch whose epilogue writes the fp32 logits once (class-contiguous rows, TMA stores) and keeps an online
	softmax per frame across the N tiles, then one streaming pass log_probs = logits - lse.  Returns (logits, log_probs,
	argmax) with logits / log_probs as [B, C, T] VIEWS of class-contiguous [B, T, C] memory.  alpha given: E4M3 sources
	(conv1d_fused_fp8)."""
	dev = sources[0].act.device
	ld = (C + 3) // 4 * 4
	logits = torch.empty(B, T_out, ld, dtype = torch.float32, device = dev)
	lse = torch.empty(B, T_out, dtype = torch.float32, device = dev)
	argmax = torch.empty(B, T_out, dtype = torch.int32, device = dev)
	if alpha is None:
		conv1d_fused(sources, B, T_out, C, bias = bias, logits = logits, log_probs = lse, argmax = argmax, epilogue = _lib.EPI_LOGITS_ROWS)
	else:
		conv1d_fused_fp8(sources, B, T_out, C, alpha, bias = bias, logits = logits, log_probs = lse, argmax = argmax, epilogue = _lib.EPI_LOGITS_ROWS)
	log_probs = torch.empty_like(logits)
	rc = _lib.load().cab_log_softmax_rows(_p(logits), _p(lse), B * T_out, C, ld, _p(log_probs), _stream())
	_lib.check(rc, 'cab_log_softmax_rows')
	return logits[:, :, :C].permute(0, 2, 1), log_probs[:, :, :C].permute(0, 2, 1), argmax


class _LogSoftmaxDim1(torch.autograd.Function):
	@staticmethod
	def forward(ctx, logits):
		lp, _ = log_softmax_argmax(logits, want_argmax = False)
		ctx.save_for_backward(lp)
		ctx.in_dtype = logits.dtype
		return lp

	@staticmethod
	def backward(ctx, grad_out):
		lp, = ctx.saved_tensors
		B, C, T = lp.shape
		go = grad_out.to(torch.float32).contiguous()
		gi = torch.empty_like(lp)
		rc = _lib.load().cab_log_softmax_bwd(_p(lp), _p(go), B, C, T, _p(gi), _stream())
		_lib.check(rc, 'cab_log_softmax_bwd')
		return gi.to(ctx.in_dtype)


def log_softmax_dim1(logits):
	"""F.log_softmax(logits, dim=1).to(float32) for [B, C, T] (models.py:316), differentiable."""
	return _LogSoftmaxDim1.apply(logits)


def topk_ids(log_probs, K):
	_need_cuda(log_probs)
	log_probs = log_probs.to(torch.float32).contiguous()
	B, C, T = log_probs.shape
	out = torch.empty(B, K, T, dtype = torch.int32, device = log_probs.device)
	rc = _lib.load().cab_topk_ids(_p(log_probs), B, C, T, K, _p(out), _stream())
	_lib.check(rc, 'cab_topk_ids')
	return out


def greedy_collapse(ids, lengths, num_classes, eps_id, space_id, is_silence, is_word_start, blank_amount_to_space):
	"""ids int32 [B,T]; returns (tokens [B,T], frames [B,T], counts [B]) int32 on device."""
	_need_cuda(ids, lengths, is_silence, is_word_start)
	ids = ids.to(torch.int32).contiguous()
	B, T = ids.shape
	ln = None if lengths is None else lengths.to(torch.int32).contiguous()
	tok = torch.empty(B, T, dtype = torch.int32, device = ids.device)
	frm = torch.empty(B, T, dtype = torch.int32, device = ids.device)
	cnt = torch.empty(B, dtype = torch.int32, device = ids.device)
	rc = _lib.load().cab_greedy_collapse(
		_p(ids), _p(ln), B, T, num_classes, eps_id, space_id, _p(is_silence), _p(is_word_start),
		blank_amount_to_space, _p(tok), _p(frm), T, _p(cnt), _stream()
	)
	_lib.check(rc, 'cab_greedy_collapse')
	return tok, frm, cnt


def top2_probs(log_probs):
	"""fp32 [B, C, T] (any strides) -> fp32 [B, 2, T]: the two largest probabilities per frame"""
	_need_cuda(log_probs)
	lp = log_probs if log_probs.dtype == torch.float32 else log_probs.float()
	B, C, T = lp.shape
	out = torch.empty(B, 2, T, dtype = torch.float32, device = lp.device)
	rc = _lib.load().cab_top2_probs(_p(lp), lp.stride(0), lp.stride(1), lp.stride(2), B, C, T, _p(out), _stream())
	_lib.check(rc, 'cab_top2_probs')
	return out


BEAM_MAX_WIDTH = 128  # beams per utterance the search kernel holds in shared memory
BEAM_MAX_CLASSES = 64  # classes per frame after pruning (min(cutoff_top_n, C))


def ctc_beam_search(log_probs, output_lengths = None, beam_width = 100, cutoff_top_n = 40, cutoff_prob = 1.0, topk = 1, blank = None, lm = None,
					alpha = 0.0, beta = 0.0):
	"""CTC prefix beam search on fp32 [B, C, T] log_probs (any strides, e.g. the class-contiguous views of the
	large-vocabulary head).  blank None: C - 1.  Returns device tensors (tokens int32 [B, topk, T], frames int32
	[B, topk, T], lengths int32 [B, topk], scores fp32 [B, topk]): the topk most probable hypotheses best first, the frame at
	which each token was emitted, and log(p_blank + p_nonblank) at the last frame (-inf, length 0 where the search kept fewer
	than topk hypotheses).  Tokens and frames are -1 past each hypothesis' length.

	lm: an lm.NGramLM built for these labels and this blank.  Then only prefixes spelling words of the LM's vocabulary are
	searched, a space that ends word w adds alpha * ln P(w | previous words) + beta, the last word gets the same term
	(alpha * -1000 + beta if it is incomplete) and the scores are these fused ones (csrc/beam.cu, cab_ctc_beam_search_lm)."""
	_need_cuda(log_probs)
	lp = log_probs if log_probs.dtype == torch.float32 else log_probs.float()
	B, C, T = lp.shape
	blank = C - 1 if blank is None else int(blank)
	N = min(int(cutoff_top_n), C)
	W, K = int(beam_width), int(topk)
	dev = lp.device
	if output_lengths is None:
		olen = torch.full((B, ), T, dtype = torch.int64, device = dev)
	else:
		olen = torch.as_tensor(output_lengths, device = dev).to(torch.int64).contiguous()
	if B == 0 or T == 0:  # nothing to search: the empty hypothesis, probability one
		tokens = torch.full((B, K, T), -1, dtype = torch.int32, device = dev)
		scores = torch.full((B, K), -math.inf, dtype = torch.float32, device = dev)
		scores[:, 0] = 0.0
		return tokens, tokens.clone(), torch.zeros(B, K, dtype = torch.int32, device = dev), scores
	lib = _lib.load()
	nbytes = ctypes.c_int64()
	_lib.check(lib.cab_ctc_beam_search_workspace(B, T, C, N, W, K, blank, float(cutoff_prob), ctypes.byref(nbytes)), 'cab_ctc_beam_search_workspace')
	ws = torch.empty(nbytes.value, dtype = torch.uint8, device = dev)
	tokens = torch.empty(B, K, T, dtype = torch.int32, device = dev)
	frames = torch.empty_like(tokens)
	lengths = torch.empty(B, K, dtype = torch.int32, device = dev)
	scores = torch.empty(B, K, dtype = torch.float32, device = dev)
	if lm is None:
		rc = lib.cab_ctc_beam_search(
			_p(lp), lp.stride(0), lp.stride(1), lp.stride(2), _p(olen), B, T, C, N, float(cutoff_prob), blank, W, K, _p(ws), nbytes.value,
			_p(tokens), _p(frames), T, _p(lengths), _p(scores), _stream()
		)
		_lib.check(rc, 'cab_ctc_beam_search')
	else:
		if lm.blank != blank:
			raise ValueError(f'convasr_b200: the LM was built with blank={lm.blank}, the search uses blank={blank}')
		rc = lib.cab_ctc_beam_search_lm(
			_p(lp), lp.stride(0), lp.stride(1), lp.stride(2), _p(olen), B, T, C, N, float(cutoff_prob), blank, W, K, _p(ws), nbytes.value,
			_p(tokens), _p(frames), T, _p(lengths), _p(scores), ctypes.byref(lm.device_struct(dev)), float(alpha), float(beta), lm.space,
			_stream()
		)
		_lib.check(rc, 'cab_ctc_beam_search_lm')
	return tokens, frames, lengths, scores


def entropy(log_probs, lengths = None, eps_id = -1):
	_need_cuda(log_probs, lengths)
	log_probs = log_probs.to(torch.float32).contiguous()
	B, C, T = log_probs.shape
	e = torch.empty(B, dtype = torch.float32, device = log_probs.device)
	w = torch.empty(B, dtype = torch.float32, device = log_probs.device)
	ln = None if lengths is None else lengths.to(torch.int64).contiguous()
	rc = _lib.load().cab_entropy(_p(log_probs), _p(ln), B, C, T, eps_id, _p(e), _p(w), _stream())
	_lib.check(rc, 'cab_entropy')
	return e, w


# ------------------------------------------------------------------------------------------
# CTC
# ------------------------------------------------------------------------------------------
def _tbc_strides(log_probs):
	# log_probs is addressed as [T, B, C] through its strides (any permuted view works)
	assert log_probs.ndim == 3 and log_probs.dtype == torch.float32
	return log_probs.stride(0), log_probs.stride(1), log_probs.stride(2)


def _ctc_args(log_probs, targets, input_lengths, target_lengths):
	_need_cuda(log_probs, targets, input_lengths, target_lengths)
	T, B, C = log_probs.shape
	targets = targets.to(torch.int64).contiguous()
	if targets.ndim != 2:
		raise ValueError('convasr_b200.ctc: targets must be padded [B, L]')
	input_lengths = torch.as_tensor(input_lengths, device = log_probs.device).to(torch.int64).contiguous()
	target_lengths = torch.as_tensor(target_lengths, device = log_probs.device).to(torch.int64).contiguous()
	return T, B, C, targets.shape[1], targets, input_lengths, target_lengths


class _CtcLoss(torch.autograd.Function):
	@staticmethod
	def forward(ctx, log_probs, targets, input_lengths, target_lengths, blank, states_per_cta):
		lp = log_probs if log_probs.dtype == torch.float32 else log_probs.float()
		T, B, C, L, targets, input_lengths, target_lengths = _ctc_args(lp, targets, input_lengths, target_lengths)
		S = 2 * L + 1
		lib = _lib.load()
		ctx.blank = blank
		ctx.in_dtype = log_probs.dtype
		ctx.states_per_cta = states_per_cta
		if states_per_cta is not None or not lib.cab_ctc_loss_one_cta_covers(L):
			# one thread-block cluster per utterance: alpha is stored only when a gradient will be wanted, beta is
			# recomputed by the backward
			alpha = None
			if ctx.needs_input_grad[0]:
				nbytes = ctypes.c_int64()
				_lib.check(lib.cab_ctc_loss_long_workspace(B, T, L, ctypes.byref(nbytes)), 'cab_ctc_loss_long_workspace')
				alpha = torch.empty(nbytes.value // 4, dtype = torch.float32, device = lp.device)
			nll = torch.empty(B, dtype = torch.float32, device = lp.device)
			offsets = torch.empty(B, 2, (T + 7) // 8 + 2, dtype = torch.float64, device = lp.device)
			st, sb, sc = _tbc_strides(lp)
			rc = lib.cab_ctc_loss_long_fwd(
				_p(lp), st, sb, sc, _p(targets), _p(input_lengths), _p(target_lengths), B, T, C, L, blank, _p(alpha), _p(offsets),
				_p(nll), int(states_per_cta or 0), _stream()
			)
			_lib.check(rc, 'cab_ctc_loss_long_fwd')
			ctx.cluster = True
			ctx.save_for_backward(lp, targets, input_lengths, target_lengths, alpha, offsets)
			return nll
		alpha = torch.empty(B, T, S, dtype = torch.float32, device = lp.device)
		# when a gradient will be wanted, alpha and beta run concurrently in one launch
		beta = torch.empty_like(alpha) if ctx.needs_input_grad[0] else None
		nll = torch.empty(B, dtype = torch.float32, device = lp.device)
		offsets = torch.empty(B, 2, (T + 7) // 8 + 2, dtype = torch.float64, device = lp.device)
		st, sb, sc = _tbc_strides(lp)
		rc = _lib.load().cab_ctc_loss_fwd(
			_p(lp), st, sb, sc, _p(targets), _p(input_lengths), _p(target_lengths), B, T, C, L, blank, _p(alpha),
			_p(beta), _p(offsets), _p(nll), _stream()
		)
		_lib.check(rc, 'cab_ctc_loss_fwd')
		ctx.beta = beta
		ctx.save_for_backward(lp, targets, input_lengths, target_lengths, alpha, offsets)
		ctx.cluster = False
		return nll

	@staticmethod
	def backward(ctx, grad_out):
		lp, targets, input_lengths, target_lengths, alpha, offsets = ctx.saved_tensors
		T, B, C = lp.shape
		L = targets.shape[1]
		if ctx.cluster:
			grad = torch.empty_strided(lp.shape, lp.stride(), dtype = torch.float32, device = lp.device)
			st, sb, sc = _tbc_strides(lp)
			go = grad_out.to(torch.float32).contiguous()
			rc = _lib.load().cab_ctc_loss_long_bwd(
				_p(lp), st, sb, sc, _p(targets), _p(input_lengths), _p(target_lengths), B, T, C, L, ctx.blank, _p(alpha), _p(offsets),
				_p(go), _p(grad), grad.stride(0), grad.stride(1), grad.stride(2), int(ctx.states_per_cta or 0), _stream()
			)
			_lib.check(rc, 'cab_ctc_loss_long_bwd')
			return grad.to(ctx.in_dtype), None, None, None, None, None
		beta_ready = ctx.beta is not None
		beta = ctx.beta if beta_ready else torch.empty_like(alpha)
		ctx.beta = None
		# gradient laid out like log_probs' memory (keeps [B,C,T]-permuted views coalesced)
		grad = torch.empty_strided(lp.shape, lp.stride(), dtype = torch.float32, device = lp.device)
		st, sb, sc = _tbc_strides(lp)
		go = grad_out.to(torch.float32).contiguous()
		rc = _lib.load().cab_ctc_loss_bwd(
			_p(lp), st, sb, sc, _p(targets), _p(input_lengths), _p(target_lengths), B, T, C, L, ctx.blank, _p(alpha),
			_p(beta), int(beta_ready), _p(offsets), _p(go), _p(grad), grad.stride(0), grad.stride(1), grad.stride(2), _stream()
		)
		_lib.check(rc, 'cab_ctc_loss_bwd')
		return grad.to(ctx.in_dtype), None, None, None, None, None


def ctc_loss(log_probs, targets, input_lengths, target_lengths, blank = 0, _states_per_cta = None):
	"""F.ctc_loss(log_probs[T,B,C], targets[B,L], ..., reduction='none', zero_infinity=False).  Targets up to 1345 labels
	run on one CTA per utterance and direction; longer ones (up to 65535 labels) on a thread-block cluster per utterance,
	with one fp32 [B, T, 2L+1] workspace when a gradient is wanted and none for the loss alone -- the same nll bit for bit
	wherever both run.  _states_per_cta (tests only) forces the cluster path with that slice size (0: the library's choice)."""
	return _CtcLoss.apply(log_probs, targets, input_lengths, target_lengths, int(blank), _states_per_cta)


_FP16_TABLES = {}


def _fp16_tables(device):
	"""exp and log of every fp16 value as computed by this host's torch, as uint16 bit patterns on the device: with them the
	fp16 alignment recursion equals the reference's fp16 arithmetic on this machine bit for bit (ctc.cu: half_fn)"""
	key = str(device)
	if key not in _FP16_TABLES:
		x = torch.arange(65536, dtype = torch.int32).to(torch.int16).view(torch.float16)
		bits = lambda t: t.view(torch.int16).to(torch.int32).bitwise_and(0xFFFF).to(torch.uint16)
		_FP16_TABLES[key] = (bits(x.exp()).to(device), bits(x.log()).to(device))
	return _FP16_TABLES[key]


CTC_ALIGN_CTA_STATES = 4096  # 2 * L_max + 1 up to which one CTA per utterance aligns (cab_ctc_alignment)


def ctc_alignment(log_probs, targets, input_lengths, target_lengths, blank = 0, _states_per_cta = None):
	"""fp16 log_probs: the recursion rounds to fp16 after every operation, as the reference does on an fp16 tensor (the
	values are handed to the kernel as their exact fp32 images).  Targets up to 2047 labels run on one CTA per utterance
	with a byte per back-pointer; longer ones (up to 65535 labels) on a thread-block cluster per utterance with 2-bit
	back-pointers -- the same result wherever both run.  _states_per_cta (tests only) forces the cluster path with that
	slice size (0: the library's choice)."""
	half = log_probs.dtype == torch.float16
	lp = log_probs if log_probs.dtype == torch.float32 else log_probs.float()
	T, B, C, L, targets, input_lengths, target_lengths = _ctc_args(lp, targets, input_lengths, target_lengths)
	S = 2 * L + 1
	lib = _lib.load()
	cluster = _states_per_cta is not None or S > CTC_ALIGN_CTA_STATES
	out = torch.empty(B, L, dtype = torch.int64, device = lp.device)
	if B == 0 or L == 0:
		return out.zero_()
	if cluster:
		nbytes = ctypes.c_int64()
		_lib.check(lib.cab_ctc_alignment_long_workspace(B, T, L, ctypes.byref(nbytes)), 'cab_ctc_alignment_long_workspace')
		bp = torch.empty(nbytes.value, dtype = torch.uint8, device = lp.device)
	else:
		bp = torch.empty(B, T, S, dtype = torch.uint8, device = lp.device)
	st, sb, sc = _tbc_strides(lp)
	tabs = _fp16_tables(lp.device) if half else (None, None)
	args = (_p(lp), st, sb, sc, _p(targets), _p(input_lengths), _p(target_lengths), B, T, C, L, blank, _p(bp), _p(out), int(half),
			_p(tabs[0]), _p(tabs[1]))
	if cluster:
		_lib.check(lib.cab_ctc_alignment_long(*args, int(_states_per_cta or 0), _stream()), 'cab_ctc_alignment_long')
	else:
		_lib.check(lib.cab_ctc_alignment(*args, _stream()), 'cab_ctc_alignment')
	return out
