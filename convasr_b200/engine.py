"""Inference engine: turns the parameters of a JasperNet-family module tree into a list of
fused-kernel launches (cab_conv1d_fused and friends) and runs them.

What the reference does per ConvBn1d repeat -- conv, BatchNorm, residual 1x1 convs + their
BatchNorms, add, activation, temporal mask (models.py:127-139) -- is ONE launch here:
BatchNorm is folded into the weights on the host exactly as nn.utils.fusion.fuse_conv_bn_eval
does for models.py:141-151, residual branches become extra K-segments of the same GEMM, and
bias/activation/mask run in the TMEM epilogue.

HBM layout: activations are bf16 channels-last [B, T, C_alloc] (C_alloc = C rounded up to 64),
weights are bf16 tap-major [taps, C_out, C_in_alloc].  The "fp32" precision tier keeps every
activation and weight as a (hi, lo) bf16 pair and accumulates hi*hi + hi*lo + lo*hi in fp32.

The "fp8" tier (inference only) stores every activation as E4M3 with one static fp32 scale per tensor (from a
calibration run of the bf16 plan, keyed by the launch that produces the tensor) and every weight as E4M3 with one
scale per output channel.  The sources of a launch share one accumulator: source j's weights absorb its input scale s_j,
W~_j = e4m3(W_j * s_j / alpha[n]) with alpha[n] = max_j(s_j * max|W_j[n]|) / 448, and the epilogue multiplies by
alpha[n].  Contracted widths are multiples of 128 there (C_alloc = C rounded up to 128).
"""
import torch
import torch.nn as nn

from . import _lib, ops

BF16 = torch.bfloat16
FP8 = torch.float8_e4m3fn
E4M3_MAX = 448.0


def _ceil_to(x, m):
	return (x + m - 1) // m * m


def _split(x):
	hi = x.to(BF16)
	lo = (x - hi.to(torch.float32)).to(BF16)
	return hi, lo


def fold_bn(conv_w, conv_b, bn):
	"""conv followed by eval-mode BatchNorm == conv with scaled weights and a bias
	(same algebra as torch.nn.utils.fusion.fuse_conv_bn_eval used at models.py:145,150)."""
	w = conv_w.detach().to(torch.float32)
	b = conv_b.detach().to(torch.float32) if conv_b is not None else torch.zeros(w.shape[0], device = w.device)
	if isinstance(bn, nn.modules.batchnorm._BatchNorm):
		if bn.running_mean is None:
			raise RuntimeError('convasr_b200: BatchNorm without running statistics cannot be folded')
		gamma = bn.weight.detach().float() if bn.weight is not None else torch.ones_like(bn.running_mean)
		beta = bn.bias.detach().float() if bn.bias is not None else torch.zeros_like(bn.running_mean)
		scale = gamma * torch.rsqrt(bn.running_var.detach().float() + bn.eps)
		w = w * scale.reshape(-1, 1, 1)
		b = (b - bn.running_mean.detach().float()) * scale + beta
	return w, b


def pack_taps(w, c_in_alloc):
	"""[C_out, C_in, k] fp32 -> fp32 tap-major [k, C_out, c_in_alloc] (zero padded channels)."""
	C_out, C_in, k = w.shape
	out = torch.zeros(k, C_out, c_in_alloc, dtype = torch.float32, device = w.device)
	out[:, :, :C_in] = w.permute(2, 0, 1)
	return out


def pack_taps_stride2(w, pad, c_in_alloc):
	"""Stride-2 conv as a stride-1 conv over the frame-pair view [B, F/2, 2*c_in_alloc]:
	out[t] = sum_k w[k] x[2t + k - pad];  with j = k - pad = 2*dp + q (q in {0,1}) the tap dp
	reads pair t+dp, channel block q.  Returns (weights [taps, C_out, 2*c_in_alloc], taps, pad_left)."""
	C_out, C_in, k = w.shape
	dp_min = (0 - pad) // 2
	dp_max = (k - 1 - pad) // 2
	taps = dp_max - dp_min + 1
	out = torch.zeros(taps, C_out, 2 * c_in_alloc, dtype = torch.float32, device = w.device)
	for kk in range(k):
		j = kk - pad
		dp = j // 2
		q = j - 2 * dp
		out[dp - dp_min, :, q * c_in_alloc:q * c_in_alloc + C_in] = w[:, :, kk]
	return out, taps, -dp_min


_ACT_CODES = {'relu': _lib.ACT_RELU, 'hardtanh': _lib.ACT_HARDTANH, 'leaky_relu': _lib.ACT_LEAKY_RELU}


def act_code(nonlinearity):
	if nonlinearity is None:
		return _lib.ACT_NONE, 0.0, 0.0
	name = nonlinearity[0]
	if name not in _ACT_CODES:
		raise NotImplementedError(f'convasr_b200: nonlinearity {nonlinearity!r} has no fused epilogue')
	if name == 'hardtanh':
		return _ACT_CODES[name], float(nonlinearity[1]), float(nonlinearity[2])
	if name == 'leaky_relu':
		return _ACT_CODES[name], float(nonlinearity[1]) if len(nonlinearity) > 1 else 0.01, 0.0
	return _ACT_CODES[name], 0.0, 0.0


def e4m3(x):
	"""fp32 -> E4M3 with saturation at +-448 (torch's float8_e4m3fn cast turns values past the largest finite into NaN;
	cvt.rn.satfinite, which the kernels use, clamps)"""
	return x.clamp(-E4M3_MAX, E4M3_MAX).to(FP8)


def fp8_scale(amax):
	"""per-tensor activation scale: x / scale spans the E4M3 range; an all-zero tensor gets 1"""
	amax = float(amax)
	return amax / E4M3_MAX if amax > 0 else 1.0


def quantize_sources_fp8(ws, scales):
	"""E4M3 weights of one launch's sources sharing an accumulator.  ws: fp32 packed weights [taps, rows, c_in] (rows may
	differ), scales: the input scale of each source.  Returns ([W~_j], alpha fp32 [max rows]) with
	alpha[n] = max_j(s_j * max|W_j[n]|) / 448 (1 where every weight of row n is zero) and W~_j = e4m3(W_j * s_j / alpha[n])."""
	rows = max(w.shape[1] for w in ws)
	peak = torch.zeros(rows, dtype = torch.float32, device = ws[0].device)
	for w, s in zip(ws, scales):
		peak[:w.shape[1]] = torch.maximum(peak[:w.shape[1]], w.abs().amax(dim = (0, 2)) * s)
	alpha = torch.where(peak > 0, peak / E4M3_MAX, torch.ones_like(peak))
	return [e4m3(w * (s / alpha[:w.shape[1]]).view(1, -1, 1)).contiguous() for w, s in zip(ws, scales)], alpha.contiguous()


class _Weights:
	"""a packed weight in the active precision tier ('fp8': the fp32 packing is kept until the plan quantises it)"""

	def __init__(self, w_f32, fp32_tier):
		if fp32_tier == 'fp8':
			self.f32, self.hi, self.lo = w_f32, None, None
		elif fp32_tier:
			self.hi, self.lo = _split(w_f32)
			self.hi, self.lo = self.hi.contiguous(), self.lo.contiguous()
		else:
			self.hi, self.lo = w_f32.to(BF16).contiguous(), None


class _Act:
	"""an activation tensor in the active precision tier: bf16 [B, T, C_alloc] (+ lo)"""

	def __init__(self, hi, lo, T, C):
		self.hi, self.lo, self.T, self.C = hi, lo, T, C


class _Gemm:
	"""one operand pair of a fused launch: which activation, which weight, conv geometry"""

	def __init__(self, src, weights, c_in_alloc, taps, dilation, pad_left, pair_view = False):
		self.src = src  # 'x' (running activation), 'tmp' (grouped conv output) or residual index
		self.weights, self.c_in_alloc, self.taps, self.dilation, self.pad_left = weights, c_in_alloc, taps, dilation, pad_left
		self.pair_view = pair_view


class _Launch:
	def __init__(self):
		self.gemms = []
		self.bias = None
		self.act = (_lib.ACT_NONE, 0.0, 0.0)
		self.mask = False
		self.C_out = 0  # real channels
		self.C_alloc = 0
		self.dT = 0  # T_out - T_in for stride 1
		self.stride2 = None  # (k, pad) of the original strided conv
		self.grouped = None  # (weight fp32, bias fp32, groups, pad_left, C_mid, C_mid_alloc)
		self.epilogue = _lib.EPI_ACT_BF16
		self.key = self.tmp_key = None  # calibration keys of the output / grouped-conv activation
		self.alpha = None  # fp8 tier: per-column accumulator multiplier [C_alloc]
		self.in_scale = self.tmp_scale = self.out_scale = 1.0  # fp8 tier: scales of the running input, grouped output, output


def next_residuals(i, n_blocks, plan, residuals, x):
	"""residual bookkeeping of JasperNet.forward after block i (models.py:306-313)"""
	if i >= n_blocks - plan.num_epilogue_modules - 1:
		return []
	if plan.residual_mode == 'dense':
		return residuals + [x]
	if plan.residual_mode:
		return [x]
	return []


class StackPlan:
	"""Packed weights + launch list for backbone and decoder of one model, one precision tier."""

	_epochs = 0

	def __init__(self, model, fp32_tier, fp8_scales = None):
		"""fp8_scales: {activation key: scale} from a calibration run (JasperNet.calibrate_fp8) selects the fp8 tier"""
		StackPlan._epochs += 1
		self.epoch = StackPlan._epochs  # monotonically increasing identity (id() can be reused after a plan is freed)
		self.fp8 = fp8_scales is not None
		self.fp32_tier = fp32_tier and not self.fp8
		self._wmode = 'fp8' if self.fp8 else self.fp32_tier
		self.align = 128 if self.fp8 else 64  # channel allocation granularity (one 128-byte swizzle row of the operand)
		self.blocks = []  # list of list of _Launch (one list per ConvBn1d)
		self.residual_mode = model.residual
		self.num_epilogue_modules = model.num_epilogue_modules
		for block in model.backbone:
			self.blocks.append(self._plan_convbn(block))
		self.heads = self._plan_decoder(model.decoder)
		# the features are packed 64 wide for a stride-2 prologue (its frame-pair view is then 128 wide), else like every activation
		self.feat_align = 64 if self.blocks[0][0].stride2 is not None else self.align
		self._assign_keys()
		if self.fp8:
			self._quantize_fp8(fp8_scales)

	def _assign_keys(self):
		"""name every activation by the launch that produces it ('feat' for the packed features); record each source's key"""
		x, residuals = 'feat', []
		for i, launches in enumerate(self.blocks):
			for j, L in enumerate(launches):
				L.key, L.tmp_key, L.in_key = ('block', i, j), ('grouped', i, j), x
				for g in L.gemms:
					g.in_key = x if g.src == 'x' else L.tmp_key if g.src == 'tmp' else residuals[g.src]
				x = L.key
			residuals = next_residuals(i, len(self.blocks), self, residuals, x)
		for h, chain in enumerate(self.heads):
			hx = x
			for j, L in enumerate(chain):
				L.key, L.tmp_key, L.in_key = ('head', h, j), ('head_grouped', h, j), hx
				for g in L.gemms:
					g.in_key = hx if g.src == 'x' else L.tmp_key
				hx = L.key

	def launches(self):
		return [L for launches in self.blocks for L in launches] + [L for chain in self.heads for L in chain]

	def _quantize_fp8(self, scales):
		missing = sorted({g.in_key for L in self.launches() for g in L.gemms if g.in_key not in scales}, key = str)
		if missing:
			raise RuntimeError(f'convasr_b200: no fp8 calibration scale for activations {missing}; call model.calibrate_fp8(x, xlen)')
		for L in self.launches():
			wq, alpha = quantize_sources_fp8([g.weights.f32 for g in L.gemms], [scales[g.in_key] for g in L.gemms])
			for g, w in zip(L.gemms, wq):
				g.weights.hi, g.weights.f32 = w, None
			L.alpha = torch.cat([alpha, torch.ones(max(L.C_alloc - alpha.numel(), 0), device = alpha.device)]).contiguous()
			L.in_scale = scales[L.in_key]
			L.tmp_scale = scales.get(L.tmp_key, 1.0)
			L.out_scale = scales.get(L.key, 1.0)

	# -- planning ---------------------------------------------------------------------------
	def _plan_convbn(self, m, final_logits = False, mask = None):
		launches = []
		n_rep = len(m.conv)
		for j in range(n_rep):
			L = _Launch()
			seq = m.conv[j]
			first = seq[0]
			k, stride, dil = first.kernel_size[0], first.stride[0], first.dilation[0]
			pad = first.padding[0]
			C_in, C_out = first.in_channels, seq[-1].out_channels
			c_in_alloc = _ceil_to(C_in, 64 if stride == 2 else self.align)  # stride 2: the pair view doubles it
			L.C_out, L.C_alloc = C_out, _ceil_to(C_out, self.align)
			L.dT = 2 * pad - dil * (k - 1)
			bias = torch.zeros(L.C_alloc, dtype = torch.float32, device = first.weight.device)
			if len(seq) == 3:  # separable: grouped conv + bias + ReLU, then pointwise (+BN)
				if stride != 1 or dil != 1:
					raise NotImplementedError('convasr_b200: strided/dilated separable conv')
				C_mid = first.out_channels
				c_mid_alloc = _ceil_to(C_mid, self.align)
				gb = first.bias.detach().float().contiguous() if first.bias is not None else None
				L.grouped = (first.weight.detach().float().contiguous(), gb, first.groups, pad, C_mid, c_mid_alloc, C_in)
				w, b = fold_bn(seq[2].weight, seq[2].bias, m.bn[j])
				L.gemms.append(_Gemm('tmp', _Weights(pack_taps(w, c_mid_alloc), self._wmode), c_mid_alloc, 1, 1, 0))
			else:
				if first.groups != 1:
					raise NotImplementedError('convasr_b200: grouped non-separable conv')
				w, b = fold_bn(first.weight, first.bias, m.bn[j])
				if stride == 2:
					if dil != 1:
						raise NotImplementedError('convasr_b200: dilated strided conv')
					wp, taps, pad_left = pack_taps_stride2(w, pad, c_in_alloc)
					L.stride2 = (k, pad)
					L.gemms.append(_Gemm('x', _Weights(wp, self._wmode), 2 * c_in_alloc, taps, 1, pad_left, pair_view = True))
				elif stride == 1:
					L.gemms.append(_Gemm('x', _Weights(pack_taps(w, c_in_alloc), self._wmode), c_in_alloc, k, dil, pad))
				else:
					raise NotImplementedError(f'convasr_b200: conv stride {stride}')
			bias[:C_out] += b
			if j == n_rep - 1:
				for r, (rc, rbn) in enumerate(zip(m.conv_residual, m.bn_residual)):
					if isinstance(rc, nn.Identity):  # 'flat' residual: identity 1x1
						w = torch.eye(C_out, device = bias.device).unsqueeze(-1)
						L.gemms.append(_Gemm(r, _Weights(pack_taps(w, L.C_alloc), self._wmode), L.C_alloc, 1, 1, 0))
					else:
						w, b = fold_bn(rc.weight, rc.bias, rbn)
						rc_in_alloc = _ceil_to(rc.in_channels, self.align)
						L.gemms.append(_Gemm(r, _Weights(pack_taps(w, rc_in_alloc), self._wmode), rc_in_alloc, 1, 1, 0))
						bias[:C_out] += b
			L.bias = bias.contiguous()
			act = m.activation.nonlinearity
			L.act = act_code(act)
			if L.act[0] in (_lib.ACT_NONE, ) and L.C_alloc != L.C_out:
				pass
			L.mask = bool(m.temporal_mask) if mask is None else mask
			launches.append(L)
		return launches

	def _plan_decoder(self, decoder):
		heads = []
		conv0 = decoder[0]
		L = _Launch()
		w, b = fold_bn(conv0.weight, conv0.bias, None)
		c_in_alloc = _ceil_to(conv0.in_channels, self.align)
		L.gemms.append(_Gemm('x', _Weights(pack_taps(w, c_in_alloc), self._wmode), c_in_alloc, conv0.kernel_size[0], 1, conv0.padding[0]))
		L.bias = b.contiguous()
		L.C_out = L.C_alloc = conv0.out_channels
		L.dT = 2 * conv0.padding[0] - (conv0.kernel_size[0] - 1)
		L.epilogue = _lib.EPI_LOGSOFTMAX if conv0.out_channels <= 256 else _lib.EPI_LOGITS_F32
		heads.append([L])
		if getattr(decoder, 'type', None) == 'bpe':
			chain = []
			for i, cb in enumerate(decoder[1]):
				chain += self._plan_convbn(cb, mask = False)  # Decoder passes no lengths (models.py:43)
			last = chain[-1]
			last.epilogue = _lib.EPI_LOGITS_F32
			last.C_alloc = last.C_out
			last.bias = last.bias[:last.C_out].contiguous()
			heads.append(chain)
		return heads

	# -- execution --------------------------------------------------------------------------
	def _sources(self, L, x, tmp, residuals):
		srcs = []
		for g in L.gemms:
			a = x if g.src == 'x' else tmp if g.src == 'tmp' else residuals[g.src]
			hi, lo = a.hi, a.lo
			T_in = a.T
			if g.pair_view:
				B, T_rows, C = hi.shape
				hi = hi.view(B, T_rows // 2, 2 * C)
				lo = lo.view(B, T_rows // 2, 2 * C) if lo is not None else None
				T_in = T_rows // 2
			srcs.append(ops.Source(hi, g.weights.hi, g.c_in_alloc, g.taps, g.dilation, g.pad_left, T_in = T_in))
			if self.fp32_tier:
				srcs.append(ops.Source(hi, g.weights.lo, g.c_in_alloc, g.taps, g.dilation, g.pad_left, T_in = T_in))
				if lo is not None:
					srcs.append(ops.Source(lo, g.weights.hi, g.c_in_alloc, g.taps, g.dilation, g.pad_left, T_in = T_in))
		return srcs

	def _fold_excess_sources(self, srcs, B, T_out, C_alloc, dev):
		"""more operand pairs than one launch has K segments (dense 'Big' models in the split tier: 10 branches x 3 products):
		the first groups run as plain linear launches (no bias / activation / mask) and re-enter the last launch as identity
		K segments of their (hi, lo) partial sum"""
		eye = None
		while len(srcs) > _lib.MAX_CONV_SOURCES:
			room = _lib.MAX_CONV_SOURCES - 4  # leave room for the identity segments of the running partial sum
			now, srcs = srcs[:room], srcs[room:]
			part_hi = torch.empty(B, T_out, C_alloc, dtype = BF16, device = dev)
			part_lo = torch.empty_like(part_hi) if self.fp32_tier else None
			ops.conv1d_fused(now, B, T_out, C_alloc, out_hi = part_hi, out_lo = part_lo)
			if eye is None:
				eye = torch.eye(C_alloc, dtype = BF16, device = dev).unsqueeze(0).contiguous()
			srcs = [ops.Source(part_hi, eye, C_alloc, 1, 1, 0, T_in = T_out)] + ([ops.Source(part_lo, eye, C_alloc, 1, 1, 0, T_in = T_out)] if part_lo is not None else []) + srcs
		return srcs

	def _run_launch(self, L, x, residuals, xlen, B, observe = None):
		dev = x.hi.device
		tmp = None
		if L.grouped is not None:
			gw, gb, groups, gpad, C_mid, c_mid_alloc, C_in = L.grouped
			if self.fp8:
				t_hi, t_lo = ops.grouped_conv1d_fp8(x.hi, x.T, C_in, L.in_scale, gw, gb, groups, gpad, c_mid_alloc, L.tmp_scale), None
			else:
				t_hi, t_lo = ops.grouped_conv1d_relu(x.hi, x.T, C_in, gw, gb, groups, gpad, ld_out = c_mid_alloc, act_lo = x.lo, want_lo = self.fp32_tier)
			tmp = _Act(t_hi, t_lo, x.T, C_mid)
			if observe is not None:
				observe(L.tmp_key, t_hi)
		if L.stride2 is not None:
			k, pad = L.stride2
			T_out = (x.T + 2 * pad - (k - 1) - 1) // 2 + 1
		else:
			T_out = x.T + L.dT
		return self.run_gemm(L, self._sources(L, x, tmp, residuals), xlen if L.mask else None, B, T_out, dev)

	def run_gemm(self, L, srcs, xlen, B, T_out, dev):
		"""the fused GEMM of launch L over its operand pairs `srcs` and its epilogue: an _Act, or per head (logits, log_probs,
		argmax); xlen: the temporal mask (None: none)"""
		code, a, b = L.act
		if self.fp8:
			return self._run_epilogue_fp8(L, srcs, xlen, B, T_out, dev)
		if L.epilogue == _lib.EPI_ACT_BF16:
			srcs = self._fold_excess_sources(srcs, B, T_out, L.C_alloc, dev)
			out_hi = torch.empty(B, T_out, L.C_alloc, dtype = BF16, device = dev)
			out_lo = torch.empty_like(out_hi) if self.fp32_tier else None
			ops.conv1d_fused(srcs, B, T_out, L.C_alloc, bias = L.bias, act = code, act_a = a, act_b = b, xlen = xlen, out_hi = out_hi, out_lo = out_lo)
			return _Act(out_hi, out_lo, T_out, L.C_out)
		if L.epilogue == _lib.EPI_LOGSOFTMAX or code != _lib.ACT_NONE:
			logits = torch.empty(B, L.C_out, T_out, dtype = torch.float32, device = dev)
		if L.epilogue == _lib.EPI_LOGSOFTMAX:
			log_probs = torch.empty_like(logits)
			argmax = torch.empty(B, T_out, dtype = torch.int32, device = dev)
			ops.conv1d_fused(srcs, B, T_out, L.C_out, bias = L.bias, logits = logits, log_probs = log_probs, argmax = argmax, epilogue = _lib.EPI_LOGSOFTMAX)
		elif code == _lib.ACT_NONE:
			return ops.large_vocab_head(srcs, B, T_out, L.C_out, L.bias)  # head 0 with a large vocabulary: fused online softmax
		else:  # the 'bpe' second head ends in ConvBn1d's activation (models.py:27-33): logits = act(.), then a separate log_softmax
			ops.conv1d_fused(srcs, B, T_out, L.C_out, bias = L.bias, act = code, act_a = a, act_b = b, logits = logits, epilogue = _lib.EPI_LOGITS_F32)
			log_probs, argmax = ops.log_softmax_argmax(logits)
		return logits, log_probs, argmax

	def _run_epilogue_fp8(self, L, srcs, xlen, B, T_out, dev):
		if len(srcs) > _lib.MAX_CONV_SOURCES:
			raise NotImplementedError(f'convasr_b200: {len(srcs)} operand pairs in one fp8 launch (at most {_lib.MAX_CONV_SOURCES})')
		code, a, b = L.act
		if L.epilogue == _lib.EPI_ACT_BF16:
			out = torch.empty(B, T_out, L.C_alloc, dtype = FP8, device = dev)
			ops.conv1d_fused_fp8(srcs, B, T_out, L.C_alloc, L.alpha, 1.0 / L.out_scale, bias = L.bias, act = code, act_a = a, act_b = b, xlen = xlen, out = out)
			return _Act(out, None, T_out, L.C_out)
		if L.epilogue == _lib.EPI_LOGSOFTMAX:
			logits = torch.empty(B, L.C_out, T_out, dtype = torch.float32, device = dev)
			log_probs = torch.empty_like(logits)
			argmax = torch.empty(B, T_out, dtype = torch.int32, device = dev)
			ops.conv1d_fused_fp8(srcs, B, T_out, L.C_out, L.alpha, bias = L.bias, logits = logits, log_probs = log_probs, argmax = argmax, epilogue = _lib.EPI_LOGSOFTMAX)
		elif code == _lib.ACT_NONE:
			return ops.large_vocab_head(srcs, B, T_out, L.C_out, L.bias, alpha = L.alpha)
		else:
			logits = torch.empty(B, L.C_out, T_out, dtype = torch.float32, device = dev)
			ops.conv1d_fused_fp8(srcs, B, T_out, L.C_out, L.alpha, bias = L.bias, act = code, act_a = a, act_b = b, logits = logits, epilogue = _lib.EPI_LOGITS_F32)
			log_probs, argmax = ops.log_softmax_argmax(logits)
		return logits, log_probs, argmax

	def run(self, feats, xlen, observe = None):
		"""feats: _Act holding the normalised features [B, F_pad, C_alloc] (E4M3 in the fp8 tier, already divided by the
		'feat' scale); returns per head (logits, log_probs, argmax).  observe(key, tensor): called with every activation the
		plan produces (calibration)."""
		B = feats.hi.shape[0]
		x = feats
		if observe is not None:
			observe('feat', feats.hi)
		residuals = []
		n_blocks = len(self.blocks)
		for i, launches in enumerate(self.blocks):
			for L in launches:
				x = self._run_launch(L, x, residuals, xlen, B, observe)
				if observe is not None:
					observe(L.key, x.hi)
			residuals = next_residuals(i, n_blocks, self, residuals, x)
		outs = []
		for chain in self.heads:
			h = x
			for L in chain:
				h = self._run_launch(L, h, [], None, B, observe)
				if observe is not None and isinstance(h, _Act):
					observe(L.key, h.hi)
			outs.append(h)
		return outs


def params_signature(module):
	"""cheap fingerprint of every parameter/buffer: plans are rebuilt when anything changes"""
	return tuple((t.data_ptr(), t._version, t.dtype) for t in list(module.parameters()) + list(module.buffers()))
