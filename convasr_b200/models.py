"""Drop-in replacement for the reference's `models` module (acoustic-model hot path only).

Same public surface as the reference (SURVEY.md section 8b): `getattr(models, name)(num_input_features,
num_classes, dropout=, decoder_type=, frontend=, dict=, ...)`, `model(x, xlen, y=, ylen=)` returning
`dict(logits=[...], log_probs=[...], olen=[...], loss=...)`, `fuse_conv_bn_eval`, `freeze`, the
same sub-module names and therefore the same `state_dict` keys -- but in eval mode `forward`
runs entirely on hand-written sm_100a kernels through the C ABI (convasr_b200/engine.py):
fused log-mel frontend, masked instance norm, one tcgen05 implicit-GEMM launch per ConvBn1d
repeat with BatchNorm folded and residual/activation/mask in the epilogue, the decoder 1x1
fused with log_softmax + argmax, and the CTC loss.

Training mode (`model.train()`) runs forward AND backward of the same module tree on this repo's kernels
(convasr_b200/training.py: batch-statistics BatchNorm, residual / dense / separable topologies, dgrad, wgrad);
there is no ATen / cuDNN path and no CPU path: tensors must be CUDA tensors.

Reference sites are cited per class (paths relative to the reference root).
"""
import math
import os
import typing

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import engine, ops

# ------------------------------------------------------------------------------------------
# frontend
# ------------------------------------------------------------------------------------------


def slaney_mel_basis(sample_rate, n_fft, n_mels, fmin = 0.0, fmax = None):
	"""The mel basis the reference obtains from librosa.filters.mel at models.py:521-523
	(Slaney mel scale, Slaney area normalisation), computed here in float64."""
	fmax = sample_rate / 2.0 if fmax is None else float(fmax)
	lin_step = 200.0 / 3.0
	knee_hz = 1000.0
	knee_mel = knee_hz / lin_step
	log_step = math.log(6.4) / 27.0

	def to_mel(hz):
		hz = np.asarray(hz, dtype = np.float64)
		return np.where(hz < knee_hz, hz / lin_step, knee_mel + np.log(np.maximum(hz, 1e-30) / knee_hz) / log_step)

	def to_hz(mel):
		mel = np.asarray(mel, dtype = np.float64)
		return np.where(mel < knee_mel, mel * lin_step, knee_hz * np.exp((mel - knee_mel) * log_step))

	bins = np.linspace(0.0, sample_rate / 2.0, n_fft // 2 + 1)
	edges = to_hz(np.linspace(to_mel(fmin), to_mel(fmax), n_mels + 2))
	rising = (bins[None, :] - edges[:-2, None]) / (edges[1:-1] - edges[:-2])[:, None]
	falling = (edges[2:, None] - bins[None, :]) / (edges[2:] - edges[1:-1])[:, None]
	tri = np.clip(np.minimum(rising, falling), 0.0, None)
	tri *= (2.0 / (edges[2:] - edges[:-2]))[:, None]
	return torch.from_numpy(tri.astype(np.float32))


class LogFilterBankFrontend(nn.Module):
	"""models.py:486-603.  Buffers/params keep the reference names: `window`, `mel.weight`
	[n_mels, n_freq, 1], `mel.bias` (= eps), and `stft.weight` in stft_mode='conv'."""

	def __init__(
		self, out_channels, sample_rate, window_size, window_stride, window, dither = 1e-5, dither0 = 0.0,
		preemphasis = 0.97, eps = torch.finfo(torch.float16).tiny, normalize_signal = True,
		debug_short_long_records_normalize_signal_multiplier = 1.0, stft_mode = None, window_periodic = True,
		normalize_features = False, **kwargs
	):
		super().__init__()
		self.debug_short_long_records_normalize_signal_multiplier = debug_short_long_records_normalize_signal_multiplier
		self.stft_mode = stft_mode
		self.dither, self.dither0 = dither, dither0  # accepted, unused -- as in the reference (:571,574)
		self.preemphasis = preemphasis
		self.normalize_signal = normalize_signal
		self.sample_rate = sample_rate
		self.win_length = int(window_size * sample_rate)
		self.hop_length = int(window_stride * sample_rate)
		self.nfft = 2**math.ceil(math.log2(self.win_length))
		self.freq_cutoff = self.nfft // 2 + 1
		self.register_buffer('window', getattr(torch, window)(self.win_length, periodic = window_periodic).float())
		basis = slaney_mel_basis(sample_rate, self.nfft, out_channels, 0.0, int(sample_rate / 2))
		self.mel = nn.Conv1d(basis.shape[1], basis.shape[0], 1).requires_grad_(False)
		with torch.no_grad():
			self.mel.weight.copy_(basis.unsqueeze(-1))
			self.mel.bias.fill_(eps)
		if stft_mode == 'conv':
			# kept for state_dict compatibility (models.py:548-561); the arithmetic is the same DFT
			fourier = torch.view_as_real(torch.fft.fft(torch.eye(self.nfft), dim = 1))
			forward_basis = fourier[:self.freq_cutoff].permute(2, 0, 1).reshape(-1, 1, self.nfft)
			off = (self.nfft - self.win_length) // 2
			wpad = F.pad(self.window, (off, self.nfft - self.win_length - off))
			self.stft = nn.Conv1d(1, forward_basis.shape[0], self.nfft, bias = False, stride = self.hop_length).requires_grad_(False)
			with torch.no_grad():
				self.stft.weight.copy_(forward_basis * wpad)
		else:
			self.stft = None
		self._tables = None

	def _device_tables(self, device):
		sig = (self.mel.weight.data_ptr(), self.mel.weight._version, self.mel.bias.data_ptr(), self.mel.bias._version, self.window.data_ptr(), str(device))
		if self._tables is None or self._tables[0] != sig:
			mel = self.mel.weight.detach().squeeze(-1).to(device = device, dtype = torch.float32).contiguous()
			log_eps = float(self.mel.bias[0])  # one D2H read when the tables are (re)built, never per call
			self._tables = (sig, mel, ops.make_mel_band(mel), ops.make_twiddle(self.nfft, device), self.window.detach().to(device = device, dtype = torch.float32).contiguous(), log_eps)
		return self._tables[1:]

	def forward(self, signal, mask = None, xlen = None, **kwargs):
		"""signal [B, T] int16/float; mask [B, T] bool as built by JasperNet.forward (models.py:290)
		or, preferably, the fractions `xlen` themselves.  Returns fp32 [B, n_mels, T // hop + 1]."""
		assert signal.ndim == 2
		if not signal.is_cuda:
			raise RuntimeError('convasr_b200: LogFilterBankFrontend runs on CUDA only (no CPU fallback); move the signal to the GPU / use --frontend-in-model')
		T = signal.shape[1]
		if xlen is None and mask is not None:
			# recover exact lengths from the prefix mask; n/T rounds so that ceil(fp32(n/T)*T) == n for n <= 2^23
			n = mask.reshape(mask.shape[0], -1).sum(dim = -1).to(torch.float32)
			xlen = (n - 0.5) / T
		mel, band, twiddle, window, log_eps = self._device_tables(signal.device)
		return ops.frontend_logmel(
			signal, xlen, window, mel, band, twiddle, self.hop_length, self.nfft, preemphasis = self.preemphasis,
			log_eps = log_eps, normalize_signal = self.normalize_signal,
			denom_multiplier = self.debug_short_long_records_normalize_signal_multiplier
		)

	def features(self, signal, xlen, norm, F_pad_even, C_pad, want_lo):
		"""signal -> instance-normalised bf16 channels-last features in one native call (what JasperNet.forward does at
		models.py:286-301); norm: the model's MaskedInstanceNorm1d or None"""
		mel, band, twiddle, window, log_eps = self._device_tables(signal.device)
		Fr = signal.shape[1] // self.hop_length + 1
		F_pad = Fr + (Fr % 2) if F_pad_even else Fr
		hi, lo, _ = ops.frontend_features(
			signal, xlen, window, mel, band, twiddle, self.hop_length, self.nfft, self.preemphasis, log_eps, self.normalize_signal,
			self.debug_short_long_records_normalize_signal_multiplier, norm is not None, norm is not None and norm.temporal_mask, norm.eps if norm is not None else 0.0,
			F_pad, C_pad, want_lo = want_lo
		)
		return hi, lo, Fr

	@staticmethod
	def compute_output_shape(time_dim_length, kernel_size, stride, padding, dilation = 1):
		return int(math.floor((time_dim_length + 2 * padding - dilation * (kernel_size - 1) - 1) / stride + 1))


def compute_output_lengths(x, lengths_fraction = None):
	"""models.py:611-614"""
	if lengths_fraction is None:
		return torch.full(x.shape[:1], x.shape[-1], device = x.device, dtype = torch.long)
	return (lengths_fraction * x.shape[-1]).ceil().long()


def temporal_mask(x, lengths):
	"""models.py:617-619"""
	return (torch.arange(x.shape[-1], device = x.device, dtype = lengths.dtype).unsqueeze(0) < lengths.unsqueeze(1)).view(x.shape[:1] + (1, ) * (len(x.shape) - 2) + x.shape[-1:])


def normalize_signal(signal, dim = -1, eps = 1e-5, denom_multiplier = 1.0):
	"""models.py:684-686 (host-side helper; the model path fuses this into the frontend kernel)"""
	signal_max = signal.abs().max(dim = dim, keepdim = True).values + eps
	return signal / (signal_max * denom_multiplier) if signal.numel() > 0 else signal


class MaskedInstanceNorm1d(nn.InstanceNorm1d):
	"""models.py:688-719; forward runs the native stats + normalise kernels."""

	def __init__(self, *args, temporal_mask = False, legacy = True, **kwargs):
		super().__init__(*args, **kwargs)
		self.temporal_mask = temporal_mask
		self.legacy = legacy

	def forward(self, x, mask = None, xlen = None):
		if self.track_running_stats or self.affine:
			raise NotImplementedError('convasr_b200: instance norm with running stats / affine parameters is not built')
		if self.temporal_mask and xlen is None and mask is not None:
			n = mask.reshape(mask.shape[0], -1).sum(dim = -1).to(torch.float32)
			xlen = (n - 0.5) / x.shape[-1]
		_, _, out = ops.instnorm_pack(x, xlen if self.temporal_mask else None, self.eps, want_f32 = True)
		return out


# ------------------------------------------------------------------------------------------
# conv blocks (parameter containers with the reference's names; compute lives in engine.py)
# ------------------------------------------------------------------------------------------


class ConvSamePadding(nn.Sequential):
	"""models.py:47-77: `padding = dilation * kernel_size // 2`; separable = grouped conv (with
	bias) -> ReLU -> pointwise conv."""

	def __init__(self, in_channels, out_channels, kernel_size, stride, dilation, bias, groups, separable):
		padding = dilation * kernel_size // 2
		if separable:
			assert dilation == 1
			layers = [
				nn.Conv1d(in_channels, out_channels, kernel_size = kernel_size, stride = stride, padding = padding, dilation = dilation, groups = groups),
				nn.ReLU(inplace = True),
				nn.Conv1d(out_channels, out_channels, kernel_size = 1, bias = bias)
			]
		else:
			layers = [nn.Conv1d(in_channels, out_channels, kernel_size = kernel_size, stride = stride, padding = padding, dilation = dilation, groups = groups, bias = bias)]
		super().__init__(*layers)


class ResidualActivation(nn.Module):
	"""models.py:350-371 (non-invertible form): y += residuals; nonlinearity; dropout."""

	def __init__(self, nonlinearity, dropout = 0, invertible = False):
		super().__init__()
		self.nonlinearity = nonlinearity
		self.dropout = dropout
		self.invertible = invertible

	def forward(self, y, residual: typing.List = []):
		for r in residual:
			y = y + r
		if self.dropout > 0 and self.training and self.nonlinearity[0] == 'relu':
			return relu_dropout(y, p = self.dropout, training = True)
		y = getattr(F, self.nonlinearity[0])(y, *self.nonlinearity[1:])
		return F.dropout(y, p = self.dropout, training = self.training)

	def extra_repr(self):
		return f'nonlinearity={self.nonlinearity}, dropout={self.dropout}, invertible={self.invertible}'


def relu_dropout(x, p = 0, inplace = False, training = False):
	"""models.py:436-443"""
	if not training or p == 0:
		return x.clamp(min = 0)
	keep = 1 - p
	drop = (torch.rand_like(x) > keep) | (x < 0)
	return x.masked_fill(drop, 0).div(keep)


class ConvBn1d(nn.Module):
	"""models.py:80-151.  Sub-module names (`conv`, `bn`, `conv_residual`, `bn_residual`) fix the
	state_dict keys; JasperNet.forward launches the fused kernel plan (eval) or the native training graph."""

	def __init__(
		self, num_channels, kernel_size, stride = 1, dropout = 0, groups = 1, num_channels_residual: typing.List = [],
		repeat = 1, dilation = 1, separable = False, temporal_mask = True, nonlinearity = ('relu', ),
		nonlinearity_reference = True, batch_norm_momentum = 0.1, inplace = False
	):
		super().__init__()
		c_in, c_out = num_channels
		self.conv = nn.ModuleList([
			ConvSamePadding(c_in if i == 0 else c_out, c_out, kernel_size = kernel_size, stride = stride, dilation = dilation, separable = separable, bias = False, groups = groups)
			for i in range(repeat)
		])
		self.bn = nn.ModuleList([nn.BatchNorm1d(c_out, momentum = batch_norm_momentum) for i in range(repeat)])
		self.conv_residual = nn.ModuleList([nn.Identity() if c is None else nn.Conv1d(c, c_out, kernel_size = 1) for c in num_channels_residual])
		self.bn_residual = nn.ModuleList([nn.Identity() if c is None else nn.BatchNorm1d(c_out, momentum = batch_norm_momentum) for c in num_channels_residual])
		self.activation = ResidualActivation(nonlinearity, dropout, invertible = inplace)
		self.temporal_mask = temporal_mask

	def forward(self, x, lengths_fraction = None, residual: typing.List = []):
		raise NotImplementedError('convasr_b200: ConvBn1d is a parameter container; it runs as part of JasperNet.forward (fused launches in eval mode, convasr_b200/training.py in training mode)')

	def fuse_conv_bn_eval(self):
		"""models.py:141-151: fold each BatchNorm into the conv before it and replace it by Identity
		(state_dict then carries `.bias` on the fused convs and no `bn.*` entries)."""
		for i in range(len(self.conv_residual)):
			conv, bn = self.conv_residual[i], self.bn_residual[i]
			if not isinstance(conv, nn.Identity) and not isinstance(bn, nn.Identity):
				self.conv_residual[i] = _fused_conv(conv, bn)
				self.bn_residual[i] = nn.Identity()
		for i in range(len(self.conv)):
			if not isinstance(self.bn[i], nn.Identity):
				self.conv[i][-1] = _fused_conv(self.conv[i][-1], self.bn[i])
				self.bn[i] = nn.Identity()


def _fused_conv(conv, bn):
	w, b = engine.fold_bn(conv.weight, conv.bias, bn)
	fused = nn.Conv1d(conv.in_channels, conv.out_channels, conv.kernel_size[0], stride = conv.stride[0], padding = conv.padding[0], dilation = conv.dilation[0], groups = conv.groups, bias = True)
	fused = fused.to(device = conv.weight.device, dtype = conv.weight.dtype)
	with torch.no_grad():
		fused.weight.copy_(w)
		fused.bias.copy_(b)
	fused.weight.requires_grad_(conv.weight.requires_grad)
	return fused


class Decoder(nn.Sequential):
	"""models.py:23-44: head 0 = 1x1 conv to num_classes[0]; 'bpe' adds two ConvBn1d(k=15)."""

	def __init__(self, input_size, num_classes, type = None):
		if type is None:
			super().__init__(nn.Conv1d(input_size, num_classes[0], kernel_size = 1))
		elif type == 'bpe':
			super().__init__(
				nn.Conv1d(input_size, num_classes[0], kernel_size = 1),
				nn.Sequential(ConvBn1d(num_channels = (input_size, input_size), kernel_size = 15), ConvBn1d(num_channels = (input_size, num_classes[1]), kernel_size = 15))
			)
		else:
			raise ValueError(f'unknown decoder type {type!r}')
		self.type = type

	def forward(self, x):
		if self.type is None:
			return (self[0](x), )
		return self[0](x), self[1](x)


# ------------------------------------------------------------------------------------------
# the network
# ------------------------------------------------------------------------------------------


class JasperNet(nn.Module):
	"""models.py:158-347.  Prologue (stride `stride1`) + 5 blocks x num_subblocks x `repeat` +
	2-module epilogue + Decoder."""

	def __init__(
		self, num_input_features, num_classes, repeat = 3, num_subblocks = 1, dilation = 1, residual = 'dense',
		kernel_sizes = [11, 13, 17, 21, 25], kernel_size_prologue = 11, kernel_size_epilogue = 29, base_width = 128,
		out_width_factors = [2, 3, 4, 5, 6], out_width_factors_large = [7, 8], separable = False, groups = 1, dropout = 0,
		dropout_prologue = 0.2, dropout_epilogue = 0.4, dropouts = [0.2, 0.2, 0.2, 0.3, 0.3], temporal_mask = True,
		nonlinearity = ('relu', ), inplace = False, stride1 = 2, stride2 = 1, decoder_type = None, dict = dict,
		frontend = None, bpe_only = False, normalize_features = True,
		normalize_features_eps = torch.finfo(torch.float16).tiny, normalize_features_track_running_stats = False,
		normalize_features_legacy = True, normalize_features_temporal_mask = True, check_time_dim_padded = True,
		precision = None
	):
		super().__init__()
		self.init_params = {name: repr(value) for name, value in locals().items()}
		if dropout == 0:
			dropout_prologue = dropout_epilogue = 0
			dropouts = [0] * len(dropouts)
		common = {'temporal_mask': temporal_mask, 'nonlinearity': nonlinearity, 'inplace': inplace}  # NB `dict` is a ctor argument here
		width = out_width_factors[0] * base_width
		blocks = [ConvBn1d(num_channels = (num_input_features, width), kernel_size = kernel_size_prologue, dropout = dropout_prologue, stride = stride1, **common)]
		skip_widths = []
		for k, p_drop, factor in zip(kernel_sizes, dropouts, out_width_factors):  # zip truncates (Wav2Letter passes 6 kernels)
			for s in range(num_subblocks):
				c_out = factor * base_width if s == num_subblocks - 1 else width
				if residual == 'dense':
					skip_widths = skip_widths + [width]
				elif residual == 'flat':
					skip_widths = [None]
				elif residual:
					skip_widths = [width]
				else:
					skip_widths = []
				blocks.append(ConvBn1d(num_channels = (width, c_out), kernel_size = k, dropout = p_drop, repeat = repeat, separable = separable, groups = groups, num_channels_residual = list(skip_widths), **common))
				# NB the reference keeps the *input* width for all sub-blocks of a block (models.py:216-219)
			width = factor * base_width
		w7, w8 = out_width_factors_large[0] * base_width, out_width_factors_large[1] * base_width
		blocks.append(ConvBn1d(num_channels = (width, w7), kernel_size = kernel_size_epilogue, dropout = dropout_epilogue, dilation = dilation, **common))
		blocks.append(ConvBn1d(num_channels = (w7, w8), kernel_size = 1, dropout = dropout_epilogue, **common))
		self.backbone = nn.ModuleList(blocks)
		self.num_epilogue_modules = 2
		self.frontend = frontend
		self.normalize_features = MaskedInstanceNorm1d(
			num_input_features, affine = False, eps = normalize_features_eps, track_running_stats = normalize_features_track_running_stats,
			temporal_mask = normalize_features_temporal_mask, legacy = normalize_features_legacy
		) if normalize_features else None
		self.decoder = Decoder(w8, num_classes, type = decoder_type)
		self.residual = residual
		self.dict = dict
		self.bpe_only = bpe_only
		self.check_time_dim_padded = check_time_dim_padded
		self.precision = precision  # None = follow the parameter dtype; 'bf16' | 'fp32' | 'fp8' (eval only)
		self._plan = None
		self._fp8_calibration = None  # (parameter signature, {activation key: scale}); deliberately not in state_dict
		self._graphs_enabled = os.environ.get('CONVASR_B200_CUDA_GRAPHS', '0') == '1'
		self._graphs_max = 4
		self._graphs = {}

	# -- precision tier -------------------------------------------------------------------
	def set_precision(self, precision):
		"""'bf16': single bf16 operands (speed tier).  'fp32': split-bf16 hi/lo operands with fp32
		accumulation (matches the reference's fp32 path to ~1e-5).  'fp8': eval-only serving tier, E4M3
		activations and weights with fp32 accumulation; needs calibrate_fp8() first.  None: decide from the
		parameter dtype (fp32 params -> 'fp32', half/bfloat16 params -> 'bf16')."""
		assert precision in (None, 'bf16', 'fp32', 'fp8')
		self.precision = precision
		self._plan = None
		return self

	def _active_precision(self):
		p = self.precision or os.environ.get('CONVASR_B200_PRECISION')
		if p:
			return p
		w = self.decoder[0].weight
		return 'fp32' if w.dtype == torch.float32 else 'bf16'

	def train(self, mode = True):
		if mode and self._active_precision() == 'fp8':
			raise RuntimeError("convasr_b200: the fp8 tier is inference only (there is no fp8 training); call set_precision('bf16') or set_precision('fp32') before model.train()")
		return super().train(mode)

	def _params_sig(self):
		# _state_epoch: bumped by everything that writes parameters / running statistics through raw pointers without
		# touching a tensor version (native training forward, CUDA-graph replays of a training step)
		return (getattr(self, '_state_epoch', 0), engine.params_signature(self.backbone), engine.params_signature(self.decoder))

	def _get_plan(self):
		prec = self._active_precision()
		sig = (prec, ) + self._params_sig()
		if self._plan is None or self._plan[0] != sig:
			scales = None
			if prec == 'fp8':
				if self._fp8_calibration is None:
					raise RuntimeError('convasr_b200: the fp8 tier needs activation scales; call model.calibrate_fp8(x, xlen) first')
				if self._fp8_calibration[0] != self._params_sig():
					raise RuntimeError('convasr_b200: parameters or running statistics changed since the fp8 calibration; call model.calibrate_fp8(x, xlen) again')
				scales = self._fp8_calibration[1]
			with torch.no_grad():
				self._plan = (sig, engine.StackPlan(self, fp32_tier = prec == 'fp32', fp8_scales = scales))
		return self._plan[1]

	@torch.no_grad()
	def calibrate_fp8(self, x, xlen = None):
		"""Static activation scales of the fp8 tier: runs the bf16 plan once on (x, xlen) -- inputs as for forward -- and
		records max |a| of every activation it produces (features, every launch output, every grouped-conv output) with
		one abs-max kernel each; scale = max / 448.  The scales belong to the current parameters: after a training step or
		any parameter change the fp8 forward raises until this is called again.  They are not part of state_dict."""
		if not x.is_cuda:
			raise RuntimeError('convasr_b200: model inputs must be CUDA tensors (there is no CPU fallback)')
		if xlen is not None:
			xlen = xlen.to(device = x.device, dtype = torch.float32).contiguous()
		if self.frontend is not None:
			x = x.squeeze(1) if x.ndim == 3 else x
		plan = engine.StackPlan(self, fp32_tier = False)
		keys, amax = [], []

		def observe(key, t):
			keys.append(key)
			amax.append(ops.absmax_bf16(t))

		hi, _, Fr, C = self._packed_features(x, xlen, False)
		plan.run(engine._Act(hi, None, Fr, C), xlen, observe = observe)
		values = torch.cat(amax).tolist()  # one device -> host copy
		self._fp8_calibration = (self._params_sig(), {k: engine.fp8_scale(v) for k, v in zip(keys, values)})
		self._plan = None
		self._graphs = {}
		return self

	# -- forward --------------------------------------------------------------------------
	def forward(self, x, xlen = None, y = None, ylen = None):
		if not x.is_cuda:
			raise RuntimeError('convasr_b200: model inputs must be CUDA tensors (there is no CPU fallback)')
		if xlen is not None:
			xlen = xlen.to(device = x.device, dtype = torch.float32).contiguous()
		if self.frontend is not None:
			assert (not self.check_time_dim_padded) or (x.shape[-1] % (32 / 2) == 0), 'Shape of input signal is not divisible by 16 '
			x = x.squeeze(1) if x.ndim == 3 else x
			n_frames = x.shape[-1] // self.frontend.hop_length + 1
		else:
			assert x.ndim == 3
			n_frames = x.shape[-1]
		assert (not self.check_time_dim_padded) or (n_frames % 32 == 0), 'Shape of features after frontend is not divisible by 32'

		if self.training:
			if self._active_precision() == 'fp8':
				raise RuntimeError("convasr_b200: the fp8 tier is inference only (there is no fp8 training); call model.eval()")
			from . import training
			why = training.unsupported_reason(self)
			if why is not None:
				raise NotImplementedError(f'convasr_b200: training of this module tree is not built ({why}); there is no ATen / cuDNN fallback')
			logits, log_probs = training.forward_training(self, x, xlen)  # frontend, conv/BN forward + backward on this repo's kernels
		else:
			logits, log_probs = self._forward_native(x, xlen)
		olen = [compute_output_lengths(l, xlen) for l in logits]
		aux = {}
		if y is not None and ylen is not None:
			loss = []
			for i, l in enumerate(log_probs):
				nll = ops.ctc_loss(l.permute(2, 0, 1), y[:, i], olen[i], ylen[:, i], blank = l.shape[1] - 1)
				loss.append(nll / ylen[:, 0])  # models.py:323
			aux = dict(loss = sum(loss) if not self.bpe_only else sum(loss[1:]))
		return self.dict(logits = logits, log_probs = log_probs, olen = olen, **aux)

	# -- CUDA graphs ------------------------------------------------------------------------
	def enable_cuda_graphs(self, enabled = True, max_cached = 4):
		"""Eval-mode forward as one CUDA-graph replay per (input shape, dtype, mask on/off): removes the
		host launch gaps between the ~25 short kernels of a step.  Inputs are copied into static buffers
		and outputs are cloned out, so semantics equal the eager path.  Opt-in because every distinct
		input shape costs one capture and one private memory pool."""
		self._graphs_enabled = bool(enabled)
		self._graphs_max = max_cached
		self._graphs = {}
		return self

	def _graphed_raw(self, x, xlen):
		plan = self._get_plan()
		key = (tuple(x.shape), x.dtype, xlen is not None, plan.epoch, x.device.index)
		entry = self._graphs.get(key)
		if entry is None:
			if len(self._graphs) >= self._graphs_max:
				self._graphs.pop(next(iter(self._graphs)))
			static_x = x.clone()
			static_xlen = xlen.clone() if xlen is not None else None
			side = torch.cuda.Stream(device = x.device)
			side.wait_stream(torch.cuda.current_stream())
			with torch.cuda.stream(side):
				for _ in range(2):
					self._raw_to_outputs(static_x, static_xlen)
			torch.cuda.current_stream().wait_stream(side)
			graph = torch.cuda.CUDAGraph()
			with torch.cuda.graph(graph):
				outs = self._raw_to_outputs(static_x, static_xlen)
			entry = (graph, static_x, static_xlen, outs)
			self._graphs[key] = entry
		graph, static_x, static_xlen, outs = entry
		static_x.copy_(x, non_blocking = True)
		if xlen is not None:
			static_xlen.copy_(xlen, non_blocking = True)
		graph.replay()
		return [(lg.clone(), lp.clone(), am.clone()) for lg, lp, am in outs]

	def _packed_features(self, x, xlen, want_lo, c_align = 64):
		"""raw input (signal when the frontend is in the model, else fp32 features [B, C, F]) -> (bf16 hi, lo or None, frames, channels):
		log-mel frontend + masked instance norm + channels-last packing (models.py:286-301)"""
		nf = self.normalize_features
		if nf is not None and (nf.track_running_stats or nf.affine):
			raise NotImplementedError('convasr_b200: instance norm with running stats / affine parameters is not built')
		stride = self.backbone[0].conv[0][0].stride[0]
		if self.frontend is not None and isinstance(self.frontend, LogFilterBankFrontend) and self.frontend.nfft == 256:
			C = self.frontend.mel.weight.shape[0]
			hi, lo, Fr = self.frontend.features(x, xlen, nf, stride == 2, engine._ceil_to(C, c_align), want_lo)
			return hi, lo, Fr, C
		feats = self.frontend(x, xlen = xlen) if self.frontend is not None else x
		B, C, Fr = feats.shape
		F_pad = Fr + (Fr % 2) if stride == 2 else Fr
		norm_xlen = xlen if (nf is not None and nf.temporal_mask) else None
		hi, lo, _ = ops.instnorm_pack(feats, norm_xlen, nf.eps if nf is not None else -1.0, F_pad = F_pad, C_pad = engine._ceil_to(C, c_align), want_lo = want_lo, normalize = nf is not None)
		return hi, lo, Fr, C

	def _raw_to_outputs(self, x, xlen):
		"""raw input (signal or features) -> per head (logits, log_probs, argmax); kernels only"""
		plan = self._get_plan()
		hi, lo, Fr, C = self._packed_features(x, xlen, plan.fp32_tier, plan.feat_align)
		if plan.fp8:
			hi = ops.quantize_e4m3(hi, plan.blocks[0][0].in_scale)
		return plan.run(engine._Act(hi, lo, Fr, C), xlen)

	def _forward_native(self, x, xlen):
		if getattr(self, '_graphs_enabled', False) and not torch.cuda.is_current_stream_capturing():
			outs = self._graphed_raw(x, xlen)
		else:
			outs = self._raw_to_outputs(x, xlen)
		logits, log_probs = [], []
		for lg, lp, am in outs:
			lp._convasr_argmax = am  # lets GreedyCTCGenerator skip its own argmax pass
			logits.append(lg)
			log_probs.append(lp)
		return tuple(logits), log_probs

	# -- reference utility surface --------------------------------------------------------
	def freeze(self, backbone = 0, decoder0 = False, frontend = False):
		"""models.py:328-339"""
		frozen = list(self.backbone[:backbone]) if backbone else []
		frozen += list(self.decoder)[:1] if decoder0 else []
		frozen += [self.frontend] if frontend and self.frontend is not None else []
		for m in frozen:
			for bn in m.modules():
				if isinstance(bn, nn.modules.batchnorm._BatchNorm):
					bn.eval()
					bn.train = lambda training: None
			for p in m.parameters():
				p.requires_grad = False

	def fuse_conv_bn_eval(self, K = None):
		"""models.py:341-343"""
		for block in self.backbone[:K]:
			block.fuse_conv_bn_eval()
		self._plan = None

	def set_temporal_mask_mode(self, enabled):
		for module in self.modules():
			module.temporal_mask = enabled
		self._plan = None


# ------------------------------------------------------------------------------------------
# the 24 configurations of models.py:819-1442
# ------------------------------------------------------------------------------------------


def _wav2letter_family(name, doc, **fixed):
	"""Wav2Letter-style constructors: explicit signature (a strict superset of the reference's,
	which rejects dict= / check_time_dim_padded=, SURVEY.md 8b) mapped onto JasperNet."""
	defaults = dict(dropout = 0.2, base_width = 128, nonlinearity = ('hardtanh', 0, 20), kernel_size_prologue = 11, kernel_size_epilogue = 29, kernel_sizes = [11, 13, 17, 21, 25], dilation = 2, num_blocks = 5)
	own = {k: fixed.pop(k) for k in list(fixed) if k in defaults}
	defaults.update(own)
	large_kernels = fixed.pop('large_kernels', False)

	def __init__(self, num_input_features, num_classes, dropout = defaults['dropout'], base_width = defaults['base_width'], nonlinearity = defaults['nonlinearity'],
				kernel_size_prologue = defaults['kernel_size_prologue'], kernel_size_epilogue = defaults['kernel_size_epilogue'], kernel_sizes = defaults['kernel_sizes'],
				dilation = defaults['dilation'], num_blocks = defaults['num_blocks'], decoder_type = None, normalize_features = True, frontend = None, **kwargs):
		args = dict(
			base_width = base_width, dropout = dropout, dropout_prologue = dropout, dropout_epilogue = dropout, dropouts = [dropout] * num_blocks,
			kernel_size_prologue = kernel_size_prologue, kernel_size_epilogue = kernel_size_epilogue,
			kernel_sizes = list(kernel_sizes) if large_kernels else [kernel_size_prologue] * num_blocks, out_width_factors = [2, 3, 4, 5, 6],
			out_width_factors_large = [7, 8], dilation = dilation, nonlinearity = nonlinearity, decoder_type = decoder_type,
			normalize_features = normalize_features, frontend = frontend
		)
		args.update(fixed)
		if fixed.get('residual') == 'flat':
			args['out_width_factors'] = [6] * num_blocks
		args.update(kwargs)
		JasperNet.__init__(self, num_input_features, num_classes, **args)

	return type(name, (JasperNet, ), dict(__init__ = __init__, __doc__ = doc))


def _jasper_family(name, doc, **fixed):
	def __init__(self, *args, **kwargs):
		merged = dict(fixed)
		merged.update(kwargs)
		JasperNet.__init__(self, *args, **merged)

	return type(name, (JasperNet, ), dict(__init__ = __init__, __doc__ = doc))


_RELU = ('relu', )
_LEAKY = ('leaky_relu', 0.01)
Wav2Letter = _wav2letter_family('Wav2Letter', 'models.py:819-853', residual = False, num_blocks = 6)
Wav2LetterResidual = _wav2letter_family('Wav2LetterResidual', 'models.py:856-892', residual = True)
Wav2LetterResidualNoDilation = _wav2letter_family('Wav2LetterResidualNoDilation', 'models.py:895-931', residual = True, dilation = 1)
Wav2LetterResidualBig = _wav2letter_family('Wav2LetterResidualBig', 'models.py:934-971', residual = True, num_subblocks = 2)
Wav2LetterDense = _wav2letter_family('Wav2LetterDense', 'models.py:974-1010', residual = 'dense')
Wav2LetterDenseNoDilation = _wav2letter_family('Wav2LetterDenseNoDilation', 'models.py:1013-1049', residual = 'dense', dilation = 1)
Wav2LetterDenseNoDilationInplace = _wav2letter_family('Wav2LetterDenseNoDilationInplace', 'models.py:1052-1089', residual = 'dense', dilation = 1, nonlinearity = _LEAKY, inplace = True)
Wav2LetterDenseLargeKernels = _wav2letter_family('Wav2LetterDenseLargeKernels', 'models.py:1092-1128', residual = 'dense', large_kernels = True)
Wav2LetterDenseNoDilationLargeKernels = _wav2letter_family('Wav2LetterDenseNoDilationLargeKernels', 'models.py:1131-1167', residual = 'dense', dilation = 1, large_kernels = True)
Wav2LetterDenseBig = _wav2letter_family('Wav2LetterDenseBig', 'models.py:1170-1207', residual = 'dense', num_subblocks = 2)
Wav2LetterDenseBigLargeKernelsNoDropoutReLu = _wav2letter_family('Wav2LetterDenseBigLargeKernelsNoDropoutReLu', 'models.py:1210-1247', residual = 'dense', num_subblocks = 2, large_kernels = True, dropout = 0.0, nonlinearity = _RELU)
Wav2LetterDenseBigLargeKernelsNoDilationNoDropoutReLu = _wav2letter_family('Wav2LetterDenseBigLargeKernelsNoDilationNoDropoutReLu', 'models.py:1250-1287', residual = 'dense', num_subblocks = 2, large_kernels = True, dropout = 0.0, nonlinearity = _RELU, dilation = 1)
Wav2LetterDenseBigLargeKernelsNoDilationNoTemporalMaskNoDropoutReLu = _wav2letter_family(
	'Wav2LetterDenseBigLargeKernelsNoDilationNoTemporalMaskNoDropoutReLu', 'models.py:1290-1328', residual = 'dense', num_subblocks = 2, large_kernels = True, dropout = 0.0,
	nonlinearity = _RELU, dilation = 1, temporal_mask = False
)
Wav2LetterFlat = _wav2letter_family('Wav2LetterFlat', 'models.py:1331-1367', residual = 'flat', kernel_size_prologue = 13, out_width_factors_large = [16, 16])

JasperNetSeparable = _jasper_family('JasperNetSeparable', 'models.py:1370-1372', separable = True, groups = 128)
JasperNetSmall = _jasper_family('JasperNetSmall', 'models.py:1375-1377', num_subblocks = 1, temporal_mask = False)
JasperNetSmallInstanceNorm = _jasper_family('JasperNetSmallInstanceNorm', 'models.py:1380-1389', num_subblocks = 1, temporal_mask = False, normalize_features_legacy = False, normalize_features_temporal_mask = False)
JasperNetSmallTrainableInstanceNorm = _jasper_family(
	'JasperNetSmallTrainableInstanceNorm', 'models.py:1392-1402', num_subblocks = 1, temporal_mask = False, normalize_features_legacy = False,
	normalize_features_temporal_mask = False, normalize_features_track_running_stats = True
)
JasperNetLarge = _jasper_family('JasperNetLarge', 'models.py:1405-1407', num_subblocks = 2, repeat = 5, temporal_mask = False)
JasperNetBig = _jasper_family('JasperNetBig', 'models.py:1410-1412', num_subblocks = 2, temporal_mask = False)
JasperNetBigNoStride = _jasper_family('JasperNetBigNoStride', 'models.py:1415-1417', num_subblocks = 2, stride1 = 1, temporal_mask = False)
JasperNetBigBpeOnly = _jasper_family('JasperNetBigBpeOnly', 'models.py:1420-1422', num_subblocks = 2, temporal_mask = False, bpe_only = True)
JasperNetResidualBig = _jasper_family('JasperNetResidualBig', 'models.py:1425-1427', num_subblocks = 2, temporal_mask = False, residual = True)
JasperNetBigInplace = _jasper_family('JasperNetBigInplace', 'models.py:1430-1442', num_subblocks = 2, temporal_mask = False, inplace = True, nonlinearity = _LEAKY)

# ------------------------------------------------------------------------------------------
# module-level helpers used by the reference's callers (train.py / transcribe.py / vis.py)
# ------------------------------------------------------------------------------------------


def entropy(log_probs, lengths = None, dim = 1, eps = 1e-9, sum = True, keepdim = False):
	"""models.py:645-658.  The default reduction runs the fused native kernel."""
	if not log_probs.is_cuda:
		raise RuntimeError('convasr_b200: entropy() runs on CUDA tensors only (there is no CPU fallback)')
	if dim == 1 and sum and not keepdim and log_probs.ndim == 3 and eps == 1e-9:
		return ops.entropy(log_probs, lengths)[0]
	# non-default reductions (other dim / keepdim / per-frame output): same formula on the GPU, unfused
	e = -(log_probs.exp() * log_probs).sum(dim = dim, keepdim = keepdim)
	if lengths is not None:
		e = e * temporal_mask(e, lengths)
	if not sum:
		return e
	return e.mean(dim = -1) if lengths is None else e.sum(dim = -1) / (eps + lengths.type_as(log_probs))


def weighted_mean_entropy(log_probs, lengths = None, dim = -2, eps = 1e-9, eps_id = -1):
	"""models.py:661-673"""
	if not log_probs.is_cuda:
		raise RuntimeError('convasr_b200: weighted_mean_entropy() runs on CUDA tensors only (there is no CPU fallback)')
	if dim in (-2, 1) and log_probs.ndim == 3 and eps == 1e-9:
		return ops.entropy(log_probs, lengths, eps_id = eps_id)[1]
	prob = log_probs.exp()
	e = -(prob * log_probs).sum(dim = dim)
	weights = 1 - prob.select(dim, eps_id)
	if lengths is not None:
		weights = weights * temporal_mask(e, lengths)
	return (e * weights).sum(dim = -1) / (eps + weights.sum(dim = -1))


def margin(log_probs, dim = 1):
	"""models.py:676-677: `torch.sub(*probs.topk(2, dim).values)`.  NB the reference unpacks the BATCH dimension, so it is
	only defined for a batch of two (top-2 of utterance 0 minus top-2 of utterance 1, [2, T]) and raises TypeError for any
	other batch size; kept as is.  The top-2 probabilities come from a native kernel."""
	if not log_probs.is_cuda:
		raise RuntimeError('convasr_b200: margin() runs on CUDA tensors only (there is no CPU fallback)')
	vals = ops.top2_probs(log_probs) if (dim == 1 and log_probs.ndim == 3) else log_probs.exp().topk(2, dim = dim).values
	return torch.sub(*vals)


def compute_capacity(model, scale = 1):
	return sum(map(torch.numel, model.parameters())) / scale


def unpad(x, lens):
	return [e[..., :l] for e, l in zip(x, lens)]


def reset_bn_running_stats_(model):
	"""models.py:726-733"""
	for bn in [m for m in model.modules() if isinstance(m, nn.modules.batchnorm._BatchNorm)]:
		nn.init.zeros_(bn.running_mean)
		nn.init.ones_(bn.running_var)
		nn.init.zeros_(bn.num_batches_tracked)
		bn.momentum = None
		bn.train()
	return model


def master_module(model):
	return model.module if isinstance(model, (nn.parallel.DistributedDataParallel, nn.DataParallel)) else model


def rle1d(tensor):
	"""models.py:778-786"""
	assert tensor.ndim == 1
	starts = torch.cat((
		torch.tensor([0], dtype = torch.long, device = tensor.device), (tensor[1:] != tensor[:-1]).nonzero(as_tuple = False).add_(1).squeeze(1),
		torch.tensor([tensor.shape[-1]], dtype = torch.long, device = tensor.device)
	))
	return starts[:-1], starts[1:] - starts[:-1], tensor[starts[:-1]]


def silence_space_mask(log_probs, speech, blank_idx, space_idx, kernel_size = 101):
	"""models.py:768-775 (host-side helper, no caller in the reference): frames that are not speech and whose best class is the
	blank, broadcast over every class except the space -> bool [B, C, T]"""
	best = log_probs.argmax(dim = 1)
	quiet = (~speech) & (best == blank_idx)
	not_space = torch.ones(log_probs.shape[1], dtype = quiet.dtype, device = quiet.device)
	not_space[space_idx] = False
	return quiet.unsqueeze(1) * not_space.view(1, -1, 1)


def sparse_topk(x, k, dim = -1, largest = True, indices_dtype = None, values_dtype = None, fill_value = 0.0):
	"""models.py:789-801: the k largest (or smallest) entries along `dim` plus what is needed to put them back"""
	top = x.topk(k, dim = dim, largest = largest)
	return dict(k = k, dim = dim, largest = largest, shape = x.shape, dtype = x.dtype, device = x.device, fill_value = fill_value,
				indices = top.indices.to(dtype = indices_dtype), values = top.values.to(dtype = values_dtype))


def sparse_topk_todense(saved, device = None):
	"""models.py:804-810: inverse of sparse_topk (everything else = fill_value)"""
	device = device or saved['device']
	dense = torch.full(saved['shape'], saved['fill_value'], dtype = saved['dtype'], device = device)
	return dense.scatter_(saved['dim'], saved['indices'].to(dtype = torch.int64, device = device), saved['values'].to(dtype = saved['dtype'], device = device))


def apply_dither(x, dither: float):
	"""models.py:622-642; both call sites in the frontend are commented out in the reference (models.py:571,574)"""
	return x + dither * torch.randn_like(x) if dither > 0.0 else x


class InplaceBatchNorm1d(nn.BatchNorm1d):
	"""models.py:402-433 by name.  In the reference this is BatchNorm1d's arithmetic with the input re-derived from the output in the
	backward (memory saving, CUDA-only ATen operators); here the *Inplace model families hold plain BatchNorm1d modules (same
	parameters, buffers and state_dict keys) and train on the native step (training.py), so this class is only the exported name."""


class InputOutputTypeCast(nn.Module):
	"""models.py:13-20"""

	def __init__(self, model, dtype):
		super().__init__()
		self.model, self.dtype = model, dtype

	def forward(self, x, *args, **kwargs):
		return self.model(x.to(self.dtype), *args, **kwargs).to(x.dtype)


def data_parallel_and_autocast(model, optimizer = None, data_parallel = True, opt_level = None, **kwargs):
	"""models.py:736-752.  apex.amp opt levels map onto the native precision tiers: None/'O0' keep
	the fp32 (split-bf16) tier, 'O1'..'O3' select the bf16 tier.  Multi-GPU inference is one
	process per GPU with utterance sharding (convasr_b200.parallel), not nn.DataParallel."""
	if opt_level not in (None, '', 'O0'):
		master_module(model).set_precision('bf16')
	return model, optimizer


def distributed_data_parallel_and_autocast(model, local_rank, optimizer = None, opt_level = None, synchronize_bn = False, **kwargs):
	"""models.py:755-765: data parallelism over NCCL / NVLink.  The model is returned UNWRAPPED with a
	parallel.GradSync attached (parameters broadcast from rank 0; the native backward all-reduces each layer's
	gradient as soon as it exists, overlapped with the rest of the backward)."""
	from . import parallel
	if synchronize_bn:
		raise NotImplementedError('convasr_b200: synchronize_bn is not built (BatchNorm statistics stay per rank, the reference default, train.py:1054)')
	if opt_level not in (None, '', 'O0'):
		model.set_precision('bf16')
	return parallel.attach_grad_sync(model), optimizer
