"""Native training step of the conv stack (forward with batch-statistics BatchNorm + backward).

What `model.train(); loss.backward()` does in the reference through autograd + cuDNN/ATen
(ConvBn1d.forward models.py:127-139, JasperNet.forward :303-317, train.py:748-774) runs here on this
repo's kernels, for EVERY topology of the model zoo (models.py:819-1442): plain stacks (Wav2Letter),
residual / dense / flat residual branches (each source through its own 1x1 conv + BatchNorm, added before
the activation of the last repeat, models.py:129-133), separable blocks (grouped conv + bias + ReLU ->
pointwise conv, models.py:50-64), frozen BatchNorm layers (model.freeze, models.py:328-339).

  step start                 bf16 operand copies of all weights         cab_pack_weights_batched
  forward, per conv repeat   [h = relu(grouped(x) + b)]                 cab_grouped_conv1d
                             y = conv(x or h) + batch sums in the epilogue  cab_conv1d_fused (tcgen05 implicit GEMM)
                             y_r = conv1x1_r(residual_r) + bias, sums   cab_conv1d_fused
                             x' = mask(dropout(act(sum BN_i(y_i))))     cab_bn_act_mask_fwd (one branch, bulk-copy
                                                                        streamed, BN finalize folded in) / cab_bn_multi_act_mask_fwd
  decoder                    logits, log_probs                          cab_conv1d_fused (LOGSOFTMAX epilogue) or
                                                                        LOGITS_F32 + cab_log_softmax_argmax (large vocabularies)
  backward, per conv repeat  dz, (dgamma, dbeta), dy per BN branch      cab_bn_act_mask_bwd / cab_act_mask_bwd_dz
                             dW = dy (x) x over time                    cab_conv1d_wgrad (tcgen05, MN-major operands)
                             dx = sum over ALL consumers of x           ONE cab_conv1d_fused launch whose K segments are the
                                  conv(dy_c, flipped W_c^T)             consumers (main conv of the next repeat + every
                                                                        residual 1x1 conv that reads x)
                             grouped conv: dW, db, dx                   cab_grouped_conv1d_wgrad / cab_grouped_conv1d (transposed)
                             all-reduce(dW) on the comm stream          parallel.GradSync (data-parallel replicas)

Precision tiers (model.set_precision): 'bf16' -- activations and operand copies in bf16, fp32 accumulation,
fp32 BatchNorm arithmetic, fp32 gradients; 'fp32' -- every activation, gradient activation and operand copy is a
(hi, lo) bf16 pair and every GEMM accumulates hi*hi + hi*lo + lo*hi (the exactness harness: the same kernel chain
meets the reference's fp32 numbers, tests/test_gpu_training.py).

On ragged batches the three GEMMs leave out tiles that lie entirely in an utterance's padding (the
previous layer's mask makes the inputs exact zeros there; masked gradient rows are never read).
"""
import os

import torch
import torch.nn as nn

from . import _lib, engine, ops

BF16 = torch.bfloat16
# Tests and tools/trace_train_layers.py set these two to False to run the other path as a reference; that path also runs for
# unmasked inputs and for repeats the fold does not cover.
_SKIP_PADDING = True  # leave tiles of pure padding out
# BatchNorm-backward channel sums accumulated by the dgrad GEMM's epilogue instead of a separate pass over (y, g)
_FOLD_BN_REDUCE = True
_GRAD_BUCKET_MB = int(os.environ.get('CONVASR_B200_GRAD_BUCKET_MB', '64'))  # data-parallel gradient bucket size; 0 = one collective per layer


def unsupported_reason(model):
	"""None when this module tree trains on the native kernels, else why not"""
	if getattr(model.decoder, 'type', None) is not None:
		return 'two-head (bpe) decoder'
	n_blocks = len(model.backbone)
	for i, block in enumerate(model.backbone):
		if block.activation.invertible and block.activation.nonlinearity[0] != 'leaky_relu':
			# the reference's invertible activation exists for leaky_relu only (models.py:383).  The *Inplace families themselves
			# train here: InplaceBatchNorm1d (models.py:411-433) is BatchNorm1d's arithmetic with the input re-derived from the
			# output in the backward, the invertible leaky_relu (models.py:376-408) is leaky_relu -- a memory optimisation of the
			# reference's implementation, not a different function; this path keeps both activations (180 GB of HBM).
			return 'invertible activation other than leaky_relu'
		if block.activation.nonlinearity[0] not in ('relu', 'hardtanh', 'leaky_relu'):
			return f'nonlinearity {block.activation.nonlinearity!r}'
		if len(block.conv_residual) + 1 > _lib.MAX_BN_BRANCHES:
			return 'too many residual branches'
		for rc, rbn in zip(block.conv_residual, block.bn_residual):
			if isinstance(rc, nn.Identity) != isinstance(rbn, nn.Identity):
				return 'fused residual branch'
			if not isinstance(rc, nn.Identity) and (rc.kernel_size[0] != 1 or type(rbn) is not nn.BatchNorm1d or rbn.weight is None or not rbn.track_running_stats or rbn.momentum is None):
				return 'residual branch layout'
		for seq, bn in zip(block.conv, block.bn):
			if type(bn) is not nn.BatchNorm1d:
				return 'BatchNorm already fused or replaced'
			if bn.weight is None or not bn.track_running_stats or bn.momentum is None:
				return 'BatchNorm without affine parameters / running statistics / momentum'
			if len(seq) == 3:
				g, pw = seq[0], seq[2]
				if g.stride[0] != 1 or g.dilation[0] != 1 or pw.kernel_size[0] != 1 or pw.bias is not None or g.in_channels % g.groups or g.out_channels % g.groups:
					return 'separable conv layout'
			elif len(seq) == 1:
				conv = seq[0]
				if conv.groups != 1 or conv.bias is not None or conv.stride[0] not in (1, 2) or (conv.stride[0] == 2 and (i != 0 or conv.dilation[0] != 1 or len(block.conv) != 1)):
					return 'conv layout'
			else:
				return 'conv layout'
	if not all(p.dtype == torch.float32 for p in model.parameters()):
		return 'parameters are not fp32'
	return None


def supported(model):
	"""can this module tree train on the native kernels?"""
	return unsupported_reason(model) is None


# ------------------------------------------------------------------------------------------
# static description of the graph
# ------------------------------------------------------------------------------------------
class _Conv:
	"""one dense conv (a GEMM): main conv of a repeat, pointwise conv of a separable pair, or a residual 1x1 conv"""

	def __init__(self, conv):
		self.m = conv
		self.k, self.stride, self.dil, self.pad = conv.kernel_size[0], conv.stride[0], conv.dilation[0], conv.padding[0]
		self.C_in, self.C_out = conv.in_channels, conv.out_channels
		self.ci_alloc, self.co_alloc = engine._ceil_to(self.C_in, 64), engine._ceil_to(self.C_out, 64)
		self.pair = self.stride == 2


class _Rep:
	def __init__(self, block, j, in_id, out_id, res_ids, salt):
		seq, self.bn = block.conv[j], block.bn[j]
		self.grouped = seq[0] if len(seq) == 3 else None
		self.conv = _Conv(seq[-1])
		self.act = engine.act_code(block.activation.nonlinearity)
		self.mask = bool(block.temporal_mask)
		self.dropout = float(block.activation.dropout)
		self.in_id, self.out_id, self.salt = in_id, out_id, salt
		self.res = []  # (source activation id, _Conv or None, bn or None)
		for r, (rc, rbn) in zip(res_ids, zip(block.conv_residual, block.bn_residual)):
			self.res.append((r, None, None) if isinstance(rc, nn.Identity) else (r, _Conv(rc), rbn))


def _graph(model):
	"""activation ids: 0 = normalised features; every repeat output gets the next id.  Residual bookkeeping of
	JasperNet.forward, models.py:306-313."""
	reps, residual, n = [], [], len(model.backbone)
	cur, next_id = 0, 1
	for i, block in enumerate(model.backbone):
		last = len(block.conv) - 1
		for j in range(len(block.conv)):
			reps.append(_Rep(block, j, cur, next_id, residual if j == last else [], salt = len(reps)))
			cur, next_id = next_id, next_id + 1
		if i >= n - model.num_epilogue_modules - 1:
			residual = []
		elif model.residual == 'dense':
			residual = residual + [cur]
		elif model.residual:
			residual = [cur]
		else:
			residual = []
	return reps


def _layers(model):
	"""compatibility view used by tests: the repeats of a plain stack"""
	return _graph(model)


# ------------------------------------------------------------------------------------------
# small helpers over the C ABI
# ------------------------------------------------------------------------------------------
def _empty_act(B, T, ld, dev, split):
	hi = torch.empty(B, T, ld, dtype = BF16, device = dev)
	return engine._Act(hi, torch.empty_like(hi) if split else None, T, ld)


def _pack(w, ci_ld, co_ld, want_dgrad):
	"""single weight, bf16 tier (kept for the kernel-level tests)"""
	return _pack_all([(w, ci_ld, co_ld, want_dgrad, 0, 0)], False)[0][:2]


def _pack_all(specs, split = False):
	"""specs: [(w fp32 [Co, Ci, K], ci_ld, co_ld, want_dgrad, mode, pad)] -> [(fwd, dgrad, fwd_lo, dgrad_lo)] bf16 operand copies
	([K, Co, ci_ld] / [K, Ci, co_ld] with flipped taps; mode 1 = stride-2 pair layout [taps2, Co, 2 * ci_ld]) in as few
	launches as the 32-item batches allow (cab_pack_weights_batched)"""
	out, items = [], []
	for spec in specs:
		w, ci_ld, co_ld, want_dgrad = spec[:4]
		mode, pad = (spec[4], spec[5]) if len(spec) > 4 else (0, 0)
		Co, Ci, K = w.shape
		if mode == 1:
			taps2 = (K - 1 - pad) // 2 - (0 - pad) // 2 + 1
			mk_f = lambda: torch.zeros(taps2, Co, 2 * ci_ld, dtype = BF16, device = w.device)
			ld_arg = 2 * ci_ld
		else:
			mk_f = lambda: (torch.zeros if ci_ld != Ci else torch.empty)(K, Co, ci_ld, dtype = BF16, device = w.device)
			ld_arg = ci_ld
		mk_d = lambda: (torch.zeros if co_ld != Co else torch.empty)(K, Ci, co_ld, dtype = BF16, device = w.device)
		fwd, fwd_lo = mk_f(), (mk_f() if split else None)
		dgr, dgr_lo = (mk_d() if want_dgrad else None), (mk_d() if want_dgrad and split else None)
		ptr = lambda t: t.data_ptr() if t is not None else None
		items.append(_lib.PackItem(w.data_ptr(), ptr(fwd), ptr(dgr), ptr(fwd_lo), ptr(dgr_lo), Co, Ci, K, ld_arg, co_ld, mode, pad))
		out.append((fwd, dgr, fwd_lo, dgr_lo))
	for lo in range(0, len(items), _lib.PACK_MAX_ITEMS):
		chunk = items[lo:lo + _lib.PACK_MAX_ITEMS]
		arr = (_lib.PackItem * len(chunk))(*chunk)
		_lib.check(_lib.load().cab_pack_weights_batched(arr, len(chunk), ops._stream()), 'cab_pack_weights_batched')
	return out


def _srcs(a, w_hi, w_lo, C_in, taps, dil, pad_left, T_in, pair = False):
	"""operand pairs of one logical GEMM: 1 in the bf16 tier, hi*hi + hi*lo + lo*hi in the split tier"""
	hi, lo = a.hi, a.lo
	if pair:
		B, rows, C = hi.shape
		hi = hi.view(B, rows // 2, 2 * C)
		lo = lo.view(B, rows // 2, 2 * C) if lo is not None else None
	out = [ops.Source(hi, w_hi, C_in, taps, dil, pad_left, T_in = T_in)]
	if w_lo is not None:
		out.append(ops.Source(hi, w_lo, C_in, taps, dil, pad_left, T_in = T_in))
		out.append(ops.Source(lo, w_hi, C_in, taps, dil, pad_left, T_in = T_in))
	return out


def _bn_finalize(sums, n_rows, C, bn):
	"""sums: fp64 [2, ld] accumulated by the conv epilogue -> [scale, shift, mean, invstd] (+ running statistics)"""
	ss = torch.empty(4, C, dtype = torch.float32, device = sums.device)
	if sums.shape[1] != C:  # the epilogue indexes the statistics with the padded channel count
		sums = sums[:, :C].contiguous()
	rc = _lib.load().cab_bn_finalize(ops._p(sums), n_rows, C, ops._p(bn.weight), ops._p(bn.bias), float(bn.eps), float(bn.momentum), ops._p(bn.running_mean), ops._p(bn.running_var), ops._p(ss), ops._stream())
	_lib.check(rc, 'cab_bn_finalize')
	return ss


def _bn_frozen_coeffs(bn):
	"""BatchNorm in eval mode inside a training model (model.freeze): normalise with the running statistics"""
	invstd = torch.rsqrt(bn.running_var.detach().float() + bn.eps)
	scale = bn.weight.detach().float() * invstd
	return torch.stack([scale, bn.bias.detach().float() - bn.running_mean.detach().float() * scale, bn.running_mean.detach().float(), invstd]).contiguous()


def _conv_bn(cv, x, T_in, B, w, bias, bn, xlen, skip, split):
	"""y = conv(x) (+ bias) with the BatchNorm batch statistics from the epilogue -> (y, ss, T_out)"""
	dev = x.hi.device
	wf, _, wf_lo, _ = w
	if cv.pair:
		taps, pad_left = wf.shape[0], -((0 - cv.pad) // 2)
		srcs = _srcs(x, wf, wf_lo, 2 * cv.ci_alloc, taps, 1, pad_left, x.hi.shape[1] // 2, pair = True)
		T_out = (T_in + 2 * cv.pad - (cv.k - 1) - 1) // 2 + 1
	else:
		srcs = _srcs(x, wf, wf_lo, cv.ci_alloc, cv.k, cv.dil, cv.pad, T_in)
		T_out = T_in + 2 * cv.pad - cv.dil * (cv.k - 1)
	y = _empty_act(B, T_out, cv.co_alloc, dev, split)
	b_pad = None
	if bias is not None:
		b_pad = torch.zeros(cv.co_alloc, dtype = torch.float32, device = dev)
		b_pad[:cv.C_out] = bias.detach()
	if not bn.training:
		ops.conv1d_fused(srcs, B, T_out, cv.co_alloc, bias = b_pad, out_hi = y.hi, out_lo = y.lo, skip = skip)
		return y, _bn_frozen_coeffs(bn), T_out, None
	sums = torch.empty(2, cv.co_alloc, dtype = torch.float64, device = dev)  # fp64 accumulators: reproducible batch statistics
	ops.conv1d_fused(srcs, B, T_out, cv.co_alloc, bias = b_pad, out_hi = y.hi, out_lo = y.lo, stats = sums, skip = skip)  # batch statistics in the epilogue
	return y, None, T_out, sums


class NativeStack(torch.autograd.Function):
	"""feats (bf16 channels-last, no grad) -> (logits, log_probs, argmax); parameters enter as explicit inputs
	so autograd routes their gradients; `holder` carries the module tree and launch geometry."""

	@staticmethod
	def forward(ctx, holder, feats, feats_lo, xlen, *params):
		model, reps, split = holder['model'], holder['reps'], holder['split']
		lib = _lib.load()
		B, dev = feats.shape[0], feats.device
		dec = model.decoder[0]
		# bf16 operand copies (hi [, lo]) of every dense conv weight, in one launch per 32 weights
		specs, slots = [], {}
		for rep in reps:
			convs = [rep.conv] + [c for _, c, _ in rep.res if c is not None]
			for cv in convs:
				slots[cv] = len(specs)
				needs_dgrad = not cv.pair
				specs.append((cv.m.weight.detach(), cv.ci_alloc, cv.co_alloc, needs_dgrad, 1 if cv.pair else 0, cv.pad if cv.pair else 0))
		specs.append((dec.weight.detach(), engine._ceil_to(dec.in_channels, 64), engine._ceil_to(dec.out_channels, 64), True, 0, 0))
		packed = _pack_all(specs, split)
		W = {cv: packed[i] for cv, i in slots.items()}
		w_dec = packed[-1]

		acts = {0: (engine._Act(feats, feats_lo, holder['n_frames'], feats.shape[2]), holder['n_frames'])}
		masked = {0: False}  # is the activation exactly zero past ceil(xlen * T)?
		saved = []
		for rep in reps:
			x, x_T = acts[rep.in_id]
			cv = rep.conv
			rec = dict(x = x, x_T = x_T)
			conv_in, conv_T = x, x_T
			if rep.grouped is not None:
				g = rep.grouped
				h_hi, h_lo = ops.grouped_conv1d(x.hi, x_T, g.in_channels, g.weight.detach(), g.bias.detach() if g.bias is not None else None, g.groups, g.padding[0], ld_out = cv.ci_alloc, act_lo = x.lo, want_lo = split, relu = True)
				conv_in, conv_T = engine._Act(h_hi, h_lo, x_T + 2 * g.padding[0] - (g.kernel_size[0] - 1), g.out_channels), x_T + 2 * g.padding[0] - (g.kernel_size[0] - 1)
				rec['h'] = conv_in
			skip = None
			if _SKIP_PADDING and xlen is not None and masked[rep.in_id] and rep.grouped is None and not cv.pair:
				# the input is exactly zero from frame ceil(xlen*x_T) on (the producer's mask), the conv has no
				# bias: output rows >= that + pad are zeros -- tiles of pure padding are not computed
				skip = (xlen, x_T, cv.pad)
			y, ss, T_out, sums = _conv_bn(cv, conv_in, conv_T, B, W[cv], None, rep.bn, xlen, skip, split)
			code, a, b = rep.act
			out = _empty_act(B, T_out, cv.co_alloc, dev, split)
			mask_ptr = ops._p(xlen if rep.mask else None)
			if not rep.res:
				# one BatchNorm branch: streamed kernel, the BN finalize (mean / invstd / running statistics) folded in
				if ss is None:
					ss = torch.empty(4, cv.C_out, dtype = torch.float32, device = dev)
					bn = rep.bn
					rc = lib.cab_bn_act_mask_fwd_stats(
						ops._p(y.hi), ops._p(y.lo), ops._p(sums), sums.shape[1], B * T_out, ops._p(bn.weight), ops._p(bn.bias), float(bn.eps), float(bn.momentum),
						ops._p(bn.running_mean), ops._p(bn.running_var), ops._p(ss), B, T_out, cv.C_out, cv.co_alloc, code, a, b, mask_ptr, ops._p(out.hi), ops._p(out.lo),
						rep.dropout, ops._p(holder['seed']), rep.salt, ops._stream()
					)
					_lib.check(rc, 'cab_bn_act_mask_fwd_stats')
				else:
					# frozen BatchNorm: ss holds the coefficients of the running statistics
					rc = lib.cab_bn_act_mask_fwd(ops._p(y.hi), ops._p(y.lo), ops._p(ss), B, T_out, cv.C_out, cv.co_alloc, code, a, b, mask_ptr, ops._p(out.hi), ops._p(out.lo), rep.dropout, ops._p(holder['seed']), rep.salt, ops._stream())
					_lib.check(rc, 'cab_bn_act_mask_fwd')
				rec.update(y = y, ss = ss, branches = None)
			else:
				if ss is None:
					ss = _bn_finalize(sums, B * T_out, cv.C_out, rep.bn)
				branches = [(None, None, y, ss, rep.bn)]
				for src_id, rcv, rbn in rep.res:
					r_act, r_T = acts[src_id]
					assert r_T == T_out, 'residual sources must have the frame count of the block output'
					if rcv is None:
						branches.append((src_id, None, r_act, None, None))
						continue
					y_r, ss_r, _, sums_r = _conv_bn(rcv, r_act, r_T, B, W[rcv], rcv.m.bias, rbn, xlen, None, split)
					if ss_r is None:
						ss_r = _bn_finalize(sums_r, B * T_out, rcv.C_out, rbn)
					branches.append((src_id, rcv, y_r, ss_r, rbn))
				arr = (_lib.BnBranch * len(branches))(*[_lib.BnBranch(t.hi.data_ptr(), t.lo.data_ptr() if t.lo is not None else None, s.data_ptr() if s is not None else None) for _, _, t, s, _ in branches])
				rc = lib.cab_bn_multi_act_mask_fwd(arr, len(branches), B, T_out, cv.C_out, cv.co_alloc, code, a, b, mask_ptr, ops._p(out.hi), ops._p(out.lo), rep.dropout, ops._p(holder['seed']), rep.salt, ops._stream())
				_lib.check(rc, 'cab_bn_multi_act_mask_fwd')
				rec.update(y = y, ss = ss, branches = branches, out = out)
			rec['T_out'] = T_out
			saved.append(rec)
			acts[rep.out_id] = (out, T_out)
			masked[rep.out_id] = rep.mask and xlen is not None
		tracked = [bn.num_batches_tracked for rep in reps for bn in [rep.bn] + [rb for _, c, rb in rep.res if c is not None] if bn.training]
		if tracked:
			torch._foreach_add_(tracked, 1)
		x, x_T = acts[reps[-1].out_id]
		C = dec.out_channels
		logits = torch.empty(B, C, x_T, dtype = torch.float32, device = dev)
		dec_srcs = _srcs(x, w_dec[0], w_dec[2], w_dec[0].shape[2], 1, 1, 0, x_T)
		bias = dec.bias.detach() if dec.bias is not None else None
		if C <= 256:
			log_probs = torch.empty_like(logits)
			argmax = torch.empty(B, x_T, dtype = torch.int32, device = dev)
			ops.conv1d_fused(dec_srcs, B, x_T, C, bias = bias, logits = logits, log_probs = log_probs, argmax = argmax, epilogue = _lib.EPI_LOGSOFTMAX)
		else:
			ops.conv1d_fused(dec_srcs, B, x_T, C, bias = bias, logits = logits, epilogue = _lib.EPI_LOGITS_F32)
			log_probs, argmax = ops.log_softmax_argmax(logits)
		ctx.holder, ctx.saved, ctx.xlen, ctx.W, ctx.w_dec, ctx.masked = holder, saved, xlen, W, w_dec, masked
		ctx.seed = holder['seed'].clone()  # the value this forward used (the live counter advances every step)
		holder['seed'].add_(len(reps) + 1)
		ctx.last = (x, x_T)
		ctx.acts = acts
		ctx.save_for_backward(log_probs)
		ctx.mark_non_differentiable(argmax)
		return logits, log_probs, argmax

	@staticmethod
	def backward(ctx, g_logits, g_log_probs, _g_argmax):
		holder, saved, xlen, W, masked = ctx.holder, ctx.saved, ctx.xlen, ctx.W, ctx.masked
		model, reps, split = holder['model'], holder['reps'], holder['split']
		log_probs, = ctx.saved_tensors
		lib = _lib.load()
		B, C, T = log_probs.shape
		dev = log_probs.device
		# gradient w.r.t. the logits
		g = None
		if g_log_probs is not None:
			g = torch.empty_like(log_probs)
			rc = lib.cab_log_softmax_bwd(ops._p(log_probs), ops._p(g_log_probs.to(torch.float32).contiguous()), B, C, T, ops._p(g), ops._stream())
			_lib.check(rc, 'cab_log_softmax_bwd')
		if g_logits is not None:
			g = g_logits.to(torch.float32).contiguous() if g is None else g + g_logits
		dec = model.decoder[0]
		c_ld = engine._ceil_to(C, 64)
		g_cl = _empty_act(B, T, c_ld, dev, split)
		sync = getattr(model, '_grad_sync', None)
		# all the small gradients (decoder bias, BN gamma / beta, grouped conv bias) live in one flat buffer: one all-reduce
		bn_list = [(rep, None) for rep in reps] + [(rep, k) for rep in reps for k, (_, c, _) in enumerate(rep.res) if c is not None]
		small_n = c_ld + sum(2 * (rep.conv.C_out if k is None else rep.res[k][1].C_out) for rep, k in bn_list) + sum(rep.grouped.out_channels for rep in reps if rep.grouped is not None)
		small = torch.zeros(small_n, dtype = torch.float32, device = dev)
		cursor = [c_ld]

		def take(n):
			v = small[cursor[0]:cursor[0] + n]
			cursor[0] += n
			return v

		max_c = max(rep.conv.C_out for rep in reps)
		partials = torch.empty(_lib.BN_SUM_REPLICAS * 2 * max_c, dtype = torch.float64, device = dev)  # scratch of the BN backward sums
		d_bias = small[:C] if dec.bias is not None else None
		rc = lib.cab_bct_to_btc(ops._p(g), B, C, T, c_ld, ops._p(g_cl.hi), ops._p(g_cl.lo), ops._p(d_bias), ops._stream())
		_lib.check(rc, 'cab_bct_to_btc')
		grads = {}

		# Gradient buckets (data-parallel replicas): the packed weight gradients are carved, in backward order, out of flat
		# buffers of ~CONVASR_B200_GRAD_BUCKET_MB; a bucket is all-reduced in ONE collective as soon as it is full -- 266 MB of
		# Wav2Letter gradients travel in 5 collectives instead of 20 (each costs a launch, ~40 us of latency at 8 ranks and a
		# window in which NCCL and the persistent GEMMs compete for SMs), still overlapped with the rest of the backward.
		bucket = dict(buf = None, used = 0, start = 0)
		bucket_floats = max(1, _GRAD_BUCKET_MB) * (1 << 18)

		def flush_bucket():
			if sync is not None and bucket['buf'] is not None and bucket['used'] > bucket['start']:
				sync.reduce(bucket['buf'][bucket['start']:bucket['used']])
			bucket['start'] = bucket['used']

		def alloc(numel):
			if sync is None:
				return torch.empty(numel, dtype = torch.float32, device = dev)
			if bucket['buf'] is None or bucket['used'] + numel > bucket['buf'].numel():
				flush_bucket()
				bucket['buf'] = torch.empty(max(bucket_floats, numel), dtype = torch.float32, device = dev)
				bucket['used'] = bucket['start'] = 0
			out = bucket['buf'][bucket['used']:bucket['used'] + numel]
			bucket['used'] += numel
			return out

		def wgrad(dy, dy_T, C_out, x, x_T, C_in, k, dil, pad, x_masked):
			return _wgrad(dy, dy_T, C_out, x, x_T, C_in, k, dil, pad, xlen if (_SKIP_PADDING and xlen is not None and x_masked) else None, defer = True, alloc = alloc)

		deferred = []  # packed weight gradients: all-reduced in their packed layout, un-packed into the parameter layout by ONE launch at the end

		def finish_weight(p, grad):
			if not p.requires_grad:
				return
			if isinstance(grad, tuple):
				packed, K, Co, Ci, transposed, pair_pad, pair_ci_alloc = grad
				out = torch.empty(Co, Ci, K, dtype = torch.float32, device = dev)
				deferred.append(_lib.UnpackItem(packed.data_ptr(), out.data_ptr(), K, Co, Ci, packed.shape[2], int(transposed), pair_pad, pair_ci_alloc))
				deferred_keep.append(packed)
				grads[p] = out
				if bucket['buf'] is not None and bucket['used'] - bucket['start'] >= bucket_floats:
					flush_bucket()  # overlaps the dgrad / wgrad of the layers still to come
				return
			grads[p] = grad
			if sync is not None:
				sync.reduce(grad)

		deferred_keep = []

		# decoder: the wide side (input channels) sits on the 128-row M side -> packed gradient is [1, Ci, Co]
		x_last, T_last = ctx.last
		last_masked = masked[reps[-1].out_id]
		skip_last = (xlen, T_last, 0) if _SKIP_PADDING and xlen is not None and last_masked else None
		if dec.weight.requires_grad:
			packed = _wgrad_packed(x_last, T_last, dec.in_channels, g_cl, T, C, 1, 1, 0, skip_last, alloc)
			finish_weight(dec.weight, (packed, 1, C, dec.in_channels, True, 0, 0))
		if dec.bias is not None and dec.bias.requires_grad:
			grads[dec.bias] = d_bias
		# pending[activation id] = contributions to its gradient: ('gemm', dy, w_dgrad (hi, lo), C_in, taps, dil, pad_left, T_in) or ('direct', act)
		pending = {reps[-1].out_id: [('gemm', g_cl, (ctx.w_dec[1], ctx.w_dec[3]), c_ld, 1, 1, 0, T)]}
		eyes = {}

		def materialize(act_id, T_act, ld, bn_reduce = None):
			"""sum of all contributions to d(loss)/d(activation): ONE fused GEMM launch over every consumer.  bn_reduce (see
			ops.conv1d_fused): fold the BatchNorm-backward reduction of the repeat that produced this activation into that launch;
			returns (gradient, folded?)"""
			contribs = pending.pop(act_id)
			if len(contribs) == 1 and contribs[0][0] == 'direct':
				return contribs[0][1], False
			srcs = []
			for c in contribs:
				if c[0] == 'gemm':
					_, dy, (w_hi, w_lo), C_in, taps, dil, pad_left, T_in = c
					srcs += _srcs(dy, w_hi, w_lo, C_in, taps, dil, pad_left, T_in)
				else:  # identity consumer ('flat' residual, grouped-conv input gradient): an eye weight as one more K segment
					a = c[1]
					n = a.hi.shape[2]
					if n not in eyes:
						eyes[n] = torch.eye(n, dtype = BF16, device = dev).unsqueeze(0).contiguous()
					srcs.append(ops.Source(a.hi, eyes[n], n, 1, 1, 0, T_in = a.T))
					if a.lo is not None:
						srcs.append(ops.Source(a.lo, eyes[n], n, 1, 1, 0, T_in = a.T))
			# gradient rows of masked frames are never read (the mask's backward selects, it does not multiply)
			skip = (xlen, T_act, 0) if (_SKIP_PADDING and xlen is not None and masked[act_id]) else None
			gx = None
			folded = False
			while srcs:
				# more consumers than one launch has K segments (dense 'Big' models in the split tier): chain launches, the
				# partial sum re-enters as an identity segment
				room = _lib.MAX_CONV_SOURCES - (0 if gx is None else (2 if split else 1))
				now, srcs = srcs[:room], srcs[room:]
				if gx is not None:
					if ld not in eyes:
						eyes[ld] = torch.eye(ld, dtype = BF16, device = dev).unsqueeze(0).contiguous()
					now = now + [ops.Source(gx.hi, eyes[ld], ld, 1, 1, 0, T_in = T_act)] + ([ops.Source(gx.lo, eyes[ld], ld, 1, 1, 0, T_in = T_act)] if split else [])
				nxt = _empty_act(B, T_act, ld, dev, split)
				fold_now = bn_reduce if (not srcs and not split) else None  # the launch that writes the final sum
				ops.conv1d_fused(now, B, T_act, ld, out_hi = nxt.hi, out_lo = nxt.lo, skip = skip, bn_reduce = fold_now)
				folded = fold_now is not None
				gx = nxt
			return gx, folded

		for rep, rec in zip(reversed(reps), reversed(saved)):
			cv = rep.conv
			T_out = rec['T_out']
			code, a, b = rep.act
			y, ss = rec['y'], rec['ss']
			bn_reduce = None
			if _FOLD_BN_REDUCE and not split and rec['branches'] is None and rep.dropout == 0 and lib.cab_bn_bwd_apply_covers(B * T_out, cv.co_alloc, 0) == 1:
				bn_reduce = (y.hi, ss, cv.C_out, code, a, b, xlen if rep.mask else None, partials)
			gx, folded = materialize(rep.out_id, T_out, cv.co_alloc, bn_reduce)
			mask_ptr = ops._p(xlen if rep.mask else None)
			sums = take(2 * cv.C_out).view(2, cv.C_out)
			dy = _empty_act(B, T_out, cv.co_alloc, dev, split)
			if rec['branches'] is None:
				fn, name = (lib.cab_bn_act_mask_bwd_apply, 'cab_bn_act_mask_bwd_apply') if folded else (lib.cab_bn_act_mask_bwd, 'cab_bn_act_mask_bwd')
				rc = fn(ops._p(y.hi), ops._p(y.lo), ops._p(gx.hi), ops._p(gx.lo), ops._p(ss), B, T_out, cv.C_out, cv.co_alloc, code, a, b, mask_ptr, ops._p(sums), ops._p(dy.hi), ops._p(dy.lo),
						rep.dropout, ops._p(ctx.seed), rep.salt, int(not rep.bn.training), ops._p(partials), ops._stream())
				_lib.check(rc, name)
			else:
				out = rec['out']
				dz = _empty_act(B, T_out, cv.co_alloc, dev, split)
				rc = lib.cab_act_mask_bwd_dz(ops._p(out.hi), ops._p(out.lo), ops._p(gx.hi), ops._p(gx.lo), B, T_out, cv.C_out, cv.co_alloc, code, a, b, mask_ptr, ops._p(dz.hi), ops._p(dz.lo), rep.dropout, ops._p(ctx.seed), rep.salt, ops._stream())
				_lib.check(rc, 'cab_act_mask_bwd_dz')
				for src_id, rcv, y_i, ss_i, bn_i in rec['branches']:
					if ss_i is None:  # identity residual: the source receives dz itself
						pending.setdefault(src_id, []).append(('direct', dz))
						continue
					main = rcv is None
					s_i = sums if main else take(2 * rcv.C_out).view(2, rcv.C_out)
					dy_i = dy if main else _empty_act(B, T_out, rcv.co_alloc, dev, split)
					rc = lib.cab_bn_act_mask_bwd(ops._p(y_i.hi), ops._p(y_i.lo), ops._p(dz.hi), ops._p(dz.lo), ops._p(ss_i), B, T_out, cv.C_out, cv.co_alloc, _lib.ACT_NONE, 0.0, 0.0, None, ops._p(s_i), ops._p(dy_i.hi), ops._p(dy_i.lo),
													0.0, None, 0, int(not bn_i.training), ops._p(partials), ops._stream())
					_lib.check(rc, 'cab_bn_act_mask_bwd')
					if main:
						continue
					if bn_i.bias.requires_grad:
						grads[bn_i.bias], grads[bn_i.weight] = s_i[0], s_i[1]
					r_act, r_T = ctx.acts[src_id]
					if rcv.m.weight.requires_grad:
						finish_weight(rcv.m.weight, wgrad(dy_i, T_out, rcv.C_out, r_act, r_T, rcv.C_in, 1, 1, 0, masked[src_id]))
					if rcv.m.bias is not None and rcv.m.bias.requires_grad:
						# a bias in front of a batch-statistics BatchNorm has an exactly zero gradient (dy sums to zero per channel);
						# with a frozen BatchNorm it is the channel sum of dy = scale * dbeta
						grads[rcv.m.bias] = torch.zeros_like(rcv.m.bias) if bn_i.training else (s_i[0] * ss_i[0]).contiguous()
					w = W[rcv]
					pending.setdefault(src_id, []).append(('gemm', dy_i, (w[1], w[3]), rcv.co_alloc, 1, 1, 0, T_out))
			if rep.bn.bias.requires_grad:
				grads[rep.bn.bias], grads[rep.bn.weight] = sums[0], sums[1]
			# the dense conv of this repeat: dW, and its contribution to the gradient of its input
			x, x_T = rec['x'], rec['x_T']
			conv_in, conv_T = (rec['h'], rec['h'].T) if rep.grouped is not None else (x, x_T)
			in_masked = masked[rep.in_id] and rep.grouped is None
			if cv.m.weight.requires_grad:
				if cv.pair:
					xv = engine._Act(x.hi.view(B, x.hi.shape[1] // 2, 2 * x.hi.shape[2]), x.lo.view(B, x.lo.shape[1] // 2, 2 * x.lo.shape[2]) if x.lo is not None else None, x.hi.shape[1] // 2, 2 * cv.ci_alloc)
					taps2 = W[cv][0].shape[0]
					packed = _wgrad_packed(dy, T_out, cv.C_out, xv, xv.T, 2 * cv.ci_alloc, taps2, 1, -((0 - cv.pad) // 2), None, alloc)
					finish_weight(cv.m.weight, (packed, cv.k, cv.C_out, cv.C_in, 2, cv.pad, cv.ci_alloc))
				else:
					finish_weight(cv.m.weight, wgrad(dy, T_out, cv.C_out, conv_in, conv_T, cv.C_in, cv.k, cv.dil, cv.pad, in_masked))
			if rep.in_id == 0 and rep.grouped is None:
				continue  # the features need no gradient
			w = W[cv]
			contrib = ('gemm', dy, (w[1], w[3]), cv.co_alloc, cv.k, cv.dil, cv.dil * (cv.k - 1) - cv.pad, T_out)  # dx[j] = sum_k' W'[k'] dy[j + k'*d - (d*(K-1) - pad)], W' = flipped, transposed weights
			if rep.grouped is None:
				pending.setdefault(rep.in_id, []).append(contrib)
				continue
			# separable pair: dh = pointwise dgrad, gated by the ReLU between the two convs; then the grouped conv's dW, db, dx
			gconv, h = rep.grouped, rec['h']
			pending[('h', rep.salt)] = [contrib]
			masked[('h', rep.salt)] = False
			dh, _ = materialize(('h', rep.salt), h.T, cv.ci_alloc)
			dzh = _empty_act(B, h.T, cv.ci_alloc, dev, split)
			rc = lib.cab_act_mask_bwd_dz(ops._p(h.hi), ops._p(h.lo), ops._p(dh.hi), ops._p(dh.lo), B, h.T, gconv.out_channels, cv.ci_alloc, _lib.ACT_RELU, 0.0, 0.0, None, ops._p(dzh.hi), ops._p(dzh.lo), 0.0, None, 0, ops._stream())
			_lib.check(rc, 'cab_act_mask_bwd_dz')
			gb = take(gconv.out_channels)
			gw = ops.grouped_conv1d_wgrad(dzh, h.T, x, x_T, gconv.in_channels, gconv.out_channels, gconv.groups, gconv.kernel_size[0], gconv.padding[0], gb)
			if gconv.weight.requires_grad:
				finish_weight(gconv.weight, gw)
			if gconv.bias is not None and gconv.bias.requires_grad:
				grads[gconv.bias] = gb
			if rep.in_id != 0:
				# dx = grouped conv of dz_h with the in-group transposed, tap-flipped weights (no bias, no ReLU)
				cin_g, cout_g, K = gconv.in_channels // gconv.groups, gconv.out_channels // gconv.groups, gconv.kernel_size[0]
				wt = gconv.weight.detach().view(gconv.groups, cout_g, cin_g, K).permute(0, 2, 1, 3).flip(3).reshape(gconv.in_channels, cout_g, K).contiguous()
				dx_hi, dx_lo = ops.grouped_conv1d(dzh.hi, h.T, gconv.out_channels, wt, None, gconv.groups, K - 1 - gconv.padding[0], ld_out = x.hi.shape[2], act_lo = dzh.lo, want_lo = split, relu = False, T_out = x_T)
				pending.setdefault(rep.in_id, []).append(('direct', engine._Act(dx_hi, dx_lo, x_T, x.hi.shape[2])))
		if sync is not None:
			flush_bucket()
			sync.reduce(small)
			sync.finish()
		for lo in range(0, len(deferred), 32):
			chunk = deferred[lo:lo + 32]
			arr = (_lib.UnpackItem * len(chunk))(*chunk)
			_lib.check(lib.cab_unpack_wgrad_batched(arr, len(chunk), ops._stream()), 'cab_unpack_wgrad_batched')
		return (None, None, None, None) + tuple(grads.get(p) for p in holder['params'])


def _padded_work(M, N):
	n_nt = (N + 255) // 256
	bn = ((N + n_nt - 1) // n_nt + 63) // 64 * 64
	return ((M + 127) // 128 * 128) * n_nt * bn


def _wgrad_packed(a, a_T, M, bx, b_T, N, taps, dil, pad, skip, alloc = None):
	"""fp32 [taps, M, ld] = sum_{b,t} a[b,t,m] * bx[b, t + tap*dil - pad, n]; three accumulated launches in the split tier"""
	out = ops.conv1d_wgrad(a.hi, a_T, M, bx.hi, b_T, N, taps, dil, pad, skip = skip, alloc = alloc)
	if a.lo is not None:
		ops.conv1d_wgrad(a.hi, a_T, M, bx.lo, b_T, N, taps, dil, pad, skip = skip, out = out)
		ops.conv1d_wgrad(a.lo, a_T, M, bx.hi, b_T, N, taps, dil, pad, skip = skip, out = out)
	return out


def _wgrad(dy, T_out, C_out, x, x_T, C_in, k, dil, pad, xlen_zero = None, defer = False, alloc = None):
	"""dW[co, ci, tap] = sum_{b,t} dy[b,t,co] * x[b, t + tap*dil - pad, ci].  Either tensor can sit on the
	128-row M side of the GEMM; pick the orientation with less tile padding (e.g. 640 -> 768 wastes 20 %
	one way and nothing the other way).  Swapping sides negates the frame shift."""
	if not isinstance(dy, engine._Act):
		dy, x = engine._Act(dy, None, T_out, C_out), engine._Act(x, None, x_T, C_in)
	# xlen_zero: x is exactly zero from frame ceil(xlen*x_T) on, so products with t + tap*dil - pad >= that vanish
	if _padded_work(C_out, C_in) <= _padded_work(C_in, C_out):
		packed = _wgrad_packed(dy, T_out, C_out, x, x_T, C_in, k, dil, pad, (xlen_zero, x_T, pad) if xlen_zero is not None else None, alloc)
		return (packed, k, C_out, C_in, False, 0, 0) if defer else _unpack(packed, k, C_out, C_in, transposed = False)
	packed = _wgrad_packed(x, x_T, C_in, dy, T_out, C_out, k, -dil, -pad, (xlen_zero, x_T, 0) if xlen_zero is not None else None, alloc)
	return (packed, k, C_out, C_in, True, 0, 0) if defer else _unpack(packed, k, C_out, C_in, transposed = True)


def _unpack(packed, K, Co, Ci, transposed, pair_pad = 0, pair_ci_alloc = 0):
	grad = torch.empty(Co, Ci, K, dtype = torch.float32, device = packed.device)
	rc = _lib.load().cab_unpack_wgrad(ops._p(packed), K, Co, Ci, packed.shape[2], int(transposed), ops._p(grad), 0, pair_pad, pair_ci_alloc, ops._stream())
	_lib.check(rc, 'cab_unpack_wgrad')
	return grad


def forward_training(model, x, xlen):
	"""raw input (signal when the frontend is in the model, else fp32 features [B, C, F]) -> (logits tuple, log_probs list)
	with autograd through the native kernels"""
	split = model._active_precision() == 'fp32'  # fp32 parameters train in the split-bf16 tier unless set_precision('bf16') / an apex opt level says otherwise
	reps = getattr(model, '_train_graph', None)
	if reps is None:
		reps = model._train_graph = _graph(model)
	hi, lo, Fr, C = model._packed_features(x, xlen, split)
	params = []
	for rep in reps:
		if rep.grouped is not None:
			params += [rep.grouped.weight] + ([rep.grouped.bias] if rep.grouped.bias is not None else [])
		params += [rep.conv.m.weight, rep.bn.weight, rep.bn.bias]
		for _, rcv, rbn in rep.res:
			if rcv is not None:
				params += [rcv.m.weight] + ([rcv.m.bias] if rcv.m.bias is not None else []) + [rbn.weight, rbn.bias]
	dec = model.decoder[0]
	params += [dec.weight] + ([dec.bias] if dec.bias is not None else [])
	seed = getattr(model, '_dropout_seed', None)
	if seed is None or seed.device != hi.device:
		# device-resident dropout counter, initialised from torch's seed so torch.manual_seed controls it
		seed = model._dropout_seed = torch.full((1, ), torch.initial_seed() & 0x7FFFFFFFFFFF, dtype = torch.int64, device = hi.device)
	holder = dict(model = model, reps = reps, params = params, n_frames = Fr, seed = seed, split = split)
	leaves = params
	if getattr(model, '_alias_params', False):
		# GraphedTrainStep: differentiate w.r.t. fresh aliases of the parameters (same storage).  A parameter's AccumulateGrad
		# node is cached while any earlier autograd graph lives and remembers the stream it was created under; an eager step
		# on the default stream whose outputs are still referenced would make the legacy stream wait on the capturing one.
		leaves = [p.detach().requires_grad_(p.requires_grad) for p in params]
		model._aliases = (params, leaves)
	logits, log_probs, argmax = NativeStack.apply(holder, hi, lo, xlen, *leaves)
	model._state_epoch = getattr(model, '_state_epoch', 0) + 1  # running statistics moved: cached eval plans are stale
	log_probs._convasr_argmax = argmax
	return (logits, ), [log_probs]


class GraphedTrainStep:
	"""One whole training step -- zero_grad, forward, CTC loss, backward, optimizer.step -- captured
	once into a CUDA graph and replayed: ~190 kernel launches per step stop paying host launch
	latency and inter-kernel gaps.  Inputs are copied into static buffers; the per-utterance loss of
	the step is returned (a clone).  Shapes are fixed at construction.  Data-parallel replicas
	(parallel.attach_grad_sync) capture their NCCL all-reduces inside the same graph, on the process
	group's communication stream, so they still overlap the backward."""

	def __init__(self, model, optimizer, x, xlen, y, ylen, warmup = 3, max_grad_norm = None):
		self.model, self.optimizer, self.max_grad_norm = model, optimizer, max_grad_norm
		self.params = [p for g in optimizer.param_groups for p in g['params']]
		self.static = [t.clone() for t in (x, xlen, y, ylen)]
		side = torch.cuda.Stream(device = x.device)
		side.wait_stream(torch.cuda.current_stream())
		with torch.cuda.stream(side):
			for _ in range(warmup):
				self._step()
		torch.cuda.current_stream().wait_stream(side)
		torch.cuda.synchronize()
		self.graph = torch.cuda.CUDAGraph()
		# thread_local: the NCCL watchdog thread may query events while this thread captures
		with torch.cuda.graph(self.graph, capture_error_mode = 'thread_local'):
			self.loss = self._step()

	def _step(self):
		sx, sxlen, sy, sylen = self.static
		self.optimizer.zero_grad(set_to_none = True)
		m = self.model.module if hasattr(self.model, 'module') else self.model
		m._alias_params = True
		try:
			out = self.model(sx, sxlen, y = sy, ylen = sylen)
		finally:
			m._alias_params = False
		loss = (out['loss'] * sylen[:, 0]).mean()  # train.py:754-755
		# gradients w.r.t. the per-step aliases (see forward_training), handed to the parameters the optimizer knows
		params, leaves = m._aliases
		pairs = [(p, l) for p, l in zip(params, leaves) if l.requires_grad]
		grads = torch.autograd.grad(loss, [l for _, l in pairs], allow_unused = True)
		for (p, _), g in zip(pairs, grads):
			p.grad = g
		m._aliases = None
		from . import optimizers
		if isinstance(self.optimizer, optimizers._FusedOptimizer):
			self.optimizer.step(max_grad_norm = self.max_grad_norm)  # clipping folded into the native step
		else:
			if self.max_grad_norm is not None:  # train.py:776-779
				torch.nn.utils.clip_grad_norm_(self.params, self.max_grad_norm, error_if_nonfinite = False)
			self.optimizer.step()
		return out['loss'].detach()

	def __call__(self, x, xlen, y, ylen):
		for dst, src in zip(self.static, (x, xlen, y, ylen)):
			dst.copy_(src, non_blocking = True)
		self.graph.replay()
		# parameters and running statistics were written by raw-pointer kernels inside the replay: nothing bumped a
		# tensor version, so cached eval plans (folded BN, packed weights) must be invalidated explicitly
		m = self.model.module if hasattr(self.model, 'module') else self.model
		m._state_epoch = getattr(m, '_state_epoch', 0) + 1
		return self.loss.clone()
