"""Streaming acoustic-model inference: log-probs chunk by chunk from cached layer context.

`StreamingModel(model).forward(chunks, states, is_eos)` takes the next PCM samples of any set of streams and returns the
log-probs of the output frames that became final, i.e. whose value no later audio can change.  Concatenated over calls
they equal `model(signal, normalisation = fixed)` on the whole signal bit for bit, eos tail included, so they can go
straight into `decoders.OnlineBeamSearchDecoder.decode_incremental`.

How a call works.  The inference plan (engine.StackPlan: folded BatchNorm, packed weights, the launch list) is cut into
steps: the frontend, every grouped conv of a separable block and every fused launch.  Output j of a conv reads inputs
[j - pad_left, j - pad_left + d(k - 1)] (the stride-2 prologue reads whole frame pairs), so an output is final once
all of those inputs are, and a launch with several sources (residual, dense, flat sums) is final up to the least of
them.  The host knows every count up front from the sample counts alone.  Per step, the rows each consumer still reads
(its left context, then the rows that became final in this call, then zeros for the padding at either end of the
stream) are gathered into one batched window, the existing kernels compute the new final rows, and those are appended
to each stream's buffer of that activation.  No final frame is computed twice.  (The grouped conv of a separable block
also computes the k - 1 rows after its new ones and discards them: its kernel takes one frame count for its input and
its output, and the window it reads ends k - 1 rows after the last new output.)  Before anything else a call moves
the live rows of every full buffer to its front (one batched copy launch for all streams and activations), so a stream
holds its context plus one chunk, however long it runs.

Normalisation is fixed per stream (models.FixedNormalisation): per-utterance statistics cannot be known before the end.
`estimate_normalisation` measures it on a prefix with the model's own abs-max and instance-norm statistics kernels.
"""
import numpy as np
import torch

from . import engine, ops
from .models import FixedNormalisation, LogFilterBankFrontend

__all__ = ['FixedNormalisation', 'estimate_normalisation', 'StreamingModel', 'AcousticStream', 'frontend_frames_final', 'tail_start']


@torch.no_grad()
def estimate_normalisation(model, signal_prefix, xlen = None):
	"""FixedNormalisation measured on `signal_prefix` [B, T] (e.g. the first seconds of each stream): the scale the
	frontend would apply to this prefix (1 / ((max|x| + 1e-5) * multiplier), rounded as the kernel rounds it) and the
	instance-norm mean and 1 / sd of its log-mel frames (over the first ceil(xlen * F) frames when the model masks them)"""
	fe = model.frontend
	if not isinstance(fe, LogFilterBankFrontend):
		raise NotImplementedError('convasr_b200: estimate_normalisation needs a model with its LogFilterBankFrontend')
	if not signal_prefix.is_cuda:
		raise RuntimeError('convasr_b200: model inputs must be CUDA tensors (there is no CPU fallback)')
	x = signal_prefix.squeeze(1) if signal_prefix.ndim == 3 else signal_prefix
	B = x.shape[0]
	xlen = None if xlen is None else xlen.to(device = x.device, dtype = torch.float32).contiguous()
	mel, band, twiddle, window, log_eps = fe._device_tables(x.device)
	absmax = torch.zeros(B, dtype = torch.float32, device = x.device)
	logmel = ops.frontend_logmel(
		x, xlen, window, mel, band, twiddle, fe.hop_length, fe.nfft, preemphasis = fe.preemphasis, log_eps = log_eps,
		normalize_signal = fe.normalize_signal, denom_multiplier = fe.debug_short_long_records_normalize_signal_multiplier, absmax = absmax
	)
	if fe.normalize_signal:
		mult = torch.tensor(fe.debug_short_long_records_normalize_signal_multiplier, dtype = torch.float32, device = x.device)
		scale = 1.0 / ((absmax + torch.tensor(1e-5, dtype = torch.float32, device = x.device)) * mult)
	else:
		scale = torch.ones(B, dtype = torch.float32, device = x.device)
	n_mels = logmel.shape[1]
	nf = model.normalize_features
	if nf is None:
		mean = torch.zeros(B, n_mels, dtype = torch.float32, device = x.device)
		invstd = torch.ones_like(mean)
	else:
		stats = torch.empty(B, n_mels, 2, dtype = torch.float32, device = x.device)
		ops.instnorm_pack(logmel, xlen if nf.temporal_mask else None, nf.eps, want_f32 = True, stats = stats)
		mean, invstd = stats[..., 0].contiguous(), (1.0 / stats[..., 1]).contiguous()
	return FixedNormalisation(scale.contiguous(), mean, invstd)


def frontend_frames_final(n_samples, is_eos, hop, nfft = 256):
	"""log-mel frames of a stream that no later sample can change once `n_samples` have arrived: frame f covers samples
	[hop f - nfft/2, hop f + nfft/2); the left pad is a reflection only when the stream is longer than nfft/2 samples
	(models.py:577-582), so a stream of at most nfft/2 samples holds its frames until eos, which adds the zero-padded
	tail up to the reference's n // hop + 1 frames.  Before eos frames are final in pairs (2m, 2m + 1): the frontend
	kernel transforms the two frames of a pair together as one complex sequence, so a frame's rounding depends on its
	partner, which must see the samples it sees in one shot."""
	total = n_samples // hop + 1
	if is_eos:
		return total
	if n_samples <= nfft // 2:
		return 0
	return min(total, (n_samples - nfft // 2) // hop + 1) & ~1


def tail_start(n_frames_final, hop, nfft = 256):
	"""first sample a stream keeps once `n_frames_final` frames are final: the sample before the window of the next frame
	(its pre-emphasis input); at most hop + nfft + 1 samples before the newest, since frames become final in pairs"""
	return max(0, hop * n_frames_final - nfft // 2 - 1)


class _Src:
	"""one input of a step: activation `node`, read at rows [j - pad, j - pad + span) for output j (pair: frame pairs)"""

	def __init__(self, node, taps, dilation, pad, pair = False):
		self.node, self.taps, self.dilation, self.pad, self.pair = node, taps, dilation, pad, pair
		self.span = dilation * (taps - 1) + 1  # rows (pairs when `pair`) one output reads

	def final_out(self, n_final):
		"""outputs whose inputs are all among the first n_final rows of the source"""
		if self.pair:
			return n_final // 2 + self.pad - self.span + 1
		return n_final + self.pad - self.span + 1

	def first_row(self, j):
		"""first source frame output j reads"""
		return 2 * (j - self.pad) if self.pair else j - self.pad


class _Step:
	"""a launch of the plan as the streaming planner sees it: sources, the one-shot output length, and what it runs"""

	def __init__(self, node, srcs, eos_len, launch = None, grouped = None, head = None):
		self.node, self.srcs, self.eos_len = node, srcs, eos_len
		self.launch, self.grouped, self.head = launch, grouped, head  # head: index of the decoder head this step ends
		self.left_context = max(s.pad * (2 if s.pair else 1) for s in srcs)
		self.right_reach = max((s.span - 1 - s.pad) * (2 if s.pair else 1) for s in srcs)


def _plan_steps(plan):
	"""engine.StackPlan -> list of _Step in launch order (nodes named by the plan's activation keys)"""
	steps = []
	add = steps.append
	for i, launches in enumerate(plan.blocks):
		for L in launches:
			srcs = []
			main = L.in_key
			if L.grouped is not None:
				gw, gb, groups, gpad, C_mid, c_mid_alloc, C_in = L.grouped
				add(_Step(L.tmp_key, [_Src(L.in_key, gw.shape[2], 1, gpad)], lambda n, x = L.in_key: n[x], grouped = L))
			for g in L.gemms:
				srcs.append(_Src(g.in_key, g.taps, g.dilation, g.pad_left, g.pair_view))
			if L.stride2 is not None:
				k, pad = L.stride2
				eos = lambda n, x = main, k = k, pad = pad: (n[x] + 2 * pad - (k - 1) - 1) // 2 + 1
			else:
				eos = lambda n, x = main, dT = L.dT: n[x] + dT
			add(_Step(L.key, srcs, eos, launch = L))
	for h, chain in enumerate(plan.heads):
		for j, L in enumerate(chain):
			srcs = [_Src(g.in_key, g.taps, g.dilation, g.pad_left, g.pair_view) for g in L.gemms]
			if L.grouped is not None:
				raise NotImplementedError('convasr_b200: streaming a separable decoder head is not built')
			add(_Step(L.key, srcs, lambda n, x = L.in_key, dT = L.dT: n[x] + dT, launch = L, head = h if j == len(chain) - 1 else None))
	return steps


class _Buf:
	"""one stream's rows of one activation: rows [start, count) live at [0, count - start) of hi / lo"""

	def __init__(self, hi, lo):
		self.hi, self.lo, self.start, self.count = hi, lo, 0, 0

	@property
	def cap(self):
		return self.hi.shape[0]


class AcousticStream:
	"""per-stream state of StreamingModel: samples so far, the final-frame count of every activation, the buffers of the
	rows later launches still read, the samples the next frames still need, and the stream's FixedNormalisation (one row)"""

	def __init__(self, owner, epoch, normalisation):
		self._owner, self._epoch = owner, epoch
		self.normalisation = normalisation
		self.norm_stats = normalisation.stats()  # [1, n_mels, 2] (mean, invstd), the pack's layout
		self.n_samples = 0
		self.finished = False
		self.tail = None  # fp32 device tensor: samples [tail_start(final frames), n_samples)
		self.final = {}  # node -> final frames
		self.bufs = {}  # node -> _Buf
		self.rebases = 0  # how often a buffer's live rows were moved to its front
		self.grows = 0  # how often a buffer was replaced by a larger one

	def bytes_held(self):
		"""device bytes this stream holds (sample tail and activation buffers)"""
		n = self.tail.numel() * 4 if self.tail is not None else 0
		for b in self.bufs.values():
			n += b.hi.numel() * b.hi.element_size() + (b.lo.numel() * b.lo.element_size() if b.lo is not None else 0)
		return n


class StreamingModel:
	"""Streaming inference of an eval-mode JasperNet-family model with its nfft = 256 LogFilterBankFrontend, in the bf16
	or fp32 tier.  One AcousticStream per stream (new_state); forward(chunks, states, is_eos) returns per head
	'log_probs' / 'logits' [B, C_h, T_new] fp32 and 'argmax' [B, T_new] int32 of the frames that became final in this
	call, and 'lengths' [B] int32 (how many of the T_new frames of each row are real): the input layout and
	output_lengths of OnlineBeamSearchDecoder.decode_incremental."""

	def __init__(self, model):
		self.model = model
		plan = self._plan()
		fe = model.frontend
		self.hop, self.nfft = fe.hop_length, fe.nfft
		self.n_mels = fe.mel.weight.shape[0]
		self._epoch = plan.epoch
		self.steps = _plan_steps(plan)
		self.consumers = {}  # node -> [(step, src)]
		for s in self.steps:
			for src in s.srcs:
				self.consumers.setdefault(src.node, []).append((s, src))
		self.heads = [s for s in self.steps if s.head is not None]
		self.lookahead_frames = self._lookahead()

	def _plan(self):
		m = self.model
		if m.training:
			raise RuntimeError('convasr_b200: streaming inference needs an eval-mode model; call model.eval()')
		if m._active_precision() == 'fp8':
			raise NotImplementedError("convasr_b200: the fp8 tier does not stream; call set_precision('bf16') or set_precision('fp32')")
		fe = m.frontend
		if not isinstance(fe, LogFilterBankFrontend) or fe.nfft != 256:
			raise NotImplementedError('convasr_b200: streaming needs the model\'s LogFilterBankFrontend with nfft = 256 (other FFT sizes are not built)')
		if m.normalize_features is not None and (m.normalize_features.track_running_stats or m.normalize_features.affine):
			raise NotImplementedError('convasr_b200: instance norm with running stats / affine parameters is not built')
		return m._get_plan()

	# -- the frame schedule (host only) ----------------------------------------------------------
	def schedule(self, n_samples, is_eos, prev = None):
		"""final frame count of every activation after `n_samples` samples (`is_eos`: the stream ends there); prev: the
		counts before (outputs of the decoder heads never run ahead of each other: all heads are final up to the least)"""
		fin = {'feat': frontend_frames_final(n_samples, is_eos, self.hop, self.nfft)}
		lens = {'feat': n_samples // self.hop + 1} if is_eos else None
		for s in self.steps:
			if is_eos:
				lens[s.node] = s.eos_len(lens)
				fin[s.node] = lens[s.node]
			else:
				fin[s.node] = max(0, min(src.final_out(fin[src.node]) for src in s.srcs))
		if not is_eos and len(self.heads) > 1:
			cap = min(fin[s.node] for s in self.heads)
			for s in self.heads:
				fin[s.node] = cap
		if prev is not None:
			for k, v in prev.items():
				fin[k] = max(fin[k], v)
		return fin

	def _lookahead(self):
		"""output frames the final frontier lags behind the audio in steady state: max over the phases of one hop of
		(frames the stream would have if it ended now) - (frames final now)"""
		out = self.heads[0].node
		base = 1 << 14
		lag = 0
		for phase in range(self.hop * 2):
			n = base * self.hop + phase
			lag = max(lag, self.schedule(n, True)[out] - self.schedule(n, False)[out])
		return lag

	# -- streams ---------------------------------------------------------------------------------
	def new_state(self, normalisation):
		"""a fresh stream; normalisation: models.FixedNormalisation of one row (n_mels channels)"""
		plan = self._plan()
		if plan.epoch != self._epoch:
			raise RuntimeError('convasr_b200: the model\'s inference plan changed (parameters, fuse_conv_bn_eval or precision) since this StreamingModel was built; build a new one')
		if not isinstance(normalisation, FixedNormalisation) or len(normalisation) != 1 or normalisation.mean.shape[1] != self.n_mels:
			raise ValueError(f'convasr_b200: new_state takes a FixedNormalisation of one row of {self.n_mels} channels')
		return AcousticStream(self, self._epoch, normalisation)

	def _check(self, chunks, states, is_eos):
		if self.model.training:
			raise RuntimeError('convasr_b200: streaming inference needs an eval-mode model; call model.eval()')
		plan = self._plan()
		if plan.epoch != self._epoch:
			raise RuntimeError('convasr_b200: the model\'s inference plan changed (parameters, fuse_conv_bn_eval or precision) after new_state; these streams cannot continue')
		if not (len(chunks) == len(states) == len(is_eos)) or len(states) == 0:
			raise ValueError('convasr_b200: chunks, states and is_eos need one entry per row (at least one row)')
		if len({id(s) for s in states}) != len(states):
			raise ValueError('convasr_b200: a stream appears in two rows of one call')
		for st in states:
			if not isinstance(st, AcousticStream) or st._owner is not self:
				raise ValueError('convasr_b200: a state belongs to another StreamingModel')
			if st.finished:
				raise RuntimeError('convasr_b200: a stream was fed after its eos')
		for c in chunks:
			if not isinstance(c, torch.Tensor) or not c.is_cuda:
				raise RuntimeError('convasr_b200: chunks must be CUDA tensors (there is no CPU fallback)')
			if c.ndim != 1 or c.dtype not in (torch.int16, torch.float32):
				raise ValueError('convasr_b200: a chunk is a 1-D int16 or fp32 tensor of samples')
		return plan

	@torch.no_grad()
	def forward(self, chunks, states, is_eos):
		plan = self._check(chunks, states, is_eos)
		B = len(states)
		dev = chunks[0].device
		eos = [bool(e) for e in is_eos]
		n_new = [int(c.numel()) for c in chunks]
		old = [st.final for st in states]
		new = [self.schedule(st.n_samples + n, e, st.final or None) for st, n, e in zip(states, n_new, eos)]
		self._rebase(states, old, new, plan, dev)
		copies = _Copies(dev)
		feats = self._frontend(chunks, states, n_new, eos, old, new, plan, dev)
		if feats is not None:
			self._append(states, 'feat', feats, old, new, copies)
		outs = {}
		for s in self.steps:
			o0 = [f.get(s.node, 0) for f in old]
			cnt = [nw[s.node] - a for nw, a in zip(new, o0)]
			n_out = max(cnt)
			if n_out == 0:
				if s.head is not None:
					outs[s.head] = None
				continue
			res = self._run_step(s, states, o0, n_out, plan, copies, dev)
			if s.head is not None:
				outs[s.head] = res
			elif s.node in self.consumers:
				self._append(states, s.node, res, old, new, copies)
		for st, n, e, c, f in zip(states, n_new, eos, chunks, new):
			st.n_samples += n
			st.final = f
			st.finished = e
		lengths = [new[b][self.heads[0].node] - old[b].get(self.heads[0].node, 0) for b in range(B)]
		result = {'log_probs': [], 'logits': [], 'argmax': [], 'lengths': torch.tensor(lengths, dtype = torch.int32).to(dev)}
		for h, s in enumerate(self.heads):
			r = outs.get(h)
			if r is None:
				C = s.launch.C_out
				r = (torch.empty(B, C, 0, device = dev), torch.empty(B, C, 0, device = dev), torch.empty(B, 0, dtype = torch.int32, device = dev))
			result['logits'].append(r[0])
			result['log_probs'].append(r[1])
			result['argmax'].append(r[2])
		return result

	__call__ = forward

	# -- frontend --------------------------------------------------------------------------------
	def _frontend(self, chunks, states, n_new, eos, old, new, plan, dev):
		B = len(states)
		f0 = [o.get('feat', 0) for o in old]
		frames = [nw['feat'] - a for nw, a in zip(new, f0)]
		tails = [st.tail.numel() if st.tail is not None else 0 for st in states]
		staged_len = [t + n for t, n in zip(tails, n_new)]
		pitch = max(4, (max(staged_len) + 3) // 4 * 4)
		staged = torch.zeros(B, pitch, dtype = torch.float32, device = dev)
		for b, (st, c) in enumerate(zip(states, chunks)):
			if tails[b]:
				staged[b, :tails[b]].copy_(st.tail)
			if n_new[b]:
				staged[b, tails[b]:staged_len[b]].copy_(c)
			keep = st.n_samples + n_new[b] - tail_start(new[b]['feat'], self.hop, self.nfft)
			st.tail = staged[b, staged_len[b] - keep:staged_len[b]].clone() if not eos[b] else None
		F = max(frames)
		if F == 0:
			return None
		rows = np.zeros((B, 5), dtype = np.int32)
		for b, st in enumerate(states):
			n_total = st.n_samples + n_new[b]
			rows[b] = (f0[b], frames[b], st.n_samples - tails[b], staged_len[b], int(n_total > self.nfft // 2))
		rows = torch.from_numpy(rows).to(dev)
		scale = torch.cat([st.normalisation.signal_scale for st in states])
		stats = torch.cat([st.norm_stats for st in states])
		fe = self.model.frontend
		mel, band, twiddle, window, log_eps = fe._device_tables(dev)
		hi, lo = ops.frontend_stream(staged, rows, F, window, mel, band, twiddle, self.hop, self.nfft, fe.preemphasis, log_eps, scale, stats,
									engine._ceil_to(self.n_mels, plan.feat_align), want_lo = plan.fp32_tier)
		return engine._Act(hi, lo, F, self.n_mels)

	# -- buffers ---------------------------------------------------------------------------------
	def _keep_from(self, node, fin):
		"""first row of `node` a consumer still reads, given the final counts `fin` of its consumers"""
		return max(0, min(src.first_row(fin.get(s.node, 0)) for s, src in self.consumers[node]))

	def _rebase(self, states, old, new, plan, dev):
		"""make room for this call's new rows in every buffer: move the live rows of a full buffer to its front, or move them
		to a larger buffer when they would overlap there; one batched copy launch for all streams and activations"""
		copies = _Copies(dev)
		for st, o, nw in zip(states, old, new):
			for node in self.consumers:
				add = nw[node] - o.get(node, 0)
				buf = st.bufs.get(node)
				keep = self._keep_from(node, o)
				if buf is None:
					if add == 0:
						continue
					buf = st.bufs[node] = self._alloc(node, 2 * (add + 16), plan, dev)
					buf.start = buf.count = keep
					continue
				live = buf.count - max(keep, buf.start)
				keep = max(keep, buf.start)
				if buf.count + add <= buf.start + buf.cap:
					continue
				need = live + add
				if need <= buf.cap and keep - buf.start >= live:  # rows [keep, count) -> [0, live): no overlap
					for a, _ in self._parts(buf):
						copies.add(a, 0, a, keep - buf.start, live)
					st.rebases += 1
				else:
					grown = self._alloc(node, 2 * need, plan, dev)
					for (a, _), (g, _) in zip(self._parts(buf), self._parts(grown)):
						copies.add(g, 0, a, keep - buf.start, live)
					grown.count = buf.count
					st.bufs[node] = buf = grown
					st.grows += 1
				buf.start = keep
		copies.run()

	def _alloc(self, node, rows, plan, dev):
		C = self._width(node, plan)
		hi = torch.empty(rows, C, dtype = torch.bfloat16, device = dev)
		return _Buf(hi, torch.empty_like(hi) if plan.fp32_tier else None)

	def _width(self, node, plan):
		if node == 'feat':
			return engine._ceil_to(self.n_mels, plan.feat_align)
		for s in self.steps:
			if s.node == node:
				return s.grouped.grouped[5] if s.grouped is not None else s.launch.C_alloc
		raise KeyError(node)

	@staticmethod
	def _parts(buf):
		return [(buf.hi, 0)] + ([(buf.lo, 1)] if buf.lo is not None else [])

	def _append(self, states, node, act, old, new, copies):
		"""rows [0, new - old) of each row of `act` (hi / lo [B, T, C]) -> the end of that stream's buffer of `node`"""
		for b, st in enumerate(states):
			n = new[b][node] - old[b].get(node, 0)
			if n == 0:
				continue
			buf = st.bufs[node]
			for src, (dst, _) in zip([act.hi] + ([act.lo] if act.lo is not None else []), self._parts(buf)):
				copies.add(dst, buf.count - buf.start, src[b], 0, n)
			buf.count += n
		copies.run()

	# -- one step --------------------------------------------------------------------------------
	def _window(self, src, states, o0, n_out, plan, copies, dev):
		"""the rows of src.node that outputs [o0[b], o0[b] + n_out) of each row read, in one [B, R, C] tensor (hi, lo):
		the stream's buffered rows where it has them, zeros before the stream start and past its final rows"""
		R = (n_out + src.span - 1) * (2 if src.pair else 1)
		C = self._width(src.node, plan)
		B = len(states)
		hi = torch.empty(B, R, C, dtype = torch.bfloat16, device = dev)
		lo = torch.empty_like(hi) if plan.fp32_tier else None
		for b, st in enumerate(states):
			a = src.first_row(o0[b])
			buf = st.bufs.get(src.node)
			c0 = min(max(a, 0), a + R)  # rows before the stream start are the left zero pad
			c1 = max(c0, min(a + R, buf.count if buf is not None else 0))  # rows past the final ones: right zero pad / don't-care
			assert c1 == c0 or c0 >= buf.start, 'convasr_b200: streaming context was dropped too early'
			for dst, part in [(hi, 0)] + ([(lo, 1)] if lo is not None else []):
				if c0 > a:
					copies.add(dst[b], 0, None, 0, c0 - a)
				if c1 > c0:
					copies.add(dst[b], c0 - a, buf.hi if part == 0 else buf.lo, c0 - buf.start, c1 - c0)
				if a + R > c1:
					copies.add(dst[b], c1 - a, None, 0, a + R - c1)
		return engine._Act(hi, lo, R, C)

	def _run_step(self, s, states, o0, n_out, plan, copies, dev):
		B = len(states)
		wins = [self._window(src, states, o0, n_out, plan, copies, dev) for src in s.srcs]
		copies.run()
		if s.grouped is not None:
			L = s.grouped
			gw, gb, groups, gpad, C_mid, c_mid_alloc, C_in = L.grouped
			w = wins[0]
			t_hi, t_lo = ops.grouped_conv1d_relu(w.hi, w.T, C_in, gw, gb, groups, 0, ld_out = c_mid_alloc, act_lo = w.lo, want_lo = plan.fp32_tier)
			return engine._Act(t_hi, t_lo, w.T, C_mid)
		L = s.launch
		srcs = []
		for src, g, w in zip(s.srcs, L.gemms, wins):
			hi, lo, T_in = w.hi, w.lo, w.T
			if src.pair:
				hi = hi.view(B, T_in // 2, 2 * hi.shape[2])
				lo = lo.view(B, T_in // 2, 2 * lo.shape[2]) if lo is not None else None
				T_in //= 2
			srcs.append(ops.Source(hi, g.weights.hi, g.c_in_alloc, g.taps, g.dilation, 0, T_in = T_in))
			if plan.fp32_tier:
				srcs.append(ops.Source(hi, g.weights.lo, g.c_in_alloc, g.taps, g.dilation, 0, T_in = T_in))
				srcs.append(ops.Source(lo, g.weights.hi, g.c_in_alloc, g.taps, g.dilation, 0, T_in = T_in))
		return plan.run_gemm(L, srcs, None, B, n_out, dev)


class _Copies:
	"""batched row copies for one cab_stream_copy launch: (dst tensor, dst row, src tensor or None = zeros, src row, rows).
	The jobs hold raw addresses, so the tensors are kept alive until the launch is queued: a buffer replaced before then
	(a stream's buffer that grew) would otherwise go back to the caching allocator, and a later allocation of this call
	(another grown buffer, the job table itself) could take its memory before the kernel has read it.  Once the launch is
	queued, later work on the stream is ordered after it, so the references can go."""

	def __init__(self, dev):
		self.dev, self.jobs, self.max_bytes, self.keep = dev, [], 0, []

	def add(self, dst, dst_row, src, src_row, rows):
		row_bytes = dst.shape[-1] * dst.element_size()
		assert src is None or src.shape[-1] == dst.shape[-1]
		nbytes = rows * row_bytes
		d = dst.data_ptr() + dst_row * row_bytes
		s = 0 if src is None else src.data_ptr() + src_row * row_bytes
		self.jobs.append((d, s, nbytes))
		self.keep.append((dst, src))
		self.max_bytes = max(self.max_bytes, nbytes)

	def run(self):
		for i in range(0, len(self.jobs), 65535):
			part = self.jobs[i:i + 65535]
			t = torch.tensor(part, dtype = torch.int64).pin_memory().to(self.dev, non_blocking = True)
			ops.stream_copy(t, max(n for _, _, n in part))
		self.jobs, self.max_bytes, self.keep = [], 0, []
