"""Drop-in replacement for the reference's `decoders` module (decoders.py:5-55).

GreedyDecoder: per-frame top-K class ids truncated to the output length -- NO blank/repeat
collapse (that lives in transcript_generators.GreedyCTCGenerator).  K=1 is the fused argmax
(ties -> lowest id, as torch.argmax); K>1 is the native top-K kernel (K <= 8).
BeamSearchDecoder: CTC prefix beam search on the GPU (csrc/beam.cu), acoustic only or fused with a word n-gram LM read
from an ARPA file (convasr_b200/lm.py); KenLM's binary format is not read.
OnlineBeamSearchDecoder: the same search resumed chunk by chunk, one state per stream; decode_incremental returns the
tokens that became final and the tails after them, at a cost per call that does not grow with the stream.
"""
import math

import torch

from . import lm as _lm
from . import ops


class GreedyDecoder:
	def decode(self, log_probs, output_lengths = None, K = 1):
		B, C, T = log_probs.shape
		lens = [T] * B if output_lengths is None else torch.as_tensor(output_lengths).tolist()
		if K == 1:
			ids = getattr(log_probs, '_convasr_argmax', None)
			if ids is None or ids.shape != (B, T):
				_, ids = ops.log_softmax_argmax(log_probs, want_log_probs = False)
			rows = ids.cpu().tolist()
			return [row[:o] for row, o in zip(rows, lens)]
		ids = ops.topk_ids(log_probs, K).cpu()
		return [ids[b, :, :o].tolist() for b, o in enumerate(lens)]


class BeamSearchDecoder:
	"""CTC prefix beam search over [B, C, T] log_probs, argument names as ctcdecode's CTCBeamDecoder.

	Each frame keeps its `cutoff_top_n` most probable classes and, with `cutoff_prob` < 1, only those (most probable
	first) until their probability sums to `cutoff_prob`; `beam_width` (at most 128) prefixes survive each frame, ranked
	by log(p_blank + p_nonblank).  `blank_id` None means the last class (C - 1), the model's convention.  `num_workers`
	is accepted for compatibility; the search runs on the GPU.

	`lm_path` ending in '.arpa' (any case): a word n-gram LM in ARPA text format (order <= 6) is fused in with ctcdecode's word-level
	rules.  `labels` are then single characters including ' '; only prefixes whose words are in the LM's vocabulary are
	searched; a space that ends word w adds `beam_alpha` * ln P(w | previous words) + `beam_beta`; after the last frame
	the last word gets the same term (ln P = -1000 if it is not a complete word) and the hypotheses are ranked by the
	fused score.  The file is parsed once per (path, mtime, labels).  Any other `lm_path` (KenLM's binary format) raises
	NotImplementedError, as does a nonzero `beam_alpha` / `beam_beta` without `lm_path`.

	`topk` means the k most probable hypotheses, best first.  Whether the reference's `decoded_scores.topk(...)` line
	selects the same ones depends on the sign of ctcdecode's scores and cannot be checked here."""

	def __init__(self, labels, lm_path = None, beam_width = 100, beam_alpha = 0, beam_beta = 0, cutoff_top_n = 40, cutoff_prob = 1.0,
				num_workers = 1, topk = 1, blank_id = None):
		if lm_path is None and (beam_alpha != 0 or beam_beta != 0):
			raise NotImplementedError('convasr_b200: beam_alpha / beam_beta weight a language model, and no lm_path was given; '
									'pass the LM as an ARPA file (KenLM\'s text format): lm_path=\'<file>.arpa\'')
		if lm_path is not None and not str(lm_path).lower().endswith('.arpa'):
			raise NotImplementedError(f'convasr_b200: lm_path={lm_path!r} does not name an uncompressed ARPA text file (*.arpa); KenLM\'s '
									'binary format and compressed files are not read. Pass the ARPA file instead (the text LM that KenLM\'s '
									'build_binary converts), decompressed')
		if not 1 <= int(beam_width) <= ops.BEAM_MAX_WIDTH:
			raise ValueError(f'convasr_b200: beam_width={beam_width} out of [1, {ops.BEAM_MAX_WIDTH}]')
		if not 1 <= int(topk) <= int(beam_width):
			raise ValueError(f'convasr_b200: topk={topk} out of [1, beam_width={beam_width}]')
		if int(cutoff_top_n) < 1:
			raise ValueError(f'convasr_b200: cutoff_top_n={cutoff_top_n} must be positive')
		if not 0.0 < float(cutoff_prob) <= 1.0:
			raise ValueError(f'convasr_b200: cutoff_prob={cutoff_prob} out of (0, 1]')
		self.labels = labels
		self.beam_width, self.cutoff_top_n, self.cutoff_prob = int(beam_width), int(cutoff_top_n), float(cutoff_prob)
		self.num_workers, self.topk, self.blank_id = num_workers, int(topk), blank_id
		self.lm_path, self.beam_alpha, self.beam_beta = lm_path, float(beam_alpha), float(beam_beta)
		self.lm = None if lm_path is None else _lm.load_arpa(lm_path, labels, blank_id)

	def decode_nbest(self, log_probs, output_lengths = None):
		"""Device tensors for rescoring and timestamps: dict(tokens int32 [B, topk, T], frames int32 [B, topk, T] (the frame
		at which each token was emitted), lengths int32 [B, topk], scores fp32 [B, topk] = log(p_blank + p_nonblank), plus
		the LM terms with an LM).  Tokens and frames are -1 past each length; a hypothesis the search did not keep has score
		-inf and length 0."""
		tokens, frames, lengths, scores = ops.ctc_beam_search(
			log_probs, output_lengths, beam_width = self.beam_width, cutoff_top_n = self.cutoff_top_n, cutoff_prob = self.cutoff_prob,
			topk = self.topk, blank = self.blank_id, lm = self.lm, alpha = self.beam_alpha, beta = self.beam_beta
		)
		return dict(tokens = tokens, frames = frames, lengths = lengths, scores = scores)

	def decode(self, log_probs, output_lengths = None):
		"""topk = 1: one token list per utterance; topk > 1: per utterance, up to topk token lists, best first."""
		return self._token_lists(self.decode_nbest(log_probs, output_lengths))

	def _token_lists(self, r):
		lengths, scores = r['lengths'].cpu().tolist(), r['scores'].cpu().tolist()
		n_max = max([max(l) for l in lengths], default = 0)
		tokens = r['tokens'][:, :, :n_max].cpu().tolist()
		out = [[tok[:l] for tok, l, s in zip(tb, lb, sb) if s > -math.inf] for tb, lb, sb in zip(tokens, lengths, scores)]
		return [o[0] if o else [] for o in out] if self.topk == 1 else out


class OnlineBeamSearchDecoder(BeamSearchDecoder):
	"""BeamSearchDecoder for posteriors that arrive over time (ctcdecode's OnlineCTCBeamDecoder): the same constructor
	and search, resumed chunk by chunk per stream (ops.ctc_beam_search_stream, csrc/beam.cu).

	    dec = OnlineBeamSearchDecoder(labels, beam_width = 100)
	    state = dec.new_state()                             # one per stream
	    for chunk, last in chunks:                          # chunk: [1, C, T_chunk] log_probs, any T_chunk >= 0
	        partial = dec.decode(chunk, [state], is_eos = last)

	After the chunk containing frame t the result is bit for bit BeamSearchDecoder's on frames 0..t of the stream
	(with an LM, the last word's term and the re-rank included).  Each call may batch any streams in any rows; a row's
	`output_lengths` entry is its frame count in this call (0 allowed).  A state belongs to the decoder that made it;
	after an is_eos call it is finished and feeding it again raises.  decode_incremental splits each result into the
	tokens that became final and the tails after them, and its cost per call does not grow with the stream."""

	def new_state(self, capacity = 1024):
		"""a new stream; `capacity` is the node table's first size in frames (it grows by doubling)"""
		return ops.BeamStreamState(config = self._config(), capacity = capacity)

	def _config(self):
		return (tuple(self.labels), self.lm_path, self.beam_width, self.beam_alpha, self.beam_beta, self.cutoff_top_n, self.cutoff_prob,
				self.topk, self.blank_id)

	def decode_nbest(self, log_probs, states, is_eos, output_lengths = None):
		"""device tensors as BeamSearchDecoder.decode_nbest, [B, topk, L] tokens and frames with L the longest stream's
		frames so far; frames count from the stream's start"""
		self._check_states(log_probs, states)
		tokens, frames, lengths, scores = ops.ctc_beam_search_stream(
			log_probs, states, is_eos, output_lengths, beam_width = self.beam_width, cutoff_top_n = self.cutoff_top_n,
			cutoff_prob = self.cutoff_prob, topk = self.topk, blank = self.blank_id, lm = self.lm, alpha = self.beam_alpha, beta = self.beam_beta
		)
		return dict(tokens = tokens, frames = frames, lengths = lengths, scores = scores)

	def decode(self, log_probs, states, is_eos, output_lengths = None):
		"""token lists as BeamSearchDecoder.decode, for each row's stream so far"""
		r = self.decode_nbest(log_probs, states, is_eos, output_lengths)
		return self._token_lists(r)

	def decode_incremental(self, log_probs, states, is_eos, output_lengths = None):
		"""The same search at a cost per call that does not grow with the stream (ops.ctc_beam_search_stream_incremental):
		per row, (the tokens that became final in this call, [the tail after everything final so far, per hypothesis the
		search kept, best first]).  All final lists of a stream concatenated, followed by tail k, are hypothesis k of
		decode() on the same frames; final tokens are never retracted.  A state's first incremental call binds it to
		decode_incremental for life; decode / decode_nbest refuse it afterwards."""
		self._check_states(log_probs, states)
		ft, _, fl, tokens, _, lengths, scores = ops.ctc_beam_search_stream_incremental(
			log_probs, states, is_eos, output_lengths, beam_width = self.beam_width, cutoff_top_n = self.cutoff_top_n,
			cutoff_prob = self.cutoff_prob, topk = self.topk, blank = self.blank_id, lm = self.lm, alpha = self.beam_alpha, beta = self.beam_beta
		)
		fl, lengths, scores = fl.cpu().tolist(), lengths.cpu().tolist(), scores.cpu().tolist()
		n_max = max([max(l) for l in lengths], default = 0)
		ft, tokens = ft[:, :max(fl, default = 0)].cpu().tolist(), tokens[:, :, :n_max].cpu().tolist()
		return [(f[:n], [tok[:l] for tok, l, s in zip(tb, lb, sb) if s > -math.inf])
				for f, n, tb, lb, sb in zip(ft, fl, tokens, lengths, scores)]

	def _check_states(self, log_probs, states):
		if any(s.finished for s in states if isinstance(s, ops.BeamStreamState)):
			raise RuntimeError('convasr_b200: a stream of this call has ended (is_eos was set on an earlier call); start a new state')
		if log_probs.shape[1] != len(self.labels):
			raise ValueError(f'convasr_b200: log_probs have {log_probs.shape[1]} classes, the decoder {len(self.labels)} labels')
		config = self._config()
		for b, s in enumerate(states):
			if not isinstance(s, ops.BeamStreamState) or s.config != config:
				raise ValueError(f'convasr_b200: the stream state of row {b} was not made by this decoder configuration (new_state())')
