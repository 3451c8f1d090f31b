"""Streaming CTC prefix beam search on the GPU (csrc/beam.cu beam_search_kernel<LM, true>, ops.ctc_beam_search_stream,
decoders.OnlineBeamSearchDecoder) against the one-shot search.

The contract is bit-identity: after the call that consumed frames 0..t of a stream, tokens, emission frames, lengths and
scores equal what ops.ctc_beam_search returns for frames 0..t of that stream with the same arguments, with and without
an LM, whatever the chunk sizes, batch partners and rows.  The one-shot references are batched (the stream's
log-probs repeated with output_lengths = t + 1); its result does not depend on the batch (tests/test_gpu_beam_search.py)."""
import ctypes
import math
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import beam_lm_oracle as LO  # noqa: E402

pytestmark = pytest.mark.gpu

CHARS = list(LO.RU) + ['*', '.', '2', ' ', '|']  # the char model's 38 labels, blank '|' last


@pytest.fixture(scope = 'module')
def dev():
	return torch.device('cuda')


@pytest.fixture(scope = 'module')
def syn_lm(tmp_path_factory):
	"""seeded 3-gram ARPA over 2 000 words of the char labels' letters"""
	from convasr_b200.lm import NGramLM
	path = str(tmp_path_factory.mktemp('lm') / 'syn.arpa')
	words = LO.random_words(2000, seed = 7, lengths = (2, 7))
	LO.write_synthetic_arpa(path, words, seed = 8, n_bigrams = 20000, n_trigrams = 20000)
	return path, words, NGramLM.from_arpa(path, CHARS)


def sentences(words, B, n_words, seed):
	rng = np.random.default_rng(seed)
	cid = {l: c for c, l in enumerate(CHARS)}
	return [[cid[ch] for ch in ' '.join(words[i] for i in rng.integers(0, len(words), n_words))] for _ in range(B)]


def posteriors(kind, B, C, T, seed, words = None):
	g = torch.Generator().manual_seed(seed)
	if kind == 'diffuse':
		return torch.randn(B, C, T, generator = g).log_softmax(1)
	if words is not None:
		return LO.planted(B, C, T, sentences(words, B, T // 30, seed + 1), C - 1, g, scale = 6.0)
	seqs = [torch.randint(0, C - 1, (T // 6, ), generator = g).tolist() for _ in range(B)]
	return LO.planted(B, C, T, seqs, C - 1, g, scale = 6.0)


def one_shot(lp, ends, kw):
	"""ops.ctc_beam_search of stream s on frames 0..t-1 for every (s, t) in ends: {(s, t): (tokens, frames, length, score)}"""
	from convasr_b200 import ops
	out = {}
	for i in range(0, len(ends), 256):
		part = ends[i:i + 256]
		x = lp[[s for s, _ in part]]
		if lp.stride(1) == 1:
			x = x.permute(0, 2, 1).contiguous().permute(0, 2, 1)
		olen = torch.tensor([t for _, t in part], device = lp.device)
		tok, frm, ln, sc = ops.ctc_beam_search(x, olen, **kw)
		for r, key in enumerate(part):
			out[key] = (tok[r], frm[r], ln[r], sc[r])
	return out


def assert_same(got, ref, key):
	"""stream row (tokens [K, L], frames, lengths [K], scores [K]) == one-shot (tokens [K, T], ...) bit for bit"""
	gt, gf, gl, gs = got
	rt, rf, rl, rs = ref
	assert torch.equal(gl, rl), (key, gl.tolist(), rl.tolist())
	assert torch.equal(gs, rs), (key, gs.tolist(), rs.tolist())
	w = min(gt.shape[-1], rt.shape[-1])
	assert torch.equal(gt[:, :w], rt[:, :w]) and torch.equal(gf[:, :w], rf[:, :w]), key
	assert bool((gt[:, w:] == -1).all()) and bool((rt[:, w:] == -1).all()), key


def run_schedule(lp, lengths, calls, kw, capacity = 1024, check_every = 1):
	"""Feed stream s's frames per `calls`: a list of calls, each a list of (stream, n_frames) rows in row order; a stream's
	last chunk (reaching its length) is its is_eos row.  Checks the partial result of every row against the one-shot
	search (every `check_every`-th call, and every is_eos row).  Returns the states."""
	from convasr_b200 import ops
	S, C, _ = lp.shape
	states = [ops.BeamStreamState(capacity = capacity) for _ in range(S)]
	pos = [0] * S
	results = []
	for ci, call in enumerate(calls):
		T = max([n for _, n in call], default = 0)
		if lp.stride(1) == 1:  # class-contiguous memory: chunks as [B, C, T] views of it too
			x = torch.zeros(len(call), T, C, device = lp.device).permute(0, 2, 1)
		else:
			x = torch.zeros(len(call), C, T, device = lp.device)
		for r, (s, n) in enumerate(call):
			x[r, :, :n] = lp[s, :, pos[s]:pos[s] + n]
		eos = [pos[s] + n == lengths[s] for s, n in call]
		out = ops.ctc_beam_search_stream(x, [states[s] for s, _ in call], eos, [n for _, n in call], **kw)
		for r, (s, n) in enumerate(call):
			pos[s] += n
			if ci % check_every == 0 or eos[r]:
				results.append(((s, pos[s]), tuple(o[r] for o in out)))
	ref = one_shot(lp, sorted({k for k, _ in results}), kw)
	for key, got in results:
		assert_same(got, ref[key], key)
	assert all(st.finished for st in states) and pos == list(lengths)
	return states


def fixed_calls(lengths, size):
	"""all unfinished streams in every call, in stream order, `size` frames each (the rest at the end)"""
	calls, pos = [], [0] * len(lengths)
	while any(p < l for p, l in zip(pos, lengths)):
		call = [(s, min(size, l - p)) for s, (p, l) in enumerate(zip(pos, lengths)) if p < l]
		for s, n in call:
			pos[s] += n
		calls.append(call)
	return calls


def random_calls(lengths, seed, max_chunk = 40, shuffle = True, zero_rows = True):
	"""random chunk sizes (0 allowed), random subsets of the unfinished streams in random row order"""
	rng = np.random.default_rng(seed)
	calls, pos = [], [0] * len(lengths)
	while any(p < l for p, l in zip(pos, lengths)):
		live = [s for s in range(len(lengths)) if pos[s] < lengths[s]]
		if shuffle:
			live = [s for s in rng.permutation(live).tolist() if rng.random() < 0.8] or live[:1]
		call = []
		for s in live:
			n = int(rng.integers(0 if zero_rows else 1, max_chunk + 1))
			n = min(n, lengths[s] - pos[s])
			pos[s] += n
			call.append((s, n))
		calls.append(call)
	return calls


C2 = dict(beam_width = 100, cutoff_top_n = 40, topk = 8)
SPLITS = [1, 7, 25, 100, 'random']


@pytest.mark.parametrize('split', SPLITS)
@pytest.mark.parametrize('kind', ['peaked', 'diffuse'])
def test_c2_chunkings_equal_the_one_shot_search(dev, kind, split):
	"""C = 38, W = 100, N = 40, T = 751, ragged lengths: final and every partial result"""
	lengths = [751, 700, 523]
	lp = posteriors(kind, 3, 38, 751, seed = 1).to(dev)
	calls = fixed_calls(lengths, split) if split != 'random' else random_calls(lengths, seed = 2, shuffle = False, zero_rows = False)
	run_schedule(lp, lengths, calls, C2)


@pytest.mark.parametrize('split', SPLITS)
@pytest.mark.parametrize('kind', ['peaked', 'diffuse'])
def test_c2_chunkings_with_lm_equal_the_one_shot_search(dev, syn_lm, kind, split):
	"""the same with the synthetic 3-gram LM: partial results include the last word's term and the re-rank"""
	path, words, lm = syn_lm
	lengths = [751, 700, 523]
	lp = posteriors(kind, 3, 38, 751, seed = 3, words = words).to(dev)
	calls = fixed_calls(lengths, split) if split != 'random' else random_calls(lengths, seed = 4, shuffle = False, zero_rows = False)
	run_schedule(lp, lengths, calls, dict(C2, lm = lm, alpha = 0.8, beta = 1.5))


@pytest.mark.parametrize('lm', [False, True])
def test_streams_move_between_rows_and_partners(dev, syn_lm, lm):
	"""six ragged streams: random subsets in random row order per call, rows with 0 new frames, ends in different calls"""
	lengths = [400, 1, 250, 399, 37, 300]
	lp = posteriors('peaked', 6, 38, 400, seed = 5, words = syn_lm[1] if lm else None).to(dev)
	kw = dict(beam_width = 64, cutoff_top_n = 40, topk = 16)
	if lm:
		kw.update(lm = syn_lm[2], alpha = 0.6, beta = 0.9)
	calls = random_calls(lengths, seed = 6)
	assert any(n == 0 for c in calls for _, n in c) and len({tuple(s for s, _ in c) for c in calls}) > 3
	run_schedule(lp, lengths, calls, kw)


def test_class_contiguous_c5000_view(dev):
	"""the large-vocabulary head's layout: [B, C, T] views of class-contiguous memory, W = 16"""
	lengths = [300, 211]
	lp = posteriors('peaked', 2, 5000, 300, seed = 7).to(dev)
	lp = lp.permute(0, 2, 1).contiguous().permute(0, 2, 1)
	run_schedule(lp, lengths, random_calls(lengths, seed = 8, max_chunk = 60), dict(beam_width = 16, cutoff_top_n = 40, topk = 4))


@pytest.mark.parametrize('cfg', [dict(beam_width = 1, cutoff_top_n = 40, topk = 1), dict(beam_width = 128, cutoff_top_n = 64, topk = 128),
									dict(beam_width = 100, cutoff_top_n = 40, topk = 8, cutoff_prob = 0.9)], ids = ['W1', 'W128_N64', 'cutoff_prob'])
@pytest.mark.parametrize('lm', [False, True])
def test_widths_and_cutoff(dev, syn_lm, cfg, lm):
	lengths = [300, 257, 120]
	C = 100 if cfg['cutoff_top_n'] == 64 and not lm else 38
	lp = posteriors('diffuse' if cfg.get('cutoff_prob') else 'peaked', 3, C, 300, seed = 9, words = syn_lm[1] if lm and C == 38 else None).to(dev)
	kw = dict(cfg)
	if lm:
		kw.update(lm = syn_lm[2], alpha = 0.8, beta = 1.5, cutoff_top_n = min(cfg['cutoff_top_n'], 38))
	run_schedule(lp, lengths, random_calls(lengths, seed = 10), kw)


@pytest.mark.parametrize('lm', [False, True])
def test_node_table_growth(dev, syn_lm, lm):
	"""node tables that start at 3 frames grow by copying, results unchanged"""
	lengths = [200, 173]
	lp = posteriors('peaked', 2, 38, 200, seed = 11, words = syn_lm[1] if lm else None).to(dev)
	kw = dict(beam_width = 100, cutoff_top_n = 40, topk = 4)
	if lm:
		kw.update(lm = syn_lm[2], alpha = 0.8, beta = 1.5)
	states = run_schedule(lp, lengths, random_calls(lengths, seed = 12, max_chunk = 9), kw, capacity = 3)
	assert all(3 < s.capacity < 2 * l + 9 for s, l in zip(states, lengths))


@pytest.mark.parametrize('lm', [False, True])
def test_ten_minute_stream(dev, syn_lm, lm):
	"""T = 30 000 frames (10 min at 20 ms), 50-frame chunks: every 60th partial and the final result"""
	T = 30000
	lp = posteriors('peaked', 1, 38, T, seed = 13, words = syn_lm[1] if lm else None).to(dev)
	kw = dict(beam_width = 100, cutoff_top_n = 40, topk = 4)
	if lm:
		kw.update(lm = syn_lm[2], alpha = 0.8, beta = 1.5)
	run_schedule(lp, [T], fixed_calls([T], 50), kw, check_every = 60)


def test_eos_returns_final_and_refuses_more(dev, syn_lm):
	from convasr_b200.decoders import BeamSearchDecoder, OnlineBeamSearchDecoder
	path = syn_lm[0]
	lp = posteriors('peaked', 2, 38, 120, seed = 14, words = syn_lm[1]).to(dev)
	for lm_path in (None, path):
		kw = dict(beam_width = 32, topk = 4) if lm_path is None else dict(lm_path = lm_path, beam_alpha = 0.8, beam_beta = 1.5, beam_width = 32, topk = 4)
		dec = OnlineBeamSearchDecoder(CHARS, **kw)
		states = [dec.new_state() for _ in range(2)]
		dec.decode(lp[:, :, :70], states, is_eos = False)
		hyp = dec.decode(lp[:, :, 70:], states, is_eos = True)
		assert hyp == BeamSearchDecoder(CHARS, **kw).decode(lp)
		nb = dec.decode_nbest(lp[:1, :, :0], [dec.new_state()], is_eos = True)
		assert nb['lengths'][0, 0] == 0 and nb['scores'][0, 0] == 0 and nb['scores'][0, 1] == -math.inf
		with pytest.raises(RuntimeError, match = 'ended'):
			dec.decode(lp[:1, :, :5], states[:1], is_eos = False)


def test_refused_calls_launch_nothing(dev, syn_lm):
	from convasr_b200 import _lib, ops
	lib = _lib.load()
	B, C, T, N, W, K = 2, 38, 10, 38, 16, 2
	lp = torch.randn(B, C, T, device = dev).log_softmax(1)
	sb = ops.beam_stream_state_bytes(W)
	states = [torch.zeros(sb, dtype = torch.uint8, device = dev) for _ in range(B)]
	nodes = [torch.empty(T, W, 2, dtype = torch.int32, device = dev) for _ in range(B)]
	nbytes = ctypes.c_int64()
	_lib.check(lib.cab_ctc_beam_search_stream_workspace(B, T, N, W, K, ctypes.byref(nbytes)), 'workspace')
	ws = torch.empty(nbytes.value, dtype = torch.uint8, device = dev)
	outs = [torch.empty(B, K, T, dtype = torch.int32, device = dev) for _ in range(2)] + [torch.empty(B, K, dtype = torch.int32, device = dev),
																							torch.empty(B, K, device = dev)]

	def rows(**kw):
		r = (_lib.BeamStreamRow * B)()
		for b in range(B):
			r[b].state, r[b].nodes, r[b].state_bytes, r[b].capacity, r[b].t0, r[b].frames = states[b].data_ptr(), nodes[b].data_ptr(), sb, T, 0, T
		for k, v in kw.items():
			setattr(r[1], k, v)
		return r

	def call(r, W = W, N = N, K = K, blank = C - 1, lm = None):
		return lib.cab_ctc_beam_search_stream(lp.data_ptr(), *lp.stride(), r, B, T, C, N, 1.0, blank, W, K, ws.data_ptr(), nbytes.value,
												outs[0].data_ptr(), outs[1].data_ptr(), T, outs[2].data_ptr(), outs[3].data_ptr(), lm, 0.5, 0.5, 36, None)

	before = _lib.launch_count()
	bad = [(dict(r = rows(finished = 1)), 'ended'), (dict(r = rows(t0 = 1)), 'overruns'), (dict(r = rows(frames = T + 1)), 'frames'),
			(dict(r = rows(state = states[0].data_ptr())), 'share'), (dict(r = rows(state_bytes = sb - 16)), 'state block'),
			(dict(r = rows(nodes = None)), 'null'), (dict(r = rows(), W = 0), 'beam_width'), (dict(r = rows(), W = 129), 'beam_width'),
			(dict(r = rows(), N = 65), 'N='), (dict(r = rows(), K = W + 1), 'K='), (dict(r = rows(), blank = C), 'blank'),
			(dict(r = rows(), lm = ctypes.byref(syn_lm[2].device_struct(dev))), 'state block')]
	for kw, msg in bad:
		assert call(**kw) != 0, msg
		assert msg in lib.cab_last_error().decode(), (msg, lib.cab_last_error())
	torch.cuda.synchronize()
	assert _lib.launch_count() == before
	assert call(rows()) == 0
	torch.cuda.synchronize()
	assert _lib.launch_count() == before + 3
	st = ops.BeamStreamState()
	with pytest.raises(ValueError, match = 'another search configuration'):
		ops.ctc_beam_search_stream(lp[:1], [st], False, beam_width = 8)
		ops.ctc_beam_search_stream(lp[:1], [st], False, beam_width = 16)


def test_decoder_stream_matches_the_one_shot_decoder_text(dev, syn_lm):
	"""OnlineBeamSearchDecoder fed in 25-frame chunks gives BeamSearchDecoder's n-best token lists after every chunk"""
	from convasr_b200.decoders import BeamSearchDecoder, OnlineBeamSearchDecoder
	path, words, _ = syn_lm
	lp = posteriors('peaked', 2, 38, 200, seed = 15, words = words).to(dev)
	kw = dict(lm_path = path, beam_alpha = 0.8, beam_beta = 1.5, beam_width = 48, topk = 3)
	on, off = OnlineBeamSearchDecoder(CHARS, **kw), BeamSearchDecoder(CHARS, **kw)
	states = [on.new_state(), on.new_state()]
	for t in range(0, 200, 25):
		part = on.decode(lp[:, :, t:t + 25], states, is_eos = t + 25 >= 200)
		assert part == off.decode(lp[:, :, :t + 25])
