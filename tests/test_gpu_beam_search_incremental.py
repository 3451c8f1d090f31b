"""Incremental streaming CTC prefix beam search on the GPU (csrc/beam.cu beam_commit_kernel, beam_tail_kernel,
beam_rebase_kernel; ops.ctc_beam_search_stream_incremental, decoders.OnlineBeamSearchDecoder.decode_incremental).

Exactness: after every call, for each hypothesis k the search kept, the final segments of a stream so far followed by
tail k equal hypothesis k of ops.ctc_beam_search on the stream's frames so far, bit for bit (tokens, frames, length,
score), with and without an LM.  Maximality: the total final length equals the depth of the deepest common ancestor of
the live beams, computed here from a full-history ops.ctc_beam_search_stream state fed the same chunks (its node table
and the beam node ids in its state block), so the commit is the exact one, not just some safe prefix."""
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
def lm3(tmp_path_factory):
	"""seeded 3-gram ARPA over 1 500 words of the char labels' letters"""
	from convasr_b200.lm import NGramLM
	path = str(tmp_path_factory.mktemp('lm_incr') / 'syn3.arpa')
	words = LO.random_words(1500, seed = 21, lengths = (2, 7))
	LO.write_synthetic_arpa(path, words, seed = 22, n_bigrams = 15000, n_trigrams = 15000)
	return path, words, NGramLM.from_arpa(path, CHARS)


def posteriors(kind, B, C, T, seed, words = None):
	"""diffuse: randn; peaked: a planted label path over randn at scale 6; confident: the planted path at scale 12 over
	0.5 * randn, so that cutoff_prob 0.99 keeps one class per frame and no second branch is ever opened"""
	g = torch.Generator().manual_seed(seed)
	if kind == 'diffuse':
		return torch.randn(B, C, T, generator = g).log_softmax(1)
	rng = np.random.default_rng(seed + 1)
	if words is not None:
		cid = {l: c for c, l in enumerate(CHARS)}
		seqs = [[cid[ch] for ch in ' '.join(words[i] for i in rng.integers(0, len(words), max(1, T // 30)))] for _ in range(B)]
	else:
		seqs = [rng.integers(0, C - 1, max(1, T // 6)).tolist() for _ in range(B)]
	if kind == 'peaked':
		return LO.planted(B, C, T, seqs, C - 1, g, scale = 6.0)
	path = torch.full((B, T), C - 1)
	for b, seq in enumerate(seqs):
		path[b, torch.linspace(0, T - 1, len(seq)).long()] = torch.tensor(seq)
	return (0.5 * torch.randn(B, C, T, generator = g) + 12.0 * torch.nn.functional.one_hot(path, C).permute(0, 2, 1)).log_softmax(1)


def random_calls(lengths, seed, max_chunk = 40):
	"""random chunk sizes (0 allowed), random subsets of the unfinished streams in random row order"""
	rng = np.random.default_rng(seed)
	calls, pos = [], [0] * len(lengths)
	while any(p < l for p, l in zip(pos, lengths)):
		live = [s for s in range(len(lengths)) if pos[s] < lengths[s]]
		live = [s for s in rng.permutation(live).tolist() if rng.random() < 0.8] or live[:1]
		call = []
		for s in live:
			n = min(int(rng.integers(0, max_chunk + 1)), lengths[s] - pos[s])
			pos[s] += n
			call.append((s, n))
		calls.append(call)
	return calls


def one_shot(lp, ends, kw):
	"""ops.ctc_beam_search of stream s on frames 0..t-1 for every (s, t) in ends, on the host"""
	from convasr_b200 import ops
	out = {}
	for i in range(0, len(ends), 256):
		part = ends[i:i + 256]
		x = lp[[s for s, _ in part]]
		if lp.stride(1) == 1:
			x = x.permute(0, 2, 1).contiguous().permute(0, 2, 1)
		olen = torch.tensor([t for _, t in part], device = lp.device)
		res = [o.cpu() for o in ops.ctc_beam_search(x, olen, **kw)]
		for r, key in enumerate(part):
			out[key] = tuple(o[r] for o in res)
	return out


def dca_depth(st, W):
	"""depth (labels from the root) of the deepest common ancestor of the live beams of a full-history stream state"""
	blk = st.state.cpu()
	nb = int(blk[:16].view(torch.int32)[1])
	if nb == 0:
		return None
	o = 16 + 28 * W  # node ids: after the header, hash, parent hash, p_b, p_nb, last (cab_ctc_beam_search_stream_state_bytes)
	ids = blk[o:o + 4 * nb].view(torch.int32).tolist()
	parent = st.nodes[:st.t0].reshape(-1, 2)[:, 0].cpu().numpy()
	chain = []
	i = ids[0]
	while i >= 0:
		chain.append(i)
		i = int(parent[i])
	depth = {n: len(chain) - k for k, n in enumerate(chain)}
	depth[-1] = 0
	best = depth[ids[0]]
	for i in ids[1:]:
		while i not in depth:
			i = int(parent[i])
		best = min(best, depth[i])
	return best


def run_incremental(lp, lengths, calls, kw, capacity = 1024, check_every = 1, maximal = True):
	"""Feed stream s's frames per `calls` (lists of (stream, n_frames) rows; the chunk reaching a stream's length is its
	is_eos row) through incremental states, and the same chunks through full-history states when `maximal`.  Checks
	exactness (every `check_every`-th call and every is_eos row) and maximality (every call).  Returns the incremental
	states and the number of rebases."""
	from convasr_b200 import ops
	S, C, _ = lp.shape
	W = kw['beam_width']
	inc = [ops.BeamStreamState(capacity = capacity) for _ in range(S)]
	full = [ops.BeamStreamState() for _ in range(S)] if maximal else None
	final_tok, final_frm = [[] for _ in range(S)], [[] for _ in range(S)]
	pos = [0] * S
	results, rebases = [], 0
	for ci, call in enumerate(calls):
		T = max([n for _, n in call], default = 0)
		if lp.stride(1) == 1:
			x = torch.zeros(len(call), T, C, device = lp.device).permute(0, 2, 1)
		else:
			x = torch.zeros(len(call), C, T, device = lp.device)
		for r, (s, n) in enumerate(call):
			x[r, :, :n] = lp[s, :, pos[s]:pos[s] + n]
		eos = [pos[s] + n == lengths[s] for s, n in call]
		bases = [inc[s].base for s, _ in call]
		ft, ff, fl, tok, frm, ln, sc = [o.cpu() for o in ops.ctc_beam_search_stream_incremental(x, [inc[s] for s, _ in call], eos, [n for _, n in call], **kw)]
		rebases += sum(inc[s].base != b for (s, _), b in zip(call, bases))
		if maximal:
			ops.ctc_beam_search_stream(x, [full[s] for s, _ in call], eos, [n for _, n in call], **kw)
		for r, (s, n) in enumerate(call):
			pos[s] += n
			final_tok[s] += ft[r, :fl[r]].tolist()
			final_frm[s] += ff[r, :fl[r]].tolist()
			assert bool((ft[r, fl[r]:] == -1).all()) and bool((ff[r, fl[r]:] == -1).all())
			if maximal:
				d = dca_depth(full[s], W)
				assert d is None or d == len(final_tok[s]), ((s, pos[s]), d, len(final_tok[s]))
			if ci % check_every == 0 or eos[r]:
				results.append(((s, pos[s]), list(final_tok[s]), list(final_frm[s]), tok[r], frm[r], ln[r], sc[r]))
	ref = one_shot(lp, sorted({k for k, *_ in results}), kw)
	for key, ftok, ffrm, tok, frm, ln, sc in results:
		rt, rf, rl, rs = ref[key]
		for k in range(tok.shape[0]):
			if rs[k] == -math.inf:
				assert sc[k] == -math.inf and ln[k] == 0, (key, k)
				continue
			assert sc[k].view(torch.int32) == rs[k].view(torch.int32), (key, k, float(sc[k]), float(rs[k]))
			n = int(ln[k])
			assert len(ftok) + n == int(rl[k]), (key, k, len(ftok), n, int(rl[k]))
			assert ftok + tok[k, :n].tolist() == rt[k, :rl[k]].tolist(), (key, k)
			assert ffrm + frm[k, :n].tolist() == rf[k, :rl[k]].tolist(), (key, k)
			assert bool((tok[k, n:] == -1).all()) and bool((frm[k, n:] == -1).all())
	assert all(st.finished for st in inc) and pos == list(lengths)
	return inc, rebases


@pytest.mark.parametrize('W,topk', [(1, 1), (7, 5), (100, 5), (128, 1)])
@pytest.mark.parametrize('kind', ['peaked', 'diffuse'])
@pytest.mark.parametrize('lm', [False, True])
def test_exact_and_maximal_over_random_schedules(dev, lm3, W, topk, kind, lm):
	"""six ragged streams, random subsets in random row order per call, 0-frame rows, ends in different calls"""
	lengths = [400, 1, 250, 399, 37, 300]
	lp = posteriors(kind, 6, 38, 400, seed = 31 + W, words = lm3[1] if lm else None).to(dev)
	kw = dict(beam_width = W, cutoff_top_n = 40, topk = topk)
	if lm:
		kw.update(lm = lm3[2], alpha = 0.8, beta = 1.5)
	calls = random_calls(lengths, seed = 6)
	assert any(n == 0 for c in calls for _, n in c)
	run_incremental(lp, lengths, calls, kw)


def test_class_contiguous_c5000_view(dev):
	"""the large-vocabulary head's layout: [B, C, T] views of class-contiguous memory, W = 16"""
	lengths = [300, 211]
	lp = posteriors('peaked', 2, 5000, 300, seed = 41).to(dev)
	lp = lp.permute(0, 2, 1).contiguous().permute(0, 2, 1)
	run_incremental(lp, lengths, random_calls(lengths, seed = 42, max_chunk = 60), dict(beam_width = 16, cutoff_top_n = 40, topk = 4))


@pytest.mark.parametrize('lm', [False, True])
def test_rebase_path(dev, lm3, lm):
	"""node tables that start at 3 frames: the window is rebased hundreds of times.  Confident posteriors make the commit
	node follow the stream within a few frames; where beams do not converge the window grows instead (the exactness
	tests above cover that)"""
	lengths = [2000, 1500]
	lp = posteriors('confident', 2, 38, 2000, seed = 51, words = lm3[1] if lm else None).to(dev)
	kw = dict(beam_width = 100, cutoff_top_n = 40, topk = 4, cutoff_prob = 0.99)
	if lm:
		kw.update(lm = lm3[2], alpha = 0.8, beta = 1.5)
	states, rebases = run_incremental(lp, lengths, random_calls(lengths, seed = 52, max_chunk = 9), kw, capacity = 3)
	assert rebases >= 100, rebases
	assert all(3 < s.capacity <= 256 and s.base > 0 for s in states), [(s.capacity, s.base) for s in states]


def test_long_stream(dev):
	"""two confident streams of 120 000 frames (40 min at 20 ms) in 100-frame chunks: the node tables stay small, the
	result equals the one-shot search over all 120 000 frames"""
	from convasr_b200 import ops
	T, B = 120000, 2
	lp = posteriors('confident', B, 38, T, seed = 61).to(dev)
	kw = dict(beam_width = 100, cutoff_top_n = 40, topk = 4, cutoff_prob = 0.99)
	states = [ops.BeamStreamState() for _ in range(B)]
	finals = [[[], []] for _ in range(B)]
	cap = 0
	for t in range(0, T, 100):
		ft, ff, fl, tok, frm, ln, sc = ops.ctc_beam_search_stream_incremental(lp[:, :, t:t + 100], states, t + 100 >= T, **kw)
		if fl.max() > 0:
			n = int(fl.max())
			ft, ff, fl = ft[:, :n].cpu(), ff[:, :n].cpu(), fl.cpu()
			for b in range(B):
				finals[b][0] += ft[b, :fl[b]].tolist()
				finals[b][1] += ff[b, :fl[b]].tolist()
		cap = max(cap, *(s.capacity for s in states))
	assert cap <= 4096, cap
	rt, rf, rl, rs = [o.cpu() for o in ops.ctc_beam_search(lp, None, **kw)]
	tok, frm, ln, sc = tok.cpu(), frm.cpu(), ln.cpu(), sc.cpu()
	for b in range(B):
		for k in range(4):
			if rs[b, k] == -math.inf:
				assert sc[b, k] == -math.inf
				continue
			n = int(ln[b, k])
			assert sc[b, k].view(torch.int32) == rs[b, k].view(torch.int32)
			assert finals[b][0] + tok[b, k, :n].tolist() == rt[b, k, :rl[b, k]].tolist()
			assert finals[b][1] + frm[b, k, :n].tolist() == rf[b, k, :rl[b, k]].tolist()


def test_decoder_incremental_matches_the_one_shot_decoder(dev, lm3):
	"""decode_incremental in 25-frame chunks: final lists plus each tail are BeamSearchDecoder's n-best lists after every
	chunk, final lists never change; a call is four launches (five when a window is rebased)"""
	from convasr_b200 import _lib
	from convasr_b200.decoders import BeamSearchDecoder, OnlineBeamSearchDecoder
	path, words, _ = lm3
	lp = posteriors('peaked', 2, 38, 300, seed = 71, words = words).to(dev)
	for lm_kw in (dict(), dict(lm_path = path, beam_alpha = 0.8, beam_beta = 1.5)):
		kw = dict(beam_width = 48, topk = 3, **lm_kw)
		on, off = OnlineBeamSearchDecoder(CHARS, **kw), BeamSearchDecoder(CHARS, **kw)
		states = [on.new_state(capacity = 16), on.new_state(capacity = 16)]
		finals = [[], []]
		for t in range(0, 300, 25):
			before = _lib.launch_count()
			bases = [s.base for s in states]
			part = on.decode_incremental(lp[:, :, t:t + 25], states, is_eos = t + 25 >= 300)
			torch.cuda.synchronize()
			assert _lib.launch_count() - before == 4 + any(s.base != b for s, b in zip(states, bases))
			ref = off.decode(lp[:, :, :t + 25])
			for b, (final, tails) in enumerate(part):
				finals[b] += final
				assert [finals[b] + tail for tail in tails] == ref[b]
		with pytest.raises(RuntimeError, match = 'ended'):
			on.decode_incremental(lp[:1, :, :5], states[:1], is_eos = False)
