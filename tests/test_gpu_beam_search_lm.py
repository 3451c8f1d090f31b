"""CTC prefix beam search with a word n-gram LM on the GPU (csrc/beam.cu beam_search_kernel<true>,
ops.ctc_beam_search(lm=...), decoders.BeamSearchDecoder(lm_path='*.arpa')) against exhaustive enumeration of the fused
objective and the float64 restatement in tests/beam_lm_oracle.py.

The kernel works in fp32 and the restatement in float64: n-best lists are compared rank by rank where the reference
scores are apart (beam_oracle.assert_nbest_equal), scores to 1e-5 relative."""
import math
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import beam_lm_oracle as LO  # noqa: E402
import beam_oracle as BO  # noqa: E402
from oracle import oracle as O  # noqa: E402
from test_lm_host import ARPA_3GRAM, BLANK, LABELS  # noqa: E402

pytestmark = pytest.mark.gpu

CHARS = list(LO.RU) + ['*', '.', '2', ' ', '|']  # the char model's 38 labels, blank '|' last


@pytest.fixture(scope = 'module')
def dev():
	return torch.device('cuda')


def nbest(out, b):
	toks, lens, scores = out['tokens'][b].cpu(), out['lengths'][b].cpu().tolist(), out['scores'][b].cpu().tolist()
	return [(tuple(toks[k, :lens[k]].tolist()), scores[k]) for k in range(len(scores)) if scores[k] > -math.inf]


def decoder(labels, path, alpha, beta, **kw):
	from convasr_b200.decoders import BeamSearchDecoder
	return BeamSearchDecoder(labels, lm_path = path, beam_alpha = alpha, beam_beta = beta, **kw)


@pytest.fixture(scope = 'module')
def hand_arpa(tmp_path_factory):
	p = tmp_path_factory.mktemp('lm') / 'hand.arpa'
	p.write_text(ARPA_3GRAM, encoding = 'utf-8')
	return str(p)


@pytest.mark.parametrize('T,alpha,beta,seed', [(4, 0.0, 0.0, 0), (5, 0.5, 1.0, 1), (5, 1.3, -0.4, 2), (5, 2.0, 0.0, 3)])
def test_exhaustive_tiny_cases(dev, hand_arpa, T, alpha, beta, seed):
	g = torch.Generator().manual_seed(seed)
	lp = (1.5 * torch.randn(3, 4, T, generator = g)).log_softmax(1)
	out = decoder(LABELS, hand_arpa, alpha, beta, beam_width = 128, topk = 128, cutoff_top_n = 4, blank_id = BLANK).decode_nbest(lp.to(dev))
	direct = LO.DirectScorer(hand_arpa)
	for b in range(3):
		ref = LO.fused_labelings(lp[b].double().numpy(), direct, LABELS, alpha, beta, BLANK, O.ctc_loss_np)
		assert len(ref) <= 128
		BO.assert_nbest_equal(nbest(out, b), ref, 1e-5)


@pytest.fixture(scope = 'module')
def syn_lm(tmp_path_factory):
	"""seeded 3-gram ARPA over 2 000 words of the char labels' letters"""
	path = str(tmp_path_factory.mktemp('lm') / 'syn.arpa')
	words = LO.random_words(2000, seed = 7, lengths = (2, 7))
	LO.write_synthetic_arpa(path, words, seed = 8, n_bigrams = 20000, n_trigrams = 20000)
	return path, words


def sentences(words, B, n_words, seed):
	rng = np.random.default_rng(seed)
	cid = {l: c for c, l in enumerate(CHARS)}
	return [[cid[ch] for ch in ' '.join(words[i] for i in rng.integers(0, len(words), n_words))] for _ in range(B)]


@pytest.mark.parametrize('kind', ['peaked', 'diffuse'])
def test_long_utterances_against_restatement(dev, syn_lm, kind, capsys):
	"""T = 751, C = 38, W = 100, N = 40, ragged lengths; peaked: a sentence of LM words planted over randn"""
	path, words = syn_lm
	B, C, T, W, alpha, beta = 3, 38, 751, 100, 0.8, 1.5
	g = torch.Generator().manual_seed(11)
	olen = torch.tensor([T, 700, 523])
	if kind == 'peaked':
		lp = LO.planted(B, C, T, sentences(words, B, 24, 12), C - 1, g, scale = 6.0)
	else:
		lp = torch.randn(B, C, T, generator = g).log_softmax(1)
	out = decoder(CHARS, path, alpha, beta, beam_width = W, topk = W, cutoff_top_n = 40).decode_nbest(lp.to(dev), olen.to(dev))
	ref = LO.lm_beam_search(lp.numpy(), LO.DirectScorer(path), CHARS, alpha, beta, olen, beam_width = W, cutoff_top_n = 40)
	same = present = 0
	for b in range(B):
		got = nbest(out, b)
		BO.assert_nbest_equal(got, [(h, s) for h, _, s in ref[b]], 1e-5, k = 10)
		same += sum(x[0] == r[0] for x, r in zip(got, ref[b]))
		# every rank: each returned hypothesis is in the restatement's list, with its score
		ref_score = {h: s for h, _, s in ref[b]}
		for h, s in got:
			if h in ref_score:
				present += 1
				assert abs(s - ref_score[h]) <= 1e-5 * max(1.0, abs(ref_score[h])), (b, h, s, ref_score[h])
	total = sum(len(r) for r in ref)
	with capsys.disabled():
		print(f'\n{kind}: {same}/{total} ranks hold the restatement\'s hypothesis, {present} returned hypotheses in its list')
	assert present == sum(len(nbest(out, b)) for b in range(B))


PLANTED_ARPA = '''\\data\\
ngram 1=8
ngram 2=4
ngram 3=2

\\1-grams:
-99\t<s>\t-0.3
-1.0\t</s>
-1.0\t<unk>
-1.2\tмама\t-0.2
-1.3\tмыла\t-0.2
-1.3\tмыло\t-0.2
-1.4\tраму\t-0.2
-1.4\tрама\t-0.2

\\2-grams:
-0.2\t<s> мама\t-0.1
-0.1\tмама мыла\t-0.1
-3.0\tмама мыло\t-0.1
-0.2\tмыла раму

\\3-grams:
-0.05\t<s> мама мыла
-0.05\tмама мыла раму

\\end\\
'''


def planted_sentence(dev):
	"""'мама мылп раму': the acoustic best path misspells the second word; at that frame 'о' is the second most probable
	class and 'а' the third"""
	cid = {l: c for c, l in enumerate(CHARS)}
	text = 'мама мылп раму'
	C, blank = len(CHARS), len(CHARS) - 1
	frames = []
	for i, ch in enumerate(text):
		frames += [[(cid[ch], 8.0)] + ([(cid['о'], 6.5), (cid['а'], 5.5)] if i == 8 else []), [(blank, 8.0)]]
	lp = torch.zeros(1, C, len(frames))
	for t, peaks in enumerate(frames):
		for c, v in peaks:
			lp[0, c, t] = v
	return lp.log_softmax(1).to(dev)


def test_planted_sentence_alpha_decides(dev, tmp_path):
	path = str(tmp_path / 'planted.arpa')
	open(path, 'w', encoding = 'utf-8').write(PLANTED_ARPA)
	lp = planted_sentence(dev)
	text = lambda alpha: ''.join(CHARS[c] for c in decoder(CHARS, path, alpha, 0.0, beam_width = 32).decode(lp)[0])  # noqa: E731
	acoustic = ''.join(CHARS[c] for c in decoder(CHARS, None, 0, 0, beam_width = 32).decode(lp)[0])
	assert acoustic == 'мама мылп раму'
	assert text(0.0) == 'мама мыло раму'  # the dictionary word nearest acoustically
	assert text(3.0) == 'мама мыла раму'  # the LM's sentence


def test_result_does_not_depend_on_the_batch(dev, syn_lm):
	path, words = syn_lm
	B, C, T = 5, 38, 300
	g = torch.Generator().manual_seed(3)
	lp = LO.planted(B, C, T, sentences(words, B, 10, 4), C - 1, g, scale = 4.0).to(dev)
	olen = torch.tensor([300, 17, 299, 0, 150], device = dev)
	dec = decoder(CHARS, path, 0.7, 0.5, beam_width = 64, topk = 8)
	full = dec.decode_nbest(lp, olen)
	for b in range(B):
		one = dec.decode_nbest(lp[b:b + 1].clone(), olen[b:b + 1])
		for key in ('tokens', 'frames', 'lengths', 'scores'):
			assert torch.equal(full[key][b:b + 1], one[key]), (b, key)
	assert full['lengths'][3, 0] == 0 and full['scores'][3, 0] == 0 and full['scores'][3, 1] == -math.inf


def test_without_lm_the_search_is_unchanged(dev):
	"""lm=None makes the acoustic call: bit-equal to ops.ctc_beam_search without the LM arguments"""
	from convasr_b200 import ops
	g = torch.Generator().manual_seed(5)
	lp = torch.randn(4, 38, 200, generator = g).log_softmax(1).to(dev)
	a = ops.ctc_beam_search(lp, beam_width = 64, topk = 4)
	b = ops.ctc_beam_search(lp, beam_width = 64, topk = 4, lm = None, alpha = 0.0, beta = 0.0)
	for x, y in zip(a, b):
		assert torch.equal(x, y)


def test_bad_arguments_are_refused_before_any_launch(dev, hand_arpa):
	import ctypes
	from convasr_b200 import _lib, ops
	from convasr_b200.lm import NGramLM
	lm = NGramLM.from_arpa(hand_arpa, LABELS, BLANK)
	lp = torch.randn(2, 4, 20, device = dev).log_softmax(1)
	good = lm.device_struct(dev)
	lib = _lib.load()
	B, C, T, N, W, K = 2, 4, 20, 4, 8, 1
	nbytes = ctypes.c_int64()
	_lib.check(lib.cab_ctc_beam_search_workspace(B, T, C, N, W, K, BLANK, 1.0, ctypes.byref(nbytes)), 'workspace')
	ws = torch.empty(nbytes.value, dtype = torch.uint8, device = dev)
	outs = [torch.empty(B, K, T, dtype = torch.int32, device = dev) for _ in range(2)] + [torch.empty(B, K, dtype = torch.int32, device = dev),
																							torch.empty(B, K, device = dev)]

	def call(s, alpha = 0.5, beta = 0.0, space = 2, blank = BLANK):
		return lib.cab_ctc_beam_search_lm(lp.data_ptr(), *lp.stride(), None, B, T, C, N, 1.0, blank, W, K, ws.data_ptr(), nbytes.value, outs[0].data_ptr(),
											outs[1].data_ptr(), T, outs[2].data_ptr(), outs[3].data_ptr(), s if s is None else ctypes.byref(s), alpha, beta, space,
											None)

	def variant(**kw):
		s = _lib.NgramLM.from_buffer_copy(good)
		for k, v in kw.items():
			if k == 'size1':
				s.sizes[1] = v
			elif k == 'table0':
				s.tables[0] = v
			else:
				setattr(s, k, v)
		return s

	before = _lib.launch_count()
	bad = [dict(s = None), dict(s = variant(order = 0)), dict(s = variant(order = 7)), dict(s = variant(num_classes = 5)), dict(s = variant(size1 = 12)),
			dict(s = variant(table0 = None)), dict(s = variant(child = None)), dict(s = variant(bos = -1)), dict(s = good, space = 3), dict(s = good, space = 4),
			dict(s = good, space = -1), dict(s = good, alpha = math.nan), dict(s = good, beta = math.inf)]
	for kw in bad:
		assert call(**kw) != 0, kw
		assert lib.cab_last_error()
	torch.cuda.synchronize()
	assert _lib.launch_count() == before
	assert call(good) == 0
	torch.cuda.synchronize()
	assert _lib.launch_count() == before + 3
	with pytest.raises(ValueError, match = 'blank'):
		ops.ctc_beam_search(lp, blank = 0, lm = lm)


def test_dropin_flow_decodes_text_with_an_arpa(dev, tmp_path):
	"""drop-in `decoders.BeamSearchDecoder(labels, lm_path='x.arpa', beam_alpha, beam_beta).decode(log_probs, olen)` -> text"""
	import importlib
	path = str(tmp_path / 'x.arpa')
	open(path, 'w', encoding = 'utf-8').write(PLANTED_ARPA)
	root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
	dropin = os.path.join(root, 'convasr_b200', 'dropin')
	saved = sys.modules.pop('decoders', None)
	sys.path.insert(0, dropin)
	try:
		decoders = importlib.import_module('decoders')
		tok = O.CharTokenizer(LO.RU)
		assert tok.idx2char == CHARS
		lp = planted_sentence(dev)
		olen = torch.tensor([lp.shape[-1]], device = dev)
		hyp = decoders.BeamSearchDecoder(tok.idx2char, lm_path = path, beam_width = 32, beam_alpha = 3.0, beam_beta = 0.5).decode(lp, olen)
		assert tok.decode(hyp) == ['мама мыла раму']
	finally:
		sys.path.remove(dropin)
		sys.modules.pop('decoders', None)
		if saved is not None:
			sys.modules['decoders'] = saved
