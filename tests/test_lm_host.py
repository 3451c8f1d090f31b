"""Word n-gram LM for the beam search (convasr_b200/lm.py), host side: ARPA back-off against hand-computed values and a
direct scorer, the probing tables through a host mirror of the kernel's lookup, the dictionary trie, the float64
restatement of the fused search against exhaustive enumeration, and the refused inputs.  No device needed; the GPU side
is tests/test_gpu_beam_search_lm.py."""
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

LABELS = ['a', 'b', ' ', '_']  # blank '_'
BLANK = 3

ARPA_3GRAM = '''
\\data\\
ngram 1=7
ngram 2=5
ngram 3=2

\\1-grams:
-1.0\t<unk>
-99\t<s>\t-0.5
-1.2\t</s>
-0.7\tab\t-0.3
-0.9\tba\t-0.2
-1.1\ta
-1.5\tbb

\\2-grams:
-0.4\t<s> ab\t-0.25
-0.6\tab ba\t-0.1
-0.8\tba a
-0.3\t<s> ba
-0.5\ta bb\t-0.05

\\3-grams:
-0.2\t<s> ab ba
-0.35\tab ba a

\\end\\
'''


def write(tmp_path, text, name = 'lm.arpa'):
	p = tmp_path / name
	p.write_text(text, encoding = 'utf-8')
	return str(p)


@pytest.fixture
def hand_lm(tmp_path):
	from convasr_b200.lm import NGramLM
	path = write(tmp_path, ARPA_3GRAM)
	return NGramLM.from_arpa(path, LABELS, BLANK), LO.DirectScorer(path)


# (completed words so far, word, log10 P by hand)
KNOWN = [
	(('ab', ), 'ba', -0.2),  # listed trigram <s> ab ba: the second word
	((), 'ab', -0.4),  # first word: <s> <s> ab unlisted, bo(<s> <s>) unlisted = 0, bigram <s> ab
	(('ba', ), 'a', -0.8),  # <s> ba a unlisted; bigram <s> ba has no back-off (0); bigram ba a
	(('ab', 'ba'), 'bb', -0.1 - 0.2 - 1.5),  # listed context ab ba (bo -0.1), listed ba (bo -0.2), unigram bb
	(('bb', 'ab'), 'ba', -0.6),  # unlisted context bb ab (0), bigram ab ba
	(('ab', 'ba'), 'a', -0.35),
	(('a', ), 'bb', -0.5),  # <s> a unlisted (0), bigram a bb
]


@pytest.mark.parametrize('ctx,w,log10p', KNOWN)
def test_arpa_back_off_known_answers(hand_lm, ctx, w, log10p):
	lm, direct = hand_lm
	assert direct.score(ctx, w) == pytest.approx(math.log(10) * log10p, abs = 1e-12)
	ids = [lm.word_id[x] for x in ('<s>', '<s>') + ctx][-2:]
	assert lm.score_ids(ids, lm.word_id[w]) == pytest.approx(math.log(10) * log10p, rel = 1e-6)


def test_oov_and_special_words(hand_lm):
	lm, direct = hand_lm
	assert direct.score((), 'zz') == direct.score((), '<unk>') == direct.score((), '</s>') == -1000.0
	assert lm.score_ids([lm.bos, lm.bos], 10 ** 6) == -1000.0
	assert sorted(lm.vocab) == ['a', 'ab', 'ba', 'bb'] and lm.order == 3


def test_tables_against_the_direct_scorer(tmp_path):
	"""every listed n-gram (its context <s>-padded) and 3000 random tuples, including unlisted contexts and OOV words,
	through the host mirror of the kernel's probing lookup"""
	from convasr_b200.lm import NGramLM
	labels = list(LO.RU) + [' ', '|']
	words = LO.random_words(300, seed = 1)
	path = str(tmp_path / 'syn.arpa')
	vocab = LO.write_synthetic_arpa(path, words, seed = 2, n_bigrams = 3000, n_trigrams = 3000)
	lm, direct = NGramLM.from_arpa(path, labels), LO.DirectScorer(path)
	for k, t in enumerate(lm.tables):
		size = len(t)
		assert size & (size - 1) == 0 and np.count_nonzero(t['key']) * 2 <= size
	ctx_of = lambda ws: [lm.word_id[x] for x in (['<s>', '<s>'] + list(ws))[-2:]]  # noqa: E731
	checked = 0
	for ws in list(direct.prob):
		h, w = ws[:-1], ws[-1]
		if w in direct.vocab and (not h or h[0] == '<s>' or '<s>' not in h):
			hc = h[h.index('<s>') + 1:] if '<s>' in h else h  # a leading <s> is the padding
			assert lm.score_ids(ctx_of(hc), lm.word_id[w]) == pytest.approx(direct.score(hc, w), rel = 1e-6, abs = 1e-6), ws
			checked += 1
	assert checked > 5000
	rng = np.random.default_rng(3)
	for _ in range(3000):
		hc = tuple(vocab[i] for i in rng.integers(3, len(vocab), rng.integers(0, 3)))
		w = vocab[rng.integers(0, len(vocab))]
		got = lm.score_ids(ctx_of(hc), lm.word_id[w]) if w in direct.vocab else -1000.0
		assert got == pytest.approx(direct.score(hc, w), rel = 1e-6, abs = 1e-6), (hc, w)


def walk(lm, text):
	"""the kernel's admissibility rule on the trie tables"""
	node = 0
	for ch in text:
		c = lm.labels.index(ch)
		if c == lm.space:
			if lm.word[node] < 0:
				return False
			node = 0
		else:
			node = lm.child[node, c]
			if node < 0:
				return False
	return True


@pytest.mark.parametrize('text,ok', [('', True), ('a', True), ('ab', True), ('ab ba', True), ('ab b', True), ('ab ba ', True), ('a bb a', True),
										(' ab', False), ('ab  ba', False), ('aa ', False), ('b ', False), ('bab', False), ('ab aa', False)])
def test_trie_admissibility(hand_lm, text, ok):
	lm, direct = hand_lm
	assert walk(lm, text) == ok
	allowed, spellable = LO.spelling(direct.vocab, LABELS, BLANK)
	runs = text.split(' ')
	ref = not text.startswith(' ') and '  ' not in text and all(r in spellable for r in runs[:-1]) and (runs[-1] in allowed or runs[-1] in spellable)
	assert ref == ok
	assert lm.nbytes == sum(t.nbytes for t in lm.tables) + lm.child.size * 4 + lm.word.size * 4 and lm.child.shape[1] == 4


@pytest.mark.parametrize('T,alpha,beta,seed', [(4, 0.0, 0.0, 0), (5, 0.0, 0.0, 1), (5, 0.5, 1.0, 2), (5, 1.3, -0.4, 3), (4, 0.0, 2.0, 4), (5, 2.0, 0.0, 5)])
def test_restatement_equals_exhaustive_enumeration(hand_lm, T, alpha, beta, seed):
	"""a beam wider than the admissible prefixes, no pruning: the fused n-best list is every admissible labeling, ranked
	by ln P_ctc + its words' bonuses + the end term"""
	_, direct = hand_lm
	g = torch.Generator().manual_seed(seed)
	lp = (1.5 * torch.randn(1, 4, T, generator = g, dtype = torch.float64)).log_softmax(1).numpy()
	ref = LO.fused_labelings(lp[0], direct, LABELS, alpha, beta, BLANK, O.ctc_loss_np)
	got = LO.lm_beam_search(lp, direct, LABELS, alpha, beta, beam_width = 4096, cutoff_top_n = 4, blank = BLANK)[0]
	assert len(got) == len(ref) > 10
	BO.assert_nbest_equal([(h, s) for h, _, s in got], ref, 1e-9)


def test_refusals(tmp_path):
	from convasr_b200.decoders import BeamSearchDecoder
	from convasr_b200.lm import NGramLM
	with pytest.raises(NotImplementedError, match = 'binary format'):
		BeamSearchDecoder(LABELS, lm_path = 'lm.bin', beam_alpha = 0.5)
	path = write(tmp_path, ARPA_3GRAM)
	with pytest.raises(ValueError, match = 'single-character'):
		NGramLM.from_arpa(path, ['ab', 'b', ' ', '_'])
	with pytest.raises(ValueError, match = 'space'):
		NGramLM.from_arpa(path, ['a', 'b', 'c', '_'])
	char_level = '\\data\\\nngram 1=4\n\n\\1-grams:\n-1\t<s>\n-1\ta\n-1\tb\n-1\t</s>\n\n\\end\\\n'
	with pytest.raises(NotImplementedError, match = 'character-level'):
		NGramLM.from_arpa(write(tmp_path, char_level, 'c.arpa'), LABELS)
	order7 = '\\data\\\n' + ''.join(f'ngram {k}=1\n' for k in range(1, 8)) + '\n'
	with pytest.raises(ValueError, match = 'order 7'):
		NGramLM.from_arpa(write(tmp_path, order7, 'o7.arpa'), LABELS)
	mismatch = ARPA_3GRAM.replace('ngram 2=5', 'ngram 2=6')
	with pytest.raises(ValueError, match = r'lm.arpa:16: the header says ngram 2=6, the section has 5'):
		NGramLM.from_arpa(write(tmp_path, mismatch), LABELS)
	with pytest.raises(ValueError, match = r':\d+: word .zz. is not a 1-gram'):
		NGramLM.from_arpa(write(tmp_path, ARPA_3GRAM.replace('ba a\n', 'ba zz\n')), LABELS)
	dup = ARPA_3GRAM.replace('ngram 2=5', 'ngram 2=6').replace('-0.3\t<s> ba\n', '-0.3\t<s> ba\n-0.35\tab ba\n')
	with pytest.raises(ValueError, match = r'lm.arpa:21: duplicate 2-gram .ab ba.'):
		NGramLM.from_arpa(write(tmp_path, dup), LABELS)
	for name in ('lm.arpa.gz', 'lm.binary'):
		with pytest.raises(NotImplementedError, match = 'compressed'):
			BeamSearchDecoder(LABELS, lm_path = name)


def test_decoder_loads_the_arpa_once(tmp_path):
	from convasr_b200.decoders import BeamSearchDecoder
	path = write(tmp_path, ARPA_3GRAM)
	d1 = BeamSearchDecoder(LABELS, lm_path = path, beam_alpha = 0.5, beam_beta = 1.0, blank_id = BLANK)
	d2 = BeamSearchDecoder(LABELS, lm_path = path, blank_id = BLANK)
	assert d1.lm is d2.lm and d1.lm.space == 2 and (d1.beam_alpha, d1.beam_beta) == (0.5, 1.0)
	with pytest.raises(NotImplementedError, match = 'KenLM'):
		BeamSearchDecoder(LABELS, beam_beta = 1.0)
	upper = write(tmp_path, ARPA_3GRAM, 'LM.ARPA')
	assert BeamSearchDecoder(LABELS, lm_path = upper, blank_id = BLANK).lm.order == 3


def test_loaded_lms_are_released(tmp_path):
	"""a file that changes replaces its entry, and at most _CACHE_MAX LMs stay loaded"""
	from convasr_b200 import lm as L
	path = write(tmp_path, ARPA_3GRAM)
	first = L.load_arpa(path, LABELS, BLANK)
	os.utime(path, ns = (1, 1))
	second = L.load_arpa(path, LABELS, BLANK)
	assert second is not first and sum(k[0] == os.path.realpath(path) for k in L._CACHE) == 1
	for i in range(L._CACHE_MAX + 1):
		L.load_arpa(write(tmp_path, ARPA_3GRAM, f'x{i}.arpa'), LABELS, BLANK)
	assert len(L._CACHE) == L._CACHE_MAX
