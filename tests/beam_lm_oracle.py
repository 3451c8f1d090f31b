"""Float64 restatement of the CTC prefix beam search with a word n-gram LM (csrc/beam.cu beam_search_kernel<true>,
ops.ctc_beam_search(lm=...)), a direct dict-based ARPA scorer, exhaustive enumeration of the fused objective, and a
seeded synthetic ARPA writer, for the tests and tools/time_beam_search_lm.py.

Rules (ctcdecode's word-level scorer, written out as the contract of the search):
- the acoustic search of beam_oracle.py: pruning, keep / repeat / merge, top W by log(p_b + p_nb), ties to the lower q;
- a prefix is admissible when every run of labels a space follows is a word of V, the last run is a prefix of a word of
  V, and no space is first or follows a space; other extensions are neither candidates nor merged;
- a space that ends word w adds alpha * lm(w | h) + beta to the extension and to a merge into the beam holding that
  prefix, lm(w | h) = ln(10) * log10 P(w | last n - 1 words, <s>-padded) by ARPA back-off, -1000 for w outside V;
- after the last frame each non-empty beam not ending in a space gets the same term for its last word (-1000 before
  alpha if incomplete), then the beams are re-ranked by it, ties to the earlier rank.
"""
import math
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import beam_oracle as BO  # noqa: E402

NEG = -math.inf
OOV = -1000.0
LN10 = math.log(10.0)
SPECIAL = ('<s>', '</s>', '<unk>')


class DirectScorer:
	"""ARPA back-off straight from the text: dicts of word tuples"""

	def __init__(self, path):
		self.prob, self.bo = {}, {}
		order, k = 0, 0
		for line in open(path, encoding = 'utf-8'):
			t = line.strip()
			if not t:
				continue
			if t.startswith('ngram '):
				order = max(order, int(t[6:].split('=')[0]))
			elif t.startswith('\\') and t.endswith('-grams:'):
				k = int(t[1:-7])
			elif t.startswith('\\'):
				k = 0
			elif k:
				parts = t.split()
				ws = tuple(parts[1:k + 1])
				self.prob[ws] = float(parts[0])
				if len(parts) == k + 2:
					self.bo[ws] = float(parts[-1])
		self.order = order
		self.vocab = {w[0] for w in self.prob if len(w) == 1 and w[0] not in SPECIAL}

	def log10p(self, h, w):
		if h + (w, ) in self.prob:
			return self.prob[h + (w, )]
		return self.bo.get(h, 0.0) + self.log10p(h[1:], w)

	def score(self, context, w):
		"""lm(w | context) in natural log; context: the completed words so far (any length, <s>-padded here)"""
		if w not in self.vocab:
			return OOV
		n = self.order
		h = (('<s>', ) * n + tuple(context))[len(context) + 1:] if n > 1 else ()
		return LN10 * self.log10p(h, w)


def spelling(words, labels, blank):
	"""prefix string -> bool [C]: the labels that extend it to a prefix of a spellable word, and the spellable words"""
	space = labels.index(' ')
	ok = {l for c, l in enumerate(labels) if c not in (blank, space)}
	spellable = {w for w in words if all(ch in ok for ch in w)}
	cid = {l: c for c, l in enumerate(labels)}
	allowed = {}
	for w in spellable:
		for i in range(len(w)):
			allowed.setdefault(w[:i], np.zeros(len(labels), dtype = bool))[cid[w[i]]] = True
	return allowed, spellable


def lm_beam_search(log_probs, scorer, labels, alpha, beta, output_lengths = None, beam_width = 100, cutoff_top_n = 40, cutoff_prob = 1.0,
					blank = None):
	"""log_probs [B, C, T] -> per utterance the beams best first by fused score: (tokens, emission frames, score)"""
	lp_all = np.asarray(log_probs, dtype = np.float64)
	B, C, T = lp_all.shape
	blank = C - 1 if blank is None else int(blank)
	space = labels.index(' ')
	W, n_ctx = int(beam_width), scorer.order - 1
	allowed, spellable = spelling(scorer.vocab, labels, blank)
	none = np.zeros(C, dtype = bool)
	results = []
	for b in range(B):
		olen = T if output_lengths is None else max(0, min(T, int(output_lengths[b])))
		frames_pruned = BO.prune(lp_all[b, :, :olen].T, cutoff_top_n, cutoff_prob)
		prefixes, emitted = [()], [()]
		pb, pnb, last = np.array([0.0]), np.array([NEG]), np.array([-1])
		word, ctx, bonus = [''], [()], np.array([0.0])
		for t in range(olen):
			cls, vals = frames_pruned[t]
			n, nb = len(cls), len(prefixes)
			where = {int(c): k for k, c in enumerate(cls)}
			kb, ks = where.get(blank), where.get(space)
			tot = np.logaddexp(pb, pnb)
			kpb = tot + vals[kb] if kb is not None else np.full(nb, NEG)
			kl = np.array([where.get(int(c), -1) for c in last])
			kpnb = np.where(kl >= 0, pnb + vals[np.maximum(kl, 0)], NEG)
			merged = np.zeros((nb, n), dtype = bool)
			rank = {p: i for i, p in enumerate(prefixes)}
			for j in range(nb):
				if kl[j] < 0 or not prefixes[j]:
					continue
				p = rank.get(prefixes[j][:-1])
				if p is None:
					continue
				e = (pb[p] if last[p] == last[j] else tot[p]) + vals[kl[j]] + bonus[j]
				kpnb[j] = np.logaddexp(kpnb[j], e)
				merged[p, kl[j]] = True
			spb = np.array([alpha * scorer.score(ctx[i], word[i]) + beta if ks is not None and word[i] in spellable else NEG for i in range(nb)])
			adm = np.stack([allowed.get(word[i], none) for i in range(nb)])[:, cls]
			ext = np.where(cls[None, :] == last[:, None], pb[:, None], tot[:, None]) + vals[None, :]
			ext[:, cls == blank] = NEG
			ext[merged] = NEG
			nonspace = (cls != space) & (cls != blank)
			ext[:, nonspace] = np.where(adm[:, nonspace], ext[:, nonspace], NEG)
			if ks is not None:
				ext[:, ks] += spb
			score = np.concatenate([np.logaddexp(kpb, kpnb)[:, None], ext], axis = 1).reshape(-1)
			q = np.nonzero(score > NEG)[0]
			q = q[np.lexsort((q, -score[q]))][:W]
			i, s = np.divmod(q, n + 1)
			new = dict(pre = [], emit = [], word = [], ctx = [], bonus = [])
			for ii, ss in zip(i.tolist(), s.tolist()):
				if ss == 0:
					new['pre'].append(prefixes[ii]); new['emit'].append(emitted[ii]); new['word'].append(word[ii]); new['ctx'].append(ctx[ii])
					new['bonus'].append(bonus[ii])
				else:
					c = int(cls[ss - 1])
					new['pre'].append(prefixes[ii] + (c, )); new['emit'].append(emitted[ii] + (t, ))
					if c == space:
						new['word'].append(''); new['ctx'].append((ctx[ii] + (word[ii], ))[-n_ctx:] if n_ctx else ())
						new['bonus'].append(spb[ii])
					else:
						new['word'].append(word[ii] + labels[c]); new['ctx'].append(ctx[ii]); new['bonus'].append(0.0)
			keep = s == 0
			k = np.maximum(s - 1, 0)
			pb = np.where(keep, kpb[i], NEG)
			pnb = np.where(keep, kpnb[i], ext[i, k])
			last = np.where(keep, last[i], cls[k])
			prefixes, emitted, word, ctx, bonus = new['pre'], new['emit'], new['word'], new['ctx'], np.array(new['bonus'])
			if not prefixes:
				break
		final = []
		for r, p in enumerate(prefixes):
			f = float(np.logaddexp(pb[r], pnb[r]))
			if p and p[-1] != space:
				f += alpha * (scorer.score(ctx[r], word[r]) if word[r] in spellable else OOV) + beta
			final.append(f)
		order = sorted(range(len(prefixes)), key = lambda r: (-final[r], r))
		results.append([(prefixes[r], emitted[r], final[r]) for r in order])
	return results


def fused_labelings(lp, scorer, labels, alpha, beta, blank, ctc_loss_np):
	"""Every admissible labeling of nonzero CTC probability for one utterance lp [C, T], ranked by ln P_ctc + the bonuses
	of its words + the end term (exhaustive; tiny T, C only)"""
	space = labels.index(' ')
	allowed, spellable = spelling(scorer.vocab, labels, blank)
	out = []
	for l, lnp in BO.labelings_by_probability(lp, blank, ctc_loss_np):
		text = ''.join(labels[c] for c in l)
		runs = text.split(' ')
		if text.startswith(' ') or '  ' in text or any(r not in spellable for r in runs[:-1]) or runs[-1] not in allowed and runs[-1] not in spellable:
			continue
		f, ctx = lnp, ()
		for w in runs[:-1]:
			f += alpha * scorer.score(ctx, w) + beta
			ctx += (w, )
		if l and l[-1] != space:
			f += alpha * (scorer.score(ctx, runs[-1]) if runs[-1] in spellable else OOV) + beta
		out.append((l, f))
	out.sort(key = lambda x: -x[1])
	return out


RU = 'абвгдеёжзийклмнопрстуфхцчшщъыьэюя'


def random_words(n, seed, alphabet = RU, lengths = (2, 9)):
	"""n distinct words over alphabet, lengths uniform in [lengths[0], lengths[1])"""
	rng = np.random.default_rng(seed)
	letters = np.array(list(alphabet))
	out, seen = [], set()
	while len(out) < n:
		m = 2 * (n - len(out)) + 16
		ln = rng.integers(lengths[0], lengths[1], m)
		ch = letters[rng.integers(0, len(letters), (m, lengths[1]))]
		for r in range(m):
			w = ''.join(ch[r, :ln[r]])
			if w not in seen:
				seen.add(w)
				out.append(w)
				if len(out) == n:
					break
	return out


def write_synthetic_arpa(path, words, seed, n_bigrams, n_trigrams):
	"""A seeded 3-gram ARPA over words: random log10 probabilities and back-offs (not normalised; the search does not
	need it), bigrams over (<s> | words) x words, trigrams extending listed bigrams; about one context in three has no
	back-off listed"""
	rng = np.random.default_rng(seed)
	vocab = ['<unk>', '<s>', '</s>'] + list(words)
	V, first = len(vocab), 3
	hist = np.concatenate([[1], np.arange(first, V)])  # <s> and the words
	bi = np.unique(rng.choice(hist, n_bigrams) * V + rng.integers(first, V, n_bigrams))
	tri_src = rng.integers(0, len(bi), n_trigrams)
	tri = np.unique(bi[tri_src] * V + rng.integers(first, V, n_trigrams))
	tri = tri[(tri // V) % V != 1]  # no <s> in the middle of a context

	def f(x):
		return f'{x:.4f}'

	with open(path, 'w', encoding = 'utf-8') as out:
		out.write(f'\\data\\\nngram 1={V}\nngram 2={len(bi)}\nngram 3={len(tri)}\n\n\\1-grams:\n')
		up = rng.uniform(-6.0, -1.5, V)
		ub = rng.uniform(-1.0, 0.0, V)
		up[1] = -99.0
		for i, w in enumerate(vocab):
			out.write(f'{f(up[i])}\t{w}' + (f'\t{f(ub[i])}' if i != 2 and rng.random() < 0.7 else '') + '\n')
		out.write('\n\\2-grams:\n')
		bp, bb, has = rng.uniform(-4.0, -0.3, len(bi)), rng.uniform(-1.0, 0.0, len(bi)), rng.random(len(bi)) < 0.7
		out.write(''.join(f'{f(bp[i])}\t{vocab[x // V]} {vocab[x % V]}' + (f'\t{f(bb[i])}' if has[i] else '') + '\n' for i, x in enumerate(bi.tolist())))
		out.write('\n\\3-grams:\n')
		tp = rng.uniform(-3.0, -0.1, len(tri))
		out.write(''.join(f'{f(tp[i])}\t{vocab[x // (V * V)]} {vocab[(x // V) % V]} {vocab[x % V]}\n' for i, x in enumerate(tri.tolist())))
		out.write('\n\\end\\\n')
	return vocab


def planted(B, C, T, label_seqs, blank, g, scale = 6.0):
	"""[B, C, T] log-probs (torch) with each utterance's label sequence planted at evenly spread frames over randn"""
	import torch
	import torch.nn.functional as F
	path = torch.full((B, T), blank)
	for b, seq in enumerate(label_seqs):
		pos = torch.linspace(0, T - 1, len(seq)).long()
		path[b, pos] = torch.tensor(seq)
	return (torch.randn(B, C, T, generator = g) + scale * F.one_hot(path, C).permute(0, 2, 1)).log_softmax(1)
