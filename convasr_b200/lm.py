"""Word n-gram language model for the GPU beam search (decoders.BeamSearchDecoder with lm_path='<file>.arpa').

`NGramLM.from_arpa(path, labels, blank)` parses an ARPA file (KenLM's text format, log10 values, order 1..6) on the
host and builds the tables `cab_ctc_beam_search_lm` reads:
- per order k, an open-addressing table in KenLM's "probing" layout: a power-of-two number of 16-byte entries
  {uint64 key, float log10 p, float log10 back-off}, key 0 = empty slot, linear probing from key & (size - 1).  The key
  of a word-id sequence folds the ids newest first through the splitmix64 step of csrc/beam.cu (`beam_hash`).  Two
  distinct n-grams of one order never share a key: the build checks it and refuses otherwise.
- a dictionary trie over label ids: child int32 [nodes, C] (-1 = no child, node 0 = the root) and the word id each
  node spells (-1 = none).  Words that use a character outside the labels cannot be spelled; they stay in the LM.

Word ids are the positions of the 1-grams in the file.  The vocabulary V is the 1-gram words except <s>, </s> and <unk>.
"""
import math
import os

import numpy as np

MAX_ORDER = 6  # KenLM's default maximum order (CAB_NGRAM_MAX_ORDER)
OOV_SCORE = -1000.0  # ctcdecode's OOV_SCORE: natural log, before alpha
SPECIAL = ('<s>', '</s>', '<unk>')

def _fold(h, ids):
	"""csrc/beam.cu beam_hash on uint64 arrays: h + 0x9E3779B97F4A7C15 * (id + 1), then the splitmix64 finaliser"""
	with np.errstate(over = 'ignore'):
		z = h + np.uint64(0x9E3779B97F4A7C15) * (ids.astype(np.uint64) + np.uint64(1))
		z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
		z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
		return z ^ (z >> np.uint64(31))


def ngram_keys(ids):
	"""int [count, k] word-id sequences (oldest first) -> uint64 [count] keys, folded newest first"""
	ids = np.asarray(ids, dtype = np.int64)
	h = np.zeros(ids.shape[0], dtype = np.uint64)
	for j in range(ids.shape[1] - 1, -1, -1):
		h = _fold(h, ids[:, j])
	return h


ENTRY = np.dtype([('key', '<u8'), ('log10_p', '<f4'), ('log10_bo', '<f4')])


def _probing_table(keys, p, bo, order):
	"""open addressing, linear probing, load <= 1/2; slots claimed in n-gram order"""
	count = len(keys)
	size = 1 << max(1, int(2 * count - 1).bit_length())
	mask = np.uint64(size - 1)
	table = np.zeros(size, dtype = ENTRY)
	if count == 0:
		return table
	if np.any(keys == 0):
		raise ValueError(f'ARPA {order}-grams: an n-gram hashes to the empty-slot key 0')
	srt = np.sort(keys)
	if np.any(srt[1:] == srt[:-1]):  # parse_arpa refuses repeated n-grams, so these are distinct ones
		raise ValueError(f'ARPA {order}-grams: two distinct n-grams share a 64-bit key')
	slot = keys & mask
	todo = np.arange(count)
	taken = np.zeros(size, dtype = bool)
	while todo.size:
		s = slot[todo]
		free = ~taken[s]
		# the first entry (in n-gram order) that asks for a free slot gets it; the others move one slot on
		_, first = np.unique(s, return_index = True)
		win = np.zeros(todo.size, dtype = bool)
		win[first] = True
		win &= free
		placed = todo[win]
		table['key'][slot[placed]] = keys[placed]
		table['log10_p'][slot[placed]] = p[placed]
		table['log10_bo'][slot[placed]] = bo[placed]
		taken[slot[placed]] = True
		todo = todo[~win]
		slot[todo] = (slot[todo] + np.uint64(1)) & mask
	return table


def parse_arpa(path):
	"""-> (order, words [list, file order], grams [per order k: (ids int64 [count, k], log10 p float64, log10 bo float64)]).
	Malformed input raises ValueError naming the line."""
	with open(path, encoding = 'utf-8') as f:
		lines = f.read().split('\n')
	i, n = 0, len(lines)

	def bad(j, what):
		return ValueError(f'{path}:{j + 1}: {what}')

	while i < n and lines[i].strip() != '\\data\\':
		if lines[i].strip():
			raise bad(i, f'expected \\data\\, got {lines[i].strip()[:40]!r}')
		i += 1
	if i == n:
		raise ValueError(f'{path}: no \\data\\ header (not an ARPA file)')
	i += 1
	counts = {}
	while i < n and lines[i].strip():
		t = lines[i].strip()
		if not t.startswith('ngram ') or '=' not in t:
			raise bad(i, f'expected "ngram k=count", got {t[:40]!r}')
		k, _, c = t[6:].partition('=')
		try:
			k, c = int(k), int(c)
		except ValueError:
			raise bad(i, f'expected "ngram k=count", got {t[:40]!r}') from None
		if k != len(counts) + 1 or c < 0:
			raise bad(i, f'ngram orders must run 1, 2, ... with counts >= 0, got {t!r}')
		counts[k] = c
		i += 1
	order = len(counts)
	if order < 1:
		raise ValueError(f'{path}: the \\data\\ header lists no n-gram counts')
	if order > MAX_ORDER:
		raise ValueError(f'{path}: order {order} exceeds {MAX_ORDER}, the largest the search supports')
	word_id = {}
	words = []
	grams = []
	for k in range(1, order + 1):
		while i < n and not lines[i].strip():
			i += 1
		if i == n or lines[i].strip() != f'\\{k}-grams:':
			raise bad(min(i, n - 1), f'expected \\{k}-grams:')
		head = i
		i += 1
		start = i
		while i < n and lines[i].strip() and not lines[i].startswith('\\'):
			i += 1
		body = lines[start:i]
		if len(body) != counts[k]:
			raise bad(head, f'the header says ngram {k}={counts[k]}, the section has {len(body)} entries')
		ids = np.empty((len(body), k), dtype = np.int64)
		p = np.empty(len(body), dtype = np.float64)
		bo = np.zeros(len(body), dtype = np.float64)
		for r, line in enumerate(body):
			parts = line.split()
			if len(parts) not in (k + 1, k + 2):
				raise bad(start + r, f'a {k}-gram line has log10 p, {k} words and an optional back-off')
			try:
				p[r] = float(parts[0])
				if len(parts) == k + 2:
					bo[r] = float(parts[-1])
			except ValueError:
				raise bad(start + r, 'unreadable number') from None
			if not (math.isfinite(p[r]) and math.isfinite(bo[r])):
				raise bad(start + r, 'values must be finite')
			ws = parts[1:k + 1]
			if k == 1:
				if ws[0] in word_id:
					raise bad(start + r, f'duplicate 1-gram {ws[0]!r}')
				word_id[ws[0]] = len(words)
				words.append(ws[0])
				ids[r, 0] = word_id[ws[0]]
			else:
				for j, w in enumerate(ws):
					wid = word_id.get(w)
					if wid is None:
						raise bad(start + r, f'word {w!r} is not a 1-gram')
					ids[r, j] = wid
		if k > 1 and len(body):
			# the same words listed twice: report the second line
			srt = np.lexsort(ids.T[::-1])
			same = np.all(ids[srt[1:]] == ids[srt[:-1]], axis = 1)
			if same.any():
				r = int(max(srt[1:][same][0], srt[:-1][same][0]))
				raise bad(start + r, f'duplicate {k}-gram {" ".join(words[x] for x in ids[r])!r}')
		grams.append((ids, p, bo))
	while i < n and not lines[i].strip():
		i += 1
	if i == n or lines[i].strip() != '\\end\\':
		raise bad(min(i, n - 1), 'expected \\end\\')
	if '<s>' not in word_id:
		raise ValueError(f'{path}: no <s> 1-gram')
	return order, words, grams


class NGramLM:
	"""Host tables and their device copies; `device_struct(device)` gives the cab_ngram_lm_t the kernel reads."""

	def __init__(self, order, words, grams, labels, blank):
		self.order, self.words = order, words
		self.word_id = {w: i for i, w in enumerate(words)}
		self.bos = self.word_id['<s>']
		self.labels = list(labels)
		self.blank = blank
		self.space = self.labels.index(' ')
		self.vocab = [w for w in words if w not in SPECIAL]
		if all(len(w) == 1 for w in self.vocab):
			raise NotImplementedError('convasr_b200: a character-level LM (every word one character) is not supported; '
										'the beam search fuses a word-level LM')
		self.tables = [_probing_table(ngram_keys(ids), p, bo, k + 1) for k, (ids, p, bo) in enumerate(grams)]
		self._build_trie()
		self._device = {}

	@classmethod
	def from_arpa(cls, path, labels, blank = None):
		"""labels: the C single-character label strings, one of them ' '; blank: the blank's label id (None = C - 1)"""
		labels = list(labels)
		for c, l in enumerate(labels):
			if not isinstance(l, str) or len(l) != 1:
				raise ValueError(f'convasr_b200: LM decoding needs single-character labels; label {c} is {l!r}')
		if ' ' not in labels:
			raise ValueError("convasr_b200: LM decoding needs a space label (' ') to end words")
		blank = len(labels) - 1 if blank is None else int(blank)
		if not 0 <= blank < len(labels) or labels[blank] == ' ':
			raise ValueError(f'convasr_b200: blank={blank} out of range or the space label')
		order, words, grams = parse_arpa(path)
		return cls(order, words, grams, labels, blank)

	def _build_trie(self):
		C = len(self.labels)
		char_id = {l: c for c, l in enumerate(self.labels) if c != self.blank and c != self.space}
		children = [{}]
		word = [-1]
		for w in self.vocab:
			if not all(ch in char_id for ch in w):
				continue  # cannot be spelled with these labels
			node = 0
			for ch in w:
				c = char_id[ch]
				nxt = children[node].get(c)
				if nxt is None:
					nxt = len(children)
					children[node][c] = nxt
					children.append({})
					word.append(-1)
				node = nxt
			word[node] = self.word_id[w]
		self.child = np.full((len(children), C), -1, dtype = np.int32)
		for node, ch in enumerate(children):
			if ch:
				self.child[node, list(ch.keys())] = list(ch.values())
		self.word = np.asarray(word, dtype = np.int32)

	@property
	def nbytes(self):
		"""bytes of the device tables: n-gram entries, trie children and node words"""
		return sum(t.nbytes for t in self.tables) + self.child.nbytes + self.word.nbytes

	def score_ids(self, context, w):
		"""ln P(w | context) by the kernel's lookup (csrc/beam.cu lm_word_score) on the host tables: context = the last
		order - 1 word ids, oldest first; OOV_SCORE when w has no 1-gram.  A host mirror for the tests."""
		n = self.order
		context = list(context)[-(n - 1):] if n > 1 else []
		assert len(context) == n - 1

		def probe(k, key):
			t = self.tables[k - 1]
			mask = len(t) - 1
			s = int(key) & mask
			while t['key'][s] != key and t['key'][s] != 0:
				s = (s + 1) & mask
			return t[s] if t['key'][s] == key else None

		bo = np.float32(0.0)
		for k in range(n, 0, -1):
			e = probe(k, ngram_keys([context[n - k:] + [w]])[0])
			if e is not None:
				return float(np.float32(2.302585093) * (bo + e['log10_p']))
			if k > 1:
				c = probe(k - 1, ngram_keys([context[n - k:]])[0])
				if c is not None:
					bo = np.float32(bo + c['log10_bo'])
		return OOV_SCORE

	def device_struct(self, device):
		"""the cab_ngram_lm_t of the tables on `device` (uploaded once per device and kept)"""
		import torch
		from . import _lib
		key = str(device)
		if key not in self._device:
			tabs = [torch.from_numpy(t.view(np.uint8)).to(device) for t in self.tables]
			child = torch.from_numpy(self.child).to(device)
			word = torch.from_numpy(self.word).to(device)
			s = _lib.NgramLM()
			s.order, s.num_classes, s.num_nodes, s.bos = self.order, len(self.labels), len(self.word), self.bos
			for k, t in enumerate(tabs):
				s.tables[k] = t.data_ptr()
				s.sizes[k] = len(self.tables[k])
			s.child, s.word = child.data_ptr(), word.data_ptr()
			self._device[key] = (s, tabs, child, word)
		return self._device[key][0]


_CACHE = {}
_CACHE_MAX = 2  # LMs kept loaded (host tables and their device copies); the least recently used one is dropped first


def load_arpa(path, labels, blank = None):
	"""NGramLM.from_arpa, cached per (real path, mtime, labels, blank): parsing runs once per file.  An entry for the same
	path with another mtime is dropped when the file changes, and at most _CACHE_MAX LMs stay loaded."""
	real = os.path.realpath(path)
	key = (real, os.stat(real).st_mtime_ns, tuple(labels), blank)
	lm = _CACHE.pop(key, None)
	if lm is None:
		for k in [k for k in _CACHE if k[0] == real and k[1] != key[1]]:
			del _CACHE[k]
		lm = NGramLM.from_arpa(real, labels, blank)
	_CACHE[key] = lm  # most recently used last
	while len(_CACHE) > _CACHE_MAX:
		del _CACHE[next(iter(_CACHE))]
	return lm
