"""Streaming CTC prefix beam search, host side (no device): the state-bytes and workspace queries, the C ABI's refusals
(checked before any launch; every refused call here names its reason) and the Python refusals of
ops.ctc_beam_search_stream and decoders.OnlineBeamSearchDecoder."""
import ctypes

import pytest
import torch

from convasr_b200 import _lib, ops
from convasr_b200.decoders import OnlineBeamSearchDecoder


def state_bytes(W, order = 0):
	n = ctypes.c_int64()
	rc = _lib.load().cab_ctc_beam_search_stream_state_bytes(W, order, ctypes.byref(n))
	return rc, n.value


@pytest.mark.parametrize('W', [1, 16, 100, 128])
@pytest.mark.parametrize('order', [0, 1, 3, 6])
def test_state_bytes(W, order):
	# header {t0, count, finished, 0}; per beam: hash, parent hash (8 + 8), p_b, p_nb, last, node, parent rank (5 x 4); with an
	# LM: trie node, bonus (2 x 4) and order - 1 context words (4 each); rounded up to 16 bytes
	per_beam = 36 + (8 + 4 * (order - 1) if order else 0)
	rc, n = state_bytes(W, order)
	assert rc == 0 and n == (16 + W * per_beam + 15) // 16 * 16
	assert ops.beam_stream_state_bytes(W, order) == n


def test_state_bytes_refusals():
	lib = _lib.load()
	for W, order in ((0, 0), (129, 0), (16, -1), (16, 7)):
		assert state_bytes(W, order)[0] != 0
		assert lib.cab_last_error()
	assert lib.cab_ctc_beam_search_stream_state_bytes(16, 0, None) != 0


def test_workspace_query():
	lib = _lib.load()
	n = ctypes.c_int64()
	assert lib.cab_ctc_beam_search_stream_workspace(2, 0, 40, 100, 4, ctypes.byref(n)) == 0 and n.value > 0
	small = n.value
	assert lib.cab_ctc_beam_search_stream_workspace(2, 50, 40, 100, 4, ctypes.byref(n)) == 0 and n.value >= small + 2 * 50 * (40 * 8 + 4)
	for args in ((0, 10, 40, 100, 4), (2, -1, 40, 100, 4), (2, 10, 65, 100, 4), (2, 10, 40, 129, 4), (2, 10, 40, 100, 101)):
		assert lib.cab_ctc_beam_search_stream_workspace(*args, ctypes.byref(n)) != 0


FAKE = 1 << 20  # a non-null address; every call below is refused before anything dereferences it


def test_c_abi_refusals_name_their_reason():
	lib = _lib.load()
	B, C, T, N, W, K = 2, 38, 10, 38, 16, 2
	sb = ops.beam_stream_state_bytes(W)

	def rows(**kw):
		r = (_lib.BeamStreamRow * B)()
		for b in range(B):
			r[b].state, r[b].nodes, r[b].state_bytes, r[b].capacity, r[b].t0, r[b].frames = FAKE * (b + 1), FAKE * 8, sb, T, 0, T
		for k, v in kw.items():
			setattr(r[1], k, v)
		return r

	def call(r, W = W, N = N, K = K, blank = C - 1, cutoff = 1.0, ws_bytes = 1 << 30, L_cap = T, lp = FAKE, T = T):
		return lib.cab_ctc_beam_search_stream(lp, C * T, T, 1, r, B, T, C, N, cutoff, blank, W, K, FAKE, ws_bytes, FAKE, FAKE, L_cap, FAKE, FAKE,
												None, 0.0, 0.0, 0, None)

	before = _lib.launch_count()
	cases = [(dict(r = rows(finished = 1)), 'has ended'), (dict(r = rows(t0 = 1)), 'overruns'), (dict(r = rows(t0 = 5, capacity = 14)), 'overruns'),
			(dict(r = rows(frames = T + 1)), 'frames='), (dict(r = rows(frames = -1)), 'frames='), (dict(r = rows(state = FAKE)), 'share a state block'),
			(dict(r = rows(state_bytes = sb - 16)), 'state block of'), (dict(r = rows(state = None)), 'null state'),
			(dict(r = rows(nodes = None)), 'null state'), (dict(r = rows(capacity = (1 << 31) // W)), 'capacity'), (dict(r = None), 'null pointer'),
			(dict(r = rows(), W = 0), 'beam_width'), (dict(r = rows(), W = 129), 'beam_width'), (dict(r = rows(), N = 0), 'N='),
			(dict(r = rows(), N = 65), 'N='), (dict(r = rows(), K = 0), 'K='), (dict(r = rows(), K = W + 1), 'K='), (dict(r = rows(), blank = C), 'blank'),
			(dict(r = rows(), blank = -1), 'blank'), (dict(r = rows(), cutoff = 0.0), 'cutoff_prob'), (dict(r = rows(), cutoff = 1.5), 'cutoff_prob'),
			(dict(r = rows(), ws_bytes = 64), 'workspace'), (dict(r = rows(), L_cap = 0), 'L_cap'), (dict(r = rows(), lp = None), 'null log_probs')]
	for kw, msg in cases:
		assert call(**kw) != 0, msg
		assert msg in lib.cab_last_error().decode(), (msg, lib.cab_last_error())
	assert _lib.launch_count() == before


def test_lm_arguments_are_checked():
	lib = _lib.load()
	B, C, T, W = 1, 38, 4, 8
	r = (_lib.BeamStreamRow * 1)()
	r[0].state, r[0].nodes, r[0].state_bytes, r[0].capacity, r[0].frames = FAKE, FAKE * 2, 1 << 20, T, T
	lm = _lib.NgramLM()
	lm.order, lm.num_classes, lm.num_nodes, lm.bos = 3, 37, 1, 0

	def call(s, space = 36, alpha = 0.5):
		return lib.cab_ctc_beam_search_stream(FAKE, C * T, T, 1, r, B, T, C, 38, 1.0, 37, W, 1, FAKE, 1 << 30, FAKE, FAKE, T, FAKE, FAKE,
												ctypes.byref(s), alpha, 0.0, space, None)

	assert call(lm) != 0 and 'classes' in lib.cab_last_error().decode()
	lm.num_classes = 38
	assert call(lm) != 0 and 'lm trie' in lib.cab_last_error().decode()
	lm.order = 9
	assert call(lm) != 0 and 'order' in lib.cab_last_error().decode()


LABELS = list('abc ') + ['_']


def test_python_refusals():
	cpu = torch.zeros(1, len(LABELS), 4)
	dec = OnlineBeamSearchDecoder(LABELS, beam_width = 8)
	other = OnlineBeamSearchDecoder(LABELS, beam_width = 16)
	st = dec.new_state()
	with pytest.raises(RuntimeError, match = 'CUDA'):  # no CPU fallback
		dec.decode(cpu, [st], is_eos = False)
	with pytest.raises(ValueError, match = 'not made by this decoder'):  # mixed configurations
		other.decode(cpu, [st], is_eos = False)
	with pytest.raises(ValueError, match = 'not made by this decoder'):
		OnlineBeamSearchDecoder(LABELS[:-2] + ['d', '_'], beam_width = 8).decode(cpu, [st], is_eos = False)
	with pytest.raises(ValueError, match = 'classes'):  # C != len(labels)
		dec.decode(torch.zeros(1, len(LABELS) + 1, 4), [st], is_eos = False)
	st.finished = True
	with pytest.raises(RuntimeError, match = 'ended'):  # fed after eos
		dec.decode(cpu, [st], is_eos = False)
	with pytest.raises(RuntimeError, match = 'ended'):
		ops.ctc_beam_search_stream(cpu, [st], True)
	s2 = ops.BeamStreamState()
	with pytest.raises(ValueError, match = 'two rows'):
		ops.ctc_beam_search_stream(torch.zeros(2, 5, 4), [s2, s2], False)
	s2.search = (5, 4, 8, 5, 1.0, 1, None, 0.0, 0.0)
	with pytest.raises(ValueError, match = 'another search configuration'):
		ops.ctc_beam_search_stream(torch.zeros(1, 5, 4), [s2], False, beam_width = 16)
	with pytest.raises(ValueError, match = 'stream states'):
		ops.ctc_beam_search_stream(torch.zeros(2, 5, 4), [ops.BeamStreamState()], False)
