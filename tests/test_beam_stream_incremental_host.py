"""Incremental streaming CTC prefix beam search, host side (no device): the workspace query, the C ABI's refusals of
cab_ctc_beam_search_stream_incremental (checked before any launch; every refused call names its reason), the window
policy of ops.BeamStreamState, and the refusal of mixing incremental and full-history calls on one state."""
import ctypes

import pytest
import torch

from convasr_b200 import _lib, ops
from convasr_b200.decoders import OnlineBeamSearchDecoder


def test_row_layout():
	assert ctypes.sizeof(_lib.BeamStreamIncrementalRow) == 72
	assert _lib.BeamStreamIncrementalRow.base.offset == 32 and _lib.BeamStreamIncrementalRow.commit.offset == 48


def test_workspace_query():
	lib = _lib.load()
	n, m = ctypes.c_int64(), ctypes.c_int64()
	assert lib.cab_ctc_beam_search_stream_incremental_workspace(2, 50, 40, 100, 4, ctypes.byref(n)) == 0
	assert lib.cab_ctc_beam_search_stream_workspace(2, 50, 40, 100, 4, ctypes.byref(m)) == 0
	assert n.value > m.value
	for args in ((0, 10, 40, 100, 4), (2, -1, 40, 100, 4), (2, 10, 65, 100, 4), (2, 10, 40, 129, 4), (2, 10, 40, 100, 101)):
		assert lib.cab_ctc_beam_search_stream_incremental_workspace(*args, ctypes.byref(n)) != 0
	assert lib.cab_ctc_beam_search_stream_incremental_workspace(2, 10, 40, 100, 4, None) != 0


FAKE = 1 << 20  # a non-null address; every call below is refused before anything dereferences it


def test_c_abi_refusals_name_their_reason():
	lib = _lib.load()
	B, C, T, N, W, K = 2, 38, 10, 38, 16, 2
	sb = ops.beam_stream_state_bytes(W)

	def rows(**kw):
		r = (_lib.BeamStreamIncrementalRow * B)()
		for b in range(B):
			r[b].state, r[b].nodes, r[b].state_bytes, r[b].capacity, r[b].t0, r[b].frames, r[b].commit = FAKE * (b + 1), FAKE * 8, sb, 4 * T, 0, T, -1
		for k, v in kw.items():
			setattr(r[1], k, v)
		return r

	def call(r, W = W, N = N, K = K, blank = C - 1, cutoff = 1.0, ws_bytes = 1 << 30, L_cap = 4 * T, lp = FAKE, T = T, out = FAKE):
		return lib.cab_ctc_beam_search_stream_incremental(lp, C * T, T, 1, r, B, T, C, N, cutoff, blank, W, K, FAKE, ws_bytes, FAKE, FAKE, FAKE, out,
															FAKE, FAKE, L_cap, FAKE, FAKE, None, 0.0, 0.0, 0, None)

	before = _lib.launch_count()
	cases = [(dict(r = rows(finished = 1)), 'has ended'), (dict(r = rows(t0 = 3 * T + 1)), 'overruns'), (dict(r = rows(t0 = 4 * T + 1)), 'overruns'),
			(dict(r = rows(frames = T + 1)), 'frames='), (dict(r = rows(frames = -1)), 'frames='), (dict(r = rows(state = FAKE)), 'share a state block'),
			(dict(r = rows(state_bytes = sb - 16)), 'state block of'), (dict(r = rows(state = None)), 'null state'),
			(dict(r = rows(nodes = None)), 'null state'), (dict(r = rows(capacity = (1 << 31) // W)), 'capacity'), (dict(r = None), 'null pointer'),
			(dict(r = rows(), out = None), 'null pointer'), (dict(r = rows(base = -1)), 'base'),
			(dict(r = rows(commit = -2)), 'commit node'), (dict(r = rows(t0 = 5, commit = 5 * W)), 'commit node'),
			(dict(r = rows(t0 = 20, commit = 10 * W + 3, shift = 11)), 'shift='), (dict(r = rows(t0 = 20, commit = 12 * W, shift = 9)), 'overlap'),
			(dict(r = rows(t0 = 20, shift = 1)), 'shift='), (dict(r = rows(t0 = 20, commit = 12 * W, shift = -1)), 'shift='),
			(dict(r = rows(t0 = 20), L_cap = 29), 'L_cap'), (dict(r = rows(t0 = 20, commit = 12 * W + 5), L_cap = 16), 'L_cap'),
			(dict(r = rows(), W = 0), 'beam_width'), (dict(r = rows(), W = 129), 'beam_width'), (dict(r = rows(), N = 0), 'N='),
			(dict(r = rows(), N = 65), 'N='), (dict(r = rows(), K = 0), 'K='), (dict(r = rows(), K = W + 1), 'K='), (dict(r = rows(), blank = C), 'blank'),
			(dict(r = rows(), blank = -1), 'blank'), (dict(r = rows(), cutoff = 0.0), 'cutoff_prob'), (dict(r = rows(), cutoff = 1.5), 'cutoff_prob'),
			(dict(r = rows(), ws_bytes = 64), 'workspace'), (dict(r = rows(), L_cap = 0), 'L_cap'), (dict(r = rows(), lp = None), 'null log_probs')]
	for kw, msg in cases:
		assert call(**kw) != 0, msg
		assert msg in lib.cab_last_error().decode(), (msg, lib.cab_last_error())
	assert _lib.launch_count() == before
	# the window bound: the frames after the commit node's frame (12) of t0 = 20, plus 10 new ones, are 17; the row then
	# passes that check and fails the next one
	assert call(rows(t0 = 20, commit = 12 * W + 5, state = FAKE), L_cap = 17) != 0 and 'share a state block' in lib.cab_last_error().decode()


def test_lm_arguments_are_checked():
	lib = _lib.load()
	B, C, T, W = 1, 38, 4, 8
	r = (_lib.BeamStreamIncrementalRow * 1)()
	r[0].state, r[0].nodes, r[0].state_bytes, r[0].capacity, r[0].frames, r[0].commit = FAKE, FAKE * 2, 1 << 20, T, T, -1
	lm = _lib.NgramLM()
	lm.order, lm.num_classes, lm.num_nodes, lm.bos = 3, 37, 1, 0

	def call(s, space = 36, alpha = 0.5):
		return lib.cab_ctc_beam_search_stream_incremental(FAKE, C * T, T, 1, r, B, T, C, 38, 1.0, 37, W, 1, FAKE, 1 << 30, FAKE, FAKE, FAKE, FAKE,
															FAKE, FAKE, T, FAKE, FAKE, ctypes.byref(s), alpha, 0.0, space, None)

	assert call(lm) != 0 and 'classes' in lib.cab_last_error().decode()
	lm.num_classes = 38
	assert call(lm) != 0 and 'lm trie' in lib.cab_last_error().decode()


def test_window_policy():
	"""the window drops the frames before the commit node's frame once that frame reaches half the capacity, and grows by
	doubling only when the frames after it and the call's frames do not fit"""
	W = 4
	s = ops.BeamStreamState(capacity = 8)
	s.nodes = torch.zeros(8, W, 2, dtype = torch.int32)
	s.state = torch.zeros(16, dtype = torch.uint8)
	s.t0, s.commit = 7, 3 * W + 1  # commit frame 3 < 8 / 2: kept
	assert s._window(1, W, 16, 'cpu') == 0 and s.capacity == 8
	s.commit = 4 * W  # frame 4: the window may start there
	assert s._window(5, W, 16, 'cpu') == 4 and s.capacity == 8
	s.commit = 4 * W + 2
	assert s._window(6, W, 16, 'cpu') == 4 and s.capacity == 16  # 3 + 6 frames do not fit in 8
	s.commit = -1
	assert s._window(2, W, 16, 'cpu') == 0 and s.capacity == 16


LABELS = list('abc ') + ['_']


def test_incremental_and_full_history_calls_do_not_mix():
	cpu = torch.zeros(1, len(LABELS), 4)
	dec = OnlineBeamSearchDecoder(LABELS, beam_width = 8)
	st = dec.new_state()
	st.incremental = True  # as after a first incremental call
	with pytest.raises(RuntimeError, match = 'incremental calls'):
		dec.decode(cpu, [st], is_eos = False)
	with pytest.raises(RuntimeError, match = 'incremental calls'):
		dec.decode_nbest(cpu, [st], is_eos = False)
	with pytest.raises(RuntimeError, match = 'incremental calls'):
		ops.ctc_beam_search_stream(cpu, [st], False, beam_width = 8)
	full = dec.new_state()
	full.search = (len(LABELS), len(LABELS) - 1, 8, 5, 1.0, 1, None, 0.0, 0.0)  # as after a full-history call
	with pytest.raises(RuntimeError, match = 'full-history calls'):
		dec.decode_incremental(cpu, [full], is_eos = False)
	with pytest.raises(RuntimeError, match = 'full-history calls'):
		ops.ctc_beam_search_stream_incremental(cpu, [full], False, beam_width = 8)


def test_python_refusals():
	cpu = torch.zeros(1, len(LABELS), 4)
	dec = OnlineBeamSearchDecoder(LABELS, beam_width = 8)
	st = dec.new_state()
	with pytest.raises(RuntimeError, match = 'CUDA'):  # no CPU fallback
		dec.decode_incremental(cpu, [st], is_eos = False)
	with pytest.raises(ValueError, match = 'not made by this decoder'):
		OnlineBeamSearchDecoder(LABELS, beam_width = 16).decode_incremental(cpu, [st], is_eos = False)
	with pytest.raises(ValueError, match = 'classes'):
		dec.decode_incremental(torch.zeros(1, len(LABELS) + 1, 4), [st], is_eos = False)
	s2 = ops.BeamStreamState()
	with pytest.raises(ValueError, match = 'two rows'):
		ops.ctc_beam_search_stream_incremental(torch.zeros(2, 5, 4), [s2, s2], False)
	s2.search, s2.incremental = (5, 4, 8, 5, 1.0, 1, None, 0.0, 0.0), True
	with pytest.raises(ValueError, match = 'another search configuration'):
		ops.ctc_beam_search_stream_incremental(torch.zeros(1, 5, 4), [s2], False, beam_width = 16)
	s2.finished = True
	with pytest.raises(RuntimeError, match = 'ended'):
		dec.decode_incremental(cpu, [s2], is_eos = False)
