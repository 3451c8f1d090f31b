"""CTC prefix beam search (decoders.BeamSearchDecoder), host side: the float64 restatement against exhaustive enumeration
of CTC probabilities, its pruning rule, the refused arguments (Python and C ABI, no device needed) and the drop-in
export.  The GPU side is tests/test_gpu_beam_search.py."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import beam_oracle as BO  # noqa: E402
from oracle import oracle as O  # noqa: E402


def random_log_probs(B, C, T, seed, scale = 1.5):
	g = torch.Generator().manual_seed(seed)
	return (scale * torch.randn(B, C, T, generator = g, dtype = torch.float64)).log_softmax(1).float().numpy()


@pytest.mark.parametrize('C,T,blank,seed', [(2, 7, 1, 0), (3, 6, 2, 1), (3, 7, 0, 2), (4, 5, 3, 3), (4, 6, 0, 4), (4, 7, 3, 5)])
def test_oracle_equals_exhaustive_ctc_ranking(C, T, blank, seed):
	"""A beam wider than the number of prefixes and no pruning: the n-best list is every labeling of nonzero probability,
	ranked by exp(-ctc_loss_np), with the same log-probability"""
	lp = random_log_probs(1, C, T, seed)
	ref = BO.labelings_by_probability(lp[0].astype(np.float64), blank, O.ctc_loss_np)
	got = BO.ctc_prefix_beam_search(lp, beam_width = 4096, cutoff_top_n = C, blank = blank)[0]
	assert [h for h, _, _ in got] == [h for h, _ in ref]
	np.testing.assert_allclose([s for _, _, s in got], [s for _, s in ref], rtol = 0, atol = 1e-9)
	# emission frames: one per token, strictly increasing, within the utterance
	for h, e, _ in got:
		assert len(e) == len(h) and list(e) == sorted(set(e)) and all(0 <= f < T for f in e)


def test_oracle_output_lengths_and_empty_utterance():
	lp = random_log_probs(3, 4, 9, 7)
	full = BO.ctc_prefix_beam_search(lp, beam_width = 16, cutoff_top_n = 4)
	cut = BO.ctc_prefix_beam_search(lp, [9, 5, 0], beam_width = 16, cutoff_top_n = 4)
	assert cut[0] == full[0]
	assert cut[1] == BO.ctc_prefix_beam_search(lp[1:2, :, :5], beam_width = 16, cutoff_top_n = 4)[0]
	assert cut[2] == [((), (), 0.0)]  # no frames: the empty labeling with probability one


def test_prune_top_n_ties_and_order():
	lp = np.log(np.array([[0.1, 0.3, 0.2, 0.3, 0.1]]))
	cls, vals = BO.prune(lp, 2)[0]
	assert cls.tolist() == [1, 3]  # the two 0.3s, ascending class order
	cls, _ = BO.prune(lp, 3)[0]
	assert cls.tolist() == [1, 2, 3]
	cls, _ = BO.prune(lp, 4)[0]
	assert cls.tolist() == [0, 1, 2, 3]  # of the tied 0.1s the lower class id
	cls, _ = BO.prune(lp, 99)[0]
	assert cls.tolist() == [0, 1, 2, 3, 4]  # N = min(cutoff_top_n, C)


def test_prune_cutoff_prob_keeps_the_crossing_class():
	lp = np.log(np.array([[0.05, 0.5, 0.25, 0.15, 0.05]]))
	assert BO.prune(lp, 5, 0.5)[0][0].tolist() == [1]  # 0.5 reaches 0.5: stop there
	assert BO.prune(lp, 5, 0.6)[0][0].tolist() == [1, 2]  # 0.5 < 0.6, 0.75 crosses it and is kept
	assert BO.prune(lp, 5, 0.8)[0][0].tolist() == [1, 2, 3]
	assert BO.prune(lp, 2, 0.99)[0][0].tolist() == [1, 2]  # cutoff_top_n still caps it
	assert BO.prune(lp, 5, 1.0)[0][0].tolist() == [0, 1, 2, 3, 4]


def test_pruned_search_only_uses_kept_classes():
	lp = random_log_probs(2, 12, 30, 11, scale = 3.0)
	res = BO.ctc_prefix_beam_search(lp, beam_width = 8, cutoff_top_n = 3, cutoff_prob = 0.9)
	for b, beams in enumerate(res):
		allowed = [set(c.tolist()) for c, _ in BO.prune(lp[b].T, 3, 0.9)]
		for h, e, s in beams:
			assert all(tok in allowed[f] for tok, f in zip(h, e))
		scores = [s for _, _, s in beams]
		assert scores == sorted(scores, reverse = True) and len(beams) <= 8


def test_language_model_arguments_raise():
	from convasr_b200.decoders import BeamSearchDecoder
	labels = list('ab_')
	for kw in (dict(lm_path = 'lm.bin'), dict(beam_alpha = 0.5), dict(beam_beta = 1.0)):
		with pytest.raises(NotImplementedError, match = 'KenLM'):
			BeamSearchDecoder(labels, **kw)
	BeamSearchDecoder(labels, lm_path = None, beam_alpha = 0, beam_beta = 0)


@pytest.mark.parametrize('kw', [dict(beam_width = 0), dict(beam_width = 129), dict(topk = 0), dict(beam_width = 4, topk = 5), dict(cutoff_top_n = 0),
								dict(cutoff_prob = 0.0), dict(cutoff_prob = 1.5)])
def test_out_of_range_arguments_raise(kw):
	from convasr_b200.decoders import BeamSearchDecoder
	with pytest.raises(ValueError):
		BeamSearchDecoder(list('ab_'), **kw)


def test_workspace_query_refuses_bad_arguments_on_the_host():
	"""cab_ctc_beam_search_workspace: the same argument checks as the search, no device work"""
	from convasr_b200 import _lib
	lib = _lib.load()
	n = ctypes.c_int64()
	# B, T, C, N, W, K, blank, cutoff_prob
	assert lib.cab_ctc_beam_search_workspace(80, 751, 38, 38, 100, 1, 37, 1.0, ctypes.byref(n)) == 0
	assert n.value >= 80 * 751 * (2 * 38 * 4 + 4 + 100 * 8)
	bad = [(80, 751, 38, 38, 0, 1, 37, 1.0), (80, 751, 38, 38, 129, 1, 37, 1.0), (2, 9, 100, 65, 16, 1, 99, 1.0), (2, 9, 38, 0, 16, 1, 37, 1.0),
			(2, 9, 38, 38, 16, 1, 38, 1.0), (2, 9, 38, 38, 16, 1, -1, 1.0), (2, 9, 38, 38, 16, 17, 37, 1.0), (2, 9, 38, 38, 16, 0, 37, 1.0),
			(2, 9, 38, 38, 16, 1, 37, 0.0), (2, 9, 38, 38, 16, 1, 37, 1.5)]
	for args in bad:
		assert lib.cab_ctc_beam_search_workspace(*args, ctypes.byref(n)) != 0, args
		assert lib.cab_last_error()
	assert 'cab_ctc_beam_search_workspace' in _lib.HOST_ONLY and 'cab_ctc_beam_search_workspace' not in _lib.trace().names
	assert 'cab_ctc_beam_search' in _lib.trace().names


def test_dropin_decoders_expose_the_beam_search():
	root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
	dropin = os.path.join(root, 'convasr_b200', 'dropin')
	sys.path.insert(0, dropin)
	saved = sys.modules.pop('decoders', None)
	try:
		import decoders
		from convasr_b200 import decoders as impl
		assert decoders.BeamSearchDecoder is impl.BeamSearchDecoder and decoders.GreedyDecoder is impl.GreedyDecoder
		d = decoders.BeamSearchDecoder(list('ab_'), beam_width = 16, topk = 2)
		assert (d.beam_width, d.topk, d.cutoff_top_n, d.cutoff_prob, d.blank_id) == (16, 2, 40, 1.0, None)
	finally:
		sys.path.remove(dropin)
		sys.modules.pop('decoders', None)
		if saved is not None:
			sys.modules['decoders'] = saved
