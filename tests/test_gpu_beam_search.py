"""CTC prefix beam search on the GPU (csrc/beam.cu, ops.ctc_beam_search, decoders.BeamSearchDecoder) against the float64
restatement in tests/beam_oracle.py and exhaustive enumeration of CTC probabilities.

The kernels work in fp32 and the restatement in float64, so two candidates whose scores differ by less than the fp32
rounding accumulated over the frames may be ranked the other way round; n-best lists are compared rank by rank where
the reference scores are apart, and scores to 1e-5 relative."""
import math
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import beam_oracle as BO  # noqa: E402
from oracle import oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope = 'module')
def dev():
	return torch.device('cuda')


def peaked(B, C, T, y, ylen, olen, blank, g, scale = 6.0):
	"""[B, C, T] log-probs of a model that has learnt something: each utterance's labels planted at evenly spread frames
	(the construction of test_gpu_long_ctc_loss.py)"""
	path = torch.full((B, T), blank)
	for b in range(B):
		pos = torch.linspace(0, int(olen[b]) - 1, int(ylen[b])).long()
		path[b, pos] = y[b, :int(ylen[b])]
	return (torch.randn(B, C, T, generator = g) + scale * F.one_hot(path, C).permute(0, 2, 1)).log_softmax(1)


def nbest(out, b):
	"""(tokens, score) of utterance b's hypotheses, best first, from decode_nbest's tensors"""
	toks, lens, scores = out['tokens'][b].cpu(), out['lengths'][b].cpu().tolist(), out['scores'][b].cpu().tolist()
	return [(tuple(toks[k, :lens[k]].tolist()), scores[k]) for k in range(len(scores)) if scores[k] > -math.inf]


def decoder(**kw):
	from convasr_b200.decoders import BeamSearchDecoder
	return BeamSearchDecoder(labels = None, **kw)


@pytest.mark.parametrize('C,T,blank,W', [(3, 6, 2, 128), (3, 6, 0, 128), (4, 4, 3, 128), (4, 4, 0, 128), (2, 7, 1, 8)])
def test_exhaustive_tiny_cases(dev, C, T, blank, W):
	"""beam wider than the number of prefixes, no pruning: every labeling of nonzero probability, ranked by its exact CTC
	probability"""
	g = torch.Generator().manual_seed(100 * C + T + blank)
	lp = (1.5 * torch.randn(3, C, T, generator = g)).log_softmax(1)
	out = decoder(beam_width = W, topk = W, cutoff_top_n = C, blank_id = blank).decode_nbest(lp.to(dev))
	for b in range(3):
		ref = BO.labelings_by_probability(lp[b].double().numpy(), blank, O.ctc_loss_np)
		assert len(ref) <= W
		BO.assert_nbest_equal(nbest(out, b), ref, 1e-5)
		orc = BO.ctc_prefix_beam_search(lp[b:b + 1].numpy(), beam_width = W, cutoff_top_n = C, blank = blank)[0]
		lens = out['lengths'][b].cpu()
		for k, (h, e, _) in enumerate(orc):
			if tuple(out['tokens'][b, k, :lens[k]].tolist()) == h:  # same rank: same emission frames
				assert tuple(out['frames'][b, k, :lens[k]].tolist()) == e


def _against_oracle(lp_dev, lp_ref, olen, W, N, cutoff_prob, k_cmp, dev):
	out = decoder(beam_width = W, topk = W, cutoff_top_n = N, cutoff_prob = cutoff_prob).decode_nbest(lp_dev, olen.to(dev))
	ref = BO.ctc_prefix_beam_search(lp_ref, olen, beam_width = W, cutoff_top_n = N, cutoff_prob = cutoff_prob)
	same = 0
	for b in range(len(ref)):
		got = nbest(out, b)
		BO.assert_nbest_equal(got, [(h, s) for h, _, s in ref[b]], 1e-5, k = k_cmp)
		same += sum(g[0] == r[0] for g, r in zip(got, ref[b]))
		h, e, _ = ref[b][0]
		if got[0][0] == h:
			assert out['frames'][b, 0, :len(h)].cpu().tolist() == list(e)
	return same, sum(len(r) for r in ref)


@pytest.mark.parametrize('C,W,scale,layout', [(38, 100, 6.0, 'bct'), (5000, 16, 10.0, 'btc')])
def test_peaked_posteriors_against_oracle(dev, C, W, scale, layout, capsys):
	"""T = 751 (15 s), ragged lengths.  C = 5000 reads the class-contiguous [B, C, T] view of the large-vocabulary head
	without a copy; there the planted class needs scale 10 to carry most of the mass (scale 6 leaves it ~5 %)."""
	B, T, L = 3, 751, 120
	g = torch.Generator().manual_seed(C)
	olen = torch.tensor([T, 700, 523])
	ylen = torch.tensor([L, 100, 77])
	y = torch.randint(0, C - 1, (B, L), generator = g)
	lp = peaked(B, C, T, y, ylen, olen, C - 1, g, scale = scale)
	lp_dev = lp.to(dev) if layout == 'bct' else lp.permute(0, 2, 1).contiguous().to(dev).permute(0, 2, 1)
	same, total = _against_oracle(lp_dev, lp.numpy(), olen, W, 40, 1.0, 10, dev)
	with capsys.disabled():
		print(f'\nC={C} W={W}: {same}/{total} ranks hold the oracle\'s hypothesis')


def test_cutoff_prob_against_oracle(dev):
	B, C, T, L = 2, 38, 400, 60
	g = torch.Generator().manual_seed(5)
	olen, ylen = torch.tensor([T, 350]), torch.tensor([L, 50])
	lp = peaked(B, C, T, torch.randint(0, C - 1, (B, L), generator = g), ylen, olen, C - 1, g, scale = 4.0)
	_against_oracle(lp.to(dev), lp.numpy(), olen, 32, 8, 0.95, 10, dev)


def test_diffuse_posteriors_top1(dev):
	"""untrained-model-like posteriors: the best score to 1e-4 relative, the same best sequence wherever the oracle's
	top-2 margin exceeds 1e-3"""
	B, C, T, W = 4, 38, 300, 100
	g = torch.Generator().manual_seed(9)
	lp = torch.randn(B, C, T, generator = g).log_softmax(1)
	olen = torch.tensor([T, 280, 250, 137])
	out = decoder(beam_width = W, topk = 2, cutoff_top_n = 40).decode_nbest(lp.to(dev), olen.to(dev))
	ref = BO.ctc_prefix_beam_search(lp.numpy(), olen, beam_width = W, cutoff_top_n = 40)
	checked = 0
	for b in range(B):
		got = nbest(out, b)
		assert abs(got[0][1] - ref[b][0][2]) <= 1e-4 * abs(ref[b][0][2])
		if ref[b][0][2] - ref[b][1][2] > 1e-3:
			assert got[0][0] == ref[b][0][0]
			checked += 1
	assert checked >= 1


def test_result_does_not_depend_on_the_batch(dev):
	B, C, T = 6, 38, 300
	g = torch.Generator().manual_seed(3)
	lp = torch.randn(B, C, T, generator = g).log_softmax(1).to(dev)
	olen = torch.tensor([300, 17, 299, 0, 150, 1], device = dev)
	dec = decoder(beam_width = 64, topk = 8)
	full = dec.decode_nbest(lp, olen)
	for b in range(B):
		one = dec.decode_nbest(lp[b:b + 1].clone(), olen[b:b + 1])
		for key in ('tokens', 'frames', 'lengths', 'scores'):
			assert torch.equal(full[key][b:b + 1], one[key]), (b, key)
	# no frames: the empty hypothesis with probability one
	assert full['lengths'][3, 0] == 0 and full['scores'][3, 0] == 0 and full['scores'][3, 1] == -math.inf


def test_bad_arguments_are_refused_before_any_launch(dev):
	from convasr_b200 import _lib, ops
	lp = torch.randn(2, 100, 20, device = dev).log_softmax(1)
	before = _lib.launch_count()
	for kw in (dict(beam_width = 0), dict(beam_width = 129), dict(cutoff_top_n = 65), dict(cutoff_top_n = 0), dict(blank = 100), dict(blank = -1),
				dict(beam_width = 16, topk = 17), dict(topk = 0), dict(cutoff_prob = 0.0)):
		with pytest.raises(RuntimeError, match = 'cab_ctc_beam_search'):
			ops.ctc_beam_search(lp, **kw)
	torch.cuda.synchronize()
	assert _lib.launch_count() == before
	ops.ctc_beam_search(lp, beam_width = 128, cutoff_top_n = 64, topk = 128)  # the limits themselves run
	assert _lib.launch_count() == before + 3
	with pytest.raises(RuntimeError, match = 'no CPU fallback'):
		ops.ctc_beam_search(lp.cpu())


def test_topk_decode_lists(dev):
	g = torch.Generator().manual_seed(1)
	lp = torch.randn(3, 6, 12, generator = g).log_softmax(1)
	olen = torch.tensor([12, 7, 3])
	ref = BO.ctc_prefix_beam_search(lp.numpy(), olen, beam_width = 8, cutoff_top_n = 6)
	one = decoder(beam_width = 8).decode(lp.to(dev), olen)
	many = decoder(beam_width = 8, topk = 3).decode(lp.to(dev), olen)
	assert one == [list(r[0][0]) for r in ref]
	assert many == [[list(h) for h, _, _ in r[:3]] for r in ref]


def test_dropin_transcribe_flow_matches_greedy_text_on_confident_posteriors(golden, dev):
	"""model -> BeamSearchDecoder -> text through the drop-in modules.  The posteriors are the model's argmax path made
	confident (p > 0.99 in every frame); there the beam's best hypothesis spells the GreedyCTCGenerator text.  The
	generator's rule that turns a run of blanks into a space is switched off (blank_amount_to_space > T): it formats
	the transcript and is not part of decoding."""
	import importlib
	root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
	dropin = os.path.join(root, 'convasr_b200', 'dropin')
	saved = {n: sys.modules.pop(n, None) for n in ('models', 'decoders', 'transcript_generators')}
	sys.path.insert(0, dropin)
	try:
		models, decoders, transcript_generators = [importlib.import_module(n) for n in ('models', 'decoders', 'transcript_generators')]
		c = golden('models')['cases'][0]
		frontend = models.LogFilterBankFrontend(out_channels = 64, sample_rate = 8000, window_size = .02, window_stride = .01, window = 'hann_window', dither = 0.0, dither0 = 0.0, stft_mode = None)
		model = models.Wav2Letter(num_input_features = 64, num_classes = [38], frontend = frontend, check_time_dim_padded = False,
									dict = lambda logits, log_probs, olen, **kwargs: (log_probs[0], logits[0], olen[0]), **c['kwargs'])
		model.load_state_dict(O.synth_state_dict(c['shapes'], seed = c['seed']), strict = False)
		model.to(dev).eval()
		x, xlen = c['signal'], c['xlen']
		with torch.no_grad():
			log_probs, _, olen = model(x.to(dev), xlen.to(dev))
		tok = O.CharTokenizer('абвгдеёжзийклмнопрстуфхцчшщъыьэюя')
		B, C, T = log_probs.shape
		path = log_probs.argmax(1).cpu()
		path[path == tok.space_id] = tok.eps_id  # keep spaces out: the generator treats them as silence
		g = torch.Generator().manual_seed(0)
		confident = (torch.randn(B, C, T, generator = g) + 14.0 * F.one_hot(path, C).permute(0, 2, 1)).log_softmax(1).to(dev)
		assert bool((confident.max(1).values.exp() > 0.99).all())
		labels = tok.idx2char
		hyp = decoders.BeamSearchDecoder(labels, beam_width = 32, cutoff_top_n = 40).decode(confident, olen)
		beam_text = tok.decode(hyp)
		gen = transcript_generators.GreedyCTCGenerator(blank_amount_to_space = T + 1)
		tr = gen.generate(tokenizer = tok, log_probs = confident, begin = torch.zeros(B, device = dev), end = torch.ones(B, device = dev),
							output_lengths = olen, time_stamps = None, segment_text_key = 'hyp')
		greedy_text = [''.join(s['hyp'] for s in t[0]) for t in tr]
		assert beam_text == greedy_text
		assert any(len(t) > 0 for t in beam_text)
	finally:
		sys.path.remove(dropin)
		for n, mod in saved.items():
			sys.modules.pop(n, None)
			if mod is not None:
				sys.modules[n] = mod
