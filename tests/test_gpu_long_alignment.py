"""ctc.alignment for long targets (beyond 2047 labels): the thread-block-cluster kernel
(ctc_align_cluster_kernel + ctc_align_backtrace_kernel, cab_ctc_alignment_long).

Host-only tests: the packed workspace query and the planted-path construction against the oracle.
GPU tests (marked gpu): the cluster path is bit-identical to the one-CTA kernel whatever the split,
exact against the oracle just past the old limit, exact on planted paths at hour scale, and runs
the transcribe-shaped flow through the drop-in modules.
"""
import ctypes
import os
import sys

import pytest
import torch

from oracle import oracle as O


def planted_path(L, C, blank, seed, T = None):
	"""log_probs [T, C] whose best path is a planted one: each label held for 1-3 frames, 0-2 blank frames before it (at least
	one between equal labels), trailing blanks up to T = 4L, lp = log_softmax(randn + 8 * one_hot(path)).
	Returns (log_probs, labels int64 [L], last frame of each label int64 [L])."""
	T = T or 4 * L
	g = torch.Generator().manual_seed(seed)
	y = torch.randint(0, C - 1, (L, ), generator = g)
	y = y + (y >= blank).long()  # any class but the blank
	runs = torch.randint(1, 4, (L, ), generator = g)
	gaps = torch.randint(0, 3, (L, ), generator = g)
	rep = torch.zeros(L, dtype = torch.bool)
	rep[1:] = y[1:] == y[:-1]
	gaps = torch.where(rep, gaps.clamp(min = 1), gaps)
	ends = torch.cumsum(gaps + runs, 0) - 1
	assert int(ends[-1]) < T
	starts = ends - runs + 1
	idx = torch.repeat_interleave(torch.arange(L), runs)
	pos = starts[idx] + torch.arange(int(runs.sum())) - (torch.cumsum(runs, 0) - runs)[idx]
	path = torch.full((T, ), blank, dtype = torch.int64)
	path[pos] = y[idx]
	lp = (torch.randn(T, C, generator = g) + 8.0 * torch.nn.functional.one_hot(path, C)).log_softmax(-1)
	return lp, y, ends


# ---------------------------------------------------------------- host only
def test_long_alignment_workspace_query_is_host_only():
	"""cab_ctc_alignment_long_workspace: the packed back-pointer table, B * T * ceil((2L+1)/4) bytes (4 two-bit codes a byte),
	decided in one place; an error naming the limit beyond L_max = 65535; no device needed"""
	from convasr_b200 import _lib
	lib = _lib.load()
	n = ctypes.c_int64()
	for B, T, L in ((80, 753, 169), (4, 30000, 8000), (1, 180000, 45000), (3, 7, 0), (2, 5, 1), (1, 1, 65535)):
		assert lib.cab_ctc_alignment_long_workspace(B, T, L, ctypes.byref(n)) == 0
		assert n.value == B * T * -(-(2 * L + 1) // 4)
	assert n.value == 32768  # S = 131071 -> 32768 bytes per frame
	assert lib.cab_ctc_alignment_long_workspace(1, 180000, 45000, ctypes.byref(n)) == 0 and n.value > 2**31  # 64-bit offsets
	assert lib.cab_ctc_alignment_long_workspace(1, 10, 65536, ctypes.byref(n)) != 0
	assert '65535' in lib.cab_last_error().decode()
	assert 'cab_ctc_alignment_long_workspace' in _lib.HOST_ONLY and 'cab_ctc_alignment_long_workspace' not in _lib.trace().names


@pytest.mark.parametrize('L,half', [(100, False), (1000, False), (100, True)])
def test_planted_path_is_the_oracle_alignment(L, half):
	"""the planted-path construction the hour-scale GPU test relies on (where the oracle is out of reach) is what the oracle
	returns at sizes it can run"""
	C, blank = 38, 37
	lp, y, ends = planted_path(L, C, blank, seed = L + int(half))
	T = lp.shape[0]
	lp = lp[:, None]
	if half:
		lp = lp.half()
	al = O.ctc_alignment(lp, y[None], torch.tensor([T]), torch.tensor([L]), blank)
	assert torch.equal(al[0], ends)


# ---------------------------------------------------------------- GPU
def _seeded_cases():
	"""the golden cases and the seeded cases of the one-CTA alignment tests: [B, C, T]-permuted views, input_lengths < T,
	tl = 0, repeated labels; fp32 and fp16"""
	root = os.path.dirname(os.path.abspath(__file__))
	cases = []
	for name in ('ctc', 'ctc_fp16'):
		for c in torch.load(os.path.join(root, 'golden', name + '.pt'), weights_only = False)['cases']:
			if c['alignment'] is not None:
				cases.append((c['log_probs'], c['targets'], c['input_lengths'], c['target_lengths'], c['blank']))
	g = torch.Generator().manual_seed(2)
	B, C, T, L = 6, 38, 300, 60
	lp = (torch.randn(B, C, T, generator = g) * 2).log_softmax(1)
	y = torch.randint(0, C - 1, (B, L), generator = g)
	y[:, 7] = y[:, 6]
	y[0, 20:24] = y[0, 19]
	ylen, olen = torch.tensor([60, 41, 17, 1, 0, 33]), torch.tensor([300, 250, 299, 120, 300, 70])
	cases.append((lp.permute(2, 0, 1), y, olen, ylen, C - 1))
	g = torch.Generator().manual_seed(4)
	B, C, T, L = 5, 38, 400, 80
	lp = (torch.randn(B, C, T, generator = g) * 3).log_softmax(1).half()
	y = torch.randint(0, C - 1, (B, L), generator = g)
	y[:, 3] = y[:, 2]
	ylen, olen = torch.tensor([80, 41, 17, 0, 33]), torch.tensor([400, 350, 399, 400, 170])
	cases.append((lp.permute(2, 0, 1), y, olen, ylen, C - 1))
	return cases


@pytest.mark.gpu
def test_cluster_alignment_is_split_invariant_and_equals_the_one_cta_kernel():
	from convasr_b200 import ctc, ops
	dev = torch.device('cuda:0')
	for lp, y, olen, ylen, blank in _seeded_cases():
		lp, y, olen, ylen = lp.to(dev), y.to(dev), olen.to(dev), ylen.to(dev)
		ref = ctc.alignment(lp, y, olen, ylen, blank = blank)
		for spc in (4, 64, 256, 0):
			got = ops.ctc_alignment(lp, y, olen, ylen, blank = blank, _states_per_cta = spc)
			assert got.dtype == torch.int64 and torch.equal(got, ref), (lp.dtype, tuple(lp.shape), spc, int((got != ref).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize('T,L,half', [(6000, 2100, False), (6000, 2100, True), (12000, 3000, False)])
def test_alignment_just_past_the_one_cta_limit_against_oracle(T, L, half):
	"""peaked posteriors (a model that has learnt something: no argmax within rounding of a tie), padded batch with
	input_lengths < T, one tl = 0 row, the [B, C, T] view"""
	from convasr_b200 import ctc
	dev = torch.device('cuda:0')
	g = torch.Generator().manual_seed(T + L)
	B, C = 3, 38
	y = torch.randint(0, C - 1, (B, L), generator = g)
	ylen = torch.tensor([L, L * 2 // 3, 0])
	olen = torch.tensor([T, T * 3 // 4, T * 5 // 6])
	path = torch.full((B, T), C - 1)
	for b in range(B):
		pos = torch.linspace(0, int(olen[b]) - 1, int(ylen[b])).long()
		path[b, pos] = y[b, :int(ylen[b])]
	lp = (torch.randn(B, C, T, generator = g) + 6.0 * torch.nn.functional.one_hot(path, C).permute(0, 2, 1)).log_softmax(1)
	if half:
		lp = lp.half()
	ref = O.ctc_alignment(lp.permute(2, 0, 1), y, olen, ylen, C - 1)
	got = ctc.alignment(lp.to(dev).permute(2, 0, 1), y.to(dev), olen.to(dev), ylen.to(dev), blank = C - 1)
	assert torch.equal(got.cpu(), ref), int((got.cpu() != ref).sum())
	assert int(got[2].abs().sum()) == 0


@pytest.mark.gpu
def test_hour_long_planted_alignment():
	"""T = 180 000 frames (one hour at 50 frames/s), L = 45 000 labels, C = 38: a 4 GB packed back-pointer table; then the
	same utterance batched with a short one whose tail CTAs hold no live state"""
	from convasr_b200 import ctc
	dev = torch.device('cuda:0')
	C, blank, L, T = 38, 37, 45000, 180000
	lp, y, ends = planted_path(L, C, blank, seed = 7, T = T)
	al = ctc.alignment(lp[:, None].to(dev), y[None].to(dev), torch.tensor([T], device = dev), torch.tensor([L], device = dev), blank = blank)
	assert torch.equal(al[0].cpu(), ends)
	del al
	torch.cuda.empty_cache()
	L2, T2 = 100, 400
	lp2, y2, ends2 = planted_path(L2, C, blank, seed = 8)
	pad = torch.full((T - T2, C), -20.0)
	pad[:, blank] = 0.0
	lpb = torch.stack([lp, torch.cat([lp2, pad])], 1)
	yb = torch.zeros(2, L, dtype = torch.int64)
	yb[0], yb[1, :L2] = y, y2
	al = ctc.alignment(lpb.to(dev), yb.to(dev), torch.tensor([T, T2], device = dev), torch.tensor([L, L2], device = dev), blank = blank)
	al = al.cpu()
	assert torch.equal(al[0], ends) and torch.equal(al[1, :L2], ends2) and int(al[1, L2:].abs().sum()) == 0


@pytest.mark.gpu
def test_dropin_transcribe_flow_aligns_three_minutes():
	"""`PYTHONPATH=convasr_b200/dropin`: 3 minutes of 8 kHz int16 PCM -> Wav2Letter (bf16 tier, eval) -> log_probs ->
	ctc.alignment with more than 2047 labels, as transcribe.py --align calls it (transcribe.py:176-183)"""
	import importlib
	root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
	dropin = os.path.join(root, 'convasr_b200', 'dropin')
	dev = torch.device('cuda:0')
	saved = {n: sys.modules.pop(n, None) for n in ('models', 'ctc')}
	sys.path.insert(0, dropin)
	try:
		models, ctc = [importlib.import_module(n) for n in ('models', 'ctc')]
		from convasr_b200 import ops
		c = torch.load(os.path.join(root, 'tests', 'golden', 'models.pt'), weights_only = False)['cases'][0]
		frontend = models.LogFilterBankFrontend(out_channels = 64, sample_rate = 8000, window_size = .02, window_stride = .01, window = 'hann_window', dither = 0.0, dither0 = 0.0, stft_mode = None)
		model = models.Wav2Letter(num_input_features = 64, num_classes = [38], frontend = frontend, check_time_dim_padded = False,
									dict = lambda logits, log_probs, olen, **kwargs: (log_probs[0], logits[0], olen[0]), **c['kwargs'])
		model.load_state_dict(O.synth_state_dict(c['shapes'], seed = c['seed']), strict = False)
		model = model.to(dev).eval().set_precision('bf16')
		g = torch.Generator().manual_seed(11)
		x = (torch.randn(2, 1440000, generator = g) * 3000).round().clamp(-32767, 32767).to(torch.int16)
		xlen = torch.tensor([1.0, 0.8])
		with torch.no_grad():
			log_probs, logits, olen = model(x.to(dev), xlen.to(dev))
		L = 2100
		y = torch.randint(0, 37, (2, L), generator = g).to(dev)
		ylen = torch.tensor([L, 1700], device = dev)
		al = ctc.alignment(log_probs.permute(2, 0, 1), y, olen, ylen, blank = 37, pack_backpointers = False)
		assert torch.equal(ctc.alignment(log_probs.permute(2, 0, 1), y, olen, ylen, blank = 37, pack_backpointers = True), al)
		assert torch.equal(ops.ctc_alignment(log_probs.permute(2, 0, 1), y, olen, ylen, blank = 37, _states_per_cta = 128), al)
		assert al.dtype == torch.int64 and al.shape == (2, L)
		for b in range(2):
			a = al[b].cpu()
			n = int(ylen[b])
			assert int(a[n:].abs().sum()) == 0
			assert bool((a[1:n] >= a[:n - 1]).all()) and int(a[:n].max()) < int(olen[b])
	finally:
		sys.path.remove(dropin)
		for n, mod in saved.items():
			sys.modules.pop(n, None)
			if mod is not None:
				sys.modules[n] = mod


@pytest.mark.gpu
def test_alignment_beyond_the_cluster_limit_is_refused_before_any_launch():
	from convasr_b200 import _lib, ctc
	dev = torch.device('cuda:0')
	lp = torch.zeros(8, 1, 5, device = dev).log_softmax(-1)
	y = torch.ones(1, 65536, dtype = torch.int64, device = dev)
	n0 = _lib.launch_count()
	with pytest.raises(RuntimeError, match = '65535'):
		ctc.alignment(lp, y, torch.tensor([8], device = dev), torch.tensor([65536], device = dev), blank = 0)
	assert _lib.launch_count() == n0
