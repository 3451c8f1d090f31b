"""Streaming acoustic model (convasr_b200.streaming) on the host: the planner's frame schedule, left context, right reach
and lookahead against a brute-force walk of the module tree, the frontend's final frames against a restatement from
the window geometry, and the refusals that need no device."""
import random

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from convasr_b200 import models, streaming

HOP = 80


def _frontend(nfft_window = .02):
	return models.LogFilterBankFrontend(64, 8000, nfft_window, .01, 'hann_window')


def _model(name, **kw):
	num_classes = kw.pop('num_classes', [38])
	args = dict(frontend = _frontend(), dropout = 0., check_time_dim_padded = False, base_width = 8)
	if name == 'JasperNetSeparable':
		args['groups'] = 8
	args.update(kw)
	return getattr(models, name)(64, num_classes, **args).eval()


ZOO = [
	'Wav2Letter', 'Wav2LetterResidual', 'Wav2LetterResidualNoDilation', 'Wav2LetterResidualBig', 'Wav2LetterDense', 'Wav2LetterDenseNoDilation',
	'Wav2LetterDenseNoDilationInplace', 'Wav2LetterDenseLargeKernels', 'Wav2LetterDenseNoDilationLargeKernels', 'Wav2LetterDenseBig',
	'Wav2LetterDenseBigLargeKernelsNoDropoutReLu', 'Wav2LetterDenseBigLargeKernelsNoDilationNoDropoutReLu',
	'Wav2LetterDenseBigLargeKernelsNoDilationNoTemporalMaskNoDropoutReLu', 'Wav2LetterFlat', 'JasperNetSeparable', 'JasperNetSmall',
	'JasperNetSmallInstanceNorm', 'JasperNetLarge', 'JasperNetBig', 'JasperNetBigNoStride', 'JasperNetBigBpeOnly', 'JasperNetResidualBig',
	'JasperNetBigInplace'
]


# ---------------------------------------------------------------- brute force over the module tree
def _dep(x, conv):
	"""which outputs of `conv` read a flagged input (x: float64 [1, 1, T] 0/1); a stride-2 conv reads whole frame pairs"""
	k, s, p, d = conv.kernel_size[0], conv.stride[0], conv.padding[0], conv.dilation[0]
	if s == 2:
		first, last = 2 * ((0 - p) // 2), 2 * ((k - 1 - p) // 2) + 1  # frames of the pairs that output 0 reads, relative to 2j
		x = F.pad(x, (-first, last))
		return (F.conv1d(x, torch.ones(1, 1, last - first + 1, dtype = x.dtype), stride = 2) > 0).double()[..., :(x.shape[-1] + first - last + 2 * p - (k - 1) - 1) // 2 + 1]
	return (F.conv1d(x, torch.ones(1, 1, k, dtype = x.dtype), padding = p, dilation = d) > 0).double()


def _convbn(block, x, residuals):
	for j in range(len(block.conv)):
		for m in block.conv[j]:
			if isinstance(m, nn.Conv1d):
				x = _dep(x, m)
	for r, rc in enumerate(block.conv_residual):
		x = torch.maximum(x, _dep(residuals[r], rc) if isinstance(rc, nn.Conv1d) else residuals[r])
	return x


def _walk(model, x):
	"""the flags of every decoder head's outputs, following JasperNet.forward (models.py:286-316)"""
	residuals = []
	n = len(model.backbone)
	for i, block in enumerate(model.backbone):
		x = _convbn(block, x, residuals)
		if i < n - model.num_epilogue_modules - 1:
			residuals = residuals + [x] if model.residual == 'dense' else [x] if model.residual else []
		else:
			residuals = []
	heads = [_dep(x, model.decoder[0])]
	if model.decoder.type == 'bpe':
		h = x
		for cb in model.decoder[1]:
			h = _convbn(cb, h, [])
		heads.append(h)
	return heads


def _brute_final(model, m, total):
	"""output frames final when the first m of `total` feature frames are (all heads final up to the least), and the
	one-shot output length"""
	x = torch.zeros(1, 1, total, dtype = torch.float64)
	x[..., m:] = 1
	heads = _walk(model, x)
	finals = [int(h[0, 0].nonzero()[0]) if h.any() else h.shape[-1] for h in heads]
	return min(finals), heads[0].shape[-1]


@pytest.mark.parametrize('name', ZOO + ['bpe'])
def test_planner_reach_matches_brute_force(name):
	model = _model('Wav2Letter', decoder_type = 'bpe', num_classes = [38, 300]) if name == 'bpe' else _model(name)
	sm = streaming.StreamingModel(model)
	out = sm.heads[0].node
	total = 1200
	for m in [1, 2, 3, 7, 40, 41, 200, 201, 333]:
		n = (m - 1) * HOP + 129
		assert streaming.frontend_frames_final(n, False, HOP) == m & ~1
		want, _ = _brute_final(model, m & ~1, total)
		assert sm.schedule(n, False)[out] == want, (name, m)
	# at the end of the stream every activation has its one-shot length
	for n in [1, 128, 129, 16000, 16001 + 79]:
		_, length = _brute_final(model, 0, n // HOP + 1)
		fin = sm.schedule(n, True)
		assert all(fin[h.node] == length for h in sm.heads)
	# left context and right reach of every stride-1 launch: the conv padding and d(k-1) - padding of the module
	convs = [c for blk in model.backbone for rep in blk.conv for c in rep if isinstance(c, nn.Conv1d) and c.groups == 1 and c.stride[0] == 1 and c.kernel_size[0] > 1]
	steps = [s for s in sm.steps if s.grouped is None and s.launch is not None and s.launch.stride2 is None and s.head is None and s.srcs[0].taps > 1]
	steps = [s for s in steps if s.node[0] == 'block']
	assert len(steps) == len(convs)
	for s, c in zip(steps, convs):
		assert s.srcs[0].pad == c.padding[0] and s.left_context == c.padding[0]
		assert s.right_reach == c.dilation[0] * (c.kernel_size[0] - 1) - c.padding[0]


def test_lookahead_matches_brute_force():
	for name in ['Wav2Letter', 'Wav2LetterDense', 'bpe']:
		model = _model('Wav2Letter', decoder_type = 'bpe', num_classes = [38, 300]) if name == 'bpe' else _model(name)
		sm = streaming.StreamingModel(model)
		lag = 0
		for phase in range(2 * HOP):
			n = 600 * HOP + phase
			fin, length = _brute_final(model, streaming.frontend_frames_final(n, False, HOP), n // HOP + 1)
			lag = max(lag, length - fin)
		assert sm.lookahead_frames == lag, (name, sm.lookahead_frames, lag)
		if name == 'Wav2Letter':
			# 15 convs of k = 11 (5 frames each), the k = 29 d = 2 epilogue (27), prologue + frontend: about 105 frames of 20 ms
			assert 100 <= lag <= 110, lag


def _frontend_final_restated(n, eos):
	"""frame f is final when every sample of its window [80 f - 128, 80 f + 128) and of its FFT partner's inside the
	stream has arrived and the left pad is decided (a reflection needs more than 128 samples), or at eos"""
	total = n // HOP + 1
	if eos:
		return total
	return sum(1 for f in range(total) if n > 128 and 80 * (f | 1) + 128 <= n)


def test_frame_schedule_on_random_chunkings():
	rng = random.Random(5)
	model = _model('Wav2LetterResidual')
	sm = streaming.StreamingModel(model)
	out = sm.heads[0].node
	for trial in range(60):
		total = rng.choice([0, 1, 60, 128, 129, 200, 1000, 5000, 12345])
		cuts = sorted(rng.randint(0, total) for _ in range(rng.randint(0, 12)))
		sizes = [b - a for a, b in zip([0] + cuts, cuts + [total])]
		sizes += [0] * rng.randint(0, 2)
		n, prev = 0, None
		for i, c in enumerate(sizes):
			n += c
			eos = i == len(sizes) - 1
			assert streaming.frontend_frames_final(n, eos, HOP) == _frontend_final_restated(n, eos)
			fin = sm.schedule(n, eos, prev)
			if not eos:
				want, _ = _brute_final(model, fin['feat'], n // HOP + 1 + 400)
				assert fin[out] == want
			if prev is not None:
				assert all(fin[k] >= prev[k] for k in prev)
			prev = fin
		_, length = _brute_final(model, 0, total // HOP + 1)
		assert prev[out] == length
		if total <= 128:
			assert all(sm.schedule(m, False)['feat'] == 0 for m in range(total + 1))


def test_refusals_without_a_device():
	m = _model('Wav2Letter')
	m.train()
	with pytest.raises(RuntimeError, match = 'eval-mode'):
		streaming.StreamingModel(m)
	m.eval()
	m.set_precision('fp8')
	with pytest.raises(NotImplementedError, match = 'fp8'):
		streaming.StreamingModel(m)
	m.set_precision(None)
	m512 = models.Wav2Letter(64, [38], frontend = _frontend(.04), dropout = 0., check_time_dim_padded = False, base_width = 8).eval()
	assert m512.frontend.nfft == 512
	with pytest.raises(NotImplementedError, match = 'nfft = 256'):
		streaming.StreamingModel(m512)
	nofe = models.Wav2Letter(64, [38], dropout = 0., check_time_dim_padded = False, base_width = 8).eval()
	with pytest.raises(NotImplementedError, match = 'LogFilterBankFrontend'):
		streaming.StreamingModel(nofe)
	sm = streaming.StreamingModel(_model('Wav2Letter'))
	with pytest.raises(ValueError, match = 'one row'):
		sm.new_state(None)
	with pytest.raises(TypeError, match = 'CUDA'):
		models.FixedNormalisation(torch.ones(1), torch.zeros(1, 64), torch.ones(1, 64))


def test_new_prototypes_match_the_ctypes_table():
	"""the streaming entry points are additions: their parameter counts match the ctypes table, the ABI version stays 3,
	and bad arguments are refused before anything is launched"""
	import ctypes
	import os
	import re
	from convasr_b200 import _lib
	root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
	src = re.sub(r'/\*.*?\*/', '', open(os.path.join(root, 'include', 'convasr_b200.h')).read(), flags = re.S)
	protos = dict(re.findall(r'\bint\s+(cab_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;', src, flags = re.S))
	for name in ('cab_frontend_features_fixed', 'cab_frontend_stream', 'cab_stream_copy'):
		assert len([p for p in protos[name].split(',') if p.strip()]) == len(_lib.SIGNATURES[name]), name
	lib = _lib.load()
	assert lib.cab_abi_version() == 3 == _lib.ABI_VERSION
	before = _lib.launch_count()
	fake = ctypes.c_void_p(1 << 20)
	assert lib.cab_stream_copy(fake, 65536, 16, None) != 0
	assert lib.cab_stream_copy(fake, 1, 15, None) != 0
	assert lib.cab_stream_copy(None, 0, 0, None) == 0
	assert lib.cab_frontend_stream(fake, 256, fake, 1, 1, 160, 80, 512, 64, fake, fake, fake, fake, 0.97, 1e-5, fake, fake, fake, 64, fake, None, None) != 0
	assert b'nfft = 256' in lib.cab_last_error()
	assert lib.cab_frontend_stream(fake, 250, fake, 1, 1, 160, 80, 256, 64, fake, fake, fake, fake, 0.97, 1e-5, fake, fake, fake, 64, fake, None, None) != 0
	assert _lib.launch_count() == before
