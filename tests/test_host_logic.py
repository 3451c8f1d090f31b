"""Host-side logic of the drop-in modules (no GPU): module tree / state_dict contract, BN
folding, weight re-packing for the strided prologue, mel basis, precision selection."""
import pytest
import torch
import torch.nn.functional as F

from convasr_b200 import engine, models
from oracle import oracle as O

ALL_MODELS = [
	'Wav2Letter', 'Wav2LetterResidual', 'Wav2LetterResidualNoDilation', 'Wav2LetterResidualBig', 'Wav2LetterDense', 'Wav2LetterDenseNoDilation',
	'Wav2LetterDenseNoDilationInplace', 'Wav2LetterDenseLargeKernels', 'Wav2LetterDenseNoDilationLargeKernels', 'Wav2LetterDenseBig',
	'Wav2LetterDenseBigLargeKernelsNoDropoutReLu', 'Wav2LetterDenseBigLargeKernelsNoDilationNoDropoutReLu',
	'Wav2LetterDenseBigLargeKernelsNoDilationNoTemporalMaskNoDropoutReLu', 'Wav2LetterFlat', 'JasperNetSeparable', 'JasperNetSmall',
	'JasperNetSmallInstanceNorm', 'JasperNetSmallTrainableInstanceNorm', 'JasperNetLarge', 'JasperNetBig', 'JasperNetBigNoStride',
	'JasperNetBigBpeOnly', 'JasperNetResidualBig', 'JasperNetBigInplace'
]


def test_all_24_configurations_resolve():
	for name in ALL_MODELS:
		assert issubclass(getattr(models, name), models.JasperNet)


def test_state_dict_keys_and_shapes_match_the_reference(golden):
	"""Keys/shapes recorded from the real reference in tests/golden/models.pt."""
	for c in golden('models')['cases']:
		if c['fused']:
			continue
		m = getattr(models, c['model'])(64, [c['num_classes']], frontend = models.LogFilterBankFrontend(64, 8000, .02, .01, 'hann_window'), dropout = 0., **c['kwargs'])
		mine = {k: tuple(v.shape) for k, v in m.state_dict().items() if not k.startswith('frontend.')}
		assert mine == c['shapes'], c['model']
		fe_keys = sorted(k for k in m.state_dict() if k.startswith('frontend.'))
		assert fe_keys == ['frontend.mel.bias', 'frontend.mel.weight', 'frontend.window']


def test_state_dict_keys_match_live_reference_for_every_class(golden):
	"""state_dict keys / shapes and backbone length of every class against the original: live where its tree is present,
	else as recorded in tests/golden/surface.pt (oracle/make_golden.py: golden_surface)"""
	from oracle import make_golden, reference_shim
	recorded = golden('surface')['state_dicts']
	ref = reference_shim.load() if reference_shim.available() else None
	assert set(ALL_MODELS) <= set(recorded)
	for name in ALL_MODELS:
		kw = make_golden.surface_kwargs(name)
		ours = getattr(models, name)(64, [38], **kw)
		b = dict(shapes = {k: tuple(v.shape) for k, v in ours.state_dict().items()}, backbone = len(ours.backbone))
		assert b == recorded[name], name
		if ref is not None:
			theirs = getattr(ref.models, name)(64, [38], **kw)
			assert dict(shapes = {k: tuple(v.shape) for k, v in theirs.state_dict().items()}, backbone = len(theirs.backbone)) == b, name


def test_wav2letter_accepts_the_callers_extra_kwargs():
	# transcribe.py:44-52 / benchmark.py:97-104 pass dict= and check_time_dim_padded= (SURVEY.md 8b)
	m = models.Wav2Letter(64, [38], base_width = 8, dict = lambda logits, log_probs, olen, **kw: logits[0], check_time_dim_padded = False)
	assert m.check_time_dim_padded is False and callable(m.dict)
	assert len(m.backbone) == 8 and [len(b.conv) for b in m.backbone] == [1, 3, 3, 3, 3, 3, 1, 1]
	assert m.backbone[6].conv[0][0].padding[0] == 29 and m.backbone[6].conv[0][0].dilation[0] == 2  # +2 frames quirk
	assert m.backbone[1].activation.nonlinearity == ('hardtanh', 0, 20)


def test_mel_basis_matches_reference(golden):
	g = golden('frontend')
	assert float((models.slaney_mel_basis(8000, 256, 64, 0.0, 4000) - g['mel']).abs().max()) < 2e-7
	fe = models.LogFilterBankFrontend(64, 8000, .02, .01, 'hann_window')
	assert (fe.win_length, fe.hop_length, fe.nfft, fe.freq_cutoff) == (160, 80, 256, 129)
	assert float(fe.mel.bias[0]) == 2.0**-14


def test_fold_bn_equals_conv_then_bn():
	torch.manual_seed(0)
	conv = torch.nn.Conv1d(6, 10, 5, padding = 2, bias = False)
	bn = torch.nn.BatchNorm1d(10).eval()
	bn.running_mean.normal_(); bn.running_var.uniform_(0.5, 1.5); bn.weight.data.uniform_(0.5, 1.5); bn.bias.data.normal_()
	x = torch.randn(2, 6, 30)
	w, b = engine.fold_bn(conv.weight, conv.bias, bn)
	assert torch.allclose(F.conv1d(x, w, b, padding = 2), bn(conv(x)), atol = 1e-5)
	w2, b2 = engine.fold_bn(conv.weight, None, torch.nn.Identity())
	assert torch.equal(w2, conv.weight) and float(b2.abs().max()) == 0


def test_fuse_conv_bn_eval_changes_keys_like_the_reference(golden):
	c = [c for c in golden('models')['cases'] if c['fused']][0]
	m = models.Wav2Letter(64, [38], **c['kwargs']).eval()
	m.load_state_dict(O.synth_state_dict(c['shapes'], seed = c['seed']), strict = False)
	n_before = len(m.state_dict())
	m.fuse_conv_bn_eval()
	keys = set(m.state_dict())
	assert not any('.bn.' in k for k in keys)
	assert 'backbone.0.conv.0.0.bias' in keys and len(keys) < n_before


@pytest.mark.parametrize('k,pad,F_', [(11, 5, 51), (11, 5, 50), (13, 6, 31), (3, 1, 9)])
def test_stride2_pair_view_repacking(k, pad, F_):
	"""The frame-pair trick: stride-2 conv == stride-1 conv over [F/2, 2C] with re-packed taps."""
	torch.manual_seed(k)
	C, Co, CA = 5, 7, 8
	w = torch.randn(Co, C, k)
	x = torch.randn(2, C, F_)
	ref = F.conv1d(x, w, stride = 2, padding = pad)
	wp, taps, pad_left = engine.pack_taps_stride2(w, pad, CA)
	F_pad = F_ + F_ % 2
	xa = torch.zeros(2, F_pad, CA)
	xa[:, :F_, :C] = x.permute(0, 2, 1)
	pairs = xa.view(2, F_pad // 2, 2 * CA)  # [B, P, 2CA]
	T_out = ref.shape[-1]
	out = torch.zeros(2, Co, T_out)
	for t in range(T_out):
		for j in range(taps):
			p = t + j - pad_left
			if 0 <= p < pairs.shape[1]:
				out[:, :, t] += pairs[:, p] @ wp[j].T
	assert torch.allclose(out, ref, atol = 1e-4)


def test_precision_selection():
	m = models.Wav2Letter(64, [38], base_width = 8)
	assert m._active_precision() == 'fp32'
	assert m.to(torch.bfloat16)._active_precision() == 'bf16'
	m2, _ = models.data_parallel_and_autocast(models.Wav2Letter(64, [38], base_width = 8), opt_level = 'O2')
	assert m2._active_precision() == 'bf16'


def test_training_graph_wiring_follows_the_reference_forward():
	"""training._graph: activation ids and residual sources per repeat follow JasperNet.forward (models.py:303-313):
	residual branches join on the LAST repeat of a block only, 'dense' accumulates every earlier block output, plain
	residual keeps the previous one, the two epilogue modules (and the block before them feeding forward) get none."""
	from convasr_b200 import training
	for name, mode in (('Wav2Letter', False), ('Wav2LetterResidual', True), ('Wav2LetterDense', 'dense'), ('Wav2LetterFlat', 'flat'), ('JasperNetSeparable', 'dense')):
		kw = dict(base_width = 128, groups = 128) if 'Separable' in name else dict(base_width = 16)
		m = getattr(models, name)(64, [38], dropout = 0., **kw)
		reps = training._graph(m)
		assert [r.in_id for r in reps] == list(range(len(reps))) and [r.out_id for r in reps] == list(range(1, len(reps) + 1))
		block_out, k = [], 0
		for i, block in enumerate(m.backbone):
			n = len(block.conv)
			for j in range(n):
				rep = reps[k + j]
				srcs = [s for s, _, _ in rep.res]
				if j < n - 1 or not mode or i == 0 or i >= len(m.backbone) - 2:
					assert srcs == [], (name, i, j)
				elif mode == 'dense':
					assert srcs == block_out[:i], (name, i, j, srcs)
				else:
					assert srcs == block_out[i - 1:i], (name, i, j, srcs)
				assert all((c is None) == (mode == 'flat') for _, c, _ in rep.res)
				assert (rep.grouped is not None) == ('Separable' in name and 0 < i < len(m.backbone) - 2)
			k += n
			block_out.append(reps[k - 1].out_id)


# ------------------------------------------------------------------------------------------ batch feed
def test_collate_matches_reference_collate_fn(golden):
	"""feed.collate == AudioTextDataset.collate_fn (datasets.py:305-332) on the items oracle/make_golden.py fed the
	reference: same shapes, dtypes (int16 PCM stays int16), zero padding to the time multiple, fp32 length fractions,
	speaker padding; also through the recycling pool (buffers come back dirty and must be re-initialised)."""
	from convasr_b200 import feed
	from oracle import make_golden
	pool = feed.PinnedPool(pin = False)
	for rep in range(2):
		for (name, items, multiple), c in zip(make_golden.feed_batches(), golden('feed')['cases']):
			assert name == c['name']
			meta, s, x, xlen, y, ylen = feed.collate(items, time_padding_multiple = multiple, pool = pool)
			assert [m['example_id'] for m in meta] == [m['example_id'] for m in c['meta']]
			for got, want in ((s, c['s']), (x, c['x']), (xlen, c['xlen']), (y, c['y']), (ylen, c['ylen'])):
				assert got.dtype == want.dtype and got.shape == want.shape and torch.equal(got, want), name
			pool.give(s, x, xlen, y, ylen)
			for t in (s, x, xlen, y, ylen):
				t.fill_(7)  # poison what went back to the pool
	# batch mode: fields arrive as lists and are zipped first (datasets.py:307-308)
	name, items, multiple = make_golden.feed_batches()[0]
	a = feed.collate(items, multiple)
	b = feed.collate(list(map(list, zip(*items))), multiple, batch_mode = True)
	assert all(torch.equal(u, v) for u, v in zip(a[1:], b[1:]))


def test_collate_matches_live_reference(golden):
	"""feed.collate against the original's collate_fn: live where its tree (with an importable datasets module) is present,
	else against its outputs recorded in tests/golden/feed.pt"""
	import types
	from convasr_b200 import feed
	from oracle import make_golden, reference_shim
	ref = reference_shim.load() if reference_shim.available() else None
	live = ref is not None and ref.datasets is not None
	for (name, items, multiple), c in zip(make_golden.feed_batches(), golden('feed')['cases']):
		if live:
			fake_self = types.SimpleNamespace(mode = ref.datasets.AudioTextDataset.DEFAULT_MODE, time_padding_multiple = multiple)
			theirs = ref.datasets.AudioTextDataset.collate_fn(fake_self, items)[1:]
		else:
			theirs = (c['s'], c['x'], c['xlen'], c['y'], c['ylen'])
		ours = feed.collate(items, multiple)
		assert all(torch.equal(a, b) and a.dtype == b.dtype for a, b in zip(ours[1:], theirs)), name


# ------------------------------------------------------------------------------------------ bench contract
def test_bench_reference_arm_prints_the_contract_line():
	"""`bench.py --impl reference` (the CPU oracle port timed on the host cores) prints ONE JSON line with the
	keys the driver reads; runs without a GPU."""
	import json
	import os
	import subprocess
	import sys
	ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
	out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--cpu-sample-batch', '2', '--workload', 'wav2letter_char_fwd_ctc_B8x10s_fp32'], capture_output = True, text = True, timeout = 600, env = dict(os.environ, CUDA_VISIBLE_DEVICES = ''))
	assert out.returncode == 0, out.stderr[-2000:]
	lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
	assert len(lines) == 1
	d = json.loads(lines[0])
	assert d['impl'] == 'reference' and d['metric'] == 'audio_seconds_per_second' and d['unit'] == 'audio-s/s'
	assert d['higher_is_better'] is True and d['value'] > 0 and d['gpu_launches'] == 0
	from oracle import reference_shim
	assert d['cpu_baseline']['kind'] == ('reference' if reference_shim.available() else 'port') and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
	assert d['config']['batch_per_gpu'] == 2  # the label says what actually ran
	assert d['e2e'] == dict(value = d['value'], unit = 'audio-s/s', h2d_bytes_per_step = 0, d2h_bytes_per_step = 0)
	assert d['config']['workload'] == 'wav2letter_char_fwd_ctc_B8x10s_fp32'


def test_native_training_coverage_by_model_class():
	"""training.unsupported_reason(): every family of the model zoo trains on the native kernels, the *Inplace ones included
	(section 8f rank 4: InplaceBatchNorm1d / the invertible leaky_relu compute BatchNorm1d / leaky_relu; only an invertible
	activation other than leaky_relu, which the reference asserts against, is refused); there is no ATen path to fall back
	to -- a module tree that is not covered raises instead."""
	from convasr_b200 import models, training
	reasons = {name: training.unsupported_reason(getattr(models, name)(64, [38], **(dict(base_width = 128) if 'Separable' in name else dict(base_width = 16)))) for name in ALL_MODELS}
	refused = {n for n, r in reasons.items() if r is not None}
	assert refused == set(), reasons
	m = models.Wav2LetterDenseNoDilationInplace(64, [38], base_width = 16)
	assert all(b.activation.invertible for b in m.backbone)
	m.backbone[1].activation.nonlinearity = ('relu', )
	assert 'invertible' in training.unsupported_reason(m)
	assert training.unsupported_reason(models.Wav2Letter(64, [38, 120], base_width = 16, decoder_type = 'bpe')) is not None
	assert not hasattr(models.JasperNet, '_forward_training')


def test_small_host_helpers_match_the_live_reference(golden):
	"""silence_space_mask / sparse_topk / sparse_topk_todense (models.py:768-810): host-side helpers of the module surface,
	against the original live where its tree is present, else as recorded in tests/golden/surface.pt"""
	import torch
	from convasr_b200 import models
	from oracle import make_golden, reference_shim
	inp = make_golden.surface_inputs()
	lp, speech = inp['lp'], inp['speech']
	mask = models.silence_space_mask(lp, speech, blank_idx = 6, space_idx = 5)
	assert mask.shape == (2, 7, 40) and not bool(mask[:, 5].any())
	quiet = (~speech) & (lp.argmax(1) == 6)
	assert torch.equal(mask[:, 0].bool(), quiet)
	x = inp['x']
	saved = models.sparse_topk(x, 2, dim = 1, indices_dtype = torch.int16, values_dtype = torch.float16, fill_value = -1.0)
	dense = models.sparse_topk_todense(saved)
	assert dense.shape == x.shape and int((dense != -1.0).sum()) == 3 * 2 * 11
	assert torch.allclose(dense.max(1).values, x.max(1).values, atol = 2e-3)
	assert issubclass(models.InplaceBatchNorm1d, torch.nn.BatchNorm1d) and models.apply_dither(x, 0.0) is x
	rec = golden('surface')
	h = rec['helpers']
	assert torch.equal(mask.bool(), h['mask'])
	assert torch.equal(saved['indices'], h['indices']) and torch.equal(saved['values'], h['values']) and torch.equal(dense, h['dense'])
	missing = set(rec['names']) - set(dir(models))
	assert missing <= {'OnnxWrapper', 'Wav2VecFrontend'}, missing  # ONNX runtime / fairseq backends: out of scope (SURVEY 2.1)
	if not reference_shim.available():
		return
	ref = reference_shim.load().models
	assert torch.equal(mask.bool(), ref.silence_space_mask(lp, speech, 6, 5).bool())
	r_saved = ref.sparse_topk(x, 2, dim = 1, indices_dtype = torch.int16, values_dtype = torch.float16, fill_value = -1.0)
	assert torch.equal(saved['indices'], r_saved['indices']) and torch.equal(saved['values'], r_saved['values'])
	assert torch.equal(dense, ref.sparse_topk_todense(r_saved))
	missing = {n for n in dir(ref) if not n.startswith('_') and callable(getattr(ref, n)) and getattr(getattr(ref, n), '__module__', None) == ref.__name__ and not hasattr(models, n)}
	assert missing <= {'OnnxWrapper', 'Wav2VecFrontend'}, missing  # ONNX runtime / fairseq backends: out of scope (SURVEY 2.1)


def test_larc_matches_the_live_reference(golden):
	"""larc_ in 'clip' and 'scale' mode against the original: live where its tree is present, else as recorded in
	tests/golden/surface.pt"""
	import torch
	from convasr_b200 import optimizers
	from oracle import make_golden, reference_shim
	ref_larc = reference_shim.load().optimizers.larc_ if reference_shim.available() else None
	for case, recorded in zip(make_golden.surface_inputs()['larc'], golden('surface')['larc']):
		ours = make_golden.larc_grads(optimizers.larc_, case)
		for theirs in [recorded] + ([make_golden.larc_grads(ref_larc, case)] if ref_larc is not None else []):
			for a, b in zip(ours, theirs):
				assert (a is None and b is None) or torch.allclose(a, b, rtol = 1e-6, atol = 0), case['mode']
