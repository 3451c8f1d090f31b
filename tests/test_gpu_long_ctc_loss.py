"""CTC loss and gradient for long targets (beyond 1345 labels): the thread-block-cluster kernel
(ctc_loss_cluster_kernel, cab_ctc_loss_long_fwd / cab_ctc_loss_long_bwd).

Host-only tests: the workspace and routing queries, and the float64 restatement used at hour scale against the oracle and
F.ctc_loss.  GPU tests (marked gpu): the cluster path gives the one-CTA kernel's nll bit for bit whatever the split, its
gradient up to the order of atomic additions; it matches float64 F.ctc_loss just past the old limit and the float64
restatement at 10 minutes and one hour; it is refused past 65535 labels; and it serves the model's loss in eval, in
native training and inside a CUDA-graph training step.
"""
import ctypes
import functools
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import oracle as O


def rel(a, b):
	a, b = a.detach().double().cpu(), b.detach().double().cpu()
	return float((a - b).norm() / (b.norm() + 1e-30))


def ctc_f64(lp, y, blank, want_grad = False):
	"""Textbook CTC in float64, vectorised over the extended states, one frame per step, on lp's device: lp [T, C] holds the
	utterance's frames only, y [L] its labels.  Returns nll (float) and, with want_grad, exp(lp) - occupancy [T, C]
	(F.ctc_loss's gradient for grad_out = 1).  Stores the float64 alpha table only when the gradient is wanted."""
	lp = lp.double()
	T, C = lp.shape
	dev = lp.device
	S = 2 * y.numel() + 1
	ninf = -math.inf

	def problem(ext):
		skip = torch.zeros(S, dtype = torch.bool, device = dev)
		skip[2:] = ext[2:] != ext[:-2]
		return ext, ~skip

	def step(a, e, noskip):
		a2 = F.pad(a, (1, 0), value = ninf)[:S]
		a3 = F.pad(a, (2, 0), value = ninf)[:S].masked_fill(noskip, ninf)
		return torch.logsumexp(torch.stack([a, a2, a3]), 0) + e

	def start(e):
		a = torch.full((S, ), ninf, dtype = torch.float64, device = dev)
		a[:2] = e[:2]
		return a

	ext = torch.full((S, ), blank, dtype = torch.int64, device = dev)
	ext[1::2] = y.to(dev)
	ext, noskip = problem(ext)
	alpha = torch.empty(T, S, dtype = torch.float64, device = dev) if want_grad else None
	a = start(lp[0, ext])
	for t in range(T):
		if t > 0:
			a = step(a, lp[t, ext], noskip)
		if want_grad:
			alpha[t] = a
	ll = float(torch.logsumexp(a[-2:], 0)) if S > 1 else float(a[0])
	if not want_grad:
		return -ll, None
	# beta: alpha of the time- and state-reversed problem
	ext_r, noskip_r = problem(ext.flip(0))
	grad = lp.exp()
	for t in range(T - 1, -1, -1):
		b = start(lp[t, ext_r]) if t == T - 1 else step(b, lp[t, ext_r], noskip_r)
		occ = (alpha[t] + b.flip(0) - ll - lp[t, ext]).exp()
		grad[t].index_add_(0, ext, -occ)
	return -ll, grad


def peaked(B, C, T, y, ylen, olen, blank, g, scale = 6.0):
	"""[B, C, T] log-probs of a model that has learnt something: each utterance's labels planted at evenly spread frames"""
	path = torch.full((B, T), blank)
	for b in range(B):
		pos = torch.linspace(0, int(olen[b]) - 1, int(ylen[b])).long()
		path[b, pos] = y[b, :int(ylen[b])]
	return (torch.randn(B, C, T, generator = g) + scale * F.one_hot(path, C).permute(0, 2, 1)).log_softmax(1)


# ---------------------------------------------------------------- host only
def test_long_ctc_loss_workspace_query_is_host_only():
	"""cab_ctc_loss_long_workspace: one fp32 [B, T, 2L+1] alpha table, 64-bit, refused past 65535 labels; no device needed"""
	from convasr_b200 import _lib
	lib = _lib.load()
	n = ctypes.c_int64()
	for B, T, L in ((80, 753, 169), (2, 30000, 8000), (1, 180000, 45000), (3, 7, 0), (1, 1, 65535)):
		assert lib.cab_ctc_loss_long_workspace(B, T, L, ctypes.byref(n)) == 0
		assert n.value == 4 * B * T * (2 * L + 1)
	assert lib.cab_ctc_loss_long_workspace(1, 180000, 45000, ctypes.byref(n)) == 0 and n.value > 2**31
	assert lib.cab_ctc_loss_long_workspace(1, 10, 65536, ctypes.byref(n)) != 0
	assert '65535' in lib.cab_last_error().decode()
	for name in ('cab_ctc_loss_long_workspace', 'cab_ctc_loss_one_cta_covers'):
		assert name in _lib.HOST_ONLY and name not in _lib.trace().names


def test_one_cta_routing_boundary():
	"""the one-CTA recursion takes every L_max whose 8 staged frames fit its shared memory: up to 1345 labels"""
	from convasr_b200 import _lib
	lib = _lib.load()
	for L in (0, 1, 169, 225, 1000, 1344, 1345):
		assert lib.cab_ctc_loss_one_cta_covers(L) == 1, L
	for L in (1346, 1347, 2047, 2048, 8000, 45000, 65535, 65536):
		assert lib.cab_ctc_loss_one_cta_covers(L) == 0, L


def test_float64_restatement_equals_oracle_and_f_ctc_loss():
	"""the vectorised restatement the long GPU tests compare against: repeats, an empty target, an infeasible target"""
	g = torch.Generator().manual_seed(0)
	T, C, blank = 30, 6, 5
	cases = [
		(torch.tensor([1, 2, 2, 3, 1]), 30),
		(torch.tensor([4, 4, 4]), 20),
		(torch.tensor([], dtype = torch.int64), 12),
		(torch.tensor([0, 0, 0, 0]), 6),  # needs 7 frames: infeasible
		(torch.tensor([2]), 1),
	]
	for y, il in cases:
		lp = torch.randn(T, C, generator = g, dtype = torch.float64).log_softmax(-1)
		nll, grad = ctc_f64(lp[:il], y, blank, want_grad = True)
		ref_nll, ref_grad = O.ctc_loss_np(lp[:, None].numpy(), y[None].numpy(), np.array([il]), np.array([y.numel()]), blank)
		torch_nll = F.ctc_loss(lp[:, None], y[None], torch.tensor([il]), torch.tensor([y.numel()]), blank = blank, reduction = 'none')
		if math.isinf(ref_nll[0]):
			assert math.isinf(nll) and math.isinf(float(torch_nll[0]))
			continue
		assert abs(nll - ref_nll[0]) < 1e-9 * max(1.0, abs(nll)) and abs(nll - float(torch_nll[0])) < 1e-9 * max(1.0, abs(nll))
		assert torch.allclose(grad, torch.from_numpy(ref_grad[:il, 0]), atol = 1e-10)


# ---------------------------------------------------------------- GPU
def _identity_cases():
	"""the golden cases ([T, B, C]) and the C2-shape cases of the bench-shape parity test (peaked and random, through the
	[B, C, T]-permuted view): (leaf log-probs, view into [T, B, C], targets, input_lengths, target_lengths, blank)"""
	root = os.path.dirname(os.path.abspath(__file__))
	ident = lambda x: x
	cases = []
	for c in torch.load(os.path.join(root, 'golden', 'ctc.pt'), weights_only = False)['cases']:
		cases.append((c['log_probs'], ident, c['targets'], c['input_lengths'], c['target_lengths'], c['blank']))
	g = torch.Generator().manual_seed(1)
	B, C, T, L = 3, 38, 753, 225
	lp_bct = torch.randn(B, C, T, generator = g).log_softmax(1)
	y = torch.randint(0, C - 1, (B, L), generator = g)
	ylen, olen = torch.tensor([225, 150, 3]), torch.tensor([753, 600, 410])
	bct = lambda x: x.permute(2, 0, 1)
	cases.append((peaked(B, C, T, y, ylen, olen, C - 1, g), bct, y, olen, ylen, C - 1))
	cases.append((lp_bct, bct, y, olen, ylen, C - 1))
	return cases


def _loss_and_grad(leaf, view, y, il, tl, blank, spc):
	x = leaf.detach().clone().requires_grad_(True)
	from convasr_b200 import ops
	nll = ops.ctc_loss(view(x), y, il, tl, blank = blank, _states_per_cta = spc)
	nll.sum().backward()
	return nll.detach(), view(x.grad)


def _check_grad(got, ref, il, tol):
	assert torch.equal(got.isnan(), ref.isnan())
	assert rel(got.nan_to_num(0.0), ref.nan_to_num(0.0)) < tol
	for b in range(got.shape[1]):  # exactly zero past the input length
		assert float(got[int(il[b]):, b].abs().max() if int(il[b]) < got.shape[0] else 0.0) == 0.0


@pytest.mark.gpu
def test_cluster_loss_is_split_invariant_and_equals_the_one_cta_kernel():
	from convasr_b200 import ops
	dev = torch.device('cuda:0')
	for leaf, view, y, il, tl, blank in _identity_cases():
		leaf, y, il, tl = leaf.to(dev), y.to(dev), il.to(dev), tl.to(dev)
		ref_nll, ref_grad = _loss_and_grad(leaf, view, y, il, tl, blank, None)
		for spc in (4, 64, 256, 0):
			nll, grad = _loss_and_grad(leaf, view, y, il, tl, blank, spc)
			assert torch.equal(nll, ref_nll), (tuple(leaf.shape), spc, (nll - ref_nll).abs().max())
			_check_grad(grad, ref_grad, il.cpu(), 1e-6)
			with torch.no_grad():
				assert torch.equal(ops.ctc_loss(view(leaf), y, il, tl, blank = blank, _states_per_cta = spc), ref_nll)


@pytest.mark.gpu
@pytest.mark.parametrize('L,C,layout,kind', [(1346, 38, 'bct', 'peaked'), (1346, 38, 'bct', 'random'), (2000, 38, 'bct', 'peaked'),
												(3000, 38, 'bct', 'peaked'), (3000, 38, 'bct', 'random'), (1346, 5000, 'btc', 'peaked')])
def test_loss_just_past_the_one_cta_limit_against_float64_f_ctc_loss(L, C, layout, kind):
	"""B = 2 with a short second utterance, T = 3.5 L; the model's [B, C, T] view or the class-contiguous [B, T, C] layout of
	the large-vocabulary head.  Bars of the existing CTC tests: nll 1e-4; gradient 1e-4 (peaked), 1e-3 (random).  On random
	log-probs the fp32 rounding of the recursion's fast exp / log (the one-CTA kernel's arithmetic, kept for a bit-identical
	nll) accumulates over the frames: 2.4e-3 measured at T = 10 500 (L = 3 000), hence 5e-3 there"""
	from convasr_b200 import ctc
	dev = torch.device('cuda:0')
	g = torch.Generator().manual_seed(L + C)
	B, T, blank = 2, L * 7 // 2, C - 1
	y = torch.randint(0, C - 1, (B, L), generator = g)
	ylen, olen = torch.tensor([L, 40]), torch.tensor([T, 300])
	lp = peaked(B, C, T, y, ylen, olen, blank, g) if kind == 'peaked' else torch.randn(B, C, T, generator = g).log_softmax(1)
	if layout == 'btc':
		lp = lp.permute(0, 2, 1).contiguous()
		view = lambda x: x.permute(1, 0, 2)
	else:
		view = lambda x: x.permute(2, 0, 1)
	ref_lp = view(lp).double().requires_grad_(True)
	ref = F.ctc_loss(ref_lp, y, olen, ylen, blank = blank, reduction = 'none')
	ref.sum().backward()
	x = lp.to(dev).requires_grad_(True)
	nll = ctc.ctc_loss(view(x), y.to(dev), olen.to(dev), ylen.to(dev), blank = blank)
	assert torch.allclose(nll.double().cpu(), ref.detach(), rtol = 1e-4)
	nll.sum().backward()
	_check_grad(view(x.grad).cpu(), ref_lp.grad, olen, 1e-4 if kind == 'peaked' else 1e-3 if T < 8000 else 5e-3)


@pytest.mark.gpu
def test_ten_minutes_loss_and_gradient_against_float64_restatement():
	"""T = 30 000 frames (10 minutes at 50 frames/s), L = 8 000 labels, batched with a short utterance"""
	from convasr_b200 import ops
	dev = torch.device('cuda:0')
	g = torch.Generator().manual_seed(10)
	B, C, T, L, blank = 2, 38, 30000, 8000, 37
	y = torch.randint(0, C - 1, (B, L), generator = g)
	ylen, olen = torch.tensor([L, 100]), torch.tensor([T, 500])
	lp = peaked(B, C, T, y, ylen, olen, blank, g).to(dev).requires_grad_(True)
	nll = ops.ctc_loss(lp.permute(2, 0, 1), y.to(dev), olen.to(dev), ylen.to(dev), blank = blank)
	nll.sum().backward()
	grad = lp.grad.permute(2, 0, 1)
	ref_grad = torch.zeros_like(grad, dtype = torch.float64)
	for b in range(B):
		il, tl = int(olen[b]), int(ylen[b])
		ref_nll, ref_grad[:il, b] = ctc_f64(lp.detach()[b, :, :il].T, y[b, :tl], blank, want_grad = True)
		assert abs(float(nll[b]) - ref_nll) <= 1e-4 * abs(ref_nll), (b, float(nll[b]), ref_nll)
	assert rel(grad, ref_grad) < 1e-4
	assert float(grad[int(olen[1]):, 1].abs().max()) == 0.0


@pytest.mark.gpu
def test_hour_long_loss_only_needs_no_workspace():
	"""T = 180 000 frames, L = 45 000 labels: a loss-only call allocates no [T, 2L+1] table (65 GB in fp32)"""
	from convasr_b200 import ops
	dev = torch.device('cuda:0')
	g = torch.Generator().manual_seed(60)
	C, T, L, blank = 38, 180000, 45000, 37
	y = torch.randint(0, C - 1, (1, L), generator = g)
	lp = peaked(1, C, T, y, torch.tensor([L]), torch.tensor([T]), blank, g).to(dev)
	yd, il, tl = y.to(dev), torch.tensor([T], device = dev), torch.tensor([L], device = dev)
	torch.cuda.synchronize()
	base = torch.cuda.memory_allocated()
	torch.cuda.reset_peak_memory_stats()
	with torch.no_grad():
		nll = ops.ctc_loss(lp.permute(2, 0, 1), yd, il, tl, blank = blank)
	torch.cuda.synchronize()
	assert torch.cuda.max_memory_allocated() - base < 64 * 2**20  # offsets and nll only; the table would be 65 GB
	ref_nll, _ = ctc_f64(lp[0].T, y[0], blank)
	assert abs(float(nll[0]) - ref_nll) <= 1e-4 * abs(ref_nll), (float(nll[0]), ref_nll)


@pytest.mark.gpu
def test_loss_beyond_the_cluster_limit_is_refused_before_any_launch():
	from convasr_b200 import _lib, ctc
	dev = torch.device('cuda:0')
	y = torch.ones(1, 65536, dtype = torch.int64, device = dev)
	for requires_grad in (False, True):
		lp = torch.zeros(8, 1, 5, device = dev).log_softmax(-1).requires_grad_(requires_grad)
		n0 = _lib.launch_count()
		with pytest.raises(RuntimeError, match = '65535'):
			ctc.ctc_loss(lp, y, torch.tensor([8], device = dev), torch.tensor([65536], device = dev), blank = 0)
		assert _lib.launch_count() == n0


def _model(dev, precision, train, seed = 7):
	from convasr_b200 import models
	m = models.Wav2Letter(64, [38], frontend = models.LogFilterBankFrontend(64, 8000, .02, .01, 'hann_window'), dropout = 0., check_time_dim_padded = False,
							base_width = 32, num_blocks = 1)
	shapes = {k: tuple(v.shape) for k, v in m.state_dict().items() if not k.startswith('frontend.')}
	sd = O.synth_state_dict(shapes, seed = seed)
	m.load_state_dict(sd, strict = False)
	m = m.to(dev).set_precision(precision)
	return (m.train() if train else m.eval()), sd


def _long_batch(seconds, L, seed):
	g = torch.Generator().manual_seed(seed)
	sig = (torch.randn(2, 8000 * seconds, generator = g) * 3000).round().clamp(-32767, 32767).to(torch.int16)
	xlen = torch.tensor([1.0, 0.8])
	y = torch.randint(0, 37, (2, 1, L), generator = g)
	ylen = torch.tensor([[L], [L * 3 // 4]])
	return sig, xlen, y, ylen


@pytest.mark.gpu
def test_model_eval_loss_of_three_minutes():
	"""Wav2Letter in eval on 3 minutes of 8 kHz audio with a 2 000-label target: out['loss'] is the float64 loss of
	out['log_probs'], each over its utterance's target length (models.py:323)"""
	dev = torch.device('cuda:0')
	m, _ = _model(dev, 'fp32', train = False)
	sig, xlen, y, ylen = _long_batch(180, 2000, seed = 11)
	with torch.no_grad():
		out = m(sig.to(dev), xlen.to(dev), y = y.to(dev), ylen = ylen.to(dev))
	loss, lp, olen = out['loss'].cpu(), out['log_probs'][0], out['olen'][0]
	assert bool(torch.isfinite(loss).all())
	for b in range(2):
		ref, _ = ctc_f64(lp[b, :, :int(olen[b])].T, y[b, 0, :int(ylen[b, 0])], 37)
		ref = ref / float(ylen[b, 0])
		assert abs(float(loss[b]) - ref) <= 1e-4 * abs(ref), (b, float(loss[b]), ref)


@pytest.mark.gpu
def test_native_training_step_cluster_path_equals_one_cta_path(monkeypatch):
	"""fp32 tier, a 1 000-label target (both kernels take it): every parameter gradient of the step within 1e-5"""
	from convasr_b200 import ops
	dev = torch.device('cuda:0')
	sig, xlen, y, ylen = [t.to(dev) for t in _long_batch(40, 1000, seed = 12)]
	grads, losses = [], []
	for forced in (False, True):
		if forced:
			monkeypatch.setattr(ops, 'ctc_loss', functools.partial(ops.ctc_loss, _states_per_cta = 0))
		m, _ = _model(dev, 'fp32', train = True)
		out = m(sig, xlen, y = y, ylen = ylen)
		(out['loss'] * ylen[:, 0]).mean().backward()
		losses.append(out['loss'].detach().cpu())
		grads.append({k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None})
	assert bool(torch.isfinite(losses[0]).all()) and torch.allclose(losses[0], losses[1], rtol = 1e-6)
	assert grads[0].keys() == grads[1].keys() and len(grads[0]) > 0
	for k in grads[0]:
		assert rel(grads[1][k], grads[0][k]) < 1e-5, k


@pytest.mark.gpu
def test_graphed_train_step_with_long_target_equals_eager_step():
	"""a 1 400-label target (the cluster path) inside training.GraphedTrainStep, against the eager step"""
	from convasr_b200 import training
	dev = torch.device('cuda:0')
	sig, xlen, y, ylen = [t.to(dev) for t in _long_batch(60, 1400, seed = 13)]
	losses = []
	for graphed in (False, True):
		m, sd = _model(dev, 'bf16', train = True)
		opt = torch.optim.SGD(m.parameters(), lr = 1e-3, momentum = 0.9)
		if graphed:
			step = training.GraphedTrainStep(m, opt, sig, xlen, y, ylen, warmup = 2)
			m.load_state_dict(sd, strict = False)
			for st in opt.state.values():
				st['momentum_buffer'].zero_()
			out = [step(sig, xlen, y, ylen) for _ in range(3)]
		else:
			out = []
			for _ in range(3):
				opt.zero_grad(set_to_none = True)
				o = m(sig, xlen, y = y, ylen = ylen)
				(o['loss'] * ylen[:, 0]).mean().backward()
				opt.step()
				out.append(o['loss'].detach().clone())
		losses.append(torch.stack(out).cpu())
	assert bool(torch.isfinite(losses[1]).all())
	assert torch.allclose(losses[0][0], losses[1][0], rtol = 1e-4, atol = 1e-4)
	assert torch.allclose(losses[0], losses[1], rtol = 2e-2, atol = 2e-2)
