"""The oracle (oracle/oracle.py) against the golden vectors minted from the real reference
(tests/golden/, generator oracle/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from oracle import oracle as O


def rel(a, b):
	return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))


def test_mel_filterbank_matches_reference(golden):
	g = golden('frontend')
	mel = O.slaney_mel_filterbank(8000, 256, 64, 0.0, 4000)
	assert mel.shape == g['mel'].shape
	assert float((mel - g['mel']).abs().max()) < 2e-7  # SURVEY.md 8c: 6.5e-8 between librosa restatements
	assert torch.equal(torch.hann_window(160, periodic = True), g['window'])


def test_frontend_and_instance_norm(golden):
	g = golden('frontend')
	for c in g['cases']:
		logmel = O.frontend_logmel(c['signal'], c['xlen'], mel = g['mel'])
		assert logmel.shape == c['logmel'].shape, c['name']
		assert float((logmel - c['logmel']).abs().max()) < 5e-5, c['name']  # fp32 log-mel, SURVEY appendix C: 7.6e-6
		feats = O.masked_instance_norm(c['logmel'], c['xlen'])
		assert float((feats - c['feats']).abs().max()) < 1e-5, c['name']
		if c['xlen'] is not None:  # padded frames are exactly zero
			F = feats.shape[-1]
			for b, n in enumerate(O.output_lengths(F, c['xlen']).tolist()):
				assert float(feats[b, :, n:].abs().max() if n < F else 0.0) == 0.0


def test_models_forward_and_loss(golden):
	g = golden('models')
	for c in g['cases']:
		sd = O.synth_state_dict(c['shapes'], seed = c['seed'])
		assert abs(sum(float(v.double().abs().sum()) for v in sd.values() if v.is_floating_point()) - c['checksum']) < 1e-6 * c['checksum']
		over = {k: v for k, v in c['kwargs'].items() if k in ('groups', )}
		logits, log_probs, olen = O.model_forward(sd, c['signal'], c['xlen'], model = c['model'], **over)
		assert torch.equal(olen[0], c['olen']), c['model']
		# fused reference (case 1) == unfused oracle up to BN folding rounding (BASELINE.md: 3.8e-7 rel)
		assert rel(logits[0], c['logits']) < 1e-4, (c['model'], rel(logits[0], c['logits']))
		assert rel(log_probs[0], c['log_probs']) < 1e-4
		C = c['num_classes']
		loss = O.ctc_loss_torch(log_probs[0].permute(2, 0, 1), c['y'][:, 0], olen[0], c['ylen'][:, 0], C - 1) / c['ylen'][:, 0]
		assert torch.allclose(loss, c['loss'], rtol = 1e-3, atol = 1e-3), c['model']


def test_ctc_loss_restatement_matches_torch(golden):
	g = golden('ctc')
	for c in g['cases']:
		nll, grad = O.ctc_loss_np(c['log_probs'].numpy(), c['targets'].numpy(), c['input_lengths'].numpy(), c['target_lengths'].numpy(), c['blank'])
		ref = c['loss'].double().numpy()
		finite = np.isfinite(ref)
		assert np.array_equal(np.isinf(nll), ~finite)
		assert np.allclose(nll[finite], ref[finite], rtol = 1e-5)
		if c['grad'] is not None:
			assert np.allclose(grad, c['grad'].double().numpy(), atol = 1e-4)  # torch computes in fp32; nll ~ 1e2 => ~1e-5 abs noise


def test_alignment_matches_reference(golden):
	g = golden('ctc')
	for c in g['cases']:
		if c['alignment'] is None:
			continue
		al = O.ctc_alignment(c['log_probs'], c['targets'], c['input_lengths'], c['target_lengths'], c['blank'])
		assert torch.equal(al, c['alignment'])


def test_fp16_alignment_matches_reference(golden):
	"""ctc.alignment on fp16 log_probs (ctc.py:29): the reference's recursion runs in fp16; the restatement rounds after every
	operation and must hit the same frames -- which differ from the fp32 answer on these inputs"""
	differing = 0
	for c in golden('ctc_fp16')['cases']:
		assert c['log_probs'].dtype == torch.float16
		al = O.ctc_alignment(c['log_probs'], c['targets'], c['input_lengths'], c['target_lengths'], c['blank'])
		assert torch.equal(al, c['alignment'])
		differing += int((O.ctc_alignment(c['log_probs'].float(), c['targets'], c['input_lengths'], c['target_lengths'], c['blank']) != c['alignment']).sum())
	assert differing > 0


def test_greedy_decode_and_generate(golden):
	g = golden('decode')
	tok = O.CharTokenizer(g['alphabet'])
	assert (tok.eps_id, tok.space_id, len(tok.idx2char)) == (37, 36, 38)
	for c in g['generate']:
		B, T = len(c['ids']), len(c['ids'][0])
		ts = [[t * 0.02 for t in range(T)]] * B if c['with_ts'] else None
		# timestamps are float32 in the reference (torch tensor .tolist())
		if ts is not None:
			ts = (torch.arange(T)[None].float() * 0.02).expand(B, -1).tolist()
		segs = O.greedy_generate(tok, c['ids'], c['olens'], ts, begin = [0.0] * B, end = [float(torch.tensor(T * 0.02))] * B)
		assert segs == c['segments']
	d = g['decode']
	assert O.greedy_decode(d['lp1'], [4]) == d['d1'] == [[0, 0, 3, 1]]
	assert O.greedy_decode(d['lp2'], K = 2) == d['d2'] == [[[0, 1], [1, 2]]]
	assert O.greedy_decode(d['lp3'], [33, 20, 1, 7]) == d['d3']
	assert O.greedy_decode(d['lp3'], [33, 20, 1, 7], K = 3) == d['d4']


def test_oracle_against_live_reference(golden):
	"""A seeded Wav2Letter (base_width 16, xlen 0.77 / 1.0) forward + ctc.alignment of the original vs the oracle: live where its
	tree is present, else against its outputs as recorded in tests/golden/surface.pt"""
	from oracle import make_golden, reference_shim
	inp = make_golden.surface_inputs()
	sig, xlen, y, ylen = inp['signal'], inp['xlen'], inp['y'], inp['ylen']
	rec = golden('surface')['forward']
	logits, log_probs, olen = O.model_forward(O.synth_state_dict(rec['shapes'], seed = 5), sig, xlen, model = 'Wav2Letter')
	assert torch.equal(olen[0], rec['olen'])
	assert rel(logits[0], rec['logits']) < 1e-4
	assert torch.equal(O.ctc_alignment(rec['log_probs'].permute(2, 0, 1), y, rec['olen'], ylen, 37), rec['alignment'])
	if not reference_shim.available():
		return
	ref = reference_shim.load()
	model = reference_shim.make_model('Wav2Letter', (38, ), base_width = 16)
	shapes = {k: tuple(v.shape) for k, v in model.state_dict().items() if not k.startswith('frontend.')}
	sd = O.synth_state_dict(shapes, seed = 5)
	model.load_state_dict(sd, strict = False)
	with torch.no_grad():
		out = model(sig, xlen)
	assert torch.equal(olen[0], out['olen'][0])
	assert rel(logits[0], out['logits'][0]) < 1e-4
	lp = out['log_probs'][0]
	al_ref = ref.ctc.alignment(lp.permute(2, 0, 1), y, olen[0], ylen, blank = 37)
	assert torch.equal(O.ctc_alignment(lp.permute(2, 0, 1), y, olen[0], ylen, 37), al_ref)


# ------------------------------------------------------------------------------------------ train mode
def golden_state_dict(c):
	sd = O.synth_state_dict(c['shapes'], seed = c['seed'])
	assert abs(sum(float(v.double().abs().sum()) for v in sd.values() if v.is_floating_point()) - c['checksum']) < 1e-6 * c['checksum']
	return sd


def oracle_train_step(c, **kw):
	"""the oracle's TRAIN-mode forward + autograd backward on a golden case -> (logits, loss[B], grads, stats)"""
	sd = golden_state_dict(c)
	n_frozen = c['kwargs'].get('freeze', 0)
	is_frozen = lambda k: any(k.startswith(f'backbone.{i}.') for i in range(n_frozen))
	leaf = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and 'running' not in k and not is_frozen(k) else v.clone()) for k, v in sd.items()}
	over = {k: v for k, v in c['kwargs'].items() if k in ('groups', )}
	over['frozen_blocks'] = n_frozen
	if 'nonlinearity' in c['kwargs']:
		over['act'] = tuple(c['kwargs']['nonlinearity'])
	stats = {}
	logits, log_probs, olen = O.model_forward(leaf, c['signal'], c['xlen'], model = c['model'], training = True, stats_out = stats, **over, **kw)
	C = c['num_classes']
	nll = O.ctc_loss_torch(log_probs[0].permute(2, 0, 1), c['y'][:, 0], olen[0], c['ylen'][:, 0], C - 1)
	nll.mean().backward()  # == (loss / ylen * ylen).mean(), train.py:754-755
	grads = {k: v.grad for k, v in leaf.items() if v.is_floating_point() and v.requires_grad and v.grad is not None}
	return logits[0].detach(), nll.detach() / c['ylen'][:, 0], grads, stats


def check_grads_against_golden(grads, golden_grads, tol, what = ''):
	"""golden gradients are strided samples + norms (oracle/make_golden.py: compress_grad).  Returns (total rel error,
	worst per-tensor rel error).  Tensors whose true gradient is zero (a conv bias in front of a batch-statistics
	BatchNorm) hold rounding noise in the reference too: they are judged against the largest tensor's scale."""
	assert set(grads) == set(golden_grads), set(grads) ^ set(golden_grads)
	gmax = max(float(gg['sample'].double().norm()) for gg in golden_grads.values())
	worst, tot_d, tot_n = 0.0, 0.0, 0.0
	for k, gg in golden_grads.items():
		g = grads[k].detach().cpu().flatten()
		assert tuple(grads[k].shape) == gg['shape'], k
		s = g[::gg['stride']]
		d = float((s.double() - gg['sample'].double()).norm())
		n = float(gg['sample'].double().norm())
		tot_d += d * d
		tot_n += n * n
		e = d / max(n, 1e-3 * gmax)
		worst = max(worst, e)
		assert e < tol, (what, k, e)
		assert abs(float(g.double().norm()) - gg['norm']) <= tol * max(gg['norm'], 1e-3 * gmax), (what, k)
	total = (tot_d / tot_n)**0.5
	assert total < tol, (what, total)
	return total, worst


def test_train_mode_oracle_matches_reference_golden(golden):
	"""TRAIN mode (batch-statistics BN, autograd) of every golden family: logits, loss, all gradients, BN running stats"""
	g = golden('train')
	for c in g['cases']:
		logits, loss, grads, stats = oracle_train_step(c)
		assert rel(logits, c['logits']) < 1e-4, (c['model'], rel(logits, c['logits']))
		assert torch.allclose(loss, c['loss'], rtol = 1e-4, atol = 1e-4), c['model']
		# a hardtanh / relu gate that flips between two fp32 implementations moves the gradient by O(1 / sqrt(elements)):
		# the kinked full-depth cases are bounded loosely, the shallow and the smooth ones tightly (O.SMOOTH_NONLINEARITY)
		deep_kinked = 'nonlinearity' not in c['kwargs'] and c['kwargs'].get('num_blocks', 5) > 1
		total, worst = check_grads_against_golden(grads, c['grads'], 5e-2 if deep_kinked else 1e-3, c['model'])
		print(c['model'], c['kwargs'], 'oracle vs reference: total grad rel', total, 'worst tensor', worst)
		sd0 = golden_state_dict(c)
		for k, v in c['stats'].items():
			got = stats.get(k, sd0[k])  # frozen BatchNorms keep their buffers
			if k.endswith('num_batches_tracked'):
				assert int(got) == int(v), k
			else:
				assert torch.allclose(got, v, rtol = 1e-4, atol = 1e-5), k


def test_inplace_family_oracle_matches_the_reference_twin(golden):
	"""*Inplace model families (section 8f rank 4): the golden comes from the reference's non-in-place twin (the in-place forward
	needs CUDA-only ATen operators, oracle/make_golden.py: golden_train_inplace); the restatement, told only the class name,
	must reproduce it"""
	for c in golden('train_inplace')['cases']:
		logits, loss, grads, stats = oracle_train_step(c)
		assert rel(logits, c['logits']) < 1e-4, (c['model'], rel(logits, c['logits']))
		assert torch.allclose(loss, c['loss'], rtol = 1e-4, atol = 1e-4), c['model']
		total, worst = check_grads_against_golden(grads, c['grads'], 5e-2, c['model'])  # leaky_relu has a kink at 0: see the test above
		print(c['model'], 'oracle vs reference twin: total grad rel', total, 'worst tensor', worst)
		for k, v in c['stats'].items():
			if not k.endswith('num_batches_tracked'):
				assert torch.allclose(stats[k], v, rtol = 1e-4, atol = 1e-5), k


def test_misc_golden_novograd_uncertainty_bpe(golden):
	g = golden('misc')
	for c in g['novograd']:
		params = [p.clone() for p in c['p0']]
		state = [{} for _ in params]
		for st in c['steps']:
			O.novograd_step(params, st['grads'], state, lr = c['lr'], betas = c['betas'], weight_decay = c['weight_decay'], dampening = c['dampening'])
			for p, q in zip(params, st['params']):
				assert torch.allclose(p, q, rtol = 1e-6, atol = 1e-7)
	for c in g['uncertainty']:
		lp, lens = c['log_probs'], c['lengths']
		assert torch.allclose(O.entropy(lp, lens), c['entropy'], rtol = 1e-5, atol = 1e-6)
		assert torch.allclose(O.entropy(lp, None), c['entropy_nolen'], rtol = 1e-5, atol = 1e-6)
		assert torch.allclose(O.weighted_mean_entropy(lp, lens, eps_id = lp.shape[1] - 1), c['wme'], rtol = 1e-5, atol = 1e-6)
		assert torch.allclose(O.weighted_mean_entropy(lp, None, eps_id = lp.shape[1] - 1), c['wme_nolen'], rtol = 1e-5, atol = 1e-6)
		assert torch.allclose(O.margin(lp[:2]), c['margin'], rtol = 1e-6, atol = 1e-7)
		with pytest.raises(TypeError):
			O.margin(torch.cat([lp, lp])[:3])
	c = g['bpe']
	sd = O.synth_state_dict(c['shapes'], seed = c['seed'])
	logits, log_probs, olen = O.model_forward(sd, c['signal'], c['xlen'], model = c['model'])
	assert len(logits) == 2
	loss = 0
	for h in range(2):
		assert torch.equal(olen[h], c['olen'][h])
		assert rel(logits[h], c['logits'][h]) < 1e-4 and rel(log_probs[h], c['log_probs'][h]) < 1e-4
		C = c['num_classes'][h]
		loss = loss + O.ctc_loss_torch(log_probs[h].permute(2, 0, 1), c['y'][:, h], olen[h], c['ylen'][:, h], C - 1) / c['ylen'][:, 0]  # models.py:323: every head / ylen[:, 0]
	assert torch.allclose(loss, c['loss'], rtol = 1e-3, atol = 1e-3)
