"""Streaming acoustic model on the GPU: streamed features, log-probs, logits and argmax concatenated over calls equal the
one-shot forward under the same FixedNormalisation bit for bit (torch.equal), in the bf16 and fp32 tiers, for random
chunkings (0-sample chunks, chunks shorter than a hop or than the lookahead, streams of at most 128 samples) and
streams moving between rows; the online recogniser; bounded memory over a 10-minute stream; refusals; and the cost of
a prefix-estimated normalisation against per-utterance statistics, reported."""
import random
import zlib

import pytest
import torch

from convasr_b200 import decoders, models, streaming
from oracle import oracle as O

pytestmark = pytest.mark.gpu

HOP = 80


@pytest.fixture(scope = 'module')
def dev():
	return torch.device('cuda:0')


def _model(name, dev, precision, **kw):
	num_classes = kw.pop('num_classes', [38])
	args = dict(frontend = models.LogFilterBankFrontend(64, 8000, .02, .01, 'hann_window'), dropout = 0., check_time_dim_padded = False, base_width = 32)
	if name == 'JasperNetSeparable':
		args['groups'] = 32
	args.update(kw)
	m = getattr(models, name)(64, num_classes, **args)
	torch.manual_seed(7)
	with torch.no_grad():
		for mod in m.modules():
			if isinstance(mod, torch.nn.BatchNorm1d):
				mod.running_mean.uniform_(-0.1, 0.1)
				mod.running_var.uniform_(0.5, 1.5)
	return m.to(dev).eval().set_precision(precision)


def _signals(lengths, seed):
	g = torch.Generator().manual_seed(seed)
	return [(torch.randn(n, generator = g) * 3000).round().clamp(-32767, 32767).to(torch.int16) for n in lengths]


def _chunkings(rng, n):
	"""random cut points, with 0-sample chunks, sub-hop chunks and long chunks"""
	cuts = sorted(rng.randint(0, n) for _ in range(rng.randint(1, 9)))
	sizes = [b - a for a, b in zip([0] + cuts, cuts + [n])]
	return sizes + [0] * rng.randint(0, 1)


def _run_streams(sm, sigs, norm, dev, rng):
	"""feed every stream in random chunks; each call batches the streams that still have chunks, in shuffled rows.
	Returns per stream and head the concatenated (logits, log_probs, argmax)."""
	plans = [_chunkings(rng, s.numel()) for s in sigs]
	pos = [0] * len(sigs)
	states = [sm.new_state(norm[i]) for i in range(len(sigs))]
	got = [[([], [], []) for _ in sm.heads] for _ in sigs]
	while any(plans):
		live = [i for i in range(len(sigs)) if plans[i]]
		rng.shuffle(live)
		chunks, eos = [], []
		for i in live:
			n = plans[i].pop(0)
			c = sigs[i][pos[i]:pos[i] + n]
			chunks.append((c.float() if rng.random() < 0.5 else c).to(dev))
			pos[i] += n
			eos.append(not plans[i])
		out = sm.forward(chunks, [states[i] for i in live], eos)
		lens = out['lengths'].tolist()
		for r, i in enumerate(live):
			for h in range(len(sm.heads)):
				got[i][h][0].append(out['logits'][h][r, :, :lens[r]])
				got[i][h][1].append(out['log_probs'][h][r, :, :lens[r]])
				got[i][h][2].append(out['argmax'][h][r, :lens[r]])
	return [[tuple(torch.cat(x, dim = -1) for x in head) for head in g] for g in got]


LENGTHS = [16000 + 37, 7001, 100, 129, 2400]


def test_streamed_features_equal_the_one_shot_frontend(dev):
	rng = random.Random(1)
	for precision in ('bf16', 'fp32'):
		m = _model('Wav2Letter', dev, precision)
		sigs = _signals(LENGTHS, 3)
		norm = streaming.estimate_normalisation(m, torch.stack([s[:2000] for s in sigs[:1]] * len(sigs)).to(dev))
		feats = {}

		class Capture(streaming.StreamingModel):
			def _frontend(self, chunks, states, n_new, eos, old, new, plan, dev):
				act = super()._frontend(chunks, states, n_new, eos, old, new, plan, dev)
				for b, st in enumerate(states):
					n = new[b]['feat'] - old[b].get('feat', 0)
					if act is not None and n:
						feats.setdefault(id(st), []).append((act.hi[b, :n], act.lo[b, :n] if act.lo is not None else None))
				return act

		sm = Capture(m)
		states = []
		orig_new_state = sm.new_state
		sm.new_state = lambda nr: states.append(orig_new_state(nr)) or states[-1]
		_run_streams(sm, sigs, norm, dev, rng)
		plan = m._get_plan()
		for i, s in enumerate(sigs):
			hi, lo, Fr = m.frontend.features(s[None].to(dev), None, m.normalize_features, True, 64, plan.fp32_tier, norm[i])
			got = feats[id(states[i])]
			g_hi = torch.cat([h for h, _ in got])
			assert g_hi.shape[0] == Fr, (precision, i)
			assert torch.equal(g_hi, hi[0, :Fr]), (precision, i, (g_hi != hi[0, :Fr]).any(-1).nonzero().flatten()[:16].tolist())
			if precision == 'fp32':
				assert torch.equal(torch.cat([l for _, l in got]), lo[0, :Fr]), i


MODELS = [
	('Wav2Letter', {}), ('Wav2LetterResidual', {}), ('Wav2LetterDense', {}), ('Wav2LetterFlat', {}), ('JasperNetSeparable', {}),
	('Wav2Letter', dict(decoder_type = 'bpe', num_classes = [38, 300])), ('Wav2Letter', dict(num_classes = [1000]))
]


@pytest.mark.parametrize('precision', ['bf16', 'fp32'])
@pytest.mark.parametrize('name,kw', MODELS, ids = [f'{n}-{"-".join(map(str, k.values())) or "ctc"}' for n, k in MODELS])
def test_streamed_model_equals_the_one_shot_forward(dev, name, kw, precision):
	rng = random.Random(zlib.crc32(f'{name}{kw}{precision}'.encode()))
	m = _model(name, dev, precision, **dict(kw))
	sigs = _signals(LENGTHS, 11)
	norm = streaming.estimate_normalisation(m, torch.stack([s[:2000] for s in sigs[:1]] * len(sigs)).to(dev))
	sm = streaming.StreamingModel(m)
	got = _run_streams(sm, sigs, norm, dev, rng)
	for i, s in enumerate(sigs):
		with torch.no_grad():
			ref = m(s[None].to(dev), normalisation = norm[i])
		for h in range(len(sm.heads)):
			lg, lp, am = got[i][h]
			T = ref['log_probs'][h].shape[-1]
			assert lp.shape[-1] == T == int(ref['olen'][h][0]), (i, h)
			assert torch.equal(lg, ref['logits'][h][0]), (i, h, 'logits')
			assert torch.equal(lp, ref['log_probs'][h][0]), (i, h, 'log_probs')
			if h == 0:
				assert torch.equal(am, ref['log_probs'][h]._convasr_argmax[0]), (i, h, 'argmax')


def test_online_recogniser_equals_one_shot_beam_search(dev):
	rng = random.Random(4)
	m = _model('Wav2LetterResidual', dev, 'fp32')
	labels = list('_абвгдеёжзийклмнопрстуфхцчшщъыьэюя 0123') [:38]
	labels[-1] = '|'
	sigs = _signals([12000, 5003, 8000], 21)
	norm = streaming.estimate_normalisation(m, torch.stack([s[:2000] for s in sigs]).to(dev))
	sm = streaming.StreamingModel(m)
	online = decoders.OnlineBeamSearchDecoder(labels, beam_width = 16)
	states = [sm.new_state(norm[i]) for i in range(len(sigs))]
	beams = [online.new_state() for _ in sigs]
	final = [[] for _ in sigs]
	tails = [None] * len(sigs)
	plans = [_chunkings(rng, s.numel()) for s in sigs]
	pos = [0] * len(sigs)
	while any(plans):
		live = [i for i in range(len(sigs)) if plans[i]]
		chunks, eos = [], []
		for i in live:
			n = plans[i].pop(0)
			chunks.append(sigs[i][pos[i]:pos[i] + n].to(dev))
			pos[i] += n
			eos.append(not plans[i])
		out = sm.forward(chunks, [states[i] for i in live], eos)
		res = online.decode_incremental(out['log_probs'][0], [beams[i] for i in live], eos, out['lengths'])
		for r, i in enumerate(live):
			final[i] += res[r][0]
			tails[i] = res[r][1]
	one_shot = decoders.BeamSearchDecoder(labels, beam_width = 16)
	for i, s in enumerate(sigs):
		with torch.no_grad():
			ref = m(s[None].to(dev), normalisation = norm[i])
		want = one_shot.decode(ref['log_probs'][0])
		assert final[i] + tails[i][0] == want[0], i


def test_memory_stays_bounded_over_a_long_stream(dev):
	"""30 000 output frames (10 minutes) in 50-frame chunks: the rebase runs and the bytes held stay under twice the live
	rows (context + one chunk) of every activation"""
	m = _model('Wav2LetterDense', dev, 'bf16')
	sm = streaming.StreamingModel(m)
	norm = models.FixedNormalisation(torch.full((1, ), 1e-4, device = dev), torch.zeros(1, 64, device = dev), torch.ones(1, 64, device = dev))
	st = sm.new_state(norm)
	chunk = 50 * 2 * HOP
	g = torch.Generator(device = dev).manual_seed(0)
	plan = m._get_plan()
	# the bound: per activation, rows a consumer still reads in steady state plus one chunk, doubled by the growth policy
	n_big = 100_000 * HOP
	fin = sm.schedule(n_big, False)
	nxt = sm.schedule(n_big + chunk, False)
	bound = 4 * (HOP + 256 + 1 + 4)
	for node in sm.consumers:
		live = fin[node] - sm._keep_from(node, fin) + (nxt[node] - fin[node])
		bound += 2 * (live + 16) * sm._width(node, plan) * 2
	held, frames = [], 0
	for call in range(600):
		x = (torch.randn(chunk, generator = g, device = dev) * 3000).round()
		out = sm.forward([x], [st], [call == 599])
		frames += int(out['lengths'][0])
		held.append(st.bytes_held() if call < 599 else held[-1])
	assert frames == sm.schedule(600 * chunk, True)[sm.heads[0].node]
	assert st.rebases > 0
	assert max(held) <= bound, (max(held), bound)
	assert max(held[300:]) == max(held[100:300])  # flat: no growth after the first minute


def test_refusals(dev):
	m = _model('Wav2Letter', dev, 'bf16')
	sm = streaming.StreamingModel(m)
	norm = models.FixedNormalisation(torch.ones(1, device = dev), torch.zeros(1, 64, device = dev), torch.ones(1, 64, device = dev))
	st = sm.new_state(norm)
	x = torch.zeros(400, dtype = torch.int16, device = dev)
	with pytest.raises(RuntimeError, match = 'CUDA'):
		sm.forward([x.cpu()], [st], [False])
	other = streaming.StreamingModel(m)
	with pytest.raises(ValueError, match = 'another StreamingModel'):
		other.forward([x], [st], [False])
	sm.forward([x], [st], [True])
	with pytest.raises(RuntimeError, match = 'after its eos'):
		sm.forward([x], [st], [False])
	st = sm.new_state(norm)
	with pytest.raises(ValueError, match = 'two rows'):
		sm.forward([x, x], [st, st], [False, False])
	m.train()
	with pytest.raises(RuntimeError, match = 'eval-mode'):
		sm.forward([x], [st], [False])
	m.eval()
	m.set_precision('fp32')
	with pytest.raises(RuntimeError, match = 'plan changed'):
		sm.forward([x], [st], [False])
	m.set_precision('bf16')
	sm = streaming.StreamingModel(m)
	st = sm.new_state(norm)
	m.fuse_conv_bn_eval()
	with pytest.raises(RuntimeError, match = 'plan changed'):
		sm.forward([x], [st], [False])
	sm = streaming.StreamingModel(m)
	st = sm.new_state(norm)
	with torch.no_grad():
		m.decoder[0].bias.add_(1.0)
	with pytest.raises(RuntimeError, match = 'plan changed'):
		sm.forward([x], [st], [False])
	with pytest.raises(RuntimeError, match = 'plan changed'):
		sm.new_state(norm)
	m.set_precision('fp8')
	with pytest.raises((NotImplementedError, RuntimeError), match = 'fp8'):
		streaming.StreamingModel(m)
	m.set_precision('bf16').train()
	with pytest.raises(RuntimeError, match = 'eval'):
		m(x[None].repeat(1, 40), normalisation = norm)


def test_normalisation_cost_is_reported(golden, dev, capsys):
	"""greedy ids and greedy text with the normalisation estimated on a prefix against today's per-utterance forward, on
	the golden models (random-init weights; their signals are about 1 s, so the prefix is the first 0.5 s, not 2 s):
	reported, not asserted"""
	from convasr_b200 import transcript_generators
	tok = O.CharTokenizer('абвгдеёжзийклмнопрстуфхцчшщъыьэюя')
	gen = transcript_generators.GreedyCTCGenerator()

	def edit(a, b):
		d = list(range(len(b) + 1))
		for i, ca in enumerate(a, 1):
			p, d[0] = d[0], i
			for j, cb in enumerate(b, 1):
				p, d[j] = d[j], min(d[j] + 1, d[j - 1] + 1, p + (ca != cb))
		return d[-1]

	lines = []
	for c in golden('models')['cases']:
		m = getattr(models, c['model'])(64, [c['num_classes']], frontend = models.LogFilterBankFrontend(64, 8000, .02, .01, 'hann_window'), dropout = 0., check_time_dim_padded = False, **c['kwargs'])
		m.load_state_dict(O.synth_state_dict(c['shapes'], seed = c['seed']), strict = False)
		m = m.to(dev).eval()
		sig = c['signal'].to(dev)
		B = sig.shape[0]
		with torch.no_grad():
			per_utt = m(sig)
			norm = streaming.estimate_normalisation(m, sig[:, :4000])
			fixed = m(sig, normalisation = norm)
		a, b = per_utt['log_probs'][0]._convasr_argmax, fixed['log_probs'][0]._convasr_argmax
		agree = float((a == b).float().mean())
		ends = dict(begin = torch.zeros(B, device = dev), end = torch.ones(B, device = dev))
		line = f'{c["model"]:20s} fused={c["fused"]}: greedy-id agreement {agree:.4f}'
		if c['num_classes'] != 38:
			lines.append(line)
			continue
		ta = gen.generate(tok, per_utt['log_probs'][0], output_lengths = per_utt['olen'][0], **ends)
		tb = gen.generate(tok, fixed['log_probs'][0], output_lengths = fixed['olen'][0], **ends)
		ha = [' '.join(s['hyp'] for s in t[0]) for t in ta]
		hb = [' '.join(s['hyp'] for s in t[0]) for t in tb]
		cer = sum(edit(x, y) for x, y in zip(hb, ha)) / max(1, sum(len(y) for y in ha))
		lines.append(line + f', CER vs per-utterance text {cer:.4f}')
	with capsys.disabled():
		print('\nnormalisation estimated on the first 0.5 s vs per-utterance statistics (random-init weights):\n  ' + '\n  '.join(lines))


def test_buffers_that_grow_together_in_one_call_stay_exact(dev):
	"""24 streams of equal length fed in lock step with growing chunks, so every stream replaces its buffers in the same
	calls (the old buffers' rows are copied out by the same launch that may write the new ones): the streamed outputs
	still equal the one-shot forward bit for bit"""
	m = _model('Wav2LetterDense', dev, 'fp32')
	sizes = [400, 1200, 5000, 20000, 3000]
	sigs = _signals([sum(sizes)] * 24, 31)
	norm = streaming.estimate_normalisation(m, torch.stack([s[:4000] for s in sigs]).to(dev))
	sm = streaming.StreamingModel(m)
	states = [sm.new_state(norm[i]) for i in range(len(sigs))]
	got = [([], [], []) for _ in sigs]
	pos, grown_together = 0, 0
	for j, n in enumerate(sizes):
		before = [st.grows for st in states]
		out = sm.forward([s[pos:pos + n].to(dev) for s in sigs], states, [j == len(sizes) - 1] * len(sigs))
		pos += n
		grown_together = max(grown_together, sum(st.grows > g for st, g in zip(states, before)))
		lens = out['lengths'].tolist()
		for r in range(len(sigs)):
			got[r][0].append(out['logits'][0][r, :, :lens[r]])
			got[r][1].append(out['log_probs'][0][r, :, :lens[r]])
			got[r][2].append(out['argmax'][0][r, :lens[r]])
	assert grown_together == len(sigs)
	for i, s in enumerate(sigs):
		with torch.no_grad():
			ref = m(s[None].to(dev), normalisation = norm[i])
		lg, lp, am = (torch.cat(x, dim = -1) for x in got[i])
		assert torch.equal(lg, ref['logits'][0][0]), i
		assert torch.equal(lp, ref['log_probs'][0][0]), i
		assert torch.equal(am, ref['log_probs'][0]._convasr_argmax[0]), i


def test_fixed_normalisation_against_per_utterance_statistics(dev):
	"""a check of the fixed-statistics kernels that does not go through them twice: the normalisation estimated on each
	whole utterance is a torch restatement of the reference's (signal scale exactly, statistics of the log-mel within
	float32 rounding), and the fixed path under it reproduces today's per-utterance path, whose only difference is
	(x - mean) * invstd in place of (x - mean) / sd: features within the split-bf16 resolution, logits to 1e-4"""
	m = _model('Wav2LetterResidual', dev, 'fp32')
	sig = torch.stack(_signals([16000, 16000, 16000], 41)).to(dev)
	sig[1] //= 7  # a different abs-max per row
	norm = streaming.estimate_normalisation(m, sig)
	amax = sig.float().abs().amax(dim = 1)
	assert torch.equal(norm.signal_scale, 1.0 / (amax + 1e-5))
	with torch.no_grad():
		logmel = m.frontend(sig).double()  # today's frontend: per-utterance abs-max
	mean = logmel.mean(dim = 2)
	sd = (((logmel - mean[..., None]) ** 2).mean(dim = 2) + m.normalize_features.eps).sqrt()
	assert torch.allclose(norm.mean.double(), mean, rtol = 0, atol = 1e-4)
	assert torch.allclose(norm.invstd.double(), 1 / sd, rtol = 5e-5, atol = 0)
	plan = m._get_plan()
	hi, lo, Fr = m.frontend.features(sig, None, m.normalize_features, True, 64, True)
	fhi, flo, _ = m.frontend.features(sig, None, m.normalize_features, True, 64, True, norm)
	want, got = hi.float() + lo.float(), fhi.float() + flo.float()
	assert (got - want).abs().max() <= 5e-5 * want.abs().max(), float((got - want).abs().max())
	assert plan.fp32_tier
	with torch.no_grad():
		a, b = m(sig), m(sig, normalisation = norm)
	r = float((a['logits'][0] - b['logits'][0]).norm() / a['logits'][0].norm())
	assert r < 1e-4, r
	wrong = models.FixedNormalisation(norm.signal_scale * 2, norm.mean, norm.invstd)
	with torch.no_grad():
		c = m(sig, normalisation = wrong)
	assert float((a['logits'][0] - c['logits'][0]).norm() / a['logits'][0].norm()) > 1e-3  # the check can fail
