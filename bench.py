"""Headline benchmark: audio-seconds per second (RTFx) of the Wav2Letter forward + CTC path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload NAME]

Default workload = BASELINE.json configs[1]: Wav2Letter-char (66.5 M params, 38 classes) TRAINING
STEP, batch 80 x 15 s of synthetic 8 kHz int16 PCM, every utterance full length (xlen = 1, as the
reference's own benchmark.py feeds it), bf16.  One step = log-mel
frontend -> instance norm -> 18 conv + batch-statistics BatchNorm + hardtanh + mask layers -> decoder
+ log_softmax -> CTC loss -> backward through everything (CTC gradient, log_softmax, decoder, BN,
dgrad and wgrad of every conv) -> clip_grad_norm(100) + SGD(momentum 0.9, weight decay 1e-3) update (the
reference's train.py defaults, train.py:657-662,776-779) as one native multi-tensor step.  The whole step
runs on this repo's kernels.  N > 1: data-parallel replicas; every layer's weight gradient is
all-reduced (NCCL) from inside the native backward as soon as it exists, inside the same CUDA graph; after the
timed steps the replicas' parameters are compared bit for bit ("replicas_identical").

"also" (every N): the same training step on a RAGGED batch; the inference path of the same shape (eval forward with
folded BatchNorm + greedy collapse + CTC loss + CTC gradient); BASELINE configs[4]: the utterance-sharded inference
sweep, 8192 utterances x 10 s split over the ranks in micro-batches of 256 (no data-path collective).
N = 1 only: BASELINE configs[0] (C1, with the reference's own CPU time beside it), configs[2] (C3), configs[3] (C4),
each with its own roofline, and "gpu_baseline": the UNMODIFIED reference (baseline/_ref, cuDNN / ATen / cuFFT) running
the headline training step on the same GPU.

value  = whole-job audio-seconds / second with the PCM already resident in HBM (CUDA events).
e2e    = same metric through the public module API with HOST buffers: pinned int16 PCM + targets
         -> H2D through convasr_b200.feed.DeviceFeeder (every step uploads its own batch; the copy of step
         i+1 overlaps the compute of step i), the step, D2H of the per-utterance loss (and the greedy
         ids for inference).
kernels = per C-ABI entry point: launches, device ms per step (CUDA events around every call of one eager
         step), algorithmic bytes / FLOPs and the fraction of the measured peak that bounds it.
N > 1  = per-GPU batch fixed (weak scaling); time = max over ranks.
--impl reference = the UNMODIFIED reference (baseline/_ref or /root/reference: models.py + torch CPU ops, all host
         threads, its own train-loop body train.py:748-779) on a bounded sample of the same workload; when the
         staged reference is absent, the oracle port (cpu_baseline.kind says which).
--dump-outputs DIR = after the timed steps of the selected workload, write what its last timed step handed back to
         the caller as DIR/<name>.npy (float32; integer outputs as float64), outputs larger than 16 MB as a fixed,
         seeded sample: training -> per-utterance loss and the updated parameters; inference -> loss, log-probs,
         their CTC gradient, greedy tokens and token counts; sweep -> loss and token counts of the whole pass.  With
         --gpus N > 1 rank 0 writes: its batch, or for the sweep its shard.
         Inputs and weights are seeded, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
	sys.path.insert(0, ROOT)

import torch

WORKLOADS = {
	# name: (model, num_classes, batch, seconds, precision, kind, lengths)
	#   lengths 'full'  : every utterance fills its row, xlen = 1 (the reference's own benchmark.py:126 style; BASELINE "80 x 15 s")
	#   lengths 'ragged': xlen ~ U(0.5, 1] (SURVEY.md 8d "recommended additionally": exercises masks); on average 25 % of every row
	#                     is padding, whose tiles the conv / wgrad kernels leave out (exact: they are structural zeros)
	'wav2letter_char_train_step_B80x15s_bf16': ('Wav2Letter', 38, 80, 15.0, 'bf16', 'train', 'full'),
	'wav2letter_char_train_step_B80x15s_bf16_ragged': ('Wav2Letter', 38, 80, 15.0, 'bf16', 'train', 'ragged'),
	'wav2letter_char_fwd_ctc_B80x15s_bf16': ('Wav2Letter', 38, 80, 15.0, 'bf16', 'infer', 'full'),
	'wav2letter_char_fwd_ctc_B80x15s_bf16_ragged': ('Wav2Letter', 38, 80, 15.0, 'bf16', 'infer', 'ragged'),
	'wav2letter_char_fwd_ctc_B8x10s_fp32': ('Wav2Letter', 38, 8, 10.0, 'fp32', 'infer', 'ragged'),  # BASELINE configs[0] (C1)
	'jasper_separable_fwd_ctc_B256x20s_bf16': ('JasperNetSeparable', 38, 256, 20.0, 'bf16', 'infer', 'full'),  # configs[2] (C3)
	'wav2letter_bpe5000_fwd_ctc_B64x15s_bf16': ('Wav2Letter', 5000, 64, 15.0, 'bf16', 'infer', 'full'),  # configs[3] (C4)
	'wav2letter_char_infer_sweep_8192x10s_bf16': ('Wav2Letter', 38, 256, 10.0, 'bf16', 'sweep', 'ragged'),  # configs[4] (C5): batch = micro-batch
}
SWEEP_UTTERANCES = 8192
DEFAULT_WORKLOAD = 'wav2letter_char_train_step_B80x15s_bf16'
SECONDARY_WORKLOADS = ['wav2letter_char_train_step_B80x15s_bf16_ragged', 'wav2letter_char_fwd_ctc_B80x15s_bf16', 'wav2letter_char_infer_sweep_8192x10s_bf16']
SINGLE_GPU_WORKLOADS = ['wav2letter_char_fwd_ctc_B8x10s_fp32', 'jasper_separable_fwd_ctc_B256x20s_bf16', 'wav2letter_bpe5000_fwd_ctc_B64x15s_bf16']
# mean DRAM bytes per launch of the tensor-pipe kernels, from the committed ncu --set full captures
NCU_DRAM_BYTES_PER_LAUNCH = {
	'wav2letter_char_train_step_B80x15s_bf16': 131.2e6,  # profiles/r01_train_step_tensor_kernels_ncu_full.csv (56 launches)
	'wav2letter_char_train_step_B80x15s_bf16_ragged': 131.2e6,
	'wav2letter_char_fwd_ctc_B80x15s_bf16': 105.0e6,  # profiles/r01_step_kernels_ncu_full.csv (conv1d_umma_kernel launches)
}
STEP_DESC = {
	'train': 'frontend+instnorm+18x(conv, batch-stat BN, hardtanh, mask)+decoder/log_softmax+CTC loss+full backward (CTC grad, BN bwd, dgrad, wgrad)+clip_grad_norm+SGD(momentum,wd) update',
	'infer': 'frontend+instnorm+conv stack (BN folded)+decoder/log_softmax/argmax+greedy CTC collapse+CTC loss+CTC grad (no conv backward)',
	'sweep': f'{SWEEP_UTTERANCES} utterances sharded over the ranks, micro-batches of 256: frontend+instnorm+conv stack (BN folded)+decoder/log_softmax/argmax+greedy CTC collapse+CTC loss; one pass over the shard',
}
SAMPLE_RATE = 8000
LENGTHS_DESC = {
	'full': 'xlen = 1: every utterance fills its row (benchmark.py:126 style)',
	'ragged': 'xlen ~ U(0.5, 1]: ~25 % of each row is padding; value counts PADDED seconds; tiles of pure padding are left out of the GEMMs (structural zeros, exact)',
}
FP32_FMA_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12  # nominal: 148 SMs x 128 fp32 lanes x 2 FLOP x 1.965 GHz (no measured fp32 peak in MEASURED_PEAKS.json)


def synth_batch(B, seconds, C, seed, lengths = 'ragged'):
	"""SURVEY.md 8(d): int16 PCM round(3000*N(0,1)); targets never the blank, lengths such that an alignment exists.
	'ragged': xlen ~ U(0.5, 1] with one full-length row; 'full': xlen = 1 (benchmark.py:126), target lengths up to
	0.3 * t_out (SURVEY C2: L <~ 225 of t = 753)."""
	g = torch.Generator().manual_seed(seed)
	T = int(seconds * SAMPLE_RATE)
	sig = (torch.randn(B, T, generator = g) * 3000).round().clamp(-32767, 32767).to(torch.int16)
	xlen = torch.rand(B, generator = g) * 0.5 + 0.5
	xlen[0] = 1.0
	t_out = (T // 80 + 1 - 1) // 2 + 1 + 2
	if lengths == 'full':
		xlen = torch.ones(B)
		L = int(0.3 * t_out)
		lo = max(1, L // 3)
	else:
		t_min = int((xlen.min() * t_out).ceil())
		L = int(0.45 * t_min)
		lo = max(1, int(0.2 * t_min / 2))
	ylen = torch.randint(lo, L + 1, (B, ), generator = g)
	y = torch.randint(0, C - 1, (B, 1, L), generator = g)
	return sig, xlen, y, ylen.unsqueeze(1)


def model_shapes(model_name, C):
	from convasr_b200 import models
	m = getattr(models, model_name)(64, [C], dropout = 0.)
	return {k: tuple(v.shape) for k, v in m.state_dict().items()}


def conv_flops_per_step(model, B, F):
	"""algorithmic 2*MAC of every conv (real channels, real frames, no padding), SURVEY.md 8(d); (dense GEMM flops,
	grouped-conv flops, output frames)"""
	import torch.nn as nn
	dense, grouped = 0, 0
	t = F
	for block in model.backbone:
		for seq in block.conv:
			for conv in seq:
				if isinstance(conv, nn.Conv1d):
					t = (t + 2 * conv.padding[0] - conv.dilation[0] * (conv.kernel_size[0] - 1) - 1) // conv.stride[0] + 1
					fl = 2 * B * t * conv.out_channels * (conv.in_channels // conv.groups) * conv.kernel_size[0]
					if conv.groups > 1:
						grouped += fl
					else:
						dense += fl
		for rc in block.conv_residual:
			if isinstance(rc, nn.Conv1d):
				dense += 2 * B * t * rc.out_channels * rc.in_channels
	d = model.decoder[0]
	dense += 2 * B * t * d.out_channels * d.in_channels
	return dense, grouped, t


def algorithmic_bytes(model, B, T, t_out, C, kind, L):
	"""algorithmic HBM bytes per step of the memory-bound entry points (SURVEY.md 8(d) per-unit figures x this batch)"""
	import torch.nn as nn
	F = T // 80 + 1
	out = {
		'cab_frontend_logmel': B * T * 2 + B * 64 * F * 4,  # int16 PCM in, fp32 log-mel out
		'cab_instnorm_pack': B * 64 * F * 4 + B * (F + F % 2) * 64 * 2,  # fp32 log-mel in, bf16 channels-last out
		'cab_ctc_loss_fwd': B * t_out * C * 4 + 2 * B * t_out * (2 * L + 1) * 4,  # log_probs read; alpha and beta written
		'cab_ctc_loss_bwd': 2 * B * t_out * C * 4 + 2 * B * t_out * (2 * L + 1) * 4,  # log_probs read, grad written; alpha, beta read
		'cab_greedy_collapse': B * t_out * 4 * 2,
		'cab_log_softmax_argmax': B * t_out * C * 4 * 2,
		'cab_log_softmax_rows': B * t_out * C * 4 * 2,  # logits read, log-probs written
		'cab_frontend_features': B * T * 2 + B * (F + F % 2) * 64 * 2,  # int16 PCM in, normalised bf16 channels-last features out (SURVEY 8d: 28.8 KB per audio-second)
	}
	if kind == 'train':
		acts, t, params = 0, F, 0
		for block in model.backbone:
			for seq in block.conv:
				conv = seq[0]
				t = (t + 2 * conv.padding[0] - conv.dilation[0] * (conv.kernel_size[0] - 1) - 1) // conv.stride[0] + 1
				acts += B * t * ((conv.out_channels + 63) // 64 * 64) * 2
				params += conv.weight.numel()
		params += model.decoder[0].weight.numel()
		n_all = sum(p.numel() for p in model.parameters() if p.requires_grad)
		out.update({
			'cab_bn_act_mask_fwd_stats': 2 * acts,  # y read, activation written
			'cab_bn_act_mask_bwd': 5 * acts,  # reduce: y, g read; apply: y, g read, dy written
			'cab_bn_act_mask_bwd_apply': 3 * acts,  # the channel sums came out of the dgrad epilogue: y, g read, dy written
			'cab_pack_weights_batched': params * (4 + 2 + 2),  # fp32 master read, forward + dgrad bf16 operands written
			'cab_unpack_wgrad': params * 8,
			'cab_unpack_wgrad_batched': params * 8,
			'cab_optimizer_step': n_all * 20 + n_all * 4,  # p, g, m read + p, m written; g read once more for the norm
			'cab_log_softmax_bwd': 3 * B * t_out * C * 4,
			'cab_bct_to_btc': B * t_out * C * 4 + B * t_out * 64 * 2,
		})
	return out


class ClockSampler:
	"""nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""

	def __init__(self, index):
		self.index, self.rows, self.proc = index, [], None

	def start(self):
		q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
		try:
			self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={q}', '--format=csv,noheader,nounits', '-lms', '100'], stdout = subprocess.PIPE, stderr = subprocess.DEVNULL, text = True)
			threading.Thread(target = self._read, daemon = True).start()
		except Exception:
			self.proc = None

	def _read(self):
		for line in self.proc.stdout:
			self.rows.append((time.time(), [c.strip() for c in line.split(',')]))

	def stop(self, t0, t1):
		if self.proc is None:
			return None
		time.sleep(0.15)
		self.proc.terminate()
		rows = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.2] or [r for _, r in self.rows[-3:]]
		if not rows:
			return None
		try:
			sm = sorted(float(r[0]) for r in rows)
			reasons = set()
			for r in rows:
				for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], r[3:7]):
					if v.lower().startswith('active'):
						reasons.add(name)
			return dict(sm_mhz = sm[len(sm) // 2], sm_max_mhz = float(rows[0][1]), power_w_max = max(float(r[2]) for r in rows), reasons = sorted(reasons), samples = len(rows))
		except Exception:
			return None


def measured_peaks():
	try:
		return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
	except Exception:
		return None


DUMP_BYTES_PER_ARRAY = 16 << 20
DUMP_BYTES_TOTAL = 64 << 20


def host_outputs(outputs):
	"""device tensors -> numpy arrays for --dump-outputs: float32, integer tensors as float64 (exact); a tensor above
	DUMP_BYTES_PER_ARRAY becomes a sample of its flattened values at indices drawn from a fixed seed, the same in every run"""
	import numpy as np
	out = {}
	for name, t in outputs.items():
		t = t.detach()
		dtype = torch.float32 if t.is_floating_point() else torch.float64
		limit = DUMP_BYTES_PER_ARRAY // (4 if dtype == torch.float32 else 8)
		if t.numel() > limit:
			idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), limit))
			t = t.flatten()[torch.from_numpy(idx).to(t.device)]
		out[name] = t.to(dtype).cpu().numpy()
	assert sum(a.nbytes for a in out.values()) <= DUMP_BYTES_TOTAL, {n: a.nbytes for n, a in out.items()}
	return out


# --------------------------------------------------------------------------------------------
# reference arms: the UNMODIFIED reference (baseline/_ref staged by __graft_entry__.build(), or /root/reference) through
# its own public API; the oracle port only when neither exists
# --------------------------------------------------------------------------------------------
def reference_available():
	from oracle import reference_shim
	return reference_shim.available()


def reference_model(model_name, C, device, seed_shapes_from = None):
	"""the reference's own module tree with this bench's seeded weights"""
	from oracle import oracle as O, reference_shim
	model = reference_shim.make_model(model_name, (C, ), frontend = True)
	shapes = {k: tuple(v.shape) for k, v in model.state_dict().items() if not k.startswith('frontend.')}
	model.load_state_dict(O.synth_state_dict(shapes, seed = 0), strict = False)
	return model.to(device)


def reference_step_fn(model, kind, C, tokenizer = None):
	"""one step of the workload through the reference's public API: its train-loop body (train.py:748-779) or its
	transcribe flow (forward + GreedyCTCGenerator.generate + loss)"""
	from oracle import reference_shim
	ref = reference_shim.load()
	if kind == 'train':
		model.train()
		opt = torch.optim.SGD(model.parameters(), lr = 1e-6, momentum = 0.9, weight_decay = 1e-3)  # train.py:657-662 defaults

		def step(sig, xlen, y, ylen):
			out = model(sig, xlen, y = y, ylen = ylen)
			loss = (out['loss'] * ylen[:, 0]).mean()  # train.py:754-755
			loss.backward()
			torch.nn.utils.clip_grad_norm_(model.parameters(), 100.0, error_if_nonfinite = False)  # train.py:776-779
			opt.step()
			opt.zero_grad()
			return out['loss'].detach()
		return step
	model.eval()
	model.fuse_conv_bn_eval()
	gen = ref.transcript_generators.GreedyCTCGenerator()
	tok = tokenizer or ref.text_tokenizers.CharTokenizerLegacy('абвгдеёжзийклмнопрстуфхцчшщъыьэюя')

	def step(sig, xlen, y, ylen):
		with torch.no_grad():
			out = model(sig, xlen, y = y, ylen = ylen)
			if C == len(tok.idx2char):
				gen.generate(tok, out['log_probs'][0], begin = torch.zeros(len(sig)), end = torch.ones(len(sig)), output_lengths = out['olen'][0])
		return out['loss']
	return step


def port_step_fn(model_name, C, kind):
	"""fallback when the reference is not staged: the oracle port of the same step"""
	from oracle import oracle as O
	shapes = {k: s for k, s in model_shapes(model_name, C).items() if not k.startswith('frontend.')}
	sd = O.synth_state_dict(shapes, seed = 0)

	def step(sig, xlen, y, ylen):
		if kind == 'train':
			leaf = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and 'running' not in k else v) for k, v in sd.items()}
			logits, log_probs, olen = O.model_forward(leaf, sig, xlen, model = model_name, training = True)
			loss = O.ctc_loss_torch(log_probs[0].permute(2, 0, 1), y[:, 0], olen[0], ylen[:, 0], C - 1).mean()
			loss.backward()
			with torch.no_grad():
				for k, v in leaf.items():
					if v.is_floating_point() and v.grad is not None:
						sd[k] = sd[k] - 1e-6 * v.grad
			return loss.detach()
		logits, log_probs, olen = O.model_forward(sd, sig, xlen, model = model_name)
		lp = log_probs[0].permute(2, 0, 1).detach().requires_grad_(True)
		loss = O.ctc_loss_torch(lp, y[:, 0], olen[0], ylen[:, 0], C - 1)
		loss.sum().backward()
		return loss.detach()
	return step


def run_cpu_reference(name, sample_B, steps, warmup):
	"""(value audio-s/s, s/step, cpu_baseline dict) of the reference's CPU path on a bounded sample of workload `name`"""
	model_name, C, B, seconds, precision, kind, lengths = WORKLOADS[name]
	kind = 'infer' if kind == 'sweep' else kind
	torch.set_num_threads(os.cpu_count())
	if reference_available():
		step, src = reference_step_fn(reference_model(model_name, C, 'cpu'), kind, C), 'reference'
		how = f'UNMODIFIED reference models.py / transcript_generators.py via oracle/reference_shim.py, torch {torch.__version__} CPU ops, fp32'
	else:
		step, src = port_step_fn(model_name, C, kind), 'port'
		how = f'oracle port (reference tree not staged under baseline/_ref): torch {torch.__version__} CPU ops, fp32'
	sig, xlen, y, ylen = synth_batch(sample_B, seconds, C, seed = 0, lengths = lengths)
	for _ in range(warmup):
		step(sig, xlen, y, ylen)
	t0 = time.perf_counter()
	for _ in range(steps):
		step(sig, xlen, y, ylen)
	dt = (time.perf_counter() - t0) / steps
	value = sample_B * seconds / dt
	return value, dt, dict(value = value, unit = 'audio-s/s', cores = torch.get_num_threads(), kind = src, sample = f'{sample_B} x {seconds:g} s utterances per step ({kind} step of {name}), {steps} steps after {warmup} warm-up, {dt:.2f} s/step; {how}')


def run_gpu_baseline(name, dev, steps = 8, warmup = 3):
	"""the UNMODIFIED reference on the same GPU through stock PyTorch kernels (cuDNN convolutions, ATen BatchNorm / hardtanh /
	ctc_loss, cuFFT frontend, torch.optim.SGD), eager, fp32 parameters with TF32 convolutions and under bf16 autocast --
	benchmark.py:116-205 method (synchronize around the timed iterations).  Library kernels: context, not a bench value."""
	if not reference_available():
		return dict(unavailable = 'reference tree not staged under baseline/_ref')
	model_name, C, B, seconds, precision, kind, lengths = WORKLOADS[name]
	out = dict(what = f'unmodified reference ({model_name}) on {torch.cuda.get_device_name(dev)}: stock PyTorch {torch.__version__} CUDA kernels, eager, {kind} step, batch {B} x {seconds:g} s', unit = 'audio-s/s')
	sig, xlen, y, ylen = [t.to(dev) for t in synth_batch(B, seconds, C, seed = 1000, lengths = lengths)]
	sig = sig.float()  # the reference casts int16 itself, but its torch.stft path wants a float signal on CUDA
	torch.backends.cudnn.benchmark = True
	for label, autocast in (('fp32_tf32_convs', False), ('bf16_autocast', True)):
		try:
			step = reference_step_fn(reference_model(model_name, C, dev), kind, C)

			def run():
				with torch.autocast('cuda', dtype = torch.bfloat16, enabled = autocast):
					return step(sig, xlen, y, ylen)
			for _ in range(warmup):
				run()
			torch.cuda.synchronize()
			t0 = time.perf_counter()
			for _ in range(steps):
				run()
			torch.cuda.synchronize()
			dt = (time.perf_counter() - t0) / steps
			out[label] = dict(value = B * seconds / dt, ms_per_step = dt * 1e3)
		except Exception as e:
			out[label] = dict(error = repr(e)[:300])
		torch.cuda.empty_cache()
	return out


# --------------------------------------------------------------------------------------------
# native arm
# --------------------------------------------------------------------------------------------
def measure(name, args, rank, world, local_rank, dev, steps, warmup, level):
	"""one workload on this rank's GPU.  level: 'full' (primary line: + e2e, cpu_baseline, clocks), 'roofline' (value +
	roofline + kernel table), 'light' (value only)"""
	from convasr_b200 import _lib, models, ops
	from oracle import oracle as O  # only for the seeded synthetic weights (outside every timed region)
	model_name, C, B, seconds, precision, kind, lengths = WORKLOADS[name]
	sweep = kind == 'sweep'
	config = dict(workload = name, lengths = LENGTHS_DESC[lengths], model = model_name, num_classes = C, batch_per_gpu = B, seconds_per_utterance = seconds, sample_rate = SAMPLE_RATE, precision = precision, kind = kind,
				step = STEP_DESC[kind], parallelism = (f'data-parallel replicas x{world} (per-layer NCCL gradient all-reduce overlapped with the backward)' if kind == 'train' else f'utterance-sharded replicas x{world} (no data-path collective)'),
				l2 = 'flushed between timed steps (256 MiB memset)', cuda_graphs = not args.no_cuda_graphs)
	frontend = models.LogFilterBankFrontend(64, SAMPLE_RATE, .02, .01, 'hann_window')
	model = getattr(models, model_name)(64, [C], frontend = frontend, dropout = 0., check_time_dim_padded = False)
	shapes = {k: tuple(v.shape) for k, v in model.state_dict().items() if not k.startswith('frontend.')}
	model.load_state_dict(O.synth_state_dict(shapes, seed = 0), strict = False)
	model = model.to(dev).set_precision(precision)
	sig, xlen, y, ylen = synth_batch(B, seconds, C, seed = 1000 + rank, lengths = lengths)
	sig_pin, xlen_pin, y_pin, ylen_pin = [t.pin_memory() for t in (sig, xlen, y, ylen)]
	sig_d, xlen_d, y_d, ylen_d = [t.to(dev) for t in (sig, xlen, y, ylen)]
	flush = torch.empty(256 << 20, dtype = torch.uint8, device = dev)
	from convasr_b200 import feed as feed_mod
	Fr = sig.shape[1] // 80 + 1
	flops_fwd, flops_grouped, t_out = conv_flops_per_step(model, B, Fr)
	first = model.backbone[0].conv[0][0]
	flops_first = 2 * B * ((Fr + 2 * first.padding[0] - first.kernel_size[0]) // first.stride[0] + 1) * first.out_channels * first.in_channels * first.kernel_size[0]
	# greedy CTC collapse tables (transcript_generators.py:8-93): blank = last class, the class before it plays the space
	sil = torch.zeros(C, dtype = torch.uint8, device = dev)
	sil[C - 1] = sil[C - 2] = 1
	ws = torch.zeros(C, dtype = torch.uint8, device = dev)
	ws[C - 2] = 1
	replicas = None

	def infer_once(s, xl, yy, yl, want_grad):
		"""eval forward (loss included through the public API) + device part of GreedyCTCGenerator + optionally the CTC gradient
		(left in the returned log-probs' .grad)"""
		with torch.no_grad():
			out = model(s, xl)
		lp = out['log_probs'][0]
		tok, frm, cnt = ops.greedy_collapse(lp._convasr_argmax, out['olen'][0], C, C - 1, C - 2, sil, ws, 10)
		lp = lp.requires_grad_(want_grad)
		nll = ops.ctc_loss(lp.permute(2, 0, 1), yy[:, 0], out['olen'][0], yl[:, 0], blank = C - 1)
		if want_grad:
			nll.sum().backward()  # grad w.r.t. the log-probs/logits only: CTC alpha || beta -> gradient scatter
		return nll, tok, cnt, lp

	if kind == 'train':
		from convasr_b200 import optimizers, training
		model.train()
		assert training.unsupported_reason(model) is None, training.unsupported_reason(model)
		net = model
		if world > 1:
			net, _ = models.distributed_data_parallel_and_autocast(model, local_rank, opt_level = 'O2' if precision == 'bf16' else None)
		# train.py defaults: SGD(momentum 0.9, weight_decay 1e-3) after clip_grad_norm_(max_norm 100) (train.py:657-662,776-779)
		train_params = [p for p in model.parameters() if p.requires_grad]
		optimizer = optimizers.SGD(train_params, lr = 1e-6, momentum = 0.9, weight_decay = 1e-3)  # native multi-tensor step
		flops = 3 * flops_fwd - flops_first  # forward + dgrad (all but the first layer) + wgrad

		def run_eager(s, xl, yy, yl):
			optimizer.zero_grad(set_to_none = True)
			out = net(s, xl, y = yy, ylen = yl)
			loss = (out['loss'] * yl[:, 0]).mean()  # train.py:754-755
			loss.backward()
			optimizer.step(max_grad_norm = 100.0)  # clip_grad_norm_ folded into the native step
			return out['loss']

		run = [run_eager]  # swapped for the CUDA-graph replay after the eager launch count

		def step_device():
			return dict(loss = run[0](sig_d, xlen_d, y_d, ylen_d))

		def step_e2e(batch):
			_, _, s, xl, yy, yl = batch  # this step's H2D was issued on the copy stream during the previous step
			return run[0](s, xl, yy, yl).detach().cpu()

		d2h = B * 4
		tensor_entries = ['cab_conv1d_fused', 'cab_conv1d_wgrad']
		kernel_label = 'conv1d_umma_kernel (forward + dgrad) + wgrad_umma_kernel'
		audio_per_step = B * seconds
	elif kind == 'infer':
		model.eval()
		flops = flops_fwd

		def step_device():
			nll, tok, cnt, lp = infer_once(sig_d, xlen_d, y_d, ylen_d, True)
			return dict(loss = nll, log_probs = lp.detach(), log_probs_grad = lp.grad, tokens = tok, token_counts = cnt)

		def step_e2e(batch):
			_, _, s, xl, yy, yl = batch
			out = model(s, xl, y = yy, ylen = yl)
			tok, frm, cnt = ops.greedy_collapse(out['log_probs'][0]._convasr_argmax, out['olen'][0], C, C - 1, C - 2, sil, ws, 10)
			return out['loss'].cpu(), tok.cpu(), cnt.cpu()

		d2h = B * 4 + B * t_out * 4 + B * 4
		tensor_entries = ['cab_conv1d_fused']
		kernel_label = 'conv1d_umma_kernel'
		audio_per_step = B * seconds
	else:  # sweep: this rank's shard of SWEEP_UTTERANCES, resident in HBM, one pass in micro-batches of B
		model.eval()
		lo, hi = (SWEEP_UTTERANCES * rank) // world, (SWEEP_UTTERANCES * (rank + 1)) // world
		n_local = hi - lo
		T = sig.shape[1]
		g = torch.Generator(device = dev).manual_seed(2000 + rank)
		shard = (torch.randn(n_local, T, generator = g, device = dev) * 3000).round().clamp(-32767, 32767).to(torch.int16)
		shard_xlen = torch.rand(n_local, generator = g, device = dev) * 0.5 + 0.5
		L = y.shape[2]
		shard_y = torch.randint(0, C - 1, (n_local, 1, L), generator = g, device = dev)
		shard_ylen = torch.randint(max(1, L // 3), L + 1, (n_local, 1), generator = g, device = dev)
		flops = flops_fwd * n_local / B

		keep = args.dump_outputs and level == 'full' and rank == 0  # per-micro-batch results are kept only for the dump

		def step_device():
			kept = []
			for a in range(0, n_local, B):
				res = infer_once(shard[a:a + B], shard_xlen[a:a + B], shard_y[a:a + B], shard_ylen[a:a + B], False)
				if keep:
					kept.append(res)
			if keep:
				return dict(loss = torch.cat([r[0] for r in kept]), token_counts = torch.cat([r[2] for r in kept]))
			return dict(loss = res[0])

		loss_host = torch.empty(n_local, dtype = torch.float32).pin_memory()
		cnt_host = torch.empty(n_local, dtype = torch.int32).pin_memory()

		def step_e2e(batches):
			# results come back through pinned buffers with asynchronous copies; one synchronisation at the end of the pass (a
			# transcription loop consumes them a micro-batch behind), so the H2D of the next micro-batch, the kernels and the D2H overlap
			a = 0
			for _, _, s, xl, yy, yl in batches:
				out = model(s, xl, y = yy, ylen = yl)
				tok, frm, cnt = ops.greedy_collapse(out['log_probs'][0]._convasr_argmax, out['olen'][0], C, C - 1, C - 2, sil, ws, 10)
				loss_host[a:a + len(s)].copy_(out['loss'], non_blocking = True)
				cnt_host[a:a + len(s)].copy_(cnt, non_blocking = True)
				a += len(s)
			torch.cuda.synchronize()
			return loss_host, cnt_host

		d2h = n_local * 8
		tensor_entries = ['cab_conv1d_fused']
		kernel_label = 'conv1d_umma_kernel'
		audio_per_step = n_local * seconds
		if level != 'full':  # one pass is ~0.4 s per GPU: as a secondary line two timed passes are enough
			steps, warmup = min(steps, 2), 1

	def barrier():
		if world > 1:
			torch.distributed.barrier()
		torch.cuda.synchronize()

	def timed(fn, n):
		"""(total ms of n calls of fn, what the last call returned)"""
		evs = []
		for _ in range(n):
			flush.zero_()
			e0, e1 = torch.cuda.Event(enable_timing = True), torch.cuda.Event(enable_timing = True)
			e0.record()
			last = fn()
			e1.record()
			evs.append((e0, e1))
		torch.cuda.synchronize()
		return sum(a.elapsed_time(b) for a, b in evs), last

	# one eager step counts this repo's kernel launches per step (graph replays bypass the counter)
	step_device()
	torch.cuda.synchronize()
	l0 = _lib.launch_count()
	step_device()
	torch.cuda.synchronize()
	launches_per_step = _lib.launch_count() - l0
	kernels, roofline = None, None
	if level in ('full', 'roofline') and not sweep:
		# per entry point: CUDA events around every C-ABI call of eager steps, on the launching stream
		n_prof = min(steps, 3)
		with _lib.trace() as tr:
			for _ in range(n_prof):
				flush.zero_()
				step_device()
		summary = tr.summary()
		peaks = measured_peaks()
		hbm_peak = peaks['hbm_gbs'] if peaks else 6550.0
		tf_peak = peaks['bf16_tflops_sustained'] if peaks else 1590.0
		abytes = algorithmic_bytes(model, B, sig.shape[1], t_out, C, kind, y.shape[2])
		kernels = []
		for entry, (calls, ms_total) in sorted(summary.items(), key = lambda kv: -kv[1][1]):
			ms_step = ms_total / n_prof
			row = dict(entry = entry, launches_per_step = calls // n_prof, ms_per_step = ms_step)
			if entry in tensor_entries:
				row.update(bound = 'tensor')
			elif entry == 'cab_grouped_conv1d':
				ach = flops_grouped / (ms_step / 1e3) / 1e12
				row.update(bound = 'fp32 fma (nominal peak, no measured figure)', achieved = ach, peak = FP32_FMA_PEAK_TFLOPS, unit = 'TFLOP/s', frac = ach / FP32_FMA_PEAK_TFLOPS)
			elif entry in abytes and ms_step > 0:
				ach = abytes[entry] / (ms_step / 1e3) / 1e9
				row.update(bound = 'hbm', algorithmic_bytes = abytes[entry], achieved = ach, peak = hbm_peak, unit = 'GB/s', frac = ach / hbm_peak)
			kernels.append(row)
		kern_ms = sum(summary[e][1] for e in tensor_entries if e in summary) / n_prof
		n_kern = sum(summary[e][0] for e in tensor_entries if e in summary) // n_prof
		achieved = flops / (kern_ms / 1e3) / 1e12
		for row in kernels:
			if row.get('bound') == 'tensor':
				row.update(note = 'see roofline: all launches of the tensor-pipe entry points together')
		roofline = dict(
			bound = 'tensor', kernel = kernel_label, achieved = achieved, peak = tf_peak, unit = 'TFLOP/s', frac = achieved / tf_peak,
			peak_source = 'MEASURED_PEAKS.json bf16_tflops_sustained (of measured)' if peaks else 'fallback 1.59 PFLOP/s (of fallback)',
			peak_burst = peaks['bf16_tflops'] if peaks else None, frac_of_burst = (achieved / peaks['bf16_tflops']) if peaks else None, traffic = NCU_DRAM_BYTES_PER_LAUNCH.get(name),
			traffic_source = 'ncu --set full dram__bytes_read.sum + dram__bytes_write.sum, mean over the launches of one step (profiles/r01_*_ncu_full.csv; round-2b capture of four dgrad launches with the folded BatchNorm-backward reduction: profiles/r02b_dgrad_fold_ncu.md -- the fold adds one read of y per dgrad launch, ~21 MB per launch averaged over the step); the kernels are L2-fed, not HBM-fed' if name in NCU_DRAM_BYTES_PER_LAUNCH else None,
			launches_per_step = n_kern, kernel_ms_per_step = kern_ms, algorithmic_gflop_per_step = flops / 1e9, mma_passes_per_flop = 3 if precision == 'fp32' else 1
		)
	if config['cuda_graphs'] and kind != 'train':
		model.enable_cuda_graphs(True)  # forward = one graph replay; greedy collapse / CTC loss / grad stay eager launches
	if config['cuda_graphs'] and kind == 'train':
		try:
			run[0] = training.GraphedTrainStep(net, optimizer, sig_d, xlen_d, y_d, ylen_d, max_grad_norm = 100.0)  # whole step = one replay
		except Exception as e:  # data-parallel capture includes the NCCL collectives; keep the eager step if a stack refuses it
			if world == 1:
				raise
			print(f'[bench] rank {rank}: CUDA-graph capture of the data-parallel step failed ({e!r}); eager step instead', file = sys.stderr)
			config['cuda_graphs'] = False
	for _ in range(warmup):
		nll = step_device()['loss']
	torch.cuda.synchronize()
	assert bool(torch.isfinite(nll).all()), 'synthetic targets must admit an alignment'
	sampler = ClockSampler(local_rank)
	if rank == 0:
		sampler.start()
	barrier()
	t_wall0 = time.time()
	ms, last = timed(step_device, steps)
	barrier()
	t_wall1 = time.time()
	clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
	result = dict(ms = ms, ms_e2e = None, steps = steps)
	if args.dump_outputs and level == 'full' and rank == 0:
		if kind == 'train':  # the step hands back the loss; its other result is the updated parameters
			last['parameters'] = torch.cat([p.detach().flatten() for p in train_params])
		if 'tokens' in last:  # the collapse leaves the entries past each row's count unwritten
			tok = last['tokens']
			last['tokens'] = torch.where(torch.arange(tok.shape[1], device = dev) < last['token_counts'][:, None], tok, 0)
		result['outputs'] = host_outputs(last)
	if roofline is not None:
		roofline['share_of_step'] = roofline['kernel_ms_per_step'] / (ms / steps)
	if kind == 'train' and world > 1:
		# data-parallel correctness, visible to the driver: after the timed steps every replica must hold bit-identical parameters
		import torch.distributed as dist
		flat = torch.cat([p.detach().flatten() for p in model.parameters() if p.requires_grad])
		digest = torch.stack([flat.double().sum(), flat.double().abs().sum(), flat.view(torch.int32).long().sum().double()])
		every = [torch.empty_like(digest) for _ in range(world)]
		dist.all_gather(every, digest)
		gnorm = optimizer.total_grad_norm.clone() if optimizer.total_grad_norm is not None else torch.zeros(1, device = dev)
		norms = [torch.empty_like(gnorm) for _ in range(world)]
		dist.all_gather(norms, gnorm)
		replicas = dict(identical = all(torch.equal(every[0], e) for e in every[1:]), param_checksum = float(every[0][1]), grad_norm_per_rank = [float(n) for n in norms], grad_norms_identical = all(torch.equal(norms[0], n) for n in norms[1:]))
		assert replicas['identical'], f'data-parallel replicas diverged: {[e.tolist() for e in every]}'
	if level == 'full' or (sweep and level != 'light'):
		# end to end through the public API with host buffers (convasr_b200/feed.py): every step uploads its own pinned host
		# batch; the copy of step i+1 is issued on a copy stream while step i computes (the timed region contains one full H2D per step)
		if sweep:
			host = [t.cpu().pin_memory() for t in (shard, shard_xlen, shard_y, shard_ylen)]

			def batches():
				return feed_mod.DeviceFeeder(((None, None) + tuple(t[a:a + B] for t in host) for a in range(0, n_local, B)), dev)
			step_e2e(batches())
			barrier()
			result['ms_e2e'] = timed(lambda: step_e2e(batches()), steps)[0]
			h2d = sum(t.numel() * t.element_size() for t in host)
		else:
			feeder = iter(feed_mod.DeviceFeeder(((None, None, sig_pin, xlen_pin, y_pin, ylen_pin) for _ in range(steps + 8)), dev))
			for _ in range(3):
				step_e2e(next(feeder))
			barrier()
			result['ms_e2e'] = timed(lambda: step_e2e(next(feeder)), steps)[0]
			h2d = sum(t.numel() * t.element_size() for t in (sig, xlen, y, ylen))
		barrier()
		result['h2d'] = h2d
	result.update(valid_fraction = float(xlen.mean()), config = config, clocks = clocks, roofline = roofline, kernels = kernels, launches = launches_per_step * steps, audio_per_step = audio_per_step,
					precision = precision, d2h = d2h, replicas = replicas, kind = kind)
	del model, flush
	torch.cuda.empty_cache()
	return result


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--gpus', type = int, default = 1)
	ap.add_argument('--steps', type = int, default = 30)
	ap.add_argument('--warmup', type = int, default = 5)
	ap.add_argument('--impl', default = 'native', choices = ['native', 'reference'])
	ap.add_argument('--workload', default = DEFAULT_WORKLOAD, choices = sorted(WORKLOADS))
	ap.add_argument('--no-cpu-baseline', action = 'store_true')
	ap.add_argument('--no-secondary', action = 'store_true')
	ap.add_argument('--no-gpu-baseline', action = 'store_true')
	ap.add_argument('--cpu-sample-batch', type = int, default = 4)
	ap.add_argument('--no-cuda-graphs', action = 'store_true')
	ap.add_argument('--dump-outputs', metavar = 'DIR', help = 'write the outputs of the last timed step as DIR/<name>.npy')
	args = ap.parse_args()
	if args.steps < 1:
		ap.error('--steps must be at least 1')
	if args.dump_outputs and args.impl != 'native':
		ap.error('--dump-outputs writes the outputs of the native timed path (--impl native)')
	model_name, C, B, seconds, precision, kind, lengths = WORKLOADS[args.workload]
	rank = int(os.environ.get('RANK', 0))
	world = int(os.environ.get('WORLD_SIZE', 1))
	local_rank = int(os.environ.get('LOCAL_RANK', 0))
	steps, warmup = args.steps, max(args.warmup, 3)

	if args.impl == 'reference':
		if rank != 0:
			return
		n_steps = max(1, min(steps, 3))
		value, sec, cpu = run_cpu_reference(args.workload, args.cpu_sample_batch, n_steps, 1)
		config = dict(workload = args.workload, lengths = LENGTHS_DESC[lengths], model = model_name, num_classes = C, batch_per_gpu = args.cpu_sample_batch, native_arm_batch_per_gpu = B, seconds_per_utterance = seconds, sample_rate = SAMPLE_RATE,
						precision = 'fp32', kind = kind, step = STEP_DESC[kind], sample = cpu['sample'])
		line = dict(
			impl = 'reference', metric = 'audio_seconds_per_second', value = value, unit = 'audio-s/s', n_gpus = args.gpus, steps = n_steps, warmup = 1, ms_per_step = sec * 1e3,
			higher_is_better = True, scaling = 'weak', vs_baseline = None, dtype = 'fp32', data = 'synthetic', config = config, cpu_baseline = cpu,
			e2e = dict(value = value, unit = 'audio-s/s', h2d_bytes_per_step = 0, d2h_bytes_per_step = 0), gpu_launches = 0
		)
		print(json.dumps(line))
		return

	# ------------------------------------------------------------------ native arm
	assert torch.cuda.is_available(), 'bench.py --impl native needs a CUDA device'
	torch.cuda.set_device(local_rank)
	dev = torch.device('cuda', local_rank)
	if world > 1:
		import torch.distributed as dist
		dist.init_process_group('nccl', device_id = dev)

	def reduce_max(vals):
		if world == 1:
			return vals
		t = torch.tensor([v if v is not None else 0.0 for v in vals], device = dev, dtype = torch.float64)
		torch.distributed.all_reduce(t, op = torch.distributed.ReduceOp.MAX)
		return t.tolist()

	cpu_baseline = None
	if rank == 0 and world == 1 and not args.no_cpu_baseline:
		_, _, cpu_baseline = run_cpu_reference(args.workload, args.cpu_sample_batch, 3, 1)
	r = measure(args.workload, args, rank, world, local_rank, dev, steps, warmup, 'full')
	if args.dump_outputs and rank == 0:
		import numpy as np
		os.makedirs(args.dump_outputs, exist_ok = True)
		for name, a in r['outputs'].items():
			np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
	ms, ms_e2e = reduce_max([r['ms'], r['ms_e2e']])
	also = None
	if not args.no_secondary and args.workload == DEFAULT_WORKLOAD:
		also = {}
		names = SECONDARY_WORKLOADS + (SINGLE_GPU_WORKLOADS if world == 1 else [])
		for name2 in names:
			level = 'roofline' if (world == 1 or WORKLOADS[name2][5] == 'sweep') else 'light'
			r2 = measure(name2, args, rank, world, local_rank, dev, steps, warmup, level)
			ms2, ms2_e2e = reduce_max([r2['ms'], r2['ms_e2e']])
			entry = dict(value = r2['audio_per_step'] * world * r2['steps'] / (ms2 / 1e3), unit = 'audio-s/s', ms_per_step = ms2 / r2['steps'], steps = r2['steps'], lengths = r2['config']['lengths'], valid_audio_fraction = r2['valid_fraction'],
						step = r2['config']['step'], precision = r2['precision'], cuda_graphs = r2['config']['cuda_graphs'], gpu_launches = r2['launches'], clocks = r2['clocks'], roofline = r2['roofline'], kernels = r2['kernels'])
			if r2['ms_e2e'] is not None:
				entry['e2e'] = dict(value = r2['audio_per_step'] * world * r2['steps'] / (ms2_e2e / 1e3), unit = 'audio-s/s', ms_per_step = ms2_e2e / r2['steps'], h2d_bytes_per_step = r2.get('h2d'), d2h_bytes_per_step = r2['d2h'])
			if name2 == 'wav2letter_char_fwd_ctc_B8x10s_fp32' and rank == 0 and not args.no_cpu_baseline:
				# BASELINE.md section 4: config C1 forward + greedy decode is the reference's own CPU-runnable case
				_, _, entry['cpu_baseline'] = run_cpu_reference(name2, 8, 3, 1)
			also[name2] = entry
		if world == 1 and not args.no_gpu_baseline:
			also['gpu_baseline'] = run_gpu_baseline(args.workload, dev)
	if rank == 0:
		audio_s = r['audio_per_step'] * world
		line = dict(
			metric = 'audio_seconds_per_second', value = audio_s * r['steps'] / (ms / 1e3), unit = 'audio-s/s', n_gpus = world, steps = r['steps'], warmup = warmup, ms_per_step = ms / r['steps'],
			higher_is_better = True, scaling = 'weak', vs_baseline = None, dtype = 'bf16' if r['precision'] == 'bf16' else 'bf16x3 (split-bf16, fp32 accumulate)', data = 'synthetic',
			config = r['config'],
			e2e = dict(value = audio_s * r['steps'] / (ms_e2e / 1e3), unit = 'audio-s/s', ms_per_step = ms_e2e / r['steps'], h2d_bytes_per_step = r.get('h2d'), d2h_bytes_per_step = r['d2h']),
			gpu_launches = r['launches'], roofline = r['roofline'], kernels = r['kernels'], cpu_baseline = cpu_baseline, clocks = r['clocks'], also = also
		)
		if r['replicas'] is not None:
			line['replicas_identical'] = r['replicas']['identical']
			line['replicas'] = r['replicas']
		print(json.dumps(line))
	if world > 1:
		torch.distributed.destroy_process_group()


if __name__ == '__main__':
	main()
