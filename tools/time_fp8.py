"""bf16 vs fp8 inference tier, alternating in one process: ms per forward (conv stack + decoder, frontend included) and
per-launch GEMM times (CUDA events around every cab_conv1d_fused / cab_conv1d_fused_fp8 call) with achieved FLOP/s.
The card name, power limit and max SM clock are read in the same call.

Shapes: C1 Wav2Letter B8 x 10 s; a C5 micro-batch Wav2Letter B256 x 10 s; C3 JasperNetSeparable B256 x 20 s; C4
Wav2Letter BPE-5000 B64 x 15 s.  Random-init weights, full-length utterances (xlen = 1), int16 signal input.
FLOPs per launch = 2 * B * T_out * C_out_alloc * sum over sources of taps * C_in_alloc (what the tensor cores execute,
padding channels included).

  python tools/time_fp8.py --out profiles/r05_time_fp8.log
"""
import argparse
import copy
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

CONFIGS = [
	('C1', 'Wav2Letter', 38, 8, 10.0),
	('C5 micro-batch', 'Wav2Letter', 38, 256, 10.0),
	('C3', 'JasperNetSeparable', 38, 256, 20.0),
	('C4', 'Wav2Letter', 5000, 64, 15.0),
]
GEMM_ENTRIES = ['cab_conv1d_fused', 'cab_conv1d_fused_fp8']


def card_info():
	name = torch.cuda.get_device_name(0)
	try:
		q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output = True, text = True, timeout = 30).stdout.strip().splitlines()[0]
	except Exception as e:  # noqa: BLE001
		q = f'nvidia-smi query failed: {e}'
	return f'{name}; power limit, max SM clock: {q}'


def launch_geometry(plan, F):
	"""(launch, T_out, FLOPs) in execution order, for a batch of one utterance"""
	out, T = [], F
	for launches in plan.blocks:
		for L in launches:
			if L.stride2 is not None:
				k, pad = L.stride2
				T = (T + 2 * pad - (k - 1) - 1) // 2 + 1
			else:
				T = T + L.dT
			out.append((L, T))
	T_body = T
	for chain in plan.heads:
		T = T_body
		for L in chain:
			T = T + L.dT
			out.append((L, T))
	res = []
	for L, T in out:
		rows = L.C_alloc if L.epilogue == 0 else L.C_out
		k_sum = sum(g.taps * g.c_in_alloc for g in L.gemms)
		res.append((L, T, 2.0 * T * rows * k_sum))
	return res


def time_forward(m, sig, xlen, n):
	e0, e1 = torch.cuda.Event(enable_timing = True), torch.cuda.Event(enable_timing = True)
	with torch.no_grad():
		e0.record()
		for _ in range(n):
			m(sig, xlen)
		e1.record()
	torch.cuda.synchronize()
	return e0.elapsed_time(e1) / n


def gemm_times(m, sig, xlen, passes):
	from convasr_b200 import _lib
	per = None
	for _ in range(passes):
		with torch.no_grad(), _lib.trace(GEMM_ENTRIES) as t:
			m(sig, xlen)
		torch.cuda.synchronize()
		ms = [e0.elapsed_time(e1) for _, e0, e1 in t.events]
		per = [[v] for v in ms] if per is None else [p + [v] for p, v in zip(per, ms)]
	return [statistics.median(p) for p in per]


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--out', default = None)
	ap.add_argument('--iters', type = int, default = 10)
	ap.add_argument('--rounds', type = int, default = 3)
	ap.add_argument('--configs', default = None, help = 'comma-separated subset of the labels (C1, C5, C3, C4)')
	args = ap.parse_args()
	if not torch.cuda.is_available():
		raise SystemExit('time_fp8.py needs a CUDA device')
	from convasr_b200 import models
	dev = torch.device('cuda:0')
	lines = [f'# tools/time_fp8.py on {card_info()}', f'# {args.rounds} alternating rounds of {args.iters} forwards per tier; ms per forward; GEMM = conv launches only']

	def emit(s):
		print(s, flush = True)
		lines.append(s)

	for label, name, C, B, secs in CONFIGS:
		if args.configs and label.split()[0] not in args.configs.split(','):
			continue
		torch.manual_seed(0)
		fe = models.LogFilterBankFrontend(64, 8000, .02, .01, 'hann_window')
		m16 = getattr(models, name)(64, [C], frontend = fe, dropout = 0., check_time_dim_padded = False).to(dev).eval().set_precision('bf16')
		m8 = copy.deepcopy(m16).set_precision('fp8')
		g = torch.Generator().manual_seed(1)
		T = int(secs * 8000)
		sig = (torch.randn(B, T, generator = g) * 3000).round().clamp(-32767, 32767).to(torch.int16).to(dev)
		xlen = torch.ones(B, device = dev)
		m8.calibrate_fp8(sig, xlen)
		for m in (m16, m8):
			time_forward(m, sig, xlen, 2)
		t16, t8 = [], []
		for _ in range(args.rounds):
			t16.append(time_forward(m16, sig, xlen, args.iters))
			t8.append(time_forward(m8, sig, xlen, args.iters))
		a16, a8 = statistics.median(t16), statistics.median(t8)
		emit(f'\n## {label}: {name} C={C}, B={B} x {secs:g} s')
		emit(f'forward ms: bf16 {", ".join(f"{v:.3f}" for v in t16)} | fp8 {", ".join(f"{v:.3f}" for v in t8)} | median speed-up {a16 / a8:.3f}x; audio-s/s bf16 {B * secs / a16 * 1e3:.0f}, fp8 {B * secs / a8 * 1e3:.0f}')
		F = T // 80 + 1  # frames of the log-mel frontend (hop 80)
		geo16 = launch_geometry(m16._get_plan(), F)
		geo8 = launch_geometry(m8._get_plan(), F)
		g16 = gemm_times(m16, sig, xlen, 5)
		g8 = gemm_times(m8, sig, xlen, 5)
		assert len(g16) == len(geo16) and len(g8) == len(geo8), (len(g16), len(geo16), len(g8), len(geo8))
		emit('launch | T_out x C_out | bf16 ms, TFLOP/s | fp8 ms, TFLOP/s | speed-up')
		tot16 = tot8 = fl16 = fl8 = 0.0
		for i, ((L, T_out, f16), (L8, _, f8), ms16, ms8) in enumerate(zip(geo16, geo8, g16, g8)):
			f16 *= B
			f8 *= B
			tot16 += ms16
			tot8 += ms8
			fl16 += f16
			fl8 += f8
			slower = '  <- slower in fp8' if ms8 > ms16 else ''
			emit(f'{i:2d} {str(L.key):22s} | {T_out:5d} x {L.C_out:5d} | {ms16:8.4f}, {f16 / ms16 / 1e9:7.1f} | {ms8:8.4f}, {f8 / ms8 / 1e9:7.1f} | {ms16 / ms8:5.2f}x{slower}')
		emit(f'GEMM total: bf16 {tot16:.3f} ms ({fl16 / tot16 / 1e9:.0f} TFLOP/s), fp8 {tot8:.3f} ms ({fl8 / tot8 / 1e9:.0f} TFLOP/s), speed-up {tot16 / tot8:.3f}x')
		del m16, m8
		torch.cuda.empty_cache()
	if args.out:
		os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok = True)
		with open(args.out, 'w') as f:
			f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
	main()
