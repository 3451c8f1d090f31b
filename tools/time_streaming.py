"""Time streaming acoustic-model inference (convasr_b200.streaming.StreamingModel) with CUDA events.

  python tools/time_streaming.py [--minutes 10] [--out profiles/r12_time_streaming.log]

Shape C2: B = 80 streams of Wav2Letter-char (66.5 M parameters, 38 classes, 64 mels, 8 kHz), bf16 tier, random int16
audio.  For chunks of 0.25, 0.5 and 1 s the 80 streams are fed from their start for `--minutes` of audio; the time
of each call (host work included: scheduling, descriptor uploads, allocation from torch's caching allocator; ended by
a device synchronise) is averaged over 20 calls around 1 k, 10 k and 30 k output frames into the streams.  Then 15 s
of audio of the 80 streams streamed from the start (the last chunk is_eos) against one one-shot forward over the same
15 s (`model(signal, normalisation = fixed)`), and, over one further streamed pass, the share of the device time of a
call that goes to launches computing fewer than 128 new rows (CUDA events around every step).  The device name,
power limit and max SM clock are printed in the same run.  Needs a CUDA device.
"""
import argparse
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from convasr_b200 import models, streaming  # noqa: E402
from time_beam_search import device_line  # noqa: E402

B, SR, HOP = 80, 8000, 80


def model():
	m = models.Wav2Letter(64, [38], frontend = models.LogFilterBankFrontend(64, SR, .02, .01, 'hann_window'), dropout = 0., check_time_dim_padded = False)
	return m.cuda().eval().set_precision('bf16')


def audio(n, seed):
	g = torch.Generator(device = 'cuda').manual_seed(seed)
	return (torch.randn(B, n, device = 'cuda', generator = g) * 3000).round().clamp(-32767, 32767).to(torch.int16)


class Timed(streaming.StreamingModel):
	"""records (new rows, device ms) of every step of a call"""

	def _run_step(self, s, states, o0, n_out, plan, copies, dev):
		if self.events is None:
			return super()._run_step(s, states, o0, n_out, plan, copies, dev)
		e0, e1 = torch.cuda.Event(enable_timing = True), torch.cuda.Event(enable_timing = True)
		e0.record()
		r = super()._run_step(s, states, o0, n_out, plan, copies, dev)
		e1.record()
		self.events.append((n_out, e0, e1))
		return r


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument('--minutes', type = float, default = 10.0)
	ap.add_argument('--out', default = None)
	args = ap.parse_args()
	lines = [device_line()]

	def log(s):
		print(s, flush = True)
		lines.append(s)

	m = model()
	sm = Timed(m)
	sm.events = None
	norm = streaming.estimate_normalisation(m, audio(2 * SR, 1))
	rows = [norm[i] for i in range(B)]
	log(f'Wav2Letter bf16, B = {B} streams, lookahead {sm.lookahead_frames} output frames ({sm.lookahead_frames * 20} ms)')
	base = audio(60 * SR, 2)  # one minute of audio, cycled
	for sec in (0.25, 0.5, 1.0):
		n = int(sec * SR)
		states = [sm.new_state(r) for r in rows]
		calls = int(args.minutes * 60 / sec)
		marks = {1000: [], 10000: [], 30000: []}
		frames = 0
		for c in range(calls):
			o = (c * n) % base.shape[1]
			chunks = [base[b, o:o + n] for b in range(B)]
			torch.cuda.synchronize()
			t0 = time.perf_counter()
			out = sm.forward(chunks, states, [False] * B)
			torch.cuda.synchronize()
			ms = (time.perf_counter() - t0) * 1e3
			frames += int(out['lengths'][0])
			for k, v in marks.items():
				if abs(frames - k) <= 10 * sec * 50 and len(v) < 20:
					v.append(ms)
		got = ', '.join(f'{k // 1000} k: {sum(v) / len(v):.2f} ms' if v else f'{k // 1000} k: not reached' for k, v in marks.items())
		log(f'chunk {sec:.2f} s ({n} samples x {B} streams): ms per call at {got}')
	sig = audio(15 * SR, 3)
	fixed = models.FixedNormalisation(norm.signal_scale, norm.mean, norm.invstd)
	with torch.no_grad():
		m(sig, normalisation = fixed)
	torch.cuda.synchronize()
	reps = 3
	t0 = time.perf_counter()
	for _ in range(reps):
		with torch.no_grad():
			m(sig, normalisation = fixed)
	torch.cuda.synchronize()
	one_shot = (time.perf_counter() - t0) * 1e3 / reps
	for sec in (0.25, 0.5, 1.0):
		n = int(sec * SR)
		calls = int(15 / sec)
		for timed_pass in (False, True):
			states = [sm.new_state(r) for r in rows]
			sm.events = [] if timed_pass else None
			torch.cuda.synchronize()
			t0 = time.perf_counter()
			for c in range(calls):
				sm.forward([sig[b, c * n:(c + 1) * n] for b in range(B)], states, [c == calls - 1] * B)
			torch.cuda.synchronize()
			total = (time.perf_counter() - t0) * 1e3
			if not timed_pass:
				log(f'chunk {sec:.2f} s: 15 s streamed in {calls} calls = {total:.1f} ms total; one-shot forward over the same 15 s = {one_shot:.1f} ms; ratio {total / one_shot:.2f}')
			else:
				small = sum(e0.elapsed_time(e1) for r, e0, e1 in sm.events if r < 128)
				every = sum(e0.elapsed_time(e1) for r, e0, e1 in sm.events)
				log(f'chunk {sec:.2f} s: launches with < 128 new rows take {small:.1f} of {every:.1f} ms of step time ({100 * small / every:.0f} %)')
		sm.events = None
	if args.out:
		with open(args.out, 'w') as f:
			f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
	main()
