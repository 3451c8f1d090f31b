"""Time the streaming CTC prefix beam search (cab_ctc_beam_search_stream) against the one-shot search, with CUDA events.

  python tools/time_beam_search_stream.py

Shape C2: B = 80 streams, T = 751 frames, C = 38, W = 100, N = 40, topk = 1, peaked posteriors (a planted label path
every 6th frame, scale 6, over randn).  For chunks of 25, 50 and 100 frames (0.5 / 1 / 2 s at 20 ms per frame) the 80
streams are fed from their first frame to the last (new states each pass, the last chunk is_eos), alternating with one
one-shot call on the whole 751 frames, 3 rounds each: ms per streaming call, µs per frame (the pass over the 751 frames
divided by 751: the streams run in parallel, their frames in sequence) and ms per one-shot call.  Acoustic and with a
seeded synthetic 3-gram LM (2 000 words, tests/beam_lm_oracle.py write_synthetic_arpa, alpha 0.8, beta 1.5).  Then the
cost of a partial result 10 minutes into the streams (30 000 frames fed in 50-frame chunks, the 751 frames cycled): a
call with 0 new frames (prune of nothing, state load / store, the back-trace over 30 000 frames of nodes) and a 50-frame
call, and torch.profiler's per-kernel times of the latter.  The timings include the host work of each call (descriptor
set-up, workspace and output allocation from torch's caching allocator).  The device name, power limit and max SM clock
are printed in the same run.  Needs a CUDA device.
"""
import os
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import beam_lm_oracle as LO  # noqa: E402
from convasr_b200 import ops  # noqa: E402
from convasr_b200.lm import NGramLM  # noqa: E402
from time_beam_search import device_line, posteriors  # noqa: E402
from time_beam_search_lm import CHARS, kernel_times  # noqa: E402


def event_ms(fn):
	e0, e1 = torch.cuda.Event(enable_timing = True), torch.cuda.Event(enable_timing = True)
	torch.cuda.synchronize()
	e0.record()
	fn()
	e1.record()
	torch.cuda.synchronize()
	return e0.elapsed_time(e1)


def stream_pass(lp, chunk, kw):
	B, _, T = lp.shape
	states = [ops.BeamStreamState() for _ in range(B)]
	calls = 0
	for t in range(0, T, chunk):
		ops.ctc_beam_search_stream(lp[:, :, t:t + chunk], states, t + chunk >= T, **kw)
		calls += 1
	return calls


def main():
	assert torch.cuda.is_available(), 'needs a CUDA device'
	print(device_line(), flush = True)
	B, C, T, W, N = 80, 38, 751, 100, 40
	lp = posteriors(B, C, T, 'peaked', 'bct')
	olen = torch.full((B, ), T, device = 'cuda', dtype = torch.int64)
	with tempfile.TemporaryDirectory() as tmp:
		path = os.path.join(tmp, 'small.arpa')
		LO.write_synthetic_arpa(path, LO.random_words(2000, seed = 1, lengths = (2, 9)), seed = 2, n_bigrams = 20000, n_trigrams = 20000)
		lm = NGramLM.from_arpa(path, CHARS)
	for label, extra in (('acoustic', {}), ('LM', dict(lm = lm, alpha = 0.8, beta = 1.5))):
		kw = dict(beam_width = W, cutoff_top_n = N, **extra)
		one_shot = lambda: ops.ctc_beam_search(lp, olen, **kw)  # noqa: E731
		for chunk in (25, 50, 100):
			stream_pass(lp, chunk, kw)  # warm-up
			one_shot()
			s_ms, o_ms = [], []
			for _ in range(3):
				calls = [0]
				s_ms.append(event_ms(lambda: calls.__setitem__(0, stream_pass(lp, chunk, kw))))
				o_ms.append(event_ms(one_shot))
			s, o = min(s_ms), min(o_ms)
			print(f'C2 B={B} T={T} W={W} N={N} {label:8s} chunk {chunk:3d}: stream {s:8.3f} ms per pass = {s / calls[0]:6.3f} ms per call '
					f'({calls[0]} calls), {1000 * s / T:6.2f} us/frame | one-shot {o:7.3f} ms, {1000 * o / T:6.2f} us/frame | stream / one-shot '
					f'{s / o:5.2f} (rounds: stream {", ".join(f"{x:.3f}" for x in s_ms)}; one-shot {", ".join(f"{x:.3f}" for x in o_ms)})', flush = True)
		# 10 minutes into the streams
		states = [ops.BeamStreamState(capacity = 30500) for _ in range(B)]
		t = 0
		while t < 30000:
			ops.ctc_beam_search_stream(lp[:, :, t % T:t % T + 50] if t % T + 50 <= T else lp[:, :, :50], states, False, **kw)
			t += 50
		torch.cuda.synchronize()
		t_start = states[0].t0
		empty = lp[:, :, :0]
		chunk50 = lp[:, :, :50]
		zero = min(event_ms(lambda: ops.ctc_beam_search_stream(empty, states, False, **kw)) for _ in range(5))
		fifty = min(event_ms(lambda: ops.ctc_beam_search_stream(chunk50, states, False, **kw)) for _ in range(5))
		k = kernel_times(lambda: ops.ctc_beam_search_stream(chunk50, states, False, **kw))
		print(f'  {label}: 10 min into the streams ({t_start} frames consumed when the timed calls start): call with 0 new frames '
				f'{zero:.3f} ms, with 50 frames {fifty:.3f} ms; profile of 50-frame calls: '
				+ ', '.join(f'{n} {v:.3f} ms ({c} launches)' for n, (v, c) in sorted(k.items())), flush = True)
		del states


if __name__ == '__main__':
	main()
