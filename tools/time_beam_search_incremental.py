"""Time the incremental streaming beam search (cab_ctc_beam_search_stream_incremental) against the full-history streaming
search (cab_ctc_beam_search_stream) as a stream grows, with CUDA events.

  python tools/time_beam_search_incremental.py

Shape C2: B = 80 streams, C = 38, W = 100, N = 40, topk = 1, fed in 50-frame chunks (1 s at 20 ms per frame) up to
30 000 frames (10 minutes), the 751 frames of tools/time_beam_search.py's posteriors cycled.  Each chunk goes to a
full-history state set and to an incremental state set in one process, one call after the other, each call timed on
its own (host work included: descriptor set-up, allocations from torch's caching allocator and, for the incremental
call, its copy of the commit nodes to the host).  Reported around 1 000, 10 000 and 30 000 frames (the median of the
calls within 250 frames of the mark): ms per call of each, the node-table window of the incremental states (frames
held, capacity) and how far the commit node lags (frames consumed minus the commit node's frame, mean and max over
the streams).  Then torch.profiler's per-kernel times of 50-frame calls of both, in a separate pass.  The top
hypothesis of both state sets is compared after the timed calls.  Peaked posteriors (a planted label every 6th frame, scale 6)
and diffuse ones (randn), acoustic and with the seeded 2 000-word 3-gram LM of the other timing scripts (alpha 0.8,
beta 1.5).  The device name, power limit and max SM clock are printed in the same run.  Needs a CUDA device.
"""
import os
import statistics
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
from time_beam_search_stream import event_ms  # noqa: E402

TOTAL, CHUNK, MARKS = 30000, 50, (1000, 10000, 30000)


def chunk_at(lp, t):
	T = lp.shape[2]
	return lp[:, :, t % T:t % T + CHUNK] if t % T + CHUNK <= T else lp[:, :, :CHUNK]


def run(label, lp, kw):
	B, W = lp.shape[0], kw['beam_width']
	full = [ops.BeamStreamState(capacity = TOTAL + 500) for _ in range(B)]
	inc = [ops.BeamStreamState() for _ in range(B)]
	finals = [[] for _ in range(B)]
	rec = []  # (frames consumed, full ms, incremental ms, window frames, capacity, lag per stream)
	t = 0
	while t < TOTAL:
		x = chunk_at(lp, t)
		f_ms = event_ms(lambda: ops.ctc_beam_search_stream(x, full, False, **kw))
		out = []
		i_ms = event_ms(lambda: out.extend(ops.ctc_beam_search_stream_incremental(x, inc, False, **kw)))
		t += CHUNK
		ft, fl = out[0].cpu(), out[2].tolist()
		for b in range(B):
			finals[b] += ft[b, :fl[b]].tolist()
		lags = [s.t0 - (s.commit // W if s.commit >= 0 else -1) for s in inc]
		rec.append((t, f_ms, i_ms, max(s.t0 for s in inc), max(s.capacity for s in inc), lags))
	for m in MARKS:
		near = [r for r in rec if abs(r[0] - m) <= 250]
		lag = [x for r in near for x in r[5]]
		print(f'  {label:18s} ~{m:5d} frames ({len(near)} calls): full-history {statistics.median(r[1] for r in near):6.3f} ms, incremental '
				f'{statistics.median(r[2] for r in near):6.3f} ms per 50-frame call | window up to {max(r[3] for r in near)} frames, capacity '
				f'{max(r[4] for r in near)} | commit lag mean {statistics.mean(lag):6.1f} frames, max {max(lag)}', flush = True)
	tok, _, ln, _ = ops.ctc_beam_search_stream(lp[:, :, :0], full, False, **kw)
	_, _, _, tail, _, tl, _ = ops.ctc_beam_search_stream_incremental(lp[:, :, :0], inc, False, **kw)
	tok, ln, tail, tl = tok.cpu(), ln.cpu(), tail.cpu(), tl.cpu()
	same = sum(finals[b] + tail[b, 0, :tl[b, 0]].tolist() == tok[b, 0, :ln[b, 0]].tolist() for b in range(B))
	print(f'  {label:18s} top hypothesis after {full[0].t0} frames: incremental (final + tail) equals full-history in {same} / {B} streams '
			f'(mean length {statistics.mean(ln[:, 0].tolist()):.0f} tokens)', flush = True)
	k_inc = kernel_times(lambda: ops.ctc_beam_search_stream_incremental(chunk_at(lp, 0), inc, False, **kw))
	k_full = kernel_times(lambda: ops.ctc_beam_search_stream(chunk_at(lp, 0), full, False, **kw))
	for name, k in (('incremental', k_inc), ('full-history', k_full)):
		print(f'  {label:18s} profile of {name} 50-frame calls at {full[0].t0} frames: '
				+ ', '.join(f'{n} {v:.3f} ms ({c} launches)' for n, (v, c) in sorted(k.items())), flush = True)


def main():
	assert torch.cuda.is_available(), 'needs a CUDA device'
	print(device_line(), flush = True)
	B, C, T, W, N = 80, 38, 751, 100, 40
	with tempfile.TemporaryDirectory() as tmp:
		path = os.path.join(tmp, 'small.arpa')
		LO.write_synthetic_arpa(path, LO.random_words(2000, seed = 1, lengths = (2, 9)), seed = 2, n_bigrams = 20000, n_trigrams = 20000)
		lm = NGramLM.from_arpa(path, CHARS)
	print(f'C2 B={B} C={C} W={W} N={N} topk=1, {CHUNK}-frame chunks to {TOTAL} frames', flush = True)
	for kind in ('peaked', 'diffuse'):
		lp = posteriors(B, C, T, kind, 'bct')
		for name, extra in (('acoustic', {}), ('LM', dict(lm = lm, alpha = 0.8, beta = 1.5))):
			run(f'{kind} {name}', lp, dict(beam_width = W, cutoff_top_n = N, **extra))


if __name__ == '__main__':
	main()
