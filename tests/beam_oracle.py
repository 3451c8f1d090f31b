"""Float64 restatement of the CTC prefix beam search of csrc/beam.cu (decoders.BeamSearchDecoder), for the tests.

Same rules as the kernels: per frame the top N = min(cutoff_top_n, C) classes by log-prob (ties -> lower class id), cut
by cutoff_prob (running sum of probabilities, most probable first, the class that crosses it kept; summed in fp32 as the
kernel does), kept in ascending class order.  Candidate q = i * (n + 1) + s of source beam i: s = 0 keeps the prefix,
s = 1 + k extends it by the k-th kept class; an extension that equals an existing beam is merged into that beam's
p_nonblank; probability zero is not a candidate; the top W by log(p_blank + p_nonblank), ties to the lower q.
Vectorised per frame: B = 8 x 751 frames takes seconds.
"""
import math

import numpy as np

NEG = -math.inf


def prune(lp, cutoff_top_n, cutoff_prob = 1.0):
	"""lp [T, C] -> per frame (classes int64 ascending, log-probs float64) of the classes the search considers"""
	lp = np.asarray(lp, dtype = np.float64)
	T, C = lp.shape
	N = min(int(cutoff_top_n), C)
	ids = np.broadcast_to(np.arange(C), lp.shape)
	top = np.lexsort((ids, -lp), axis = -1)[:, :N]  # descending value, ties -> lower class id
	vals = np.take_along_axis(lp, top, axis = 1)
	out = []
	for t in range(T):
		n = N
		if cutoff_prob < 1.0:
			cum = np.cumsum(np.exp(vals[t]).astype(np.float32), dtype = np.float32)
			hit = np.nonzero(cum >= np.float32(cutoff_prob))[0]
			n = int(hit[0]) + 1 if hit.size else N
		keep = np.sort(top[t, :n])
		out.append((keep, lp[t, keep]))
	return out


def ctc_prefix_beam_search(log_probs, output_lengths = None, beam_width = 100, cutoff_top_n = 40, cutoff_prob = 1.0, blank = None):
	"""log_probs [B, C, T] (numpy or torch) -> per utterance the surviving beams best first, each (tokens tuple, emission
	frames tuple, score = log(p_blank + p_nonblank))"""
	lp_all = np.asarray(log_probs, dtype = np.float64)
	B, C, T = lp_all.shape
	blank = C - 1 if blank is None else int(blank)
	W = int(beam_width)
	results = []
	for b in range(B):
		olen = T if output_lengths is None else max(0, min(T, int(output_lengths[b])))
		frames_pruned = prune(lp_all[b, :, :olen].T, cutoff_top_n, cutoff_prob)
		prefixes, emitted = [()], [()]
		pb, pnb, last = np.array([0.0]), np.array([NEG]), np.array([-1])
		for t in range(olen):
			cls, vals = frames_pruned[t]
			n, nb = len(cls), len(prefixes)
			where = {int(c): k for k, c in enumerate(cls)}
			kb = where.get(blank)
			tot = np.logaddexp(pb, pnb)
			kpb = tot + vals[kb] if kb is not None else np.full(nb, NEG)
			kl = np.array([where.get(int(c), -1) for c in last])
			kpnb = np.where(kl >= 0, pnb + vals[np.maximum(kl, 0)], NEG)
			merged = np.zeros((nb, n), dtype = bool)
			rank = {p: i for i, p in enumerate(prefixes)}
			for j in range(nb):
				if kl[j] < 0 or not prefixes[j]:
					continue
				p = rank.get(prefixes[j][:-1])
				if p is None:
					continue
				e = (pb[p] if last[p] == last[j] else tot[p]) + vals[kl[j]]
				kpnb[j] = np.logaddexp(kpnb[j], e)
				merged[p, kl[j]] = True
			ext = np.where(cls[None, :] == last[:, None], pb[:, None], tot[:, None]) + vals[None, :]
			ext[:, cls == blank] = NEG
			ext[merged] = NEG
			score = np.concatenate([np.logaddexp(kpb, kpnb)[:, None], ext], axis = 1).reshape(-1)
			q = np.nonzero(score > NEG)[0]
			q = q[np.lexsort((q, -score[q]))][:W]
			i, s = np.divmod(q, n + 1)
			new_pre, new_emit = [], []
			for ii, ss in zip(i.tolist(), s.tolist()):
				if ss == 0:
					new_pre.append(prefixes[ii])
					new_emit.append(emitted[ii])
				else:
					new_pre.append(prefixes[ii] + (int(cls[ss - 1]), ))
					new_emit.append(emitted[ii] + (t, ))
			keep = s == 0
			k = np.maximum(s - 1, 0)
			pb = np.where(keep, kpb[i], NEG)
			pnb = np.where(keep, kpnb[i], ext[i, k])
			last = np.where(keep, last[i], cls[k])
			prefixes, emitted = new_pre, new_emit
			if not prefixes:
				break
		final = np.logaddexp(pb, pnb) if prefixes else np.array([])
		results.append([(p, e, float(sc)) for p, e, sc in zip(prefixes, emitted, final)])
	return results


def labelings_by_probability(lp, blank, ctc_loss_np):
	"""Every labeling of nonzero CTC probability for one utterance lp [C, T], ranked by exp(-nll) (exhaustive; tiny T, C
	only).  ctc_loss_np: the oracle's float64 CTC."""
	C, T = lp.shape
	symbols = [c for c in range(C) if c != blank]
	out = [((), float(np.sum(lp[blank])))]
	frontier = [()]
	for _ in range(T):
		frontier = [p + (c, ) for p in frontier for c in symbols]
		for p in frontier:
			nll, _ = ctc_loss_np(lp.T[:, None, :], [list(p)], [T], [len(p)], blank)
			if math.isfinite(nll[0]):
				out.append((p, -float(nll[0])))
	out.sort(key = lambda x: -x[1])
	return out


def assert_nbest_equal(got, ref, tol, k = None):
	"""got, ref: lists of (tokens, score) best first.  The first k ranks (all, and then the same length, when k is None)
	hold the same hypotheses, except that two whose reference scores are within tol of each other may trade places; every
	score is within tol (relative, for |score| > 1) of the reference score of its hypothesis."""
	if k is None:
		assert len(got) == len(ref), (len(got), len(ref))
	ref_score = {tuple(h): s for h, s in ref}
	for r, ((h, s), (hr, sr)) in enumerate(list(zip(got, ref))[:k]):
		h = tuple(h)
		assert h in ref_score, (r, h)
		scale = max(1.0, abs(sr))
		assert abs(ref_score[h] - sr) <= tol * scale, (r, h, hr, ref_score[h], sr)
		assert abs(s - ref_score[h]) <= tol * scale, (r, h, s, ref_score[h])
