"""Drop-in replacement for the reference's `ctc` module (ctc.py:6-75): forced alignment on the
GPU (convasr_b200/csrc/ctc.cu).  Targets of up to 2047 labels run on one CTA per utterance
(ctc_align_kernel); longer ones, up to 65535 labels (hour-long recordings), on a thread-block
cluster per utterance (ctc_align_cluster_kernel + ctc_align_backtrace_kernel).

All of the reference's behaviours are reproduced, including the batch-coupled ones (recursion
over all T frames of the padded batch, terminal state read after the last global frame,
back-trace from input_length-1, finite "zero", stay-preferred argmax ties) -- SURVEY.md A12 -- and
its fp16 mode: on fp16 log_probs every operation of the recursion rounds to fp16 ("zero" = finfo(float16).min).
`pack_backpointers` only changes the reference's memory format, never its result, and is ignored
here: the short-target kernel keeps one byte per back-pointer, the cluster kernel always packs
four 2-bit back-pointers per byte (B * T * ceil((2L+1)/4) bytes).
"""
import torch

from . import ops


def alignment(
	log_probs, targets, input_lengths, target_lengths, blank: int = 0, pack_backpointers: bool = False,
	finfo_min_fp32: float = torch.finfo(torch.float32).min, finfo_min_fp16: float = torch.finfo(torch.float16).min
):
	"""log_probs [T, B, C] (any strides), targets [B, L] -> int64 [B, L]: for every target label the
	last frame index at which the best path sits in it (zeros past target_length)."""
	if log_probs.dtype not in (torch.float32, torch.float16):
		raise NotImplementedError(f'convasr_b200.ctc.alignment: {log_probs.dtype} log_probs (the reference handles float32 and float16, ctc.py:29)')
	return ops.ctc_alignment(log_probs, targets, input_lengths, target_lengths, blank = blank)


def ctc_loss(log_probs, targets, input_lengths, target_lengths, blank = 0, reduction = 'none'):
	"""torch.nn.functional.ctc_loss(..., zero_infinity=False) as called at models.py:323."""
	nll = ops.ctc_loss(log_probs, targets, input_lengths, target_lengths, blank = blank)
	if reduction == 'none':
		return nll
	if reduction == 'sum':
		return nll.sum()
	if reduction == 'mean':
		tl = torch.as_tensor(target_lengths, device = nll.device).clamp(min = 1).to(nll.dtype)
		return (nll / tl).mean()
	raise ValueError(reduction)
