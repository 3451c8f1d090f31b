"""ctypes binding of libconvasr_b200.so (the C ABI declared in include/convasr_b200.h).

There is no fallback: if the shared object is missing or a call fails, a RuntimeError is raised.
"""
import ctypes
import os

from . import build as _build

_LIB = None

c_int = ctypes.c_int
c_i32 = ctypes.c_int32
c_i64 = ctypes.c_int64
c_float = ctypes.c_float
c_void_p = ctypes.c_void_p


class ConvSource(ctypes.Structure):
	_fields_ = [
		('act', c_void_p), ('wgt', c_void_p), ('T_in', c_i32), ('T_rows', c_i32), ('ld_ch', c_i32), ('ch_off', c_i32),
		('C_in', c_i32), ('w_rows', c_i32), ('w_ld_ch', c_i32), ('w_ch_off', c_i32), ('taps', c_i32),
		('dilation', c_i32), ('pad_left', c_i32)
	]


class ConvEpilogue(ctypes.Structure):
	_fields_ = [
		('B', c_i32), ('T_out', c_i32), ('C_out', c_i32), ('block_n', c_i32), ('epilogue', c_i32), ('act', c_i32),
		('act_a', c_float), ('act_b', c_float), ('bias', c_void_p), ('xlen_frac', c_void_p), ('out_hi', c_void_p),
		('out_lo', c_void_p), ('out_T_rows', c_i32), ('out_ld_ch', c_i32), ('logits', c_void_p),
		('log_probs', c_void_p), ('argmax', c_void_p), ('stats', c_void_p), ('skip_frac', c_void_p), ('skip_T', c_i32),
		('skip_margin', c_i32),
		# BatchNorm-backward reduction folded into a dgrad launch
		('bnr_y', c_void_p), ('bnr_ss', c_void_p), ('bnr_xlen_frac', c_void_p), ('bnr_partials', c_void_p), ('bnr_C', c_i32), ('bnr_act', c_i32),
		('bnr_act_a', c_float), ('bnr_act_b', c_float)
	]


class PackItem(ctypes.Structure):
	_fields_ = [('w', c_void_p), ('fwd', c_void_p), ('dgrad', c_void_p), ('fwd_lo', c_void_p), ('dgrad_lo', c_void_p), ('Co', c_i32), ('Ci', c_i32), ('K', c_i32), ('ci_ld', c_i32), ('co_ld', c_i32), ('mode', c_i32), ('pad', c_i32)]


class UnpackItem(ctypes.Structure):
	_fields_ = [('packed', c_void_p), ('grad', c_void_p), ('K', c_i32), ('Co', c_i32), ('Ci', c_i32), ('ld', c_i32), ('transposed', c_i32), ('pair_pad', c_i32), ('pair_ci_alloc', c_i32)]


class BnBranch(ctypes.Structure):
	_fields_ = [('y', c_void_p), ('y_lo', c_void_p), ('ss', c_void_p)]


NGRAM_MAX_ORDER = 6  # CAB_NGRAM_MAX_ORDER


class NgramLM(ctypes.Structure):  # cab_ngram_lm_t
	_fields_ = [('order', c_i32), ('num_classes', c_i32), ('num_nodes', c_i32), ('bos', c_i32), ('tables', c_void_p * NGRAM_MAX_ORDER),
				('sizes', c_i64 * NGRAM_MAX_ORDER), ('child', c_void_p), ('word', c_void_p)]


class BeamStreamRow(ctypes.Structure):  # cab_beam_stream_t
	_fields_ = [('state', c_void_p), ('nodes', c_void_p), ('state_bytes', c_i64), ('capacity', c_i64), ('t0', c_i64), ('frames', c_i32),
				('is_eos', c_i32), ('finished', c_i32), ('reserved', c_i32)]


class BeamStreamIncrementalRow(ctypes.Structure):  # cab_beam_stream_incremental_t
	_fields_ = [('state', c_void_p), ('nodes', c_void_p), ('state_bytes', c_i64), ('capacity', c_i64), ('base', c_i64), ('t0', c_i64),
				('commit', c_i32), ('shift', c_i32), ('frames', c_i32), ('is_eos', c_i32), ('finished', c_i32), ('reserved', c_i32)]


ACT_NONE, ACT_RELU, ACT_HARDTANH, ACT_LEAKY_RELU = 0, 1, 2, 3
EPI_ACT_BF16, EPI_LOGSOFTMAX, EPI_LOGITS_F32, EPI_LOGITS_ROWS = 0, 1, 2, 3
MAX_CONV_SOURCES = 18
MAX_BN_BRANCHES = 12
PACK_MAX_ITEMS = 32
ABI_VERSION = 3

# name -> argtypes; every function returns int except the three introspection calls
BN_SUM_REPLICAS = 8  # CAB_BN_SUM_REPLICAS

SIGNATURES = {
	'cab_frontend_logmel': [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
							c_void_p, c_void_p, c_float, c_float, c_int, c_float, c_void_p, c_void_p, c_void_p],
	'cab_frontend_features': [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float, c_int, c_float,
								c_int, c_int, c_float, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
	'cab_frontend_features_fixed': [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float,
									c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p],
	'cab_frontend_stream': [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float,
							c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p],
	'cab_stream_copy': [c_void_p, c_int, c_i64, c_void_p],
	'cab_instnorm_pack': [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_int, c_int, c_void_p, c_void_p,
						c_void_p, c_void_p, c_void_p],
	'cab_conv1d_fused': [ctypes.POINTER(ConvSource), c_int, ctypes.POINTER(ConvEpilogue), c_void_p],
	'cab_conv1d_fused_fp8': [ctypes.POINTER(ConvSource), c_int, ctypes.POINTER(ConvEpilogue), c_void_p, c_float, c_void_p],
	'cab_absmax_bf16': [c_void_p, c_i64, c_void_p, c_void_p],
	'cab_quantize_e4m3': [c_void_p, c_i64, c_float, c_void_p, c_void_p],
	'cab_conv1d_wgrad': [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
						c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p],
	'cab_bn_batch_stats': [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_float, c_void_p, c_void_p,
							c_void_p, c_void_p, c_void_p],
	'cab_bn_finalize': [c_void_p, c_int, c_int, c_void_p, c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p],
	'cab_bn_act_mask_fwd': [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p, c_float,
							c_void_p, c_i64, c_void_p],
	'cab_bn_act_mask_bwd': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_void_p,
							c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_i64, c_int, c_void_p, c_void_p],
	'cab_bn_act_mask_bwd_apply': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_void_p,
								c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_i64, c_int, c_void_p, c_void_p],
	'cab_bn_bwd_apply_covers': [c_int, c_int, c_int],
	'cab_bn_multi_act_mask_fwd': [ctypes.POINTER(BnBranch), c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p,
								c_float, c_void_p, c_i64, c_void_p],
	'cab_act_mask_bwd_dz': [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p,
							c_float, c_void_p, c_i64, c_void_p],
	'cab_pack_weight': [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p],
	'cab_pack_weights_batched': [ctypes.POINTER(PackItem), c_int, c_void_p],
	'cab_unpack_wgrad': [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p],
	'cab_unpack_wgrad_batched': [ctypes.POINTER(UnpackItem), c_int, c_void_p],
	'cab_bct_to_btc': [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
	'cab_optimizer_step': [c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
							c_void_p, c_void_p, c_void_p, c_float, c_float, c_float, c_float, c_float, c_int, c_float, c_void_p, c_void_p, c_void_p],
	'cab_grouped_conv1d': [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
								c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p],
	'cab_grouped_conv1d_fp8': [c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
								c_void_p, c_int, c_int, c_float, c_void_p],
	'cab_grouped_conv1d_wgrad': [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
								c_void_p, c_void_p, c_void_p],
	'cab_bn_act_mask_fwd_stats': [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p,
								c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_i64, c_void_p],
	'cab_log_softmax_argmax': [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
	'cab_log_softmax_bwd': [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
	'cab_log_softmax_rows': [c_void_p, c_void_p, c_i64, c_int, c_int, c_void_p, c_void_p],
	'cab_ctc_loss_fwd': [c_void_p, c_i64, c_i64, c_i64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
						c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
	'cab_ctc_loss_bwd': [c_void_p, c_i64, c_i64, c_i64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
						c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_i64, c_i64, c_i64, c_void_p],
	'cab_ctc_loss_one_cta_covers': [c_int],
	'cab_ctc_loss_long_workspace': [c_int, c_int, c_int, ctypes.POINTER(c_i64)],
	'cab_ctc_loss_long_fwd': [c_void_p, c_i64, c_i64, c_i64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
								c_void_p, c_void_p, c_void_p, c_int, c_void_p],
	'cab_ctc_loss_long_bwd': [c_void_p, c_i64, c_i64, c_i64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
								c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_i64, c_i64, c_int, c_void_p],
	'cab_ctc_alignment':[c_void_p, c_i64, c_i64, c_i64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
						c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p],
	'cab_ctc_alignment_long': [c_void_p, c_i64, c_i64, c_i64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
								c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p],
	'cab_ctc_alignment_long_workspace': [c_int, c_int, c_int, ctypes.POINTER(c_i64)],
	'cab_topk_ids': [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
	'cab_greedy_collapse': [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p,
							c_void_p, c_int, c_void_p, c_void_p],
	'cab_top2_probs': [c_void_p, c_i64, c_i64, c_i64, c_int, c_int, c_int, c_void_p, c_void_p],
	'cab_entropy': [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
	'cab_ctc_beam_search_workspace': [c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, ctypes.POINTER(c_i64)],
	'cab_ctc_beam_search': [c_void_p, c_i64, c_i64, c_i64, c_void_p, c_int, c_int, c_int, c_int, c_float, c_int, c_int, c_int, c_void_p, c_i64,
							c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p],
	'cab_ctc_beam_search_lm': [c_void_p, c_i64, c_i64, c_i64, c_void_p, c_int, c_int, c_int, c_int, c_float, c_int, c_int, c_int, c_void_p, c_i64,
								c_void_p, c_void_p, c_int, c_void_p, c_void_p, ctypes.POINTER(NgramLM), c_float, c_float, c_int, c_void_p],
	'cab_ctc_beam_search_stream_state_bytes': [c_int, c_int, ctypes.POINTER(c_i64)],
	'cab_ctc_beam_search_stream_workspace': [c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_i64)],
	'cab_ctc_beam_search_stream': [c_void_p, c_i64, c_i64, c_i64, ctypes.POINTER(BeamStreamRow), c_int, c_int, c_int, c_int, c_float, c_int, c_int,
									c_int, c_void_p, c_i64, c_void_p, c_void_p, c_int, c_void_p, c_void_p, ctypes.POINTER(NgramLM), c_float, c_float,
									c_int, c_void_p],
	'cab_ctc_beam_search_stream_incremental_workspace': [c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_i64)],
	'cab_ctc_beam_search_stream_incremental': [c_void_p, c_i64, c_i64, c_i64, ctypes.POINTER(BeamStreamIncrementalRow), c_int, c_int, c_int, c_int,
												c_float, c_int, c_int, c_int, c_void_p, c_i64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
												c_int, c_void_p, c_void_p, ctypes.POINTER(NgramLM), c_float, c_float, c_int, c_void_p],
}
HOST_ONLY = {'cab_bn_bwd_apply_covers', 'cab_ctc_alignment_long_workspace', 'cab_ctc_loss_one_cta_covers', 'cab_ctc_loss_long_workspace',
			'cab_ctc_beam_search_workspace', 'cab_ctc_beam_search_stream_state_bytes', 'cab_ctc_beam_search_stream_workspace',
			'cab_ctc_beam_search_stream_incremental_workspace'}  # queries that launch nothing (left out of the per-entry-point device timing)
INTROSPECTION = {'cab_abi_version': c_int, 'cab_last_error': ctypes.c_char_p, 'cab_launch_count': c_i64}


def lib_path():
	return os.environ.get('CONVASR_B200_LIB') or _build.LIB_PATH


def load():
	"""Load (building first if the .so is absent and nvcc exists).  Raises loudly otherwise."""
	global _LIB
	if _LIB is not None:
		return _LIB
	path = lib_path()
	if path == _build.LIB_PATH and _build.needs_build():
		# missing, or older than its sources: rebuild (under a file lock; concurrent ranks wait and then load the result)
		try:
			_build.build()
		except Exception as e:
			if not os.path.exists(path):
				raise RuntimeError(
					f'convasr_b200: native library {path} is missing and could not be built ({e}); there is no fallback path'
				) from e
			# no compiler on this machine (a GPU box running a snapshot): the shipped library is used as is; an ABI
			# mismatch is caught below
	elif not os.path.exists(path):
		raise RuntimeError(f'convasr_b200: native library {path} is missing; there is no fallback path')
	lib = ctypes.CDLL(path)
	for name, argtypes in SIGNATURES.items():
		fn = getattr(lib, name)
		fn.argtypes = argtypes
		fn.restype = c_int
	for name, restype in INTROSPECTION.items():
		fn = getattr(lib, name)
		fn.argtypes = []
		fn.restype = restype
	if lib.cab_abi_version() != ABI_VERSION:
		raise RuntimeError(f'convasr_b200: ABI version mismatch ({lib.cab_abi_version()} != {ABI_VERSION}): stale {path}? rebuild with python -m convasr_b200.build --force')
	_LIB = lib
	return lib


def check(rc, what):
	if rc != 0:
		msg = load().cab_last_error()
		raise RuntimeError(f'convasr_b200: {what} failed (rc={rc}): {msg.decode() if msg else "?"}')


def launch_count():
	return int(load().cab_launch_count())


class trace:
	"""Per-entry-point device timing for bench.py: `with _lib.trace() as t:` wraps every C-ABI call in a pair of CUDA
	events on the launching (current torch) stream; afterwards t.summary() = {entry point: (calls, total ms)}.
	Eager launches only (a CUDA-graph replay does not pass through here)."""

	def __init__(self, names = None):
		self.names = list(names) if names is not None else [n for n in SIGNATURES if n not in HOST_ONLY]
		self.events = []

	def __enter__(self):
		import torch
		lib = load()
		self._orig = {}
		for name in self.names:
			fn = getattr(lib, name)
			self._orig[name] = fn

			def make(fn, name):
				def traced(*a):
					e0, e1 = torch.cuda.Event(enable_timing = True), torch.cuda.Event(enable_timing = True)
					e0.record()
					rc = fn(*a)
					e1.record()
					self.events.append((name, e0, e1))
					return rc
				return traced

			setattr(lib, name, make(fn, name))
		return self

	def __exit__(self, *exc):
		lib = load()
		for name, fn in self._orig.items():
			setattr(lib, name, fn)
		return False

	def summary(self):
		import torch
		torch.cuda.synchronize()
		out = {}
		for name, e0, e1 in self.events:
			n, ms = out.get(name, (0, 0.0))
			out[name] = (n + 1, ms + e0.elapsed_time(e1))
		return out
