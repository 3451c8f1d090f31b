"""In-tree nvcc build of libconvasr_b200.so (sm_100a only).

`python -m convasr_b200.build` or `__graft_entry__.build()`.  The shared object lands next to
the package so it travels with a repo snapshot; it is git-ignored (built artefact).
"""
import os
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, 'csrc')
LIB_PATH = os.path.join(PKG_DIR, 'libconvasr_b200.so')
SOURCES = ['api.cu', 'frontend.cu', 'conv_gemm.cu', 'wgrad_gemm.cu', 'ctc.cu', 'train.cu', 'optim.cu', 'grouped_conv.cu', 'beam.cu']
HEADERS = ['common.cuh', os.path.join('..', '..', 'include', 'convasr_b200.h')]

NVCC_FLAGS = [
	'-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '--use_fast_math=false',
	'-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=default', '--expt-relaxed-constexpr'
]


def _nvcc():
	cand = os.environ.get('NVCC') or '/usr/local/cuda/bin/nvcc'
	return cand if os.path.exists(cand) else 'nvcc'


HASH_PATH = LIB_PATH + '.srchash'


def source_hash():
	"""content hash of everything the library is built from (mtimes do not survive a snapshot copy to a GPU box)"""
	import hashlib
	h = hashlib.sha256()
	for d in [os.path.join(CSRC, s) for s in SOURCES + HEADERS]:
		h.update(open(d, 'rb').read())
	h.update(' '.join(NVCC_FLAGS).encode())
	return h.hexdigest()


def needs_build():
	if not os.path.exists(LIB_PATH) or not os.path.exists(HASH_PATH):
		return True
	return open(HASH_PATH).read().strip() != source_hash()


def build(force = False, verbose = False):
	"""Compile and link under an exclusive file lock: ranks of one torchrun that all find the library stale take
	turns, the first one builds (objects and the .so go to temporary names, then os.replace), the others see a
	fresh library when they get the lock."""
	import fcntl
	if not force and not needs_build():
		return LIB_PATH
	with open(os.path.join(PKG_DIR, '.build.lock'), 'w') as lock:
		fcntl.flock(lock, fcntl.LOCK_EX)
		try:
			if not force and not needs_build():
				return LIB_PATH
			return _build_locked(verbose)
		finally:
			fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose):
	objs = []
	procs = []
	for src in SOURCES:
		obj = os.path.join(CSRC, src.replace('.cu', '.o'))
		cmd = [_nvcc(), *[f for f in NVCC_FLAGS if f != '--use_fast_math=false'], '-c', os.path.join(CSRC, src), '-o', obj]
		if verbose:
			cmd.insert(1, '-Xptxas=-v')
		procs.append((src, subprocess.Popen(cmd, stdout = subprocess.PIPE, stderr = subprocess.STDOUT, text = True)))
		objs.append(obj)
	failed = False
	for src, proc in procs:
		out, _ = proc.communicate()
		if proc.returncode != 0:
			failed = True
			sys.stderr.write(f'--- nvcc failed for {src} ---\n{out}\n')
		elif verbose and out:
			sys.stderr.write(f'--- {src} ---\n{out}\n')
	if failed:
		raise RuntimeError('convasr_b200: nvcc compilation failed')
	tmp = LIB_PATH + f'.tmp{os.getpid()}'
	link = [_nvcc(), '-shared', '-o', tmp, *objs, '-gencode', 'arch=compute_100a,code=sm_100a', '-lcudart']
	res = subprocess.run(link, stdout = subprocess.PIPE, stderr = subprocess.STDOUT, text = True)
	if res.returncode != 0:
		raise RuntimeError('convasr_b200: link failed\n' + res.stdout)
	os.replace(tmp, LIB_PATH)
	with open(HASH_PATH, 'w') as f:
		f.write(source_hash())
	return LIB_PATH


if __name__ == '__main__':
	print(build(force = '--force' in sys.argv, verbose = '-v' in sys.argv))
