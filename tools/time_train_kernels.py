"""Times the activation-sized BatchNorm training kernels at the layer shapes of the headline workload (C2: B = 80, T = 751,
widths 256 ... 1024, weighted by how many layers have that width), L2 flushed before every call."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from convasr_b200 import _lib, ops
lib = _lib.load(); dev = 'cuda'
B, T = 80, 751
flush = torch.empty(256 << 20, dtype = torch.uint8, device = dev)
def timeit(fn, n = 7):
	for _ in range(2): fn()
	ts = []
	for _ in range(n):
		flush.zero_()
		e0, e1 = torch.cuda.Event(enable_timing = True), torch.cuda.Event(enable_timing = True)
		e0.record(); fn(); e1.record(); torch.cuda.synchronize()
		ts.append(e0.elapsed_time(e1) * 1e3)
	ts.sort(); return ts[len(ts) // 2]
tot = dict(fwd = 0.0, bwd = 0.0, apply = 0.0)
rows = []
for C, count in ((256, 4), (384, 3), (512, 3), (640, 3), (768, 3), (896, 1), (1024, 1)):
	y = torch.randn(B, T, C, device = dev).to(torch.bfloat16)
	g = torch.randn(B, T, C, device = dev).to(torch.bfloat16)
	out = torch.empty_like(y); dy = torch.empty_like(y)
	gamma = torch.ones(C, device = dev); beta = torch.full((C, ), 8.0, device = dev)
	rm = torch.zeros(C, device = dev); rv = torch.ones(C, device = dev)
	raw = torch.zeros(2, C, dtype = torch.float64, device = dev)
	raw[0] = y.float().sum((0, 1)).double(); raw[1] = (y.float() ** 2).sum((0, 1)).double()
	ss = torch.empty(4, C, device = dev); sums = torch.empty(2, C, device = dev); part = torch.zeros(_lib.BN_SUM_REPLICAS * 2 * C, dtype = torch.float64, device = dev)
	xlen = torch.ones(B, device = dev)
	t_f = timeit(lambda: _lib.check(lib.cab_bn_act_mask_fwd_stats(ops._p(y), None, ops._p(raw), C, B * T, ops._p(gamma), ops._p(beta), 1e-5, 0.1, ops._p(rm), ops._p(rv), ops._p(ss), B, T, C, C, 2, 0.0, 20.0, ops._p(xlen), ops._p(out), None, 0.0, None, 0, ops._stream()), 'fwd'))
	t_b = timeit(lambda: _lib.check(lib.cab_bn_act_mask_bwd(ops._p(y), None, ops._p(g), None, ops._p(ss), B, T, C, C, 2, 0.0, 20.0, ops._p(xlen), ops._p(sums), ops._p(dy), None, 0.0, None, 0, 0, ops._p(part), ops._stream()), 'bwd'))
	t_a = timeit(lambda: _lib.check(lib.cab_bn_act_mask_bwd_apply(ops._p(y), None, ops._p(g), None, ops._p(ss), B, T, C, C, 2, 0.0, 20.0, ops._p(xlen), ops._p(sums), ops._p(dy), None, 0.0, None, 0, 0, ops._p(part), ops._stream()), 'apply'))
	mb = y.numel() * 2 / 1e6
	rows.append(f'C={C}: fwd {t_f:.1f} us ({2 * mb / t_f:.2f} TB/s) bwd {t_b:.1f} apply {t_a:.1f} us ({3 * mb / t_a:.2f} TB/s)')
	tot['fwd'] += count * t_f; tot['bwd'] += count * t_b; tot['apply'] += count * t_a
print(f'18-layer totals: fwd {tot["fwd"]:.0f} us, bwd(reduce+apply) {tot["bwd"]:.0f} us, apply-only {tot["apply"]:.0f} us | ' + ' | '.join(rows))
