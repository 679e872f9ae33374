"""Developer aid: in-kernel cycle counters of the shared-memory solve kernel (CTA 0, per warp and phase).

    LRBMS_DEVTOOLS=1 python -m pylrbms_b200.build --force && python tools/solve_timing.py [--solver window|auto]

Needs a library built with -DLRBMS_DEVTOOLS (never the shipped build)."""
import os, sys, numpy as np, ctypes as C
os.environ['LRBMS_SOLVE_TIMING'] = '1'
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
solver = 'window'
if '--solver' in sys.argv:
    i = sys.argv.index('--solver'); solver = sys.argv[i + 1]; del sys.argv[i:i + 2]
import torch, bench
from pylrbms_b200 import LRBMSReductor, discretize
a = bench.parse_args()
data, bases = bench.make_inputs(a)
d, _ = discretize(data); rd = LRBMSReductor(d, bases=bases).reduce()
rd.set_solver(solver)
n_mu = 148 * 8
theta = torch.from_numpy(rd.thetas(bench.make_mus(a, 0, n_mu))).cuda()
rd.solve_device(theta)                  # counters are overwritten by every launch: one launch = 8 parameters on CTA 0
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record(); rd.solve_device(theta); e1.record(); e1.synchronize()
plan = rd.online_plan
out = np.zeros(128, dtype=np.int64)
n = plan.handle.lib.lrbms_online_debug_timing(plan.p, out.ctypes.data, 128)
assert n == 128, plan.handle.lib.lrbms_last_error(plan.handle.h)
t = out.reshape(16, 8) / 8.0            # per parameter
names = ['meta', 'chain|Y', 'ubar', 'X', 'endbar', 'epi', 'back', 'store']
div, what = 160, 'column'
print('kernel', rd.solve_kernel_name, ' launch of', n_mu, 'parameters: %.3f ms' % e0.elapsed_time(e1))
print('cycles per parameter, per warp:')
print('warp ' + ' '.join('%9s' % n for n in names) + '   total')
for w in range(16):
    print('%4d ' % w + ' '.join('%9.0f' % v for v in t[w]) + '  %9.0f' % t[w].sum())
print('per %s (update warps, mean): ' % what, ' '.join('%s=%.0f' % (n, t[1:, k].mean() / div) for k, n in enumerate(names[:7])),
      ' warp 0: ', ' '.join('%s=%.0f' % (n, t[0, k] / div) for k, n in enumerate(names[:7])))
