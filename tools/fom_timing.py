"""Fine-scale solve d.solve_batch (lrbms_affine_pcg_solve) at C2: OS2015, 8 x 8 subdomains, 32 x 32 cells, n = 393 216.

Records the card and its power limit, wall time (device synchronised, after warm-up) for batches of 1, 32 and 128
parameters, iterations and attained true residuals, SciPy splu on the host for a sample of the same parameters, the
energy-norm error against splu, and the effectivity eta(mu) / |||u_h - R u_N||| of the N = 20 reduced model over 32
parameters.  Then, recorded but not asserted, the Jacobi-CG behaviour on the contrast-1e6 SPE10-like field (4 x 4, 16 cells).

    python tools/fom_timing.py [--out FILE]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spl
import torch

from pylrbms_b200 import LRBMSReductor, discretize
from pylrbms_b200._lib import LrbmsError
from pylrbms_b200.parameters import theta_matrix
from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases, spe10_like_problem

ap = argparse.ArgumentParser()
ap.add_argument('--out', default=None)
args = ap.parse_args()
lines = []


def log(s=''):
    print(s, flush=True)
    lines.append(s)


if not torch.cuda.is_available():
    raise SystemExit('fom_timing.py needs the B200: there is no CPU path to time')
card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
log('card: ' + card + ' (name, power limit, max SM clock)')


def host_system(data, d, mu):
    th = theta_matrix(list(d.operator.coefficients) + list(d.rhs.coefficients), [mu], d.parameter_type)[0]
    S = data.num_subdomains
    A = None
    for q in range(data.Q):
        blocks = [[None] * S for _ in range(S)]
        for (i, j), M in data.lhs[q].items():
            blocks[i][j] = M
        A = th[q] * sp.bmat(blocks, format='csc') if A is None else A + th[q] * sp.bmat(blocks, format='csc')
    return A.tocsc(), th[data.Q] * np.concatenate(data.rhs)


data = assemble_block_swipdg((8, 8), 32)
d, _ = discretize(data)
n = d.solution_space.dim
lo, hi = data.parameter_range
log('C2: n = %d, nnz per component = %d' % (n, d.affine_system(range(data.num_subdomains))[0].nnz))
rng = np.random.default_rng(2024)
d.solve_batch(rng.uniform(lo, hi, 2))                                 # warm-up: operator upload, module load
results = {}
for size in (1, 32, 128):
    mus = rng.uniform(lo, hi, size)
    torch.cuda.synchronize()
    t = time.perf_counter()
    U = d.solve_batch(mus)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t
    info = d.last_solve_info
    it, rr = info['iterations'], info['relative_residual']
    groups = (size + 31) // 32
    results[size] = (mus, U, dt)
    log('batch %4d: %.3f s, %.1f parameters/s, %.1f us per iteration per group of 32 (%d groups, %d iterations for the '
        'slowest); iterations min / median / max %d / %d / %d; true relative residual max %.2e, median %.2e'
        % (size, dt, size / dt, 1e6 * dt / it.max() / groups, groups, it.max(), it.min(), int(statistics.median(it)),
           it.max(), rr.max(), float(np.median(rr))))

mus32, U32, dt32 = results[32]
U32d = U32.data
n_lu = 4
t_lu, errs = [], []
for k in range(n_lu):
    A, b = host_system(data, d, mus32[k])
    t = time.perf_counter()
    u_ref = spl.splu(A).solve(b)
    t_lu.append(time.perf_counter() - t)
    if k < 2:
        e = U32d[k] - u_ref
        errs.append(np.sqrt(e @ (A @ e)) / np.sqrt(u_ref @ (A @ u_ref)))
log('SciPy splu on the host (%d cores visible), one factorisation per parameter: %.2f s per parameter (mean of the first '
    '%d of the 32-batch) = %.3f parameters/s; GPU batch of 32: %.1f parameters/s' % (
        os.cpu_count(), float(np.mean(t_lu)), n_lu, 1.0 / float(np.mean(t_lu)), 32 / dt32))
log('energy-norm error against splu (relative): ' + ', '.join('%.2e' % e for e in errs))

bases = make_local_bases(data, 20, seed=1002)
red = LRBMSReductor(d, bases={'domain_%d' % i: bases[i] for i in range(data.num_subdomains)})
rd = red.reduce()
uN = rd.solve_batch(mus32)
eta = np.asarray(rd.estimate_batch(uN, mus32))
R = red.reconstruct(uN).data
offs = np.concatenate([[0], np.cumsum(data.n)])
err = np.zeros(32)
for i in range(data.num_subdomains):
    E = (U32d - R)[:, offs[i]:offs[i + 1]]
    err += np.einsum('kd,kd->k', E, (data.energy[i] @ E.T).T)
eff = eta / np.sqrt(err)
log('effectivity eta / |||u_h - R u_N||| (N = 20, 32 parameters): min %.3f, max %.3f' % (eff.min(), eff.max()))

data6 = assemble_block_swipdg((4, 4), 16, problem=spe10_like_problem(seed=1003, contrast=1e6))
d6, _ = discretize(data6)
mus6 = np.linspace(*data6.parameter_range, 4)
try:
    d6.solve_batch(mus6)
    log('SPE10-like contrast 1e6 (4 x 4, 16 cells, n = %d): converged' % d6.solution_space.dim)
except LrbmsError as e:
    log('SPE10-like contrast 1e6 (4 x 4, 16 cells, n = %d): raised: %s' % (d6.solution_space.dim, e))
inf6 = d6.last_solve_info
log('  iterations %s, true relative residuals %s, status %s' % (
    list(inf6['iterations']), ['%.2e' % r for r in inf6['relative_residual']], list(inf6['status'])))
if args.out:
    with open(args.out, 'w') as f:
        f.write('\n'.join(lines) + '\n')
