"""Weak greedy (pylrbms_b200.greedy) step by step at C2: OS2015, 8 x 8 subdomains, 32 x 32 cells, n = 393 216, 4 096 training
parameters, bases started from the constant shape function (LRBMSReductor(d), incremental re-projection on).

Two runs of 5 extensions each: k = 1 parameter per extension (extend_basis(method='pod', pod_modes=1)) and k = 32
(pod_modes=4).  Every step records the reduce time, the sweep of the training set (solve + estimate, eta to the host), the
fine solve of the k selected parameters cold (d.solve_batch, zero initial guess) and warm (the same lrbms_affine_pcg_solve
call and options, started from the reconstructed reduced solutions), their iterations, the time of the warm-start guess
itself, the extension time and the basis sizes.  A step whose extension finds nothing above pod_rtol ends the run, as it
ends greedy(); the true error of the snapshots against the reduced model of the final bases is then logged.  The k = 32 run also
times the Gram-Schmidt extension of the first step's 32 snapshots on a copy of the initial bases.  The card, its power
limit and SM clocks are read in the same run.  Every time is a host clock around work that ends in a device synchronise.

    python tools/greedy_timing.py [--out FILE] [--n-train 4096] [--steps 5]
"""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from pylrbms_b200 import ExtensionError, LRBMSReductor, discretize, reduction_error_analysis
from pylrbms_b200.greedy import select_worst
from pylrbms_b200.kernels import affine_pcg_solve
from pylrbms_b200.parameters import theta_matrix
from pylrbms_b200.swipdg_fixture import assemble_block_swipdg

ap = argparse.ArgumentParser()
ap.add_argument('--out', default=None)
ap.add_argument('--n-train', type=int, default=4096)
ap.add_argument('--steps', type=int, default=5)
args = ap.parse_args()
lines = []


def log(s=''):
    print(s, flush=True)
    lines.append(s)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


if not torch.cuda.is_available():
    raise SystemExit('greedy_timing.py needs the B200: there is no CPU path to time')
card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm', '--format=csv,noheader'],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
log('card: ' + card + ' (name, power limit, SM clock, max SM clock)')

data = assemble_block_swipdg((8, 8), 32)
d, _ = discretize(data)
S, n = data.num_subdomains, d.solution_space.dim
train = np.random.default_rng(2026).uniform(*data.parameter_range, args.n_train)
log('C2: n = {}, {} subdomains, {} training parameters, {} extensions per run'.format(n, S, len(train), args.steps))
# warm-up: modules, the affine pattern, a first plan and online plan (not timed)
d.solve_batch(train[:1])
warm_red = LRBMSReductor(d)
warm_red.reduce().sweep_eta_into(train[:64], torch.empty(64, dtype=torch.float64, pin_memory=True))
del warm_red


def warm_solve(mus, guess):
    """d.solve_batch(mus) (default options) from the initial guess ``guess`` instead of zero: returns the iterations."""
    pattern, values, rhs = d.affine_system(range(S))
    theta = torch.from_numpy(theta_matrix(list(d.operator.coefficients) + list(d.rhs.coefficients), mus,
                                          d.parameter_type)).cuda()
    x = torch.zeros((n, max(4, (len(mus) + 3) // 4 * 4)), dtype=torch.float64, device='cuda')
    row = 0
    for b in guess._blocks:
        x[row:row + b.dim, :len(mus)] = b.dofmajor()
        row += b.dim
    _, it, rr, st = affine_pcg_solve(pattern, values, rhs, theta, x, 1e-9, max(100, 10 * n), 3)
    assert np.all(st == 0) and np.all(rr <= 1e-9)
    return it


summary = {}
for k, pod_modes in ((1, 1), (32, 4)):
    log()
    log('k = {} parameters per extension, extend_basis(method=\'pod\', pod_modes={})'.format(k, pod_modes))
    log('step |  N min/max  sum N | reduce s | sweep ms | cold solve s  iters mean/max | guess ms | warm solve s  iters '
        'mean/max | extend ms | max eta')
    red = LRBMSReductor(d)
    red.incremental = True
    eta_host = torch.empty(len(train), dtype=torch.float64, pin_memory=True)
    rows = []
    for step in range(args.steps):
        N = [len(red.bases[s.id]) for s in d.solution_space.subspaces]
        rd, t_reduce = timed(red.reduce)
        (bad, _, _), t_sweep = timed(lambda: rd.sweep_eta_into(train, eta_host))
        assert bad == 0
        eta = eta_host.numpy().copy()
        sel = train[select_worst(eta, k)]
        guess, t_guess = timed(lambda: red.reconstruct(rd.solve_batch(sel)))
        U, t_cold = timed(lambda: d.solve_batch(sel))
        it_cold = d.last_solve_info['iterations'].copy()
        it_warm, t_warm = timed(lambda: warm_solve(sel, guess))
        if k == 32 and step == 0:
            gs = LRBMSReductor(d)
            _, t_gs = timed(lambda: gs.extend_basis(U))
            summary['gs'] = (t_gs, sum(len(gs.bases[s.id]) for s in d.solution_space.subspaces) - sum(N))
            del gs
        try:
            _, t_ext = timed(lambda: red.extend_basis(U, method='pod', pod_modes=pod_modes))
        except ExtensionError:
            ana = reduction_error_analysis(d, red, red.reduce(), sel, U_h=U)
            log('{:4d} | {:4d}/{:<4d} {:6d} | ExtensionError: no mode above pod_rtol; the snapshots\' relative errors against the '
                'reduced model are {:.2e} .. {:.2e} (cold {:.0f}, warm {:.0f} iterations)'.format(
                    step, min(N), max(N), sum(N), ana.relative_errors.min(), ana.relative_errors.max(), it_cold.mean(),
                    it_warm.mean()))
            break
        rows.append(dict(t_reduce=t_reduce, t_sweep=t_sweep, t_cold=t_cold, t_warm=t_warm, t_guess=t_guess, t_ext=t_ext,
                         it_cold=it_cold, it_warm=it_warm,
                         added=sum(len(red.bases[s.id]) for s in d.solution_space.subspaces) - sum(N)))
        log('{:4d} | {:4d}/{:<4d} {:6d} | {:8.3f} | {:8.2f} | {:12.3f}  {:7.0f}/{:<5d} | {:8.2f} | {:12.3f}  {:7.0f}/{:<5d} | '
            '{:9.2f} | {:.4e}'.format(step, min(N), max(N), sum(N), t_reduce, 1e3 * t_sweep, t_cold, it_cold.mean(),
                                      int(it_cold.max()), 1e3 * t_guess, t_warm, it_warm.mean(), int(it_warm.max()),
                                      1e3 * t_ext, float(eta.max())))
    summary[k] = rows

log()
log('summary')
for k in (1, 32):
    rows = summary[k]
    cold = sum(r['t_cold'] for r in rows)
    warm = sum(r['t_warm'] for r in rows)
    added = sum(r['added'] for r in rows)
    it_c = np.concatenate([r['it_cold'] for r in rows])
    it_w = np.concatenate([r['it_warm'] for r in rows])
    step = [r['t_reduce'] + r['t_sweep'] + r['t_cold'] + r['t_ext'] for r in rows]      # one step of greedy()
    ext_share = [r['t_ext'] / s for r, s in zip(rows, step)]
    log('k = {:2d}: fine solve per solved parameter cold {:.3f} s, warm {:.3f} s; per added basis vector cold {:.4f} s '
        '({} vectors); iterations cold mean {:.0f}, warm mean {:.0f} ({:+.1f} %); extension {:.2f}-{:.2f} % of a step'
        .format(k, cold / (k * len(rows)), warm / (k * len(rows)), cold / max(1, added), added, it_c.mean(), it_w.mean(),
                100.0 * (it_w.mean() / it_c.mean() - 1.0), 100 * min(ext_share), 100 * max(ext_share)))
t_gs, n_gs = summary['gs']
log('Gram-Schmidt extension of the 32 snapshots of the first k = 32 step: {:.3f} s ({} vectors appended); POD: {:.3f} s'
    .format(t_gs, n_gs, summary[32][0]['t_ext']))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write('\n'.join(lines) + '\n')
