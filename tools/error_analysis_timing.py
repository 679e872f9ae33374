"""Reduction error analysis (reduction_error_analysis, csrc/error_norms.cu) at C2: OS2015, 8 x 8 subdomains, 32 x 32 cells,
n = 393 216, N = 20 per subdomain, 128 parameters.

Records the card, its power limit and SM clock (read in the same run); CUDA-event times of the two new kernels
(lrbms_recon_error, lrbms_segmented_form with the local energy products and with the affine operator), each warmed up and
preceded by a 256 MB L2 flush, against the bytes they must move (counted from shapes) at 7.7 TB/s; the same error
measurement done by the composed VectorArray path (reductor.reconstruct, -, CsrOperator.pairwise_apply2) and by the host
loop of tools/fom_timing.py; and the share of the whole analysis spent in the fine-scale solve.

    python tools/error_analysis_timing.py [--out FILE] [--n-mu 128] [--reps 20]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from pylrbms_b200 import LRBMSReductor, discretize, reduction_error_analysis
from pylrbms_b200.error_analysis import _dofmajor, _energy_system
from pylrbms_b200.kernels import recon_error, segmented_form
from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases
from pylrbms_b200.vectorarray import _round_cap

ap = argparse.ArgumentParser()
ap.add_argument('--out', default=None)
ap.add_argument('--n-mu', type=int, default=128)
ap.add_argument('--reps', type=int, default=20)
args = ap.parse_args()
lines = []
HBM = 7.7e12


def log(s=''):
    print(s, flush=True)
    lines.append(s)


if not torch.cuda.is_available():
    raise SystemExit('error_analysis_timing.py needs the B200: there is no CPU path to time')
card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm', '--format=csv,noheader'],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
log('card: ' + card + ' (name, power limit, SM clock, max SM clock)')

data = assemble_block_swipdg((8, 8), 32)
d, _ = discretize(data)
S, n, n_mu = data.num_subdomains, d.solution_space.dim, args.n_mu
bases = make_local_bases(data, 20, seed=1002)
red = LRBMSReductor(d, bases={'domain_%d' % i: bases[i] for i in range(S)})
rd = red.reduce()
mus = np.random.default_rng(2024).uniform(*data.parameter_range, n_mu)
reduction_error_analysis(d, red, rd, mus[:2])                          # warm-up: modules, patterns, plans

torch.cuda.synchronize()
t0 = time.perf_counter()
res = reduction_error_analysis(d, red, rd, mus)
torch.cuda.synchronize()
t_all = time.perf_counter() - t0
torch.cuda.synchronize()
t0 = time.perf_counter()
U_h = d.solve_batch(mus)
torch.cuda.synchronize()
t_solve = time.perf_counter() - t0
torch.cuda.synchronize()
t0 = time.perf_counter()
res2 = reduction_error_analysis(d, red, rd, mus, U_h=U_h)
torch.cuda.synchronize()
t_rest = time.perf_counter() - t0
assert np.array_equal(res.errors, res2.errors)
log('C2: n = %d, S = %d, N = 20, %d parameters' % (n, S, n_mu))
log('whole analysis (fine solve included): %.3f s; fine solve alone: %.3f s (%.1f %% of the whole); analysis with U_h '
    'given (reduced sweep + error kernels + host copies): %.1f ms' % (t_all, t_solve, 100 * t_solve / t_all, 1e3 * t_rest))
log('effectivity eta / |||u_h - R u_N||| over %d parameters: min %.3f, max %.3f; max error %.3e (relative %.3e)' % (
    n_mu, res.min_effectivity, res.max_effectivity, res.max_error, res.relative_errors.max()))

# ---- kernel times
U_N, _ = rd.sweep(mus)
u_h = _dofmajor(U_h, n, n_mu)
u_N = U_N.device_tensor.contiguous()
subs = d.solution_space.subspaces
bl = [red.bases[s.id] for s in subs]
E_pat, E_vals, offs = _energy_system(d)
A_pat, A_vals, _ = d.affine_system(range(S))
from pylrbms_b200.parameters import theta_matrix                        # noqa: E402
theta = torch.from_numpy(theta_matrix(list(d.operator.coefficients) + list(d.rhs.coefficients), mus,
                                      d.parameter_type)).cuda()
e = torch.empty((n, _round_cap(n_mu)), dtype=torch.float64, device='cuda')
out_l = torch.empty((S, n_mu), dtype=torch.float64, device='cuda')
out_o = torch.empty((1, n_mu), dtype=torch.float64, device='cuda')
flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')


def time_call(fn):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(args.reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    return statistics.median(ts), min(ts), max(ts)


N_tot = sum(len(b) for b in bl)
Q = A_vals.shape[0]
bytes_recon = 8 * (2 * n * n_mu + n * 20 + n_mu * N_tot)                # u_h read, e written, V, u_N
bytes_energy = 8 * n * n_mu + 12 * E_pat.nnz + 4 * (n + 1)             # e read once, pattern with one value array
bytes_op = 8 * n * n_mu + (4 + 8 * Q) * A_pat.nnz + 4 * (n + 1) + 8 * Q * n_mu
cases = [('lrbms_recon_error (e = u_h - R u_N)', lambda: recon_error(bl, rd.block_dims, u_h, u_N, e), bytes_recon),
         ('lrbms_segmented_form, local energy products (Q = 1, %d segments, nnz %d)' % (S, E_pat.nnz),
          lambda: segmented_form(E_pat, E_vals, offs, e, n_mu, out=out_l), bytes_energy),
         ('lrbms_segmented_form, affine operator (Q = %d, one segment, nnz %d)' % (Q, A_pat.nnz),
          lambda: segmented_form(A_pat, A_vals, [0, n], e, n_mu, theta=theta, out=out_o), bytes_op)]
log('kernel times: CUDA events around one library call (host table upload + launches), median / min / max of %d, each '
    'after 3 warm-up calls and a 256 MB write that evicts L2 (126 MB); the error scratch is %.0f MB, u_h %.0f MB'
    % (args.reps, 8e-6 * n * e.shape[1], 8e-6 * n * u_h.stride(0)))
for name, fn, nbytes in cases:
    med, lo, hi = time_call(fn)
    log('  %s: %.1f us (%.1f .. %.1f); %.1f MB from shapes -> %.2f TB/s = %.0f %% of 7.7 TB/s (HBM bound %.1f us)' % (
        name, 1e6 * med, 1e6 * lo, 1e6 * hi, 1e-6 * nbytes, nbytes / med * 1e-12, 100 * nbytes / med / HBM,
        1e6 * nbytes / HBM))
assert np.array_equal(np.sqrt(np.maximum(out_l.cpu().numpy(), 0)), res.local_errors)

# ---- the composed VectorArray path: reconstruct (one lincomb per subdomain), difference, SpMM + pairwise dot per subdomain
def composed():
    R = red.reconstruct(U_N)
    D = U_h - R
    return np.sqrt(sum(d.operators['local_energy_dg_product_%d' % i].pairwise_apply2(D._blocks[i], D._blocks[i])
                       for i in range(S)))


composed()
ts = []
for _ in range(3):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    err_c = composed()
    torch.cuda.synchronize()
    ts.append(time.perf_counter() - t0)
log('composed path (reductor.reconstruct, -, CsrOperator.pairwise_apply2 per subdomain): %.1f ms (median of 3, wall '
    'clock to a device synchronise); energy errors agree with the analysis to %.1e relative' % (
        1e3 * statistics.median(ts), np.max(np.abs(err_c - res.errors) / res.errors)))

# ---- the host loop of tools/fom_timing.py
t0 = time.perf_counter()
Ud = U_h.data
Rd = red.reconstruct(U_N).data
err = np.zeros(n_mu)
for i in range(S):
    E = (Ud - Rd)[:, offs[i]:offs[i + 1]]
    err += np.einsum('kd,kd->k', E, (data.energy[i] @ E.T).T)
t_host = time.perf_counter() - t0
log('host loop of tools/fom_timing.py (%d cores visible; device-to-host copies included): %.2f s; energy errors agree '
    'with the analysis to %.1e relative' % (os.cpu_count(), t_host, np.max(np.abs(np.sqrt(err) - res.errors) / res.errors)))
if args.out:
    with open(args.out, 'w') as f:
        f.write('\n'.join(lines) + '\n')
