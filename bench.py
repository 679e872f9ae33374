#!/usr/bin/env python
"""Benchmark of the LRBMS hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port) on host cores
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step returned, DIR/*.npy

Workload (BASELINE.json configs[1], SURVEY.md section 8d row C2): OS2015 academic multiscale example, 8x8
subdomains, 6144 fine DG dofs each, local basis size 20 (n_red = 1280), Q = 2 affine terms; online batch of
10 000 parameters per GPU, uniform in [0.1, 1].  Synthetic inputs: the operators come from the structured P1-SWIPDG
assembler in ``pylrbms_b200.swipdg_fixture`` (DUNE is not available), the bases are seeded and orthonormalised in
the local energy products.

A *step* = one sweep of the hot path over one parameter batch: assemble + factor + solve + estimate for every
parameter (``lrbms_online_solve`` + ``lrbms_online_estimate``) followed by the estimator max (``lrbms_eta_max``; for
N > 1 one NCCL all-reduce(max) -- the "estimator-max gather", the only collective of the path).  ``value`` counts
solves+estimates per second with the coefficient matrix already in HBM; ``e2e`` goes through the public API
(``ReducedModel.sweep_into``) from host parameters to host results.  The offline half of the metric (projection
HBM GB/s) is measured in the same run on the same workload and reported under ``offline``.

One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'online reduced solves+estimates/s (mu-batched)'
UNIT = 'solves+estimates/s'



def ncu_traffic(kernel, workload):
    """DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed ``ncu --set full`` capture
    of this round (``profiles/traffic.json``, written by ``tools/ncu_summary.py`` from the raw pages).  An entry only counts
    if it was captured from the *same kernel source* (sha256 of the .cu file, recorded next to the numbers) and the same
    workload string -- after a kernel change the figure goes to null instead of silently going stale."""
    import hashlib
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            table = json.load(f)
        e = table[kernel]
        with open(os.path.join(ROOT, 'pylrbms_b200', 'csrc', e['source']), 'rb') as f:
            sha = hashlib.sha256(f.read()).hexdigest()
        if sha != e['source_sha256'] or e['workload'] != workload:
            return None
        return float(e['dram_bytes_per_launch'])
    except Exception:
        return None


# ----------------------------------------------------------------------------------------------------------
#  workload
# ----------------------------------------------------------------------------------------------------------

def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--subdomains', type=int, default=8, help='subdomains per direction (8 -> 8x8, config C2)')
    ap.add_argument('--cells', type=int, default=32, help='cells per subdomain and direction (32 -> n_i = 6144)')
    ap.add_argument('--basis', type=int, default=20, help='local basis size')
    ap.add_argument('--n-mu', type=int, default=10000, help='parameters per GPU and step')
    ap.add_argument('--cpu-sample', type=int, default=24, help='parameters per CPU-baseline step')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-offline', action='store_true')
    ap.add_argument('--offline-only', action='store_true', help='stop after the offline half (and its sharded run at N > 1)')
    ap.add_argument('--no-parity', action='store_true', help='skip the oracle parity gate (it runs whenever the oracle fits)')
    ap.add_argument('--eta-only', action='store_true', help='e2e ships eta only (ReducedModel.sweep_eta_into), not the solutions')
    ap.add_argument('--no-c5', dest='c5', action='store_false', help='skip the 125 000-parameter-per-GPU sweep (configs[4])')
    ap.add_argument('--no-c3-sharded', dest='c3_sharded', action='store_false',
                    help='at N > 1: skip the subdomain-sharded offline projection of configs[2] (SPE10-like, 16x16 subdomains)')
    ap.add_argument('--problem', default='os2015', choices=['os2015', 'spe10'],
                    help="spe10: the high-contrast (1e6) SPE10-like field of configs[2]")
    ap.add_argument('--config', default=None, choices=['c2', 'c3', 'c4', 'c5'],
                    help='shorthand for a BASELINE.json configuration: c2 = the default; c3 = --problem spe10 --subdomains 16 '
                         '--n-mu 2048; c4 = --synthetic3d 4,4,4 --subdomains 8 --basis 40 --n-mu 64 (full-size reduced system, '
                         'small fine grid); c5 = --n-mu 125000 --eta-only')
    ap.add_argument('--seed', type=int, default=1002)
    ap.add_argument('--synthetic3d', default=None, metavar='HX,HY,HZ',
                    help='seeded synthetic operators with 3D structure (config C4 shape): --subdomains per direction, '
                         'HX x HY x HZ cells of 4 dofs per subdomain (16,16,12 -> n_i = 12288); offline measurements only')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='after the timed steps, write what the last online step returned (u, eta, info, eta_max, and '
                         'the parameters mu they belong to) as DIR/<name>.npy in float64; at most 64 MB, a fixed seeded '
                         'sample of the parameters when all of them would not fit (rank 0 only)')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and (a.impl != 'b200' or a.offline_only):
        ap.error('--dump-outputs writes the outputs of the online step of --impl b200; it cannot be combined with '
                 '--impl reference or --offline-only')
    if a.config == 'c3':
        a.problem, a.subdomains, a.n_mu, a.c5 = 'spe10', 16, 2048, False
    elif a.config == 'c4':
        a.synthetic3d, a.subdomains, a.basis, a.n_mu, a.c5 = '4,4,4', 8, 40, 64, False
    elif a.config == 'c5':
        a.n_mu, a.eta_only, a.c5 = 125000, True, False
    return a


def problem_name(a):
    return 'OS2015' if a.problem == 'os2015' else 'SPE10-like (contrast 1e6)'


def workload_name(a):
    if a.synthetic3d:
        h = [int(x) for x in a.synthetic3d.split(',')]
        return 'synthetic 3D {0}x{0}x{0} subdomains, n_i={1}, N={2}, Q=2, {3} mu per GPU'.format(
            a.subdomains, 4 * h[0] * h[1] * h[2], a.basis, a.n_mu)
    return '{0} {1}x{1} subdomains, n_i={2}, N={3}, Q=2, {4} mu per GPU'.format(problem_name(a), a.subdomains, 6 * a.cells ** 2,
                                                                               a.basis, a.n_mu)


def make_inputs(a):
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases
    if a.synthetic3d:
        from pylrbms_b200.synthetic_fixture import make_random_local_bases, synthetic_block_operators
        h = tuple(int(x) for x in a.synthetic3d.split(','))
        data = synthetic_block_operators((a.subdomains,) * 3, h, seed=a.seed)
        bases = make_random_local_bases(data, a.basis, seed=a.seed)
        return data, {'domain_%d' % i: bases[i] for i in range(data.num_subdomains)}
    problem = None
    if a.problem == 'spe10':
        from pylrbms_b200.swipdg_fixture import spe10_like_problem
        problem = spe10_like_problem(seed=1003, contrast=1e6)
    data = assemble_block_swipdg((a.subdomains, a.subdomains), a.cells, problem=problem)
    bases = make_local_bases(data, a.basis, seed=a.seed)
    return data, {'domain_%d' % i: bases[i] for i in range(data.num_subdomains)}


def make_mus(a, rank, n, data=None):
    rng = np.random.default_rng(a.seed + 7919 * rank)
    lo, hi = tuple(data.parameter_range) if data is not None else (0.1, 1.0)
    return rng.uniform(lo, hi, n)


def survey_flops_per_mu(a, data, rd):
    return survey_flops_model(rd.block_dims, data.neighborhoods, data.Q, rd.half_bandwidth)


def survey_flops_model(N, nbh, Q, half_bandwidth):
    """Algorithmic flops of one solve+estimate, SURVEY.md section 8d: assemble 2 Q B N^2, banded Cholesky n b^2,
    two triangular solves 4 n b, estimator sum_i 2 (d_i^2 + 2 (Q d_i)^2 + Q^2 N^2 + Q^2 N d_i + Q d_i), with b the scalar half
    bandwidth of the lexicographically ordered reduced operator (2D: (sx + 1) N; 3D: (sx sy + 1) N) and d_i the summed basis
    sizes over the neighbourhood of subdomain i."""
    n = int(sum(N))
    B = sum(len(x) for x in nbh)                  # diagonal + directed face-neighbour blocks
    b = half_bandwidth + 1
    est = 0
    for s_, nb in enumerate(nbh):
        d = sum(N[k] for k in nb)
        est += 2 * (d * d + 2 * (Q * d) ** 2 + Q * Q * N[s_] ** 2 + Q * Q * N[s_] * d + Q * d)
    solve = 2 * Q * sum(N[i] * N[j] for i, nb in enumerate(nbh) for j in nb) + n * b * b + 4 * n * b
    return dict(solve=float(solve), estimate=float(est), total=float(solve + est), n_red=n, blocks=B, half_bandwidth=b)


# ----------------------------------------------------------------------------------------------------------
#  clocks
# ----------------------------------------------------------------------------------------------------------

class ClockSampler:
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.FIELDS,
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); power.append(float(r[2]))
                for name, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'power_w_max': max(power) if power else None, 'samples': len(sm), 'reasons': sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------
#  reference arm: the reference's CPU algorithm (oracle port) on the host cores
# ----------------------------------------------------------------------------------------------------------

def cpu_reference_model(a):
    """Offline phase with the oracle (NumPy/SciPy restatement of pylrbms on pyMOR); returns the reduced model."""
    from oracle import lrbms_oracle as O
    data, bases = make_inputs(a)
    t = time.perf_counter()
    d = O.build_discretization(data)
    red = O.LRBMSReductor(d, bases=bases)
    rd = red.reduce()
    return rd, time.perf_counter() - t


def cpu_online_step(rd, mus):
    """What the reference does per parameter: ``U = rd.solve(mu); eta = rd.estimate(U, mu)`` (online_enrichment.py:72-74)."""
    out = []
    for mu in mus:
        U = rd.solve(mu)
        out.append(rd.estimate(U, mu))
    return out


class VectorisedCpuModel:
    """SURVEY.md section 8d, CPU variant (ii): the same reduced model evaluated the way a careful CPU implementation
    would -- banded Cholesky (LAPACK dpbsv) on the block-banded reduced operator instead of a dense LU, and every estimator
    form restricted to the rows / columns it really touches instead of dense n_red-sized mat-vecs.  Reported next to the
    reference-faithful figure so that the GPU / CPU ratio is not inflated by the reference's dense storage."""

    def __init__(self, rd):
        import scipy.sparse as sp
        self.rd, est = rd, rd.estimator
        A = [np.asarray(o.matrix) for o in rd.operator.operators]
        n = A[0].shape[0]
        nz = np.nonzero(sum(np.abs(M) for M in A))
        self.b = int(np.max(np.abs(nz[0] - nz[1]))) if len(nz[0]) else 0
        self.ab = []
        for M in A:                                    # lower banded storage: ab[k, j] = M[j + k, j]
            ab = np.zeros((self.b + 1, n))
            for k in range(self.b + 1):
                ab[k, :n - k] = np.diagonal(M, -k)
            self.ab.append(ab)
        self.fr = [sp.csr_matrix(np.asarray(o.matrix)) for o in est.flux_reconstruction.operators]

        def restrict(M):
            M = np.asarray(M)
            r, c = np.nonzero(np.abs(M).sum(axis=1))[0], np.nonzero(np.abs(M).sum(axis=0))[0]
            return r, c, np.ascontiguousarray(M[np.ix_(r, c)])
        self.sub = []
        for ii, s_ in enumerate(est.subdomains):
            ops = rd.operators
            self.sub.append(dict(
                nc=restrict(ops['nc_%d' % s_].matrix), r_fd=restrict(ops['r_fd_%d' % s_]._array.data),
                r_dd=restrict(ops['r_dd_%d' % s_].matrix), df_bb=restrict(ops['df_bb_%d' % s_].matrix),
                df_aa=[(c, restrict(o.matrix)) for o, c in zip(ops['df_aa_%d' % s_].operators, ops['df_aa_%d' % s_].coefficients)],
                df_ab=[(c, restrict(o.matrix)) for o, c in zip(ops['df_ab_%d' % s_].operators, ops['df_ab_%d' % s_].coefficients)]))

    @staticmethod
    def _form(x, rcm, y):
        r, c, M = rcm
        return x[r] @ (M @ y[c])

    def step(self, mus):
        from scipy.linalg import solveh_banded
        rd, est = self.rd, self.rd.estimator
        out = []
        for mu_ in mus:
            mu = rd.parse_parameter(mu_)
            th = [c.evaluate(mu) for c in rd.operator.coefficients]
            ab = th[0] * self.ab[0]
            for q in range(1, len(th)):
                ab = ab + th[q] * self.ab[q]
            f = rd.rhs.as_source_array(mu).data[0]
            u = solveh_banded(ab, f, lower=True)
            thf = [c.evaluate(mu) for c in est.flux_reconstruction.coefficients]
            ur = sum(t * (S @ u) for t, S in zip(thf, self.fr))
            S_ = len(self.sub)
            nc, r, df = np.zeros(S_), np.zeros(S_), np.zeros(S_)
            for ii, T in enumerate(self.sub):
                nc[ii] = self._form(u, T['nc'], u)
                rr, cc, M = T['r_fd']
                r[ii] = est.local_eta_rf_squared[ii] - 2.0 * float(M[0] @ ur[cc]) + self._form(ur, T['r_dd'], ur)
                df[ii] = sum(c.evaluate(mu) * self._form(u, R, u) for c, R in T['df_aa']) + self._form(ur, T['df_bb'], ur) + \
                    2.0 * sum(c.evaluate(mu) * self._form(u, R, ur) for c, R in T['df_ab'])
                r[ii] *= (1.0 / np.pi ** 2) / est.min_diffusion_evs[ii] * est.subdomain_diameters[ii] ** 2
            a_bar = est.alpha(est.lambda_coeffs, mu, est.mu_bar)
            g_bar = est.gamma(est.lambda_coeffs, mu, est.mu_bar)
            a_hat = est.alpha(est.lambda_coeffs, mu, est.mu_hat)
            out.append((np.sqrt(g_bar) * np.linalg.norm(nc) + np.linalg.norm(r + df) / np.sqrt(a_hat)) / np.sqrt(a_bar))
        return out


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core the BLAS can take."""
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        pass


def cpu_threads():
    try:
        from threadpoolctl import threadpool_info
        n = max([p.get('num_threads', 1) for p in threadpool_info()] + [1])
        return int(n)
    except Exception:
        return os.cpu_count() or 1


def run_reference(a):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    use_all_host_threads()
    rd, t_off = cpu_reference_model(a)
    mus = make_mus(a, 0, a.cpu_sample)
    for _ in range(max(1, a.warmup) if a.warmup else 0):
        cpu_online_step(rd, mus[:max(1, a.cpu_sample // 4)])
    t = time.perf_counter()
    for _ in range(a.steps):
        cpu_online_step(rd, mus)
    dt = time.perf_counter() - t
    value = a.cpu_sample * a.steps / dt
    cores = cpu_threads()
    sample = '{} parameters per step of the same reduced model (n_red={}), dense unblocked operators, numpy.linalg.solve + ' \
             '6 quadratic forms per subdomain per parameter'.format(a.cpu_sample, rd.solution_space.dim)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': a.gpus, 'steps': a.steps,
        'warmup': a.warmup, 'ms_per_step': 1e3 * dt / a.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': workload_name(a), 'cpu_sample_mu_per_step': a.cpu_sample,
                   'note': 'pyMOR/DUNE are not installable here; this is the NumPy/SciPy restatement of the reference path (oracle/)'},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample,
                         'offline_reduce_s': t_off},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------
#  B200 arm
# ----------------------------------------------------------------------------------------------------------

def measure_fp64_gemm_peak(torch):
    """cuBLAS DGEMM 4096^3, best of 5 (burst) -- the FP64 tensor-pipe denominator; MEASURED_PEAKS.json has no FP64 figure."""
    n = 4096
    a = torch.randn((n, n), dtype=torch.float64, device='cuda')
    b = torch.randn((n, n), dtype=torch.float64, device='cuda')
    torch.matmul(a, b)
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record(); e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def measured_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            p = json.load(f)
        return float(p['hbm_gbs']), 'MEASURED_PEAKS.json hbm_gbs (measured)'
    except Exception:
        return 6650.0, 'fallback 6.65 TB/s (B200_PROFILING.md)'


def offline_workload_name(a):
    if a.synthetic3d:
        return workload_name(a)
    return '{0} {1}x{1} subdomains, n_i={2}, N={3}, Q=2 (offline)'.format(problem_name(a), a.subdomains, 6 * a.cells ** 2, a.basis)


def measure_offline(a, torch, planner, d, bases, fp64_peak, flush_l2, t_reduce_first, reductor):
    """Kernel-only timing of the batched projection (inputs resident in HBM) + the wall time of reductor.reduce()."""
    from pylrbms_b200 import LRBMSReductor
    st = planner.stats()
    for _ in range(max(3, a.warmup)):
        planner.run()
    times_all, times_proj = [], []
    for _ in range(a.steps):
        flush_l2()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        planner.spmm_plans[0].run()        # stage 0: Oswald / flux-reconstruction images of the bases (rows a2, a3)
        e1.record()
        for p in planner.spmm_plans[1:]:   # later stages belong to the projection: D R, and A^T L of the narrow-left chains
            p.run()
        planner.project_plan.run()
        e2.record()
        e2.synchronize()
        times_all.append(e0.elapsed_time(e2)); times_proj.append(e1.elapsed_time(e2))
    hbm_peak, hbm_src = measured_peaks()
    pp = planner.project_plan
    t_proj = float(np.mean(times_proj)) * 1e-3
    # EXECUTED work of the plan that was timed: the later SpMM stages + the projection plan (tight byte count: every array
    # once).  This is what `frac` is computed from.  The SURVEY section 8d formulation (every operator chain applied matrix by
    # matrix to the right-hand array, as the reference defines the operators) asks for more flops than the restructured plan
    # executes; it is reported as an aside (`*_survey_formulation`), not as the roofline fraction.
    ex_flops = pp.flops + sum(p.flops for p in planner.spmm_plans[1:])
    ex_bytes = pp.algorithmic_bytes + sum(p.algorithmic_bytes for p in planner.spmm_plans[1:])
    acct = LRBMSReductor(d, bases=bases)
    acct.fuse_chains, acct.narrow_left = False, False
    acct_plan = acct.build_plan()
    sv_bytes = acct_plan.project_plan.algorithmic_bytes_survey
    sv_flops = acct_plan.project_plan.flops
    del acct, acct_plan
    tfs, gbs = ex_flops / t_proj / 1e12, ex_bytes / t_proj / 1e9
    ai = ex_flops / ex_bytes
    crossover = fp64_peak * 1e12 / (hbm_peak * 1e9)
    tensor_bound = ai > crossover
    roof = {'bound': 'tensor' if tensor_bound else 'hbm',
            'kernel': 'projection plan (all buckets of one run: spmm_kernel, project_kernel, gram_kernel)',
            'achieved': tfs if tensor_bound else gbs, 'peak': fp64_peak if tensor_bound else hbm_peak,
            'unit': 'TFLOP/s' if tensor_bound else 'GB/s',
            'frac': tfs / fp64_peak if tensor_bound else gbs / hbm_peak,
            'traffic': ncu_traffic('projection_plan', offline_workload_name(a)),
            'peak_source': 'cuBLAS DGEMM 4096^3 measured in this run (FP64 tensor pipe)' if tensor_bound else hbm_src,
            'counts': 'executed by the timed plan', 'flops': ex_flops, 'bytes': ex_bytes,
            'arithmetic_intensity_flop_per_byte': ai, 'crossover_flop_per_byte': crossover,
            'fp64_tflops': tfs, 'fp64_peak_tflops': fp64_peak, 'fp64_frac': tfs / fp64_peak,
            'hbm_gbs': gbs, 'hbm_peak_gbs': hbm_peak, 'hbm_frac': gbs / hbm_peak, 'hbm_peak_source': hbm_src,
            'survey_formulation': {'flops': sv_flops, 'bytes': sv_bytes, 'fp64_frac': sv_flops / t_proj / 1e12 / fp64_peak,
                                   'hbm_frac': sv_bytes / t_proj / 1e9 / hbm_peak,
                                   'note': 'SURVEY 8d work count of the operators as the reference defines them; the plan '
                                           'executes less (fused chains, narrow-left), so this is not a kernel efficiency'}}
    # end to end through the public API: reductor.reduce() from the bases to a reduced model whose blocks are readable
    reductor.reuse_plan = False
    t_e2e = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rd_ = reductor.reduce()
        rd_.operator.operators[0].sblocks[0]            # reduced blocks live in rd_'s buffer
        torch.cuda.synchronize()
        t_e2e.append(time.perf_counter() - t0)
    return {
        'metric': 'offline projection HBM GB/s', 'unit': 'GB/s', 'value': sv_bytes / t_proj / 1e9,
        'value_note': 'BASELINE metric: SURVEY 8d algorithmic bytes / projection time; roofline.frac uses executed counts',
        'workload': offline_workload_name(a),
        'ms_all_stages': float(np.mean(times_all)), 'ms_projection': float(np.mean(times_proj)),
        'ms_projection_covers': 'SpMM stages >= 1 (divergence images, A^T L of narrow-left chains) + the projection plan; '
                                'stage 0 (Oswald / flux-reconstruction images of the bases) is the rest of ms_all_stages',
        'projection_descriptors': planner.n_project_descs, 'spmm_descriptors': planner.n_spmm_descs,
        'launches_per_reduce': st['launches'], 'roofline': roof,
        'e2e': {'api': 'LRBMSReductor.reduce()', 'first_call_s': t_reduce_first, 'repeat_call_s': float(np.min(t_e2e)),
                'what': 'wall time incl. host planning, plan creation and all kernels; first call also pays one-off operator '
                        'preparation (fused chain products, transposes) and CUDA module load'},
    }


def measure_sharded_offline(a, torch, dist, d, bases, flush_l2, barrier, ms_unsharded, label):
    """Strong scaling of the offline half: the same operator set, subdomains split over the ranks, reduced regions exchanged
    over peer memory (NCCL all-gather timed beside it).  The gathered buffer must equal the unsharded result bit for bit (checked here)."""
    from pylrbms_b200 import LRBMSReductor
    world = dist.get_world_size()
    red_s = LRBMSReductor(d, bases=bases, shard=True)
    red_s.reduce()
    ps = red_s.last_plan
    for _ in range(3):
        ps.run(); ps.exchange()
    t_run, t_all = [], []
    for _ in range(a.steps):
        flush_l2()
        barrier()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        ps.run()
        e1.record()
        ps.exchange()
        e2.record()
        e2.synchronize()
        t_run.append(e0.elapsed_time(e1)); t_all.append(e0.elapsed_time(e2))
    # the same exchange through NCCL (one in-place all-gather), timed beside the peer-memory path
    from pylrbms_b200.distributed import exchange_kind, exchange_regions
    t_nccl = []
    for it in range(3 + a.steps):
        flush_l2()
        barrier()
        e0, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(2))
        e0.record()
        exchange_regions(ps.out, ps.region_starts)
        e1.record()
        e1.synchronize()
        if it >= 3:
            t_nccl.append(e0.elapsed_time(e1))
    tt = torch.tensor([float(np.mean(t_run)), float(np.mean(t_all)), float(np.mean(t_nccl))], dtype=torch.float64, device='cuda')
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    # bitwise check against the unsharded projection of the same bases on this rank
    red_u = LRBMSReductor(d, bases=bases)
    rd_u = red_u.reduce()
    rd_s = red_s.reduce()
    same = True
    for name in ('operator', 'nc_0', 'r_dd_%d' % (len(rd_u.block_dims) - 1)):
        ou, os_ = rd_u.operators[name], rd_s.operators[name]
        for gu, gs in zip(getattr(ou, 'operators', [ou]), getattr(os_, 'operators', [os_])):
            same = same and bool(np.array_equal(gu.to_dense(), gs.to_dense()))
    flag = torch.tensor([1.0 if same else 0.0], dtype=torch.float64, device='cuda')
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if flag.item() != 1.0:
        raise SystemExit('bench.py: sharded offline projection differs from the unsharded one')
    return {
        'workload': label, 'n_gpus': world, 'scaling': 'strong', 'partition': 'contiguous strips of subdomains per rank',
        'ms_all_stages_max_over_ranks': float(tt[0].item()), 'ms_with_exchange_max_over_ranks': float(tt[1].item()),
        'ms_all_stages_1gpu_unsharded_this_rank': ms_unsharded,
        'speedup_vs_unsharded': ms_unsharded / float(tt[0].item()),
        'speedup_vs_unsharded_incl_exchange': ms_unsharded / float(tt[1].item()),
        'exchange': '%s; equal-stride rank regions, %d doubles in total' % (exchange_kind(), int(ps.out.numel())),
        'ms_exchange_max_over_ranks': float(tt[1].item()) - float(tt[0].item()),
        'ms_exchange_nccl_all_gather_max_over_ranks': float(tt[2].item()),
        'bitwise_equal_to_unsharded': True,
        'projection_descriptors_this_rank': ps.n_project_descs,
    }


def parity_gate(a, rd, mus_all, rd_ref=None):
    """BASELINE.md section 2: no timing counts without parity.  The reduced model the GPU arm just timed is compared with the
    oracle's on the same inputs: every reduced operator / product (max-norm, relative to the operator), and for a sample of
    the benchmark's own parameters u(mu) in the energy norm, eta and its three parts -- through ``sweep_into`` (the e2e
    entry point) and ``sweep``.  Raises SystemExit on failure."""
    from oracle.parity import RTOL, compare_online, compare_operators, reference_online
    import torch
    if rd_ref is None:
        rd_ref = cpu_reference_model(a)
    rd_ref_pair, rd_ref = rd_ref, rd_ref[0]
    worst, checked = 0.0, 0
    for name, err in compare_operators(rd, rd_ref).items():
        if not err <= RTOL:
            raise SystemExit('bench.py: PARITY FAILURE, reduced operator {}: rel err {:.3e}'.format(name, err))
        worst, checked = max(worst, err), checked + 1
    n = a.cpu_sample
    mus = np.asarray(mus_all[:n])
    ref = reference_online(rd_ref, mus)
    u_host = torch.empty((n, rd.n_red), dtype=torch.float64).pin_memory()
    eta_host = torch.empty(n, dtype=torch.float64).pin_memory()
    if rd.sweep_into(mus, u_host, eta_host) != 0:
        raise SystemExit('bench.py: PARITY FAILURE, a reduced system was flagged as not positive definite')
    e1 = compare_online(rd, rd_ref, mus, U=u_host.numpy(), eta=eta_host.numpy(), ref=ref)
    e2 = compare_online(rd, rd_ref, mus, ref=ref)
    for tag, errs in (('sweep_into', e1), ('sweep', e2)):
        for name, err in errs.items():
            if name.endswith('_plain') or name == 'cancellation':
                continue
            lim = RTOL
            if not err <= lim:
                raise SystemExit('bench.py: PARITY FAILURE, {} {}: rel err {:.3e}'.format(tag, name, err))
            worst, checked = max(worst, err), checked + n
    return {'max_rel': worst, 'checked': checked, 'tol': RTOL, 'n_mu': n, 'by_quantity': {'sweep_into': e1, 'sweep': e2}, 'reduced_operators': len(rd_ref.operators) + len(rd_ref.products),
            'what': 'every reduced operator and product vs the oracle (max-norm rel.); u(mu) in the energy norm, eta, nc / r / df '
                    'and indicators for the first {} benchmark parameters, through ReducedModel.sweep_into and .sweep'.format(n),
            'oracle': "oracle/: restatement of the reference's reductor.py / estimators.py, bit-identical to those files executed "
                      "unmodified on stand-ins for pyMOR / dune-gdt (oracle/reference_run.py, tests/golden/reference_run__*.npz)"}, rd_ref_pair


def sparse_solve_gate(rd, mus, n_check=2):
    """Configurations the oracle cannot hold (its dense unblocked storage, SURVEY.md row a10): the solutions the GPU arm just
    timed are checked against an independent CPU solver -- SciPy's SuperLU on the block-sparse reduced operator assembled
    on the host from the projected blocks -- in the energy norm (1e-10), plus the residual.  The projected blocks themselves
    are covered against the oracle by the -m gpu tests at these block sizes (tests/test_gpu_configs.py)."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spl
    offs = np.concatenate([[0], np.cumsum(rd.block_dims)])
    mats = []
    for op in rd.operator.operators:
        rows, cols, vals = [], [], []
        for (i, j), B in op.blocks().items():
            r, c = np.meshgrid(np.arange(offs[i], offs[i + 1]), np.arange(offs[j], offs[j + 1]), indexing='ij')
            rows.append(r.ravel()); cols.append(c.ravel()); vals.append(B.ravel())
        mats.append(sp.csc_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(rd.n_red,) * 2))
    f_terms = [o.to_dense()[0] for o in rd.rhs.operators]
    pick = np.linspace(0, len(mus) - 1, n_check).astype(int)
    U, eta = rd.sweep(np.asarray(mus)[pick])
    worst_e, worst_r = 0.0, 0.0
    for k, m in enumerate(pick):
        th = rd.thetas([mus[m]])[0]
        A = sum(t * M for t, M in zip(th[:len(mats)], mats)).tocsc()
        f = sum(t * v for t, v in zip(th[len(mats):], f_terms))
        lu = spl.splu(A)
        u_ref = lu.solve(f)
        u_ref += lu.solve(f - A @ u_ref)
        e = U.data[k] - u_ref
        worst_e = max(worst_e, float(np.sqrt(e @ (A @ e)) / np.sqrt(u_ref @ (A @ u_ref))))
        worst_r = max(worst_r, float(np.linalg.norm(A @ U.data[k] - f) / np.linalg.norm(f)))
    if not (worst_e <= 1e-10 and np.all(np.isfinite(eta)) and np.all(eta > 0)):
        raise SystemExit('bench.py: PARITY FAILURE against the CPU sparse solve: energy-norm error {:.3e}'.format(worst_e))
    return {'max_rel': worst_e, 'checked': int(n_check), 'tol': 1e-10, 'kind': 'independent CPU sparse direct solve (SciPy SuperLU) on the '
            'same block-sparse reduced operator, energy norm; the oracle cannot hold this configuration (dense unblocked storage)',
            'residual_rel': worst_r}


DUMP_BYTES = 48 << 20          # --dump-outputs stays below 64 MB in all


def dump_outputs(out_dir, mus, u, eta, info, mx, am):
    """Write what one online step returned -- reduced solutions ``u`` (n_mu x n_red), ``eta``, the factorisation flags
    ``info`` and ``eta_max`` = [max, argmax] -- with the parameters ``mu`` they belong to, as float64 ``<name>.npy`` files.
    When every parameter's row does not fit ``DUMP_BYTES``, the rows of a fixed, seeded sample of the parameters are
    written (their positions in the batch are ``index``), so that two runs with the same arguments compare row for row."""
    import torch
    n_mu, n_red = u.shape
    rows = max(1, DUMP_BYTES // (8 * (n_red + 4)))
    idx = np.arange(n_mu) if rows >= n_mu else np.sort(np.random.default_rng(0).choice(n_mu, rows, replace=False))
    sel = torch.from_numpy(idx).to(u.device)
    arrays = {'index': idx.astype(np.float64), 'mu': np.asarray(mus, dtype=np.float64)[idx],
              'u': u.index_select(0, sel).cpu().numpy(), 'eta': eta.index_select(0, sel).cpu().numpy(),
              'info': info.index_select(0, sel).cpu().numpy().astype(np.float64),
              'eta_max': np.array([float(mx.item()), float(am.item())])}
    os.makedirs(out_dir, exist_ok=True)
    for name, x in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), x)


def run_b200(a):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device -- the B200 path has no CPU fallback (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from pylrbms_b200 import build
    build.build()
    from pylrbms_b200 import LRBMSReductor, discretize

    # ---- setup (untimed): host assembly, upload, offline reduction -- every rank holds the full (small) reduced model
    data, bases = make_inputs(a)
    d, _ = discretize(data)
    reductor = LRBMSReductor(d, bases=bases)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rd = reductor.reduce()
    torch.cuda.synchronize()
    t_reduce_first = time.perf_counter() - t0
    planner = reductor.last_plan
    rd.online_plan                                     # build the online plan (symbolic phase + operator upload)

    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device='cuda')     # 256 MB > 126 MB L2
    fp64_peak = measure_fp64_gemm_peak(torch)

    def flush_l2():
        flush.fill_(1.0)

    # ---- offline half: the batched projection of every operator
    offline = None
    if not a.no_offline:
        offline = measure_offline(a, torch, planner, d, bases, fp64_peak, flush_l2, t_reduce_first, reductor)
        rd = reductor.reduce()                         # (measure_offline re-ran reduce(): keep the model of the last plan)
        rd.online_plan
        if world > 1:
            offline['sharded'] = measure_sharded_offline(a, torch, dist, d, bases, flush_l2, barrier, offline['ms_all_stages'],
                                                         offline_workload_name(a))
        if world > 1 and a.c3_sharded and not a.synthetic3d and (a.problem, a.subdomains) != ('spe10', 16):
            # configs[2]: high-contrast SPE10-like field on 16 x 16 subdomains, offline projection + estimator Grams at N GPUs
            import copy
            a3 = copy.copy(a)
            a3.problem, a3.subdomains = 'spe10', 16
            data3, bases3 = make_inputs(a3)
            d3, _ = discretize(data3)
            red3 = LRBMSReductor(d3, bases=bases3)
            red3.reduce()
            p3 = red3.last_plan
            for _ in range(3):
                p3.run()
            t3 = []
            for _ in range(a.steps):
                flush_l2()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); p3.run(); e1.record(); e1.synchronize()
                t3.append(e0.elapsed_time(e1))
            del red3, p3
            offline['sharded_c3'] = measure_sharded_offline(a3, torch, dist, d3, bases3, flush_l2, barrier, float(np.mean(t3)),
                                                            offline_workload_name(a3))
            del d3, data3, bases3
            torch.cuda.empty_cache()
    if a.offline_only:
        if rank == 0:
            print(json.dumps({'metric': 'offline projection HBM GB/s', 'value': offline['value'], 'unit': 'GB/s', 'n_gpus': world,
                              'dtype': 'f64', 'data': 'synthetic', 'config': {'workload': offline_workload_name(a)},
                              'higher_is_better': True, 'offline': offline}))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- online half
    n_mu = a.n_mu
    mus = make_mus(a, rank, n_mu, data)
    theta = torch.from_numpy(rd.thetas(mus)).cuda()
    u = torch.empty((n_mu, rd.n_red), dtype=torch.float64, device='cuda')
    eta = torch.empty(n_mu, dtype=torch.float64, device='cuda')
    info = torch.empty(n_mu, dtype=torch.int32, device='cuda')
    rd._workspace(n_mu)

    def step():
        rd.solve_device(theta, u, info)
        ev_mid = torch.cuda.Event(enable_timing=True); ev_mid.record()
        rd.estimate_device(theta, u, eta)
        mx, am = rd.eta_max_device(eta)
        if world > 1:
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        return ev_mid, mx, am

    for _ in range(max(3, a.warmup)):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t_step, t_solve = [], []
    barrier()
    for _ in range(a.steps):
        flush_l2()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ev_mid, mx, am = step()
        e1.record()
        e1.synchronize()
        t_step.append(e0.elapsed_time(e1)); t_solve.append(e0.elapsed_time(ev_mid))
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, mus, u, eta, info, mx, am)
    if int(info.abs().max().item()) != 0:
        raise SystemExit('bench.py: a reduced system was flagged as not positive definite')
    total_ms = torch.tensor([float(np.sum(t_step))], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_s = float(total_ms.item()) * 1e-3
    value = world * n_mu * a.steps / total_s

    # ---- end to end through the public API: host parameters -> host results, copies inside the timed region
    e2e_steps = a.steps
    if a.eta_only:
        eta_host = torch.empty(n_mu, dtype=torch.float64).pin_memory()

        def e2e_call():
            bad, mx_, am_ = rd.sweep_eta_into(mus, eta_host)
            return bad, mx_
        d2h = int(eta.numel() * 8)
        api = 'ReducedModel.sweep_eta_into(mus, eta_host)'
    else:
        u_host = torch.empty((n_mu, rd.n_red), dtype=torch.float64).pin_memory()
        eta_host = torch.empty(n_mu, dtype=torch.float64).pin_memory()

        def e2e_call():
            bad = rd.sweep_into(mus, u_host, eta_host)
            return bad, float(eta_host.max())
        d2h = int((u.numel() + eta.numel()) * 8)
        api = 'ReducedModel.sweep_into(mus, u_host, eta_host)'
    for _ in range(2):
        e2e_call()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        bad, mx_ = e2e_call()
        if bad:
            raise SystemExit('bench.py: a reduced system was flagged as not positive definite (e2e)')
        if world > 1:
            m = torch.tensor([mx_], dtype=torch.float64, device='cuda')
            dist.all_reduce(m, op=dist.ReduceOp.MAX)
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * n_mu * e2e_steps / float(e2e_s.item())

    # ---- configs[4]: the 1M-parameter sweep, 125 000 parameters per GPU, estimator-max gather, eta-only results
    c5 = None
    if a.c5 and not a.synthetic3d:
        n5 = 125000
        mus5 = make_mus(a, 100 + rank, n5, data)
        eta5 = torch.empty(n5, dtype=torch.float64).pin_memory()
        from pylrbms_b200.distributed import gather_estimator_max

        def c5_call():
            bad5, mx5, am5 = rd.sweep_eta_into(mus5, eta5)
            if bad5:
                raise SystemExit('bench.py: a reduced system was flagged as not positive definite (C5)')
            lo5 = rank * n5
            return gather_estimator_max(torch.tensor([mx5], dtype=torch.float64, device='cuda'),
                                        torch.tensor([am5], dtype=torch.int64, device='cuda'), lo5)
        c5_call()
        barrier()
        t0 = time.perf_counter()
        reps5 = a.steps
        for _ in range(reps5):
            gmax, garg = c5_call()
        barrier()
        t5 = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t5, op=dist.ReduceOp.MAX)
        c5 = {'workload': '{} parameters ({} per GPU), 64 subdomains, estimator-max gather'.format(world * n5, n5),
              'value': world * n5 * reps5 / float(t5.item()), 'unit': UNIT, 'n_gpus': world,
              'api': 'ReducedModel.sweep_eta_into + distributed.gather_estimator_max (one all-gather of (max, argmax) pairs per sweep)',
              'h2d_bytes_per_sweep': int(n5 * theta.shape[1] * 8), 'd2h_bytes_per_sweep': int(n5 * 8),
              'eta_max': gmax, 'argmax_global': garg, 'seconds_per_sweep': float(t5.item()) / reps5}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel: the solve kernel the plan selected (name, flop count from the library)
    fl = survey_flops_per_mu(a, data, rd)
    solve_s = float(np.mean(t_solve)) * 1e-3
    achieved = fl['solve'] * n_mu / solve_s / 1e12
    solve_name = rd.solve_kernel_name
    executed = rd.solve_flops_executed
    roofline = {'bound': 'tensor', 'kernel': solve_name, 'achieved': achieved, 'peak': fp64_peak, 'unit': 'TFLOP/s',
                'frac': achieved / fp64_peak,
                'traffic': ncu_traffic(solve_name, workload_name(a)),
                'peak_source': 'cuBLAS DGEMM 4096^3 measured in this run (FP64; MEASURED_PEAKS.json has no FP64 figure)',
                'algorithmic_flops_per_mu': fl['solve'], 'executed_flops_per_mu': executed,
                'executed_tflops': executed * n_mu / solve_s / 1e12, 'executed_frac': executed * n_mu / solve_s / 1e12 / fp64_peak,
                'ms_per_launch': 1e3 * solve_s, 'share_of_step': float(np.sum(t_solve) / np.sum(t_step))}

    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps, 'warmup': max(3, a.warmup),
        'ms_per_step': 1e3 * total_s / a.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': workload_name(a), 'n_red': fl['n_red'], 'reduced_blocks': fl['blocks'],
                   'half_bandwidth': rd.half_bandwidth,
                   'l2': 'flushed between timed steps (256 MB write); factor scratch per step also exceeds L2',
                   'parallelism': 'mu-sharded x{}'.format(world), 'flops_per_mu_survey': fl['total']},
        'clocks': clocks,
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': int(theta.numel() * 8),
                'd2h_bytes_per_step': d2h, 'api': api},
        'gpu_launches': int(a.steps * gpu_launches_per_step(rd)),
        'roofline': roofline,
        'offline': offline,
    }
    if c5 is not None:
        line['c5_sweep'] = c5
    rd_ref = None
    if not a.no_parity and not a.synthetic3d and oracle_feasible(a):
        line['parity'], rd_ref = parity_gate(a, rd, mus)
    elif not a.no_parity:
        line['parity'] = sparse_solve_gate(rd, mus)
    if not a.no_cpu_baseline and world == 1 and oracle_feasible(a):
        line['cpu_baseline'] = cpu_baseline(a, rd_ref)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def oracle_feasible(a):
    """The reference-faithful oracle stores every reduced operator as an unblocked dense matrix (SURVEY.md row a10):
    ~5 GB at 8x8 subdomains, N = 20; beyond ~100 subdomains it does not fit a host."""
    return a.subdomains ** 2 * a.basis <= 2000 and not a.synthetic3d


def gpu_launches_per_step(rd):
    """Kernels of this repo launched per timed step: the solve (1 launch for the CTA-per-parameter kernels, 3 per block column
    + 2 per chunk for the band solver), estimate_kernel, combine_kernel, eta_max_kernel."""
    return int(rd.online_plan.info(0)) + 1


def cpu_baseline(a, rd_ref=None):
    use_all_host_threads()
    rd, t_off = rd_ref if rd_ref is not None else cpu_reference_model(a)
    mus = make_mus(a, 0, a.cpu_sample)
    cpu_online_step(rd, mus[:2])
    t = time.perf_counter()
    cpu_online_step(rd, mus)
    dt = time.perf_counter() - t
    # variant (ii) of SURVEY.md section 8d: banded Cholesky + restricted estimator forms; checked against variant (i)
    vm = VectorisedCpuModel(rd)
    ref = cpu_online_step(rd, mus[:2])
    got = vm.step(mus[:2])
    assert np.allclose(got, ref, rtol=1e-9, atol=0.0), (got, ref)
    n_vec = 8 * a.cpu_sample
    mus_v = make_mus(a, 1, n_vec)
    t = time.perf_counter()
    vm.step(mus_v)
    dt_v = time.perf_counter() - t
    return {'value': a.cpu_sample / dt, 'unit': UNIT, 'cores': cpu_threads(), 'kind': 'port',
            'sample': '{} parameters of the same workload, one at a time as the reference does (dense unblocked operators, '
                      'numpy.linalg.solve, 6 quadratic forms per subdomain)'.format(a.cpu_sample),
            'offline_reduce_s': t_off,
            'vectorised': {'value': n_vec / dt_v, 'unit': UNIT, 'sample': '{} parameters'.format(n_vec),
                           'what': 'same reduced model, banded Cholesky (scipy.linalg.solveh_banded, half-bandwidth {}) and estimator '
                                   'forms restricted to the rows / columns they touch; agrees with the reference-faithful variant to '
                                   '1e-9'.format(vm.b)}}


if __name__ == '__main__':
    args = parse_args()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)
