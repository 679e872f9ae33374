"""The online estimator (``estimate_kernel<kTMU>`` + ``combine_kernel``) against the exactly rounded reference of
``oracle/exact_forms.py``, at every tile width, through the C ABI; plan coexistence (the kernels' shared-memory limits);
``lrbms_eta_max``; and at C2 the split of the GPU / oracle difference into evaluation error on each side and input difference.

Rounding bound of the kernel (``online.cu`` estimate_kernel), per subdomain: each product ``c x_r M_rk y_k`` passes at most

    K = kend + 1      the DMMA k loop over the right vector, padded to a multiple of 4, + 1 for theta_q u_k staged rounded
      + 1 + 1         the left vector's own theta_q u_k rounding, the product with the left vector
      + 3             the 8-row shuffle reduction of a tile
      + 3             coef * theta_a * theta_b and the product with the tile's dot
      + n_w           the per-warp accumulation over that warp's (term, 8-row tile) items, n_w = ceil(tiles / 16)
      + 16            the cross-warp sum over the 16 warps
      + 2             r only: + ||f||^2, * r_scale

roundings, so ``|got - exact| <= gamma_K S`` with ``gamma_K = K u / (1 - K u)``, ``u = 2^-53`` and ``S`` the part summed over
absolute values (``EstimatorForms.evaluate``'s ``S_*``).
"""
import ctypes as C

import numpy as np
import pytest

from oracle import exact_forms as X
from test_gpu_kernels import _random_reduced_system, dev

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
EPS = 2.0 ** -52
PARTS = ('nc', 'r', 'df')


def _torch():
    import torch
    return torch


def gamma(k):
    k = np.asarray(k, dtype=np.float64)
    return k * U / (1.0 - k * U)


def kernel_K(forms, sizes, nbh, Q):
    """``(3, S)``: the K of the module docstring per part and subdomain."""
    dsub = [sum(sizes[k] for k in nbh[i]) for i in range(len(sizes))]
    tiles = np.zeros(len(sizes), dtype=np.int64)
    kend = np.zeros(len(sizes), dtype=np.int64)
    for (part, sub, left, right, factors, M) in forms.forms:
        tiles[sub] += (M.shape[0] + 7) // 8
        kend[sub] = max(kend[sub], (M.shape[1] + 3) // 4 * 4)
    K = (kend + 1) + (1 + 1) + 3 + 3 + (tiles + 15) // 16 + 16
    return np.stack([K, K + 2, K])


# ------------------------------------------------------------------------------------------------------------
#  C-ABI plans with explicit estimator terms
# ------------------------------------------------------------------------------------------------------------

def _chain_system(rng, sizes, Q, Qf):
    """Subdomains on a chain (k couples to k - 1 and k + 1): neighbourhoods of two or three members, ragged."""
    return _random_reduced_system(rng, len(sizes), 1, list(sizes), Q=Q, Qf=Qf,
                                  couplings=[(k + 1, k) for k in range(len(sizes) - 1)])


def _plan(handle, sysd, terms, rf2, rsc, tbar, that, alpha_first, solver=0):
    from pylrbms_b200 import _lib as L
    S, sizes, off, blocks, Q, Qf = sysd['S'], sysd['sizes'], sysd['off'], sysd['blocks'], sysd['Q'], sysd['Qf']
    bi = L.host_i32([b[0] for b in blocks]); bj = L.host_i32([b[1] for b in blocks])
    packed, offsets, pos = [], np.zeros(Q * len(blocks), dtype=np.int64), 0
    for q in range(Q):
        for b, (i, j) in enumerate(blocks):
            blk = sysd['dense'][q][off[i]:off[i + 1], off[j]:off[j + 1]]
            offsets[q * len(blocks) + b] = pos
            packed.append(blk.ravel())
            pos += blk.size
    d_blocks, d_rhs = dev(np.concatenate(packed)), dev(sysd['rhs'])
    nbh_ptr = L.host_i32(np.concatenate([[0], np.cumsum([len(x) for x in sysd['nbh']])]))
    nbh_idx = L.host_i32(np.concatenate(sysd['nbh']))
    sysc = L.ReducedSystem()
    sysc.n_sub = S; sysc.basis_sizes = sizes.ctypes.data; sysc.Q = Q; sysc.Qf = Qf; sysc.n_blocks = len(blocks)
    sysc.block_i = bi.ctypes.data; sysc.block_j = bj.ctypes.data; sysc.block_offset = offsets.ctypes.data
    sysc.lhs_blocks = d_blocks.data_ptr(); sysc.rhs = d_rhs.data_ptr()
    sysc.nbh_ptr = nbh_ptr.ctypes.data; sysc.nbh_idx = nbh_idx.ctypes.data
    sysc.solver = solver
    keep = [bi, bj, offsets, d_blocks, d_rhs, nbh_ptr, nbh_idx, sizes]
    if terms:
        mats, carr, moff = [], [], 0
        for (i, out, lk, rk, qa, qb, coef, M) in terms:
            mats.append(np.ascontiguousarray(M, dtype=np.float64).ravel())
            carr.append(L.EstimatorTerm(i, out, lk, rk, M.shape[0], M.shape[1], qa, qb, coef, moff))
            moff += M.size
        d_mats = dev(np.concatenate(mats))
        tarr = (L.EstimatorTerm * len(carr))(*carr)
        rf2h, rsch, tb, th = L.host_f64(rf2), L.host_f64(rsc), L.host_f64(tbar), L.host_f64(that)
        sysc.n_terms = len(carr); sysc.terms = C.cast(tarr, C.c_void_p); sysc.est_matrices = d_mats.data_ptr()
        sysc.rf_squared = rf2h.ctypes.data; sysc.r_scale = rsch.ctypes.data
        sysc.theta_bar = tb.ctypes.data; sysc.theta_hat = th.ctypes.data
        sysc.alpha_returns_first = alpha_first
        keep += [d_mats, tarr, rf2h, rsch, tb, th]
    p = C.c_void_p()
    handle.check(handle.lib.lrbms_online_plan_create(handle.h, C.byref(sysc), C.byref(p)))
    return L.Plan(handle, p, keep)


def _estimate(handle, plan, theta, u, S, poison=True):
    """``lrbms_online_estimate`` on the given ``theta (n_mu, Q + Qf)`` and ``u (n_mu, n_red)``: ``(parts, eta, indicators)``."""
    from pylrbms_b200._lib import current_stream_ptr, ptr
    torch = _torch()
    n_mu = theta.shape[0]
    ws = C.c_size_t()
    handle.check(handle.lib.lrbms_online_workspace_bytes(plan.p, n_mu, C.byref(ws)))
    work = torch.empty(max(ws.value, 8), dtype=torch.uint8, device='cuda')
    eta = torch.full((n_mu,), np.nan, dtype=torch.float64, device='cuda')
    parts = torch.full((3, S, n_mu), np.nan, dtype=torch.float64, device='cuda')
    ind = torch.full((S, n_mu), np.nan, dtype=torch.float64, device='cuda')
    d_theta, d_u = dev(theta), dev(u)
    if poison:
        handle.check(handle.lib.lrbms_debug_poison_shared(handle.h, current_stream_ptr()))
    handle.check(handle.lib.lrbms_online_estimate(plan.p, n_mu, ptr(d_theta), ptr(d_u), ptr(eta), ptr(parts), ptr(ind),
                                                  ptr(work), ws.value, current_stream_ptr()))
    torch.cuda.synchronize()
    return parts.cpu().numpy(), eta.cpu().numpy(), ind.cpu().numpy()


def _spec(Q):
    """The reference's term shapes (estimators.py:71-91): (out, left, right, qa, qb, coef)."""
    s = [(X.OUT_NC, X.VEC_UN, X.VEC_UN, -1, -1, 1.0), (X.OUT_R, X.VEC_ONE, X.VEC_UR, -1, -1, -2.0),
         (X.OUT_R, X.VEC_UR, X.VEC_UR, -1, -1, 1.0)]
    s += [(X.OUT_DF, X.VEC_UI, X.VEC_UI, a, b, 1.0) for a in range(Q) for b in range(Q)]
    s += [(X.OUT_DF, X.VEC_UR, X.VEC_UR, -1, -1, 1.0)]
    s += [(X.OUT_DF, X.VEC_UI, X.VEC_UR, a, -1, 2.0) for a in range(Q)]
    return s


def _dims(sizes, nbh, Q):
    dsub = [int(sum(sizes[k] for k in nbh[i])) for i in range(len(sizes))]
    return {X.VEC_ONE: lambda i: 1, X.VEC_UI: lambda i: int(sizes[i]), X.VEC_UN: lambda i: dsub[i],
            X.VEC_UR: lambda i: Q * dsub[i]}


def random_family(rng, sysd, n_mu):
    """Nothing cancels: positive matrices, solutions, coefficients; theta spread over two decades."""
    sizes, nbh, Q, Qf = sysd['sizes'], sysd['nbh'], sysd['Q'], sysd['Qf']
    dim = _dims(sizes, nbh, Q)
    terms = []
    for i in range(len(sizes)):
        for (out, lk, rk, qa, qb, coef) in _spec(Q):
            terms.append((i, out, lk, rk, qa, qb, abs(coef), rng.uniform(0.5, 1.5, (dim[lk](i), dim[rk](i)))))
    theta = 10.0 ** rng.uniform(-1.0, 1.0, (n_mu, Q + Qf))
    u = rng.uniform(0.5, 1.5, (n_mu, sysd['n']))
    rf2, rsc = rng.uniform(0.5, 1.5, len(sizes)), rng.uniform(0.1, 0.3, len(sizes))
    return terms, theta, u, rf2, rsc


def cancelling_family(rng, sysd, n_mu, delta=1e-3):
    """Estimator-shaped terms that cancel: ``RDD = B B^T``, ``r_fd = RDD x*``, ``rf2 = x*^T RDD x*`` and ``U_r`` within
    ``delta`` of ``x*``, so ``r = (U_r - x*)^T RDD (U_r - x*)`` is a small difference of large terms; ``df`` is the square
    ``|sum_a theta_a G_a u_i - H U_r|^2`` with ``H x* = sum_a theta*_a G_a u*_i``; ``nc = u^T (C C^T) u``."""
    sizes, nbh, Q, Qf, off = sysd['sizes'], sysd['nbh'], sysd['Q'], sysd['Qf'], sysd['off']
    S = len(sizes)
    th0 = rng.uniform(0.5, 2.0, Q + Qf)
    u0 = rng.standard_normal(sysd['n'])
    theta = th0 * (1.0 + delta * rng.uniform(-1, 1, (n_mu, Q + Qf)))
    u = u0 * (1.0 + delta * rng.uniform(-1, 1, (n_mu, sysd['n'])))
    terms, rf2 = [], np.zeros(S)
    for i in range(S):
        xs = np.concatenate([th0[q] * u0[off[k]:off[k + 1]] for k in nbh[i] for q in range(Q)])
        ui = u0[off[i]:off[i + 1]]
        n_r, n_i, d = len(xs), int(sizes[i]), len(xs) // Q
        B = rng.standard_normal((n_r, n_r)) / np.sqrt(n_r)
        RDD = B @ B.T
        terms.append((i, X.OUT_R, X.VEC_ONE, X.VEC_UR, -1, -1, -2.0, (RDD @ xs)[None, :]))
        terms.append((i, X.OUT_R, X.VEC_UR, X.VEC_UR, -1, -1, 1.0, RDD))
        rf2[i] = xs @ RDD @ xs
        Cm = rng.standard_normal((d, d)) / np.sqrt(d)
        terms.append((i, X.OUT_NC, X.VEC_UN, X.VEC_UN, -1, -1, 1.0, Cm @ Cm.T))
        G = [rng.standard_normal((n_i, n_i)) for _ in range(Q)]
        g = sum(th0[a] * G[a] @ ui for a in range(Q))
        H0 = rng.standard_normal((n_i, n_r)) / np.sqrt(n_r)
        H = H0 + np.outer(g - H0 @ xs, xs) / (xs @ xs)
        for a in range(Q):
            for b in range(Q):
                terms.append((i, X.OUT_DF, X.VEC_UI, X.VEC_UI, a, b, 1.0, G[a].T @ G[b]))
        terms.append((i, X.OUT_DF, X.VEC_UR, X.VEC_UR, -1, -1, 1.0, H.T @ H))
        for a in range(Q):
            terms.append((i, X.OUT_DF, X.VEC_UI, X.VEC_UR, a, -1, -2.0, G[a].T @ H))
    return terms, theta, u, rf2, rng.uniform(0.1, 0.3, S)


def _eta_from_parts(parts, theta, Q, tbar, that, alpha_first):
    """estimators.py:99-109 in float64 on the kernel's own parts."""
    rb, rh = theta[:, :Q] / np.asarray(tbar)[:Q], theta[:, :Q] / np.asarray(that)[:Q]
    a_bar = rb[:, 0] if alpha_first else rb.min(axis=1)
    a_hat = rh[:, 0] if alpha_first else rh.min(axis=1)
    g_bar = rb.max(axis=1)
    nc, rd = parts[0], parts[1] + parts[2]
    eta = (np.sqrt(g_bar) * np.sqrt(np.sum(nc * nc, axis=0)) + np.sqrt(np.sum(rd * rd, axis=0)) / np.sqrt(a_hat)) / np.sqrt(a_bar)
    ind = (2.0 / a_bar) * (g_bar * nc ** 2 + (1.0 / a_hat) * rd ** 2)
    return eta, ind


# (tile the plan must pick, Q, Qf, alpha_returns_first, basis sizes on a chain, n_mu)
TILE_CASES = [
    (64, 2, 1, 1, [37, 41, 39, 5], 3 * 64 + 17),        # largest neighbourhood 117 dofs
    (64, 2, 2, 0, [40, 41, 39], 1),
    (32, 1, 1, 0, [5, 11, 7, 3], 3 * 32 + 9),
    (32, 3, 2, 1, [9, 13, 6, 1, 8], 3 * 32 + 1),
    (32, 2, 1, 1, [3, 11, 7, 20, 1, 9], 1),
    (16, 2, 1, 0, [97, 103, 101], 3 * 16 + 5),
    (16, 3, 1, 1, [61, 73, 67], 3 * 16 + 11),
    (16, 1, 2, 1, [199, 201, 200], 1),
    (8, 2, 2, 1, [161, 173, 167], 3 * 8 + 5),
    (8, 3, 1, 0, [117, 119, 121], 3 * 8 + 3),
    (8, 2, 1, 0, [161, 173, 167], 1),
]


@pytest.mark.parametrize('family', ['random', 'cancelling'])
@pytest.mark.parametrize('tmu,Q,Qf,alpha_first,sizes,n_mu', TILE_CASES)
def test_estimator_against_exact_reference(handle, tmu, Q, Qf, alpha_first, sizes, n_mu, family):
    rng = np.random.default_rng([tmu, Q, Qf, alpha_first, sum(sizes), n_mu, family == 'random'])
    sysd = _chain_system(rng, sizes, Q, Qf)
    make = random_family if family == 'random' else cancelling_family
    terms, theta, u, rf2, rsc = make(rng, sysd, n_mu)
    tbar, that = rng.uniform(0.5, 1.5, Q), rng.uniform(0.5, 1.5, Q)
    plan = _plan(handle, sysd, terms, rf2, rsc, tbar, that, alpha_first)
    assert int(plan.info(9)) == tmu, 'plan picked {} parameters per CTA'.format(plan.info(9))
    S = len(sizes)
    parts, eta, ind = _estimate(handle, plan, theta, u, S)
    forms = X.terms_from_cabi(terms, sizes, sysd['nbh'], Q, rf2, rsc)
    ex = forms.evaluate(theta, u)
    K = kernel_K(forms, sizes, sysd['nbh'], Q)
    worst = {}
    for k, name in enumerate(PARTS):
        err = np.abs(parts[k] - ex[name])
        ratio = err / (EPS * ex['S_' + name])
        worst[name] = (float(ratio.max()), float((err / np.abs(ex[name])).max()))
        if family == 'random':
            assert np.all(err <= 1e-13 * np.abs(ex[name])), (name, float((err / np.abs(ex[name])).max()))
        assert np.all(err <= gamma(K[k][:, None]) * ex['S_' + name]), (name, float(ratio.max()))
    print('tile {} {}: |got - exact| / (eps S), rel:'.format(tmu, family), worst,
          'cancellation S / |r|: {:.1e}'.format(float((ex['S_r'] / np.abs(ex['r'])).max())))
    # eta and indicators from the kernel's own parts
    reta, rind = _eta_from_parts(parts, theta, Q, tbar, that, alpha_first)
    assert np.all(np.abs(eta - reta) <= 8 * EPS * np.abs(reta))
    assert np.all(np.abs(ind - rind) <= 8 * EPS * np.abs(rind))
    # batch composition: the same parameters permuted / in a smaller batch give bit-identical parts
    if n_mu > 1:
        perm = rng.permutation(n_mu)
        p2, e2, i2 = _estimate(handle, plan, theta[perm], u[perm], S)
        assert np.array_equal(p2, parts[:, :, perm]) and np.array_equal(e2, eta[perm]) and np.array_equal(i2, ind[:, perm])
        sub = perm[:max(1, n_mu // 3)]
        p3, e3, _ = _estimate(handle, plan, theta[sub], u[sub], S)
        assert np.array_equal(p3, parts[:, :, sub]) and np.array_equal(e3, eta[sub])


@pytest.mark.parametrize('Q,sizes,tmu', [
    (2, [41, 42, 41], 32),          # 124-dof neighbourhood: 64 parameters need 232 320 dynamic bytes, 272 static do not fit
    (2, [155, 157, 156], 8),        # 468 dofs: 16 parameters need 232 320 dynamic bytes
    (3, [116, 117, 117], 8),        # 350 dofs: 16 parameters need 232 448 dynamic bytes
])
def test_estimator_tile_counts_static_shared_memory(handle, Q, sizes, tmu):
    """A tile whose dynamic shared memory fits the per-block limit but not beside the kernel's static shared memory must
    not be picked: the plan takes the next smaller tile, and its results match the exact reference."""
    rng = np.random.default_rng(sum(sizes) + Q)
    sysd = _chain_system(rng, sizes, Q, 1)
    n_mu = 2 * tmu + 3
    terms, theta, u, rf2, rsc = random_family(rng, sysd, n_mu)
    plan = _plan(handle, sysd, terms, rf2, rsc, np.ones(Q), np.ones(Q), 1)
    assert int(plan.info(9)) == tmu
    parts, eta, _ = _estimate(handle, plan, theta, u, len(sizes))
    ex = X.terms_from_cabi(terms, sizes, sysd['nbh'], Q, rf2, rsc).evaluate(theta, u)
    for k, name in enumerate(PARTS):
        assert np.all(np.abs(parts[k] - ex[name]) <= 1e-13 * np.abs(ex[name])), name


# ------------------------------------------------------------------------------------------------------------
#  plans that live together: no plan may lower another's shared-memory limit
# ------------------------------------------------------------------------------------------------------------

def _solve(handle, plan, theta, n_red):
    from pylrbms_b200._lib import current_stream_ptr, ptr
    torch = _torch()
    n_mu = theta.shape[0]
    ws = C.c_size_t()
    handle.check(handle.lib.lrbms_online_workspace_bytes(plan.p, n_mu, C.byref(ws)))
    work = torch.empty(max(ws.value, 8), dtype=torch.uint8, device='cuda')
    u = torch.zeros((n_mu, n_red), dtype=torch.float64, device='cuda')
    info = torch.full((n_mu,), -1, dtype=torch.int32, device='cuda')
    handle.check(handle.lib.lrbms_online_solve(plan.p, n_mu, ptr(dev(theta)), ptr(u), ptr(info), ptr(work), ws.value,
                                               current_stream_ptr()))
    torch.cuda.synchronize()
    assert int(info.abs().sum().item()) == 0
    return u.cpu().numpy()


@pytest.mark.parametrize('solver,large,small', [
    (1, (8, 8, 20, 2), (2, 2, 8, 1)),         # window kernel (v2)
])
def test_large_solve_plan_runs_after_smaller_plan(handle, solver, large, small):
    """The dynamic shared-memory limit is an attribute of the kernel, shared by all plans: creating a plan with a smaller
    footprint must not make the next launch of a larger plan that is still alive fail, nor change its results."""
    rng = np.random.default_rng(solver)
    big = _random_reduced_system(rng, large[0], large[1], [large[2]] * (large[0] * large[1]), Q=large[3])
    sml = _random_reduced_system(rng, small[0], small[1], [small[2]] * (small[0] * small[1]), Q=small[3])
    pb = _plan(handle, big, None, None, None, None, None, 1, solver=solver)
    assert int(pb.info(6)) == solver
    theta = np.column_stack([np.ones(5), rng.uniform(0.1, 1.0, 5), rng.uniform(0.5, 2.0, 5)])
    u1 = _solve(handle, pb, theta, big['n'])
    ps = _plan(handle, sml, None, None, None, None, None, 1, solver=solver)
    assert int(ps.info(6)) == solver
    _solve(handle, ps, theta if small[3] == 2 else theta[:, [0, 2]], sml['n'])
    u2 = _solve(handle, pb, theta, big['n'])
    assert np.array_equal(u1, u2)


def test_large_estimator_plan_runs_after_smaller_plan(handle):
    """As above for the estimator: both plans run estimate_kernel<64> (the limit is per template instantiation), the
    second with fewer dynamic bytes (116- against 121-dof neighbourhoods, both above 48 KB)."""
    rng = np.random.default_rng(64)
    big = _chain_system(rng, [40, 41, 40], 2, 1)
    terms, theta, u, rf2, rsc = random_family(rng, big, 70)
    pb = _plan(handle, big, terms, rf2, rsc, np.ones(2), np.ones(2), 1)
    p1, e1, _ = _estimate(handle, pb, theta, u, 3, poison=False)
    small = _chain_system(rng, [38, 40, 38], 2, 1)
    ts, th_s, u_s, rf2_s, rsc_s = random_family(rng, small, 5)
    ps = _plan(handle, small, ts, rf2_s, rsc_s, np.ones(2), np.ones(2), 1)
    assert int(pb.info(9)) == int(ps.info(9)) == 64
    _estimate(handle, ps, th_s, u_s, 3, poison=False)
    p2, e2, _ = _estimate(handle, pb, theta, u, 3, poison=False)
    assert np.array_equal(p1, p2) and np.array_equal(e1, e2)


def test_apply_inverse_then_sweep(handle, c1_model):
    """``rd.operator.assemble(mu).apply_inverse(f)`` builds a one-term plan with a smaller window kernel footprint; the
    model's own sweep afterwards must still run and reproduce its earlier results."""
    rd = c1_model
    assert int(rd.online_plan.info(6)) == 1, 'the model must run the window kernel for this test to cover its limit'
    mus = np.linspace(0.1, 1.0, 5)
    U1, eta1 = rd.sweep(mus)
    mu = rd.parse_parameter(0.5)
    f = rd.rhs.operators[0].to_dense()
    v = rd.operator.assemble(mu).apply_inverse(f)
    assert np.all(np.isfinite(np.asarray(v.data)))
    U2, eta2 = rd.sweep(mus)
    assert np.array_equal(np.asarray(U1.data), np.asarray(U2.data)) and np.array_equal(eta1, eta2)


# ------------------------------------------------------------------------------------------------------------
#  lrbms_eta_max
# ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize('n', [1, 1023, 1025, 100_000])
def test_eta_max(handle, n):
    from pylrbms_b200._lib import current_stream_ptr, ptr
    torch = _torch()
    rng = np.random.default_rng(n)
    base = rng.uniform(0.0, 1.0, n)
    cases = {'random': base}
    for where in (0, n - 1):
        e = base.copy(); e[where] = 2.0
        cases['max at {}'.format(where)] = e
    if n > 1:
        e = base.copy(); hit = np.sort(rng.choice(n, min(n, 3), replace=False)); e[hit] = 2.0
        cases['tie'] = e
        cases['all equal'] = np.full(n, 0.5)
        e = base.copy(); e[[n - 1, 0]] = 2.0
        cases['tie first and last'] = e
    for name, e in cases.items():
        mx = torch.zeros(1, dtype=torch.float64, device='cuda'); am = torch.full((1,), -7, dtype=torch.int64, device='cuda')
        handle.check(handle.lib.lrbms_eta_max(handle.h, n, ptr(dev(e)), ptr(mx), ptr(am), current_stream_ptr()))
        torch.cuda.synchronize()
        assert mx.item() == e.max() and am.item() == int(np.argmax(e)), name


# ------------------------------------------------------------------------------------------------------------
#  model level
# ------------------------------------------------------------------------------------------------------------

def _models(shape, cells, N, seed, problem=None):
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases
    from pylrbms_b200 import discretize, LRBMSReductor
    from oracle import lrbms_oracle as O
    data = assemble_block_swipdg(shape, cells, problem=problem)
    bases = make_local_bases(data, N, seed=seed)
    bd = {'domain_%d' % i: bases[i] for i in range(data.num_subdomains)}
    return data, LRBMSReductor(discretize(data)[0], bases=bd), O.LRBMSReductor(O.build_discretization(data), bases=bd)


@pytest.fixture(scope='module')
def c1_model(handle):
    data, red, _ = _models((4, 4), 16, 8, 1001)
    return red.reduce()


@pytest.fixture(scope='module')
def c2_models(handle):
    data, red, red_ref = _models((8, 8), 32, 20, 1002)
    return data, red.reduce(), red_ref, red_ref.reduce()


def model_exact(rd, mus, U, subdomains=None):
    """Exact parts of a ``ReducedModel``'s estimator on ``U`` (front-end (ii))."""
    parsed = [rd.parse_parameter(m) for m in mus]
    forms = X.terms_from_model(rd, subdomains)
    theta = X.flux_thetas(rd.estimator.flux_reconstruction.coefficients, parsed)
    return forms, forms.evaluate(theta, np.asarray(U), subdomains=subdomains, factor_args=parsed)


def model_K(rd, forms, subdomains):
    Q = len(rd.estimator.flux_reconstruction.coefficients)
    K = kernel_K(forms, rd.block_dims, [list(rd.neighborhoods[s]) for s in range(len(rd.block_dims))], Q)
    return K[:, list(subdomains)]


def _exact_eta(ex, rd, mus):
    """eta from the exact parts (float64 combine, estimators.py:99-102)."""
    est = rd.estimator
    out = []
    for k, mu in enumerate(mus):
        mu_p = rd.parse_parameter(mu)
        lam = est.lambda_coeffs
        a_bar, g_bar, a_hat = est.alpha(lam, mu_p, est.mu_bar), est.gamma(lam, mu_p, est.mu_bar), est.alpha(lam, mu_p, est.mu_hat)
        nc, rd_ = ex['nc'][:, k], ex['r'][:, k] + ex['df'][:, k]
        out.append((np.sqrt(g_bar) * np.linalg.norm(nc) + np.linalg.norm(rd_) / np.sqrt(a_hat)) / np.sqrt(a_bar))
    return np.array(out)


def test_c2_three_way_distances(handle, c2_models):
    """C2 (8 x 8, N = 20): split the GPU / oracle difference of the estimator into (1) the GPU's evaluation error on its own
    operators and u, (2) the oracle's evaluation error on its own, (3) the difference of the exact values on the two input
    sets.  Printed in units of eps S and relative to the value; (1) is asserted against the kernel's gamma_K S bound."""
    from oracle.parity import reference_online
    data, rd, red_ref, rd_ref = c2_models
    lo, hi = data.parameter_range
    mus = np.linspace(lo, hi, 8)
    Ug, eta_g, parts_g, _ = rd.sweep(mus, decompose=True)
    parts_g = np.stack(parts_g)
    forms, exg = model_exact(rd, mus, Ug.data)
    U_ref, eta_ref, parts_ref, _, _, _, _ = reference_online(rd_ref, mus)
    d = red_ref.d
    parsed = [d.parse_parameter(m) for m in mus]
    exo = X.terms_from_oracle(red_ref).evaluate(X.flux_thetas(d.estimator.lambda_coeffs, parsed), U_ref, factor_args=parsed)
    K = model_K(rd, forms, range(len(rd.block_dims)))
    report = {}
    for k, name in enumerate(PARTS):
        S = exg['S_' + name]
        d1 = np.abs(parts_g[k] - exg[name]); d2 = np.abs(parts_ref[k] - exo[name]); d3 = np.abs(exg[name] - exo[name])
        val = np.abs(exg[name]).max(axis=0)
        report[name] = ['{:.2f} eps S / {:.1e} rel'.format(float((x / (EPS * S)).max()), float((x.max(axis=0) / val).max()))
                        for x in (d1, d2, d3)]
        assert np.all(d1 <= gamma(K[k][:, None]) * S), name
    e_g, e_o = _exact_eta(exg, rd, mus), _exact_eta(exo, rd, mus)
    report['eta'] = ['{:.1e} rel'.format(float(np.max(np.abs(x) / e_g))) for x in (eta_g - e_g, eta_ref - e_o, e_g - e_o)]
    for name, (a, b, c) in report.items():
        print('C2 {:4s} (1) GPU vs exact(GPU inputs) {}   (2) oracle vs exact(oracle inputs) {}   (3) exact(GPU) vs '
              'exact(oracle) {}'.format(name, a, b, c))


def test_sweep_eta_into_matches_sweep(handle, c2_models):
    """``sweep_eta_into`` (the chunked eta-only sweep with max / argmax) against ``sweep`` on the same parameters:
    bit-identical eta, max and argmax for every chunk size; duplicated parameters tie and resolve to the lowest index.
    The batch is larger than the default chunk (128 parameters per SM), and no chunk but 1 divides it."""
    import torch
    _, rd, _, _ = c2_models
    rng = np.random.default_rng(9)
    default_chunk = 128 * rd.online_plan.handle.sm_count
    base = rng.uniform(0.1, 1.0, default_chunk // 2 + 151)
    mus = np.concatenate([base, base[::-1]])          # every eta twice
    _, eta = rd.sweep(mus)
    tile = int(rd.online_plan.info(9))
    assert all(len(mus) % c for c in (7, tile - 1, default_chunk))
    ref_arg = int(np.argmax(eta))
    assert eta[ref_arg] == eta[len(mus) - 1 - ref_arg] and ref_arg < len(mus) - 1 - ref_arg
    for chunk in (1, 7, tile - 1, None):
        eta_host = torch.empty(len(mus), dtype=torch.float64).pin_memory()
        bad, mx, am = rd.sweep_eta_into(mus, eta_host, chunk=chunk)
        assert bad == 0
        assert np.array_equal(eta_host.numpy(), eta), chunk
        assert mx == eta.max() and am == ref_arg, (chunk, mx, am)
