"""Reduction error analysis on the device (``reduction_error_analysis``, ``csrc/error_norms.cu``):

1. the reconstruction error ``e = u_h - V u_N`` against a double-double reference (ragged bases, an empty basis, a reduced
   solution of an older model with fewer basis vectors), and the C ABI's argument checks;
2. the segmented quadratic forms (local energy products, ``e^T A(mu) e``) against double-double evaluations, on C1 (also
   with more than one 256-parameter launch) and on the 3D synthetic operators;
3. errors, local errors, eta and effectivities against the oracle with SciPy's direct solve (C1 and the 3 x 2 grid);
4. every parameter's results bit-identical whatever batch it is analysed in, and the same bits for a reduced model that
   predates an extension of the bases;
5. snapshot reproduction: at the training parameters of the bases the error is at the solver's floor;
6. C2 at full size against a host recomputation;
7. (CPU) the argument checks of the host layer.
"""
import ctypes as C
import types

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spl

from oracle.exact_forms import EPS, dd_add, dd_mul, two_prod

gpu = pytest.mark.gpu


def _theta(d, mus):
    from pylrbms_b200.parameters import theta_matrix
    return theta_matrix(list(d.operator.coefficients) + list(d.rhs.coefficients), mus, d.parameter_type)


def _host_system(data, th):
    S = data.num_subdomains
    A = None
    for q in range(data.Q):
        blocks = [[None] * S for _ in range(S)]
        for (i, j), M in data.lhs[q].items():
            blocks[i][j] = M
        A = th[q] * sp.bmat(blocks, format='csc') if A is None else A + th[q] * sp.bmat(blocks, format='csc')
    return A.tocsc(), th[data.Q] * np.concatenate(data.rhs)


def _dd_tree_sum(h, l):
    """Sum of double-double values along axis 0 (pairwise, every addition error-free up to the dd renormalisation)."""
    while h.shape[0] > 1:
        if h.shape[0] % 2:
            h = np.concatenate([h, np.zeros_like(h[:1])])
            l = np.concatenate([l, np.zeros_like(l[:1])])
        h, l = dd_add(h[0::2], l[0::2], h[1::2], l[1::2])
    return h[0], l[0]


def _dd_csr_form(M, x, rows=None):
    """``sum_{r in rows} x[r] (M x)[r]`` per column of ``x (n, n_mu)`` in double-double, and ``|x|^T |M| |x|`` over the
    same rows.  ``M``: SciPy CSR."""
    M = sp.csr_matrix(M)
    rows = np.arange(M.shape[0]) if rows is None else np.asarray(rows)
    Ms = M[rows]
    cnt = np.diff(Ms.indptr)
    wh = np.zeros((len(rows), x.shape[1]))
    wl = np.zeros_like(wh)
    for j in range(int(cnt.max()) if cnt.size else 0):
        sel = np.flatnonzero(cnt > j)
        k = Ms.indptr[sel] + j
        p, e = two_prod(Ms.data[k][:, None], x[Ms.indices[k]])
        wh[sel], wl[sel] = dd_add(wh[sel], wl[sel], p, e)
    xr = x[rows]
    p, e = two_prod(xr, wh)
    vh, vl = _dd_tree_sum(p, e + xr * wl)
    scale = np.einsum('rm,rm->m', np.abs(xr), abs(Ms) @ np.abs(x))
    return vh + vl, scale


def _partition_k(n_s, n_total, sm_count, max_row):
    """Number of roundings a form of the kernel chains for one segment: the CSR row, the rows of a lane, the warps of a
    CTA and the CTAs of the segment (row partition of csrc/error_norms.cu)."""
    R = max(8, -(-n_total // (8 * sm_count)))
    c_s = -(-n_s // R)
    return max_row + 2 + (-(-R // 8)) + 8 + c_s


def _c1_setup(sizes_fn=lambda i: 4 + i % 7, empty=5):
    from pylrbms_b200 import LRBMSReductor, discretize
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases
    data = assemble_block_swipdg((4, 4), 16)
    S = data.num_subdomains
    bases = make_local_bases(data, [sizes_fn(i) for i in range(S)], seed=11)
    if empty is not None:
        bases[empty] = np.zeros((0, int(data.n[empty])))
    d, _ = discretize(data)
    red = LRBMSReductor(d, bases={'domain_%d' % i: bases[i] for i in range(S)})
    return data, d, red, bases


# ---------------------------------------------------------------------------------------------------------------------
#  1. reconstruction
# ---------------------------------------------------------------------------------------------------------------------

@gpu
def test_recon_error_matches_double_double(handle):
    import torch
    from pylrbms_b200.kernels import recon_error
    from pylrbms_b200.vectorarray import _round_cap
    data, d, red, bases = _c1_setup()
    S = data.num_subdomains
    subs = d.solution_space.subspaces
    old = [max(0, len(b) - (i % 3)) for i, b in enumerate(bases)]         # an older model: fewer vectors per subdomain
    assert any(o < len(b) for o, b in zip(old, bases)) and old[5] == 0
    n, n_mu = d.solution_space.dim, 37
    rng = np.random.default_rng(3)
    uh_host = rng.standard_normal((n, n_mu))
    uN_host = rng.standard_normal((n_mu, sum(old)))
    ld = _round_cap(n_mu)
    assert ld % 4 == 0 and ld % 32 and ld > n_mu
    u_h = torch.zeros((n, ld), dtype=torch.float64, device='cuda')
    u_h[:, :n_mu] = torch.from_numpy(uh_host)
    u_h[:, n_mu:] = float('nan')                                          # lanes past n_mu are never read
    u_h_before = u_h.clone()
    e = torch.full((n, ld + 3), float('nan'), dtype=torch.float64, device='cuda')
    recon_error([red.bases[s.id] for s in subs], old, u_h, torch.from_numpy(uN_host).cuda(), e)
    got = e.cpu().numpy()
    assert np.all(np.isnan(got[:, n_mu:])), 'columns past n_mu were written'
    assert torch.equal(u_h[:, :n_mu], u_h_before[:, :n_mu]), 'u_h was modified'
    got = got[:, :n_mu]
    row, red_off = 0, 0
    for i in range(S):
        n_i, N = int(data.n[i]), old[i]
        V = bases[i][:N].T                                                 # (n_i, N)
        c = uN_host[:, red_off:red_off + N]                                # (n_mu, N)
        h, l = np.zeros((n_i, n_mu)), np.zeros((n_i, n_mu))
        for k in range(N):
            p, err = two_prod(V[:, k:k + 1], c[None, :, k])
            h, l = dd_add(h, l, p, err)
        uh = uh_host[row:row + n_i]
        rh, rl = dd_add(uh, np.zeros_like(uh), -h, -l)
        ref = rh + rl
        bound = (N + 2) * EPS * (np.abs(uh) + np.abs(V) @ np.abs(c).T)
        assert np.all(np.abs(got[row:row + n_i] - ref) <= bound), i
        if N == 0:
            assert np.array_equal(got[row:row + n_i], uh), 'an empty basis must give e = u_h'
        row, red_off = row + n_i, red_off + N


@gpu
def test_cabi_argument_checks(handle):
    import torch
    from pylrbms_b200._lib import ReconBlock, ptr
    lib, h = handle.lib, handle.h
    V = torch.zeros((10, 4), dtype=torch.float64, device='cuda')
    x = torch.zeros((10, 8), dtype=torch.float64, device='cuda')
    uN = torch.zeros((8, 4), dtype=torch.float64, device='cuda')
    e = torch.zeros((10, 8), dtype=torch.float64, device='cuda')
    ws = torch.zeros(4096, dtype=torch.float64, device='cuda')
    blk = (ReconBlock * 1)(ReconBlock(V.data_ptr(), 4, 3, 3, 0, 0, 10, 0))
    args = lambda b, ldu: (h, 1, C.cast(b, C.c_void_p), 8, ptr(x), ldu, ptr(uN), 4, 4, ptr(e), 8, ptr(ws), 8 * 4096, None)
    assert lib.lrbms_recon_error(*args(blk, 8)) == 0
    assert lib.lrbms_recon_error(*args(blk, 7)) == -1 and b'leading dimension' in lib.lrbms_last_error(h)
    bad = (ReconBlock * 1)(ReconBlock(V.data_ptr(), 4, 3, 4, 0, 0, 10, 0))   # N = 4 > len = 3
    assert lib.lrbms_recon_error(*args(bad, 8)) == -1 and b'exceeds the basis length' in lib.lrbms_last_error(h)
    rowptr = torch.arange(11, dtype=torch.int32, device='cuda')
    colind = torch.arange(10, dtype=torch.int32, device='cuda')
    vals = torch.ones((5, 10), dtype=torch.float64, device='cuda')
    th = torch.ones((8, 5), dtype=torch.float64, device='cuda')
    seg = np.array([0, 10], dtype=np.int32)
    out = torch.zeros((1, 8), dtype=torch.float64, device='cuda')
    form = lambda Q, ldt, theta: lib.lrbms_segmented_form(h, 10, Q, ptr(rowptr), ptr(colind), ptr(vals), 10, 1, ptr(seg), 8,
                                                          theta, ldt, ptr(x), 8, ptr(out), 8, ptr(ws), 8 * 4096, None)
    assert form(5, 5, ptr(th)) == -5 and b'at most 4' in lib.lrbms_last_error(h)
    assert form(3, 2, ptr(th)) == -1 and b'ldt < Q' in lib.lrbms_last_error(h)
    assert form(2, 5, None) == -1
    assert form(4, 5, ptr(th)) == 0


# ---------------------------------------------------------------------------------------------------------------------
#  2. quadratic forms
# ---------------------------------------------------------------------------------------------------------------------

def _check_forms(handle, data, d, x_host, mus):
    """Local energy forms and x^T A(mu) x of the kernel against double-double, within gamma |x|^T |M| |x|."""
    import torch
    from pylrbms_b200.error_analysis import _energy_system
    from pylrbms_b200.kernels import segmented_form
    from pylrbms_b200.vectorarray import _round_cap
    S = data.num_subdomains
    n, n_mu = x_host.shape
    x = torch.zeros((n, _round_cap(n_mu)), dtype=torch.float64, device='cuda')
    x[:, :n_mu] = torch.from_numpy(x_host)
    E_pat, E_vals, offs = _energy_system(d)
    local = segmented_form(E_pat, E_vals, offs, x, n_mu).cpu().numpy()
    for i in range(S):
        Ei = sp.csr_matrix(data.energy[i])
        ref, scale = _dd_csr_form(Ei, x_host[offs[i]:offs[i + 1]])
        k = _partition_k(int(data.n[i]), n, handle.sm_count, int(np.diff(Ei.indptr).max()))
        assert np.all(np.abs(local[i] - ref) <= k * EPS * scale), i
    A_pat, A_vals, _ = d.affine_system(range(S))
    th = _theta(d, mus)
    opf = segmented_form(A_pat, A_vals, [0, n], x, n_mu, theta=torch.from_numpy(th).cuda()).cpu().numpy()[0]
    vh, vl, scale = np.zeros(n_mu), np.zeros(n_mu), np.zeros(n_mu)
    for q in range(data.Q):
        blocks = [[None] * S for _ in range(S)]
        for (i, j), M in data.lhs[q].items():
            blocks[i][j] = M
        Aq = sp.bmat(blocks, format='csr')
        fq, sq = _dd_csr_form(Aq, x_host)
        h, l = dd_mul(fq, np.zeros_like(fq), th[:, q])
        vh, vl = dd_add(vh, vl, h, l)
        scale += np.abs(th[:, q]) * sq
    k = _partition_k(n, n, handle.sm_count, int(np.diff(A_pat.rowptr.cpu().numpy()).max())) + data.Q
    assert np.all(np.abs(opf - (vh + vl)) <= k * EPS * scale)
    return local, opf


@gpu
def test_forms_match_double_double_c1(handle):
    import torch
    from pylrbms_b200.kernels import recon_error
    data, d, red, bases = _c1_setup(empty=None)                            # reduce() needs a vector in every basis
    subs = d.solution_space.subspaces
    mus = np.linspace(*data.parameter_range, 6)
    U_h = d.solve_batch(mus)
    rd = red.reduce()
    uN = rd.solve_batch(mus).device_tensor
    n = d.solution_space.dim
    e = torch.zeros((n, 8), dtype=torch.float64, device='cuda')
    buf = U_h._blocks[0]._buf.as_strided((n, len(mus)), (U_h._blocks[0].ld, 1))
    recon_error([red.bases[s.id] for s in subs], rd.block_dims, buf, uN, e)        # the kernel's own e
    _check_forms(handle, data, d, e[:, :len(mus)].cpu().numpy(), mus)


@gpu
def test_forms_match_double_double_3d(handle):
    from pylrbms_b200 import discretize
    from pylrbms_b200.synthetic_fixture import synthetic_block_operators
    data = synthetic_block_operators((3, 2, 2), (2, 2, 2))
    d, _ = discretize(data)
    mus = np.linspace(*data.parameter_range, 5)
    x = np.random.default_rng(5).standard_normal((d.solution_space.dim, len(mus)))
    _check_forms(handle, data, d, x, mus)


@gpu
def test_forms_more_than_one_launch_chunk(handle):
    """300 parameters: lrbms_segmented_form runs two 256-parameter launches; both are held to double-double, and the
    columns of the second launch equal the same parameters formed on their own."""
    import torch
    from pylrbms_b200.error_analysis import _energy_system
    from pylrbms_b200.kernels import segmented_form
    from pylrbms_b200.vectorarray import _round_cap
    data, d, _, _ = _c1_setup(empty=None)
    n_mu = 300
    mus = np.random.default_rng(8).uniform(*data.parameter_range, n_mu)
    x = np.random.default_rng(6).standard_normal((d.solution_space.dim, n_mu))
    local, opf = _check_forms(handle, data, d, x, mus)
    sel = slice(250, 262)
    n, k = x.shape[0], sel.stop - sel.start
    xs = torch.zeros((n, _round_cap(k)), dtype=torch.float64, device='cuda')
    xs[:, :k] = torch.from_numpy(x[:, sel])
    E_pat, E_vals, offs = _energy_system(d)
    assert np.array_equal(segmented_form(E_pat, E_vals, offs, xs, k).cpu().numpy(), local[:, sel])
    A_pat, A_vals, _ = d.affine_system(range(data.num_subdomains))
    th = torch.from_numpy(np.ascontiguousarray(_theta(d, mus)[sel])).cuda()
    assert np.array_equal(segmented_form(A_pat, A_vals, [0, n], xs, k, theta=th).cpu().numpy()[0], opf[sel])


# ---------------------------------------------------------------------------------------------------------------------
#  3. against the oracle
# ---------------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize('grid,cells', [((4, 4), 16), ((3, 2), 4)])
def test_analysis_matches_oracle(handle, grid, cells):
    from pylrbms_b200 import LRBMSReductor, discretize, reduction_error_analysis
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases
    from oracle import lrbms_oracle as O
    data = assemble_block_swipdg(grid, cells)
    S = data.num_subdomains
    bases = make_local_bases(data, [4 + (i % 7) for i in range(S)], seed=11)
    bd = {'domain_%d' % i: bases[i] for i in range(S)}
    d, _ = discretize(data)
    red, red_ref = LRBMSReductor(d, bases=bd), O.LRBMSReductor(O.build_discretization(data), bases=bd)
    rd, rd_ref = red.reduce(), red_ref.reduce()
    mus = np.linspace(*data.parameter_range, 5)
    res = reduction_error_analysis(d, red, rd, mus)
    assert res.fom_info is not None and np.all(res.fom_info['status'] == 0)
    assert res.errors.shape == (5,) and res.local_errors.shape == (S, 5) and res.indicators.shape == (S, 5)
    offs = np.concatenate([[0], np.cumsum(data.n)])
    for k, mu in enumerate(mus):
        th = _theta(d, [mu])[0]
        A, b = _host_system(data, th)
        u_ref = spl.spsolve(A, b)
        U_ref = rd_ref.solve(mu)
        E = u_ref - red_ref.reconstruct(U_ref).data[0]
        loc = np.array([E[offs[i]:offs[i + 1]] @ (data.energy[i] @ E[offs[i]:offs[i + 1]]) for i in range(S)])
        norm_u = np.sqrt(sum(u_ref[offs[i]:offs[i + 1]] @ (data.energy[i] @ u_ref[offs[i]:offs[i + 1]]) for i in range(S)))
        err_ref = np.sqrt(loc.sum())
        tol = 1e-9 * norm_u
        assert abs(res.errors[k] - err_ref) <= tol, (mu, res.errors[k], err_ref)
        assert np.all(np.abs(res.local_errors[:, k] - np.sqrt(loc)) <= tol)
        assert abs(res.relative_errors[k] - err_ref / norm_u) <= 1e-9
        assert abs(res.operator_errors[k] - np.sqrt(E @ (A @ E))) <= 1e-9 * np.sqrt(u_ref @ (A @ u_ref))
        eta_ref, _, ind_ref = rd_ref.estimate(U_ref, mu, decompose=True)
        assert abs(res.eta[k] - eta_ref) <= 1e-10 * abs(eta_ref)
        assert np.abs(res.indicators[:, k] - ind_ref[:, 0]).max() <= 1e-9 * np.abs(ind_ref).max()
        assert abs(res.effectivities[k] - eta_ref / err_ref) <= 1e-8 * eta_ref / err_ref
    assert res.argmax == int(np.argmax(res.errors)) and res.max_error == res.errors.max()
    assert res.min_effectivity == res.effectivities.min() and res.max_effectivity == res.effectivities.max()
    print(grid, 'effectivities', res.effectivities, 'operator / energy', res.operator_errors / res.errors)


# ---------------------------------------------------------------------------------------------------------------------
#  4. bit reproducibility
# ---------------------------------------------------------------------------------------------------------------------

_FIELDS = ('errors', 'operator_errors', 'relative_errors', 'effectivities')


@gpu
def test_analysis_is_batch_independent(handle):
    """C1 (S = 16: the subdomain sums must not follow NumPy's pairwise order, which differs for one column and several).
    The single-parameter analyses solve their own u_h; the batches take theirs from one pooled solve, indexed into separate
    buffers, so they also go through the gather of u_h into one dof-major buffer."""
    from pylrbms_b200 import reduction_error_analysis
    from pylrbms_b200._lib import current_stream_ptr
    from pylrbms_b200.error_analysis import _dofmajor
    data, d, red, _ = _c1_setup(empty=None)
    assert data.num_subdomains >= 8
    rd = red.reduce()
    rng = np.random.default_rng(9)
    pool = rng.uniform(*data.parameter_range, 70)
    U_pool = d.solve_batch(pool)
    keys = (0, 1, 30, 31, 32, 33, 69)
    solo = {k: reduction_error_analysis(d, red, rd, pool[[k]]) for k in keys}
    n = d.solution_space.dim
    U_sub = U_pool[np.arange(3)]
    assert _dofmajor(U_sub, n, 3).data_ptr() != U_sub._blocks[0].device_ptr, 'expected the gathered copy'

    def same(res, pos, k):
        for f in _FIELDS:
            assert np.array_equal(getattr(res, f)[pos:pos + 1], getattr(solo[k], f)), (f, pos, k)
        assert np.array_equal(res.local_errors[:, pos], solo[k].local_errors[:, 0])

    for size in (1, 31, 32, 33, 70):
        for permute, budget in ((False, None), (True, None), (True, 8 * n * 10)):
            idx = rng.permutation(size) if permute else np.arange(size)
            if budget is not None:
                d.fom_workspace_budget = budget                     # error scratch of 10 parameters
            try:
                res = reduction_error_analysis(d, red, rd, pool[idx], U_h=U_pool[idx])
            finally:
                d.__dict__.pop('fom_workspace_budget', None)
            for pos, k in enumerate(idx):
                if k in solo:
                    same(res, pos, k)
    handle.check(handle.lib.lrbms_debug_poison_shared(handle.h, current_stream_ptr()))
    res = reduction_error_analysis(d, red, rd, pool[[33, 0]])
    same(res, 0, 33)
    same(res, 1, 0)


@gpu
def test_analysis_of_an_older_reduced_model(handle):
    """A reduced model reduced before the bases were extended is analysed with the leading block_dims[i] vectors of the
    grown bases (reductor.reconstruct semantics): the same bits as before the extension."""
    from pylrbms_b200 import reduction_error_analysis
    data, d, red, _ = _c1_setup(empty=None)
    rd_old = red.reduce()
    mus = np.linspace(*data.parameter_range, 7)
    before = reduction_error_analysis(d, red, rd_old, mus)
    dims = [len(red.bases[s.id]) for s in d.solution_space.subspaces]
    red.extend_basis(d.solve_batch(mus[[1, 4]]))
    grown = [len(red.bases[s.id]) for s in d.solution_space.subspaces]
    assert all(g >= n for g, n in zip(grown, dims)) and sum(grown) > sum(dims) and list(rd_old.block_dims) == dims
    after = reduction_error_analysis(d, red, rd_old, mus)
    for f in _FIELDS + ('local_errors', 'eta', 'indicators'):
        assert np.array_equal(getattr(after, f), getattr(before, f)), f
    rd_new = red.reduce()
    assert np.all(reduction_error_analysis(d, red, rd_new, mus).errors[[1, 4]] < before.errors[[1, 4]])


# ---------------------------------------------------------------------------------------------------------------------
#  5. snapshot reproduction
# ---------------------------------------------------------------------------------------------------------------------

@gpu
def test_snapshots_are_reproduced(handle):
    from pylrbms_b200 import LRBMSReductor, discretize, reduction_error_analysis
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg
    data = assemble_block_swipdg((4, 4), 16)
    d, _ = discretize(data)
    lo, hi = data.parameter_range
    train = np.linspace(lo, hi, 4)
    red = LRBMSReductor(d)
    red.extend_basis(d.solve_batch(train))
    rd = red.reduce()
    test = np.concatenate([train, np.random.default_rng(1).uniform(lo, hi, 12)])
    res = reduction_error_analysis(d, red, rd, test)
    print('relative energy errors at the training parameters', res.relative_errors[:4], 'elsewhere min / max',
          res.relative_errors[4:].min(), res.relative_errors[4:].max())
    # measured on a B200: 5e-13 ... 9e-13 at the training parameters (the fine solve's rtol of 1e-9 sets this floor), 3e-8 and
    # more elsewhere
    assert np.all(res.relative_errors[:4] <= 1e-8)
    assert np.all(res.errors[4:] > 0)


# ---------------------------------------------------------------------------------------------------------------------
#  6. C2 at full size
# ---------------------------------------------------------------------------------------------------------------------

@gpu
def test_c2_effectivities_match_host(handle):
    from pylrbms_b200 import LRBMSReductor, discretize, reduction_error_analysis
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases
    data = assemble_block_swipdg((8, 8), 32)
    d, _ = discretize(data)
    assert d.solution_space.dim == 393216
    S = data.num_subdomains
    bases = make_local_bases(data, 20, seed=1002)
    red = LRBMSReductor(d, bases={'domain_%d' % i: bases[i] for i in range(S)})
    rd = red.reduce()
    mus = np.random.default_rng(2024).uniform(*data.parameter_range, 32)
    U_h = d.solve_batch(mus)
    res = reduction_error_analysis(d, red, rd, mus, U_h=U_h)
    assert res.fom_info is None
    uN = rd.solve_batch(mus)
    eta = np.asarray(rd.estimate_batch(uN, mus))
    D = U_h.data - red.reconstruct(uN).data
    offs = np.concatenate([[0], np.cumsum(data.n)])
    err = np.zeros(len(mus))
    for i in range(S):
        Ei = D[:, offs[i]:offs[i + 1]]
        err += np.einsum('kd,kd->k', Ei, (data.energy[i] @ Ei.T).T)
    eff = eta / np.sqrt(err)
    assert np.all(np.abs(res.effectivities - eff) <= 1e-9 * eff)
    print('C2 effectivity range (N = 20, 32 parameters): %.3f .. %.3f' % (res.min_effectivity, res.max_effectivity))


# ---------------------------------------------------------------------------------------------------------------------
#  7. host layer, no device
# ---------------------------------------------------------------------------------------------------------------------

def _fakes(dims=(3, 2), lens=(3, 2), n=(10, 12)):
    subs = [types.SimpleNamespace(id='domain_%d' % i, dim=n[i]) for i in range(len(n))]
    d = types.SimpleNamespace(solution_space=types.SimpleNamespace(subspaces=subs))
    reductor = types.SimpleNamespace(d=d, bases={s.id: [None] * lens[i] for i, s in enumerate(subs)})
    rd = types.SimpleNamespace(block_dims=list(dims))
    return d, reductor, rd


def test_host_argument_checks():
    from pylrbms_b200.error_analysis import _check_arguments, reduction_error_analysis
    d, reductor, rd = _fakes()
    assert _check_arguments(d, reductor, rd, [0.1, 0.2], None) == (2, 2)
    with pytest.raises(ValueError, match='another discretization'):
        reduction_error_analysis(types.SimpleNamespace(solution_space=d.solution_space), reductor, rd, [0.1])
    with pytest.raises(ValueError, match='3 subdomain blocks'):
        reduction_error_analysis(d, reductor, types.SimpleNamespace(block_dims=[1, 1, 1]), [0.1])
    d2, reductor2, rd2 = _fakes(dims=(3, 3), lens=(3, 2))
    with pytest.raises(ValueError, match='subdomain 1: the reduced model uses 3 basis vectors, the reductor has 2'):
        reduction_error_analysis(d2, reductor2, rd2, [0.1])
    with pytest.raises(ValueError, match='at least one parameter'):
        reduction_error_analysis(d, reductor, rd, [])
    blocks = [types.SimpleNamespace(dim=10), types.SimpleNamespace(dim=12)]
    with pytest.raises(ValueError, match='2 solutions for 3 parameters'):
        reduction_error_analysis(d, reductor, rd, [0.1, 0.2, 0.3], U_h=_Arr(blocks, 2))
    with pytest.raises(ValueError, match='not an array of the solution space'):
        reduction_error_analysis(d, reductor, rd, [0.1, 0.2], U_h=_Arr([types.SimpleNamespace(dim=10)] * 2, 2))


class _Arr:
    def __init__(self, blocks, n):
        self._blocks, self._n = blocks, n

    def __len__(self):
        return self._n
