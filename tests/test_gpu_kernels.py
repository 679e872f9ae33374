"""GPU unit tests of the individual kernels, called through the C ABI (ctypes) and checked against NumPy/SciPy.

Tolerance: FP64 throughout, 1e-10 relative (BASELINE.json north_star) -- measured relative to the natural scale
of each result (the Frobenius norm of the block / the largest |entry|), never entry-wise on cancelling sums.
"""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

RTOL = 1e-10


def _torch():
    import torch
    return torch


def dev(a, dtype=None):
    torch = _torch()
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def rel(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    scale = max(np.abs(b).max() if b.size else 0.0, 1e-300)
    return (np.abs(a - b).max() if b.size else 0.0) / scale


def random_csr(rng, n_rows, n_cols, nnz_per_row, empty_row_fraction=0.0):
    rows, cols = [], []
    for r in range(n_rows):
        if rng.random() < empty_row_fraction:
            continue
        k = int(min(n_cols, max(1, rng.poisson(nnz_per_row))))
        c = rng.choice(n_cols, size=k, replace=False)
        rows.extend([r] * k)
        cols.extend(c.tolist())
    vals = rng.standard_normal(len(rows))
    M = sp.csr_matrix((vals, (rows, cols)), shape=(n_rows, n_cols))
    M.sort_indices()
    return M


class DevCsr:
    def __init__(self, M):
        torch = _torch()
        self.M = M
        self.rowptr = dev(M.indptr.astype(np.int32))
        self.colind = dev(M.indices.astype(np.int32)) if M.nnz else torch.zeros(1, dtype=torch.int32, device='cuda')
        self.values = dev(M.data.astype(np.float64)) if M.nnz else torch.zeros(1, dtype=torch.float64, device='cuda')


def dofmajor(rng, n, N, ld=None):
    """Random dof-major array (n x ld) with garbage in the padding columns."""
    ld = N if ld is None else ld
    a = rng.standard_normal((n, ld))
    return a


# ------------------------------------------------------------------------------------------------------------
#  VectorArray kernels
# ------------------------------------------------------------------------------------------------------------

def test_va_kernels(handle):
    from pylrbms_b200._lib import current_stream_ptr, ptr, host_f64, host_i32
    torch = _torch()
    lib, h = handle.lib, handle.h
    rng = np.random.default_rng(0)
    for dim, length, ld in ((1000, 7, 8), (6144, 20, 20), (33, 1, 4), (5, 256, 256)):
        x = rng.standard_normal((dim, ld))
        y = rng.standard_normal((dim, ld))
        alpha = rng.standard_normal(length)
        # scal
        dy = dev(y)
        handle.check(lib.lrbms_va_scal(h, dim, length, ptr(host_f64(alpha)), length, ptr(dy), ld, current_stream_ptr()))
        ref = y.copy(); ref[:, :length] *= alpha
        assert rel(dy.cpu().numpy(), ref) < 1e-15
        # axpy (per-vector alpha, and broadcast x of length 1)
        dy, dx = dev(y), dev(x)
        handle.check(lib.lrbms_va_axpy(h, dim, length, ptr(host_f64(alpha)), length, ptr(dx), ld, length, ptr(dy), ld,
                                       current_stream_ptr()))
        ref = y.copy(); ref[:, :length] += alpha * x[:, :length]
        assert rel(dy.cpu().numpy(), ref) < 1e-15
        dy = dev(y)
        handle.check(lib.lrbms_va_axpy(h, dim, length, ptr(host_f64(alpha[:1])), 1, ptr(dx), ld, 1, ptr(dy), ld,
                                       current_stream_ptr()))
        ref = y.copy(); ref[:, :length] += alpha[0] * x[:, :1]
        assert rel(dy.cpu().numpy(), ref) < 1e-15
        # pairwise dot
        out = torch.zeros(length, dtype=torch.float64, device='cuda')
        handle.check(lib.lrbms_va_pairwise_dot(h, dim, length, ptr(dx), ld, ptr(dev(y)), ld, ptr(out), current_stream_ptr()))
        ref = np.einsum('da,da->a', x[:, :length], y[:, :length])
        assert np.abs(out.cpu().numpy() - ref).max() <= RTOL * np.sqrt(dim)
        # lincomb
        n_out = 5
        if length * n_out * 8 <= 48 * 1024:
            Cf = rng.standard_normal((length, n_out))
            dout = torch.full((dim, 8), 7.0, dtype=torch.float64, device='cuda')
            handle.check(lib.lrbms_va_lincomb(h, dim, length, n_out, ptr(dx), ld, ptr(dev(Cf)), n_out, ptr(dout), 8,
                                              current_stream_ptr()))
            got = dout.cpu().numpy()
            assert rel(got[:, :n_out], x[:, :length] @ Cf) < 1e-13
            assert np.all(got[:, n_out:] == 7.0)
        # copy_cols with a permutation, into an offset
        if length <= 128:
            src = rng.permutation(length).astype(np.int32)
            dout = torch.zeros((dim, 2 * ld + 1), dtype=torch.float64, device='cuda')
            handle.check(lib.lrbms_va_copy_cols(h, dim, length, ptr(host_i32(src)), ptr(dx), ld, ptr(dout), 2 * ld + 1, 1,
                                                current_stream_ptr()))
            got = dout.cpu().numpy()
            assert np.array_equal(got[:, 1:1 + length], x[:, src])
        # transposes
        rm = rng.standard_normal((length, dim))
        dm = torch.zeros((dim, ld), dtype=torch.float64, device='cuda')
        handle.check(lib.lrbms_va_transpose_in(h, dim, length, ptr(dev(rm)), ptr(dm), ld, current_stream_ptr()))
        assert np.array_equal(dm.cpu().numpy()[:, :length], rm.T)
        back = torch.zeros((length, dim), dtype=torch.float64, device='cuda')
        handle.check(lib.lrbms_va_transpose_out(h, dim, length, ptr(dm), ld, ptr(back), current_stream_ptr()))
        assert np.array_equal(back.cpu().numpy(), rm)


# ------------------------------------------------------------------------------------------------------------
#  SpMM
# ------------------------------------------------------------------------------------------------------------

def test_spmm_batched(handle):
    from pylrbms_b200._lib import SpmmDesc, make_spmm_plan
    torch = _torch()
    rng = np.random.default_rng(1)
    cases = [(1536, 1536, 12, 8, 8, 0.0), (777, 333, 5, 20, 24, 0.3), (64, 4000, 3, 1, 1, 0.0), (130, 50, 20, 100, 100, 0.5),
             (6144, 512, 2, 40, 40, 0.9), (3, 3, 2, 67, 70, 0.0)]
    descs, keep, refs = [], [], []
    for (nr, nc, k, N, ld, efrac) in cases:
        A = random_csr(rng, nr, nc, k, efrac)
        V = dofmajor(rng, nc, N, ld)
        dA, dV = DevCsr(A), dev(V)
        W = torch.full((nr, ld), -3.0, dtype=torch.float64, device='cuda')
        descs.append(SpmmDesc(dA.rowptr.data_ptr(), dA.colind.data_ptr(), dA.values.data_ptr(), nr, nc, dV.data_ptr(), ld, N,
                              W.data_ptr(), ld))
        keep.append((dA, dV, W))
        refs.append((A @ V[:, :N], N))
    plan = make_spmm_plan(handle, descs, keep)
    for _ in range(2):      # run twice: plans are reusable
        plan.run()
    torch.cuda.synchronize()
    for (dA, dV, W), (ref, N) in zip(keep, refs):
        got = W.cpu().numpy()
        assert rel(got[:, :N], ref) < 1e-13
        assert np.all(got[:, N:] == -3.0), 'padding columns must not be written'
    assert plan.launches >= 1 and plan.flops > 0


# ------------------------------------------------------------------------------------------------------------
#  fused projection
# ------------------------------------------------------------------------------------------------------------

def _project_case(rng, nr, nc, k, NL, NR, efrac, identity=False, ldpad=0, alpha=1.0):
    torch = _torch()
    from pylrbms_b200._lib import ProjectDesc
    if identity:
        nc = nr
        A = None
    else:
        A = random_csr(rng, nr, nc, k, efrac)
    VL = dofmajor(rng, nr, NL, NL + ldpad)
    VR = dofmajor(rng, nc, NR, NR + ldpad)
    dA = DevCsr(A) if A is not None else None
    dVL, dVR = dev(VL), dev(VR)
    ldo = NR + 3
    out = torch.full((NL, ldo), 11.0, dtype=torch.float64, device='cuda')
    desc = ProjectDesc(dA.rowptr.data_ptr() if dA else None, dA.colind.data_ptr() if dA else None,
                       dA.values.data_ptr() if dA else None, nr, nc, dVL.data_ptr(), NL + ldpad, NL, dVR.data_ptr(),
                       NR + ldpad, NR, out.data_ptr(), ldo, alpha)
    W = (A @ VR[:, :NR]) if A is not None else VR[:, :NR]
    ref = alpha * (VL[:, :NL].T @ W)
    # scale for the tolerance: the sum of |terms|, i.e. what a backward-stable dot product is accurate against
    scale = np.abs(VL[:, :NL]).T @ np.abs(W)
    return desc, (dA, dVL, dVR, out), ref, scale, NR


def test_project_batched(handle):
    from pylrbms_b200._lib import make_project_plan
    torch = _torch()
    rng = np.random.default_rng(2)
    cases = [
        dict(nr=1536, nc=1536, k=12, NL=8, NR=8, efrac=0.0),
        dict(nr=6144, nc=6144, k=12, NL=20, NR=20, efrac=0.0),
        dict(nr=6144, nc=6144, k=6, NL=20, NR=20, efrac=0.97),           # coupling block: few populated rows
        dict(nr=1000, nc=700, k=4, NL=13, NR=27, efrac=0.2, ldpad=3),     # ragged sizes
        dict(nr=12288, nc=12288, k=20, NL=40, NR=40, efrac=0.0),
        dict(nr=3000, nc=3000, k=0, NL=20, NR=20, efrac=0.0, identity=True),   # Gram matrix V^T V
        dict(nr=2000, nc=2000, k=7, NL=100, NR=100, efrac=0.0),           # two-step (SpMM, then dense)
        dict(nr=500, nc=900, k=7, NL=1, NR=200, efrac=0.0),               # functional x wide basis
        dict(nr=900, nc=500, k=7, NL=200, NR=1, efrac=0.0, alpha=-2.0),
        dict(nr=5, nc=5, k=2, NL=3, NR=2, efrac=0.0),
        dict(nr=1, nc=1, k=1, NL=1, NR=1, efrac=0.0),
        dict(nr=40000, nc=40000, k=12, NL=24, NR=16, efrac=0.0),          # many row splits -> cross-CTA combine
    ]
    descs, keep, refs = [], [], []
    for c in cases:
        d, k, ref, scale, NR = _project_case(rng, **c)
        descs.append(d); keep.append(k); refs.append((ref, scale, NR))
    plan = make_project_plan(handle, descs, keep)
    results = []
    for _ in range(3):
        plan.run()
        torch.cuda.synchronize()
        results.append([k[3].cpu().numpy().copy() for k in keep])
    for idx, ((ref, scale, NR), got) in enumerate(zip(refs, results[0])):
        err = np.abs(got[:, :NR] - ref) / np.maximum(scale, 1e-300)
        assert err.max() < 1e-13, 'case {}: rel err {}'.format(idx, err.max())
        assert np.all(got[:, NR:] == 11.0), 'case {}: padding written'.format(idx)
    # bit-reproducible run to run (fixed-order reductions)
    for r in results[1:]:
        for a, b in zip(results[0], r):
            assert np.array_equal(a, b)
    assert plan.algorithmic_bytes > 0 and plan.algorithmic_bytes_survey >= plan.algorithmic_bytes * 0.5


def test_project_symmetric_flag(handle):
    """``symmetric = 1``: only the lower output chunks are computed, the upper ones are mirrored (exactly symmetric)."""
    from pylrbms_b200._lib import make_project_plan, ProjectDesc
    torch = _torch()
    rng = np.random.default_rng(4)
    n, N = 3000, 100
    B = random_csr(rng, n, n, 4)
    A = sp.csr_matrix(B + B.T)
    A.sort_indices()
    dA = DevCsr(A)
    V = dofmajor(rng, n, N)
    dV = dev(V)
    outs = []
    for sym in (0, 1):
        out = torch.full((N, N), np.nan, dtype=torch.float64, device='cuda')
        d = ProjectDesc(dA.rowptr.data_ptr(), dA.colind.data_ptr(), dA.values.data_ptr(), n, n, dV.data_ptr(), N, N,
                        dV.data_ptr(), N, N, out.data_ptr(), N, 1.0, sym, 0)
        plan = make_project_plan(handle, [d], [dA, dV, out])
        plan.run()
        torch.cuda.synchronize()
        outs.append(out.cpu().numpy())
    ref = V.T @ (A @ V)
    scale = np.abs(V).T @ np.abs(A @ V)
    for got in outs:
        assert (np.abs(got - ref) / scale).max() < 1e-13
    # off-diagonal output chunks are mirrored exactly, diagonal chunks are symmetric up to rounding
    assert np.array_equal(outs[1][64:, :32], outs[1][:32, 64:].T)
    assert (np.abs(outs[1] - outs[1].T) / scale).max() < 1e-13
    # identity operator (plain Gram matrix), symmetric
    out = torch.full((N, N), np.nan, dtype=torch.float64, device='cuda')
    d = ProjectDesc(None, None, None, n, n, dV.data_ptr(), N, N, dV.data_ptr(), N, N, out.data_ptr(), N, 1.0, 1, 0)
    plan = make_project_plan(handle, [d], [dV, out])
    plan.run()
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    assert np.abs(got - V.T @ V).max() < 1e-10 and np.array_equal(got[64:, :32], got[:32, 64:].T)


def test_project_all_zero_operator(handle):
    """An operator without any stored entry projects to exact zeros (no NaN from untouched scratch)."""
    from pylrbms_b200._lib import make_project_plan, ProjectDesc
    torch = _torch()
    rng = np.random.default_rng(3)
    nr = 5000
    A = sp.csr_matrix((nr, nr))
    dA = DevCsr(A)
    V = dev(dofmajor(rng, nr, 20))
    out = torch.full((20, 20), np.nan, dtype=torch.float64, device='cuda')
    d = ProjectDesc(dA.rowptr.data_ptr(), dA.colind.data_ptr(), dA.values.data_ptr(), nr, nr, V.data_ptr(), 20, 20,
                    V.data_ptr(), 20, 20, out.data_ptr(), 20, 1.0)
    plan = make_project_plan(handle, [d], [dA, V, out])
    plan.run()
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), np.zeros((20, 20)))


# ------------------------------------------------------------------------------------------------------------
#  peer-memory exchange kernel (one GPU: the "peers" are local buffers; tools/check_peer_exchange.py is the
#  multi-GPU check against NCCL)
# ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize('n_doubles,n_dst', [(32, 1), (1120, 7), (700_128, 3), (2_800_128, 7)])
def test_peer_push_copies_region_to_every_destination(handle, n_doubles, n_dst):
    from pylrbms_b200._lib import current_stream_ptr
    torch = _torch()
    lib, h = handle.lib, handle.h
    g = torch.Generator(device='cuda').manual_seed(n_doubles + n_dst)
    src = torch.rand(n_doubles + 64, generator=g, dtype=torch.float64, device='cuda')
    dsts = [torch.full((n_doubles + 64,), -1.0, dtype=torch.float64, device='cuda') for _ in range(n_dst)]
    off = 32                                                     # regions start at multiples of 32 doubles
    arr = (C.c_uint64 * n_dst)(*[t.data_ptr() + 8 * off for t in dsts])
    handle.check(lib.lrbms_peer_push(h, C.c_void_p(src.data_ptr() + 8 * off), 8 * n_doubles, n_dst, C.cast(arr, C.c_void_p), 0,
                                     current_stream_ptr()))
    torch.cuda.synchronize()
    for t in dsts:
        assert torch.equal(t[off:off + n_doubles], src[off:off + n_doubles])
        assert bool((t[:off] == -1.0).all()) and bool((t[off + n_doubles:] == -1.0).all())   # nothing outside the region


def test_peer_push_rejects_bad_arguments(handle):
    from pylrbms_b200._lib import LrbmsError, current_stream_ptr
    torch = _torch()
    lib, h = handle.lib, handle.h
    buf = torch.zeros(256, dtype=torch.float64, device='cuda')
    arr = (C.c_uint64 * 2)(buf.data_ptr(), buf.data_ptr() + 1024)
    for n_bytes, n_dst, multicast, src_off in [(24, 1, 0, 0), (64, 17, 0, 0), (64, 2, 1, 0), (64, 1, 0, 8)]:
        with pytest.raises(LrbmsError):
            handle.check(lib.lrbms_peer_push(h, C.c_void_p(buf.data_ptr() + src_off), n_bytes, n_dst, C.cast(arr, C.c_void_p),
                                             multicast, current_stream_ptr()))
    # an empty push is a no-op
    handle.check(lib.lrbms_peer_push(h, C.c_void_p(buf.data_ptr()), 0, 1, C.cast(arr, C.c_void_p), 0, current_stream_ptr()))


# ------------------------------------------------------------------------------------------------------------
#  online: solve / estimate against dense NumPy
# ------------------------------------------------------------------------------------------------------------

def _random_reduced_system(rng, sx, sy, sizes, Q=2, Qf=1, couplings=None):
    """Random SPD block-sparse affine system on an sx x sy subdomain grid (or with the given symmetric list of coupled
    subdomain pairs) + random estimator terms."""
    S = sx * sy
    sizes = np.asarray(sizes, dtype=np.int32)
    assert len(sizes) == S
    off = np.concatenate([[0], np.cumsum(sizes)])
    n = int(off[-1])
    nbh, blocks = [], []
    for s in range(S):
        ix, iy = s % sx, s // sx
        nb = [s]
        if couplings is not None:
            nb += [j for (i, j) in couplings if i == s] + [i for (i, j) in couplings if j == s]
        else:
            if iy > 0: nb.append(s - sx)
            if ix > 0: nb.append(s - 1)
            if ix < sx - 1: nb.append(s + 1)
            if iy < sy - 1: nb.append(s + sx)
        nbh.append(sorted(set(nb)))
        for j in sorted(set(nb)):
            blocks.append((s, j))
    dense = []
    for q in range(Q):
        M = np.zeros((n, n))
        for (i, j) in blocks:
            if i >= j:
                B = rng.standard_normal((sizes[i], sizes[j])) * (0.15 if i != j else 1.0)
                if i == j:
                    B = B @ B.T + (4.0 if q == 0 else 0.5) * sizes[i] * np.eye(sizes[i])
                M[off[i]:off[i + 1], off[j]:off[j + 1]] = B
                M[off[j]:off[j + 1], off[i]:off[i + 1]] = B.T
        dense.append(M)
    rhs = rng.standard_normal((Qf, n))
    return dict(S=S, sizes=sizes, off=off, n=n, nbh=nbh, blocks=blocks, dense=dense, rhs=rhs, Q=Q, Qf=Qf)


def _make_online_plan(handle, sysd, terms_spec=None, rng=None, alpha_first=1, solver=0):
    from pylrbms_b200 import _lib as L
    torch = _torch()
    S, sizes, off, blocks, Q, Qf = sysd['S'], sysd['sizes'], sysd['off'], sysd['blocks'], sysd['Q'], sysd['Qf']
    bi = L.host_i32([b[0] for b in blocks]); bj = L.host_i32([b[1] for b in blocks])
    packed, offsets = [], np.zeros(Q * len(blocks), dtype=np.int64)
    pos = 0
    for q in range(Q):
        for b, (i, j) in enumerate(blocks):
            blk = sysd['dense'][q][off[i]:off[i + 1], off[j]:off[j + 1]]
            offsets[q * len(blocks) + b] = pos
            packed.append(blk.ravel())
            pos += blk.size
    d_blocks = dev(np.concatenate(packed))
    d_rhs = dev(sysd['rhs'])
    nbh_ptr = L.host_i32(np.concatenate([[0], np.cumsum([len(x) for x in sysd['nbh']])]))
    nbh_idx = L.host_i32(np.concatenate(sysd['nbh']))
    keep = [bi, bj, offsets, d_blocks, d_rhs, nbh_ptr, nbh_idx, sizes]
    sysc = L.ReducedSystem()
    sysc.n_sub = S; sysc.basis_sizes = sizes.ctypes.data; sysc.Q = Q; sysc.Qf = Qf; sysc.n_blocks = len(blocks)
    sysc.block_i = bi.ctypes.data; sysc.block_j = bj.ctypes.data; sysc.block_offset = offsets.ctypes.data
    sysc.lhs_blocks = d_blocks.data_ptr(); sysc.rhs = d_rhs.data_ptr()
    sysc.nbh_ptr = nbh_ptr.ctypes.data; sysc.nbh_idx = nbh_idx.ctypes.data
    sysc.solver = solver
    est = None
    if terms_spec is not None:
        mats, terms, moff = [], [], 0
        dsub = [int(sum(sizes[k] for k in sysd['nbh'][i])) for i in range(S)]
        dim_of = {L.VEC_ONE: lambda i: 1, L.VEC_UI: lambda i: int(sizes[i]), L.VEC_UN: lambda i: dsub[i],
                  L.VEC_UR: lambda i: Q * dsub[i]}
        est_terms = []
        for i in range(S):
            for (out_kind, lk, rk, qa, qb, coef) in terms_spec:
                r, c = dim_of[lk](i), dim_of[rk](i)
                M = rng.standard_normal((r, c)) / np.sqrt(max(r, c))
                mats.append(M.ravel())
                terms.append(L.EstimatorTerm(i, out_kind, lk, rk, r, c, qa, qb, coef, moff))
                est_terms.append((i, out_kind, lk, rk, qa, qb, coef, M))
                moff += M.size
        d_mats = dev(np.concatenate(mats))
        tarr = (L.EstimatorTerm * len(terms))(*terms)
        rf2 = L.host_f64(rng.uniform(0.5, 1.5, S)); rsc = L.host_f64(rng.uniform(0.1, 0.3, S))
        tbar = L.host_f64([1.0, 0.7][:Q] + [1.0] * max(0, Q - 2)); that = L.host_f64([1.0, 0.4][:Q] + [1.0] * max(0, Q - 2))
        sysc.n_terms = len(terms); sysc.terms = C.cast(tarr, C.c_void_p); sysc.est_matrices = d_mats.data_ptr()
        sysc.rf_squared = rf2.ctypes.data; sysc.r_scale = rsc.ctypes.data
        sysc.theta_bar = tbar.ctypes.data; sysc.theta_hat = that.ctypes.data
        sysc.alpha_returns_first = alpha_first
        keep += [d_mats, tarr, rf2, rsc, tbar, that]
        est = dict(terms=est_terms, rf2=rf2, rsc=rsc, tbar=tbar, that=that, dsub=dsub)
    p = C.c_void_p()
    handle.check(handle.lib.lrbms_online_plan_create(handle.h, C.byref(sysc), C.byref(p)))
    return L.Plan(handle, p, keep), est


def _run_sweep(handle, plan, sysd, theta, with_est):
    from pylrbms_b200._lib import ptr, current_stream_ptr
    torch = _torch()
    n_mu = theta.shape[0]
    ws = C.c_size_t()
    handle.check(handle.lib.lrbms_online_workspace_bytes(plan.p, n_mu, C.byref(ws)))
    work = torch.empty(max(ws.value, 8), dtype=torch.uint8, device='cuda')
    d_theta = dev(theta)
    u = torch.zeros((n_mu, sysd['n']), dtype=torch.float64, device='cuda')
    info = torch.full((n_mu,), -1, dtype=torch.int32, device='cuda')
    if not with_est:
        handle.check(handle.lib.lrbms_online_solve(plan.p, n_mu, ptr(d_theta), ptr(u), ptr(info), ptr(work), ws.value,
                                                   current_stream_ptr()))
        torch.cuda.synchronize()
        return u.cpu().numpy(), info.cpu().numpy()
    eta = torch.zeros(n_mu, dtype=torch.float64, device='cuda')
    parts = torch.zeros((3, sysd['S'], n_mu), dtype=torch.float64, device='cuda')
    ind = torch.zeros((sysd['S'], n_mu), dtype=torch.float64, device='cuda')
    handle.check(handle.lib.lrbms_online_sweep(plan.p, n_mu, ptr(d_theta), ptr(u), ptr(eta), ptr(parts), ptr(ind), ptr(info),
                                               ptr(work), ws.value, current_stream_ptr()))
    torch.cuda.synchronize()
    return u.cpu().numpy(), info.cpu().numpy(), eta.cpu().numpy(), parts.cpu().numpy(), ind.cpu().numpy()


@pytest.mark.parametrize('sx,sy,sizes', [
    (1, 1, [5]),
    (2, 2, [8, 8, 8, 8]),
    (3, 2, [3, 11, 7, 20, 1, 9]),                    # ragged, not multiples of the 8x8 tile
    (4, 4, [20] * 16),
    (8, 8, [20] * 64),                               # C2 reduced-system shape
])
@pytest.mark.parametrize('solver', [1, 3])
def test_online_solve_matches_dense(handle, sx, sy, sizes, solver):
    """Both solve kernels (lrbms_sm100.h LRBMS_SOLVER_*): 1 the shared-memory window kernel (what AUTO picks when the
    window fits one SM), 3 the block-banded out-of-HBM Cholesky (what AUTO picks for large systems).  Any other solver
    value is rejected at plan creation."""
    from pylrbms_b200._lib import LrbmsError
    rng = np.random.default_rng(10 + sx * 7 + sy)
    sysd = _random_reduced_system(rng, sx, sy, sizes)
    for retired in (2, 4):
        with pytest.raises(LrbmsError, match='unknown solver'):
            _make_online_plan(handle, sysd, solver=retired)
    plan, _ = _make_online_plan(handle, sysd, solver=solver)
    out = C.c_double()
    handle.check(handle.lib.lrbms_plan_info(plan.p, 6, C.byref(out)))
    assert int(out.value) == solver
    n_mu = 37 if sysd['n'] < 500 else 700      # more parameters than resident CTAs for the big case
    theta = np.column_stack([np.ones(n_mu), rng.uniform(0.1, 1.0, n_mu), rng.uniform(0.5, 2.0, n_mu)])
    u, info = _run_sweep(handle, plan, sysd, theta, with_est=False)
    assert np.all(info == 0)
    for m in range(0, n_mu, max(1, n_mu // 25)):
        A = theta[m, 0] * sysd['dense'][0] + theta[m, 1] * sysd['dense'][1]
        f = theta[m, 2] * sysd['rhs'][0]
        ref = np.linalg.solve(A, f)
        # energy-norm relative error and residual check (SURVEY.md section 7 "1e-10 parity through a solve")
        e = u[m] - ref
        assert np.sqrt(e @ A @ e) <= RTOL * np.sqrt(ref @ A @ ref), 'mu {}'.format(m)
        assert np.linalg.norm(A @ u[m] - f) <= RTOL * np.linalg.norm(f) * np.linalg.cond(A) ** 0.5


def _grid3d_couplings(nx, ny, nz):
    idx = lambda x, y, z: (z * ny + y) * nx + x
    out = []
    for z in range(nz):
        for y in range(ny):
            for x in range(nx):
                if x + 1 < nx: out.append((idx(x + 1, y, z), idx(x, y, z)))
                if y + 1 < ny: out.append((idx(x, y + 1, z), idx(x, y, z)))
                if z + 1 < nz: out.append((idx(x, y, z + 1), idx(x, y, z)))
    return out


@pytest.mark.parametrize('shape,N,n_mu', [
    ((16, 16), 20, 300),          # BASELINE configs[2] reduced-system shape: n_red = 5 120, half bandwidth 339
    ((4, 4, 4), 40, 24),          # configs[3] structure (six face neighbours, N = 40) at 4x4x4: n_red = 2 560, half bandwidth 679
    ((5, 3, 2), [33, 40, 17, 64, 1, 40, 25, 40, 40, 9, 40, 40, 31, 40, 40] * 2, 11),   # ragged sizes, not multiples of 64
])
def test_band_solver_large_systems(handle, shape, N, n_mu):
    """The block-banded out-of-HBM Cholesky: AUTO must select it when the factor window exceeds one SM's shared memory, and
    it must reproduce the dense solve in the energy norm (1e-10) with a clean residual; chunked runs (workspace for fewer
    parameters than the batch) must give bit-identical results."""
    torch = _torch()
    from pylrbms_b200._lib import ptr, current_stream_ptr
    rng = np.random.default_rng(5 + len(shape) + shape[0])
    S = int(np.prod(shape))
    sizes = [N] * S if np.isscalar(N) else list(N)
    if len(shape) == 2:
        sysd = _random_reduced_system(rng, shape[0], shape[1], sizes)
    else:
        sysd = _random_reduced_system(rng, S, 1, sizes, couplings=_grid3d_couplings(*shape))
    plan, _ = _make_online_plan(handle, sysd)            # AUTO
    out = C.c_double()
    handle.check(handle.lib.lrbms_plan_info(plan.p, 6, C.byref(out)))
    assert int(out.value) == 3, 'AUTO did not select the band solver'
    theta = np.column_stack([np.ones(n_mu), rng.uniform(0.1, 1.0, n_mu), rng.uniform(0.5, 2.0, n_mu)])
    u, info = _run_sweep(handle, plan, sysd, theta, with_est=False)
    assert np.all(info == 0)
    for m in np.linspace(0, n_mu - 1, 3).astype(int):
        A = theta[m, 0] * sysd['dense'][0] + theta[m, 1] * sysd['dense'][1]
        f = theta[m, 2] * sysd['rhs'][0]
        ref = np.linalg.solve(A, f)
        e = u[m] - ref
        assert np.sqrt(e @ A @ e) <= RTOL * np.sqrt(ref @ A @ ref), 'mu {}'.format(m)
        assert np.linalg.norm(A @ u[m] - f) <= RTOL * np.linalg.norm(f) * np.linalg.cond(A) ** 0.5
    # chunked: a workspace that holds the factors of 5 parameters only
    ws = C.c_size_t()
    handle.check(handle.lib.lrbms_online_workspace_bytes(plan.p, 5, C.byref(ws)))
    d_theta = dev(theta)
    u2 = torch.zeros((n_mu, sysd['n']), dtype=torch.float64, device='cuda')
    info2 = torch.ones(n_mu, dtype=torch.int32, device='cuda')
    work = torch.empty(ws.value, dtype=torch.uint8, device='cuda')
    handle.check(handle.lib.lrbms_online_solve(plan.p, n_mu, ptr(d_theta), ptr(u2), ptr(info2), ptr(work), ws.value,
                                               current_stream_ptr()))
    torch.cuda.synchronize()
    assert np.array_equal(u2.cpu().numpy(), u) and int(info2.abs().sum().item()) == 0
    # not positive definite: reported per parameter, the others unaffected
    theta_bad = theta[:4].copy()
    theta_bad[2, :2] = [-1.0, -1.0]
    ub, infob = _run_sweep(handle, plan, sysd, theta_bad, with_est=False)
    assert infob[2] > 0 and np.all(infob[[0, 1, 3]] == 0) and np.array_equal(ub[[0, 1, 3]], u[[0, 1, 3]])


@pytest.mark.parametrize('solver', [1])
def test_online_solve_is_bit_reproducible(handle, solver):
    """The column pipeline of solve_kernel_v2 lets the two halves of its update warps run the triangular solve and the pair
    loop in opposite order with a single barrier per tile column; a data race there would show as run-to-run differences.
    Same parameters in a different order and batch size must give bit-identical solutions."""
    rng = np.random.default_rng(77)
    sysd = _random_reduced_system(rng, 8, 8, [20] * 64)              # C2 reduced-system shape
    plan, _ = _make_online_plan(handle, sysd, solver=solver)
    n_mu = 900                                                       # six parameters per resident CTA
    theta = np.column_stack([np.ones(n_mu), rng.uniform(0.1, 1.0, n_mu), rng.uniform(0.5, 2.0, n_mu)])
    u1, info1 = _run_sweep(handle, plan, sysd, theta, with_est=False)
    u2, info2 = _run_sweep(handle, plan, sysd, theta, with_est=False)
    assert np.all(info1 == 0) and np.array_equal(u1, u2)
    perm = rng.permutation(n_mu)[:333]
    u3, _ = _run_sweep(handle, plan, sysd, theta[perm], with_est=False)
    assert np.array_equal(u3, u1[perm])
    # every parameter against the dense solve, not a sample
    for m in range(n_mu):
        A = theta[m, 0] * sysd['dense'][0] + theta[m, 1] * sysd['dense'][1]
        ref = np.linalg.solve(A, theta[m, 2] * sysd['rhs'][0])
        e = u1[m] - ref
        assert np.sqrt(e @ A @ e) <= RTOL * np.sqrt(ref @ A @ ref), 'mu {}'.format(m)


def test_online_solve_barrier_schedule(handle):
    """A sparsity pattern in which a target has a pair with source column J - 2 but no carrier tile in column J - 1: the
    symbolic phase must pick the barrier schedule of solve_kernel_v2 and the kernel must still reproduce the dense solve."""
    from pylrbms_b200._lib import Symbolic
    rng = np.random.default_rng(21)
    # subdomains 2 and 3 couple to 0 (fill in (3, 2) from source 0); subdomain 1 is isolated: no tile (3, 1) or (2, 1)
    couplings = [(2, 0), (3, 0), (5, 4), (6, 4), (6, 2)]
    sizes = [8, 8, 8, 8, 16, 8, 11]
    sysd = _random_reduced_system(rng, len(sizes), 1, sizes, couplings=couplings)
    sym = Symbolic(sysd['sizes'], [b[0] for b in sysd['blocks']], [b[1] for b in sysd['blocks']])
    assert sym.staggered == 0
    plan, _ = _make_online_plan(handle, sysd)
    n_mu = 41
    theta = np.column_stack([np.ones(n_mu), rng.uniform(0.1, 1.0, n_mu), rng.uniform(0.5, 2.0, n_mu)])
    u, info = _run_sweep(handle, plan, sysd, theta, with_est=False)
    assert np.all(info == 0)
    for m in range(n_mu):
        A = theta[m, 0] * sysd['dense'][0] + theta[m, 1] * sysd['dense'][1]
        ref = np.linalg.solve(A, theta[m, 2] * sysd['rhs'][0])
        e = u[m] - ref
        assert np.sqrt(e @ A @ e) <= RTOL * np.sqrt(ref @ A @ ref), 'mu {}'.format(m)


def test_online_solve_flags_indefinite_system(handle):
    rng = np.random.default_rng(5)
    sysd = _random_reduced_system(rng, 2, 2, [6, 6, 6, 6])
    plan, _ = _make_online_plan(handle, sysd)
    theta = np.array([[1.0, 0.5, 1.0], [1.0, -50.0, 1.0]])     # second parameter makes A indefinite
    u, info = _run_sweep(handle, plan, sysd, theta, with_est=False)
    assert info[0] == 0 and info[1] > 0


def _estimate_reference(sysd, est, theta, u, alpha_first=True):
    from pylrbms_b200 import _lib as L
    S, sizes, off, Q = sysd['S'], sysd['sizes'], sysd['off'], sysd['Q']
    n_mu = theta.shape[0]
    parts = np.zeros((3, S, n_mu))
    for m in range(n_mu):
        th = theta[m]
        for (i, out_kind, lk, rk, qa, qb, coef, M) in est['terms']:
            un = np.concatenate([u[m, off[k]:off[k + 1]] for k in sysd['nbh'][i]])
            ur = np.concatenate([np.concatenate([th[q] * u[m, off[k]:off[k + 1]] for q in range(Q)]) for k in sysd['nbh'][i]])
            vec = {L.VEC_ONE: np.ones(1), L.VEC_UI: u[m, off[i]:off[i + 1]], L.VEC_UN: un, L.VEC_UR: ur}
            c = coef * (th[qa] if qa >= 0 else 1.0) * (th[qb] if qb >= 0 else 1.0)
            parts[out_kind, i, m] += c * (vec[lk] @ (M @ vec[rk]))
        parts[1, :, m] = (est['rf2'] + parts[1, :, m]) * est['rsc']
    eta = np.zeros(n_mu)
    ind = np.zeros((S, n_mu))
    for m in range(n_mu):
        rb = theta[m, :Q] / est['tbar'][:Q]; rh = theta[m, :Q] / est['that'][:Q]
        a_bar = rb[0] if alpha_first else rb.min()
        a_hat = rh[0] if alpha_first else rh.min()
        g_bar = rb.max()
        nc, r, df = parts[0, :, m], parts[1, :, m], parts[2, :, m]
        eta[m] = (np.sqrt(g_bar) * np.linalg.norm(nc) + np.linalg.norm(r + df) / np.sqrt(a_hat)) / np.sqrt(a_bar)
        ind[:, m] = (2.0 / a_bar) * (g_bar * nc ** 2 + (r + df) ** 2 / a_hat)
    return parts, eta, ind


@pytest.mark.parametrize('sx,sy,sizes,alpha_first', [
    (2, 2, [8, 8, 8, 8], 1),
    (3, 2, [3, 11, 7, 20, 1, 9], 0),
    (4, 4, [20] * 16, 1),
])
def test_online_sweep_estimator_matches_numpy(handle, sx, sy, sizes, alpha_first):
    from pylrbms_b200 import _lib as L
    from pylrbms_b200._lib import current_stream_ptr as _cs
    rng = np.random.default_rng(20 + sx)
    sysd = _random_reduced_system(rng, sx, sy, sizes)
    spec = [  # the term set of reference estimators.py:71-85 (shapes as in SURVEY.md section 8a a7-a9)
        (L.OUT_NC, L.VEC_UN, L.VEC_UN, -1, -1, 1.0),
        (L.OUT_R, L.VEC_ONE, L.VEC_UR, -1, -1, -2.0),
        (L.OUT_R, L.VEC_UR, L.VEC_UR, -1, -1, 1.0),
        (L.OUT_DF, L.VEC_UI, L.VEC_UI, 0, 0, 1.0), (L.OUT_DF, L.VEC_UI, L.VEC_UI, 0, 1, 1.0),
        (L.OUT_DF, L.VEC_UI, L.VEC_UI, 1, 0, 1.0), (L.OUT_DF, L.VEC_UI, L.VEC_UI, 1, 1, 1.0),
        (L.OUT_DF, L.VEC_UR, L.VEC_UR, -1, -1, 1.0),
        (L.OUT_DF, L.VEC_UI, L.VEC_UR, 0, -1, 2.0), (L.OUT_DF, L.VEC_UI, L.VEC_UR, 1, -1, 2.0),
    ]
    plan, est = _make_online_plan(handle, sysd, spec, rng, alpha_first=alpha_first)
    n_mu = 45                       # not a multiple of the 32-parameter tile
    theta = np.column_stack([np.ones(n_mu), rng.uniform(0.1, 1.0, n_mu), np.ones(n_mu)])
    # every SM's shared memory holds NaNs before the sweep: rows of the staged neighbourhood vectors that a term reads
    # beyond its own extent (unaligned slices, neighbourhoods smaller than the largest) must have been zero-filled
    handle.check(handle.lib.lrbms_debug_poison_shared(handle.h, _cs()))
    u, info, eta, parts, ind = _run_sweep(handle, plan, sysd, theta, with_est=True)
    assert np.all(np.isfinite(eta)) and np.all(np.isfinite(parts))
    assert np.all(info == 0)
    rparts, reta, rind = _estimate_reference(sysd, est, theta, u, alpha_first=bool(alpha_first))
    for kind in range(3):
        assert rel(parts[kind], rparts[kind]) < RTOL
    assert rel(eta, reta) < RTOL
    assert rel(ind, rind) < RTOL
    # eta max / argmax
    torch = _torch()
    mx = torch.zeros(1, dtype=torch.float64, device='cuda'); am = torch.zeros(1, dtype=torch.int64, device='cuda')
    from pylrbms_b200._lib import ptr, current_stream_ptr
    handle.check(handle.lib.lrbms_eta_max(handle.h, n_mu, ptr(dev(eta)), ptr(mx), ptr(am), current_stream_ptr()))
    assert mx.item() == eta.max() and am.item() == int(np.argmax(eta))
