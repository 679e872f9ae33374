"""The LRBMS reductor: offline Galerkin projection of every block, coupling and estimator operator (K1 + K2).

Drop-in for the reference's ``LRBMSReductor`` (``reductor.py:17-78``) and the fork-only base class it delegates to,
``pymor.reductors.system.GenericRBSystemReductor`` (SURVEY.md Appendix A.3-A.5): same constructor, ``bases``
dictionary keyed by space id, ``extend_basis`` / ``extend_basis_local`` / ``reduce`` / ``reconstruct`` /
``reconstruct_local``.

How ``reduce()`` differs in execution (not in result):

* the reference projects block by block and vector by vector -- ``N_j`` ``mv`` calls plus ``N_i N_j`` scalar dots per
  block, a Python loop over every operator of ``d.operators`` (``reductor.py:70`` -> ``project_system``).  Here the
  operator *structure* is read once by a planner that emits one descriptor per output block; **all** blocks of
  **all** operators go into a single batched fused projection plan (``lrbms_project_plan_create``), preceded by at
  most two batched SpMM stages (the Oswald / flux-reconstruction images of the bases, ``reductor.py:36-60``, and
  the divergence images needed by ``r_dd``, reference ``discretize...:747-748``);
* the OI / RT image bases are written straight into per-target-subdomain *slabs*
  ``[component_i of bases['OI_k']]_{k in N(i)}`` so the estimator Grams ``nc_i, r_dd_i, df_bb_i, df_ab_i, r_fd_i`` are
  one projection each over the whole neighbourhood instead of ``|N(i)|^2`` block projections;
* reduced operators stay block sparse (no ``unblock`` to dense ``n_red^2`` storage, SURVEY.md row a10);
  ``to_dense()`` reproduces the unblocked matrix for comparison.

With ``torch.distributed`` initialised and ``shard=True`` each rank projects the blocks owned by its strip of
subdomains and the reduced data is exchanged with one broadcast per rank region (the all-gather that the
reference's dead ``Allreduce(SUM)`` of zero-padded blocks amounts to, ``reductor.py:93``).
"""
from __future__ import annotations

import numpy as np

import ctypes as C

from . import _lib
from ._lib import Handle, current_stream_ptr, make_project_plan, make_spmm_plan, ptr
from .distributed import exchange_regions, owner_rank, rank_and_world, region_layout
from .kernels import project_desc, spmm_desc
from .operators import (BlockColumnOperator, BlockEmbeddingOperator, BlockOperator, BlockProjectionOperator,
                        BlockRowOperator, Concatenation, CsrOperator, LincombOperator, VectorFunctional)
from .reduced import ReducedBlockOperator, ReducedFluxReconstruction, ReducedModel, ReducedOswaldInterpolation, SuperBlock
from .vectorarray import BlockVectorArray, GpuVectorArray, ReducedVectorArray


def _torch():
    import torch
    return torch


class ExtensionError(Exception):
    """Raised by ``extend_basis`` when nothing could be added (pyMOR ``ExtensionError``; caught at reference
    ``online_adaptive_lrbms.py:118``)."""


# ----------------------------------------------------------------------------------------------------------
#  generic reductor: bases, extension, reconstruction
# ----------------------------------------------------------------------------------------------------------

class GenericRBSystemReductor:
    def __init__(self, d, bases=None, products=None):
        self.d = d
        subs = d.solution_space.subspaces
        self._sub_index = {s.id: k for k, s in enumerate(subs)}
        self.bases = {s.id: s.empty() for s in subs}
        if bases is not None:
            items = bases.items() if isinstance(bases, dict) else zip([s.id for s in subs], bases)
            for k, v in items:
                space = subs[self._sub_index[k]]
                self.bases[k] = v.copy() if isinstance(v, GpuVectorArray) else space.from_data(v)
        self.products = list(products) if products is not None else [None] * len(subs)
        assert len(self.products) == len(subs)

    # -- basis extension: Gram-Schmidt in the local product (pyMOR gram_schmidt semantics, re-orthogonalisation)
    def extend_basis_local(self, U, atol=1e-13, rtol=1e-13, reiteration_threshold=1e-1):
        sid = U.space.id
        basis = self.bases[sid]
        product = self.products[self._sub_index[sid]]
        added = 0
        for k in range(len(U)):
            v = U[k]
            norm = initial_norm = float(np.sqrt(max(self._norm2(v, product), 0.0)))
            if norm < atol:
                continue
            if len(basis) > 0:
                while True:
                    Pv = product.apply(v) if product is not None else v
                    coeff = basis.dot(Pv)[:, 0]                               # <b_j, v>_P for all j in one launch
                    v.axpy(-1.0, basis.lincomb(coeff[None, :]))
                    old_norm, norm = norm, float(np.sqrt(max(self._norm2(v, product), 0.0)))
                    if norm / initial_norm < rtol or norm / old_norm >= reiteration_threshold:
                        break
                if norm / initial_norm < rtol:
                    continue
            v.scal(1.0 / norm)
            basis.append(v)
            added += 1
        if added == 0:
            raise ExtensionError
        return added

    @staticmethod
    def _norm2(v, product):
        if product is None:
            return float(v.pairwise_dot(v)[0])
        return float(product.pairwise_apply2(v, v)[0])

    def extend_basis(self, U, method='gram_schmidt', pod_modes=1, pod_rtol=1e-13):
        """Extend every local basis by the restrictions of the block array ``U`` (pyMOR ``extend_basis``).

        ``method='gram_schmidt'``: each restriction goes through :meth:`extend_basis_local`, vector by vector.
        ``method='pod'``: all subdomains at once -- the projection error of ``U`` onto the current bases (two classical
        Gram-Schmidt passes in the local product), a POD of it per subdomain and at most ``pod_modes`` modes appended
        whose singular value exceeds ``pod_rtol`` times the largest local norm of ``U``; the modes are orthonormalised
        against the basis and among themselves (pyMOR ``pod_orthonormalize=True``).  See :func:`_extend_basis_pod`.
        Either way :class:`ExtensionError` is raised when no subdomain received a vector."""
        if method == 'pod':
            return _extend_basis_pod(self, U, int(pod_modes), float(pod_rtol))
        if method != 'gram_schmidt':
            raise ValueError("extend_basis: method must be 'gram_schmidt' or 'pod', not {!r}".format(method))
        ok = False
        for blk in U._blocks:
            try:
                self.extend_basis_local(blk)
                ok = True
            except ExtensionError:
                pass
        if not ok:
            raise ExtensionError

    # -- reconstruction (reference online_adaptive_lrbms.py:143; reductor.py:76)
    def _offsets(self):
        subs = self.d.solution_space.subspaces
        return np.concatenate([[0], np.cumsum([len(self.bases[s.id]) for s in subs])]).astype(np.int64)

    def reconstruct_local(self, u, space_id):
        """pyMOR semantics ``RB[:u.dim].lincomb(u)``: a solution of an earlier reduced model stays reconstructible after the
        basis was extended (the enrichment loop does exactly that, reference ``reductor.py:75-78``)."""
        k = self._sub_index[space_id]
        dims = getattr(u, 'block_dims', None)
        offs = np.concatenate([[0], np.cumsum(dims)]).astype(np.int64) if dims is not None else self._offsets()
        coeff = u.device_tensor[:, offs[k]:offs[k + 1]] if isinstance(u, ReducedVectorArray) else \
            np.atleast_2d(np.asarray(u.data if hasattr(u, 'data') else u))[:, offs[k]:offs[k + 1]]
        basis = self.bases[space_id]
        n = int(offs[k + 1] - offs[k])
        if n < len(basis):
            basis = basis[:n]
        return basis.lincomb(coeff)

    def reconstruct(self, u):
        subs = self.d.solution_space.subspaces
        return self.d.solution_space.make_array([self.reconstruct_local(u, s.id) for s in subs])

    def reduce(self):
        return self._reduce()


# ----------------------------------------------------------------------------------------------------------
#  POD extension of every local basis in one pass
# ----------------------------------------------------------------------------------------------------------

def _run_project(descs, keep):
    """One projection plan over ``descs`` (at most one descriptor per subdomain and quantity), run once."""
    if descs:
        plan = make_project_plan(Handle.get(), descs, keep)
        plan.run()
        plan.destroy()


def _inner_with_bases(csrs, Xs, bases, width):
    """``C[m, off_i + j] = <x_{i,m}, v_{i,j}>_{P_i}`` for all subdomains with one projection plan: ``(width, sum N_i)``, the
    coefficient layout of ``lrbms_recon_error``."""
    torch = _torch()
    offs = np.concatenate([[0], np.cumsum([len(V) for V in bases])]).astype(np.int64)
    C = torch.zeros((width, int(offs[-1])), dtype=torch.float64, device='cuda')
    descs = [project_desc(csr, X.dim, X.device_ptr, X.ld, len(X), V.device_ptr, V.ld, len(V), C.data_ptr() + 8 * int(offs[i]),
                          int(offs[-1])) for i, (csr, X, V) in enumerate(zip(csrs, Xs, bases)) if len(X) and len(V)]
    _run_project(descs, [C])
    return C


def _grams(csrs, arrays_list, width):
    """``G[t, i] = X_i^T P_i X_i`` (``width x width``, leading ``len(X_i)`` rows / columns) for every array list ``t`` and
    subdomain ``i``, symmetric descriptors, one projection plan; returned on the host."""
    torch = _torch()
    S = len(csrs)
    G = torch.zeros((len(arrays_list), S, width, width), dtype=torch.float64, device='cuda')
    descs = []
    for t, Xs in enumerate(arrays_list):
        for i, (csr, X) in enumerate(zip(csrs, Xs)):
            if len(X):
                descs.append(project_desc(csr, X.dim, X.device_ptr, X.ld, len(X), X.device_ptr, X.ld, len(X),
                                          G[t, i].data_ptr(), width, symmetric=csr is None or csr.symmetric))
    _run_project(descs, [G])
    G = G.cpu().numpy()
    return 0.5 * (G + np.swapaxes(G, -1, -2))


def _combine(views, counts, coeffs):
    """``Y_i = X_i A_i`` for every subdomain in one ``lrbms_recon_error`` launch: ``views[i]`` holds ``counts[i]`` columns,
    ``coeffs[i]`` is ``(counts[i], m_i)``.  Returns the dof-major ``(n, >= max m_i)`` result; columns past ``m_i`` of a
    subdomain are zero."""
    torch = _torch()
    from .kernels import recon_error
    from .vectorarray import _round_cap
    width = max(a.shape[1] for a in coeffs)
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    coef = np.zeros((width, int(offs[-1])))
    for i, a in enumerate(coeffs):
        coef[:a.shape[1], offs[i]:offs[i + 1]] = -a.T             # e = 0 - X (-A) = X A
    n = sum(X.dim for X in views)
    zero = torch.zeros((n, _round_cap(width)), dtype=torch.float64, device='cuda')
    Y = torch.empty((n, _round_cap(width)), dtype=torch.float64, device='cuda')
    return recon_error(views, counts, zero, torch.from_numpy(coef).cuda(), Y)


def _views(subs, rows, X, counts):
    """The subdomain blocks of a dof-major ``(n, >= max counts)`` buffer as arrays of ``counts[i]`` vectors (no copy)."""
    return [s.from_dofmajor(X[rows[i]:rows[i + 1]], counts[i]) for i, s in enumerate(subs)]


def _subtract_projection(subs, rows, csrs, bases, X, counts):
    """``X_i - V_i (V_i^T P_i X_i)`` for every subdomain: one projection plan and one ``lrbms_recon_error`` launch."""
    torch = _torch()
    from .kernels import recon_error
    from .vectorarray import _round_cap
    width = max(counts)
    C = _inner_with_bases(csrs, _views(subs, rows, X, counts), bases, width)
    out = torch.zeros((X.shape[0], _round_cap(width)), dtype=torch.float64, device='cuda')
    if C.shape[1] == 0:                      # every basis is empty
        out[:, :width] = X[:, :width]
        return out
    return recon_error(bases, [len(V) for V in bases], X, C, out)


def pod_modes_from_gram(G, norm_max, pod_modes, pod_rtol):
    """Host half of the POD extension for one subdomain: ``(W, sigma)`` of the at most ``pod_modes`` leading eigenpairs of
    the Gram matrix ``G`` of the projection error with ``sigma > pod_rtol * norm_max``, in descending order, each
    eigenvector signed so that its entry of largest magnitude is positive."""
    lam, W = np.linalg.eigh(G)
    lam, W = lam[::-1], W[:, ::-1]
    sigma = np.sqrt(np.maximum(lam, 0.0))
    m = min(int(pod_modes), int(np.count_nonzero(sigma > pod_rtol * norm_max)))
    W, sigma = W[:, :m].copy(), sigma[:m]
    for j in range(m):
        if W[np.argmax(np.abs(W[:, j])), j] < 0:
            W[:, j] = -W[:, j]
    return W, sigma


def cholesky_leading(G):
    """Lower Cholesky factor of the largest leading block of ``G`` that is numerically positive definite: ``(m, L)``.
    A mode that the re-orthogonalisation reduced to rounding noise is dropped with everything after it."""
    for m in range(G.shape[0], 0, -1):
        try:
            return m, np.linalg.cholesky(G[:m, :m])
        except np.linalg.LinAlgError:
            continue
    return 0, np.zeros((0, 0))


def _extend_basis_pod(reductor, U, pod_modes, pod_rtol):
    """``extend_basis(U, method='pod')`` on the device.  Per subdomain ``i`` (``U_i``: restriction of ``U``, ``V_i``: basis,
    ``P_i``: the reductor's product, the Euclidean one when it is None):

    1. ``R = U - V (V^T P U)`` twice (CGS2): one projection plan and one ``lrbms_recon_error`` launch per pass;
    2. ``G_i = R_i^T P_i R_i`` and ``U_i^T P_i U_i`` in one plan, to the host;
    3. host ``eigh``: at most ``pod_modes`` modes with ``sigma > pod_rtol max_j |u_{i,j}|_{P_i}``;
    4. ``Y_i = R_i W_i / sigma_i`` (one launch), one more CGS pass against ``V``, Cholesky QR of ``Y_i^T P_i Y_i`` (one plan, one
       launch), and the result is appended.

    Returns the number of vectors appended to each basis; raises :class:`ExtensionError` when that is zero everywhere."""
    from .error_analysis import _dofmajor
    if pod_modes < 1:
        raise ValueError('pod_modes must be at least 1')
    subs = reductor.d.solution_space.subspaces
    S, k = len(subs), len(U)
    if len(U._blocks) != S or any(b.dim != s.dim for b, s in zip(U._blocks, subs)):
        raise ValueError('U is not an array of the solution space of the reductor')
    if k == 0:
        raise ExtensionError
    rows = np.concatenate([[0], np.cumsum([s.dim for s in subs])]).astype(np.int64)
    n = int(rows[-1])
    bases = [reductor.bases[s.id] for s in subs]
    csrs = [p.csr if p is not None else None for p in reductor.products]
    u = _dofmajor(U, n, k)
    R = u
    for _ in range(2):
        R = _subtract_projection(subs, rows, csrs, bases, R, [k] * S)
    views = lambda X, counts: _views(subs, rows, X, counts)
    G, H = _grams(csrs, [views(R, [k] * S), views(u, [k] * S)], k)
    modes = [pod_modes_from_gram(G[i], np.sqrt(np.maximum(np.diag(H[i]), 0.0)).max(), pod_modes, pod_rtol)
             for i in range(S)]
    counts = [W.shape[1] for W, _ in modes]
    if max(counts) == 0:
        raise ExtensionError
    Y = _combine(views(R, [k] * S), [k] * S, [W / sigma for W, sigma in modes])
    Y = _subtract_projection(subs, rows, csrs, bases, Y, counts)
    Gy = _grams(csrs, [views(Y, counts)], max(counts))[0]
    factors = [cholesky_leading(Gy[i, :counts[i], :counts[i]]) for i in range(S)]
    counts = [m for m, _ in factors]
    if max(counts) == 0:
        raise ExtensionError
    inv = [np.linalg.inv(L).T if m else np.zeros((0, 0)) for m, L in factors]   # Z = Y L^{-T}
    Z = _combine(views(Y, counts), counts, inv)
    for i, s in enumerate(subs):
        if counts[i]:
            bases[i].append(s.from_dofmajor(Z[rows[i]:rows[i + 1]], counts[i]))
    return counts


# ----------------------------------------------------------------------------------------------------------
#  projection planner
# ----------------------------------------------------------------------------------------------------------

class _ArrayRef:
    """A dof-major device array seen by the kernels: pointer, row stride, number of vectors, number of dofs.

    ``key`` names the array across two plans of one reductor and ``labels`` says what every column *is* -- row ``c`` is
    ``(k, q, a)``: image under the q-th affine component (0 for the basis itself and its Oswald image) of basis vector
    ``a`` of subdomain ``k``; ``k = -1`` marks data that never changes (right-hand sides).  Incremental re-projection
    (SURVEY.md section 8f rank 2) uses both to tell old columns from the ones an enrichment appended."""
    __slots__ = ('ptr', 'ld', 'N', 'dim', 'keep', 'stage', 'key', 'labels')

    def __init__(self, ptr, ld, N, dim, keep=None, stage=0, key=None, labels=None):
        self.ptr, self.ld, self.N, self.dim, self.keep = int(ptr), int(ld), int(N), int(dim), keep
        self.stage = stage        # SpMM stage that produces the data (0: bases and their OI / RT images)
        self.key = key if key is not None else ('static', int(ptr), int(ld), int(N))
        self.labels = labels if labels is not None else \
            np.stack([np.full(int(N), -1), np.zeros(int(N), dtype=np.int64), np.arange(int(N))], axis=1).astype(np.int64)

    _of_cache = {}

    @staticmethod
    def of(arr):
        """Reference of a vector array; cached by object for the duration of one ``build_plan`` (cleared there)."""
        hit = _ArrayRef._of_cache.get(id(arr))
        if hit is None or hit.keep is not arr:
            hit = _ArrayRef._of_cache[id(arr)] = _ArrayRef(arr.device_ptr, arr.ld, len(arr), arr.dim, arr,
                                                           key=getattr(arr, '_plan_key', None),
                                                           labels=getattr(arr, '_plan_labels', None))
        return hit


def _labels(k, qs, n):
    """Column labels ``(k, q, a)`` in q-major order for ``n`` basis vectors of subdomain ``k``."""
    qs = list(qs)
    return np.stack([np.full(len(qs) * n, k), np.repeat(qs, n), np.tile(np.arange(n), len(qs))], axis=1).astype(np.int64)


class _Planner:
    """Collects SpMM stages and projection jobs for one ``reduce()``; owns the reduced output buffer."""

    def __init__(self, handle, owner_rank_of=None, rank=0, world=1, prev=None):
        self.h = handle
        # incremental re-projection: the previous plan of this reductor (its output buffer holds every old entry) and the
        # basis sizes it was built for; None -> everything is projected from scratch
        self.prev = prev
        self.N_old = list(prev.block_dims) if prev is not None else None
        self.narrow_left = True        # L^T A R with a narrow L and a wide R is computed as (A^T L)^T R
        self.fuse_cache = None         # {ids of the chained matrices: (fused CsrOperator, keepalive)}; None: chains are not fused
        self.job_index = {}            # job key -> (token, L labels, R labels)
        self.inc_jobs = []             # jobs that exist in the previous plan: only new rows / columns are computed
        self.gathers, self.scatters = [], []
        self.jobs = []                 # (owner, csr|None, n_rows, L ref, R ref, out offset, ldo, alpha)
        self.spmm_stages = [[]]
        self._spmm_cache = {}
        self._out_size = 0
        self.keep = []
        self.owner_rank_of = owner_rank_of or (lambda owner: 0)
        self.rank, self.world = rank, world
        self.scratch_pool, self.scratch_used = None, []
        self._arena, self.arena_block = [], 64 * 1024 * 1024          # arena blocks of 64 Mi doubles (512 MB)
        self.scratch_owner = None     # the reductor: keeps one projection scratch buffer for all of its plans
        self.unit_rows = 0
        self.timings = {}
        self._region_sizes = [0] * world
        self._pending = []            # deferred allocations: (owner_rank, size) -> resolved into offsets at finalize

    def _scratch(self, rows, ld):
        """Scratch arrays are carved out of a few large arena blocks (one device allocation per 512 MB instead of one per
        array: 192 arrays at 8 x 8 subdomains) and recycled from the previous plan of the same reductor."""
        pool = self.scratch_pool
        key = (rows, ld)
        if pool is not None and pool.get(key):
            t = pool[key].pop()
        else:
            t = self._arena_take(rows * ld).view(rows, ld)
        self.scratch_used.append((key, t))
        return t

    def _arena_take(self, n, zero=False):
        """``n`` doubles from the current arena block (32-double aligned); a new block when it is exhausted."""
        torch = _torch()
        n_al = (int(n) + 31) // 32 * 32
        blk = self._arena[-1] if self._arena else None
        if blk is None or blk[1] + n_al > blk[0].numel():
            size = max(n_al, self.arena_block)
            blk = [torch.empty(size, dtype=torch.float64, device='cuda'), 0]
            self._arena.append(blk)
        t = blk[0][blk[1]:blk[1] + int(n)]
        blk[1] += n_al
        if zero:
            t.zero_()
        return t

    # -- output allocation: grouped per owner rank so that each rank's results are one contiguous region
    def alloc(self, owner, size):
        r = self.owner_rank_of(owner)
        token = len(self._pending)
        self._pending.append((r, int(size)))
        return token

    def mine(self, owner):
        return self.owner_rank_of(owner) == self.rank

    def spmm(self, owner, csr, V):
        """Schedule ``W = csr @ V`` (cached) one stage after the one that produces ``V``; returns the ref of ``W``."""
        key = (id(csr), V.ptr, V.ld, V.N)
        if key in self._spmm_cache:
            return self._spmm_cache[key]
        stage = V.stage + 1
        ld = max(4, (V.N + 3) // 4 * 4)
        W = self._scratch(max(1, csr.shape[0]), ld)
        ref = _ArrayRef(W.data_ptr(), ld, V.N, csr.shape[0], W, stage, key=('spmm', id(csr), V.key), labels=V.labels)
        while len(self.spmm_stages) <= stage:
            self.spmm_stages.append([])
        if self.mine(owner):
            self.spmm_stages[stage].append(spmm_desc(csr, V.ptr, V.ld, V.N, W.data_ptr(), ld))
        self.keep += [csr, V.keep, W]
        self._spmm_cache[key] = ref
        return ref

    def project(self, owner, csr, L, R, alpha=1.0):
        """Schedule ``alpha * L^T csr R`` (``csr=None``: identity); returns the output token (row-major ``L.N x R.N``)."""
        token = self.alloc(owner, L.N * R.N)
        if L.N and R.N:
            # work of this block in the units the library sizes its row partition with, summed over ALL ranks' blocks: every
            # rank cuts the rows of a block exactly like the unsharded plan (bit-identical sharded results)
            n_r = csr.shape[0] if csr is not None else L.dim
            gram = L.N > 40 and R.N > 40
            cw = 80 if gram else 40
            self.unit_rows += (-(-L.N // cw)) * (-(-R.N // cw)) * n_r * (3 if gram else 1)
        key = (id(csr) if csr is not None else None, L.key, R.key, float(alpha))
        self.job_index[key] = (token, L.labels, R.labels)
        if L.N and R.N and self.mine(owner):
            n_rows = csr.shape[0] if csr is not None else L.dim
            sym = (L.ptr == R.ptr and L.ld == R.ld and L.N == R.N and (csr is None or csr.symmetric))
            if self.prev is not None and key in self.prev.job_index:
                self.inc_jobs.append((token, csr, n_rows, L, R, alpha, sym, key))
            else:
                self.jobs.append((token, csr, n_rows, L, R, R.N, alpha, sym and L.N > 40))
        self.keep += [csr, L.keep, R.keep]
        return token

    # -- incremental jobs ------------------------------------------------------------------------------------------
    def _is_new(self, labels):
        k, a = labels[:, 0], labels[:, 2]
        n_old = np.asarray(self.N_old + [0], dtype=np.int64)        # k = -1 (static data) -> index -1 -> 0, never new
        return (k >= 0) & (a >= n_old[k])

    def _gather_ref(self, ref, cols):
        """A compact copy of columns ``cols`` of ``ref`` (cached per array), filled at run time -- after the SpMM stages
        that produce ``ref`` -- by one ``lrbms_va_copy_cols`` launch."""
        if ref.key in self._gather_cache:
            return self._gather_cache[ref.key]
        torch = _torch()
        n = len(cols)
        ld = max(4, (n + 3) // 4 * 4)
        buf = torch.zeros((max(1, ref.dim), ld), dtype=torch.float64, device='cuda')
        idx = np.ascontiguousarray(cols, dtype=np.int32)
        src_ptr, src_ld, dim, h = ref.ptr, ref.ld, ref.dim, self.h

        def run():
            for c0 in range(0, n, 256):
                cnt = min(256, n - c0)
                chunk = np.ascontiguousarray(idx[c0:c0 + cnt])
                h.check(h.lib.lrbms_va_copy_cols(h.h, dim, cnt, ptr(chunk), src_ptr, src_ld, buf.data_ptr(), ld, c0,
                                                 current_stream_ptr()))
        if dim and n:
            self.gathers.append(run)
        out = _ArrayRef(buf.data_ptr(), ld, n, ref.dim, [buf, ref.keep])
        self._gather_cache[ref.key] = out
        return out

    @staticmethod
    def _codes(labels):
        """One sortable integer per column label ``(k, q, a)``."""
        return ((labels[:, 0] + 1) * 64 + labels[:, 1]) * (1 << 20) + labels[:, 2]

    def _plan_incremental(self, base, descs):
        """Turn every incremental job into (at most) two narrow projections plus one entry of the block-remap launch:

            G[old, old]  <- the previous plan's output
            G[:, new]     = alpha L^T A R[:, new]                             (all rows x new columns)
            G[new, old]   = (alpha R^T A^T L[:, new])^T restricted to old     (new rows; from G[:, new]^T if symmetric)
        """
        torch = _torch()
        prev = self.prev
        self._gather_cache = {}
        todo, maps, tmp_sizes = [], [], []
        map_cache = {}

        def col_map(ref, plabels):
            """``[N]`` int32: index in the previous array for old columns, ``-(1 + rank among the new ones)`` for new ones;
            None if an old column is missing from the previous array."""
            ck = (ref.key, id(plabels))
            if ck not in map_cache:
                new = self._is_new(ref.labels)
                m = np.empty(ref.N, dtype=np.int32)
                m[new] = -1 - np.arange(int(new.sum()), dtype=np.int32)
                old_codes = self._codes(ref.labels[~new])
                pc = self._codes(plabels)
                order = np.argsort(pc, kind='stable')
                pos = np.searchsorted(pc[order], old_codes)
                ok = len(pc) > 0 or len(old_codes) == 0
                if ok and len(old_codes):
                    pos = np.minimum(pos, len(pc) - 1)
                    ok = bool(np.all(pc[order][pos] == old_codes))
                if ok and len(old_codes):
                    m[~new] = order[pos].astype(np.int32)
                map_cache[ck] = (m, np.nonzero(new)[0]) if ok else None
            return map_cache[ck]

        for (token, csr, n_rows, L, R, alpha, sym, key) in self.inc_jobs:
            ptoken, pL, pR = prev.job_index[key]
            rm, cm = col_map(L, pL), col_map(R, pR)
            if rm is None or cm is None:
                # an "old" column the previous plan did not have: project this block from scratch
                self.jobs.append((token, csr, n_rows, L, R, R.N, alpha, sym and L.N > 40))
                continue
            (row_map, rows_new), (cmap, cols_new) = rm, cm
            n_cn, n_rn = len(cols_new), len(rows_new)
            need_rows = n_rn > 0 and n_cn < R.N and not sym
            todo.append((token, ptoken, L.N, R.N, len(pR), n_cn, n_rn if need_rows else 0, len(maps), len(maps) + 1,
                         len(tmp_sizes), len(tmp_sizes) + 1))
            maps += [row_map, cmap]
            tmp_sizes += [L.N * n_cn, R.N * n_rn if need_rows else 0]
            if n_cn:
                Rn = self._gather_ref(R, cols_new)
                descs.append((csr, n_rows, L, Rn, len(tmp_sizes) - 2, alpha))
            if need_rows:
                Ln = self._gather_ref(L, rows_new)
                csr_t = csr.T if csr is not None else None
                descs.append((csr_t, csr_t.shape[0] if csr_t is not None else R.dim, R, Ln, len(tmp_sizes) - 1, alpha))
                self.keep.append(csr_t)
        # one buffer for every narrow projection result, one for every index map
        tmp_off = np.concatenate([[0], np.cumsum(tmp_sizes)]).astype(np.int64)
        tmp = torch.zeros(max(1, int(tmp_off[-1])), dtype=torch.float64, device='cuda')
        map_off = np.concatenate([[0], np.cumsum([len(m) for m in maps])]).astype(np.int64)
        maps_dev = torch.from_numpy(np.concatenate(maps) if maps else np.zeros(1, dtype=np.int32)).cuda()
        real = []
        for d_ in descs:
            if isinstance(d_, tuple):
                csr, n_rows, L, R, slot, alpha = d_
                real.append(project_desc(csr, n_rows, L.ptr, L.ld, L.N, R.ptr, R.ld, R.N, tmp.data_ptr() + 8 * int(tmp_off[slot]),
                                         R.N, alpha))
            else:
                real.append(d_)
        descs[:] = real
        remap = (_lib.RemapDesc * max(1, len(todo)))()
        out_ptr, prev_ptr, tp, mp = self.out.data_ptr(), prev.out.data_ptr(), tmp.data_ptr(), maps_dev.data_ptr()
        for n, (token, ptoken, NL, NR, pNR, n_cn, n_rn, mr, mc, t1, t2) in enumerate(todo):
            r = remap[n]
            r.dst, r.NL, r.NR = out_ptr + 8 * int(self.offsets[token]), NL, NR
            r.prev, r.pNR = prev_ptr + 8 * int(prev.offsets[ptoken]), pNR
            r.n_cn, r.cols_new = n_cn, (tp + 8 * int(tmp_off[t1])) if n_cn else None
            r.n_rn, r.rows_new = n_rn, (tp + 8 * int(tmp_off[t2])) if n_rn else None
            r.row_map, r.col_map = mp + 4 * int(map_off[mr]), mp + 4 * int(map_off[mc])
        n_remap, h = len(todo), self.h

        def scatter():
            if n_remap:
                h.check(h.lib.lrbms_remap_blocks(h.h, n_remap, C.cast(remap, C.c_void_p), current_stream_ptr()))
        self.scatters.append(scatter)
        self.keep += [tmp, maps_dev, remap]

    def finalize(self):
        """Allocate the output buffer, resolve tokens to offsets, create the plans."""
        torch = _torch()
        self.offsets, starts = region_layout(self._pending, self.world)
        self.region_starts = starts
        self.out = torch.zeros(max(1, int(starts[-1])), dtype=torch.float64, device='cuda')
        base = self.out.data_ptr()
        descs = []
        if self.inc_jobs:
            self._plan_incremental(base, descs)
        for (token, csr, n_rows, L, R, ldo, alpha, sym) in self.jobs:
            descs.append(project_desc(csr, n_rows, L.ptr, L.ld, L.N, R.ptr, R.ld, R.N, base + 8 * int(self.offsets[token]),
                                      ldo, alpha, symmetric=sym))
        import time as _time
        _t = _time.perf_counter()
        self.spmm_plans = [make_spmm_plan(self.h, st, []) for st in self.spmm_stages if st]
        self.timings['spmm_plan_create_s'] = _time.perf_counter() - _t
        _t = _time.perf_counter()
        self.project_plan = make_project_plan(self.h, descs, [], scratch_owner=self.scratch_owner,
                                              unit_rows_hint=self.unit_rows) if descs else None
        self.timings['project_plan_create_s'] = _time.perf_counter() - _t
        self.n_project_descs = len(descs)
        self.n_spmm_descs = sum(len(st) for st in self.spmm_stages)
        self.n_incremental_jobs = len(self.inc_jobs)

    def run(self):
        for p in self.spmm_plans:
            p.run()
        for g in self.gathers:
            g()
        if self.project_plan is not None:
            self.project_plan.run()
        for sc in self.scatters:
            sc()

    def release_previous(self):
        """Drop the reference to the previous plan once this plan's results are complete (no chain of old plans)."""
        if self.inc_jobs:
            self.rerunnable = False          # the copies from the previous plan cannot be repeated
        self.prev = None
        self.gathers, self.scatters = [], []

    def exchange(self):
        """Multi-GPU: all-gather of the ranks' disjoint contiguous result regions -- over peer memory (NVLink stores or
        NVSwitch multicast, ``distributed.PeerStaging``) on an NCCL group, one NCCL all-gather otherwise."""
        if self.world > 1:
            exchange_regions(self.out, self.region_starts, handle=self.h)

    # -- accounting for bench / roofline
    def stats(self):
        s = dict(launches=0, bytes=0.0, bytes_survey=0.0, flops=0.0, ctas=0)
        for p in self.spmm_plans + ([self.project_plan] if self.project_plan is not None else []):
            s['launches'] += p.launches
            s['bytes'] += p.algorithmic_bytes
            s['bytes_survey'] += p.algorithmic_bytes_survey
            s['flops'] += p.flops
            s['ctas'] += int(p.info(1))
        return s


def _gather_columns(planner, arrays):
    """Concatenate dof-major arrays column-wise.  Zero-copy when they already are adjacent column slices of one
    slab (which is how ``LRBMSReductor`` lays out the OI / RT image bases); otherwise one device copy."""
    arrays = list(arrays)
    nonempty = [a for a in arrays if len(a) > 0]          # empty bases contribute no columns (and have no address)
    if not nonempty:
        return _ArrayRef.of(arrays[0])
    arrays = nonempty
    if len(arrays) == 1:
        return _ArrayRef.of(arrays[0])
    adjacent = all(a.ld == arrays[0].ld for a in arrays) and all(
        arrays[k + 1].device_ptr == arrays[k].device_ptr + 8 * len(arrays[k]) for k in range(len(arrays) - 1))
    total = sum(len(a) for a in arrays)
    refs = [_ArrayRef.of(a) for a in arrays]
    key = ('cat',) + tuple(r.key for r in refs)
    labels = np.concatenate([r.labels for r in refs], axis=0)
    if adjacent:
        return _ArrayRef(arrays[0].device_ptr, arrays[0].ld, total, arrays[0].dim, arrays, key=key, labels=labels)
    if any(getattr(a, '_is_view', False) for a in arrays):
        # slab views are filled by the plan's first SpMM stage, i.e. after planning: copying them now would copy zeros
        raise NotImplementedError('image bases of one neighbourhood must be adjacent column slices of one slab')
    cat = GpuVectorArray(arrays[0].space, None, total)
    pos = 0
    for a in arrays:
        cat._copy_cols_from(a, None, pos)
        pos += len(a)
    cat._plan_key, cat._plan_labels = key, labels
    return _ArrayRef.of(cat)


def _selection(op, bases):
    """Interpret a *selection* operator at either end of a ``Concatenation`` chain.

    Returns ``(subspace indices, arrays)``: which subspaces of the block source (range) take part and the basis
    array each contributes, or ``None`` if ``op`` is not a selection."""
    if isinstance(op, (BlockRowOperator, BlockColumnOperator)):
        blocks = op._blocks.ravel()
        spaces = op.source.subspaces if isinstance(op, BlockRowOperator) else op.range.subspaces
        idx, arrs = [], []
        for kk, b in enumerate(blocks):
            if b is None:
                continue
            if not isinstance(b, (BlockProjectionOperator, BlockEmbeddingOperator)):
                return None
            basis = bases[spaces[kk].id]
            assert isinstance(basis, BlockVectorArray), 'basis of block space {} must be a block array'.format(spaces[kk].id)
            idx.append(kk)
            arrs.append(basis._blocks[b.index])
        return idx, arrs
    if isinstance(op, (BlockProjectionOperator, BlockEmbeddingOperator)):
        space = op.source if isinstance(op, BlockProjectionOperator) else op.range
        return [op.index], [bases[space.subspaces[op.index].id]]
    return None


_DIMS_CACHE = {}
_SPACE_TOKENS = {}


def _dims(space, bases):
    """Basis sizes over the subspaces of ``space``.  Hundreds of operators carry their own (equal) block-space objects with
    one subspace per subdomain, so the sizes are cached per *subspace-id tuple* (interned once per space object) for the
    duration of one ``build_plan`` (cleared there) instead of being recomputed O(S) times per operator."""
    token = getattr(space, '_dims_token', None)
    if token is None:
        subs = space.subspaces if hasattr(space, 'subspaces') else [space]
        token = _SPACE_TOKENS.setdefault(tuple(s.id for s in subs), len(_SPACE_TOKENS))
        try:
            space._dims_token = token
        except AttributeError:
            pass
    hit = _DIMS_CACHE.get(token)
    if hit is None:
        subs = space.subspaces if hasattr(space, 'subspaces') else [space]
        hit = _DIMS_CACHE[token] = [1 if s.id == 'SCALARS' else len(bases[s.id]) for s in subs]
    return hit


def plan_projection(op, bases, planner, owner=None, name=None):
    """Emit the projection jobs of ``op`` (SURVEY.md Appendix A.3/A.4) and return its reduced counterpart."""
    if isinstance(op, LincombOperator):
        return LincombOperator([plan_projection(o, bases, planner, owner) for o in op.operators], op.coefficients,
                               name=op.name)
    if isinstance(op, VectorFunctional):
        # reduced right-hand side: f_red[j] = V_j^T f_j (reference discretize...:596-598; Appendix A.3 "RB=None")
        arr = op._array
        blocks = arr._blocks if isinstance(arr, BlockVectorArray) else [arr]
        subs = op.source.subspaces if isinstance(arr, BlockVectorArray) else [op.source]
        sblocks = []
        for j, (s, f) in enumerate(zip(subs, blocks)):
            V = bases[s.id]
            token = planner.project(j if owner is None else owner, None, _ArrayRef.of(f), _ArrayRef.of(V))
            sblocks.append(SuperBlock([0], [j], token, 1, len(V)))
        return ReducedBlockOperator(planner, sblocks, [1], _dims(op.source, bases), name=op.name or name, functional=True)
    if isinstance(op, CsrOperator):
        L, R = bases[op.range.id], bases[op.source.id]
        token = planner.project(owner if owner is not None else 0, op.csr, _ArrayRef.of(L), _ArrayRef.of(R))
        return ReducedBlockOperator(planner, [SuperBlock([0], [0], token, len(L), len(R))], [len(L)], [len(R)],
                                    name=op.name or name)
    if isinstance(op, BlockOperator) and op._block_range and op._block_source:
        sblocks = []
        for i, j, b in op.nonzero_blocks():
            if not isinstance(b, CsrOperator):
                raise NotImplementedError('block ({}, {}) of {} is a {}; only sparse-matrix blocks are projected'
                                          .format(i, j, op.name, type(b).__name__))
            L, R = bases[op.range.subspaces[i].id], bases[op.source.subspaces[j].id]
            token = planner.project(i if owner is None else owner, b.csr, _ArrayRef.of(L), _ArrayRef.of(R))
            sblocks.append(SuperBlock([i], [j], token, len(L), len(R)))
        return ReducedBlockOperator(planner, sblocks, _dims(op.range, bases), _dims(op.source, bases), name=op.name or name)
    if isinstance(op, Concatenation):
        return _plan_chain(op, bases, planner, owner if owner is not None else 0, name)
    raise NotImplementedError('no projection rule for {} ({})'.format(type(op).__name__, getattr(op, 'name', None)))


def _plan_chain(op, bases, planner, owner, name):
    """``Concatenation([left, M_1 .. M_k, right])`` with selections (or a functional) at the ends and sparse matrices
    in the middle -- the shape of every estimator operator (reference ``discretize...:733-770``)."""
    chain = op.flat()
    # ---- right end
    sel = _selection(chain[-1], bases)
    if sel is None:
        raise NotImplementedError('{}: the right end of the chain must be a block selection'.format(op.name))
    col_idx, col_arrays = sel
    R = _gather_columns(planner, col_arrays)
    col_sizes = [len(a) for a in col_arrays]
    chain = chain[:-1]
    # ---- left end
    functional = False
    if isinstance(chain[0], VectorFunctional):
        L = _ArrayRef.of(chain[0]._array)
        row_idx, row_sizes, functional = [0], [1], True
        chain = chain[1:]
    else:
        sel = _selection(chain[0], bases)
        if sel is None:
            raise NotImplementedError('{}: the left end of the chain must be a block selection or a functional'.format(op.name))
        row_idx, row_arrays = sel
        L = _gather_columns(planner, row_arrays)
        row_sizes = [len(a) for a in row_arrays]
        chain = chain[1:]
    if not all(isinstance(m, CsrOperator) for m in chain):
        raise NotImplementedError('{}: only sparse matrices may sit between the selections'.format(op.name))
    # ---- several sparse matrices in a row (r_dd: D^T M D): their product is formed once on the host and cached for the
    #      life of the reductor -- the operators are static -- so the chain costs one SpMM and, for r_dd, a Gram over the
    #      m_i flux dofs instead of the n_i DG dofs.  Same result up to the order of summation.
    if len(chain) >= 2 and planner.fuse_cache is not None:
        chain = [fuse_chain(chain, planner.fuse_cache)]
    # ---- (A^T ...)-prefix: L^T A^T = (A L)^T, one SpMM on the left array (shared with the right side through the cache)
    while len(chain) > 1 and chain[0].transposed_of is not None:
        L = planner.spmm(owner, chain[0].transposed_of.csr, L)
        chain = chain[1:]
    # ---- all but one remaining matrix are applied to the right array
    while len(chain) > 1:
        R = planner.spmm(owner, chain[-1].csr, R)
        chain = chain[:-1]
    csr = chain[0].csr if chain else None
    if csr is not None and planner.narrow_left and (L.N > 40 or R.N > 40) and 2 * L.N <= R.N:
        # too wide for the fused kernel, and the left side is the narrow one: L^T A R = (A^T L)^T R.  One narrow SpMM on
        # the left array instead of a scratch SpMM over all columns of R (df_ab: 20 instead of 200 columns, r_fd: 1)
        L = planner.spmm(owner, csr.T, L)
        csr = None
    token = planner.project(owner, csr, L, R)
    rdims = [1] if functional else _dims(op.range, bases)
    return ReducedBlockOperator(planner, [SuperBlock(row_idx, col_idx, token, sum(row_sizes), sum(col_sizes),
                                                     row_sizes, col_sizes)],
                                rdims, _dims(op.source, bases), name=op.name or name, functional=functional)


def _walk_csr(op, out):
    """All CsrOperators reachable from ``op`` (Lincomb / Block / Concatenation containers)."""
    if isinstance(op, CsrOperator):
        out.append(op)
    elif isinstance(op, (LincombOperator, Concatenation)):
        for o in op.operators:
            _walk_csr(o, out)
    elif isinstance(op, BlockOperator):
        for b in op._blocks.ravel():
            if b is not None:
                _walk_csr(b, out)
    return out


def fuse_chain(chain, cache):
    """The product of consecutive sparse matrices of an operator chain, formed once and cached (key: the matrices)."""
    key = tuple(id(m.csr) for m in chain)
    if key not in cache:
        from .kernels import DeviceCsr
        P = chain[0].csr.host
        for m in chain[1:]:
            P = P @ m.csr.host
        P = P.tocsr()
        P.sort_indices()
        cache[key] = (CsrOperator(DeviceCsr(P), source_id=chain[-1].source.id, range_id=chain[0].range.id, name='fused_chain'),
                      [m.csr for m in chain])
    return cache[key][0]


def prepare_operators(d):
    """One-off preparation that depends on the operators only -- done when the discretization is built, not in the first
    ``reduce()``: symmetry flags of the square matrices (a symmetric Gram is computed on its lower output chunks only), the
    products of chained sparse matrices (``r_dd``: ``D^T M D``) and the transposes that chains with a narrow left side apply
    to that side (``df_ab``, ``r_fd``).  All three are cached on the matrices / on ``d`` and shared by every reductor of ``d``."""
    cache = d.__dict__.setdefault('_fused_chains', {})
    ops = list(d.operators.values()) + list(d.products.values())
    for op in ops:
        for c in _walk_csr(op, []):
            if c.csr.shape[0] == c.csr.shape[1]:
                c.csr.symmetric
        for cc in ([op] if isinstance(op, Concatenation) else
                   [o for o in getattr(op, 'operators', []) if isinstance(o, Concatenation)]):
            chain = [m for m in cc.flat() if isinstance(m, CsrOperator)]
            flat = cc.flat()
            if len(chain) >= 2 and all(isinstance(m, CsrOperator) for m in flat[1:-1]) and len(chain) == len(flat) - 2:
                fused = fuse_chain(chain, cache)
                if fused.csr.shape[0] == fused.csr.shape[1]:
                    fused.csr.symmetric
                chain = [fused]
            # narrow left end (a functional or a single subspace) against a neighbourhood on the right: (A^T L)^T R
            left = flat[0]
            narrow = isinstance(left, (VectorFunctional, BlockProjectionOperator, BlockEmbeddingOperator))
            if narrow and len(chain) == 1:
                chain[0].csr.T


# ----------------------------------------------------------------------------------------------------------
#  LRBMS reductor
# ----------------------------------------------------------------------------------------------------------

class LRBMSReductor(GenericRBSystemReductor):
    """reference ``reductor.py:17-78``."""

    def __init__(self, d, bases=None, products=None, order=None, num_cpus=1, solver_options=None, shard=False):
        assert order is None or 0 <= order <= 1
        self.solver_options = solver_options
        self.num_cpus = num_cpus            # accepted and ignored, like the reference (reductor.py:19,84)
        self.shard = bool(shard)
        self.reuse_plan = False
        self.fuse_chains = True             # products of consecutive sparse matrices in an operator chain are formed once (host)
        self.narrow_left = True             # chains with a narrow left and a wide right side apply the matrix to the left side
        self.incremental = False            # reduce() after an enrichment projects only the new rows / columns (8f rank 2)
        super().__init__(d, bases=bases, products=products)
        if order is None and bases is None:
            order = 0
        if order is not None:
            for ii in range(len(d.solution_space.subspaces)):
                self.extend_basis_local(d.shape_functions(ii, order))
        self.last_plan = None

    # -- sharding of subdomains over ranks: contiguous strips (SURVEY.md section 8e)
    def _shard_info(self):
        return rank_and_world() if self.shard else (0, 1)

    def build_plan(self, incremental=False):
        """Plan the whole offline projection for the current bases (no kernel runs yet).

        ``incremental=True`` (SURVEY.md section 8f rank 2): the previous plan of this reductor is taken as the source of
        every reduced entry whose row *and* column belong to basis vectors that already existed; only the rows / columns
        of vectors appended since (``extend_basis_local``) are projected, and only their Oswald / flux-reconstruction
        images are computed.  The reference re-projects everything after each enrichment (``online_enrichment.py:49-51``)."""
        torch = _torch()
        d = self.d
        subs = d.solution_space.subspaces
        S = len(subs)
        rank, world = self._shard_info()
        owner_rank_of = (lambda owner: owner_rank(owner, S, world)) if world > 1 else None
        old = self.last_plan
        prev = None
        if incremental and world == 1 and old is not None and getattr(old, 'reusable', False) and \
                all(len(self.bases[s.id]) >= n for s, n in zip(subs, old.block_dims)):
            prev = old
        planner = _Planner(Handle.get(), owner_rank_of, rank, world, prev=prev)
        planner.scratch_owner = self
        _DIMS_CACHE.clear()
        _ArrayRef._of_cache.clear()
        if self.fuse_chains:
            planner.fuse_cache = d.__dict__.setdefault('_fused_chains', {})      # shared with prepare_operators(d)
        planner.narrow_left = self.narrow_left
        if old is not None and getattr(old, 'reusable', False):
            # the reduced model of the previous plan is no longer referenced: recycle its scratch arrays
            pool = {}
            for key, t in old.scratch_used:
                pool.setdefault(key, []).append(t)
            planner.scratch_pool = pool
        N = [len(self.bases[s.id]) for s in subs]
        for k, sp_ in enumerate(subs):                          # what the columns of every basis are (see _ArrayRef)
            self.bases[sp_.id]._plan_key = ('V', k)
            self.bases[sp_.id]._plan_labels = _labels(k, [0], N[k])
        V = [_ArrayRef.of(self.bases[s.id]) for s in subs]
        N_old = prev.block_dims if prev is not None else [0] * S

        # ---- Oswald-interpolation and flux-reconstruction images of the bases (reference reductor.py:36-60), written
        #      into per-target-subdomain slabs: slab_i = [component i of bases['OI_k']]_{k in N(i)}
        oi = d.estimator.oswald_interpolation_error
        fr = d.estimator.flux_reconstruction
        Q = len(fr.operators)
        nbh = [oi._blocks[k, k].neighborhood for k in range(S)]
        targets = [[] for _ in range(S)]                       # targets[i] = sorted k with i in N(k)
        for k in range(S):
            for i in nbh[k]:
                targets[i].append(k)
        oi_slab, rt_slab, oi_col, rt_col = [], [], [], []
        shapes, total = [], 0
        for i in range(S):
            cols = np.concatenate([[0], np.cumsum([N[k] for k in targets[i]])]).astype(int)
            oi_col.append(dict(zip(targets[i], cols[:-1])))
            rt_col.append(dict(zip(targets[i], Q * cols[:-1])))
            ld_o = max(4, (cols[-1] + 3) // 4 * 4)
            ld_r = max(4, (Q * cols[-1] + 3) // 4 * 4)
            m_i = fr.operators[0]._blocks[i, i].range.subspaces[nbh[i].index(i)].dim
            shapes.append((subs[i].dim, ld_o, m_i, ld_r, total))
            total += (subs[i].dim * ld_o + 31) // 32 * 32 + (m_i * ld_r + 31) // 32 * 32
        slab_buf = torch.zeros(max(1, total), dtype=torch.float64, device='cuda')      # one allocation, one memset
        for (n_i, ld_o, m_i, ld_r, pos) in shapes:
            oi_slab.append(slab_buf[pos:pos + n_i * ld_o].view(n_i, ld_o))
            pos += (n_i * ld_o + 31) // 32 * 32
            rt_slab.append(slab_buf[pos:pos + m_i * ld_r].view(m_i, ld_r))
        for k in range(S):
            oi_k = oi._blocks[k, k]
            comps_o, comps_r = [], []
            n0, n1 = N_old[k], N[k]                               # columns [0, n0) exist in the previous plan's slabs
            lab_o, lab_r = _labels(k, [0], N[k]), _labels(k, range(Q), N[k])
            for c, i in enumerate(nbh[k]):
                view_o = oi_slab[i][:, oi_col[i][k]:oi_col[i][k] + N[k]]
                arr_o = oi_k.range.subspaces[c].from_dofmajor(view_o, N[k])
                arr_o._plan_key, arr_o._plan_labels = ('oi', i, k), lab_o
                comps_o.append(arr_o)
                if prev is not None and n0:
                    pc = prev.oi_col[i][k]
                    view_o[:, :n0] = prev.oi_slab[i][:, pc:pc + n0]
                if n1 > n0 and planner.mine(i):
                    planner.spmm_stages[0].append(spmm_desc(oi_k.components[c], V[k].ptr + 8 * n0, V[k].ld, n1 - n0,
                                                            view_o.data_ptr() + 8 * n0, oi_slab[i].stride(0)))
                view_r = rt_slab[i][:, rt_col[i][k]:rt_col[i][k] + Q * N[k]]
                rt_space = fr.operators[0]._blocks[k, k].range.subspaces[c]
                arr_r = rt_space.from_dofmajor(view_r, Q * N[k])
                arr_r._plan_key, arr_r._plan_labels = ('rt', i, k), lab_r
                comps_r.append(arr_r)
                for q in range(Q):                               # q-major ordering of the RT basis (reductor.py:55-60)
                    fr_kq = fr.operators[q]._blocks[k, k]
                    if prev is not None and n0:
                        pc = prev.rt_col[i][k] + q * n0
                        view_r[:, q * n1:q * n1 + n0] = prev.rt_slab[i][:, pc:pc + n0]
                    if n1 > n0 and planner.mine(i):
                        planner.spmm_stages[0].append(spmm_desc(fr_kq.components[c], V[k].ptr + 8 * n0, V[k].ld, n1 - n0,
                                                                view_r.data_ptr() + 8 * (q * n1 + n0), rt_slab[i].stride(0)))
            self.bases[oi.range.subspaces[k].id] = BlockVectorArray(comps_o, oi.range.subspaces[k])
            self.bases[fr.range.subspaces[k].id] = BlockVectorArray(comps_r, fr.range.subspaces[k])
        planner.oi_slab, planner.rt_slab, planner.oi_col, planner.rt_col = oi_slab, rt_slab, oi_col, rt_col
        planner.keep += [oi_slab, rt_slab, slab_buf]

        # ---- every operator and product of the discretization (reference reductor.py:70 -> GenericRBSystemReductor._reduce)
        red_ops, red_products = {}, {}
        for name, op in d.operators.items():
            owner = None
            tail = name.rsplit('_', 1)[-1]
            if tail.isdigit() and name not in ('operator', 'rhs'):
                owner = int(tail)                                # nc_i, r_fd_i, ..., local_energy_dg_product_i
            red_ops[name] = plan_projection(op, self.bases, planner, owner, name)
        for name, op in d.products.items():
            red_products[name] = plan_projection(op, self.bases, planner, None, name)
        import time as _time
        _t = _time.perf_counter()
        planner.finalize()
        planner.timings['finalize_s'] = _time.perf_counter() - _t
        planner.block_dims = N
        planner.red_ops, planner.red_products = red_ops, red_products
        self.last_plan = planner
        return planner

    def _plan_key(self):
        subs = self.d.solution_space.subspaces
        return tuple((self.bases[s.id].device_ptr, self.bases[s.id].ld, len(self.bases[s.id])) for s in subs) + self._shard_info()

    def _reduce(self):
        d = self.d
        key = self._plan_key()
        if self.reuse_plan and self.last_plan is not None and getattr(self, '_last_key', None) == key and \
                getattr(self.last_plan, 'rerunnable', True):
            # same basis buffers and sizes as last time: the plan is still valid.  Opt-in, because the reduced model
            # returned earlier shares the plan's output buffer and is overwritten by this run.
            planner = self.last_plan
        else:
            import time as _time
            _t = _time.perf_counter()
            planner = self.build_plan(incremental=self.incremental)
            planner.timings['build_plan_s'] = _time.perf_counter() - _t
            self._last_key = key
        planner.run()
        planner.exchange()
        planner.release_previous()
        planner.reusable = True       # its SpMM scratch may be recycled by the next plan of this reductor (same stream)
        N = planner.block_dims
        fr = d.estimator.flux_reconstruction
        red_estimator = d.estimator.with_(
            flux_reconstruction=ReducedFluxReconstruction(fr.coefficients, N),
            oswald_interpolation_error=ReducedOswaldInterpolation(N))
        rd = ReducedModel(planner.red_ops['operator'], planner.red_ops['rhs'], products=planner.red_products,
                          operators=planner.red_ops, estimator=red_estimator, parameter_type=d.parameter_type,
                          block_dims=N, neighborhoods=d.neighborhoods, parameter_range=getattr(d, 'parameter_range', None),
                          keepalive=planner)
        return rd

    def enrich_local(self, subdomain, U, mu=None):
        """reference ``reductor.py:75-78``: needs the fine-scale local corrector solve
        (``discretize...:227-316``), which is outside the hot path (SURVEY.md section 8f rank 4)."""
        if not hasattr(self.d, 'solve_for_local_correction'):
            raise NotImplementedError('enrich_local needs d.solve_for_local_correction (fine-scale neighbourhood solve)')
        Us = [self.reconstruct_local(U, 'domain_{}'.format(sdi)) for sdi in self.d.neighborhoods[subdomain]]
        local_correction = self.d.solve_for_local_correction(subdomain, Us, mu, inverse_options=self.solver_options)
        self.extend_basis_local(local_correction)
