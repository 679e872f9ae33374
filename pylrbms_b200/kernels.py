"""Thin host helpers over the C ABI: device CSR storage, descriptor builders, one-shot SpMM / projection calls.

Everything numerical happens inside ``liblrbms_sm100`` (``include/lrbms_sm100.h``); this module only packs
pointers.  One-shot helpers create a plan, run it and drop it -- the reductor batches all of its blocks into a
single plan instead (:mod:`pylrbms_b200.reductor`).
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

from ._lib import Handle, ProjectDesc, SpmmDesc, make_project_plan, make_spmm_plan


def _torch():
    import torch
    return torch


class DeviceCsr:
    """CSR matrix resident in HBM: ``rowptr`` / ``colind`` int32, ``values`` float64.

    Replaces ``IstlRowMajorSparseMatrixDouble`` (reference ``discretize_elliptic_block_swipdg.py:10-14``)."""

    def __init__(self, matrix):
        torch = _torch()
        M = sp.csr_matrix(matrix)
        if not M.has_sorted_indices:
            M = M.copy()
            M.sort_indices()
        self.shape = tuple(int(s) for s in M.shape)
        self.nnz = int(M.nnz)
        self.rowptr = torch.from_numpy(np.ascontiguousarray(M.indptr, dtype=np.int32)).cuda()
        self.colind = torch.from_numpy(np.ascontiguousarray(M.indices if M.nnz else np.zeros(1), dtype=np.int32)).cuda()
        self.values = torch.from_numpy(np.ascontiguousarray(M.data if M.nnz else np.zeros(1), dtype=np.float64)).cuda()
        self._host = M
        self._T = None
        self._symmetric = None

    @classmethod
    def from_device(cls, rowptr, colind, values, shape):
        """Wrap CSR arrays that already live in HBM (int32 ``rowptr`` / ``colind`` with sorted column indices, float64
        ``values``); the host copy is made only if somebody asks for it."""
        self = cls.__new__(cls)
        self.shape = tuple(int(s) for s in shape)
        self.nnz = int(values.numel())
        self.rowptr, self.colind, self.values = rowptr, colind, values
        self._host = None
        self._T = None
        self._symmetric = None
        return self

    @property
    def host(self):
        """The host CSR this was uploaded from (kept for the transposed upload and for inspection)."""
        if self._host is None:
            self._host = sp.csr_matrix((self.values.cpu().numpy(), self.colind.cpu().numpy(), self.rowptr.cpu().numpy()),
                                       shape=self.shape)
        return self._host

    @property
    def T(self):
        if self._T is None:
            self._T = DeviceCsr(self._host.T.tocsr())
            self._T._T = self
        return self._T

    @property
    def symmetric(self):
        """True if the matrix equals its transpose up to rounding of the assembly (checked once, on the host copy)."""
        if self._symmetric is None:
            M = self._host
            if M.shape[0] != M.shape[1]:
                self._symmetric = False
            elif M.nnz == 0:
                self._symmetric = True
            else:
                D = abs(M - M.T)
                self._symmetric = bool(D.max() <= 1e-13 * abs(M).max())
        return self._symmetric

    @property
    def device_bytes(self):
        return 4 * (self.shape[0] + 1) + 12 * self.nnz


def spmm_desc(csr, V_ptr, ldv, N, W_ptr, ldw):
    return SpmmDesc(csr.rowptr.data_ptr(), csr.colind.data_ptr(), csr.values.data_ptr(), csr.shape[0], csr.shape[1],
                    V_ptr, ldv, N, W_ptr, ldw)


def project_desc(csr, n_rows, VL_ptr, ldl, NL, VR_ptr, ldr, NR, out_ptr, ldo, alpha=1.0, symmetric=False):
    """``csr=None`` selects the identity operator (Gram matrix ``VL^T VR``).  ``symmetric=True`` asserts that the
    operator is symmetric and ``VL`` / ``VR`` are the same array (only the lower output chunks are computed)."""
    sym = 1 if (symmetric and VL_ptr == VR_ptr and ldl == ldr and NL == NR) else 0
    if csr is None:
        return ProjectDesc(None, None, None, n_rows, n_rows, VL_ptr, ldl, NL, VR_ptr, ldr, NR, out_ptr, ldo, float(alpha), sym, 0)
    assert csr.shape[0] == n_rows
    return ProjectDesc(csr.rowptr.data_ptr(), csr.colind.data_ptr(), csr.values.data_ptr(), csr.shape[0], csr.shape[1],
                       VL_ptr, ldl, NL, VR_ptr, ldr, NR, out_ptr, ldo, float(alpha), sym, 0)


def spmm_once(csr, V, range_space):
    """``W = A V`` for a :class:`GpuVectorArray` ``V``; returns a new array in ``range_space``."""
    from .vectorarray import GpuVectorArray
    W = GpuVectorArray(range_space, None, len(V))
    if len(V) == 0 or csr.shape[0] == 0:
        return W
    h = Handle.get()
    plan = make_spmm_plan(h, [spmm_desc(csr, V.device_ptr, V.ld, len(V), W.device_ptr, W.ld)], [csr, V, W])
    plan.run()
    plan.destroy()
    return W


def project_once(csr, VL, VR, alpha=1.0):
    """``alpha * VL^T (A VR)`` as a host ``(len(VL), len(VR))`` array (``csr=None``: ``VL^T VR``)."""
    torch = _torch()
    NL, NR = len(VL), len(VR)
    if NL == 0 or NR == 0:
        return np.zeros((NL, NR))
    out = torch.zeros((NL, NR), dtype=torch.float64, device='cuda')
    if VL.dim == 0:
        return out.cpu().numpy()
    h = Handle.get()
    d = project_desc(csr, VL.dim, VL.device_ptr, VL.ld, NL, VR.device_ptr, VR.ld, NR, out.data_ptr(), NR, alpha)
    plan = make_project_plan(h, [d], [csr, VL, VR, out])
    plan.run()
    plan.destroy()
    return out.cpu().numpy()


def pcg_solve(csr, b, x0=None, rtol=1e-12, max_iter=None):
    """Solve ``A x = b`` for a symmetric positive definite :class:`DeviceCsr` ``A`` with the Jacobi-preconditioned CG of
    ``lrbms_pcg_solve``.  ``b`` / ``x0``: 1-D float64 CUDA tensors.  Returns ``(x, iterations, relative residual)``."""
    import ctypes as C
    torch = _torch()
    n = csr.shape[0]
    assert csr.shape[0] == csr.shape[1] == b.numel()
    h = Handle.get()
    x = torch.zeros(n, dtype=torch.float64, device='cuda') if x0 is None else x0.clone().contiguous()
    nbytes = C.c_size_t()
    h.check(h.lib.lrbms_pcg_workspace_bytes(h.h, n, C.byref(nbytes)))
    ws = torch.empty(max(1, nbytes.value // 8), dtype=torch.float64, device='cuda')
    iters, relres = C.c_int32(), C.c_double()
    from ._lib import current_stream_ptr
    h.check(h.lib.lrbms_pcg_solve(h.h, n, csr.rowptr.data_ptr(), csr.colind.data_ptr(), csr.values.data_ptr(),
                                  b.contiguous().data_ptr(), x.data_ptr(), float(rtol),
                                  int(max_iter if max_iter is not None else max(100, 10 * n)), C.byref(iters), C.byref(relres),
                                  ws.data_ptr(), nbytes.value, current_stream_ptr()))
    return x, iters.value, relres.value


def affine_pcg_workspace_bytes(n, n_mu):
    """Device workspace ``lrbms_affine_pcg_solve`` needs for ``n_mu`` parameters of an ``n``-dof system."""
    import ctypes as C
    h = Handle.get()
    nbytes = C.c_size_t()
    h.check(h.lib.lrbms_affine_pcg_workspace_bytes(h.h, int(n), int(n_mu), C.byref(nbytes)))
    return nbytes.value


def affine_pcg_solve(pattern, values, rhs, theta, x, rtol, max_iter, max_restarts):
    """Solve ``(sum_q theta[k, q] A_q) x_k = sum_f theta[k, Q + f] rhs_f`` for every row ``k`` of ``theta`` with
    ``lrbms_affine_pcg_solve``.  ``pattern``: :class:`DeviceCsr` whose ``rowptr`` / ``colind`` every component shares;
    ``values``: ``(Q, nnz)`` and ``rhs``: ``(Qf, n)`` float64 CUDA tensors; ``theta``: ``(n_mu, Q + Qf)`` CUDA tensor;
    ``x``: dof-major ``(n, >= n_mu)`` CUDA view (row stride ``ld``), initial guess in, solution out.
    Returns ``(x, iterations, true relative residual, status)``, the last three host arrays of length ``n_mu``."""
    import ctypes as C
    from ._lib import current_stream_ptr, ptr
    torch = _torch()
    n, n_mu = pattern.shape[0], theta.shape[0]
    Q, Qf = values.shape[0], rhs.shape[0]
    assert values.is_contiguous() and rhs.is_contiguous() and theta.is_contiguous() and theta.shape[1] == Q + Qf
    assert x.shape[0] == n and x.shape[1] >= n_mu and x.stride(1) == 1
    h = Handle.get()
    nbytes = affine_pcg_workspace_bytes(n, n_mu)
    ws = torch.empty(max(1, nbytes // 8), dtype=torch.float64, device='cuda')
    iters = np.zeros(n_mu, dtype=np.int32)
    relres = np.zeros(n_mu, dtype=np.float64)
    status = np.zeros(n_mu, dtype=np.int32)
    h.check(h.lib.lrbms_affine_pcg_solve(h.h, n, Q, ptr(pattern.rowptr), ptr(pattern.colind), ptr(values), Qf, ptr(rhs),
                                         n_mu, ptr(theta), ptr(x), x.stride(0), float(rtol), int(max_iter),
                                         int(max_restarts), ptr(iters), ptr(relres), ptr(status), ptr(ws), nbytes,
                                         current_stream_ptr()))
    return x, iters, relres, status


def recon_error(bases, block_dims, u_h, u_N, e):
    """``e = u_h - R u_N`` for all subdomains in one launch (``lrbms_recon_error``).  ``bases``: the local bases (one
    :class:`GpuVectorArray` per subdomain, in row order); ``block_dims``: the coefficients per subdomain in ``u_N`` (the first
    ``block_dims[i]`` vectors of basis ``i`` are used); ``u_h`` / ``e``: dof-major ``(n, >= n_mu)`` CUDA views; ``u_N``:
    ``(n_mu, n_red)`` CUDA tensor with unit column stride.  Returns ``e``."""
    import ctypes as C
    from ._lib import ReconBlock, current_stream_ptr, ptr
    torch = _torch()
    n_mu, n_red = u_N.shape
    assert len(bases) == len(block_dims) and u_N.stride(1) == 1 and u_h.stride(1) == 1 and e.stride(1) == 1
    assert u_h.shape[0] == e.shape[0] and u_h.shape[1] >= n_mu and e.shape[1] >= n_mu
    blocks = (ReconBlock * max(1, len(bases)))()
    row, red = 0, 0
    for i, (V, N) in enumerate(zip(bases, block_dims)):
        blocks[i] = ReconBlock(V.device_ptr, V.ld, len(V), int(N), red, row, V.dim, 0)
        row, red = row + V.dim, red + int(N)
    assert row == u_h.shape[0], 'the bases do not cover the rows of u_h'
    h = Handle.get()
    nbytes = C.c_size_t()
    h.check(h.lib.lrbms_recon_error_workspace_bytes(h.h, len(bases), C.cast(blocks, C.c_void_p), n_mu, n_red, C.byref(nbytes)))
    ws = torch.empty(max(1, nbytes.value // 8 + 1), dtype=torch.float64, device='cuda')
    h.check(h.lib.lrbms_recon_error(h.h, len(bases), C.cast(blocks, C.c_void_p), n_mu, ptr(u_h), u_h.stride(0), ptr(u_N),
                                    n_red, max(n_red, u_N.stride(0)), ptr(e), e.stride(0), ptr(ws),
                                    ws.numel() * 8, current_stream_ptr()))
    return e


def segmented_form(pattern, values, seg_ptr, x, n_mu, theta=None, out=None):
    """``out[s, m] = sum over the rows of segment s of x[r, m] (sum_q theta[m, q] A_q x[:, m])[r]``
    (``lrbms_segmented_form``).  ``pattern``: :class:`DeviceCsr` whose ``rowptr`` / ``colind`` the components share;
    ``values``: ``(Q, nnz)`` CUDA tensor; ``seg_ptr``: host row offsets of the segments; ``x``: dof-major ``(n, >= n_mu)``
    CUDA view; ``theta``: ``(n_mu, >= Q)`` CUDA tensor with unit column stride, or None for theta = 1 (Q = 1).
    Returns ``out``, an ``(n_seg, n_mu)`` CUDA tensor."""
    import ctypes as C
    from ._lib import current_stream_ptr, host_i32, ptr
    torch = _torch()
    seg = host_i32(seg_ptr)
    n_seg = seg.size - 1
    Q, nnz = values.shape
    assert values.is_contiguous() and x.stride(1) == 1 and x.shape[0] == pattern.shape[0]
    if theta is not None:
        assert theta.shape[0] >= n_mu and theta.stride(1) == 1
    if out is None:
        out = torch.empty((n_seg, max(1, n_mu)), dtype=torch.float64, device='cuda')[:, :n_mu]
    h = Handle.get()
    nbytes = C.c_size_t()
    h.check(h.lib.lrbms_segmented_form_workspace_bytes(h.h, n_seg, ptr(seg), C.byref(nbytes)))
    ws = torch.empty(max(1, nbytes.value // 8 + 1), dtype=torch.float64, device='cuda')
    h.check(h.lib.lrbms_segmented_form(h.h, pattern.shape[0], Q, ptr(pattern.rowptr), ptr(pattern.colind), ptr(values), nnz,
                                       n_seg, ptr(seg), int(n_mu), ptr(theta),
                                       theta.stride(0) if theta is not None else 0, ptr(x), x.stride(0), ptr(out),
                                       out.stride(0), ptr(ws), ws.numel() * 8, current_stream_ptr()))
    return out
