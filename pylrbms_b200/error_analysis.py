"""Reduction error of a parameter batch on the device: true errors, local errors and effectivities.

``reduction_error_analysis`` is the counterpart of pyMOR's ``reduction_error_analysis`` for the LRBMS reductor, and of the
reference driver's "max discretization error" loop (``scripts/online_adaptive_lrbms.py:49-53,141-143``: reduce, solve
reduced, ``reductor.reconstruct``, difference to ``d.solve(mu)``, norm -- one parameter and one subdomain at a time).  Here a
whole batch goes through three kernels of ``csrc/error_norms.cu``:

* ``lrbms_recon_error``: ``e = u_h - R u_N`` for every subdomain in one launch, into one reused scratch buffer (``u_h`` is
  left intact: the caller gets it back);
* ``lrbms_segmented_form`` with the block-diagonal local energy products: the squared local errors
  ``e_i^T (local_energy_dg_product_i) e_i`` (their sum is the energy norm ``tools/fom_timing.py`` uses), and the same of
  ``u_h`` for the relative errors;
* ``lrbms_segmented_form`` with the affine operator: ``|||e|||_mu^2 = e^T A(mu) e`` over the whole domain only (row partials
  of a coupled operator are not norms).

Every parameter's numbers are bit-identical whatever batch, position or chunk it is analysed in.
"""
from __future__ import annotations

import numpy as np


class ReductionErrorAnalysis:
    """Result of :func:`reduction_error_analysis`; host NumPy arrays, ``(n_mu,)`` or ``(S, n_mu)``:

    ``errors`` (energy norm of ``u_h - R u_N``), ``operator_errors`` (``|||u_h - R u_N|||_mu``), ``local_errors``,
    ``relative_errors`` (``errors`` over the energy norm of ``u_h``), ``eta``, ``indicators``, ``effectivities``
    (``eta / errors``), ``local_effectivities`` (``indicators / local_errors``); ``max_error`` and its index ``argmax``,
    ``min_effectivity``, ``max_effectivity``; ``fom_info``, the ``last_solve_info`` of the fine-scale solve (None when the
    caller passed ``U_h``).  A zero error gives an effectivity of ``inf``."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def __repr__(self):
        return ('ReductionErrorAnalysis(n_mu={}, max_error={:.3e} at #{}, effectivity {:.3g} .. {:.3g})'
                .format(len(self.errors), self.max_error, self.argmax, self.min_effectivity, self.max_effectivity))


def _check_arguments(d, reductor, rd, mus, U_h):
    """Shapes and sizes only (no device work): returns ``(S, n_mu)``."""
    subs = d.solution_space.subspaces
    S = len(subs)
    if reductor.d is not d:
        raise ValueError('the reductor was built for another discretization')
    dims = [int(n) for n in rd.block_dims]
    if len(dims) != S:
        raise ValueError('the reduced model has {} subdomain blocks, the discretization {} subdomains'.format(len(dims), S))
    for i, s in enumerate(subs):
        if dims[i] > len(reductor.bases[s.id]):
            raise ValueError('subdomain {}: the reduced model uses {} basis vectors, the reductor has {}'.format(
                i, dims[i], len(reductor.bases[s.id])))
    n_mu = len(mus)
    if n_mu == 0:
        raise ValueError('need at least one parameter')
    if U_h is not None:
        if len(U_h) != n_mu:
            raise ValueError('U_h holds {} solutions for {} parameters'.format(len(U_h), n_mu))
        if len(U_h._blocks) != S or any(b.dim != s.dim for b, s in zip(U_h._blocks, subs)):
            raise ValueError('U_h is not an array of the solution space of d')
    return S, n_mu


def _dofmajor(U_h, n, n_mu):
    """``(n, >= n_mu)`` dof-major view of the fine solutions: the buffer ``d.solve_batch`` returned its blocks from, or a
    gathered copy when the blocks are not consecutive rows of one buffer."""
    import torch
    from .vectorarray import GpuVectorArray, _round_cap
    blocks = U_h._blocks
    b0 = blocks[0]._buf
    ld, row, base = b0.stride(0), 0, b0.data_ptr()
    consecutive = True
    for b in blocks:
        t = b._buf
        consecutive = consecutive and t.stride(0) == ld and t.stride(1) == 1 and t.data_ptr() == base + 8 * ld * row and \
            t.untyped_storage().data_ptr() == b0.untyped_storage().data_ptr()
        row += b.dim
    if consecutive and ld >= n_mu:
        return b0.as_strided((n, n_mu), (ld, 1))
    buf = torch.empty((n, _round_cap(n_mu)), dtype=torch.float64, device='cuda')
    row = 0
    for b in blocks:
        GpuVectorArray(b.space, buf[row:row + b.dim], 0)._copy_cols_from(b, None, 0)
        row += b.dim
    return buf


def _sum_subdomains(a):
    """``a[0] + a[1] + ... + a[S-1]`` per column, in that order.  (``a.sum(axis=0)`` is not a fixed order: for a single
    column NumPy sums the contiguous data pairwise with interleaved accumulators, for several columns row by row, so the
    bits of a parameter would depend on the batch size.)"""
    acc = a[0].copy()
    for row in a[1:]:
        acc += row
    return acc


def _energy_system(d):
    """The block-diagonal sum of the ``local_energy_dg_product_i`` as one device CSR (``(pattern, values (1, nnz))``) and
    the subdomain row offsets; built once per discretization."""
    import torch
    from .kernels import DeviceCsr
    hit = d.__dict__.get('_energy_cache')
    if hit is None:
        S = len(d.solution_space.subspaces)
        mats = [d.operators['local_energy_dg_product_{}'.format(i)].csr for i in range(S)]
        offs = np.concatenate([[0], np.cumsum([m.shape[0] for m in mats])]).astype(np.int64)
        nnz = np.concatenate([[0], np.cumsum([m.nnz for m in mats])]).astype(np.int64)
        rowptr = torch.cat([m.rowptr[:-1].to(torch.int64) + int(nnz[i]) for i, m in enumerate(mats)] +
                           [torch.tensor([int(nnz[-1])], dtype=torch.int64, device='cuda')]).to(torch.int32)
        colind = torch.cat([m.colind[:m.nnz] + int(offs[i]) for i, m in enumerate(mats)])
        values = torch.cat([m.values[:m.nnz] for m in mats]).reshape(1, -1).contiguous()
        pattern = DeviceCsr.from_device(rowptr, colind, values[0], (int(offs[-1]), int(offs[-1])))
        hit = d._energy_cache = (pattern, values, offs)
    return hit


def reduction_error_analysis(d, reductor, rd, mus, U_h=None, inverse_options=None):
    """True reduction errors and estimator effectivities of the reduced model ``rd`` (built by ``reductor`` from ``d``)
    over the parameter batch ``mus``; returns a :class:`ReductionErrorAnalysis`.

    ``U_h`` (a block array of ``len(mus)`` fine solutions) defaults to ``d.solve_batch(mus, inverse_options)``; a failing
    fine solve raises :class:`LrbmsError` as ``solve_batch`` does.  ``rd.sweep(mus, decompose=True)`` gives ``u_N``, ``eta``
    and the local indicators; a reduced system that is not positive definite raises there.  ``u_N`` is reconstructed with
    the first ``rd.block_dims[i]`` vectors of each local basis (``reductor.reconstruct`` semantics: the bases may have
    grown since ``rd`` was reduced).  The batch runs in chunks whose error scratch fits ``d.fom_workspace_budget``; the
    results do not depend on the chunking."""
    import torch
    from .kernels import recon_error, segmented_form
    from .parameters import theta_matrix
    from .vectorarray import _round_cap
    mus = list(mus)
    S, n_mu = _check_arguments(d, reductor, rd, mus, U_h)
    subs = d.solution_space.subspaces
    fom_info = None
    if U_h is None:
        U_h = d.solve_batch(mus, inverse_options=inverse_options)
        fom_info = {k: np.array(v) for k, v in d.last_solve_info.items()}
    U_N, eta, _, indicators = rd.sweep(mus, decompose=True)
    n = d.solution_space.dim
    u_h = _dofmajor(U_h, n, n_mu)
    u_N = U_N.device_tensor.contiguous()
    bases = [reductor.bases[s.id] for s in subs]
    E_pat, E_vals, offs = _energy_system(d)
    A_pat, A_vals, _ = d.affine_system(range(S))
    theta = torch.from_numpy(theta_matrix(list(d.operator.coefficients) + list(d.rhs.coefficients), mus,
                                          d.parameter_type)).cuda()
    chunk = int(max(1, min(n_mu, d.fom_workspace_budget // max(1, 8 * n))))
    e = torch.empty((n, _round_cap(chunk)), dtype=torch.float64, device='cuda')
    local_sq = torch.empty((S, n_mu), dtype=torch.float64, device='cuda')
    uh_sq = torch.empty((S, n_mu), dtype=torch.float64, device='cuda')
    op_sq = torch.empty((1, n_mu), dtype=torch.float64, device='cuda')
    for c0 in range(0, n_mu, chunk):
        c1 = min(n_mu, c0 + chunk)
        recon_error(bases, rd.block_dims, u_h[:, c0:], u_N[c0:c1], e)
        segmented_form(E_pat, E_vals, offs, e, c1 - c0, out=local_sq[:, c0:c1])
        segmented_form(A_pat, A_vals, [0, n], e, c1 - c0, theta=theta[c0:c1], out=op_sq[:, c0:c1])
        segmented_form(E_pat, E_vals, offs, u_h[:, c0:], c1 - c0, out=uh_sq[:, c0:c1])
    local_sq, uh_sq, op_sq = local_sq.cpu().numpy(), uh_sq.cpu().numpy(), op_sq.cpu().numpy()[0]
    local_errors = np.sqrt(np.maximum(local_sq, 0.0))
    errors = np.sqrt(np.maximum(_sum_subdomains(local_sq), 0.0))
    norms = np.sqrt(np.maximum(_sum_subdomains(uh_sq), 0.0))
    eta = np.asarray(eta, dtype=np.float64)
    with np.errstate(divide='ignore', invalid='ignore'):
        relative = np.where(norms > 0, errors / np.where(norms > 0, norms, 1.0), np.where(errors > 0, np.inf, 0.0))
        eff = np.where(errors > 0, eta / np.where(errors > 0, errors, 1.0), np.inf)
        local_eff = np.where(local_errors > 0, indicators / np.where(local_errors > 0, local_errors, 1.0), np.inf)
    k = int(np.argmax(errors))
    return ReductionErrorAnalysis(errors=errors, operator_errors=np.sqrt(np.maximum(op_sq, 0.0)), local_errors=local_errors,
                                  relative_errors=relative, eta=eta, indicators=np.asarray(indicators),
                                  effectivities=eff, local_effectivities=local_eff, max_error=float(errors[k]), argmax=k,
                                  min_effectivity=float(eff.min()), max_effectivity=float(eff.max()), fom_info=fom_info)
