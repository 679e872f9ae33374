"""The block-SWIPDG discretization object the LRBMS hot path consumes, resident in HBM.

``discretize(data)`` restates the assembly-independent part of the reference's ``discretize()``
(``discretize_elliptic_block_swipdg.py:581-811``; SURVEY.md Appendix B): it wraps host-assembled CSR blocks
(:class:`pylrbms_b200.swipdg_fixture.BlockSwipdgData`, standing in for dune-gdt assembly, which is out of scope)
into the same operator dictionary -- same names, same source / range spaces, same compositions -- with every
matrix uploaded to the device once.  Matrices that appear in several operators share one upload.
"""
from __future__ import annotations

import numpy as np

from .estimators import EllipticEstimator
from .kernels import DeviceCsr
from .operators import (BlockDiagonalOperator, BlockOperator, BlockProjectionOperator, BlockRowOperator, Concatenation,
                        CsrOperator, FluxReconstructionOperator, LincombOperator, OswaldInterpolationErrorOperator,
                        VectorFunctional)
from .parameters import ProductParameterFunctional, as_functional, parse_parameter
from .vectorarray import GpuVectorSpace


class BlockSwipdgDiscretization:
    """``DuneDiscretization`` stand-in (reference ``discretize...:203-225``): ``operator``, ``rhs``, ``operators``,
    ``products``, ``estimator``, ``solution_space``, ``neighborhoods``, ``shape_functions``."""

    def __init__(self, operator, rhs, products=None, operators=None, estimator=None, parameter_type=None,
                 neighborhoods=None, shape_function_data=None, solution_space=None, parameter_range=None, name=None):
        self.operator, self.rhs = operator, rhs
        self.products = dict(products or {})
        self.operators = dict(operators or {})
        self.operators.setdefault('operator', operator)
        self.operators.setdefault('rhs', rhs)
        self.estimator = estimator
        self.parameter_type = dict(parameter_type or {})
        self.parameter_range = parameter_range
        self.neighborhoods = neighborhoods
        self._shape_function_data = shape_function_data
        self.solution_space = solution_space if solution_space is not None else operator.source
        self.name = name
        self.linear = True

    def with_(self, **kw):
        import copy
        new = copy.copy(self)
        for k, v in kw.items():
            setattr(new, k, v)
        if 'operators' in kw:
            new.operator = kw['operators'].get('operator', new.operator)
            new.rhs = kw['operators'].get('rhs', new.rhs)
        return new

    def parse_parameter(self, mu):
        return parse_parameter(mu, self.parameter_type)

    #: device workspace bytes one call of the batched fine-scale solve may use; larger batches are solved in chunks
    #: (each parameter's result does not depend on the chunking)
    fom_workspace_budget = 4 << 30

    def affine_system(self, subdomains):
        """The affine components of the operator restricted to ``subdomains`` (in that order) on ONE sparsity pattern:
        ``(pattern, values, rhs)`` with ``pattern`` a :class:`DeviceCsr` (its ``values`` are scratch for the caller),
        ``values`` the ``(Q, nnz)`` component values and ``rhs`` the ``(Qf, n)`` right-hand side terms, all in HBM, so
        that ``A(mu) = sum_q theta_q A_q`` is one pass over Q value arrays on the device.  Built once per subdomain tuple;
        the union pattern is formed on the device from (row * n + column) keys."""
        import scipy.sparse as sp
        import torch
        key = tuple(int(k) for k in subdomains)
        cache = self.__dict__.setdefault('_affine_cache', {})
        if key not in cache:
            keys, datas, n_nb = [], [], 0
            for op in self.operator.operators:
                blocks = [[(op._blocks[k, l].csr.host if op._blocks[k, l] is not None else None) for l in key] for k in key]
                M = sp.bmat(blocks, format='csr')
                M.sum_duplicates()
                n_nb = M.shape[0]
                kk = np.repeat(np.arange(n_nb, dtype=np.int64), np.diff(M.indptr)) * n_nb + M.indices
                keys.append(torch.from_numpy(kk).cuda())
                datas.append(torch.from_numpy(np.ascontiguousarray(M.data, dtype=np.float64)).cuda())
            key_p = torch.unique(torch.cat(keys), sorted=True)
            vals = torch.zeros((len(keys), key_p.numel()), dtype=torch.float64, device='cuda')
            for q in range(len(keys)):
                vals[q, torch.searchsorted(key_p, keys[q])] = datas[q]
            rows_p = torch.div(key_p, n_nb, rounding_mode='floor')
            rowptr = torch.zeros(n_nb + 1, dtype=torch.int64, device='cuda')
            rowptr[1:] = torch.cumsum(torch.bincount(rows_p, minlength=n_nb), 0)
            A_dev = DeviceCsr.from_device(rowptr.to(torch.int32), (key_p - rows_p * n_nb).to(torch.int32), vals[0].clone(),
                                          (n_nb, n_nb))
            f = torch.stack([torch.cat([torch.from_numpy(o._array._blocks[k].to_numpy()[0]).cuda() for k in key])
                             for o in self.rhs.operators]).contiguous()
            cache[key] = (A_dev, vals, f)
        return cache[key]

    def solve(self, mu=None, inverse_options=None):
        """``d.solve(mu)``: the fine-scale solution for one parameter (reference ``LincombOperator.assemble(mu)`` +
        ``apply_inverse``, dune-istl); a block array of length 1.  See :meth:`solve_batch`."""
        return self.solve_batch(None if mu is None and not self.parameter_type else [self.parse_parameter(mu)],
                                inverse_options=inverse_options)

    def solve_batch(self, mus, inverse_options=None):
        """Fine-scale solutions for a parameter batch with the mu-batched Jacobi-preconditioned CG
        (``lrbms_affine_pcg_solve``), from a zero initial guess.  ``inverse_options`` may hold ``rtol`` (true relative
        residual, default 1e-9: the FP64 rounding of b - A x alone leaves up to ~1e-10 at C2, n = 393 216),
        ``maxiter`` (default max(100, 10 n)) and ``restarts`` (default 3).  Returns a :class:`BlockVectorArray` of length
        ``len(mus)`` whose blocks are views of one dof-major result buffer.
        ``self.last_solve_info`` holds the per-parameter ``iterations``, ``relative_residual`` and ``status``
        (0 converged, 1 not converged, 2 operator not positive definite); any non-zero status raises
        :class:`LrbmsError` and no solution is returned."""
        import torch
        from ._lib import LrbmsError
        from .kernels import affine_pcg_solve, affine_pcg_workspace_bytes
        from .parameters import theta_matrix
        from .vectorarray import BlockVectorArray, _round_cap
        S = len(self.solution_space.subspaces)
        pattern, values, rhs = self.affine_system(range(S))
        coeffs = list(self.operator.coefficients) + list(self.rhs.coefficients)
        theta = torch.from_numpy(theta_matrix(coeffs, mus, self.parameter_type)).cuda()
        n, n_mu = pattern.shape[0], theta.shape[0]
        opts = dict(inverse_options or {})
        rtol = float(opts.get('rtol', 1e-9))
        maxiter = int(opts['maxiter']) if opts.get('maxiter') is not None else max(100, 10 * n)
        restarts = int(opts.get('restarts', 3))
        buf = torch.zeros((n, _round_cap(n_mu)), dtype=torch.float64, device='cuda')
        per_32 = affine_pcg_workspace_bytes(n, 32)
        chunk = max(1, int(self.fom_workspace_budget * 32 // per_32))
        info = {k: np.zeros(n_mu, dtype=dt) for k, dt in (('iterations', np.int32), ('relative_residual', np.float64),
                                                            ('status', np.int32))}
        for c0 in range(0, n_mu, chunk):
            c1 = min(n_mu, c0 + chunk)
            _, it, rr, st = affine_pcg_solve(pattern, values, rhs, theta[c0:c1], buf[:, c0:], rtol, maxiter, restarts)
            info['iterations'][c0:c1], info['relative_residual'][c0:c1], info['status'][c0:c1] = it, rr, st
        self.last_solve_info = info
        bad = np.flatnonzero(info['status'])
        if bad.size:
            k = int(bad[0])
            raise LrbmsError('fine-scale solve failed for parameter #{}: status {} ({}), relative residual {:.3e} '
                             '(rtol {:.1e}) after {} iterations'.format(
                                 k, int(info['status'][k]), {1: 'not converged', 2: 'operator not positive definite'}
                                 .get(int(info['status'][k]), 'unknown'), info['relative_residual'][k], rtol,
                                 int(info['iterations'][k])))
        offs = np.concatenate([[0], np.cumsum([s.dim for s in self.solution_space.subspaces])])
        blocks = [sub.from_dofmajor(buf[offs[i]:offs[i + 1]], n_mu) for i, sub in enumerate(self.solution_space.subspaces)]
        return BlockVectorArray(blocks, self.solution_space)

    def estimate(self, U, mu=None, decompose=False):
        """Estimate for a *fine-scale* block array ``U`` through the generic operator chain, one parameter at a time,
        exactly as the reference does (``estimators.py:45-112``)."""
        return self.estimator.estimate(U, self.parse_parameter(mu), self, decompose=decompose)

    def solve_for_local_correction(self, subdomain, Us, mu=None, inverse_options=None):
        """Local corrector problem on the neighbourhood of ``subdomain`` (reference ``discretize...:227-316``).

        The reference assembles the SWIPDG operator on the neighbourhood grid with dune-gdt, solves
        ``(sum_q theta_q(mu) A_q^nbh) c = f^nbh`` (the current solution ``Us`` does not enter: its boundary functional is
        commented out, ``:247-260``) and restricts ``c`` to the subdomain.  Assembly is outside the hot path, so here the
        neighbourhood operator is the principal submatrix of the global block operator over the neighbourhood: the
        one-sided coupling terms the diagonal blocks carry on the outer interfaces act as the weakly imposed homogeneous
        Dirichlet condition of the oversampling problem.  The solve runs on the GPU (``lrbms_pcg_solve``);
        ``inverse_options`` may hold ``{'rtol': ..., 'maxiter': ...}``.  ``Us`` is accepted for signature parity."""
        from .kernels import pcg_solve
        mu = self.parse_parameter(mu)
        nb = list(self.neighborhoods[subdomain])
        A_dev, vals_q, f = self.affine_system(nb)
        f = f[0]
        theta = [c.evaluate(mu) if hasattr(c, 'evaluate') else float(c) for c in self.operator.coefficients]
        values = float(theta[0]) * vals_q[0]
        for q in range(1, vals_q.shape[0]):
            values += float(theta[q]) * vals_q[q]                      # left to right, as the reference's LincombOperator assembles
        A_dev.values = values
        opts = dict(inverse_options or {})
        # CG to the requested recurrence residual, then restarts from the iterate: a restart recomputes the TRUE residual
        # b - A x (the recurrence residual drifts away from it), so the iterate reaches the attainable accuracy eps * cond(A) of
        # a direct solve -- what the reference's apply_inverse (dune-istl / a sparse direct solver) delivers.  The enriched
        # reduced model then matches a direct-solve enrichment to ~1e-10 instead of the 1e-7 of a single CG run.
        rtol = float(opts.get('rtol', 1e-13))
        x, iters, relres = pcg_solve(A_dev, f, rtol=rtol, max_iter=opts.get('maxiter'))
        restarts = 0
        for _ in range(int(opts.get('restarts', 3))):
            x2, it2, rr2 = pcg_solve(A_dev, f, x0=x, rtol=0.1 * rtol, max_iter=opts.get('maxiter'))
            restarts += 1
            iters += it2
            improved = rr2 < 0.5 * relres
            if rr2 <= relres:
                x, relres = x2, rr2
            if it2 == 0 or not improved:
                break
        self.last_local_correction_info = {'iterations': iters, 'relative_residual': relres, 'size': int(A_dev.shape[0]),
                                           'restarts': restarts}
        if not relres <= rtol:
            # the reference's apply_inverse raises on solver failure; an unconverged corrector must not enter a basis
            from ._lib import LrbmsError
            raise LrbmsError('local corrector solve on subdomain {} did not converge: relative residual {:.3e} > {:.1e} after '
                             '{} iterations'.format(subdomain, relres, rtol, iters))
        sizes = [self.solution_space.subspaces[k].dim for k in nb]
        start = int(np.sum(sizes[:nb.index(subdomain)]))
        local = x[start:start + sizes[nb.index(subdomain)]]
        return self.solution_space.subspaces[subdomain].from_data(local.cpu().numpy()[None, :])

    def shape_functions(self, subdomain, order=0):
        """reference ``discretize...:187-200``: constant 1, then x, y, x*y."""
        sf = self._shape_function_data[subdomain]
        return self.solution_space.subspaces[subdomain].from_data(sf[:(1 if order == 0 else 4)])


def discretize(data, alpha_returns_first=True):
    """Build the device-resident operator set of SURVEY.md Appendix B from host CSR data.

    Returns ``(d, data_dict)`` like the reference's ``discretize()`` (``discretize...:811``)."""
    S, Q = data.num_subdomains, data.Q
    lambda_coeffs = [as_functional(c, data.parameter_type) for c in data.coefficients]
    dom = [GpuVectorSpace(int(data.n[i]), 'domain_{}'.format(i)) for i in range(S)]

    # ---- block lhs (discretize...:475-507, 586)
    block_ops = []
    for q in range(Q):
        ops = np.full((S, S), None, dtype=object)
        for (i, j), M in data.lhs[q].items():
            ops[i, j] = CsrOperator(M, source_id=dom[j].id, range_id=dom[i].id, name='local_block_{}-{}'.format(i, j))
        block_ops.append(BlockOperator(ops, range_spaces=dom, source_spaces=dom, name='BlockOp'))
    block_op = LincombOperator(block_ops, lambda_coeffs, name='lhs')
    solution_space = block_op.source
    # ---- block rhs (discretize...:523-527, 598)
    rhs_blocks = [dom[i].from_data(data.rhs[i]) for i in range(S)]
    block_rhs = LincombOperator([VectorFunctional(solution_space.make_array(rhs_blocks))], [1.], name='rhs')

    # ---- Oswald interpolation error / flux reconstruction (discretize...:606-618)
    oi_op = BlockDiagonalOperator(
        [OswaldInterpolationErrorOperator(i, solution_space, data.neighborhoods[i],
                                          [data.oi[(i, k)] for k in data.neighborhoods[i]]) for i in range(S)],
        name='oswald_interpolation_error')
    fr_op = LincombOperator(
        [BlockDiagonalOperator([FluxReconstructionOperator(i, solution_space, data.neighborhoods[i], data.m,
                                                           [data.fr[q][(i, k)] for k in data.neighborhoods[i]])
                                for i in range(S)]) for q in range(Q)],
        lambda_coeffs, name='flux_reconstruction')

    operators, local_l2_products = {}, []
    for ii in range(S):
        neighborhood = data.neighborhoods[ii]
        did, rid = 'domain_{}'.format(ii), 'LOCALRT_{}'.format(ii)
        # local products (discretize...:644-691)
        name = 'local_energy_dg_product_{}'.format(ii)
        operators[name] = CsrOperator(data.energy[ii], source_id=did, range_id=did, name=name)
        local_l2_product = CsrOperator(data.l2[ii], source_id=did, range_id=did, name='local_l2_product_{}'.format(ii))
        local_l2_products.append(local_l2_product)
        local_elliptic_product = CsrOperator(data.elliptic[ii], source_id=did, range_id=did)
        # projections (discretize...:695-717)
        local_projection = BlockProjectionOperator(solution_space, ii)
        ops = [None] * S
        for kk in neighborhood:
            component = data.neighborhoods[kk].index(ii)
            assert fr_op.range.subspaces[kk].subspaces[component].id == rid
            ops[kk] = BlockProjectionOperator(fr_op.range.subspaces[kk], component)
        local_rt_projection = BlockRowOperator(ops, source_spaces=fr_op.range.subspaces,
                                               name='local_rt_projection_{}'.format(ii))
        ops = [None] * S
        for kk in neighborhood:
            component = data.neighborhoods[kk].index(ii)
            assert oi_op.range.subspaces[kk].subspaces[component].id == did
            ops[kk] = BlockProjectionOperator(oi_op.range.subspaces[kk], component)
        local_oi_projection = BlockRowOperator(ops, source_spaces=oi_op.range.subspaces,
                                               name='local_oi_projection_{}'.format(ii))
        # divergence (discretize...:721-729)
        local_div_op = CsrOperator(data.div[ii], source_id=rid, range_id=did, name='local_divergence_{}'.format(ii))
        # nonconformity (discretize...:733-735)
        operators['nc_{}'.format(ii)] = Concatenation([local_oi_projection.T, local_elliptic_product, local_oi_projection],
                                                      name='nonconformity_{}'.format(ii))
        # residual (discretize...:739-748); only built for a single rhs term, like the reference
        local_div = Concatenation([local_div_op, local_rt_projection])
        local_rhs = VectorFunctional(block_rhs.operators[0]._array._blocks[ii])
        operators['r_fd_{}'.format(ii)] = Concatenation([local_rhs, local_div], name='r1_{}'.format(ii))
        operators['r_dd_{}'.format(ii)] = Concatenation([local_div.T, local_l2_product, local_div], name='r2_{}'.format(ii))
        # diffusive flux (discretize...:319-378, 752-770)
        aa_ops = []
        for q in range(Q):
            for q2 in range(Q):
                df_ops = np.full((S, S), None, dtype=object)
                df_ops[ii, ii] = CsrOperator(data.aa[q][q2][ii], source_id=did, range_id=did)
                aa_ops.append(BlockOperator(df_ops, range_spaces=dom, source_spaces=dom))
        operators['df_aa_{}'.format(ii)] = LincombOperator(
            aa_ops, [ProductParameterFunctional([c1, c2]) for c1 in lambda_coeffs for c2 in lambda_coeffs],
            name='diffusive_flux_aa_{}'.format(ii))
        bbm = CsrOperator(data.bb[ii], source_id=rid, range_id=rid)
        operators['df_bb_{}'.format(ii)] = Concatenation([local_rt_projection.T, bbm, local_rt_projection],
                                                         name='diffusive_flux_bb_{}'.format(ii))
        operators['df_ab_{}'.format(ii)] = LincombOperator(
            [Concatenation([local_projection.T, CsrOperator(data.ab[q][ii], source_id=rid, range_id=did),
                            local_rt_projection]) for q in range(Q)],
            lambda_coeffs, name='diffusive_flux_ab_{}'.format(ii))

    estimator = EllipticEstimator(list(range(S)), data.min_diffusion_evs, data.subdomain_diameters,
                                  data.local_eta_rf_squared, lambda_coeffs, data.mu_bar, data.mu_hat, fr_op, oi_op,
                                  alpha_returns_first=alpha_returns_first)
    l2_product = BlockDiagonalOperator(local_l2_products, name='l2')
    d = BlockSwipdgDiscretization(block_op, block_rhs, products={'l2': l2_product}, operators=operators,
                                  estimator=estimator, parameter_type=data.parameter_type,
                                  neighborhoods=data.neighborhoods, shape_function_data=data.shape_functions,
                                  solution_space=solution_space, parameter_range=data.parameter_range,
                                  name=data.meta.get('problem'))
    info = {'num_subdomains': S, 'neighborhoods': data.neighborhoods, 'n': data.n, 'm': data.m,
            'local_products': [operators['local_energy_dg_product_{}'.format(i)] for i in range(S)]}
    from .reductor import prepare_operators
    prepare_operators(d)              # symmetry flags, fused chain products, transposes: operator-only, done once here
    return d, info
