"""The reduced model: block-sparse reduced operators in HBM and the mu-batched online phase (K3 + K4 + K5).

``ReducedModel`` stands in for the ``StationaryDiscretization`` the reference's ``reductor.reduce()`` returns:
``rd.solve(mu)`` (reference ``online_enrichment.py:72``, ``scripts/online_adaptive_lrbms.py:141``) and
``rd.estimate(U, mu=, decompose=)`` (``online_enrichment.py:61,74``) keep their signatures; ``solve_batch``,
``estimate_batch`` and ``sweep`` are the parameter-batched forms the reference does not have (it handles one mu per
call, SURVEY.md section 2.3).

Execution: the reference assembles ``sum_q theta_q(mu) A_q`` as a dense unblocked ``n_red x n_red`` NumPy matrix, runs
``numpy.linalg.solve`` on it and evaluates six dense mat-vec quadratic forms per subdomain
(``estimators.py:70-91``).  Here the reduced blocks never leave their packed block-sparse layout; one call of
``lrbms_online_sweep`` assembles, factors (8x8-tile sparse Cholesky on FP64 tensor cores), solves and estimates a
whole batch of parameters.
"""
from __future__ import annotations

import copy
import ctypes as C

import numpy as np

from . import _lib
from ._lib import Handle, LrbmsError, current_stream_ptr, host_f64, host_i32, ptr
from .parameters import ParameterFunctional, ProductParameterFunctional, parse_parameter, theta_matrix
from .vectorarray import ReducedVectorArray


def _torch():
    import torch
    return torch


class _Dim:
    def __init__(self, dim, id_=None):
        self.dim, self.id = int(dim), id_


class SuperBlock:
    """One dense output of the projection plan covering ``row_idx x col_idx`` subspaces (row-major ``rows x cols``)."""
    __slots__ = ('row_idx', 'col_idx', 'token', 'rows', 'cols', 'row_sizes', 'col_sizes')

    def __init__(self, row_idx, col_idx, token, rows, cols, row_sizes=None, col_sizes=None):
        self.row_idx, self.col_idx, self.token = list(row_idx), list(col_idx), token
        self.rows, self.cols = int(rows), int(cols)
        self.row_sizes = list(row_sizes) if row_sizes is not None else [self.rows]
        self.col_sizes = list(col_sizes) if col_sizes is not None else [self.cols]


class ReducedBlockOperator:
    """A projected (block) operator: dense super-blocks inside the planner's output buffer.

    ``to_dense()`` is what the reference's ``unblock`` would store (``reductor.py:46,66``; SURVEY.md row a10)."""
    linear = True

    def __init__(self, owner, sblocks, range_dims, source_dims, name=None, functional=False):
        self._owner = owner                 # object with .out (device buffer) and .offsets (token -> offset)
        self.sblocks = list(sblocks)
        self.range_dims, self.source_dims = list(range_dims), list(source_dims)
        self.range, self.source = _Dim(sum(self.range_dims)), _Dim(sum(self.source_dims))
        self.name, self.functional = name, functional

    def offset(self, sb):
        return int(self._owner.offsets[sb.token])

    def device_block(self, sb):
        o = self.offset(sb)
        return self._owner.out[o:o + sb.rows * sb.cols].view(sb.rows, sb.cols)

    @property
    def buffer(self):
        return self._owner.out

    def blocks(self):
        """``{(i, j): dense block}`` keyed by range / source subspace position (host copies)."""
        out = {}
        for sb in self.sblocks:
            M = self.device_block(sb).cpu().numpy()
            ro = np.concatenate([[0], np.cumsum(sb.row_sizes)])
            co = np.concatenate([[0], np.cumsum(sb.col_sizes)])
            for a, i in enumerate(sb.row_idx):
                for b, j in enumerate(sb.col_idx):
                    out[(i, j)] = M[ro[a]:ro[a + 1], co[b]:co[b + 1]]
        return out

    def to_dense(self):
        ro = np.concatenate([[0], np.cumsum(self.range_dims)])
        co = np.concatenate([[0], np.cumsum(self.source_dims)])
        M = np.zeros((ro[-1], co[-1]))
        for (i, j), B in self.blocks().items():
            M[ro[i]:ro[i + 1], co[j]:co[j + 1]] = B
        return M

    matrix = property(to_dense)

    def as_source_array(self, mu=None):
        assert self.functional
        return self.to_dense()

    def assemble(self, mu=None):
        return self

    def with_(self, **kw):
        new = copy.copy(self)
        for k, v in kw.items():
            setattr(new, k, v)
        return new

    # -- LincombOperator.assemble(mu) support: sum_q c_q A_q on the packed blocks (va_axpy kernel, one vector of length rows*cols)
    def lincomb_assemble(self, ops, coefficients, name=None):
        torch = _torch()
        h = Handle.get()
        keyed = [{(tuple(sb.row_idx), tuple(sb.col_idx)): (o, sb) for sb in o.sblocks} for o in ops]
        if any(set(k) != set(keyed[0]) for k in keyed[1:]):
            raise NotImplementedError('assemble: affine components with different block patterns')
        total = sum(sb.rows * sb.cols for sb in self.sblocks)
        holder = _Buffer(torch.zeros(max(1, total), dtype=torch.float64, device='cuda'))
        sblocks, pos = [], 0
        for sb in self.sblocks:
            key = (tuple(sb.row_idx), tuple(sb.col_idx))
            size = sb.rows * sb.cols
            holder.offsets.append(pos)
            nsb = SuperBlock(sb.row_idx, sb.col_idx, len(holder.offsets) - 1, sb.rows, sb.cols, sb.row_sizes, sb.col_sizes)
            for q, (c, k) in enumerate(zip(coefficients, keyed)):
                o, osb = k[key]
                src = o.buffer.data_ptr() + 8 * o.offset(osb)
                a = host_f64([c])
                if size:
                    h.check(h.lib.lrbms_va_axpy(h.h, size, 1, ptr(a), 1, src, 1, 1, holder.out.data_ptr() + 8 * pos, 1,
                                                current_stream_ptr()))
            sblocks.append(nsb)
            pos += size
        return ReducedBlockOperator(holder, sblocks, self.range_dims, self.source_dims, name=name, functional=self.functional)

    def apply_inverse(self, V, mu=None):
        """Solve with this (assembled, symmetric positive definite) reduced operator: a one-term online plan."""
        if hasattr(V, '__len__') and len(V) != 1:
            raise NotImplementedError('apply_inverse: exactly one right-hand side vector (got {})'.format(len(V)))
        model = ReducedModel(_SingleTerm(self), _SingleTerm(_HostFunctional(V)), block_dims=self.source_dims)
        return model.solve(None)


class _Buffer:
    def __init__(self, out):
        self.out, self.offsets = out, []


class _SingleTerm:
    def __init__(self, op):
        self.operators, self.coefficients = [op], [1.0]


class _HostFunctional:
    """Right-hand side given as a host / reduced array (used by ``apply_inverse``)."""
    functional = True

    def __init__(self, V):
        self._v = np.asarray(V.data if hasattr(V, 'data') else V, dtype=np.float64).reshape(-1)

    def device_vector(self):
        torch = _torch()
        return torch.from_numpy(self._v.copy()).cuda()


class ReducedFluxReconstruction:
    """Reduced flux reconstruction ``fr_red`` (reference ``reductor.py:61-66``): per subdomain the map
    ``u_i -> [theta_0(mu) u_i; ...; theta_{Q-1}(mu) u_i]``.  Never materialised online -- the estimator kernel folds the
    ``theta_q`` in (SURVEY.md row a13); ``matrix(mu)`` builds the unblocked matrix for inspection."""

    def __init__(self, coefficients, block_dims):
        self.coefficients, self.block_dims = list(coefficients), list(block_dims)

    def matrix(self, mu=None):
        Q, N = len(self.coefficients), self.block_dims
        th = [c.evaluate(mu) if isinstance(c, ParameterFunctional) else float(c) for c in self.coefficients]
        n = sum(N)
        M = np.zeros((Q * n, n))
        r = c = 0
        for Ni in N:
            for q in range(Q):
                M[r + q * Ni:r + (q + 1) * Ni, c:c + Ni] = th[q] * np.eye(Ni)
            r += Q * Ni
            c += Ni
        return M

    def apply(self, U, mu=None):
        torch = _torch()
        th = [c.evaluate(mu) if isinstance(c, ParameterFunctional) else float(c) for c in self.coefficients]
        u = U.device_tensor
        offs = np.concatenate([[0], np.cumsum(self.block_dims)])
        parts = [th[q] * u[:, offs[k]:offs[k + 1]] for k in range(len(self.block_dims)) for q in range(len(th))]
        return ReducedVectorArray(torch.cat(parts, dim=1), [len(th) * n for n in self.block_dims])


class ReducedOswaldInterpolation:
    """Reduced Oswald interpolation error ``oi_red`` = identity (reference ``reductor.py:44-46``)."""

    def __init__(self, block_dims):
        self.block_dims = list(block_dims)

    def matrix(self, mu=None):
        return np.eye(sum(self.block_dims))

    def apply(self, U, mu=None):
        return U


# ----------------------------------------------------------------------------------------------------------
#  reduced model
# ----------------------------------------------------------------------------------------------------------

class ReducedModel:
    def __init__(self, operator, rhs, products=None, operators=None, estimator=None, parameter_type=None,
                 block_dims=None, neighborhoods=None, parameter_range=None, keepalive=None):
        self.operator, self.rhs = operator, rhs
        self.products = dict(products or {})
        self.operators = dict(operators or {})
        self.estimator = estimator
        self.parameter_type = dict(parameter_type or {})
        self.parameter_range = parameter_range
        self.block_dims = [int(n) for n in block_dims]
        self.neighborhoods = neighborhoods
        self.solution_space = _Dim(sum(self.block_dims), 'STATE')
        self._keep = keepalive
        self._plan = None
        self._plan_has_estimator = False
        self._work = {}
        self.linear = True
        self.solver = 'auto'        # 'auto' | 'window' | 'banded' (lrbms_sm100.h LRBMS_SOLVER_*)

    def with_(self, **kw):
        new = copy.copy(self)
        for k, v in kw.items():
            setattr(new, k, v)
        new._plan, new._work = None, {}
        return new

    @property
    def n_red(self):
        return self.solution_space.dim

    def parse_parameter(self, mu):
        return parse_parameter(mu, self.parameter_type)

    # -- coefficient evaluation on the host (theta_q are tiny expressions; reference: ExpressionParameterFunctional)
    def thetas(self, mus):
        """``(n_mu, Q + Qf)`` coefficient matrix for a parameter batch."""
        return theta_matrix(list(self.operator.coefficients) + list(self.rhs.coefficients), mus, self.parameter_type)

    # -- online plan -------------------------------------------------------------------------------------
    def _theta_index(self, functional, lam):
        for q, c in enumerate(lam):
            if c is functional:
                return q
        raise NotImplementedError('estimator coefficient {} is not one of the affine coefficients of the operator'.format(functional))

    def _estimator_terms(self):
        """Map the reduced estimator operators onto kernel terms (reference ``estimators.py:71-85``)."""
        L = _lib
        est, ops, lam = self.estimator, self.operators, list(self.operator.coefficients)
        fr = est.flux_reconstruction
        if not (len(fr.coefficients) == len(lam) and all(a is b for a, b in zip(fr.coefficients, lam))):
            raise NotImplementedError('the flux reconstruction must share the affine coefficients of the operator')
        terms = []

        def single(op, what):
            if len(op.sblocks) != 1:
                raise NotImplementedError('{}: expected one dense neighbourhood block'.format(what))
            return op.sblocks[0]

        for ii, sub in enumerate(est.subdomains):
            nb = list(self.neighborhoods[sub])
            nc = ops['nc_{}'.format(sub)]
            sb = single(nc, 'nc')
            assert sb.row_idx == nb and sb.col_idx == nb
            terms.append((sub, L.OUT_NC, L.VEC_UN, L.VEC_UN, sb.rows, sb.cols, -1, -1, 1.0, nc.offset(sb)))
            rfd = ops['r_fd_{}'.format(sub)]
            sb = single(rfd, 'r_fd')
            assert sb.col_idx == nb and sb.rows == 1
            terms.append((sub, L.OUT_R, L.VEC_ONE, L.VEC_UR, 1, sb.cols, -1, -1, -2.0, rfd.offset(sb)))
            rdd = ops['r_dd_{}'.format(sub)]
            sb = single(rdd, 'r_dd')
            assert sb.row_idx == nb and sb.col_idx == nb
            terms.append((sub, L.OUT_R, L.VEC_UR, L.VEC_UR, sb.rows, sb.cols, -1, -1, 1.0, rdd.offset(sb)))
            aa = ops['df_aa_{}'.format(sub)]
            for o, c in zip(aa.operators, aa.coefficients):
                sb = single(o, 'df_aa')
                assert sb.row_idx == [sub] and sb.col_idx == [sub]
                if not (isinstance(c, ProductParameterFunctional) and len(c.factors) == 2):
                    raise NotImplementedError('df_aa coefficients must be products of two affine coefficients')
                qa, qb = self._theta_index(c.factors[0], lam), self._theta_index(c.factors[1], lam)
                terms.append((sub, L.OUT_DF, L.VEC_UI, L.VEC_UI, sb.rows, sb.cols, qa, qb, 1.0, o.offset(sb)))
            bb = ops['df_bb_{}'.format(sub)]
            sb = single(bb, 'df_bb')
            assert sb.row_idx == nb and sb.col_idx == nb
            terms.append((sub, L.OUT_DF, L.VEC_UR, L.VEC_UR, sb.rows, sb.cols, -1, -1, 1.0, bb.offset(sb)))
            ab = ops['df_ab_{}'.format(sub)]
            for o, c in zip(ab.operators, ab.coefficients):
                sb = single(o, 'df_ab')
                assert sb.row_idx == [sub] and sb.col_idx == nb
                terms.append((sub, L.OUT_DF, L.VEC_UI, L.VEC_UR, sb.rows, sb.cols, self._theta_index(c, lam), -1, 2.0,
                              o.offset(sb)))
        return terms

    def _build_plan(self):
        torch = _torch()
        L = _lib
        h = Handle.get()
        lhs_terms, rhs_terms = self.operator.operators, self.rhs.operators
        Q, Qf, S = len(lhs_terms), len(rhs_terms), len(self.block_dims)
        pattern = [(sb.row_idx[0], sb.col_idx[0]) for sb in lhs_terms[0].sblocks]
        for o in lhs_terms:
            if [(sb.row_idx[0], sb.col_idx[0]) for sb in o.sblocks] != pattern or any(len(sb.row_idx) != 1 for sb in o.sblocks):
                raise NotImplementedError('all affine components of the reduced operator need the same block pattern')
        buf = lhs_terms[0].buffer
        if any(o.buffer is not buf for o in lhs_terms):
            raise NotImplementedError('affine components of the reduced operator must share one device buffer')
        bi = host_i32([p[0] for p in pattern])
        bj = host_i32([p[1] for p in pattern])
        boff = np.ascontiguousarray([o.offset(sb) for o in lhs_terms for sb in o.sblocks], dtype=np.int64)
        sizes = host_i32(self.block_dims)
        n_red = int(sizes.sum())
        # right-hand side terms as one (Qf, n_red) device matrix
        rows = []
        for o in rhs_terms:
            if isinstance(o, _HostFunctional):
                rows.append(o.device_vector())
            else:
                v = torch.zeros(n_red, dtype=torch.float64, device='cuda')
                offs = np.concatenate([[0], np.cumsum(self.block_dims)])
                for sb in o.sblocks:
                    j = sb.col_idx[0]
                    v[offs[j]:offs[j + 1]] = o.device_block(sb).reshape(-1)
                rows.append(v)
        rhs = torch.stack(rows).contiguous()
        sysc = L.ReducedSystem()
        sysc.n_sub, sysc.basis_sizes, sysc.Q, sysc.Qf = S, sizes.ctypes.data, Q, Qf
        sysc.n_blocks, sysc.block_i, sysc.block_j, sysc.block_offset = len(pattern), bi.ctypes.data, bj.ctypes.data, boff.ctypes.data
        sysc.lhs_blocks, sysc.rhs = buf.data_ptr(), rhs.data_ptr()
        sysc.solver = {'auto': L.SOLVER_AUTO, 'window': L.SOLVER_WINDOW, 'banded': L.SOLVER_BANDED}[self.solver]
        keep = [bi, bj, boff, sizes, rhs, buf]
        has_est = self.estimator is not None and all('nc_{}'.format(s) in self.operators for s in self.estimator.subdomains)
        if has_est:
            est = self.estimator
            if len(est.subdomains) != S:
                raise NotImplementedError('the batched estimator needs all subdomains on this rank')
            terms = self._estimator_terms()
            if any(self.operators['nc_{}'.format(s)].buffer is not buf for s in est.subdomains):
                raise NotImplementedError('estimator operators must share the reduced operator device buffer')
            tarr = (L.EstimatorTerm * len(terms))(*[L.EstimatorTerm(*t) for t in terms])
            nbh_ptr = host_i32(np.concatenate([[0], np.cumsum([len(self.neighborhoods[s]) for s in range(S)])]))
            nbh_idx = host_i32(np.concatenate([self.neighborhoods[s] for s in range(S)]))
            rf2, rsc = host_f64(est.local_eta_rf_squared), host_f64(est.r_scale())
            lam = list(self.operator.coefficients)
            tbar = host_f64([c.evaluate(est.mu_bar) if isinstance(c, ParameterFunctional) else float(c) for c in lam])
            that = host_f64([c.evaluate(est.mu_hat) if isinstance(c, ParameterFunctional) else float(c) for c in lam])
            sysc.nbh_ptr, sysc.nbh_idx = nbh_ptr.ctypes.data, nbh_idx.ctypes.data
            sysc.n_terms, sysc.terms, sysc.est_matrices = len(terms), C.cast(tarr, C.c_void_p), buf.data_ptr()
            sysc.rf_squared, sysc.r_scale = rf2.ctypes.data, rsc.ctypes.data
            sysc.theta_bar, sysc.theta_hat = tbar.ctypes.data, that.ctypes.data
            sysc.alpha_returns_first = 1 if est.alpha_returns_first else 0
            keep += [tarr, nbh_ptr, nbh_idx, rf2, rsc, tbar, that]
        p = C.c_void_p()
        h.check(h.lib.lrbms_online_plan_create(h.h, C.byref(sysc), C.byref(p)))
        self._plan = _lib.Plan(h, p, keep)
        self._plan_has_estimator = has_est
        self._Q, self._Qf = Q, Qf
        return self._plan

    @property
    def online_plan(self):
        if self._plan is None:
            self._build_plan()
        return self._plan

    def set_solver(self, solver):
        """Select the solve kernel of the online plan ('auto', 'window', 'banded'); drops a built plan."""
        if solver != self.solver:
            self.solver, self._plan, self._work = solver, None, {}
        return self

    @property
    def solve_kernel_name(self):
        """Name of the solve kernel the plan selected (from the library, not from configuration)."""
        return _lib.SOLVER_NAMES[int(self.online_plan.info(6))]

    @property
    def solve_flops_executed(self):
        """Factorisation flops per parameter the selected kernel executes."""
        return self.online_plan.info(7)

    @property
    def half_bandwidth(self):
        return int(self.online_plan.info(8))

    def _workspace(self, n_mu):
        torch = _torch()
        plan = self.online_plan
        need = C.c_size_t()
        plan.handle.check(plan.handle.lib.lrbms_online_workspace_bytes(plan.p, int(n_mu), C.byref(need)))
        w = self._work.get('ws')
        if w is None or w.numel() < need.value:
            w = torch.empty(max(256, need.value), dtype=torch.uint8, device='cuda')
            self._work['ws'] = w
        return w, need.value

    # -- device-level entry points (bench and multi-GPU use these; inputs / outputs are device tensors) -----
    def solve_device(self, theta, u=None, info=None):
        torch = _torch()
        plan = self.online_plan
        n_mu = theta.shape[0]
        if u is None:
            u = torch.empty((n_mu, self.n_red), dtype=torch.float64, device='cuda')
        if info is None:
            info = torch.empty(n_mu, dtype=torch.int32, device='cuda')
        w, nbytes = self._workspace(n_mu)
        plan.handle.check(plan.handle.lib.lrbms_online_solve(plan.p, n_mu, ptr(theta), ptr(u), ptr(info), ptr(w), nbytes,
                                                             current_stream_ptr()))
        return u, info

    def estimate_device(self, theta, u, eta=None, parts=None, indicators=None):
        torch = _torch()
        plan = self.online_plan
        if not self._plan_has_estimator:
            raise LrbmsError('this reduced model has no estimator operators')
        n_mu = theta.shape[0]
        if eta is None:
            eta = torch.empty(n_mu, dtype=torch.float64, device='cuda')
        w, nbytes = self._workspace(n_mu)
        plan.handle.check(plan.handle.lib.lrbms_online_estimate(plan.p, n_mu, ptr(theta), ptr(u), ptr(eta), ptr(parts),
                                                                ptr(indicators), ptr(w), nbytes, current_stream_ptr()))
        return eta

    def sweep_device(self, theta, u=None, eta=None, parts=None, indicators=None, info=None):
        """solve + estimate for a device-resident ``(n_mu, Q + Qf)`` coefficient matrix; everything stays in HBM."""
        torch = _torch()
        plan = self.online_plan
        if not self._plan_has_estimator:
            raise LrbmsError('this reduced model has no estimator operators')
        n_mu = theta.shape[0]
        if u is None:
            u = torch.empty((n_mu, self.n_red), dtype=torch.float64, device='cuda')
        if eta is None:
            eta = torch.empty(n_mu, dtype=torch.float64, device='cuda')
        if info is None:
            info = torch.empty(n_mu, dtype=torch.int32, device='cuda')
        w, nbytes = self._workspace(n_mu)
        plan.handle.check(plan.handle.lib.lrbms_online_sweep(plan.p, n_mu, ptr(theta), ptr(u), ptr(eta), ptr(parts),
                                                             ptr(indicators), ptr(info), ptr(w), nbytes, current_stream_ptr()))
        return u, eta, info

    def eta_max_device(self, eta):
        torch = _torch()
        h = Handle.get()
        mx = torch.empty(1, dtype=torch.float64, device='cuda')
        am = torch.empty(1, dtype=torch.int64, device='cuda')
        h.check(h.lib.lrbms_eta_max(h.h, eta.numel(), ptr(eta), ptr(mx), ptr(am), current_stream_ptr()))
        return mx, am

    # -- pyMOR-facing API -----------------------------------------------------------------------------------
    def _check_info(self, info):
        bad = info.nonzero()
        if bad.numel():
            k = int(bad[0].item())
            raise LrbmsError('reduced operator is not positive definite for parameter #{} (pivot {})'.format(k, int(info[k].item())))

    def solve_batch(self, mus):
        torch = _torch()
        theta = torch.from_numpy(self.thetas(mus)).cuda()
        u, info = self.solve_device(theta)
        self._check_info(info)
        return ReducedVectorArray(u, self.block_dims)

    def solve(self, mu=None):
        """``rd.solve(mu)`` -> reduced solution array of length 1."""
        return self.solve_batch(None if mu is None and not self.parameter_type else [self.parse_parameter(mu)])

    def estimate_batch(self, U, mus, decompose=False):
        """``eta`` per parameter: ``U[k]`` is the reduced solution for ``mus[k]``.  With ``decompose`` also the three
        ``(S, n_mu)`` arrays ``(nc, r, df)`` and the ``(S, n_mu)`` local indicators (reference ``estimators.py:104-110``)."""
        torch = _torch()
        theta = torch.from_numpy(self.thetas(mus)).cuda()
        u = U.device_tensor if isinstance(U, ReducedVectorArray) else torch.from_numpy(np.ascontiguousarray(U.data)).cuda()
        n_mu, S = theta.shape[0], len(self.block_dims)
        if u.shape[0] != n_mu:
            raise ValueError('need one reduced solution per parameter ({} vs {})'.format(u.shape[0], n_mu))
        parts = torch.empty((3, S, n_mu), dtype=torch.float64, device='cuda') if decompose else None
        ind = torch.empty((S, n_mu), dtype=torch.float64, device='cuda') if decompose else None
        eta = self.estimate_device(theta, u.contiguous(), parts=parts, indicators=ind)
        if decompose:
            p = parts.cpu().numpy()
            return eta.cpu().numpy(), (p[0], p[1], p[2]), ind.cpu().numpy()
        return eta.cpu().numpy()

    def _estimate_with(self, estimator, U, mu, decompose):
        if estimator is not self.estimator:
            return self.with_(estimator=estimator)._estimate_with(estimator, U, mu, decompose)
        n = len(U)
        mus = [mu] * n
        res = self.estimate_batch(U, mus, decompose=decompose)
        if decompose:
            eta, parts, ind = res
            return (float(eta[0]) if n == 1 else eta), parts, ind
        return float(res[0]) if n == 1 else res

    def estimate(self, U, mu=None, decompose=False):
        """``rd.estimate(U, mu=mu, decompose=False)`` (reference ``online_enrichment.py:61,74``)."""
        return self.estimator.estimate(U, self.parse_parameter(mu), self, decompose=decompose)

    def sweep_into(self, mus, u_host, eta_host):
        """End-to-end batched sweep with caller-provided (ideally pinned) host outputs: host parameters -> coefficient
        matrix -> H2D -> solve + estimate -> D2H of all reduced solutions ``(n_mu, n_red)`` and ``eta`` ``(n_mu,)``.
        Returns the number of parameters flagged as not positive definite (0 = all fine)."""
        torch = _torch()
        th = self.thetas(mus)
        n_mu = th.shape[0]
        bufs = self._work.get('e2e')
        if bufs is None or bufs[0].shape[0] != n_mu:
            bufs = (torch.empty(th.shape, dtype=torch.float64).pin_memory(),
                    torch.empty(th.shape, dtype=torch.float64, device='cuda'),
                    torch.empty((n_mu, self.n_red), dtype=torch.float64, device='cuda'),
                    torch.empty(n_mu, dtype=torch.float64, device='cuda'),
                    torch.empty(n_mu, dtype=torch.int32, device='cuda'))
            self._work['e2e'] = bufs
        th_pin, th_dev, u, eta, info = bufs
        th_pin.copy_(torch.from_numpy(th))
        th_dev.copy_(th_pin, non_blocking=True)
        # The batch goes through in (up to) four chunks so that the device->host copy of one chunk's solutions overlaps
        # the kernels of the next; chunks are multiples of the persistent solve grid (one parameter per CTA and round).
        grid = max(1, self.online_plan.handle.sm_count)
        chunk = n_mu
        if n_mu >= 32 * grid:
            chunk = ((n_mu + 3) // 4 + grid - 1) // grid * grid
        copy_stream = self._work.get('copy_stream')
        if copy_stream is None:
            copy_stream = self._work['copy_stream'] = torch.cuda.Stream()
        main = torch.cuda.current_stream()
        for lo in range(0, n_mu, chunk):
            hi = min(n_mu, lo + chunk)
            self.sweep_device(th_dev[lo:hi], u[lo:hi], eta[lo:hi], info=info[lo:hi])
            ev = torch.cuda.Event()
            ev.record(main)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev)
                u_host[lo:hi].copy_(u[lo:hi], non_blocking=True)
                eta_host[lo:hi].copy_(eta[lo:hi], non_blocking=True)
        bad = int((info != 0).sum().item())          # synchronises the compute stream
        copy_stream.synchronize()                    # ... and the copies
        main.wait_stream(copy_stream)
        return bad

    def sweep_eta_into(self, mus, eta_host, chunk=None):
        """End-to-end sweep for callers that want the estimator only (parameter-space searches, greedy training: the
        maximiser is then solved once more on its own): host parameters -> H2D -> solve + estimate chunk by chunk ->
        D2H of ``eta`` ``(n_mu,)``.  The reduced solutions stay in one chunk-sized device buffer and never cross PCIe
        (8 n_red bytes per parameter in ``sweep_into`` -- 102 MB per 10 000 parameters at n_red = 1 280).
        Returns ``(bad, eta_max, argmax)``: the number of parameters flagged as not positive definite, the largest
        ``eta`` and its index."""
        torch = _torch()
        th = self.thetas(mus)
        n_mu = th.shape[0]
        grid = max(1, self.online_plan.handle.sm_count)
        if chunk is None:
            chunk = min(n_mu, 128 * grid)
        key = ('eta_only', n_mu, chunk)
        bufs = self._work.get(key)
        if bufs is None:
            bufs = (torch.empty(th.shape, dtype=torch.float64).pin_memory(),
                    torch.empty(th.shape, dtype=torch.float64, device='cuda'),
                    torch.empty((chunk, self.n_red), dtype=torch.float64, device='cuda'),
                    torch.empty(n_mu, dtype=torch.float64, device='cuda'),
                    torch.empty(n_mu, dtype=torch.int32, device='cuda'))
            self._work = {k: v for k, v in self._work.items() if not (isinstance(k, tuple) and k[0] == 'eta_only')}
            self._work[key] = bufs
        th_pin, th_dev, u, eta, info = bufs
        th_pin.copy_(torch.from_numpy(th))
        th_dev.copy_(th_pin, non_blocking=True)
        for lo in range(0, n_mu, chunk):
            hi = min(n_mu, lo + chunk)
            self.sweep_device(th_dev[lo:hi], u[:hi - lo], eta[lo:hi], info=info[lo:hi])
        mx, am = self.eta_max_device(eta)
        eta_host.copy_(eta, non_blocking=True)
        bad = int((info != 0).sum().item())          # synchronises the stream (the copy of eta is ordered before it)
        return bad, float(mx.item()), int(am.item())

    def sweep_sharded(self, mus):
        """Multi-GPU online sweep (SURVEY.md section 8e): every rank solves + estimates its slice of ``mus`` and the ranks
        exchange only the estimator maximum.  Returns ``(U_local, eta_local, (lo, hi), eta_max, argmax)`` with ``argmax``
        the index into the *global* batch."""
        from .distributed import gather_estimator_max, mu_slice, rank_and_world
        torch = _torch()
        mus = np.asarray(mus, dtype=np.float64)
        rank, world = rank_and_world()
        lo, hi = mu_slice(len(mus), rank, world)
        theta = torch.from_numpy(self.thetas(mus[lo:hi])).cuda()
        u, eta, info = self.sweep_device(theta)
        self._check_info(info)
        mx, am = self.eta_max_device(eta)
        eta_max, argmax = gather_estimator_max(mx, am, lo)
        return ReducedVectorArray(u, self.block_dims), eta, (lo, hi), eta_max, argmax

    def sweep(self, mus, decompose=False):
        """Solve and estimate a parameter batch in one call: ``(U, eta)`` or ``(U, eta, (nc, r, df), indicators)``."""
        torch = _torch()
        theta = torch.from_numpy(self.thetas(mus)).cuda()
        n_mu, S = theta.shape[0], len(self.block_dims)
        parts = torch.empty((3, S, n_mu), dtype=torch.float64, device='cuda') if decompose else None
        ind = torch.empty((S, n_mu), dtype=torch.float64, device='cuda') if decompose else None
        u, eta, info = self.sweep_device(theta, parts=parts, indicators=ind)
        self._check_info(info)
        U = ReducedVectorArray(u, self.block_dims)
        if decompose:
            p = parts.cpu().numpy()
            return U, eta.cpu().numpy(), (p[0], p[1], p[2]), ind.cpu().numpy()
        return U, eta.cpu().numpy()
