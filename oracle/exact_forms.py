"""Nearly exactly rounded evaluation of the estimator forms ``nc``, ``r``, ``df`` (reference ``estimators.py:71-91``).

TEST INFRASTRUCTURE, like everything under ``oracle/``: the arbiter the GPU estimator and the oracle are both held to.

Every estimator part of subdomain ``i`` is a sum of bilinear forms ``c * x^T M y``: ``x`` and ``y`` are slices of the
reduced solution ``u`` or the reconstructed flux coefficients ``U_r = [theta_q u_k]_(k in N(i), q)``, ``c`` is a constant
or a product of affine coefficients ``theta_a theta_b``.  Two plain FP64 evaluations of such a sum may differ by about
``eps * S`` where ``S`` is the same sum over absolute values; with the forms of the estimator ``S`` exceeds the value by
up to ~3e7, so neither of them is a reference for the other.  This module evaluates each part of the given double
inputs in double-double arithmetic (error-free transforms in vectorised NumPy) and rounds once at the end:

* ``theta_q u_k``, the products of the coefficient factors and every ``M_rc y_c`` are split exactly into two doubles
  (``two_prod``: Veltkamp splitting, NumPy has no fma);
* ``w = M y`` is accumulated per row as an unevaluated double-double (Dot2 of Ogita, Rump and Oishi, SIAM J. Sci. Comput.
  26 (2005), without the final rounding), ``x^T w`` likewise, then the forms of one part are summed in double-double, and
  for ``r`` the constant ``||f||^2`` is added and the scale ``r_scale`` applied in double-double.

Error bound.  With ``u = 2^-53``, ``R`` and ``C`` the largest row / column count of a form of the part and ``n_f`` the
number of its forms, the double-double value ``v`` of a part satisfies

    |v - exact| <= E,      E = 4 ((R + 2)^2 + (C + 2)^2 + n_f + 8) u^2 S,

and the returned double ``fl(v)`` therefore lies within ``u |exact| + E`` of the exact value of the inputs.  For the
shapes of this project (``R, C <= 2 * 7 * 40 = 560``) ``E`` is at most ``3e-26 S``: below ``3e-17 |value|`` where
``S / |value| <= 1e9``, and below ``1e-18 |value|`` at the cancellation of about 3e7 seen at C2.  The result is
the exact value rounded once, except when the exact value lies within ``E`` of a rounding boundary, where it is the
neighbouring double (faithful).  ``numpy.longdouble`` would leave ``u_x87 * S = 5e-20 * 3e7 |value|``, three digits of
margin only, and does not exist on every platform.  ``tests/test_exact_forms.py`` holds the bound against ``fractions``.

Three front-ends build the term list:
(i)   ``terms_from_cabi``: the ``(subdomain, out_kind, left, right, qa, qb, coef, M)`` tuples of the C ABI's estimator terms;
(ii)  ``terms_from_model``: a :class:`pylrbms_b200.reduced.ReducedModel`, read through its public block access and restated
      from the reference's term list (``estimators.py:71-91``), independent of ``ReducedModel._estimator_terms``;
(iii) ``terms_from_oracle``: the oracle's reduced model through ``oracle.lrbms_oracle.reduced_blocks`` (no unblocked storage).
Each returns an :class:`EstimatorForms`; ``EstimatorForms.evaluate(theta_or_mus, u)`` returns the parts.
"""
from __future__ import annotations

import numpy as np

U = 2.0 ** -53                     # unit roundoff of IEEE double
EPS = 2.0 ** -52
_SPLIT = 134217729.0               # 2^27 + 1 (Veltkamp)

OUT_NC, OUT_R, OUT_DF = 0, 1, 2
VEC_ONE, VEC_UI, VEC_UN, VEC_UR = 0, 1, 2, 3       # lrbms_sm100.h LRBMS_VEC_*


# ------------------------------------------------------------------------------------------------------------
#  error-free transforms (element-wise on arrays)
# ------------------------------------------------------------------------------------------------------------

def two_sum(a, b):
    s = a + b
    z = s - a
    return s, (a - (s - z)) + (b - z)


def split(a):
    c = _SPLIT * a
    hi = c - (c - a)
    return hi, a - hi


def two_prod(a, b, a_split=None, b_split=None):
    p = a * b
    ah, al = split(a) if a_split is None else a_split
    bh, bl = split(b) if b_split is None else b_split
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def dd_mul(vh, vl, c):
    """(vh + vl) * c for a double c, renormalised."""
    p, e = two_prod(vh, c)
    e = e + vl * c
    s = p + e
    return s, e - (s - p)


def dd_add(ah, al, bh, bl):
    s, e = two_sum(ah, bh)
    e = e + (al + bl)
    h = s + e
    return h, e - (h - s)


# ------------------------------------------------------------------------------------------------------------
#  one stack of equally shaped forms
# ------------------------------------------------------------------------------------------------------------

def dd_forms(M, xh, xl, yh, yl):
    """``x^T M y`` for a stack of forms: ``M (F, R, C)``, ``x (F, R, n)``, ``y (F, C, n)`` as double-double pairs.
    Returns ``(vh, vl) (F, n)`` and ``|x|^T |M| |y|``."""
    F, R, C = M.shape
    n = yh.shape[2]
    Ms = split(M)
    ys = split(yh)
    wh = np.zeros((F, R, n))
    wc = np.zeros((F, R, n))
    for c in range(C):
        a = M[:, :, c, None]
        b = yh[:, None, c, :]
        p, e = two_prod(a, b, (Ms[0][:, :, c, None], Ms[1][:, :, c, None]), (ys[0][:, None, c, :], ys[1][:, None, c, :]))
        wh, q = two_sum(wh, p)
        wc += q + e + a * yl[:, None, c, :]
    wl = wc                                   # w = wh + wl (unevaluated)
    vh = np.zeros((F, n))
    vc = np.zeros((F, n))
    xs = split(xh)
    ws = split(wh)
    for r in range(R):
        p, e = two_prod(xh[:, r], wh[:, r], (xs[0][:, r], xs[1][:, r]), (ws[0][:, r], ws[1][:, r]))
        vh, q = two_sum(vh, p)
        vc += q + e + (xh[:, r] * wl[:, r] + xl[:, r] * wh[:, r])
    h = vh + vc
    scale = np.einsum('frn,frc,fcn->fn', np.abs(xh), np.abs(M), np.abs(yh))
    return (h, vc - (h - vh)), scale


# ------------------------------------------------------------------------------------------------------------
#  term lists
# ------------------------------------------------------------------------------------------------------------

class EstimatorForms:
    """The estimator of one reduced model as a list of forms.

    ``forms``: ``(part, sub, left, right, factors, M)`` with ``left / right`` in ``VEC_*`` and ``factors`` a list of
    ``('theta', q)`` / ``('const', value)`` / ``('fn', callable(mus) -> (n_mu,) array)``; ``sizes`` the basis size per
    subdomain; ``nbh[i]`` the neighbourhood of ``i`` in the order the ``M`` of ``i`` use; ``Q`` the number of flux
    coefficients; ``rf2`` and ``r_scale`` per subdomain."""

    def __init__(self, forms, sizes, nbh, Q, rf2, r_scale):
        self.forms, self.sizes, self.nbh, self.Q = forms, [int(s) for s in sizes], [list(x) for x in nbh], int(Q)
        self.rf2, self.r_scale = np.asarray(rf2, dtype=np.float64), np.asarray(r_scale, dtype=np.float64)
        self.offsets = np.concatenate([[0], np.cumsum(self.sizes)]).astype(np.int64)

    @property
    def n_sub(self):
        return len(self.sizes)

    def _vector(self, kind, sub, theta, u):
        """``(hi, lo)`` of shape ``(len, n_mu)``; theta ``(n_mu, >= Q)``, u ``(n_mu, n_red)``."""
        off = self.offsets
        n = u.shape[0]
        if kind == VEC_ONE:
            return np.ones((1, n)), np.zeros((1, n))
        if kind == VEC_UI:
            x = u[:, off[sub]:off[sub + 1]].T
            return np.ascontiguousarray(x), np.zeros_like(x)
        if kind == VEC_UN:
            x = np.concatenate([u[:, off[k]:off[k + 1]] for k in self.nbh[sub]], axis=1).T
            return np.ascontiguousarray(x), np.zeros_like(x)
        hs, ls = [], []
        for k in self.nbh[sub]:
            for q in range(self.Q):
                h, l = two_prod(theta[:, q][None, :], u[:, off[k]:off[k + 1]].T)
                hs.append(h); ls.append(l)
        return np.concatenate(hs, axis=0), np.concatenate(ls, axis=0)

    def evaluate(self, theta, u, subdomains=None, factor_args=None, chunk_elems=4_000_000):
        """Parts of the estimator for ``theta (n_mu, >= Q)`` (the flux coefficients ``theta_q`` first) and the reduced
        solutions ``u (n_mu, n_red)``.  ``factor_args`` is passed to ``('fn', f)`` factors (e.g. the parameters).

        Returns a dict of ``(n_sel, n_mu)`` arrays over ``subdomains`` (default: all): ``nc, r_pre, r, df`` (each the exact
        value rounded once, ``r_pre = ||f||^2 - 2 r_fd + r_dd`` before the scale), their sums over absolute values
        ``S_nc, S_r_pre, S_r, S_df`` and the error bound ``E_*`` of the module docstring for each."""
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        u = np.ascontiguousarray(u, dtype=np.float64)
        n_mu = u.shape[0]
        subs = list(range(self.n_sub)) if subdomains is None else [int(s) for s in subdomains]
        where = {s: k for k, s in enumerate(subs)}
        ns = len(subs)
        acc_h, acc_l, S = np.zeros((3, ns, n_mu)), np.zeros((3, ns, n_mu)), np.zeros((3, ns, n_mu))
        shape_max = np.zeros((3, ns, 2), dtype=np.int64)
        n_forms = np.zeros((3, ns), dtype=np.int64)
        # group by shape so that equally shaped forms are evaluated as one stack
        groups = {}
        for f in self.forms:
            part, sub, left, right, factors, M = f
            if sub in where:
                groups.setdefault(M.shape, []).append(f)
        for shape, fl in groups.items():
            per = max(1, chunk_elems // max(1, shape[0] * max(shape[1], 1) + (shape[0] + shape[1]) * n_mu))
            for lo in range(0, len(fl), per):
                chunk = fl[lo:lo + per]
                Ms = np.stack([f[5] for f in chunk]).astype(np.float64)
                xs = [self._vector(f[2], f[1], theta, u) for f in chunk]
                ys = [self._vector(f[3], f[1], theta, u) for f in chunk]
                (vh, vl), sc = dd_forms(Ms, np.stack([x[0] for x in xs]), np.stack([x[1] for x in xs]),
                                        np.stack([y[0] for y in ys]), np.stack([y[1] for y in ys]))
                for k, (part, sub, left, right, factors, M) in enumerate(chunk):
                    h, l, s = vh[k], vl[k], sc[k]
                    for kind, val in factors:
                        if kind == 'theta':
                            c = theta[:, val]
                        elif kind == 'fn':
                            c = np.asarray(val(factor_args), dtype=np.float64)
                        else:
                            c = np.full(n_mu, float(val))
                        h, l = dd_mul(h, l, c)
                        s = s * np.abs(c)
                    j = where[sub]
                    acc_h[part, j], acc_l[part, j] = dd_add(acc_h[part, j], acc_l[part, j], h, l)
                    S[part, j] += s
                    shape_max[part, j] = np.maximum(shape_max[part, j], M.shape)
                    n_forms[part, j] += 1
        idx = np.array(subs, dtype=np.int64)
        rf2, rsc = self.rf2[idx][:, None], self.r_scale[idx][:, None]
        rh, rl = dd_add(acc_h[1], acc_l[1], np.broadcast_to(rf2, (ns, n_mu)).copy(), np.zeros((ns, n_mu)))
        S_r_pre = S[1] + np.abs(rf2)
        sh, sl = dd_mul(rh, rl, np.broadcast_to(rsc, (ns, n_mu)).copy())
        R, Cc = shape_max[..., 0][..., None], shape_max[..., 1][..., None]
        E = 4.0 * ((R + 2.0) ** 2 + (Cc + 2.0) ** 2 + n_forms[..., None] + 8.0) * U * U * S
        E_r_pre = E[1] + 4.0 * 8 * U * U * S_r_pre
        return dict(nc=acc_h[0] + acc_l[0], df=acc_h[2] + acc_l[2], r_pre=rh + rl, r=sh + sl,
                    S_nc=S[0], S_df=S[2], S_r_pre=S_r_pre, S_r=S_r_pre * np.abs(rsc),
                    E_nc=E[0], E_df=E[2], E_r_pre=E_r_pre, E_r=(E_r_pre + 8 * U * U * S_r_pre) * np.abs(rsc))


# ---- (i) the C ABI's term tuples -----------------------------------------------------------------------------

def terms_from_cabi(terms, sizes, nbh, Q, rf2, r_scale):
    """``terms``: ``(subdomain, out_kind, left, right, qa, qb, coef, M)`` as the C ABI's ``lrbms_estimator_term_t`` list
    (``M`` a host array).  Factors: ``coef``, then ``theta_qa``, then ``theta_qb`` (-1 = none)."""
    forms = []
    for (sub, out_kind, left, right, qa, qb, coef, M) in terms:
        factors = [('const', float(coef))]
        if qa >= 0:
            factors.append(('theta', int(qa)))
        if qb >= 0:
            factors.append(('theta', int(qb)))
        forms.append((int(out_kind), int(sub), int(left), int(right), factors, np.asarray(M, dtype=np.float64)))
    return EstimatorForms(forms, sizes, nbh, Q, rf2, r_scale)


# ---- the reference's term list (estimators.py:71-91) on neighbourhood matrices -----------------------------------

def _functional_factors(c):
    """A coefficient functional as a list of factors, evaluated at the parameters passed to ``evaluate``."""
    factors = getattr(c, 'factors', None)
    if factors is None:
        factors = [c]
    out = []
    for f in factors:
        if hasattr(f, 'evaluate'):
            out.append(('fn', lambda mus, f=f: np.array([f.evaluate(m) for m in mus], dtype=np.float64)))
        else:
            out.append(('const', float(f)))
    return out


def _reference_forms(sub, mats):
    """The reference's six operators of one subdomain as forms:
    ``nc = u_o^T NC u_o`` (u_o = u over the neighbourhood, the reduced Oswald interpolation is the identity);
    ``r = ||f||^2 - 2 r_fd U_r + U_r^T RDD U_r``; ``df = sum_ab theta_a theta_b u_i^T AA_ab u_i + U_r^T BB U_r
    + 2 sum_a theta_a u_i^T AB_a U_r``.  ``mats``: ``nc, r_fd, r_dd, df_bb`` matrices, ``df_aa`` and ``df_ab`` lists of
    ``(coefficient functional, matrix)``."""
    forms = [(OUT_NC, sub, VEC_UN, VEC_UN, [], mats['nc']),
             (OUT_R, sub, VEC_ONE, VEC_UR, [('const', -2.0)], mats['r_fd']),
             (OUT_R, sub, VEC_UR, VEC_UR, [], mats['r_dd'])]
    for c, M in mats['df_aa']:
        forms.append((OUT_DF, sub, VEC_UI, VEC_UI, _functional_factors(c), M))
    forms.append((OUT_DF, sub, VEC_UR, VEC_UR, [], mats['df_bb']))
    for c, M in mats['df_ab']:
        forms.append((OUT_DF, sub, VEC_UI, VEC_UR, [('const', 2.0)] + _functional_factors(c), M))
    return forms


def _assemble(blocks, rows, cols, row_sizes, col_sizes):
    """Dense matrix over ``rows x cols`` subspace positions from ``{(i, j): block}`` (absent blocks are zero)."""
    ro = np.concatenate([[0], np.cumsum(row_sizes)])
    co = np.concatenate([[0], np.cumsum(col_sizes)])
    M = np.zeros((ro[-1], co[-1]))
    for a, i in enumerate(rows):
        for b, j in enumerate(cols):
            B = blocks.get((i, j))
            if B is not None:
                M[ro[a]:ro[a + 1], co[b]:co[b + 1]] = np.asarray(B).reshape(ro[a + 1] - ro[a], co[b + 1] - co[b])
    return M


def _flux_q(est):
    return len(est.flux_reconstruction.coefficients)


# ---- (ii) the CUDA reduced model -----------------------------------------------------------------------------------

def terms_from_model(rd, subdomains=None):
    """The reduced estimator operators of a :class:`pylrbms_b200.reduced.ReducedModel` (device blocks copied to the host
    through ``ReducedBlockOperator.blocks()``).  ``evaluate`` then takes ``theta = rd.thetas(mus)``, ``u`` and
    ``factor_args = mus`` (parsed parameters)."""
    est, ops = rd.estimator, rd.operators
    Q = _flux_q(est)
    N = rd.block_dims
    subs = list(range(len(N))) if subdomains is None else list(subdomains)
    forms = []
    for sub in subs:
        nb = list(rd.neighborhoods[sub])
        NR = [Q * N[k] for k in nb]

        def dense(op, rows, cols, rs, cs):
            return _assemble(op.blocks(), rows, cols, rs, cs)
        rfd_blocks = ops['r_fd_{}'.format(sub)].blocks()
        rfd_rows = {i for (i, j) in rfd_blocks}
        assert len(rfd_rows) == 1, 'r_fd_{}: one row expected'.format(sub)
        mats = dict(nc=dense(ops['nc_{}'.format(sub)], nb, nb, [N[k] for k in nb], [N[k] for k in nb]),
                    r_fd=_assemble(rfd_blocks, list(rfd_rows), nb, [1], NR),
                    r_dd=dense(ops['r_dd_{}'.format(sub)], nb, nb, NR, NR),
                    df_bb=dense(ops['df_bb_{}'.format(sub)], nb, nb, NR, NR),
                    df_aa=[(c, dense(o, [sub], [sub], [N[sub]], [N[sub]]))
                           for c, o in zip(ops['df_aa_{}'.format(sub)].coefficients, ops['df_aa_{}'.format(sub)].operators)],
                    df_ab=[(c, dense(o, [sub], nb, [N[sub]], NR))
                           for c, o in zip(ops['df_ab_{}'.format(sub)].coefficients, ops['df_ab_{}'.format(sub)].operators)])
        forms += _reference_forms(sub, mats)
    nbh = [list(rd.neighborhoods[s]) for s in range(len(N))]
    return EstimatorForms(forms, N, nbh, Q, est.local_eta_rf_squared, est.r_scale())


# ---- (iii) the oracle's reduced model --------------------------------------------------------------------------------

def terms_from_oracle(reductor, subdomains=None):
    """The oracle's reduced estimator operators, block by block through ``oracle.lrbms_oracle.reduced_blocks`` (the
    reductor needs its image bases: ``reductor.image_bases(unblocked=False)`` or ``reductor.reduce()``).  ``evaluate``
    then takes ``theta`` with the flux coefficients ``lambda_q(mu)`` first, the oracle's ``u`` and ``factor_args = mus``."""
    from oracle.lrbms_oracle import reduced_blocks
    from oracle.pymor_like import LincombOperator
    d = reductor.d
    est = d.estimator
    Q = _flux_q(est)
    S = len(d.solution_space.subspaces)
    N = [len(reductor.bases['domain_{}'.format(i)]) for i in range(S)]
    subs = list(range(S)) if subdomains is None else list(subdomains)
    forms = []
    for sub in subs:
        nb = list(d.neighborhoods[sub])
        NR = [Q * N[k] for k in nb]
        rb = lambda name, q=None: reduced_blocks(reductor, '{}_{}'.format(name, sub), q)

        def lincomb(name, rows, cols, rs, cs):
            op = d.operators['{}_{}'.format(name, sub)]
            assert isinstance(op, LincombOperator)
            return [(c, _assemble(rb(name, q), rows, cols, rs, cs)) for q, c in enumerate(op.coefficients)]
        mats = dict(nc=_assemble(rb('nc'), nb, nb, [N[k] for k in nb], [N[k] for k in nb]),
                    r_fd=_assemble(rb('r_fd'), [0], nb, [1], NR),
                    r_dd=_assemble(rb('r_dd'), nb, nb, NR, NR),
                    df_bb=_assemble(rb('df_bb'), nb, nb, NR, NR),
                    df_aa=lincomb('df_aa', [sub], [sub], [N[sub]], [N[sub]]),
                    df_ab=lincomb('df_ab', [sub], nb, [N[sub]], NR))
        forms += _reference_forms(sub, mats)
    r_scale = (1.0 / np.pi ** 2) / np.asarray(est.min_diffusion_evs, dtype=np.float64) * \
        np.asarray(est.subdomain_diameters, dtype=np.float64) ** 2
    return EstimatorForms(forms, N, [list(x) for x in d.neighborhoods], Q, est.local_eta_rf_squared, r_scale)


def flux_thetas(coefficients, mus):
    """``(n_mu, Q)``: the flux coefficients ``lambda_q(mu)`` for ``EstimatorForms.evaluate``."""
    return np.array([[c.evaluate(m) for c in coefficients] for m in mus], dtype=np.float64).reshape(len(mus), len(coefficients))
