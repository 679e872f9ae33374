"""CPU tests of ``oracle/exact_forms.py``, the exactly rounded reference of the estimator forms.

The evaluator is held to ``fractions.Fraction`` (exact rational arithmetic on the same double inputs) on small random
term lists, with constructed cancellation down to 1e-12 of the summed magnitude; the oracle's own estimator is held to the
evaluator on the committed golden case, which pins the arbiter to the reference's formulas (``estimators.py:71-91``).
"""
import os
import sys
from fractions import Fraction

import numpy as np
import pytest

from oracle import exact_forms as X

HERE = os.path.dirname(os.path.abspath(__file__))
U = 2.0 ** -53


def gamma(k):
    return k * U / (1.0 - k * U)


def _exact_parts(forms, theta, u):
    """Parts of an ``EstimatorForms`` in rational arithmetic: ``(4, S, n_mu)`` Fractions (nc, r_pre, r, df)."""
    n_mu = u.shape[0]
    off = forms.offsets
    out = [[[Fraction(0)] * n_mu for _ in range(forms.n_sub)] for _ in range(4)]
    for m in range(n_mu):
        uf = [Fraction(float(x)) for x in u[m]]
        th = [Fraction(float(x)) for x in theta[m]]

        def vec(kind, sub):
            if kind == X.VEC_ONE:
                return [Fraction(1)]
            if kind == X.VEC_UI:
                return uf[off[sub]:off[sub + 1]]
            if kind == X.VEC_UN:
                return [v for k in forms.nbh[sub] for v in uf[off[k]:off[k + 1]]]
            return [th[q] * v for k in forms.nbh[sub] for q in range(forms.Q) for v in uf[off[k]:off[k + 1]]]
        for (part, sub, left, right, factors, M) in forms.forms:
            x, y = vec(left, sub), vec(right, sub)
            c = Fraction(1)
            for kind, val in factors:
                c *= th[val] if kind == 'theta' else Fraction(float(val))
            tot = Fraction(0)
            for r in range(M.shape[0]):
                if x[r] == 0:
                    continue
                tot += x[r] * sum((Fraction(float(M[r, k])) * y[k] for k in range(M.shape[1])), Fraction(0))
            idx = {X.OUT_NC: 0, X.OUT_R: 1, X.OUT_DF: 3}[part]
            out[idx][sub][m] += c * tot
        for s in range(forms.n_sub):
            out[1][s][m] += Fraction(float(forms.rf2[s]))
            out[2][s][m] = out[1][s][m] * Fraction(float(forms.r_scale[s]))
    return out


def _random_case(rng, sizes, nbh, Q, n_mu, spread=2.0):
    """Random C-ABI term list over the reference's term shapes (estimators.py:71-91), plus a few extra shapes."""
    S = len(sizes)
    dsub = [sum(sizes[k] for k in nbh[i]) for i in range(S)]
    dim = {X.VEC_ONE: lambda i: 1, X.VEC_UI: lambda i: sizes[i], X.VEC_UN: lambda i: dsub[i], X.VEC_UR: lambda i: Q * dsub[i]}
    spec = [(X.OUT_NC, X.VEC_UN, X.VEC_UN, -1, -1, 1.0), (X.OUT_R, X.VEC_ONE, X.VEC_UR, -1, -1, -2.0),
            (X.OUT_R, X.VEC_UR, X.VEC_UR, -1, -1, 1.0), (X.OUT_DF, X.VEC_UR, X.VEC_UR, -1, -1, 1.0),
            (X.OUT_NC, X.VEC_UI, X.VEC_UN, Q - 1, -1, 0.75)]
    spec += [(X.OUT_DF, X.VEC_UI, X.VEC_UI, a, b, 1.0) for a in range(Q) for b in range(Q)]
    spec += [(X.OUT_DF, X.VEC_UI, X.VEC_UR, a, -1, 2.0) for a in range(Q)]
    terms = []
    for i in range(S):
        for (out, lk, rk, qa, qb, coef) in spec:
            M = rng.standard_normal((dim[lk](i), dim[rk](i))) * np.exp(rng.uniform(-3, 3))
            terms.append((i, out, lk, rk, qa, qb, coef, M))
    theta = 10.0 ** rng.uniform(-spread / 2, spread / 2, (n_mu, Q + 1))
    u = rng.standard_normal((n_mu, sum(sizes)))
    rf2, rsc = rng.uniform(0.5, 1.5, S), rng.uniform(0.1, 0.3, S)
    return terms, theta, u, rf2, rsc


def _cancel(forms, terms, theta, u, levels):
    """Adjust the first entry of the last term of each part so that the part of subdomain 0, parameter 0 comes to
    ``level * S``: constructed cancellation."""
    for part, level in levels.items():
        idx = [k for k, t in enumerate(terms) if t[0] == 0 and t[1] == part]
        k = idx[-1]
        ex = _exact_parts(forms, theta[:1], u[:1])
        val = {X.OUT_NC: ex[0], X.OUT_R: ex[1], X.OUT_DF: ex[3]}[part][0][0]
        S = {X.OUT_NC: 'S_nc', X.OUT_R: 'S_r_pre', X.OUT_DF: 'S_df'}[part]
        s = forms.evaluate(theta[:1], u[:1])[S][0, 0]
        sub, out, lk, rk, qa, qb, coef, M = terms[k]
        xv = forms._vector(lk, sub, theta[:1], u[:1])
        yv = forms._vector(rk, sub, theta[:1], u[:1])
        c = Fraction(coef) * (Fraction(theta[0, qa]) if qa >= 0 else 1) * (Fraction(theta[0, qb]) if qb >= 0 else 1)
        x0 = Fraction(xv[0][0, 0]) + Fraction(xv[1][0, 0])
        y0 = Fraction(yv[0][0, 0]) + Fraction(yv[1][0, 0])
        M = M.copy()
        M[0, 0] = float(Fraction(M[0, 0]) - (val - Fraction(level * s)) / (c * x0 * y0))
        terms[k] = (sub, out, lk, rk, qa, qb, coef, M)
        forms = X.terms_from_cabi(terms, forms.sizes, forms.nbh, forms.Q, forms.rf2, forms.r_scale)
    return forms, terms


@pytest.mark.parametrize('sizes,nbh,Q,cancel', [
    ([3, 5], [[0, 1], [0, 1]], 1, {}),
    ([2, 7, 4], [[0, 1], [0, 1, 2], [1, 2]], 2, {X.OUT_NC: 1e-12, X.OUT_R: 1e-9, X.OUT_DF: 1e-12}),
    ([5, 1, 3], [[0, 2], [1], [0, 1, 2]], 3, {X.OUT_NC: 1e-6, X.OUT_R: 1e-12, X.OUT_DF: 1e-10}),
    ([4], [[0]], 1, {X.OUT_R: 1e-12}),
])
def test_exact_forms_against_fractions(sizes, nbh, Q, cancel):
    rng = np.random.default_rng(len(sizes) * 10 + Q)
    n_mu = 3
    terms, theta, u, rf2, rsc = _random_case(rng, sizes, nbh, Q, n_mu)
    forms = X.terms_from_cabi(terms, sizes, nbh, Q, rf2, rsc)
    if cancel:
        forms, terms = _cancel(forms, terms, theta, u, cancel)
    got = forms.evaluate(theta, u)
    ex = _exact_parts(forms, theta, u)
    worst = 0.0
    for k, name in enumerate(('nc', 'r_pre', 'r', 'df')):
        for s in range(len(sizes)):
            for m in range(n_mu):
                e = ex[k][s][m]
                g = got[name][s, m]
                err = abs(Fraction(g) - e)
                assert err <= U * abs(e) + Fraction(got['E_' + name][s, m]), (name, s, m)
                assert g == float(e), '{} sub {} mu {}: {!r} is not the exact value rounded once ({!r})'.format(
                    name, s, m, g, float(e))
                assert got['S_' + name][s, m] >= abs(float(e)) * (1 - 1e-12)
                worst = max(worst, float(err / (U * abs(e))) if e else 0.0)
    # the constructed cancellation reached the requested depth
    for part, level in cancel.items():
        name, k = {X.OUT_NC: ('nc', 0), X.OUT_R: ('r_pre', 1), X.OUT_DF: ('df', 3)}[part]
        ratio = abs(float(ex[k][0][0])) / got['S_' + name][0, 0]
        assert 0.3 * level <= ratio <= 3 * level, (name, ratio)
    print('worst |got - exact| / (u |exact|):', worst)


def test_two_prod_and_split_are_exact():
    rng = np.random.default_rng(3)
    a = rng.standard_normal(2000) * 10.0 ** rng.uniform(-30, 30, 2000)
    b = rng.standard_normal(2000) * 10.0 ** rng.uniform(-30, 30, 2000)
    p, e = X.two_prod(a, b)
    h, l = X.split(a)
    for k in range(0, 2000, 7):
        assert Fraction(p[k]) + Fraction(e[k]) == Fraction(a[k]) * Fraction(b[k])
        assert Fraction(h[k]) + Fraction(l[k]) == Fraction(a[k])
    s, t = X.two_sum(a, b)
    for k in range(0, 2000, 7):
        assert Fraction(s[k]) + Fraction(t[k]) == Fraction(a[k]) + Fraction(b[k])


def _golden_oracle():
    sys.path.insert(0, os.path.join(HERE, 'golden'))
    import make_golden
    from oracle import lrbms_oracle as O
    name = 'os2015_2x2_N5'
    gold = np.load(os.path.join(HERE, 'golden', name + '.npz'))
    data, bases = make_golden.build_case(name)
    S = data.num_subdomains
    red = O.LRBMSReductor(O.build_discretization(data), bases={'domain_%d' % i: bases[i] for i in range(S)})
    return gold, red, red.reduce()


def test_oracle_estimate_within_rounding_bound_of_exact_on_golden():
    """The oracle's ``estimate`` (the reference's line-by-line restatement) on the golden case: each part lies within
    ``gamma_K S`` of the exact value of its inputs, K = 2 Q n_red + 16 (numpy's dense products over the unblocked operators,
    any summation order; the flux reconstruction is one rounding per entry; the additions and the scale).  The front-end
    over ``reduced_blocks`` and a restatement over the golden's unblocked matrices give the same exact values."""
    gold, red, rd = _golden_oracle()
    d = red.d
    est = d.estimator
    mus = gold['mus']
    forms = X.terms_from_oracle(red)
    Q, n_red = forms.Q, int(sum(forms.sizes))
    theta = X.flux_thetas(est.lambda_coeffs, [d.parse_parameter(m) for m in mus])
    U_or = np.array([rd.solve(m).data[0] for m in mus])
    assert np.abs(U_or - gold['U']).max() <= 1e-12 * np.abs(gold['U']).max()
    ex = forms.evaluate(theta, U_or, factor_args=[d.parse_parameter(m) for m in mus])
    K = 2 * Q * n_red + 16
    worst = {}
    for k, mu in enumerate(mus):
        _, parts, _ = rd.estimate(rd.solve(mu), mu, decompose=True)
        for name, p in zip(('nc', 'r', 'df'), parts):
            got = np.asarray(p)[:, 0]
            err = np.abs(got - ex[name][:, k])
            assert np.all(err <= gamma(K) * ex['S_' + name][:, k]), (name, mu, err, ex['S_' + name][:, k])
            worst[name] = max(worst.get(name, 0.0), float((err / (2 * U * ex['S_' + name][:, k])).max()))
        # the frozen golden parts are the same evaluation
        assert np.abs(gold['parts'][k] - np.stack([np.asarray(p)[:, 0] for p in parts])).max() <= \
            1e-12 * np.abs(gold['parts'][k]).max()
    print('oracle |got - exact| / (eps S) per part:', worst)
    # the same forms restated over the golden's unblocked matrices (every subdomain's neighbourhood = the whole system)
    S = len(forms.sizes)
    allnb = [list(range(S))] * S
    fl = []
    for i in range(S):
        g = lambda key: gold['red__{}_{}__{}'.format(key, i, 0)]
        fl += [(X.OUT_NC, i, X.VEC_UN, X.VEC_UN, [], g('nc')), (X.OUT_R, i, X.VEC_ONE, X.VEC_UR, [('const', -2.0)], g('r_fd')),
               (X.OUT_R, i, X.VEC_UR, X.VEC_UR, [], g('r_dd')), (X.OUT_DF, i, X.VEC_UR, X.VEC_UR, [], g('df_bb'))]
        fl += [(X.OUT_DF, i, X.VEC_UI, X.VEC_UN, [('theta', a), ('theta', b)],
                gold['red__df_aa_{}__{}'.format(i, a * Q + b)][_rows_of_idx(forms, i)]) for a in range(Q) for b in range(Q)]
        fl += [(X.OUT_DF, i, X.VEC_UI, X.VEC_UR, [('const', 2.0), ('theta', a)], gold['red__df_ab_{}__{}'.format(i, a)][_rows_of_idx(forms, i)])
               for a in range(Q)]
    ex2 = X.EstimatorForms(fl, forms.sizes, allnb, Q, forms.rf2, forms.r_scale).evaluate(theta, U_or)
    for name in ('nc', 'r', 'df'):
        assert np.all(np.abs(ex2[name] - ex[name]) <= 1e-13 * ex['S_' + name]), name


def _rows_of_idx(forms, i):
    return slice(int(forms.offsets[i]), int(forms.offsets[i + 1]))

