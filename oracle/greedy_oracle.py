"""TEST INFRASTRUCTURE ONLY -- CPU oracle, part 3: greedy basis generation and the POD basis extension.

NumPy / SciPy restatements, on top of ``oracle/pymor_like.py`` and ``oracle/lrbms_oracle.py``, of pyMOR's ``pod`` (method of
snapshots), of ``extend_basis(U, method='pod', pod_modes=m)`` with ``pod_orthonormalize=True`` and of the ``greedy`` loop
[ext] with several parameters per extension.  Like ``pymor_like.py`` this layer restates published pyMOR semantics and is
unpinned (pyMOR is not installable here); the fine solves use SciPy ``spsolve`` on the assembled sparse A(mu).  Only
``tests/`` may import this file; the product package never does.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

from .lrbms_oracle import ExtensionError
from .pymor_like import VA


# ----------------------------------------------------------------------------------------------------------
#  POD (pyMOR ``pod``, method of snapshots)
# ----------------------------------------------------------------------------------------------------------

def pod(A, product=None, modes=None, atol=0.0):
    """pyMOR ``pod`` by the method of snapshots: eigendecomposition of the Gram matrix ``A^T P A`` (``numpy.linalg.eigh``),
    singular values ``sqrt(max(lambda, 0))`` in descending order, at most ``modes`` of them with ``sigma > atol``.  Each
    eigenvector is signed so that its entry of largest magnitude is positive (so modes compare without a sign ambiguity).
    Returns ``(POD modes A W / sigma as a VA, sigma)``."""
    X = A.data
    G = X @ (product.matrix @ X.T) if product is not None else X @ X.T
    G = 0.5 * (G + G.T)
    lam, W = np.linalg.eigh(G)
    lam, W = lam[::-1], W[:, ::-1]
    sigma = np.sqrt(np.maximum(lam, 0.0))
    m = int(np.count_nonzero(sigma > atol))
    if modes is not None:
        m = min(m, int(modes))
    W, sigma = W[:, :m].copy(), sigma[:m]
    for j in range(m):
        if W[np.argmax(np.abs(W[:, j])), j] < 0:
            W[:, j] = -W[:, j]
    return VA((W / sigma).T @ X, A.space), sigma


# ----------------------------------------------------------------------------------------------------------
#  POD basis extension and greedy basis generation (pyMOR extend_basis(method='pod') / greedy [ext])
# ----------------------------------------------------------------------------------------------------------

def extend_basis_pod(reductor, U, pod_modes=1, pod_rtol=1e-13):
    """pyMOR ``extend_basis(U, method='pod', pod_modes=m)`` with ``pod_orthonormalize=True``, per subdomain ``i``: the
    projection error ``R`` of ``U_i`` onto the basis (classical Gram-Schmidt twice, in the reductor's product), its POD
    (:func:`pod`) with at most ``pod_modes`` modes of ``sigma > pod_rtol max_j |u_{i,j}|``, one more Gram-Schmidt
    pass of the modes against the basis and a Cholesky QR among themselves (of the largest leading block that is
    numerically positive definite).  Returns the number of vectors appended per subdomain; raises ExtensionError if none."""
    import scipy.linalg as sla
    subs = reductor.d.solution_space.subspaces
    counts = []
    for i, s in enumerate(subs):
        basis, P = reductor.bases[s.id], reductor.products[i]
        ip = (lambda X, Y: X @ (P.matrix @ Y.T)) if P is not None else (lambda X, Y: X @ Y.T)
        V, u = basis.data, U._blocks[i].data
        R = u.copy()
        for _ in range(2):
            if len(V):
                R = R - ip(R, V) @ V
        norm_max = np.sqrt(np.maximum(np.diag(ip(u, u)), 0.0)).max()
        Y = pod(VA(R, s), product=P, modes=pod_modes, atol=pod_rtol * norm_max)[0].data
        if len(V) and len(Y):
            Y = Y - ip(Y, V) @ V
        G = ip(Y, Y)
        G = 0.5 * (G + G.T)
        for m in range(len(Y), -1, -1):
            try:
                L = np.linalg.cholesky(G[:m, :m]) if m else None
                break
            except np.linalg.LinAlgError:
                continue
        if m:
            basis.append(VA(sla.solve_triangular(L, Y[:m], lower=True), basis.space))
        counts.append(m)
    if sum(counts) == 0:
        raise ExtensionError
    return counts


def sparse_fine_solve(d, mus):
    """Fine-scale solutions of ``d`` for the parameters ``mus`` with SciPy ``spsolve`` on the assembled sparse A(mu)."""
    import scipy.sparse.linalg as spla
    subs = d.solution_space.subspaces
    S = len(subs)
    out = []
    for mu in mus:
        mu = d.parse_parameter(mu)
        A = None
        for op, c in zip(d.operator.operators, d.operator.coefficients):
            M = sp.bmat([[(op._blocks[k, l].matrix if op._blocks[k, l] is not None else None) for l in range(S)]
                         for k in range(S)], format='csc')
            theta = c.evaluate(mu) if hasattr(c, 'evaluate') else float(c)
            A = theta * M if A is None else A + theta * M
        f = d.rhs.as_source_array(mu).data[0]
        out.append(spla.spsolve(A.tocsc(), f))
    return d.solution_space.from_data(np.array(out))


def _operator_error(d, U_h, U_N, mu):
    """``|||u_h - u_N|||_mu`` of two fine-scale arrays of length 1 with the sparse A(mu)."""
    subs = d.solution_space.subspaces
    S = len(subs)
    mu = d.parse_parameter(mu)
    E = U_h.data[0] - U_N.data[0]
    AE = np.zeros_like(E)
    for op, c in zip(d.operator.operators, d.operator.coefficients):
        M = sp.bmat([[(op._blocks[k, l].matrix if op._blocks[k, l] is not None else None) for l in range(S)]
                     for k in range(S)], format='csr')
        AE += (c.evaluate(mu) if hasattr(c, 'evaluate') else float(c)) * (M @ E)
    return float(np.sqrt(max(E @ AE, 0.0)))


def greedy(d, reductor, samples, use_estimator=True, atol=None, rtol=None, max_extensions=None, extension_params=None,
           mus_per_extension=1):
    """pyMOR ``greedy(d, reductor, samples, ...)`` with several parameters per extension: reduce; the error of every sample
    (``eta`` of the reduced solution, or ``|||u_h - R u_N|||_mu`` against ``spsolve``); stop on ``atol`` / ``rtol`` (relative
    to the first maximum) / ``max_extensions``; otherwise solve the ``mus_per_extension`` samples with the largest error
    (descending, ties: lower index first) and extend the bases (``method='pod'`` -> :func:`extend_basis_pod`); an
    ExtensionError ends the loop.  Returns the dict of ``pylrbms_b200.greedy``."""
    params = dict(extension_params or {})
    method = params.pop('method', 'gram_schmidt')
    samples = np.asarray(samples)
    k = min(int(mus_per_extension), len(samples))
    U_train = None if use_estimator else [sparse_fine_solve(d, [mu]) for mu in samples]
    max_errs, max_err_mus, extension_mus = [], [], []
    extensions = 0
    while True:
        rd = reductor.reduce()
        errors = np.zeros(len(samples))
        for j, mu in enumerate(samples):
            U_N = rd.solve(mu)
            if use_estimator:
                errors[j] = float(np.atleast_1d(rd.estimate(U_N, mu))[0])
            else:
                errors[j] = _operator_error(d, U_train[j], reductor.reconstruct(U_N), mu)
        worst = np.argsort(-errors, kind='stable')[:k]
        max_errs.append(float(errors[worst[0]]))
        max_err_mus.append(samples[worst[0]])
        if atol is not None and max_errs[-1] <= atol:
            break
        if rtol is not None and max_errs[-1] <= rtol * max_errs[0]:
            break
        if max_extensions is not None and extensions >= max_extensions:
            break
        U = sparse_fine_solve(d, samples[worst])
        try:
            if method == 'pod':
                extend_basis_pod(reductor, U, **params)
            else:
                reductor.extend_basis(U)
        except ExtensionError:
            break
        extensions += 1
        extension_mus.append(samples[worst])
    return {'rd': rd, 'max_errs': np.array(max_errs), 'max_err_mus': max_err_mus, 'extension_mus': extension_mus,
            'extensions': extensions}
