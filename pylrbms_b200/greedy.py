"""Greedy basis generation over a training set (pyMOR ``greedy(d, reductor, samples, ...)``).

Every step reduces, evaluates an error measure on the whole training set, and extends the bases by the fine solutions of
the ``mus_per_extension`` worst parameters:

* ``use_estimator=True`` (weak greedy): ``eta`` of every sample from ``rd.sweep_eta_into`` (``lrbms_online_sweep``); the
  selected parameters are solved with ``d.solve_batch`` (``lrbms_affine_pcg_solve``) from a zero initial guess (measured
  at C2, ``profiles/r06_greedy_timing.txt``: starting from the reconstructed reduced solutions does not save iterations);
* ``use_estimator=False`` (strong greedy): the true error ``|||u_h - R u_N|||_mu`` from ``reduction_error_analysis``; the fine
  solutions of all samples are computed once and stay in HBM.

The fine solve of up to 32 parameters costs about as much as that of one (``affine_iterate_kernel`` gives one lane to each
parameter of a warp-row), so several parameters per extension are cheap; ``reductor.extend_basis(U, method='pod',
pod_modes=m)`` then keeps at most ``m`` new vectors per subdomain from them.
"""
from __future__ import annotations

import logging
import time

import numpy as np

logger = logging.getLogger('pylrbms_b200.greedy')


def _take(samples, idx):
    """The samples at the positions ``idx``, in that order, in the container type ``samples`` came in."""
    if isinstance(samples, np.ndarray):
        return samples[np.asarray(idx, dtype=np.int64)]
    return [samples[int(i)] for i in idx]


def select_worst(errors, k):
    """Indices of the ``k`` largest ``errors`` in descending order; equal errors keep ascending index order."""
    return np.argsort(-np.asarray(errors, dtype=np.float64), kind='stable')[:k]


def greedy(d, reductor, samples, use_estimator=True, atol=None, rtol=None, max_extensions=None, extension_params=None,
           mus_per_extension=1, inverse_options=None):
    """Weak (``use_estimator=True``) or strong greedy basis generation over the training set ``samples``.

    Loop: ``rd = reductor.reduce()``; the error of every sample (``eta``, or ``|||u_h - R u_N|||_mu``); stop when the maximum
    is at most ``atol``, at most ``rtol`` times the first maximum, or after ``max_extensions`` extensions; otherwise solve the
    ``mus_per_extension`` samples with the largest error (ties: lower index first) and call
    ``reductor.extend_basis(U, **extension_params)``.  An :class:`ExtensionError` ends the loop (logged).  A reduced system
    that is not positive definite, or a failing fine solve, raises :class:`LrbmsError`.

    ``samples``: whatever ``rd.thetas`` and ``d.solve_batch`` take (an array of parameters or a list).  With
    ``reductor.incremental = True`` every ``reduce()`` after the first projects only the new basis vectors; ``greedy`` does
    not change reductor settings.  Two runs on the same inputs give bit-identical bases and errors.

    Returns a dict: ``rd`` (reduced model of the final bases), ``max_errs`` (``extensions + 1`` entries, one per reduced
    model), ``max_err_mus``, ``extension_mus`` (the parameters added at each extension), ``extensions``, ``time``."""
    from ._lib import LrbmsError
    from .reductor import ExtensionError
    t0 = time.perf_counter()
    if reductor.d is not d:
        raise ValueError('the reductor was built for another discretization')
    if not isinstance(samples, np.ndarray):
        samples = list(samples)
    n = len(samples)
    if n == 0:
        raise ValueError('need at least one training parameter')
    k = int(mus_per_extension)
    if k < 1 or k != mus_per_extension:
        raise ValueError('mus_per_extension must be a positive integer')
    if max_extensions is not None and max_extensions < 0:
        raise ValueError('max_extensions must be non-negative')
    if (atol is not None and atol < 0) or (rtol is not None and rtol < 0):
        raise ValueError('atol and rtol must be non-negative')
    k = min(k, n)
    params = dict(extension_params or {})
    U_train, eta_host = None, None
    if use_estimator:
        import torch
        eta_host = torch.empty(n, dtype=torch.float64, pin_memory=torch.cuda.is_available())
    else:
        from .error_analysis import reduction_error_analysis
        U_train = d.solve_batch(samples, inverse_options=inverse_options)
    max_errs, max_err_mus, extension_mus = [], [], []
    extensions = 0
    while True:
        rd = reductor.reduce()
        if use_estimator:
            bad = rd.sweep_eta_into(samples, eta_host)[0]
            if bad:
                raise LrbmsError('greedy: the reduced operator is not positive definite for {} training parameters'.format(bad))
            errors = eta_host.numpy().copy()
        else:
            errors = reduction_error_analysis(d, reductor, rd, samples, U_h=U_train).operator_errors
        worst = select_worst(errors, k)
        max_errs.append(float(errors[worst[0]]))
        max_err_mus.append(_take(samples, worst[:1])[0])
        logger.info('greedy step %d: max error %.6e at sample #%d', extensions, max_errs[-1], int(worst[0]))
        if atol is not None and max_errs[-1] <= atol:
            break
        if rtol is not None and max_errs[-1] <= rtol * max_errs[0]:
            break
        if max_extensions is not None and extensions >= max_extensions:
            break
        selected = _take(samples, worst)
        U = d.solve_batch(selected, inverse_options=inverse_options) if use_estimator else U_train[worst]
        try:
            reductor.extend_basis(U, **params)
        except ExtensionError:
            logger.info('greedy: no basis could be extended; stopping after %d extensions', extensions)
            break
        extensions += 1
        extension_mus.append(selected)
    return {'rd': rd, 'max_errs': np.array(max_errs), 'max_err_mus': max_err_mus, 'extension_mus': extension_mus,
            'extensions': extensions, 'time': time.perf_counter() - t0}
