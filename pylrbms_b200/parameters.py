"""Parameter functionals theta_q(mu) of the affine decomposition, vectorised over a parameter batch.

Mirrors the pyMOR functionals pylrbms uses (reference ``OS2015_academic_problem.py:43-44``,
``local_thermalblock_problem.py:50-51``, ``thermalblock_problem.py:47-50``,
``discretize_elliptic_block_swipdg.py:757-759``).  ``evaluate(mu)`` keeps the single-parameter pyMOR meaning;
``evaluate_batch(mus)`` returns one value per row of the batch and is what feeds the mu-batched kernels.
"""
from __future__ import annotations

import numpy as np

_SAFE = {'sin': np.sin, 'cos': np.cos, 'exp': np.exp, 'sqrt': np.sqrt, 'pi': np.pi, 'abs': np.abs,
         'min': np.minimum, 'max': np.maximum, 'log': np.log, 'tan': np.tan, 'tanh': np.tanh}


def parse_parameter(mu, parameter_type):
    """pyMOR ``parse_parameter``: number / sequence / dict -> ``{name: array of shape parameter_type[name]}``."""
    if mu is None:
        return {}
    if isinstance(mu, dict):
        return {k: np.asarray(v, dtype=float).reshape(parameter_type.get(k, np.shape(v)) or (1,)) for k, v in mu.items()}
    mu = np.atleast_1d(np.asarray(mu, dtype=float)).ravel()
    out, pos = {}, 0
    for k in sorted(parameter_type):
        size = int(np.prod(parameter_type[k])) if parameter_type[k] else 1
        out[k] = mu[pos:pos + size].reshape(parameter_type[k] or (1,))
        pos += size
    if pos != mu.size:
        raise ValueError('parameter of size {} does not match parameter type {}'.format(mu.size, parameter_type))
    return out


def parse_parameter_batch(mus, parameter_type):
    """Batch version: ``mus`` is a sequence of parameters, an ``(n_mu,)`` / ``(n_mu, dim)`` array, or a dict of
    ``(n_mu, ...)`` arrays.  Returns ``({name: (n_mu, size) array}, n_mu)``."""
    if isinstance(mus, dict):
        out = {}
        n_mu = None
        for k, v in mus.items():
            v = np.asarray(v, dtype=float)
            v = v.reshape(v.shape[0], -1)
            n_mu = v.shape[0] if n_mu is None else n_mu
            if v.shape[0] != n_mu:
                raise ValueError('inconsistent batch sizes in parameter dict')
            out[k] = v
        return out, int(n_mu or 0)
    if isinstance(mus, (list, tuple)) and len(mus) and isinstance(mus[0], dict):
        keys = sorted(mus[0])
        return ({k: np.stack([np.asarray(m[k], dtype=float).ravel() for m in mus]) for k in keys}, len(mus))
    arr = np.asarray(mus, dtype=float)
    if arr.ndim == 1:
        arr = arr[:, None]
    total = sum(int(np.prod(parameter_type[k])) if parameter_type[k] else 1 for k in parameter_type)
    if arr.shape[1] != total:
        raise ValueError('parameter batch of shape {} does not match parameter type {}'.format(arr.shape, parameter_type))
    out, pos = {}, 0
    for k in sorted(parameter_type):
        size = int(np.prod(parameter_type[k])) if parameter_type[k] else 1
        out[k] = arr[:, pos:pos + size]
        pos += size
    return out, arr.shape[0]


def theta_matrix(coefficients, mus, parameter_type):
    """``(n_mu, len(coefficients))`` matrix of the coefficients evaluated on a parameter batch (``mus=None``: one row
    for a parameter-independent model) -- the layout the mu-batched kernels read."""
    if mus is None:
        return np.array([[float(c) if not isinstance(c, ParameterFunctional) else c.evaluate(None) for c in coefficients]])
    batch, n_mu = parse_parameter_batch(mus, parameter_type)
    cols = [c.evaluate_batch(batch, n_mu) if isinstance(c, ParameterFunctional) else np.full(n_mu, float(c))
            for c in coefficients]
    return np.ascontiguousarray(np.stack(cols, axis=1))


class ParameterFunctional:
    def evaluate(self, mu=None):
        raise NotImplementedError

    def evaluate_batch(self, mus, n_mu):
        raise NotImplementedError

    def __call__(self, mu=None):
        return self.evaluate(mu)


class ConstantParameterFunctional(ParameterFunctional):
    def __init__(self, value):
        self.value = float(value)

    def evaluate(self, mu=None):
        return self.value

    def evaluate_batch(self, mus, n_mu):
        return np.full(n_mu, self.value)


class ExpressionParameterFunctional(ParameterFunctional):
    """``ExpressionParameterFunctional('1.1 + sin(diffusion)', {'diffusion': (1,)})``."""

    def __init__(self, expression, parameter_type=None):
        self.expression, self.parameter_type = str(expression), dict(parameter_type or {})
        self._code = compile(self.expression, '<theta>', 'eval')

    def evaluate(self, mu=None):
        env = dict(_SAFE)
        for k, v in (mu or {}).items():
            v = np.asarray(v, dtype=float).ravel()
            env[k] = float(v[0]) if v.size == 1 else v
        return float(eval(self._code, {'__builtins__': {}}, env))     # noqa: S307 - restricted namespace

    def evaluate_batch(self, mus, n_mu):
        env = dict(_SAFE)
        for k, v in mus.items():
            env[k] = v[:, 0] if v.shape[1] == 1 else v.T
        val = eval(self._code, {'__builtins__': {}}, env)             # noqa: S307
        return np.broadcast_to(np.asarray(val, dtype=float), (n_mu,)).copy()


class ProjectionParameterFunctional(ParameterFunctional):
    """Picks one component of a parameter (reference ``thermalblock_problem.py:47-50``)."""

    def __init__(self, component_name, component_shape=(1,), coordinates=(0,)):
        self.name, self.shape = component_name, tuple(component_shape)
        self.coordinates = tuple(np.atleast_1d(coordinates).tolist())

    def evaluate(self, mu=None):
        return float(np.asarray(mu[self.name], dtype=float).reshape(self.shape or (1,))[self.coordinates])

    def evaluate_batch(self, mus, n_mu):
        flat = int(np.ravel_multi_index(self.coordinates, self.shape or (1,)))
        return np.ascontiguousarray(mus[self.name][:, flat])


class ProductParameterFunctional(ParameterFunctional):
    """Product of evaluations (reference ``discretize_elliptic_block_swipdg.py:757-759``)."""

    def __init__(self, factors):
        self.factors = [f if isinstance(f, ParameterFunctional) else ConstantParameterFunctional(f) for f in factors]

    def evaluate(self, mu=None):
        out = 1.0
        for f in self.factors:
            out = out * f.evaluate(mu)
        return out

    def evaluate_batch(self, mus, n_mu):
        out = np.ones(n_mu)
        for f in self.factors:
            out = out * f.evaluate_batch(mus, n_mu)
        return out


def as_functional(c, parameter_type=None):
    if isinstance(c, ParameterFunctional):
        return c
    if isinstance(c, str):
        return ExpressionParameterFunctional(c, parameter_type)
    return ConstantParameterFunctional(c)


def evaluate(c, mu):
    return c.evaluate(mu) if isinstance(c, ParameterFunctional) else float(c)
