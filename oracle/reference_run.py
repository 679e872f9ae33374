"""TEST INFRASTRUCTURE ONLY -- runs the REFERENCE'S OWN source files for the hot path on seeded inputs.

``estimators.py``, ``reductor.py`` and ``online_enrichment.py`` of the reference are loaded *unmodified* from
``$LRBMS_REFERENCE_DIR`` (a pylrbms checkout's ``python/dune/pylrbms``, never copied) and executed on top of stand-ins for their third-party
dependencies, none of which can be installed here:

* **pyMOR** (the fork ``git+https://zivgitlab.uni-muenster.de/srave_01/pymor.git@master``, pymor-0.5, branch-pinned only):
  ``oracle/pymor_like.py`` restates the published semantics of the pieces the three files import
  (``NumpyMatrixOperator``, ``BlockDiagonalOperator``, ``LincombOperator``, ``unblock``, ``ImmutableInterface.with_``,
  ``pymor.parallel.mpi.norm``) and ``oracle/lrbms_oracle.GenericRBSystemReductor`` the fork-only base class;
* **dune-gdt / dune-xt** (assembly, visualisation) -- not on the path: the operators come from the same host-assembled
  ``BlockSwipdgData`` containers every other test uses; ``make_discrete_function`` / ``DuneGDTVisualizer`` are only
  imported, never called on the path;
* **mpi4py** -- single process: ``mpi_norm`` is the Frobenius norm, ``MPI.COMM_WORLD`` a placeholder.

What this pins: every line of arithmetic that lives in the reference's own files -- the estimator
(``estimators.py:45-130``: the three local quantities, the residual scaling, ``alpha`` returning inside its loop, ``gamma``,
eta, the indicators), the reductor (``reductor.py:32-73``: Oswald / flux-reconstruction image bases, q-major RT ordering,
the reduced ``fr_red`` / ``oi_red`` operators), Doerfler marking and the enrichment loop (``online_enrichment.py:9-93``).
What it does not pin: pyMOR's projection / unblock / Gram-Schmidt algorithms (restated, see above) and anything DUNE
assembles.  ``tests/golden/make_reference_golden.py`` writes the outputs as fixtures; ``tests/test_oracle_golden.py``
checks the oracle's own restatement of those files against them without needing the reference.
"""
from __future__ import annotations

import contextlib
import copy
import importlib.util
import logging
import os
import sys
import types

import numpy as np

# the ``python/dune/pylrbms`` directory of a pylrbms checkout; the reference is not part of this repository
REFERENCE_DIR = os.environ.get('LRBMS_REFERENCE_DIR', '')


class _Logger(logging.Logger):
    """pyMOR's logger surface as far as the three files use it (``info3``, ``warn``, ``block``)."""

    def info3(self, *a, **k):
        self.info(*a, **k)

    def info2(self, *a, **k):
        self.info(*a, **k)

    def warn(self, *a, **k):
        self.warning(*a, **k)

    @contextlib.contextmanager
    def block(self, *a, **k):
        yield self


def _logger(name):
    old = logging.getLoggerClass()
    logging.setLoggerClass(_Logger)
    try:
        lg = logging.getLogger('reference_run.' + name)
    finally:
        logging.setLoggerClass(old)
    return lg


class BasicInterface:
    """``pymor.core.interfaces.BasicInterface``: a ``logger`` per class."""

    @property
    def logger(self):
        return _logger(type(self).__name__)


class ImmutableInterface(BasicInterface):
    """``with_``: a copy with some ``__init__`` attributes replaced (pyMOR re-runs ``__init__`` with the stored arguments;
    for classes whose ``__init__`` only stores its arguments, as here, that is a shallow copy plus ``setattr``)."""

    def with_(self, **kwargs):
        new = copy.copy(self)
        for k, v in kwargs.items():
            setattr(new, k, v)
        return new


def _module(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    return m


def install_dependency_stand_ins():
    """Register the stand-in modules under the names the reference imports.  Refuses to shadow a real installation."""
    from . import lrbms_oracle as O
    from . import pymor_like as P
    for real in ('pymor', 'mpi4py'):
        if real in sys.modules and not getattr(sys.modules[real], '_lrbms_stand_in', False):
            raise RuntimeError(real + ' is really installed: run the reference on it instead of the stand-ins')

    class GenericRBSystemReductor(O.GenericRBSystemReductor, BasicInterface):
        pass

    class _Comm:
        rank, size = 0, 1

    mods = {
        'pymor': _module('pymor', _lrbms_stand_in=True),
        'pymor.algorithms': _module('pymor.algorithms'),
        'pymor.algorithms.system': _module('pymor.algorithms.system', unblock=P.unblock),
        'pymor.core': _module('pymor.core'),
        'pymor.core.interfaces': _module('pymor.core.interfaces', ImmutableInterface=ImmutableInterface,
                                         BasicInterface=BasicInterface),
        'pymor.operators': _module('pymor.operators'),
        'pymor.operators.block': _module('pymor.operators.block', BlockDiagonalOperator=P.BlockDiagonalOperator,
                                         BlockOperator=P.BlockOperator),
        'pymor.operators.constructions': _module('pymor.operators.constructions', LincombOperator=P.LincombOperator,
                                                 VectorArrayOperator=P.VectorArrayOperator),
        'pymor.operators.numpy': _module('pymor.operators.numpy', NumpyMatrixOperator=P.MatrixOperator),
        'pymor.reductors': _module('pymor.reductors'),
        'pymor.reductors.system': _module('pymor.reductors.system', GenericRBSystemReductor=GenericRBSystemReductor),
        'pymor.parallel': _module('pymor.parallel'),
        'pymor.parallel.mpi': _module('pymor.parallel.mpi', norm=O.mpi_norm),
        'pymor.bindings': _module('pymor.bindings'),
        'pymor.bindings.dunegdt': _module('pymor.bindings.dunegdt', DuneGDTVisualizer=object),
        'pymor.vectorarrays': _module('pymor.vectorarrays'),
        'pymor.vectorarrays.list': _module('pymor.vectorarrays.list', ListVectorArray=P.VA),
        'pymor.vectorarrays.numpy': _module('pymor.vectorarrays.numpy', NumpyVectorArray=P.VA),
        'mpi4py': _module('mpi4py', _lrbms_stand_in=True, MPI=types.SimpleNamespace(COMM_WORLD=_Comm(), SUM='sum', DOUBLE='d')),
    }
    # dune.gdt: only imported (visualisation helper), never called on the path
    if 'dune' not in sys.modules:
        mods['dune'] = _module('dune')
    mods['dune.gdt'] = _module('dune.gdt')
    mods['dune.gdt.discretefunction'] = _module('dune.gdt.discretefunction', make_discrete_function=None)
    for name, m in mods.items():
        sys.modules.setdefault(name, m)


def load_reference(reference_dir=REFERENCE_DIR):
    """The reference's three modules, executed from where they lie.  Returns a namespace with ``estimators``, ``reductor``,
    ``online_enrichment``."""
    if not os.path.isdir(reference_dir):
        raise FileNotFoundError('reference sources not found at {!r}: set LRBMS_REFERENCE_DIR to the python/dune/pylrbms '
                                'directory of a pylrbms checkout'.format(reference_dir))
    install_dependency_stand_ins()
    out = types.SimpleNamespace()
    for name in ('estimators', 'reductor', 'online_enrichment'):
        spec = importlib.util.spec_from_file_location('lrbms_reference_' + name, os.path.join(reference_dir, name + '.py'))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        setattr(out, name, mod)
    return out


def build_reference_objects(data, bases, order=None, energy_products=False):
    """The oracle's operator dictionary (host-assembled inputs) with the REFERENCE's estimator and reductor on top."""
    from . import lrbms_oracle as O
    ref = load_reference()
    d = O.build_discretization(data)
    oe = d.estimator                                             # the oracle's: only its constructor arguments are reused
    grid = types.SimpleNamespace(subdomains_on_rank=list(range(data.num_subdomains)))
    est = ref.estimators.EllipticEstimator(grid, oe.min_diffusion_evs, oe.subdomain_diameters, oe.local_eta_rf_squared,
                                           oe.lambda_coeffs, oe.mu_bar, oe.mu_hat, oe.flux_reconstruction,
                                           oe.oswald_interpolation_error, mpi_comm=None)
    d = d.with_(estimator=est)
    S = data.num_subdomains
    products = [d.operators['local_energy_dg_product_%d' % i] for i in range(S)] if energy_products else None
    red = ref.reductor.LRBMSReductor(d, bases=None if bases is None else {'domain_%d' % i: bases[i] for i in range(S)},
                                     products=products, order=order)
    return ref, d, red


def reference_outputs(data, bases, mus):
    """Same dictionary as ``tests/golden/make_golden.py::oracle_outputs``, computed by the reference's classes."""
    from .pymor_like import LincombOperator
    ref, d, red = build_reference_objects(data, bases)
    rd = red.reduce()
    out = {'mus': np.asarray(mus), 'block_dims': np.array(rd.block_dims)}
    for name, op in list(rd.operators.items()) + [('product_' + k, v) for k, v in rd.products.items()]:
        terms = op.operators if isinstance(op, LincombOperator) else [op]
        for q, t in enumerate(terms):
            M = t.matrix if hasattr(t, 'matrix') else t._array.data
            out['red__{}__{}'.format(name, q)] = np.asarray(M)
    for key in sorted(k for k in red.bases if str(k).startswith(('OI_', 'RT_'))):
        out['basis__' + key] = np.asarray(red.bases[key].data)
    U, eta, parts, ind = [], [], [], []
    for mu in mus:
        u = rd.solve(mu)
        e, p, i_ = rd.estimate(u, mu, decompose=True)
        U.append(u.data[0]); eta.append(e); parts.append(np.stack([x[:, 0] for x in p])); ind.append(i_[:, 0])
    out.update(U=np.array(U), eta=np.array(eta), parts=np.array(parts), indicators=np.array(ind))
    # the same estimator code on the FINE-SCALE operators (d.estimate of the reconstructed solution, estimators.py:45-112
    # with the grid-walking flux reconstruction / Oswald operators replaced by their matrices)
    f_eta, f_parts, f_ind = [], [], []
    for k, mu in enumerate(mus):
        U_fine = red.reconstruct(rd.solve(mu))
        e, p, i_ = d.estimate(U_fine, mu, decompose=True)
        f_eta.append(e); f_parts.append(np.stack([x[:, 0] for x in p])); f_ind.append(i_[:, 0])
    out.update(fine_eta=np.array(f_eta), fine_parts=np.array(f_parts), fine_indicators=np.array(f_ind))
    # Doerfler marking (online_enrichment.py:9-22) on the indicators of the first parameter
    for theta in (0.2, 0.5, 0.9, 1.0):
        out['doerfler_%g' % theta] = np.array(ref.online_enrichment.doerfler_marking(list(ind[0]), theta), dtype=np.int64)
    return out


def reference_enrichment(data, bases, mu, enrichment_steps, theta=0.5, max_age=2):
    """The reference's ``AdaptiveEnrichment.solve`` (``online_enrichment.py:63-93``) driving its own reductor / estimator."""
    ref, d, red = build_reference_objects(data, bases)
    rd = red.reduce()
    block_space = types.SimpleNamespace(num_blocks=data.num_subdomains)
    ae = ref.online_enrichment.AdaptiveEnrichment(None, d, block_space, red, rd, 1e-14, theta, max_age)
    log = []
    U, rd, red = ae.solve(mu, enrichment_steps=enrichment_steps,
                          callback=lambda rd_, U_, mu_, info: log.append((float(info['eta']), int(info['global RB size']),
                                                                          int(info['local_problem_solves']))))
    return {'eta': np.array([l[0] for l in log]), 'rb_size': np.array([l[1] for l in log]),
            'local_problem_solves': np.array([l[2] for l in log]), 'U': np.asarray(U.data[0]),
            'block_dims': np.array(rd.block_dims)}


def reference_enrichment_sequence(data, mus, theta=0.5, max_age=2, target_error=1e-12):
    """The enrichment scenario of ``tests/test_adaptive_enrichment.py``: bases initialised with the order-0 DG shape
    functions (``reductor.py:24-30``), local energy products for the Gram-Schmidt extension, ONE enrichment step per
    parameter of ``mus`` with the reference's ``AdaptiveEnrichment`` (``online_enrichment.py:63-93``) and ``enrich_local``
    (``reductor.py:75-78``).  The corrector problem itself is the oracle's restatement of the dune-gdt neighbourhood solve."""
    ref, d, red = build_reference_objects(data, None, order=0, energy_products=True)
    block_space = types.SimpleNamespace(num_blocks=data.num_subdomains)
    ae = ref.online_enrichment.AdaptiveEnrichment(None, d, block_space, red, red.reduce(), target_error, theta, max_age)
    log = []
    U = rd = None
    for mu in mus:
        U, rd, _ = ae.solve(mu, enrichment_steps=1,
                            callback=lambda rd_, U_, mu_, info: log.append((float(info['eta']), int(info['global RB size']),
                                                                            int(info['local_problem_solves']))))
    u_fine = np.concatenate([b.data[0] for b in red.reconstruct(U)._blocks])
    return {'mus': np.asarray(mus, dtype=float), 'eta': np.array([l[0] for l in log]), 'rb_size': np.array([l[1] for l in log]),
            'local_problem_solves': np.array([l[2] for l in log]), 'block_dims': np.array(rd.block_dims),
            'u_fine': u_fine, 'args': np.array([theta, max_age, target_error])}
