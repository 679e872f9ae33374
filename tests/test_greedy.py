"""Greedy basis generation (``pylrbms_b200.greedy``) and the POD basis extension (``extend_basis(method='pod')``):

1. (CPU) the greedy's control flow on fake models: the atol / rtol / max_extensions stops, the stop on ExtensionError,
   top-k selection with ties, ``len(max_errs) == extensions + 1``, argument errors; the oracle's POD against an SVD;
2. the POD extension against the oracle on C1 and the 3D synthetic operators (ragged and empty bases, k = 1 and 5 snapshots,
   a subdomain already in the span, every subdomain in the span, the ``pod_modes`` cap; with and without products), and
   ``method='pod'`` with one snapshot against ``gram_schmidt``;
3. weak and strong greedy against the oracle greedy on C1; the strong greedy's maximum error does not increase; two runs
   are bit-identical; k = 5 selects the top 5 of ``rd.sweep``'s eta;
4. C2 at full size: a weak greedy with k = 32 and ``pod_modes=4``, then the error analysis on test parameters.
"""
import types

import numpy as np
import pytest

gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------
#  1. host logic, no device
# ---------------------------------------------------------------------------------------------------------------------

class _FakeRd:
    def __init__(self, errors, log):
        self.errors, self.log = np.asarray(errors, dtype=np.float64), log

    def sweep_eta_into(self, mus, eta_host):
        import torch
        assert len(mus) == len(self.errors)
        eta_host.copy_(torch.from_numpy(self.errors))
        return 0, float(self.errors.max()), int(np.argmax(self.errors))


class _FakeReductor:
    """``reduce()`` returns the next error vector of ``schedule``; ``extend_basis`` raises ExtensionError from call number
    ``fail_at`` on."""

    def __init__(self, d, schedule, fail_at=None):
        self.d, self.schedule, self.fail_at = d, list(schedule), fail_at
        self.log, self.n_reduce, self.n_extend = [], 0, 0

    def reduce(self):
        rd = _FakeRd(self.schedule[min(self.n_reduce, len(self.schedule) - 1)], self.log)
        self.n_reduce += 1
        return rd

    def extend_basis(self, U, **kw):
        from pylrbms_b200.reductor import ExtensionError
        self.log.append(('extend', U, kw))
        if self.fail_at is not None and self.n_extend >= self.fail_at:
            raise ExtensionError
        self.n_extend += 1


class _FakeD:
    def __init__(self):
        self.solves = []

    def solve_batch(self, mus, inverse_options=None):
        self.solves.append((list(mus), inverse_options))
        return ('U', list(mus))


def _fake_run(schedule, samples=(0.1, 0.2, 0.3, 0.4, 0.5), fail_at=None, **kw):
    from pylrbms_b200.greedy import greedy
    d = _FakeD()
    red = _FakeReductor(d, schedule, fail_at)
    res = greedy(d, red, np.asarray(samples), **kw)
    assert len(res['max_errs']) == res['extensions'] + 1 == len(res['max_err_mus'])
    assert len(res['extension_mus']) == res['extensions'] == red.n_extend
    assert red.n_reduce == res['extensions'] + 1
    return res, d, red


def test_greedy_stops_on_max_extensions():
    sched = [[1, 5, 3, 2, 4], [1, 0.5, 3, 2, 4], [1, 0.5, 0.3, 2, 4], [1, 0.5, 0.3, 2, 0.4]]
    res, d, red = _fake_run(sched, max_extensions=3)
    assert res['extensions'] == 3
    assert list(res['max_errs']) == [5, 4, 4, 2]
    assert [list(m) for m in res['extension_mus']] == [[0.2], [0.5], [0.5]]
    assert list(res['max_err_mus']) == [0.2, 0.5, 0.5, 0.4]
    assert [s[0] for s in d.solves] == [[0.2], [0.5], [0.5]]
    res, _, _ = _fake_run(sched, max_extensions=0)
    assert res['extensions'] == 0 and list(res['max_errs']) == [5]


def test_greedy_stops_on_atol_and_rtol():
    sched = [[8, 1, 1, 1, 1], [2, 1, 1, 1, 1], [1, 0.9, 0.1, 0.1, 0.1], [0.5, 0.1, 0.1, 0.1, 0.1]]
    res, _, _ = _fake_run(sched, atol=1.0)
    assert res['extensions'] == 2 and list(res['max_errs']) == [8, 2, 1]          # max <= atol stops
    res, _, _ = _fake_run(sched, rtol=0.25)
    assert res['extensions'] == 1 and list(res['max_errs']) == [8, 2]             # 2 <= 0.25 * 8
    res, _, _ = _fake_run(sched, atol=0.1, rtol=0.01, max_extensions=3)
    assert res['extensions'] == 3 and list(res['max_errs']) == [8, 2, 1, 0.5]
    res, _, _ = _fake_run([[0, 0, 0, 0, 0]], rtol=0.5)
    assert res['extensions'] == 0                                                   # 0 <= rtol * 0


def test_greedy_stops_on_extension_error():
    sched = [[1, 5, 3, 2, 4], [1, 0.5, 3, 2, 4]]
    res, _, red = _fake_run(sched, fail_at=1, max_extensions=5, extension_params={'method': 'pod', 'pod_modes': 2})
    assert res['extensions'] == 1 and list(res['max_errs']) == [5, 4]
    assert [e[2] for e in red.log if e[0] == 'extend'] == [{'method': 'pod', 'pod_modes': 2}] * 2


def test_greedy_top_k_with_ties():
    from pylrbms_b200.greedy import select_worst
    assert list(select_worst([1, 3, 3, 2, 3, 0], 4)) == [1, 2, 4, 3]
    assert list(select_worst([2.0, 2.0, 2.0], 5)) == [0, 1, 2]
    sched = [[1, 3, 3, 2, 3], [0, 0, 0, 0, 0]]
    res, d, _ = _fake_run(sched, mus_per_extension=4, max_extensions=1)
    assert list(res['extension_mus'][0]) == [0.2, 0.3, 0.5, 0.4]
    assert res['max_err_mus'][0] == 0.2
    # more samples than parameters per extension: all of them, in order of decreasing error
    res, d, _ = _fake_run(sched, samples=[0.1, 0.2, 0.3, 0.4, 0.5], mus_per_extension=32, max_extensions=1)
    assert d.solves[0][0] == [0.2, 0.3, 0.5, 0.4, 0.1]


def test_greedy_strong_uses_columns_of_the_training_solutions(monkeypatch):
    from pylrbms_b200 import error_analysis
    sched = [[1, 5, 3, 2, 4], [1, 0.5, 3, 2, 4], [0.1] * 5]

    class _UTrain:
        def __getitem__(self, idx):
            return ('columns', list(idx))

    calls = []

    def fake_analysis(d, reductor, rd, mus, U_h=None, inverse_options=None):
        calls.append(U_h)
        return types.SimpleNamespace(operator_errors=rd.errors)

    monkeypatch.setattr(error_analysis, 'reduction_error_analysis', fake_analysis)
    from pylrbms_b200.greedy import greedy
    d = _FakeD()
    d.solve_batch = lambda mus, inverse_options=None: _UTrain()
    red = _FakeReductor(d, sched)
    res = greedy(d, red, [0.1, 0.2, 0.3, 0.4, 0.5], use_estimator=False, atol=0.2, mus_per_extension=2)
    assert res['extensions'] == 2 and list(res['max_errs']) == [5, 4, 0.1]
    assert [e[1] for e in red.log if e[0] == 'extend'] == [('columns', [1, 4]), ('columns', [4, 2])]
    assert res['extension_mus'] == [[0.2, 0.5], [0.5, 0.3]]
    assert len(calls) == 3 and all(isinstance(c, _UTrain) for c in calls)


def test_greedy_argument_errors():
    from pylrbms_b200.greedy import greedy
    d = _FakeD()
    red = _FakeReductor(d, [[1.0]])
    with pytest.raises(ValueError, match='another discretization'):
        greedy(_FakeD(), red, [0.1])
    with pytest.raises(ValueError, match='at least one'):
        greedy(d, red, [])
    for k in (0, -1, 1.5):
        with pytest.raises(ValueError, match='mus_per_extension'):
            greedy(d, red, [0.1], mus_per_extension=k)
    with pytest.raises(ValueError, match='max_extensions'):
        greedy(d, red, [0.1], max_extensions=-1)
    with pytest.raises(ValueError, match='non-negative'):
        greedy(d, red, [0.1], atol=-1.0)
    assert red.n_reduce == 0


def test_oracle_pod_matches_svd():
    import scipy.sparse as sp
    from oracle.greedy_oracle import pod
    from oracle.pymor_like import VA, MatrixOperator, Space
    rng = np.random.default_rng(4)
    space = Space(60)
    X = rng.standard_normal((7, 60)) * np.array([1, 0.5, 0.3, 0.1, 1e-3, 1e-5, 1e-7])[:, None]
    B = sp.random(60, 60, density=0.1, random_state=5)
    M = (B @ B.T + sp.eye(60)).tocsr()
    for P in (None, MatrixOperator(M)):
        L = np.linalg.cholesky(M.toarray()) if P is not None else np.eye(60)
        _, s, Vt = np.linalg.svd(X @ L, full_matrices=False)          # P-orthonormal modes: rows of Vt L^{-1}
        ref = np.linalg.solve(L.T, Vt.T).T
        modes, sigma = pod(VA(X, space), product=P, modes=4)
        assert len(modes) == 4 and np.allclose(sigma, s[:4], rtol=1e-10)
        for j in range(4):
            sign = np.sign(modes.data[j] @ (M @ ref[j]) if P is not None else modes.data[j] @ ref[j])
            assert np.abs(modes.data[j] - sign * ref[j]).max() <= 1e-8 * np.abs(ref[j]).max()
        G = modes.data @ (M @ modes.data.T) if P is not None else modes.data @ modes.data.T
        assert np.abs(G - np.eye(4)).max() < 1e-10
        # the threshold drops modes with sigma <= atol; the sign rule makes the largest eigenvector entry positive
        assert len(pod(VA(X, space), product=P, atol=0.5 * s[5])[0]) == 6
        W = (modes.data @ (M.toarray() if P is not None else np.eye(60)) @ X.T).T / sigma     # W = X^T P modes / sigma
        assert np.all(W[np.argmax(np.abs(W), axis=0), np.arange(4)] > 0)


# ---------------------------------------------------------------------------------------------------------------------
#  2. POD extension on the device against the oracle
# ---------------------------------------------------------------------------------------------------------------------

def _orthonormal(X, M):
    G = X @ (M @ X.T)
    return np.linalg.solve(np.linalg.cholesky(0.5 * (G + G.T)), X)


def _fixture(name):
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg
    from pylrbms_b200.synthetic_fixture import synthetic_block_operators
    return assemble_block_swipdg((4, 4), 16) if name == 'c1' else synthetic_block_operators((3, 2, 2), (2, 2, 2), seed=1004)


def _pod_setup(name, with_products, seed=7):
    """Device and oracle reductors on the same ragged bases (one empty), orthonormal in the product they use."""
    import scipy.sparse as sp
    from oracle import lrbms_oracle as O
    from oracle.pymor_like import BlockSpace, MatrixOperator, Space
    from pylrbms_b200 import GenericRBSystemReductor, discretize
    data = _fixture(name)
    d, _ = discretize(data)
    S = data.num_subdomains
    rng = np.random.default_rng(seed)
    mats = [sp.csr_matrix(data.energy[i]) if with_products else sp.eye(int(data.n[i]), format='csr') for i in range(S)]
    bases = [_orthonormal(rng.standard_normal((1 + i % 4, int(data.n[i]))), mats[i]) for i in range(S)]
    bases[1] = np.zeros((0, int(data.n[1])))
    prods = [d.operators['local_energy_dg_product_%d' % i] for i in range(S)] if with_products else None
    red = GenericRBSystemReductor(d, bases={'domain_%d' % i: bases[i] for i in range(S)}, products=prods)
    space_ref = BlockSpace([Space(int(data.n[i]), 'domain_%d' % i) for i in range(S)])
    d_ref = types.SimpleNamespace(solution_space=space_ref)
    red_ref = O.GenericRBSystemReductor(d_ref, bases={'domain_%d' % i: bases[i] for i in range(S)},
                                        products=[MatrixOperator(m) for m in mats] if with_products else None)
    return data, d, red, red_ref, mats, bases


def _snapshots(data, bases, k, in_span, rng):
    """``k`` snapshots with decaying scales (well separated singular values); on the subdomains ``in_span`` they are
    combinations of the basis vectors."""
    S = data.num_subdomains
    U = rng.standard_normal((k, int(np.sum(data.n)))) * (0.5 ** np.arange(k))[:, None]
    offs = np.concatenate([[0], np.cumsum(data.n)])
    for i in in_span:
        U[:, offs[i]:offs[i + 1]] = rng.standard_normal((k, len(bases[i]))) @ bases[i]
    return U


def _check_extension(data, red, red_ref, mats, bases, kw, counts_expected=None):
    S = data.num_subdomains
    for i in range(S):
        a = red.bases['domain_%d' % i].to_numpy()
        b = red_ref.bases['domain_%d' % i].data
        assert a.shape == b.shape, (i, a.shape, b.shape)
        if len(a):
            assert np.abs(a - b).max() <= 1e-9 * np.abs(b).max(), (i, np.abs(a - b).max())
            G = a @ (mats[i] @ a.T)
            assert np.abs(G - np.eye(len(a))).max() < 1e-11, (i, np.abs(G - np.eye(len(a))).max())
        if counts_expected is not None:
            assert len(a) - len(bases[i]) == counts_expected[i], (i, len(a), len(bases[i]))


@gpu
@pytest.mark.parametrize('name', ['c1', '3d'])
@pytest.mark.parametrize('with_products', [True, False])
@pytest.mark.parametrize('k,pod_modes', [(1, 1), (5, 3), (5, 8)])
def test_pod_extension_matches_oracle(handle, name, with_products, k, pod_modes):
    from oracle import greedy_oracle as G
    from oracle import lrbms_oracle as O
    from pylrbms_b200 import ExtensionError
    data, d, red, red_ref, mats, bases = _pod_setup(name, with_products)
    S = data.num_subdomains
    rng = np.random.default_rng(100 + k)
    in_span = [2, S - 1]
    U = _snapshots(data, bases, k, in_span, rng)
    counts = red.extend_basis(d.solution_space.from_data(U), method='pod', pod_modes=pod_modes)
    counts_ref = G.extend_basis_pod(red_ref, _ref_array(red_ref, U), pod_modes=pod_modes)
    expected = [0 if i in in_span else min(k, pod_modes) for i in range(S)]
    assert list(counts) == list(counts_ref) == expected
    _check_extension(data, red, red_ref, mats, bases, {}, expected)
    # every subdomain in the span (now including the new vectors): nothing is appended, ExtensionError
    grown = [red_ref.bases['domain_%d' % i].data for i in range(S)]
    U2 = _snapshots(data, grown, 3, range(S), rng)
    before = [len(red.bases['domain_%d' % i]) for i in range(S)]
    with pytest.raises(ExtensionError):
        red.extend_basis(d.solution_space.from_data(U2), method='pod', pod_modes=2)
    with pytest.raises(O.ExtensionError):
        G.extend_basis_pod(red_ref, _ref_array(red_ref, U2), pod_modes=2)
    assert [len(red.bases['domain_%d' % i]) for i in range(S)] == before


def _ref_array(red_ref, U):
    """``U`` (pyMOR layout) as a block array of the oracle reductor's solution space."""
    return red_ref.d.solution_space.from_data(U)


@gpu
@pytest.mark.parametrize('with_products', [True, False])
def test_pod_with_one_snapshot_equals_gram_schmidt(handle, with_products):
    from pylrbms_b200 import GenericRBSystemReductor
    data, d, red, _, mats, bases = _pod_setup('c1', with_products)
    S = data.num_subdomains
    red_gs = GenericRBSystemReductor(d, bases={'domain_%d' % i: bases[i] for i in range(S)}, products=red.products)
    U = _snapshots(data, bases, 1, [3], np.random.default_rng(2))
    red.extend_basis(d.solution_space.from_data(U), method='pod')
    red_gs.extend_basis(d.solution_space.from_data(U))
    for i in range(S):
        a, b = red.bases['domain_%d' % i].to_numpy(), red_gs.bases['domain_%d' % i].to_numpy()
        assert a.shape == b.shape == (len(bases[i]) + (i != 3), int(data.n[i]))
        assert np.abs(a - b).max() <= 1e-10 * np.abs(b).max()
    with pytest.raises(ValueError, match='method'):
        red.extend_basis(d.solution_space.from_data(U), method='svd')
    with pytest.raises(ValueError, match='pod_modes'):
        red.extend_basis(d.solution_space.from_data(U), method='pod', pod_modes=0)


# ---------------------------------------------------------------------------------------------------------------------
#  3. greedy against the oracle greedy
# ---------------------------------------------------------------------------------------------------------------------

_C1 = {}


def _c1():
    if not _C1:
        from oracle import lrbms_oracle as O
        from pylrbms_b200 import discretize
        data = _fixture('c1')
        _C1.update(data=data, d=discretize(data)[0], d_ref=O.build_discretization(data))
    return _C1['data'], _C1['d'], _C1['d_ref']


_TRAIN = np.array([0.1, 0.19, 0.31, 0.42, 0.55, 0.63, 0.77, 0.86, 1.0])


@gpu
@pytest.mark.parametrize('use_estimator', [True, False])
@pytest.mark.parametrize('params,k', [(None, 1), ({'method': 'pod', 'pod_modes': 2}, 3)])
def test_greedy_matches_oracle(handle, use_estimator, params, k):
    from oracle import lrbms_oracle as O
    from oracle import greedy_oracle as G
    from pylrbms_b200 import LRBMSReductor, greedy
    data, d, d_ref = _c1()
    red = LRBMSReductor(d)
    red.incremental = True
    # The oracle solves exactly, the device to a relative residual: the strong greedy's errors fall to 5e-9 of the first, so its
    # fine solves go to the attainable residual at C1; eta levels off where its residual terms cancel, and there the
    # snapshots' solver error moves it by ~1e-10 absolute (1e-7 relative).  Both are compared up to 1e-10 of the first max.
    opts = None if use_estimator else {'rtol': 1e-11}
    res = greedy(d, red, _TRAIN, use_estimator=use_estimator, max_extensions=3, extension_params=params,
                 mus_per_extension=k, inverse_options=opts)
    ref = G.greedy(d_ref, O.LRBMSReductor(d_ref), _TRAIN, use_estimator=use_estimator, max_extensions=3,
                   extension_params=params, mus_per_extension=k)
    assert res['extensions'] == ref['extensions'] >= 2
    assert [list(m) for m in res['extension_mus']] == [list(m) for m in ref['extension_mus']]
    floor = 1e-10 * ref['max_errs'][0]
    assert np.all(np.abs(res['max_errs'] - ref['max_errs']) <= 1e-8 * ref['max_errs'] + floor), (res['max_errs'],
                                                                                                 ref['max_errs'])
    assert list(res['rd'].block_dims) == [len(red.bases['domain_%d' % i]) for i in range(data.num_subdomains)]
    print('use_estimator', use_estimator, params, 'max_errs', res['max_errs'], 'extension_mus', res['extension_mus'])
    if not use_estimator:
        errs = res['max_errs']
        assert np.all(errs[1:] <= errs[:-1] * (1 + 1e-10)), errs         # Galerkin optimality, nested spaces


@gpu
def test_greedy_is_deterministic(handle):
    from pylrbms_b200 import LRBMSReductor, greedy
    data, d, _ = _c1()
    runs = []
    for _ in range(2):
        red = LRBMSReductor(d)
        red.incremental = True
        res = greedy(d, red, np.linspace(*data.parameter_range, 40), max_extensions=3,
                     extension_params={'method': 'pod', 'pod_modes': 2}, mus_per_extension=4)
        runs.append((res, [red.bases['domain_%d' % i].to_numpy() for i in range(data.num_subdomains)]))
    (a, ba), (b, bb) = runs
    assert np.array_equal(a['max_errs'], b['max_errs'])
    assert all(np.array_equal(x, y) for x, y in zip(ba, bb))
    assert [list(m) for m in a['extension_mus']] == [list(m) for m in b['extension_mus']]


@gpu
def test_greedy_selects_top_k_of_sweep(handle):
    from pylrbms_b200 import LRBMSReductor, greedy
    data, d, _ = _c1()
    train = np.random.default_rng(12).uniform(*data.parameter_range, 50)
    _, eta = LRBMSReductor(d).reduce().sweep(train)
    top = np.argsort(-eta, kind='stable')[:5]
    assert np.all(np.diff(np.sort(eta)[::-1][:6]) < 0)                    # no ties among the leaders
    res = greedy(d, LRBMSReductor(d), train, max_extensions=1, mus_per_extension=5)
    assert list(res['extension_mus'][0]) == list(train[top])
    assert res['max_errs'][0] == eta[top[0]] and res['max_err_mus'][0] == train[top[0]]


# ---------------------------------------------------------------------------------------------------------------------
#  4. C2 at full size
# ---------------------------------------------------------------------------------------------------------------------

@gpu
def test_greedy_c2_weak_pod(handle):
    from pylrbms_b200 import LRBMSReductor, discretize, greedy, reduction_error_analysis
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg
    data = assemble_block_swipdg((8, 8), 32)
    d, _ = discretize(data)
    assert d.solution_space.dim == 393216
    rng = np.random.default_rng(2026)
    train = rng.uniform(*data.parameter_range, 1024)
    red = LRBMSReductor(d)
    red.incremental = True
    res = greedy(d, red, train, max_extensions=3, extension_params={'method': 'pod', 'pod_modes': 4}, mus_per_extension=32)
    # the solution manifold of this one-parameter problem is narrow: the extension may find nothing above pod_rtol before
    # the third step, which ends the greedy (ExtensionError)
    assert res['extensions'] >= 1 and all(len(m) == 32 for m in res['extension_mus'])
    assert res['max_errs'][-1] < res['max_errs'][0]
    test = rng.uniform(*data.parameter_range, 64)
    ana = reduction_error_analysis(d, red, res['rd'], test)
    assert np.all(ana.errors <= ana.eta)
    print('C2 greedy max eta', res['max_errs'], 'basis sizes', sorted(set(res['rd'].block_dims)),
          'effectivities %.3f .. %.3f' % (ana.min_effectivity, ana.max_effectivity), 'time %.1f s' % res['time'])
