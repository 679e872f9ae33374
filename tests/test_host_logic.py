"""CPU tests of the host-side logic that needs no GPU: parameter functionals, batch parsing, sharding arithmetic,
the fixture generator's structure (SURVEY.md Appendix B) and bench.py's flop model."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_parameter_functionals_single_and_batched():
    from pylrbms_b200.parameters import (ExpressionParameterFunctional, ProductParameterFunctional,
                                         ProjectionParameterFunctional, parse_parameter, parse_parameter_batch)
    pt = {'diffusion': (1,)}
    one = ExpressionParameterFunctional('1.', pt)
    dif = ExpressionParameterFunctional('diffusion', pt)
    lt = ExpressionParameterFunctional('1.1 + sin(diffusion)', pt)         # local_thermalblock_problem.py:50-51
    mu = parse_parameter(0.3, pt)
    assert mu['diffusion'].shape == (1,) and one.evaluate(mu) == 1.0 and dif.evaluate(mu) == 0.3
    assert abs(lt.evaluate(mu) - (1.1 + np.sin(0.3))) < 1e-15
    prod = ProductParameterFunctional([dif, lt])
    assert abs(prod.evaluate(mu) - 0.3 * (1.1 + np.sin(0.3))) < 1e-15
    mus = np.linspace(0.1, 1.0, 11)
    batch, n = parse_parameter_batch(mus, pt)
    assert n == 11
    for f in (one, dif, lt, prod):
        vals = f.evaluate_batch(batch, n)
        assert vals.shape == (11,)
        assert np.allclose(vals, [f.evaluate(parse_parameter(m, pt)) for m in mus], rtol=0, atol=1e-15)
    # list-of-dicts and dict-of-arrays forms, multi-component parameters (thermalblock_problem.py:47-50)
    pt2 = {'diffusion': (2, 2)}
    proj = ProjectionParameterFunctional('diffusion', (2, 2), (1, 0))
    arr = np.arange(12.0).reshape(3, 4)
    b2, n2 = parse_parameter_batch(arr, pt2)
    assert n2 == 3 and np.array_equal(proj.evaluate_batch(b2, n2), arr[:, 2])
    assert proj.evaluate(parse_parameter(arr[1], pt2)) == arr[1, 2]
    b3, n3 = parse_parameter_batch([parse_parameter(m, pt) for m in mus], pt)
    assert n3 == 11 and np.array_equal(b3['diffusion'][:, 0], mus)
    with pytest.raises(ValueError):
        parse_parameter([1.0, 2.0], pt)


def test_sharding_arithmetic():
    from pylrbms_b200.distributed import mu_slice, owner_rank, region_layout, subdomains_on_rank
    for S, world in ((64, 8), (64, 3), (5, 8), (256, 4)):
        owners = [owner_rank(s, S, world) for s in range(S)]
        assert owners == sorted(owners) and set(owners) <= set(range(world))          # contiguous strips
        assert sum(len(subdomains_on_rank(S, r, world)) for r in range(world)) == S
    for n, world in ((10000, 8), (7, 3), (1000000, 8), (3, 8)):
        cuts = [mu_slice(n, r, world) for r in range(world)]
        assert cuts[0][0] == 0 and cuts[-1][1] == n and all(cuts[r][1] == cuts[r + 1][0] for r in range(world - 1))
        assert max(b - a for a, b in cuts) - min(b - a for a, b in cuts) <= 1
    pending = [(0, 4), (1, 3), (0, 2), (2, 5), (1, 1)]
    offsets, starts = region_layout(pending, 3)
    # equal strides (largest region, 6 doubles, rounded up to 32) so that the exchange is one in-place all-gather
    assert list(starts) == [0, 32, 64, 96] and list(offsets) == [0, 32, 4, 64, 35]
    offsets1, starts1 = region_layout(pending, 1) if False else region_layout([(0, 4), (0, 3)], 1)
    assert list(starts1) == [0, 7] and list(offsets1) == [0, 4]                    # single rank: tight packing


def test_fixture_structure_matches_appendix_b():
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases
    data = assemble_block_swipdg((3, 2), 4)
    S = data.num_subdomains
    assert S == 6 and data.Q == 2 and data.coefficients == ['1.', 'diffusion']
    for i in range(S):
        assert i in data.neighborhoods[i] and data.neighborhoods[i] == sorted(data.neighborhoods[i])
        assert data.n[i] == 6 * 16
        for q in range(2):
            assert (i, i) in data.lhs[q]
            for j in data.neighbors[i]:
                C = data.lhs[q][(i, j)]
                # coupling blocks are populated only on interface-element rows (discretize...:560-561)
                assert 0 < np.count_nonzero(np.diff(C.indptr)) < data.n[i] / 2
                assert abs(C - data.lhs[q][(j, i)].T).max() < 1e-14           # symmetric IPDG
        for k in data.neighborhoods[i]:
            assert data.oi[(k, i)].shape == (data.n[i], data.n[k])
            assert data.fr[0][(k, i)].shape == (data.m[i], data.n[k])
        assert data.div[i].shape == (data.n[i], data.m[i]) and data.bb[i].shape == (data.m[i], data.m[i])
    bases = make_local_bases(data, [3, 4, 5, 6, 7, 8], seed=0)
    for i, V in enumerate(bases):
        G = V @ (data.energy[i] @ V.T)
        assert np.abs(G - np.eye(V.shape[0])).max() < 1e-10


def test_bench_flop_model_matches_survey():
    sys.path.insert(0, ROOT)
    import bench
    nbh = []
    for s_ in range(64):
        ix, iy = s_ % 8, s_ // 8
        nbh.append(sorted([s_] + [s_ - 8] * (iy > 0) + [s_ - 1] * (ix > 0) + [s_ + 1] * (ix < 7) + [s_ + 8] * (iy < 7)))
    fl = bench.survey_flops_model([20] * 64, nbh, 2, 179)
    assert fl['n_red'] == 1280 and fl['blocks'] == 288 and fl['half_bandwidth'] == 180      # SURVEY.md section 8d, C2 row
    assert abs(fl['solve'] - (0.46e6 + 41.5e6 + 0.92e6)) < 0.1e6


@pytest.mark.parametrize('n_mu,n_red', [(7, 5), (10000, 1280)])
def test_bench_dump_outputs(tmp_path, n_mu, n_red):
    """``bench.py --dump-outputs``: float64 .npy files under 64 MB in all; above the budget the same seeded parameter sample
    every time, rows consistent with the batch they were taken from."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    mus = np.linspace(0.1, 1.0, n_mu)
    u = torch.arange(n_mu * n_red, dtype=torch.float64).reshape(n_mu, n_red)
    eta = torch.from_numpy(mus ** 2)
    info = torch.zeros(n_mu, dtype=torch.int32)
    mx, am = eta.max().reshape(1), eta.argmax().reshape(1)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), mus, u, eta, info, mx, am)
    names = sorted(p.name for p in (tmp_path / 'a').iterdir())
    assert names == ['eta.npy', 'eta_max.npy', 'index.npy', 'info.npy', 'mu.npy', 'u.npy']
    assert sum((tmp_path / 'a' / n).stat().st_size for n in names) <= 64 << 20
    out = {n[:-4]: np.load(tmp_path / 'a' / n) for n in names}
    for n in names:
        assert out[n[:-4]].dtype == np.float64 and np.array_equal(out[n[:-4]], np.load(tmp_path / 'b' / n))
    idx = out['index'].astype(np.int64)
    assert (len(idx) == n_mu) == (n_mu * n_red * 8 < bench.DUMP_BYTES) and np.all(np.diff(idx) > 0)
    assert np.array_equal(out['u'], u.numpy()[idx]) and np.array_equal(out['mu'], mus[idx])
    assert np.array_equal(out['eta'], mus[idx] ** 2) and not out['info'].any()
    assert list(out['eta_max']) == [1.0, n_mu - 1]


def test_synthetic_3d_fixture_structure():
    """The seeded synthetic operator set with 3D structure (config C4 shape): symmetry and definiteness where the hot path
    relies on them, interface-only coupling blocks, six-neighbour subdomain graph, determinism by seed."""
    import scipy.sparse as sp
    from pylrbms_b200.synthetic_fixture import make_random_local_bases, synthetic_block_operators
    data = synthetic_block_operators((3, 2, 2), (2, 2, 2), seed=5)
    again = synthetic_block_operators((3, 2, 2), (2, 2, 2), seed=5)
    other = synthetic_block_operators((3, 2, 2), (2, 2, 2), seed=6)
    S = data.num_subdomains
    assert S == 12 and data.Q == 2 and max(len(nb) for nb in data.neighborhoods) == 5      # 3x2x2: at most 4 face neighbours
    assert synthetic_block_operators((3, 3, 3), (1, 1, 1), seed=1).neighborhoods[13] == [4, 10, 12, 13, 14, 16, 22]
    for q in range(2):
        for key, M in data.lhs[q].items():
            assert (abs(M - again.lhs[q][key])).nnz == 0
            i, j = key
            assert abs(M - data.lhs[q][(j, i)].T).max() == 0.0                               # A_q[j, i] = A_q[i, j]^T
    assert abs(data.lhs[0][(0, 0)] - other.lhs[0][(0, 0)]).max() > 0
    # coupling blocks: non-zero rows only (interface cells), fewer than the diagonal block has
    for (i, j), M in data.lhs[0].items():
        if i != j:
            rows = np.unique(M.nonzero()[0])
            assert 0 < len(rows) < M.shape[0]
    # A(mu) = A_0 + mu A_1 is SPD over the parameter range
    n = int(data.n.sum())
    off = np.concatenate([[0], np.cumsum(data.n)])
    for mu in data.parameter_range:
        A = np.zeros((n, n))
        for (i, j) in data.lhs[0]:
            A[off[i]:off[i + 1], off[j]:off[j + 1]] = (data.lhs[0][(i, j)] + mu * data.lhs[1][(i, j)]).toarray()
        assert np.abs(A - A.T).max() == 0.0 and np.linalg.eigvalsh(A).min() > 0.0
    for i in range(S):
        for M in (data.l2[i], data.energy[i], data.elliptic[i]):
            assert abs(M - M.T).max() <= 1e-15 and np.linalg.eigvalsh(M.toarray()).min() > 0.0
        assert abs(data.bb[i] - data.bb[i].T).max() == 0.0
        assert abs(data.aa[0][1][i] - data.aa[1][0][i].T).max() == 0.0
        assert data.div[i].shape == (data.n[i], data.m[i]) and data.ab[1][i].shape == (data.n[i], data.m[i])
        for k in data.neighborhoods[i]:
            assert data.oi[(i, k)].shape == (data.n[k], data.n[i])
            assert data.fr[1][(i, k)].shape == (data.m[k], data.n[i])
    # bases: orthonormal in the local energy product, shape functions first
    bases = make_random_local_bases(data, [3 + (i % 4) for i in range(S)], seed=2)
    for i, V in enumerate(bases):
        G = V @ (data.energy[i] @ V.T)
        assert np.abs(G - np.eye(len(V))).max() < 1e-10


def test_peer_staging_offsets_and_halves(monkeypatch):
    """The address arithmetic of the peer-memory exchange, run on host memory: three simulated ranks, the exchange kernel
    replaced by ``memmove`` to the same destination addresses, several exchanges in a row (alternating staging halves) with
    fresh data each time.  (The kernel itself and the real symmetric memory are covered on the GPU.)"""
    import ctypes as C

    import torch

    from pylrbms_b200 import _lib
    from pylrbms_b200.distributed import PeerStaging, region_layout
    world = 3
    pending = [(0, 40), (1, 70), (1, 3), (2, 11)]
    _, starts = region_layout(pending, world)
    total = int(starts[-1])
    assert all(int(x) % 32 == 0 for x in starts)
    capacity = total + 64
    bufs = [torch.full((2 * capacity,), -7.0, dtype=torch.float64) for _ in range(world)]

    class FakeLib:
        calls = 0

        @staticmethod
        def lrbms_peer_push(h, src, n_bytes, n_dst, dst_arr, multicast, stream):
            assert multicast == 0 and n_dst == world - 1 and n_bytes % 16 == 0
            dsts = C.cast(dst_arr, C.POINTER(C.c_uint64))
            for d in range(n_dst):
                C.memmove(dsts[d], src.value, n_bytes)
            FakeLib.calls += 1
            return 0

    class FakeHandle:
        lib, h = FakeLib, None

        @staticmethod
        def check(rc):
            assert rc == 0

    monkeypatch.setattr(_lib, 'current_stream_ptr', lambda: C.c_void_p(0))
    stagings = []
    for r in range(world):
        st = object.__new__(PeerStaging)
        st.capacity, st.buf, st.rank, st.world = capacity, bufs[r], r, world
        st.peer_ptrs, st.multicast_ptr, st.exchanges = [b.data_ptr() for b in bufs], 0, 0
        stagings.append(st)
    for it in range(5):
        outs = []
        for r in range(world):
            out = torch.zeros(total, dtype=torch.float64)
            out[int(starts[r]):int(starts[r + 1])] = torch.arange(int(starts[r + 1] - starts[r]), dtype=torch.float64) + 1000 * r + 10000 * it
            outs.append(out)
        halves = [stagings[r]._push(FakeHandle, outs[r], starts) for r in range(world)]
        assert halves == [it & 1] * world
        for r in range(world):
            stagings[r]._collect(outs[r], starts, halves[r])
        for r in range(1, world):
            assert torch.equal(outs[r], outs[0])
        for r in range(world):
            seg = outs[0][int(starts[r]):int(starts[r + 1])]
            assert seg[0] == 1000 * r + 10000 * it and seg[-1] == seg[0] + len(seg) - 1
    assert FakeLib.calls == 5 * world
    # a rank never writes its own staging buffer, and nothing lands outside the two halves' used parts
    for r in range(world):
        own = bufs[r].view(2, capacity)[:, int(starts[r]):int(starts[r + 1])]
        assert bool((own == -7.0).all()) and bool((bufs[r].view(2, capacity)[:, total:] == -7.0).all())
