"""Elimination order of the subdomains in the shared-memory window solve (lrbms_symbolic_reorder).

CPU: the symbolic phase picks the Cuthill-McKee (anti-diagonal) order on the 8 x 8 subdomain grid and keeps the given order
where no other order is strictly cheaper or fits; perm / iperm / row_map are consistent permutations; the permuted schedule
replays to a Cholesky factor of P A P^T.  GPU: plans that factor in a permuted order solve the unpermuted system to 1e-12 in
the energy norm, write u in the caller's row order, report a failed pivot as the caller's row, and stay bit-reproducible
across batch order."""
import numpy as np
import pytest

from test_gpu_kernels import _make_online_plan, _random_reduced_system, _run_sweep

B200_OPTIN = 232448          # shared memory per block (opt-in) of sm_100


def _grid_couplings(sx, sy, diagonal=False):
    out = []
    for s in range(sx * sy):
        ix, iy = s % sx, s // sx
        if ix + 1 < sx: out.append((s + 1, s))
        if iy + 1 < sy: out.append((s + sx, s))
        if diagonal and ix + 1 < sx and iy + 1 < sy: out.append((s + sx + 1, s))
    return out


def _relabel(couplings, perm):
    """Subdomain perm[k] gets label k."""
    lab = np.argsort(perm)
    return [(int(max(lab[i], lab[j])), int(min(lab[i], lab[j]))) for (i, j) in couplings]


def _blocks(S, couplings):
    blocks = [(i, i) for i in range(S)]
    for (i, j) in couplings:
        blocks += [(i, j), (j, i)]
    return blocks


def _symbolic(sizes, blocks):
    from pylrbms_b200._lib import Symbolic
    return Symbolic(np.asarray(sizes, dtype=np.int32), [b[0] for b in blocks], [b[1] for b in blocks])


# systems whose reordered schedule the GPU tests run: (name, subdomain count, sizes, couplings)
_RNG = np.random.default_rng(1)
# rows of a 6 x 6 grid in order, the subdomains of each row numbered in a random order (a fully random numbering has a
# factor window too wide for one SM in the given order, and AUTO decides on the given order)
_SCRAMBLE = np.concatenate([6 * r + _RNG.permutation(6) for r in range(6)])
CASES = {
    'c2': (64, [20] * 64, _grid_couplings(8, 8)),
    # ragged sizes, zero-size subdomain included
    'ragged_scrambled': (36, [int(x) for x in _RNG.integers(0, 30, 36)], _relabel(_grid_couplings(6, 6), _SCRAMBLE)),
    # not a 5-point grid: a triangulated 7 x 5 grid (each subdomain also couples to its lower-right diagonal neighbour)
    'triangulated': (35, [int(x) for x in _RNG.integers(5, 26, 35)], _grid_couplings(7, 5, diagonal=True)),
}


def test_cuthill_mckee_on_the_c2_grid(built_library):
    sym = _symbolic([20] * 64, _blocks(64, _grid_couplings(8, 8)))
    tiles0, pairs0 = sym.n_tiles, sym.n_pairs
    assert sym.order == 0 and list(sym.get(15)) == list(range(64))
    assert sym.reorder(2, B200_OPTIN - 1024) == 1
    perm = sym.get(15)
    # level sets of a breadth-first search from subdomain 0: the anti-diagonals ix + iy, each ordered by parent position
    levels = [int(p % 8 + p // 8) for p in perm]
    assert perm[0] == 0 and levels == sorted(levels)
    assert list(perm[:6]) == [0, 1, 8, 2, 9, 16]
    given, cm, rcm = sym.order_costs
    assert 0 < cm < given and rcm >= cm
    assert sym.n_tiles < tiles0 and sym.n_pairs < pairs0
    assert sym.n_tiles == 2634 and tiles0 == 3195
    assert sym.staggered == 1


def test_given_order_kept_when_nothing_is_cheaper(built_library):
    # a chain of subdomains in its natural order: Cuthill-McKee reproduces it, its reverse costs the same -> tie -> given
    S = 12
    sym = _symbolic([20] * S, _blocks(S, [(i + 1, i) for i in range(S - 1)]))
    assert sym.reorder(2, B200_OPTIN - 1024) == 0
    assert list(sym.get(15)) == list(range(S)) and list(sym.get(17)) == list(range(sym.n_red))
    # the C2 grid with no shared memory to spare: every candidate is rejected, the costs are still reported
    sym = _symbolic([20] * 64, _blocks(64, _grid_couplings(8, 8)))
    assert sym.reorder(2, 0) == 0
    assert all(c > 0 for c in sym.order_costs)
    # re-planning twice is refused
    from pylrbms_b200._lib import LrbmsError
    sym = _symbolic([20] * 64, _blocks(64, _grid_couplings(8, 8)))
    sym.reorder(2, B200_OPTIN - 1024)
    with pytest.raises(LrbmsError):
        sym.reorder(2, B200_OPTIN - 1024)


@pytest.mark.parametrize('name', sorted(CASES))
def test_permutation_round_trips_and_replays(built_library, name):
    S, sizes, couplings = CASES[name]
    sym = _symbolic(sizes, _blocks(S, couplings))
    sym.reorder(2, B200_OPTIN - 1024)
    assert sym.order in (1, 2), 'expected a reordered schedule for {}'.format(name)
    perm, iperm, row_map = sym.get(15), sym.get(16), sym.get(17)
    assert sorted(perm) == list(range(S)) and np.array_equal(perm[iperm], np.arange(S))
    assert np.array_equal(iperm[perm], np.arange(S))
    n = sym.n_red
    assert sorted(row_map) == list(range(n))
    # subdomains keep their rows contiguous, in their own order, at the position perm gives them
    off = np.concatenate([[0], np.cumsum(sizes)])
    expect = np.concatenate([np.arange(off[p], off[p + 1]) for p in perm])
    assert np.array_equal(row_map, expect)
    # replay the permuted schedule (left-looking 8x8 tiles) to a Cholesky factor of P A P^T
    rng = np.random.default_rng(9)
    A = np.zeros((n, n))
    for i in range(S):
        B = rng.standard_normal((sizes[i], sizes[i]))
        A[off[i]:off[i + 1], off[i]:off[i + 1]] = B @ B.T + 4.0 * max(1, sizes[i]) * np.eye(sizes[i])
    for (i, j) in couplings:
        B = 0.2 * rng.standard_normal((sizes[i], sizes[j]))
        A[off[i]:off[i + 1], off[j]:off[j + 1]] = B
        A[off[j]:off[j + 1], off[i]:off[i + 1]] = B.T
    npad, ntc, n_tiles = sym.n_pad, sym.n_tile_cols, sym.n_tiles
    Ap = np.eye(npad)
    Ap[:n, :n] = A[np.ix_(row_map, row_map)]
    col_ptr, row_idx, pair_ptr, pair_a, pair_b, a_map = (sym.get(k) for k in range(6))
    L = np.zeros((n_tiles, 8, 8))
    for J in range(ntc):
        for tgt in range(col_ptr[J], col_ptr[J + 1]):
            I = row_idx[tgt]
            T = Ap[8 * I:8 * I + 8, 8 * J:8 * J + 8].copy()
            assert a_map[tgt] >= 0 or not np.any(T)
            for p in range(pair_ptr[tgt], pair_ptr[tgt + 1]):
                T -= L[pair_a[p]] @ L[pair_b[p]].T
            if tgt == col_ptr[J]:
                Ljj = np.linalg.cholesky(T)
                L[tgt] = Ljj
            else:
                L[tgt] = np.linalg.solve(Ljj, T.T).T
    Ld = np.zeros((npad, npad))
    for J in range(ntc):
        for p in range(col_ptr[J], col_ptr[J + 1]):
            Ld[8 * row_idx[p]:8 * row_idx[p] + 8, 8 * J:8 * J + 8] = L[p]
    assert np.abs(Ld @ Ld.T - Ap).max() < 1e-12 * np.abs(Ap).max()


# ---------------------------------------------------------------------------------------------------------------------
#  GPU
# ---------------------------------------------------------------------------------------------------------------------
def _system(name, seed):
    S, sizes, couplings = CASES[name]
    rng = np.random.default_rng(seed)
    sysd = _random_reduced_system(rng, S, 1, sizes, couplings=couplings)
    return sysd, rng


def _thetas(rng, n_mu):
    return np.column_stack([np.ones(n_mu), rng.uniform(0.1, 1.0, n_mu), rng.uniform(0.5, 2.0, n_mu)])


def _energy_errors(sysd, theta, u):
    out = []
    for m in range(theta.shape[0]):
        A = theta[m, 0] * sysd['dense'][0] + theta[m, 1] * sysd['dense'][1]
        ref = np.linalg.solve(A, theta[m, 2] * sysd['rhs'][0])       # dense LU of the unpermuted system
        e = u[m] - ref
        out.append(np.sqrt(e @ A @ e) / np.sqrt(ref @ A @ ref))
    return np.array(out)


@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(CASES))
def test_reordered_solve_matches_dense_lu(handle, name):
    sysd, rng = _system(name, 31)
    plan, _ = _make_online_plan(handle, sysd)
    assert int(plan.info(6)) == 1, 'the window kernel must run for this test'
    n_mu = 300
    theta = _thetas(rng, n_mu)
    u, info = _run_sweep(handle, plan, sysd, theta, with_est=False)
    assert np.all(info == 0)
    err = _energy_errors(sysd, theta, u)
    assert err.max() <= 1e-12, 'worst energy-norm error {:.3e}'.format(err.max())


@pytest.mark.gpu
def test_u_layout_and_failed_pivot_row(handle):
    """One subdomain's diagonal block of the second operator term is strongly negative: for a large theta_1 the first
    non-positive pivot is the first row of that subdomain in the caller's numbering, whatever the elimination order."""
    sysd, rng = _system('c2', 32)
    s0 = 27
    off = sysd['off']
    sysd['dense'][1][off[s0]:off[s0 + 1], off[s0]:off[s0 + 1]] = -1.0e3 * np.eye(sysd['sizes'][s0])
    plan, _ = _make_online_plan(handle, sysd)
    theta = _thetas(rng, 6)
    theta[:, 1] = 1.0e-3                                              # positive definite
    good_u, good_info = _run_sweep(handle, plan, sysd, theta, with_est=False)
    assert np.all(good_info == 0)
    assert _energy_errors(sysd, theta, good_u).max() <= 1e-12        # u is in the caller's row order
    bad = theta.copy()
    bad[[1, 4], 1] = 10.0
    u, info = _run_sweep(handle, plan, sysd, bad, with_est=False)
    assert list(info[[1, 4]]) == [off[s0] + 1] * 2, info
    keep = [0, 2, 3, 5]
    assert np.all(info[keep] == 0) and np.array_equal(u[keep], good_u[keep])


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['c2', 'ragged_scrambled'])
def test_reordered_solve_is_bit_reproducible(handle, name):
    sysd, rng = _system(name, 33)
    plan, _ = _make_online_plan(handle, sysd)
    n_mu = 700
    theta = _thetas(rng, n_mu)
    u1, info1 = _run_sweep(handle, plan, sysd, theta, with_est=False)
    assert np.all(info1 == 0)
    for k in range(2):
        perm = rng.permutation(n_mu)[:[511, 97][k]]
        u2, _ = _run_sweep(handle, plan, sysd, theta[perm], with_est=False)
        assert np.array_equal(u2, u1[perm])
