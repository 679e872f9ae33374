"""The fine-scale solve ``d.solve(mu)`` / ``d.solve_batch(mus)`` (``lrbms_affine_pcg_solve``, mu-batched Jacobi CG):

1. parity with a direct solve (SciPy) in the energy norm of A(mu), 1e-10, on 2D / 3D / high-contrast fixtures and at C2 size;
2. every parameter's result bit-identical whatever batch it is solved in (size, position, chunking, stale shared memory);
3. failures reported per parameter: a non-definite column gets status 2 without disturbing its neighbours; an iteration
   budget nobody meets raises with status 1 and returns nothing;
4. the true error of the reduced model, |||u_h - R u_N|||, as the oracle computes it;
5. the reference's published indicator norms with u_h from the GPU solve.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spl

pytestmark = pytest.mark.gpu

RTOL = 1e-10


def _theta(d, mus):
    from pylrbms_b200.parameters import theta_matrix
    return theta_matrix(list(d.operator.coefficients) + list(d.rhs.coefficients), mus, d.parameter_type)


def _host_system(data, th):
    """A(mu) (CSC) and b(mu) on the host from the fixture's blocks."""
    S = data.num_subdomains
    mats = []
    for q in range(data.Q):
        blocks = [[None] * S for _ in range(S)]
        for (i, j), M in data.lhs[q].items():
            blocks[i][j] = M
        mats.append(sp.bmat(blocks, format='csc'))
    A = mats[0] * th[0]
    for q in range(1, data.Q):
        A = A + mats[q] * th[q]
    return A.tocsc(), th[data.Q] * np.concatenate(data.rhs)


def _energy_rel_err(A, u, u_ref):
    e = u - u_ref
    return np.sqrt(e @ (A @ e)) / np.sqrt(u_ref @ (A @ u_ref))


def _fixture(name):
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, spe10_like_problem
    from pylrbms_b200.synthetic_fixture import synthetic_block_operators
    if name == 'c1':
        return assemble_block_swipdg((4, 4), 16), 16
    if name == '3x2':
        return assemble_block_swipdg((3, 2), 4), 6
    if name == '3d':
        return synthetic_block_operators((3, 2, 2), (2, 2, 2), seed=1004), 6
    if name == 'spe10_c50':
        return assemble_block_swipdg((4, 4), 16, problem=spe10_like_problem(seed=1003, contrast=50)), 6
    raise KeyError(name)


@pytest.mark.parametrize('name', ['c1', '3x2', '3d', 'spe10_c50'])
def test_fom_solve_matches_spsolve(handle, name):
    from pylrbms_b200 import discretize
    data, n_mu = _fixture(name)
    d, _ = discretize(data)
    lo, hi = data.parameter_range
    mus = np.linspace(lo, hi, n_mu)
    U = d.solve_batch(mus)
    info = d.last_solve_info
    assert len(U) == n_mu and np.all(info['status'] == 0) and np.all(info['relative_residual'] <= 1e-9)
    Ud = U.data
    for k, mu in enumerate(mus):
        A, b = _host_system(data, _theta(d, [mu])[0])
        u_ref = spl.spsolve(A, b)                    # the oracle's fine-scale solve (tests/test_reference_anchor.py)
        err = _energy_rel_err(A, Ud[k], u_ref)
        assert err <= RTOL, (name, mu, err)
    print(name, 'iterations', info['iterations'].min(), info['iterations'].max(), 'relres', info['relative_residual'].max())


def test_fom_solve_c2_matches_splu(handle):
    from pylrbms_b200 import discretize
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg
    data = assemble_block_swipdg((8, 8), 32)
    d, _ = discretize(data)
    assert d.solution_space.dim == 393216
    mus = np.array([0.1, 0.4, 0.7, 1.0])
    Ud = d.solve_batch(mus).data
    assert np.all(d.last_solve_info['status'] == 0)
    for k, th in enumerate(_theta(d, mus)):
        A, b = _host_system(data, th)
        u_ref = spl.splu(A).solve(b)
        assert _energy_rel_err(A, Ud[k], u_ref) <= RTOL, mus[k]
    print('C2 iterations', d.last_solve_info['iterations'], 'relres', d.last_solve_info['relative_residual'])


def test_fom_solve_is_batch_independent(handle):
    """d.solve(mu) equals its row of d.solve_batch bit for bit: batch sizes 1, 31, 32, 33, 70, permuted batches, a chunk
    budget that splits the batch, and after the shared memory of every SM was filled with NaNs."""
    from pylrbms_b200 import discretize
    from pylrbms_b200._lib import current_stream_ptr
    from pylrbms_b200.kernels import affine_pcg_workspace_bytes
    data, _ = _fixture('3x2')
    d, _ = discretize(data)
    lo, hi = data.parameter_range
    rng = np.random.default_rng(7)
    pool = rng.uniform(lo, hi, 70)
    solo = {k: d.solve(pool[k]).data[0] for k in (0, 1, 30, 31, 32, 33, 69)}
    n = d.solution_space.dim
    for size in (1, 31, 32, 33, 70):
        for permute, budget in ((False, None), (True, None), (True, affine_pcg_workspace_bytes(n, 32) * 10 // 32)):
            idx = np.arange(size)
            if permute:
                idx = rng.permutation(idx)
            if budget is not None:
                d.fom_workspace_budget = budget                     # chunks of 10 parameters
            try:
                Ud = d.solve_batch(pool[idx]).data
            finally:
                d.__dict__.pop('fom_workspace_budget', None)
            for pos, k in enumerate(idx):
                if k in solo:
                    assert np.array_equal(Ud[pos], solo[k]), (size, permute, budget, k, pos)
    handle.check(handle.lib.lrbms_debug_poison_shared(handle.h, current_stream_ptr()))
    Ud = d.solve_batch(pool[[33, 0]]).data
    assert np.array_equal(Ud[0], solo[33]) and np.array_equal(Ud[1], solo[0])


def test_affine_pcg_status_per_parameter(handle):
    """C ABI: the coefficient row (-1, 0, 1) makes A = -A_0 negative definite: that column stops with status 2 in the
    first iteration, every other column converges to the bits of its solo solve."""
    import torch
    from pylrbms_b200 import discretize
    from pylrbms_b200.kernels import affine_pcg_solve
    data, _ = _fixture('3x2')
    d, _ = discretize(data)
    pattern, values, rhs = d.affine_system(range(data.num_subdomains))
    n = pattern.shape[0]
    theta = _theta(d, [0.2, 0.5, 0.9, 1.0])
    theta[1] = [-1.0, 0.0, 1.0]
    assert theta.shape[1] == 3
    th = torch.from_numpy(theta).cuda()
    x = torch.zeros((n, 4), dtype=torch.float64, device='cuda')
    _, it, rr, st = affine_pcg_solve(pattern, values, rhs, th, x, 1e-9, 10 * n, 3)
    assert list(st) == [0, 2, 0, 0] and it[1] == 0, (st, it)
    assert np.all(x[:, 1].cpu().numpy() == 0.0)                      # the frozen column was never written
    for k in (0, 2, 3):
        xs = torch.zeros((n, 1), dtype=torch.float64, device='cuda')
        _, it_s, rr_s, st_s = affine_pcg_solve(pattern, values, rhs, th[k:k + 1].contiguous(), xs, 1e-9, 10 * n, 3)
        assert st_s[0] == 0 and it_s[0] == it[k] and rr_s[0] == rr[k]
        assert torch.equal(xs[:, 0], x[:, k])


def test_fom_solve_raises_when_not_converged(handle):
    from pylrbms_b200 import discretize
    from pylrbms_b200._lib import LrbmsError
    data, _ = _fixture('3x2')
    d, _ = discretize(data)
    mus = np.linspace(*data.parameter_range, 5)
    with pytest.raises(LrbmsError, match=r'parameter #0: status 1'):
        d.solve_batch(mus, inverse_options={'maxiter': 5})
    info = d.last_solve_info
    assert np.all(info['status'] == 1) and np.all(info['iterations'] == 5) and np.all(info['relative_residual'] > 1e-9)


def test_true_reduction_error_matches_oracle(handle):
    """|||d.solve(mu) - R rd.solve(mu)||| in the energy product (sum of local_energy_dg_product_i) at C1 with ragged bases."""
    from pylrbms_b200 import LRBMSReductor, discretize
    from pylrbms_b200.swipdg_fixture import make_local_bases
    from oracle import lrbms_oracle as O
    data, _ = _fixture('c1')
    S = data.num_subdomains
    sizes = [4 + (i % 7) for i in range(S)]
    bases = make_local_bases(data, sizes, seed=11)
    bd = {'domain_%d' % i: bases[i] for i in range(S)}
    d, _ = discretize(data)
    red, red_ref = LRBMSReductor(d, bases=bd), O.LRBMSReductor(O.build_discretization(data), bases=bd)
    rd, rd_ref = red.reduce(), red_ref.reduce()
    offs = np.concatenate([[0], np.cumsum(data.n)])

    def energy(v):
        return np.sqrt(sum(v[offs[i]:offs[i + 1]] @ (data.energy[i] @ v[offs[i]:offs[i + 1]]) for i in range(S)))

    for mu in np.linspace(*data.parameter_range, 4):
        u_h = d.solve(mu).data[0]
        err = energy(u_h - red.reconstruct(rd.solve(mu)).data[0])
        u_ref = spl.spsolve(*_host_system(data, _theta(d, [mu])[0]))
        err_ref = energy(u_ref - red_ref.reconstruct(rd_ref.solve(mu)).data[0])
        assert abs(err - err_ref) <= 1e-9 * energy(u_ref), (mu, err, err_ref)


def test_published_indicator_norms_from_gpu_solve(handle):
    """d.solve(1.0) + d.estimate reproduce the reference's printed indicator norms (tolerances of
    tests/test_reference_anchor.py) and the estimate of the SciPy solution to 1e-9."""
    from test_reference_anchor import PUBLISHED
    from pylrbms_b200 import discretize
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg
    data = assemble_block_swipdg((4, 4), 2)
    d, _ = discretize(data)
    U = d.solve(1.0)
    assert len(U) == 1 and d.last_solve_info['status'][0] == 0
    eta, (nc, r, df), _ = d.estimate(U, mu=1.0, decompose=True)
    got = {'nc': np.sqrt(np.sum(nc)), 'r': np.sqrt(np.sum(r)), 'df': np.sqrt(np.sum(df))}
    assert abs(got['r'] - PUBLISHED['r']) <= 0.01 * PUBLISHED['r'], got
    assert abs(got['nc'] - PUBLISHED['nc']) <= 0.15 * PUBLISHED['nc'], got
    assert abs(got['df'] - PUBLISHED['df']) <= 0.15 * PUBLISHED['df'], got
    A, b = _host_system(data, _theta(d, [1.0])[0])
    u = spl.spsolve(A, b)
    off = np.concatenate([[0], np.cumsum(data.n)])
    subs = d.solution_space.subspaces
    U_sp = d.solution_space.make_array([subs[i].from_data(u[None, off[i]:off[i + 1]]) for i in range(data.num_subdomains)])
    eta_sp = d.estimate(U_sp, mu=1.0)
    assert abs(eta - eta_sp) <= 1e-9 * abs(eta_sp)
