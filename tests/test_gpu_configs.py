"""Parity at the configurations BASELINE.json names, through the public API, against the oracle (1e-10, energy norm for
the solutions):

* C1  OS2015, 4 x 4 subdomains, 16 x 16 cells (n_i = 1 536), N = 8              -- everything
* C2  OS2015, 8 x 8 subdomains, 32 x 32 cells (n_i = 6 144), N = 20             -- everything, incl. ``sweep_into``'s chunks
* C3  high-contrast (1e6) SPE10-like field, 4 x 4 subdomains                     -- everything
      the same field on 16 x 16 subdomains (n_red = 5 120: band solver)          -- every reduced block; solves against a dense
      LU of the oracle's unblocked system operator.  The oracle's full ``reduce()`` cannot run at this size: the reference
      design stores every estimator operator as an unblocked dense ``n_red x Q n_red`` matrix (SURVEY.md row a10), 256 x 6 of
      them here.
* the reference's published indicator norms (``scripts/linearelliptic_block_swipdg_decomp.py:41-43``) through the CUDA
  fine-scale estimator.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-10


def _models(shape, cells, N, seed, problem=None):
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases
    from pylrbms_b200 import discretize, LRBMSReductor
    from oracle import lrbms_oracle as O
    data = assemble_block_swipdg(shape, cells, problem=problem)
    bases = make_local_bases(data, N, seed=seed)
    bd = {'domain_%d' % i: bases[i] for i in range(data.num_subdomains)}
    red_ref = O.LRBMSReductor(O.build_discretization(data), bases=bd)
    red = LRBMSReductor(discretize(data)[0], bases=bd)
    return data, red, red_ref


def _full_parity(data, red, red_ref, n_mu=8):
    from oracle.parity import assert_parity, compare_online, reference_online
    rd, rd_ref = red.reduce(), red_ref.reduce()
    lo, hi = data.parameter_range
    mus = np.linspace(lo, hi, n_mu)
    worst, n = assert_parity(rd, rd_ref, mus, RTOL)
    # the batched device entry point with host buffers (what bench.py's e2e leg calls)
    import torch
    u_host = torch.empty((n_mu, rd.n_red), dtype=torch.float64).pin_memory()
    eta_host = torch.empty(n_mu, dtype=torch.float64).pin_memory()
    assert rd.sweep_into(mus, u_host, eta_host) == 0
    errs = compare_online(rd, rd_ref, mus, U=u_host.numpy(), eta=eta_host.numpy())
    assert errs['u_energy'] <= RTOL and errs['eta'] <= RTOL, errs
    return rd, rd_ref, worst


def test_c1_os2015_4x4(handle):
    data, red, red_ref = _models((4, 4), 16, 8, 1001)
    rd, _, worst = _full_parity(data, red, red_ref, n_mu=16)
    assert rd.n_red == 128 and rd.solve_kernel_name == 'solve_kernel_v2'
    print('C1 worst rel err', worst)


def test_c2_os2015_8x8(handle):
    data, red, red_ref = _models((8, 8), 32, 20, 1002)
    rd, rd_ref, worst = _full_parity(data, red, red_ref, n_mu=8)
    assert rd.n_red == 1280 and rd.solve_kernel_name == 'solve_kernel_v2'
    # a batch large enough for sweep_into's four-chunk pipeline (>= 32 parameters per resident CTA); sampled check
    from oracle.parity import compare_online
    import torch
    rng = np.random.default_rng(5)
    n_mu = 32 * rd.online_plan.handle.sm_count + 77
    mus = rng.uniform(0.1, 1.0, n_mu)
    u_host = torch.empty((n_mu, rd.n_red), dtype=torch.float64).pin_memory()
    eta_host = torch.empty(n_mu, dtype=torch.float64).pin_memory()
    assert rd.sweep_into(mus, u_host, eta_host) == 0
    pick = np.concatenate([[0, n_mu - 1], rng.choice(n_mu, 6, replace=False)])
    errs = compare_online(rd, rd_ref, mus[pick], U=u_host.numpy()[pick], eta=eta_host.numpy()[pick])
    assert errs['u_energy'] <= RTOL and errs['eta'] <= RTOL, errs
    print('C2 worst rel err', worst, errs)


def test_c3_spe10_contrast_4x4(handle):
    from pylrbms_b200.swipdg_fixture import spe10_like_problem
    data, red, red_ref = _models((4, 4), 16, 20, 1003, problem=spe10_like_problem(seed=1003, contrast=1e6))
    rd, _, worst = _full_parity(data, red, red_ref, n_mu=8)
    print('C3 (4x4) worst rel err', worst)


def test_c3_spe10_contrast_16x16(handle):
    from pylrbms_b200.swipdg_fixture import spe10_like_problem
    from pylrbms_b200.operators import LincombOperator
    from oracle import lrbms_oracle as O
    from oracle.pymor_like import LincombOperator as RefLincomb, unblock
    data, red, red_ref = _models((16, 16), 16, 20, 1003, problem=spe10_like_problem(seed=1003, contrast=1e6))
    rd = red.reduce()
    assert rd.n_red == 5120 and rd.solve_kernel_name == 'band_update_kernel'
    red_ref.image_bases(unblocked=False)
    d_ref = red_ref.d
    worst = 0.0
    for name in list(d_ref.operators) + list(d_ref.products):
        got = rd.operators[name] if name in rd.operators else rd.products[name]
        gots = got.operators if isinstance(got, LincombOperator) else [got]
        ref_op = d_ref.operators[name] if name in d_ref.operators else d_ref.products[name]
        for q, g in enumerate(gots):
            ref = O.reduced_blocks(red_ref, name, q if isinstance(ref_op, RefLincomb) else None)
            gb = g.blocks()
            scale = max(np.abs(v).max() for v in ref.values())
            for key, B in ref.items():
                err = np.abs(gb[key] - B).max() / scale
                worst = max(worst, err)
                assert err <= RTOL, '{} block {}: rel err {:.3e}'.format(name, key, err)
    # online: the oracle's unblocked system operator and right-hand side, dense LU per parameter as the reference does
    op_ref = unblock(O.project_system(d_ref.operator, red_ref.bases, red_ref.bases))
    rhs_ref = unblock(O.project_system(d_ref.rhs, red_ref.bases, red_ref.bases))
    lo, hi = data.parameter_range
    mus = np.linspace(lo, hi, 8)
    U, eta, parts, ind = rd.sweep(mus, decompose=True)
    for k, mu in enumerate(mus):
        mu_p = rd.parse_parameter(mu)
        A = np.asarray(op_ref.assemble(mu_p).matrix)
        f = np.asarray(rhs_ref.as_source_array(mu_p).data[0])
        u_ref = np.linalg.solve(A, f)
        e = U.data[k] - u_ref
        assert np.sqrt(e @ A @ e) <= RTOL * np.sqrt(u_ref @ A @ u_ref), 'mu {}'.format(mu)
    print('C3 (16x16) worst block rel err', worst)
    # the estimator on all 256 subdomains against the exact value of the GPU's own reduced operators and u, and the
    # estimator constants against the oracle's: with the blocks and solutions above this closes the chain to eta
    _check_estimator(rd, mus, U, eta, parts, ind, range(data.num_subdomains), 'C3 (16x16)')
    est, est_ref = rd.estimator, d_ref.estimator
    rf2_ref = np.asarray(est_ref.local_eta_rf_squared, dtype=np.float64)
    assert np.all(np.abs(est.local_eta_rf_squared - rf2_ref) <= 1e-13 * np.abs(rf2_ref))
    rs_ref = (1.0 / np.pi ** 2) / np.asarray(est_ref.min_diffusion_evs) * np.asarray(est_ref.subdomain_diameters) ** 2
    assert np.all(np.abs(est.r_scale() - rs_ref) <= 1e-15 * rs_ref)
    for mu in mus:
        mu_p, mu_r = rd.parse_parameter(mu), d_ref.parse_parameter(mu)
        for f in ('alpha', 'gamma'):
            for bar, bar_ref in ((est.mu_bar, est_ref.mu_bar), (est.mu_hat, est_ref.mu_hat)):
                got = getattr(est, f)(est.lambda_coeffs, mu_p, bar)
                ref = getattr(est_ref, f)(est_ref.lambda_coeffs, mu_r, bar_ref)
                assert abs(got - ref) <= 1e-15 * abs(ref), (f, mu)


def _check_estimator(rd, mus, U, eta, parts, ind, subdomains, what):
    """The parts of ``rd.sweep(decompose=True)`` on ``subdomains`` within the kernel's rounding bound gamma_K S of their exact
    value (oracle/exact_forms.py, tests/test_gpu_estimator.py); eta and the indicators of every subdomain as the float64
    combine of the kernel's own parts (estimators.py:99-109)."""
    from test_gpu_estimator import EPS, PARTS, gamma, model_K, model_exact
    subs = list(subdomains)
    forms, ex = model_exact(rd, mus, U.data, subs)
    K = model_K(rd, forms, subs)
    worst = {}
    for k, name in enumerate(PARTS):
        got = np.asarray(parts[k])[subs]
        err = np.abs(got - ex[name])
        assert np.all(err <= gamma(K[k][:, None]) * ex['S_' + name]), name
        worst[name] = float((err / (EPS * ex['S_' + name])).max())
    est = rd.estimator
    nc, rdf = np.asarray(parts[0]), np.asarray(parts[1]) + np.asarray(parts[2])
    for k, mu in enumerate(mus):
        mu_p = rd.parse_parameter(mu)
        lam = est.lambda_coeffs
        a_bar, g_bar, a_hat = est.alpha(lam, mu_p, est.mu_bar), est.gamma(lam, mu_p, est.mu_bar), est.alpha(lam, mu_p, est.mu_hat)
        e = (np.sqrt(g_bar) * np.sqrt(np.sum(nc[:, k] ** 2)) + np.sqrt(np.sum(rdf[:, k] ** 2)) / np.sqrt(a_hat)) / np.sqrt(a_bar)
        assert abs(eta[k] - e) <= 8 * EPS * e
        i_ref = (2.0 / a_bar) * (g_bar * nc[:, k] ** 2 + (1.0 / a_hat) * rdf[:, k] ** 2)
        assert np.all(np.abs(np.asarray(ind)[:, k] - i_ref) <= 8 * EPS * np.abs(i_ref))
    print(what, 'estimator |got - exact| / (eps S):', worst)


def test_published_indicator_norms_cuda(handle):
    """``scripts/linearelliptic_block_swipdg_decomp.py:41-43`` through the CUDA fine-scale estimator (see
    tests/test_reference_anchor.py for what the three numbers are and why the tolerances are 1 % / 15 %)."""
    from test_reference_anchor import PUBLISHED, fom_solution
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg
    from pylrbms_b200 import discretize
    from oracle import lrbms_oracle as O
    data = assemble_block_swipdg((4, 4), 2)
    d_ref = O.build_discretization(data)
    U_ref, u = fom_solution(data, d_ref, 1.0)
    d, _ = discretize(data)
    off = np.concatenate([[0], np.cumsum(data.n)])
    subs = d.solution_space.subspaces
    U = d.solution_space.make_array([subs[i].from_data(u[None, off[i]:off[i + 1]]) for i in range(data.num_subdomains)])
    eta, (nc, r, df), _ = d.estimate(U, mu=1.0, decompose=True)
    eta_ref, (nc_ref, r_ref, df_ref), _ = d_ref.estimate(U_ref, 1.0, decompose=True)
    assert abs(eta - eta_ref) <= 1e-9 * abs(eta_ref)
    got = {'nc': np.sqrt(np.sum(nc)), 'r': np.sqrt(np.sum(r)), 'df': np.sqrt(np.sum(df))}
    assert abs(got['r'] - PUBLISHED['r']) <= 0.01 * PUBLISHED['r'], got
    assert abs(got['nc'] - PUBLISHED['nc']) <= 0.15 * PUBLISHED['nc'], got
    assert abs(got['df'] - PUBLISHED['df']) <= 0.15 * PUBLISHED['df'], got


def test_c4_3d_8x8x8_N40_full_size_online(handle):
    """BASELINE configs[3]: 3D structure (six face neighbours), 8 x 8 x 8 subdomains, local basis size 40 -> block-sparse
    reduced system with 20 480 dofs, scalar half bandwidth 2 599.  The reduced model comes from the real offline path on
    seeded synthetic operators with a small fine grid (n_i = 192: the online cost does not depend on n_i); the online solve runs
    at FULL size on the band solver.  The reference's dense path cannot run here (one unblocked operator is 3.4 GB and it
    stores hundreds), so the check is against an independent CPU solver on the same block-sparse reduced operator
    (SciPy's SuperLU): energy-norm error and residual at 1e-10, plus bit-identical results for a different batch composition.
    The estimator runs on 17 parameters and is held to the exact value of its forms on a sample of 16 subdomains."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spl
    from pylrbms_b200 import LRBMSReductor, discretize
    from pylrbms_b200.synthetic_fixture import make_random_local_bases, synthetic_block_operators
    data = synthetic_block_operators((8, 8, 8), (3, 4, 4), seed=1004)
    bases = make_random_local_bases(data, 40, seed=1004)
    S = data.num_subdomains
    rd = LRBMSReductor(discretize(data)[0], bases={'domain_%d' % i: bases[i] for i in range(S)}).reduce()
    assert rd.n_red == 20480 and rd.solve_kernel_name == 'band_update_kernel' and rd.half_bandwidth == 2599
    lo, hi = data.parameter_range
    # 17 parameters: the estimator runs 16 per CTA here (seven-member neighbourhoods of 280 dofs), so two tiles
    mus17 = np.linspace(lo, hi, 17)
    U17, eta17, parts, ind = rd.sweep(mus17, decompose=True)
    assert int(rd.online_plan.info(9)) == 16
    # a sample of subdomains: corners, edges, faces, interior (seven-member neighbourhoods)
    at = lambda x, y, z: (z * 8 + y) * 8 + x
    sample = [at(0, 0, 0), at(7, 7, 7), at(7, 0, 0), at(0, 7, 7), at(3, 0, 0), at(0, 4, 7), at(7, 5, 0), at(2, 7, 7),
              at(0, 3, 4), at(4, 0, 5), at(5, 6, 7), at(7, 2, 3), at(3, 3, 3), at(4, 4, 4), at(1, 6, 2), at(5, 2, 6)]
    _check_estimator(rd, mus17, U17, eta17, parts, ind, sample, 'C4 (8x8x8)')
    pick = [0, 8, 16]
    mus = mus17[pick]
    Ud, eta = np.asarray(U17.data)[pick], eta17[pick]
    # the block-sparse reduced operator on the host
    offs = np.concatenate([[0], np.cumsum(rd.block_dims)])
    mats = []
    for op in rd.operator.operators:
        rows, cols, vals = [], [], []
        for (i, j), B in op.blocks().items():
            r, c = np.meshgrid(np.arange(offs[i], offs[i + 1]), np.arange(offs[j], offs[j + 1]), indexing='ij')
            rows.append(r.ravel()); cols.append(c.ravel()); vals.append(B.ravel())
        mats.append(sp.csc_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(rd.n_red,) * 2))
    f_terms = [o.to_dense()[0] for o in rd.rhs.operators]
    for k in (0, 2):
        th = rd.thetas([mus[k]])[0]
        A = sum(t * M for t, M in zip(th[:len(mats)], mats)).tocsc()
        f = sum(t * v for t, v in zip(th[len(mats):], f_terms))
        lu = spl.splu(A)
        u_ref = lu.solve(f)
        u_ref += lu.solve(f - A @ u_ref)                                # one step of refinement on the CPU side
        e = Ud[k] - u_ref
        assert np.sqrt(e @ (A @ e)) <= RTOL * np.sqrt(u_ref @ (A @ u_ref))
        assert np.linalg.norm(A @ Ud[k] - f) <= RTOL * np.linalg.norm(f) * 100
    U2, eta2 = rd.sweep(mus[[2, 0]])
    assert np.array_equal(U2.data[0], Ud[2]) and np.array_equal(U2.data[1], Ud[0]) and eta2[0] == eta[2]
