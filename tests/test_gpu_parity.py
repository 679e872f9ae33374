"""Parity of the CUDA hot path with the CPU oracle (``oracle/``) on the same seeded inputs, through the public
Python API (which calls the C ABI).  FP64; tolerance 1e-10 relative (BASELINE.json north_star), measured relative
to the scale of each block / each quantity, never entry-wise on cancelling sums (SURVEY.md section 7 "hard parts").

Covered reference behaviour: ``LRBMSReductor.reduce()`` (reductor.py:33-73 -> every operator of
discretize...:581-770), ``rd.solve(mu)``, ``rd.estimate(U, mu, decompose=True)`` (estimators.py:45-130 with its
quirks), ``reductor.reconstruct`` / ``extend_basis_local``.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-10


def _setup(num_subdomains, cells, basis_size, seed, problem=None):
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases
    from pylrbms_b200 import discretize, LRBMSReductor
    from oracle import lrbms_oracle as O
    if isinstance(cells, tuple):        # seeded synthetic operators with 3D structure (synthetic_fixture.py)
        from pylrbms_b200.synthetic_fixture import make_random_local_bases, synthetic_block_operators
        data = synthetic_block_operators(num_subdomains, cells, seed=1000 + seed)
        bases = make_random_local_bases(data, basis_size, seed=seed)
    else:
        data = assemble_block_swipdg(num_subdomains, cells, problem=problem)
        bases = make_local_bases(data, basis_size, seed=seed)
    S = data.num_subdomains
    d_ref = O.build_discretization(data)
    red_ref = O.LRBMSReductor(d_ref, bases={'domain_%d' % i: bases[i] for i in range(S)})
    d, _ = discretize(data)
    red = LRBMSReductor(d, bases={'domain_%d' % i: bases[i] for i in range(S)})
    return data, d_ref, red_ref, d, red


def _blockwise(red_op):
    """{(q, i, j): block} for a reduced operator of the CUDA path (Lincomb or single)."""
    from pylrbms_b200.operators import LincombOperator
    ops = red_op.operators if isinstance(red_op, LincombOperator) else [red_op]
    return {(q,) + k: v for q, o in enumerate(ops) for k, v in o.blocks().items()}


def _blockwise_ref(red_ref, name):
    from oracle import lrbms_oracle as O
    from oracle.pymor_like import LincombOperator
    d = red_ref.d
    op = d.operators[name] if name in d.operators else d.products[name]
    nq = len(op.operators) if isinstance(op, LincombOperator) else 1
    out = {}
    for q in range(nq):
        for k, v in O.reduced_blocks(red_ref, name, q if isinstance(op, LincombOperator) else None).items():
            out[(q,) + k] = v
    return out


CASES = [
    ((2, 2), 4, 5, 1),                       # tiny
    ((3, 2), 4, [3, 7, 4, 6, 5, 8], 2),      # ragged local basis sizes (after enrichment, online_enrichment.py:49-51)
    ((4, 4), 8, 8, 3),                       # C1-like
    # 3D structure of config C4 (six face neighbours), synthetic operators
    ((2, 2, 2), (2, 2, 2), [5, 6, 7, 4, 8, 6, 5, 7], 11),
    ((3, 3, 3), (2, 2, 2), 8, 12),           # the centre subdomain has a seven-member neighbourhood
    ((3, 3, 3), (3, 3, 3), 40, 13),          # N = 40: 16-parameter estimator CTAs
]


@pytest.mark.parametrize('num_subdomains,cells,basis_size,seed', CASES)
def test_reduce_matches_oracle_blockwise(handle, num_subdomains, cells, basis_size, seed):
    data, d_ref, red_ref, d, red = _setup(num_subdomains, cells, basis_size, seed)
    rd_ref = red_ref.reduce()
    rd = red.reduce()
    names = list(d.operators) + list(d.products)
    assert set(names) == set(list(d_ref.operators) + list(d_ref.products))
    worst = 0.0
    for name in names:
        got = _blockwise(rd.operators[name] if name in rd.operators else rd.products[name])
        ref = _blockwise_ref(red_ref, name)
        scale = max(np.abs(v).max() for v in ref.values())
        for key, B in ref.items():
            assert key in got, '{}: block {} missing'.format(name, key)
            assert got[key].shape == B.shape
            err = np.abs(got[key] - B).max() / scale
            worst = max(worst, err)
            assert err < RTOL, '{} block {}: rel err {:.3e}'.format(name, key, err)
        for key, B in got.items():          # blocks the oracle found to be structurally zero must be (near) zero here
            if key not in ref:
                assert np.abs(B).max() <= RTOL * scale, '{}: spurious block {}'.format(name, key)
    # OI / RT image bases (reference reductor.py:36-60), including the q-major ordering of the RT basis
    for k in range(data.num_subdomains):
        for sid in ('OI_%d' % k, 'RT_%d' % k):
            a, b = red.bases[sid].to_numpy(), red_ref.bases[sid].data
            assert a.shape == b.shape
            assert np.abs(a - b).max() <= 1e-13 * max(1.0, np.abs(b).max())
    # unblocked form of the system operator (what the reference stores, reductor.py:46,66)
    for q in range(data.Q):
        assert np.abs(rd.operator.operators[q].to_dense() - rd_ref.operator.operators[q].matrix).max() < RTOL * \
            np.abs(rd_ref.operator.operators[q].matrix).max()
    print('worst block error', worst)


@pytest.mark.parametrize('num_subdomains,cells,basis_size,seed', CASES)
def test_solve_and_estimate_match_oracle(handle, num_subdomains, cells, basis_size, seed):
    data, d_ref, red_ref, d, red = _setup(num_subdomains, cells, basis_size, seed)
    rd_ref = red_ref.reduce()
    rd = red.reduce()
    mus = np.linspace(data.parameter_range[0], data.parameter_range[1], 7)
    # single-parameter API, exactly the reference call sequence (online_enrichment.py:72-74)
    for mu in mus[[0, 3, 6]]:
        U_ref = rd_ref.solve(mu)
        U = rd.solve(mu)
        A = rd_ref.operator.assemble(rd_ref.parse_parameter(mu)).matrix
        e = U.data[0] - U_ref.data[0]
        assert np.sqrt(e @ A @ e) <= RTOL * np.sqrt(U_ref.data[0] @ A @ U_ref.data[0])
        eta_ref, parts_ref, ind_ref = rd_ref.estimate(U_ref, mu, decompose=True)
        eta, parts, ind = rd.estimate(U, mu=mu, decompose=True)
        assert abs(eta - eta_ref) <= RTOL * abs(eta_ref)
        # r = ||f||^2 - 2 r_fd + r_dd cancels: compare relative to the scaled ||f||^2 (SURVEY.md section 7)
        r_scale = np.abs(rd.estimator.local_eta_rf_squared * rd.estimator.r_scale())
        for got, ref, scale in zip(parts, parts_ref, (None, r_scale, None)):
            s = np.abs(ref).max() if scale is None else max(np.abs(ref).max(), scale.max())
            assert np.abs(got[:, 0] - ref[:, 0]).max() <= RTOL * s
        assert np.abs(ind[:, 0] - ind_ref[:, 0]).max() <= 10 * RTOL * np.abs(ind_ref).max()
        assert isinstance(rd.estimate(U, mu=mu), float)
    # batched API: one sweep for all parameters equals the per-parameter results
    U_b, eta_b, parts_b, ind_b = rd.sweep(mus, decompose=True)
    assert U_b.data.shape == (len(mus), rd.n_red)
    for k, mu in enumerate(mus):
        U_ref = rd_ref.solve(mu)
        eta_ref, parts_ref, ind_ref = rd_ref.estimate(U_ref, mu, decompose=True)
        A = rd_ref.operator.assemble(rd_ref.parse_parameter(mu)).matrix
        e = U_b.data[k] - U_ref.data[0]
        assert np.sqrt(e @ A @ e) <= RTOL * np.sqrt(U_ref.data[0] @ A @ U_ref.data[0])       # energy norm, 1e-10
        assert abs(eta_b[k] - eta_ref) <= RTOL * abs(eta_ref)
        assert np.abs(ind_b[:, k] - ind_ref[:, 0]).max() <= 10 * RTOL * np.abs(ind_ref).max()
    # estimate_batch on given solutions
    eta_c = rd.estimate_batch(U_b, mus)
    assert np.array_equal(eta_c, eta_b)


def test_alpha_minimum_option(handle):
    """``alpha_returns_first=False`` gives the mathematically intended minimum (SURVEY.md row a15)."""
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases, os2015_problem
    from pylrbms_b200 import discretize, LRBMSReductor
    from oracle import lrbms_oracle as O
    data = assemble_block_swipdg((2, 2), 4, problem=os2015_problem(mu_bar=0.6, mu_hat=0.3))
    bases = make_local_bases(data, 4, seed=4)
    bd = {'domain_%d' % i: bases[i] for i in range(4)}
    for flag in (True, False):
        rd_ref = O.LRBMSReductor(O.build_discretization(data, alpha_returns_first=flag), bases=bd).reduce()
        rd = LRBMSReductor(discretize(data, alpha_returns_first=flag)[0], bases=bd).reduce()
        for mu in (0.15, 0.9):
            U_ref = rd_ref.solve(mu)
            eta_ref, _, ind_ref = rd_ref.estimate(U_ref, mu, decompose=True)
            eta, _, ind = rd.estimate(rd.solve(mu), mu=mu, decompose=True)
            assert abs(eta - eta_ref) <= RTOL * abs(eta_ref)
            assert np.abs(ind[:, 0] - ind_ref[:, 0]).max() <= 10 * RTOL * np.abs(ind_ref).max()


def test_reconstruct_and_extend_basis(handle):
    data, d_ref, red_ref, d, red = _setup((2, 2), 4, 4, 5)
    rd_ref, rd = red_ref.reduce(), red.reduce()
    mu = 0.4
    U_ref, U = rd_ref.solve(mu), rd.solve(mu)
    # reconstruct (reference online_adaptive_lrbms.py:143) and reconstruct_local (reductor.py:76)
    Uh_ref, Uh = red_ref.reconstruct(U_ref), red.reconstruct(U)
    assert np.abs(Uh.data - Uh_ref.data).max() <= RTOL * np.abs(Uh_ref.data).max()
    loc = red.reconstruct_local(U, 'domain_2').to_numpy()
    assert np.abs(loc - red_ref.reconstruct_local(U_ref, 'domain_2').data).max() <= RTOL * np.abs(loc).max()
    # fine-scale estimate of the reconstructed solution through the generic operator chain equals the reduced one
    eta_fine = d.estimate(Uh, mu=mu)
    eta_red = rd.estimate(U, mu=mu)
    assert abs(eta_fine - eta_red) <= 1e-8 * abs(eta_red)
    # extend_basis_local with the local energy product (reference online_adaptive_lrbms.py:104-119), then re-reduce
    from oracle import lrbms_oracle as O
    from oracle.pymor_like import VA
    from pylrbms_b200 import LRBMSReductor
    prods_ref = [d_ref.operators['local_energy_dg_product_%d' % i] for i in range(4)]
    prods = [d.operators['local_energy_dg_product_%d' % i] for i in range(4)]
    red_ref2 = O.LRBMSReductor(d_ref, products=prods_ref, order=1)
    red2 = LRBMSReductor(d, products=prods, order=1)
    rng = np.random.default_rng(0)
    for i in range(4):
        new = rng.standard_normal((2, int(data.n[i])))
        new[1] = red_ref2.bases['domain_%d' % i].data[0] * 3.0          # linearly dependent: must be rejected
        red_ref2.extend_basis_local(VA(new, d_ref.solution_space.subspaces[i]))
        red2.extend_basis_local(d.solution_space.subspaces[i].from_data(new))
        a, b = red2.bases['domain_%d' % i].to_numpy(), red_ref2.bases['domain_%d' % i].data
        assert a.shape == b.shape == (5, int(data.n[i]))
        assert np.abs(a - b).max() <= 1e-9 * np.abs(b).max()
        G = prods[i].apply2(red2.bases['domain_%d' % i], red2.bases['domain_%d' % i])
        assert np.abs(G - np.eye(5)).max() < 1e-11
    from pylrbms_b200 import ExtensionError
    with pytest.raises(ExtensionError):
        red2.extend_basis_local(red2.bases['domain_0'][0])
    rd2_ref, rd2 = red_ref2.reduce(), red2.reduce()
    eta_ref = rd2_ref.estimate(rd2_ref.solve(mu), mu)
    eta = rd2.estimate(rd2.solve(mu), mu=mu)
    assert abs(eta - eta_ref) <= 1e-9 * abs(eta_ref)


def test_vectorarray_interface(handle):
    """The VectorArray surface listed in SURVEY.md section 8b against NumPy."""
    from pylrbms_b200 import GpuVectorSpace
    rng = np.random.default_rng(7)
    sp_ = GpuVectorSpace(1000, 'domain_0')
    A, B = rng.standard_normal((6, 1000)), rng.standard_normal((6, 1000))
    a, b = sp_.from_data(A), sp_.make_array(B)
    assert len(a) == 6 and a.dim == 1000 and a.space == sp_
    assert np.array_equal(a.to_numpy(), A) and np.array_equal(a.data, A)
    assert np.abs(a.dot(b) - A @ B.T).max() < 1e-11
    assert np.abs(a.pairwise_dot(b) - np.einsum('ij,ij->i', A, B)).max() < 1e-11
    assert np.abs(a.l2_norm() - np.linalg.norm(A, axis=1)).max() < 1e-12
    c = a.copy(); c.scal(2.0); c.axpy(-0.5, b)
    assert np.abs(c.data - (2 * A - 0.5 * B)).max() < 1e-14
    c = a.copy(); c.axpy(np.arange(6.0), b[0])
    assert np.abs(c.data - (A + np.arange(6.0)[:, None] * B[0])).max() < 1e-14
    assert np.abs((a - b).data - (A - B)).max() == 0
    C_ = rng.standard_normal((3, 6))
    assert np.abs(a.lincomb(C_).data - C_ @ A).max() < 1e-12
    e = sp_.empty(reserve=4)
    assert len(e) == 0
    e.append(a); e.append(b[[1, 3]])
    assert len(e) == 8 and np.array_equal(e.data, np.vstack([A, B[[1, 3]]]))
    assert np.array_equal(a[2:4].data, A[2:4])
    z = sp_.zeros(3)
    assert z.is_zero() and not a.is_zero() and z.data.shape == (3, 1000)


def test_empty_local_bases(handle):
    """Subdomains without any basis function (an empty ``bases['domain_k']``, the state before the first enrichment of a
    subdomain) contribute zero-sized blocks; everything else must still match the oracle."""
    from pylrbms_b200.swipdg_fixture import assemble_block_swipdg, make_local_bases
    from pylrbms_b200 import discretize, LRBMSReductor
    from oracle import lrbms_oracle as O
    data = assemble_block_swipdg((3, 2), 4)
    bases = make_local_bases(data, [3, 0, 4, 5, 0, 2], seed=2)
    bd = {'domain_%d' % i: bases[i] for i in range(6)}
    rd_ref = O.LRBMSReductor(O.build_discretization(data), bases=bd).reduce()
    rd = LRBMSReductor(discretize(data)[0], bases=bd).reduce()
    assert rd.block_dims == [3, 0, 4, 5, 0, 2] and rd.n_red == 14
    for q in range(2):
        A, B = rd.operator.operators[q].to_dense(), rd_ref.operator.operators[q].matrix
        assert A.shape == B.shape == (14, 14) and np.abs(A - B).max() <= RTOL * np.abs(B).max()
    mus = np.array([0.2, 0.9])
    U, eta, parts, ind = rd.sweep(mus, decompose=True)
    for k, mu in enumerate(mus):
        U_ref = rd_ref.solve(mu)
        eta_ref, parts_ref, _ = rd_ref.estimate(U_ref, mu, decompose=True)
        A = rd_ref.operator.assemble(rd_ref.parse_parameter(mu)).matrix
        e = U.data[k] - U_ref.data[0]
        assert np.sqrt(e @ A @ e) <= RTOL * np.sqrt(U_ref.data[0] @ A @ U_ref.data[0])
        assert abs(eta[k] - eta_ref) <= RTOL * abs(eta_ref)
        assert np.abs(parts[0][:, k] - parts_ref[0][:, 0]).max() <= RTOL * max(np.abs(parts_ref[0]).max(), 1e-300)


def test_error_behaviour(handle):
    """Errors surface as exceptions carrying the library's message (C ABI: negative status + lrbms_last_error); a reduced
    operator that is not positive definite is reported, not silently 'solved'."""
    import ctypes as C
    from pylrbms_b200 import LrbmsError
    from pylrbms_b200._lib import ProjectDesc, make_project_plan, ptr, current_stream_ptr
    with pytest.raises(LrbmsError, match='null pointer'):
        make_project_plan(handle, [ProjectDesc(None, None, None, 4, 4, None, 1, 1, None, 1, 1, None, 1, 1.0, 0, 0)])
    with pytest.raises(LrbmsError, match='inconsistent sizes'):
        import torch
        t = torch.zeros(16, dtype=torch.float64, device='cuda')
        make_project_plan(handle, [ProjectDesc(None, None, None, 4, 4, t.data_ptr(), 1, 2, t.data_ptr(), 1, 2, t.data_ptr(), 2, 1.0, 0, 0)])
    data, d_ref, red_ref, d, red = _setup((2, 2), 4, 4, 9)
    rd = red.reduce()
    with pytest.raises(LrbmsError, match='not positive definite'):
        rd.solve(50.0)                       # lambda = 1 + (1 - mu) cos(..)cos(..) < 0 in the interior: indefinite
    with pytest.raises(ValueError):
        rd.estimate_batch(rd.solve_batch([0.5, 0.6]), [0.5])          # one solution per parameter
    # workspace too small is rejected by the library
    import torch
    plan = rd.online_plan
    theta = torch.from_numpy(rd.thetas([0.5])).cuda()
    u = torch.zeros((1, rd.n_red), dtype=torch.float64, device='cuda')
    info = torch.zeros(1, dtype=torch.int32, device='cuda')
    w = torch.zeros(64, dtype=torch.uint8, device='cuda')
    rc = plan.handle.lib.lrbms_online_solve(plan.p, 1, ptr(theta), ptr(u), ptr(info), ptr(w), 64, current_stream_ptr())
    assert rc == -1 and b'workspace too small' in plan.handle.lib.lrbms_last_error(plan.handle.h)


@pytest.mark.parametrize('num_subdomains,cells,basis_size', [((3, 2), 4, [3, 5, 4, 6, 5, 4]), ((2, 2, 2), (2, 2, 2), 5)])
def test_incremental_reprojection_matches_full(handle, num_subdomains, cells, basis_size):
    """SURVEY.md section 8f rank 2: after an enrichment only the rows / columns of the appended basis vectors are
    projected; everything else is taken from the previous plan.  The result must equal a from-scratch projection of the
    same bases (the reference's behaviour, ``online_enrichment.py:49-51``) and the oracle's."""
    from pylrbms_b200 import LRBMSReductor, discretize
    data, d_ref, red_ref, d, red = _setup(num_subdomains, cells, basis_size, 21)
    S = data.num_subdomains
    rng = np.random.default_rng(3)
    # extend in the local energy product, as the reference does (scripts/online_adaptive_lrbms.py:107): the given bases are
    # orthonormal in it, which is what makes the Gram-Schmidt result independent of the order of the projections
    red.products = [d.operators['local_energy_dg_product_%d' % k] for k in range(S)]
    red_ref.products = [d_ref.operators['local_energy_dg_product_%d' % k] for k in range(S)]
    red.incremental = True
    rd0 = red.reduce()
    assert red.last_plan.n_incremental_jobs == 0
    flops_full = red.last_plan.stats()['flops']
    for step, enriched in enumerate(([1], [0, S - 1], list(range(S)))):      # one, two, all subdomains; twice the same one
        for k in enriched:
            sid = 'domain_%d' % k
            new = rng.standard_normal((1 + (k + step) % 2, int(data.n[k])))
            red.extend_basis_local(d.solution_space.subspaces[k].from_data(new))
            red_ref.extend_basis_local(d_ref.solution_space.subspaces[k].make_array(new))
        rd = red.reduce()
        plan = red.last_plan
        assert plan.n_incremental_jobs > 0
        if len(enriched) < S:
            assert plan.stats()['flops'] < 0.8 * flops_full
        # from-scratch projection of the same bases through a fresh reductor
        bases_now = {'domain_%d' % k: red.bases['domain_%d' % k].to_numpy() for k in range(S)}
        rd_full = LRBMSReductor(d, bases=bases_now).reduce()
        rd_ref = red_ref.reduce()
        for name in list(d.operators) + list(d.products):
            got = _blockwise(rd.operators[name] if name in rd.operators else rd.products[name])
            full = _blockwise(rd_full.operators[name] if name in rd_full.operators else rd_full.products[name])
            ref = _blockwise_ref(red_ref, name)
            scale = max(np.abs(v).max() for v in ref.values())
            assert set(got) == set(full)
            for key, B in full.items():
                assert np.abs(got[key] - B).max() <= RTOL * scale, '{} block {} (incremental vs full)'.format(name, key)
            for key, B in ref.items():
                assert np.abs(got[key] - B).max() <= RTOL * scale, '{} block {} (incremental vs oracle)'.format(name, key)
        mus = np.linspace(data.parameter_range[0], data.parameter_range[1], 4)
        U, eta, _, _ = rd.sweep(mus, decompose=True)
        U2, eta2, _, _ = rd_full.sweep(mus, decompose=True)
        for k, mu in enumerate(mus):
            A = sum(c * o.to_dense() for c, o in zip(rd_full.thetas([mu])[0], rd_full.operator.operators))
            e = U.data[k] - U2.data[k]
            assert np.sqrt(e @ A @ e) <= RTOL * np.sqrt(U2.data[k] @ A @ U2.data[k])
        assert np.abs(eta - eta2).max() <= RTOL * np.abs(eta2).max()


def test_projection_is_bit_reproducible(handle):
    """Two projections of the same bases -- the same plan run again, and a second reductor with its own buffers -- must agree
    bit for bit.  120-column estimator Grams (three-member neighbourhoods, N = 20, Q = 2) split into output chunks of 7 + 8
    tiles: a gram CTA covers 8 + 8 and once stored the surplus tile row, racing with the mirrored chunk that owns it."""
    import torch
    from pylrbms_b200 import LRBMSReductor
    data, d_ref, red_ref, d, red = _setup((2, 2), 8, 20, 31)

    def dense(rd):
        return {(name, q): o.to_dense() for name, op in rd.operators.items() for q, o in enumerate(getattr(op, 'operators', [op]))}
    rd = red.reduce()
    A = dense(rd)
    for _ in range(3):
        red.last_plan.run()
        torch.cuda.synchronize()
        B = dense(rd)
        assert all(np.array_equal(A[k], B[k]) for k in A)
    bases = {'domain_%d' % k: red.bases['domain_%d' % k].to_numpy() for k in range(4)}
    C_ = dense(LRBMSReductor(d, bases=bases).reduce())
    bad = [k for k in A if not np.array_equal(A[k], C_[k])]
    assert not bad, bad
