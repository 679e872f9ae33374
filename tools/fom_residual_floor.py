"""Attainable true residual of the fine-scale solve: lrbms_affine_pcg_solve at C1 and C2 (mu = 0.1, 1.0) for rtol 1e-10 ...
1e-14 and 3 / 20 restarts, with the energy-norm error against SciPy splu (plus one refinement step) and the true residual
of that splu solution evaluated on the host.  Sets the default rtol of d.solve_batch (profiles/r04_fom_residual_floor.txt).

    python tools/fom_residual_floor.py
"""
import sys, os, time
sys.path.insert(0, os.getcwd())
import numpy as np, torch, scipy.sparse as sp, scipy.sparse.linalg as spl
from pylrbms_b200 import discretize
from pylrbms_b200.kernels import affine_pcg_solve
from pylrbms_b200.parameters import theta_matrix
from pylrbms_b200.swipdg_fixture import assemble_block_swipdg

def host(data, th):
    S = data.num_subdomains; A = None
    for q in range(data.Q):
        B = [[None] * S for _ in range(S)]
        for (i, j), M in data.lhs[q].items(): B[i][j] = M
        M = sp.bmat(B, format='csc'); A = th[q] * M if A is None else A + th[q] * M
    return A.tocsc(), th[data.Q] * np.concatenate(data.rhs)

for shape, cells in (((4, 4), 16), ((8, 8), 32)):
    data = assemble_block_swipdg(shape, cells); d, _ = discretize(data)
    pat, vals, rhs = d.affine_system(range(data.num_subdomains)); n = pat.shape[0]
    mus = np.array([0.1, 1.0])
    th = theta_matrix(list(d.operator.coefficients) + list(d.rhs.coefficients), mus, d.parameter_type)
    refs = []
    for k in range(2):
        A, b = host(data, th[k]); lu = spl.splu(A); u = lu.solve(b); u += lu.solve(b - A @ u); refs.append((A, u, b))
    for rtol in (1e-10, 1e-11, 1e-12, 1e-13, 1e-14):
        for rs in (3, 20):
            x = torch.zeros((n, 2), dtype=torch.float64, device='cuda')
            torch.cuda.synchronize(); t = time.perf_counter()
            _, it, rr, st = affine_pcg_solve(pat, vals, rhs, torch.from_numpy(th).cuda(), x, rtol, 10 * n, rs)
            torch.cuda.synchronize(); dt = time.perf_counter() - t
            X = x.cpu().numpy()
            errs = []
            for k, (A, u, b) in enumerate(refs):
                e = X[:, k] - u; errs.append(np.sqrt(e @ (A @ e)) / np.sqrt(u @ (A @ u)))
            print(shape, cells, 'rtol %.0e restarts %d: status %s iters %s true relres %s energy err %s  %.2fs' % (
                rtol, rs, list(st), list(it), ['%.2e' % v for v in rr], ['%.2e' % v for v in errs], dt), flush=True)
            print('   splu residual', ['%.2e' % (np.linalg.norm(b - A @ u) / np.linalg.norm(b)) for A, u, b in refs], flush=True)
