"""Compare the outputs two builds wrote with ``bench.py --dump-outputs`` (same arguments and seed).

    python tools/compare_dumps.py DIR_A DIR_B

Prints one JSON line: whether the parameters and the factorisation flags are identical, the largest per-row relative
difference of the reduced solutions u (max-norm of the row difference over the max-norm of the row) and the largest relative
difference of eta.  Exit status 1 if the parameters or flags differ or u differs by more than 1e-12 per row."""
import json
import os
import sys

import numpy as np


def main(a, b):
    load = lambda d, n: np.load(os.path.join(d, n + '.npy'))
    same_mu = bool(np.array_equal(load(a, 'index'), load(b, 'index')) and np.array_equal(load(a, 'mu'), load(b, 'mu')))
    same_info = bool(np.array_equal(load(a, 'info'), load(b, 'info')))
    ua, ub = load(a, 'u'), load(b, 'u')
    u_row = float((np.abs(ua - ub).max(axis=1) / np.abs(ub).max(axis=1)).max())
    ea, eb = load(a, 'eta'), load(b, 'eta')
    eta_rel = float((np.abs(ea - eb) / np.abs(eb)).max())
    out = {'rows': int(ua.shape[0]), 'same_mu': same_mu, 'same_info': same_info, 'u_max_row_rel': u_row,
           'eta_max_rel': eta_rel, 'eta_max': [load(a, 'eta_max').tolist(), load(b, 'eta_max').tolist()]}
    print(json.dumps(out))
    return 0 if same_mu and same_info and u_row <= 1e-12 else 1


if __name__ == '__main__':
    sys.exit(main(sys.argv[1], sys.argv[2]))
