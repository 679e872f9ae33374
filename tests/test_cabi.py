"""CPU-only checks of the C-ABI boundary: the library builds, loads without a GPU, exports every symbol that
``include/lrbms_sm100.h`` declares, fails loudly (no CPU fallback) when no device is present, and the host-only
symbolic phase produces a schedule that reproduces a dense Cholesky when replayed in NumPy."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'lrbms_sm100.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(lrbms_[a-z0-9_]+)\s*\(', text)))


def test_header_symbols_are_exported(built_library):
    lib = C.CDLL(built_library)
    declared = _declared_symbols()
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), 'symbol {} declared in include/lrbms_sm100.h is not exported'.format(name)


def test_binding_covers_header(built_library):
    from pylrbms_b200 import _lib
    assert sorted(_lib.EXPORTS) == _declared_symbols()
    lib = _lib.load_library()
    assert lib.lrbms_version() == 101


_NO_DEVICE_CHECK = '''
import ctypes as C
import sys
sys.path.insert(0, sys.argv[1])
from pylrbms_b200 import _lib
lib = _lib.load_library()
h = C.c_void_p()
rc = lib.lrbms_create(0, C.byref(h))
assert rc == -3 and not h.value, rc                  # LRBMS_ERR_NO_DEVICE
assert b'no CPU fallback' in lib.lrbms_last_error(None)
try:
    _lib.Handle.get()
except _lib.LrbmsError:
    pass
else:
    raise AssertionError('Handle.get() succeeded without a device')
'''


def test_no_cpu_fallback(built_library):
    """Without a CUDA device a handle cannot be created and the package raises instead of falling back.  Checked in a child
    process that sees no device (CUDA_VISIBLE_DEVICES empty), so that it also runs where a GPU is present."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    r = subprocess.run([sys.executable, '-c', _NO_DEVICE_CHECK, ROOT], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def _grid_blocks(sx, sy):
    blocks = []
    for s in range(sx * sy):
        ix, iy = s % sx, s // sx
        nb = [s]
        if iy > 0: nb.append(s - sx)
        if ix > 0: nb.append(s - 1)
        if ix < sx - 1: nb.append(s + 1)
        if iy < sy - 1: nb.append(s + sx)
        blocks += [(s, j) for j in sorted(nb)]
    return blocks


@pytest.mark.parametrize('sx,sy,sizes', [(1, 1, [5]), (2, 2, [8] * 4), (3, 2, [3, 11, 7, 20, 1, 9]), (4, 4, [20] * 16),
                                         (3, 3, [0, 4, 9, 2, 0, 17, 8, 8, 1])])
def test_symbolic_schedule_replays_to_cholesky(built_library, sx, sy, sizes):
    """Replay the left-looking 8x8-tile schedule of csrc/symbolic.cpp in NumPy: its pair lists are what the window
    schedule of solve_kernel_v2 is built from."""
    from pylrbms_b200._lib import Symbolic
    rng = np.random.default_rng(3)
    blocks = _grid_blocks(sx, sy)
    sizes = np.asarray(sizes, dtype=np.int32)
    off = np.concatenate([[0], np.cumsum(sizes)])
    n = int(off[-1])
    A = np.zeros((n, n))
    for (i, j) in blocks:
        if i >= j:
            B = rng.standard_normal((sizes[i], sizes[j])) * 0.2
            if i == j:
                B = B @ B.T + 3.0 * max(1, sizes[i]) * np.eye(sizes[i])
            A[off[i]:off[i + 1], off[j]:off[j + 1]] = B
            A[off[j]:off[j + 1], off[i]:off[i + 1]] = B.T
    f = rng.standard_normal(n)
    sym = Symbolic(sizes, [b[0] for b in blocks], [b[1] for b in blocks])
    assert sym.n_red == n and sym.n_pad == (n + 7) // 8 * 8
    ntc, n_tiles = sym.n_tile_cols, sym.n_tiles
    col_ptr, row_idx, pair_ptr, pair_a, pair_b, a_map = (sym.get(k) for k in range(6))
    assert col_ptr[-1] == n_tiles and pair_ptr[-1] == sym.n_pairs
    npad = sym.n_pad
    Ap = np.eye(npad); Ap[:n, :n] = A
    fp = np.zeros(npad); fp[:n] = f
    # every non-zero tile of the lower triangle of A must be in the pattern and flagged as an operator tile
    for J in range(ntc):
        rows = row_idx[col_ptr[J]:col_ptr[J + 1]]
        assert rows[0] == J and np.all(np.diff(rows) > 0)
        for I in range(J, ntc):
            t = Ap[8 * I:8 * I + 8, 8 * J:8 * J + 8]
            if np.any(t != 0) and not (I == J and np.array_equal(t, np.eye(8))):
                p = col_ptr[J] + np.searchsorted(rows, I)
                assert row_idx[p] == I and a_map[p] >= 0
    L = np.zeros((n_tiles + ntc, 8, 8))
    for J in range(ntc):
        for tgt in list(range(col_ptr[J], col_ptr[J + 1])) + [n_tiles + J]:
            if tgt < n_tiles:
                I = row_idx[tgt]
                T = Ap[8 * I:8 * I + 8, 8 * J:8 * J + 8].copy() if a_map[tgt] >= 0 else np.zeros((8, 8))
                if a_map[tgt] < 0:
                    assert not np.any(Ap[8 * I:8 * I + 8, 8 * J:8 * J + 8])
            else:
                T = np.zeros((8, 8)); T[0] = fp[8 * J:8 * J + 8]
            for p in range(pair_ptr[tgt], pair_ptr[tgt + 1]):
                a, b = pair_a[p], pair_b[p]
                # operands must already be final: they live in earlier tile columns
                assert (a < col_ptr[J] or a >= n_tiles) and b < col_ptr[J]
                T -= L[a] @ L[b].T
            if tgt == col_ptr[J]:
                Ljj = np.linalg.cholesky(T)
                L[tgt] = Ljj
            else:
                L[tgt] = np.linalg.solve(Ljj, T.T).T
    Ld = np.zeros((npad, npad))
    for J in range(ntc):
        for p in range(col_ptr[J], col_ptr[J + 1]):
            I = row_idx[p]
            Ld[8 * I:8 * I + 8, 8 * J:8 * J + 8] = L[p]
    assert np.abs(Ld @ Ld.T - Ap).max() < 1e-12 * np.abs(Ap).max()
    y = np.concatenate([L[n_tiles + J][0] for J in range(ntc)])
    assert np.allclose(Ld @ y, fp, rtol=0, atol=1e-12 * np.abs(fp).max())
    assert sym.flops > 0 and sym.max_targets >= 2
    # ---- shared-memory window schedule of solve_kernel_v2
    win_slot, late_ptr, win_a, win_b, xo_ptr, xo_idx = (sym.get(k) for k in range(6, 12))
    n_slots = sym.n_win_slots
    # a tile (I, K) is written after column K has been formed and last read while column I is formed; two tiles whose
    # lifetimes [K, I] overlap must not share a slot (column K's tiles are written after tiles of row K were last read)
    owner_until = {}
    for J in range(ntc):
        for p in range(col_ptr[J], col_ptr[J + 1]):
            if row_idx[p] == J:
                assert win_slot[p] == -1
                continue
            s_ = win_slot[p]
            assert 0 <= s_ < n_slots
            assert owner_until.get(s_, -1) <= J, 'slot {} reused while still live'.format(s_)
            owner_until[s_] = row_idx[p]
    for J in range(ntc):
        items = xo_idx[xo_ptr[J]:xo_ptr[J + 1]]
        assert sorted(items) == list(range(col_ptr[J], col_ptr[J + 1])) + [n_tiles + J]
        early = [late_ptr[t_] - pair_ptr[t_] for t_ in items]
        assert early == sorted(early, reverse=True)
        for t_ in items:
            # early pairs: source columns <= J - 3 (staggered schedule) or <= J - 2 (patterns without carrier tiles)
            lims = (col_ptr[max(J - 2, 0)], col_ptr[J - 1]) if J >= 1 else (0, 0)
            for p in range(pair_ptr[t_], pair_ptr[t_ + 1]):
                assert J == 0 or any((pair_b[p] >= lim) == (p >= late_ptr[t_]) for lim in lims)
                assert win_b[p] == win_slot[pair_b[p]]
                assert win_a[p] == (win_slot[pair_a[p]] if pair_a[p] < n_tiles else -(pair_a[p] - n_tiles + 1))


def test_symbolic_schedule_variant(built_library):
    """Band patterns (2D grids of subdomains) get the staggered schedule of solve_kernel_v2; a pattern in which a target has
    a source-(J-2) pair but no carrier tile falls back to the barrier schedule.  Either way the pair lists are complete
    (the replay test above) and late_ptr splits them at the right source column."""
    from pylrbms_b200._lib import Symbolic
    blocks = _grid_blocks(8, 8)
    sym = Symbolic(np.full(64, 20, dtype=np.int32), [b[0] for b in blocks], [b[1] for b in blocks])
    assert sym.staggered == 1
    # subdomains 2 and 3 (one 8x8 tile each) couple to 0, which fills tile (3, 2) from source column 0 = J - 2; subdomain 1 is
    # isolated, so neither tile (3, 1) nor (2, 1) exists to carry that pair
    S = 4
    blocks = [(i, i) for i in range(S)] + [(2, 0), (0, 2), (3, 0), (0, 3)]
    sym2 = Symbolic(np.full(S, 8, dtype=np.int32), [b[0] for b in blocks], [b[1] for b in blocks])
    assert sym2.staggered == 0
    col_ptr, row_idx, pair_ptr, pair_a, pair_b = (sym2.get(k) for k in range(5))
    late_ptr = sym2.get(7)
    back = 2 if sym2.staggered else 1
    for J in range(sym2.n_tile_cols):
        for tgt in list(range(col_ptr[J], col_ptr[J + 1])) + [sym2.n_tiles + J]:
            lim = col_ptr[max(J - back, 0)] if J >= 1 else 0
            for p in range(pair_ptr[tgt], pair_ptr[tgt + 1]):
                assert J == 0 or (pair_b[p] >= lim) == (p >= late_ptr[tgt])
