"""ctypes binding of ``liblrbms_sm100.so`` (C ABI declared in ``include/lrbms_sm100.h``).

There is no CPU fallback anywhere in this package: if the shared library is missing, or no sm_100 device is
present when a handle is requested, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'liblrbms_sm100.so')

EXPORTS = [
    'lrbms_version', 'lrbms_create', 'lrbms_destroy', 'lrbms_last_error', 'lrbms_device_sm_count', 'lrbms_set_option', 'lrbms_debug_poison_shared',
    'lrbms_va_scal', 'lrbms_va_axpy', 'lrbms_va_pairwise_dot', 'lrbms_va_lincomb', 'lrbms_va_copy_cols',
    'lrbms_va_transpose_in', 'lrbms_va_transpose_out',
    'lrbms_spmm_plan_create', 'lrbms_project_plan_create', 'lrbms_project_plan_scratch_bytes',
    'lrbms_project_plan_create_ws', 'lrbms_plan_run', 'lrbms_plan_destroy', 'lrbms_plan_info',
    'lrbms_symbolic_create', 'lrbms_symbolic_destroy', 'lrbms_symbolic_info', 'lrbms_symbolic_get', 'lrbms_symbolic_reorder',
    'lrbms_online_plan_create', 'lrbms_online_workspace_bytes', 'lrbms_online_solve', 'lrbms_online_estimate',
    'lrbms_online_sweep', 'lrbms_eta_max', 'lrbms_online_debug_timing',
    'lrbms_pcg_workspace_bytes', 'lrbms_pcg_solve', 'lrbms_affine_pcg_workspace_bytes', 'lrbms_affine_pcg_solve',
    'lrbms_recon_error_workspace_bytes', 'lrbms_recon_error', 'lrbms_segmented_form_workspace_bytes', 'lrbms_segmented_form',
    'lrbms_remap_blocks', 'lrbms_peer_push',
]

VEC_ONE, VEC_UI, VEC_UN, VEC_UR = 0, 1, 2, 3
OUT_NC, OUT_R, OUT_DF = 0, 1, 2
SOLVER_AUTO, SOLVER_WINDOW, SOLVER_BANDED = 0, 1, 3
SOLVER_NAMES = {1: 'solve_kernel_v2', 3: 'band_update_kernel'}


class LrbmsError(RuntimeError):
    pass


class SpmmDesc(C.Structure):
    _fields_ = [('rowptr', C.c_void_p), ('colind', C.c_void_p), ('values', C.c_void_p),
                ('n_rows', C.c_int32), ('n_cols', C.c_int32),
                ('V', C.c_void_p), ('ldv', C.c_int32), ('N', C.c_int32),
                ('W', C.c_void_p), ('ldw', C.c_int32)]


class ProjectDesc(C.Structure):
    _fields_ = [('rowptr', C.c_void_p), ('colind', C.c_void_p), ('values', C.c_void_p),
                ('n_rows', C.c_int32), ('n_cols', C.c_int32),
                ('VL', C.c_void_p), ('ldl', C.c_int32), ('NL', C.c_int32),
                ('VR', C.c_void_p), ('ldr', C.c_int32), ('NR', C.c_int32),
                ('out', C.c_void_p), ('ldo', C.c_int32),
                ('alpha', C.c_double), ('symmetric', C.c_int32), ('reserved', C.c_int32)]


class RemapDesc(C.Structure):
    _fields_ = [('dst', C.c_void_p), ('NL', C.c_int32), ('NR', C.c_int32), ('prev', C.c_void_p), ('pNR', C.c_int32),
                ('n_cn', C.c_int32), ('cols_new', C.c_void_p), ('rows_new', C.c_void_p), ('n_rn', C.c_int32),
                ('reserved', C.c_int32), ('row_map', C.c_void_p), ('col_map', C.c_void_p)]


class ReconBlock(C.Structure):
    _fields_ = [('V', C.c_void_p), ('ldv', C.c_int32), ('len', C.c_int32), ('N', C.c_int32), ('red_offset', C.c_int32),
                ('row_offset', C.c_int64), ('n_rows', C.c_int32), ('reserved', C.c_int32)]


class EstimatorTerm(C.Structure):
    _fields_ = [('subdomain', C.c_int32), ('out_kind', C.c_int32), ('left_kind', C.c_int32), ('right_kind', C.c_int32),
                ('rows', C.c_int32), ('cols', C.c_int32), ('qa', C.c_int32), ('qb', C.c_int32),
                ('coef', C.c_double), ('matrix_offset', C.c_int64)]


class ReducedSystem(C.Structure):
    _fields_ = [('n_sub', C.c_int32), ('basis_sizes', C.c_void_p), ('Q', C.c_int32), ('Qf', C.c_int32),
                ('n_blocks', C.c_int32), ('block_i', C.c_void_p), ('block_j', C.c_void_p), ('block_offset', C.c_void_p),
                ('lhs_blocks', C.c_void_p), ('rhs', C.c_void_p),
                ('nbh_ptr', C.c_void_p), ('nbh_idx', C.c_void_p), ('n_terms', C.c_int32), ('terms', C.c_void_p),
                ('est_matrices', C.c_void_p), ('rf_squared', C.c_void_p), ('r_scale', C.c_void_p),
                ('theta_bar', C.c_void_p), ('theta_hat', C.c_void_p), ('alpha_returns_first', C.c_int32),
                ('solver', C.c_int32)]


_lib = None
_lock = threading.Lock()


def load_library():
    """dlopen the library (no GPU needed for this step) and declare the prototypes."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise LrbmsError('{} not found: build it with `python -m pylrbms_b200.build` (there is no CPU fallback)'
                             .format(LIB_PATH))
        lib = C.CDLL(LIB_PATH)
        vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
        P = C.POINTER
        protos = {
            'lrbms_version': (C.c_int, []),
            'lrbms_create': (C.c_int, [C.c_int, P(vp)]),
            'lrbms_destroy': (C.c_int, [vp]),
            'lrbms_last_error': (C.c_char_p, [vp]),
            'lrbms_device_sm_count': (C.c_int, [vp, P(C.c_int)]),
            'lrbms_set_option': (C.c_int, [vp, i32, i32]),
            'lrbms_debug_poison_shared': (C.c_int, [vp, vp]),
            'lrbms_va_scal': (C.c_int, [vp, i64, i32, vp, i32, vp, i32, vp]),
            'lrbms_va_axpy': (C.c_int, [vp, i64, i32, vp, i32, vp, i32, i32, vp, i32, vp]),
            'lrbms_va_pairwise_dot': (C.c_int, [vp, i64, i32, vp, i32, vp, i32, vp, vp]),
            'lrbms_va_lincomb': (C.c_int, [vp, i64, i32, i32, vp, i32, vp, i32, vp, i32, vp]),
            'lrbms_va_copy_cols': (C.c_int, [vp, i64, i32, vp, vp, i32, vp, i32, i32, vp]),
            'lrbms_va_transpose_in': (C.c_int, [vp, i64, i32, vp, vp, i32, vp]),
            'lrbms_va_transpose_out': (C.c_int, [vp, i64, i32, vp, i32, vp, vp]),
            'lrbms_spmm_plan_create': (C.c_int, [vp, i32, vp, P(vp)]),
            'lrbms_project_plan_create': (C.c_int, [vp, i32, vp, P(vp)]),
            'lrbms_project_plan_scratch_bytes': (C.c_int, [i32, vp, P(C.c_size_t)]),
            'lrbms_project_plan_create_ws': (C.c_int, [vp, i32, vp, vp, C.c_size_t, i64, P(vp)]),
            'lrbms_plan_run': (C.c_int, [vp, vp]),
            'lrbms_plan_destroy': (C.c_int, [vp]),
            'lrbms_plan_info': (C.c_int, [vp, i32, P(dbl)]),
            'lrbms_symbolic_create': (C.c_int, [i32, vp, i32, vp, vp, P(vp)]),
            'lrbms_symbolic_destroy': (C.c_int, [vp]),
            'lrbms_symbolic_info': (C.c_int, [vp, i32, P(i64)]),
            'lrbms_symbolic_get': (i64, [vp, i32, vp, i64]),
            'lrbms_symbolic_reorder': (C.c_int, [vp, i32, i64]),
            'lrbms_online_plan_create': (C.c_int, [vp, vp, P(vp)]),
            'lrbms_online_workspace_bytes': (C.c_int, [vp, i64, P(C.c_size_t)]),
            'lrbms_online_solve': (C.c_int, [vp, i64, vp, vp, vp, vp, C.c_size_t, vp]),
            'lrbms_online_estimate': (C.c_int, [vp, i64, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]),
            'lrbms_online_sweep': (C.c_int, [vp, i64, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]),
            'lrbms_eta_max': (C.c_int, [vp, i64, vp, vp, vp, vp]),
            'lrbms_online_debug_timing': (C.c_int, [vp, vp, i32]),
            'lrbms_remap_blocks': (C.c_int, [vp, i32, vp, vp]),
            'lrbms_peer_push': (C.c_int, [vp, vp, i64, i32, vp, i32, vp]),
            'lrbms_pcg_workspace_bytes': (C.c_int, [vp, i64, P(C.c_size_t)]),
            'lrbms_pcg_solve': (C.c_int, [vp, i32, vp, vp, vp, vp, vp, dbl, i32, P(i32), P(dbl), vp, C.c_size_t, vp]),
            'lrbms_affine_pcg_workspace_bytes': (C.c_int, [vp, i64, i64, P(C.c_size_t)]),
            'lrbms_affine_pcg_solve': (C.c_int, [vp, i32, i32, vp, vp, vp, i32, vp, i64, vp, vp, i32, dbl, i32, i32,
                                                 vp, vp, vp, vp, C.c_size_t, vp]),
            'lrbms_recon_error_workspace_bytes': (C.c_int, [vp, i32, vp, i64, i32, P(C.c_size_t)]),
            'lrbms_recon_error': (C.c_int, [vp, i32, vp, i64, vp, i32, vp, i32, i32, vp, i32, vp, C.c_size_t, vp]),
            'lrbms_segmented_form_workspace_bytes': (C.c_int, [vp, i32, vp, P(C.c_size_t)]),
            'lrbms_segmented_form': (C.c_int, [vp, i32, i32, vp, vp, vp, i64, i32, vp, i64, vp, i32, vp, i32, vp, i32,
                                               vp, C.c_size_t, vp]),
        }
        for name, (res, args) in protos.items():
            fn = getattr(lib, name)          # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


class Handle:
    """One library context per CUDA device."""
    _handles = {}

    def __init__(self, device=0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.lrbms_create(int(device), C.byref(h))
        if rc != 0:
            raise LrbmsError('lrbms_create(device={}) failed ({}): {}'.format(
                device, rc, self.lib.lrbms_last_error(None).decode()))
        self.h = h
        self.device = int(device)
        n = C.c_int()
        self.lib.lrbms_device_sm_count(self.h, C.byref(n))
        self.sm_count = n.value

    def check(self, rc):
        if rc != 0:
            raise LrbmsError('liblrbms_sm100 error {}: {}'.format(rc, self.lib.lrbms_last_error(self.h).decode()))

    @classmethod
    def get(cls, device=None):
        import torch
        if device is None:
            if not torch.cuda.is_available():
                raise LrbmsError('no CUDA device: pylrbms_b200 runs on B200 (sm_100a) only and has no CPU fallback')
            device = torch.cuda.current_device()
        device = int(device)
        if device not in cls._handles:
            cls._handles[device] = Handle(device)
        return cls._handles[device]


def current_stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def host_i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def host_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def ptr(a):
    """Pointer of a numpy array (host) or torch tensor (device) as c_void_p; None -> NULL."""
    if a is None:
        return C.c_void_p(0)
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    return C.c_void_p(a.data_ptr())


class Plan:
    """RAII wrapper of lrbms_plan_t."""

    def __init__(self, handle, plan_ptr, keepalive=()):
        self.handle, self.p, self._keep = handle, plan_ptr, list(keepalive)

    def run(self, stream=None):
        self.handle.check(self.handle.lib.lrbms_plan_run(self.p, stream if stream is not None else current_stream_ptr()))

    def info(self, what):
        out = C.c_double()
        self.handle.check(self.handle.lib.lrbms_plan_info(self.p, int(what), C.byref(out)))
        return out.value

    @property
    def launches(self):
        return int(self.info(0))

    @property
    def algorithmic_bytes(self):
        return self.info(2)

    @property
    def algorithmic_bytes_survey(self):
        return self.info(5)

    @property
    def flops(self):
        return self.info(3)

    def destroy(self):
        if self.p is not None and self.p.value:
            self.handle.lib.lrbms_plan_destroy(self.p)
            self.p = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def make_spmm_plan(handle, descs, keepalive=()):
    arr = (SpmmDesc * len(descs))(*descs)
    p = C.c_void_p()
    handle.check(handle.lib.lrbms_spmm_plan_create(handle.h, len(descs), C.cast(arr, C.c_void_p), C.byref(p)))
    return Plan(handle, p, keepalive)


def make_project_plan(handle, descs, keepalive=(), scratch_owner=None, unit_rows_hint=0):
    """``scratch_owner``: an object with a ``_proj_scratch`` attribute (a CUDA tensor or None).  The plan's scratch then
    lives in that tensor (grown when too small, reused by the owner's later plans) instead of inside the plan."""
    arr = (ProjectDesc * len(descs))(*descs)
    p = C.c_void_p()
    if scratch_owner is None:
        handle.check(handle.lib.lrbms_project_plan_create_ws(handle.h, len(descs), C.cast(arr, C.c_void_p), None, 0,
                                                             int(unit_rows_hint), C.byref(p)))
        return Plan(handle, p, keepalive)
    import torch
    need = C.c_size_t()
    handle.check(handle.lib.lrbms_project_plan_scratch_bytes(len(descs), C.cast(arr, C.c_void_p), C.byref(need)))
    buf = getattr(scratch_owner, '_proj_scratch', None)
    if buf is None or buf.numel() * 8 < need.value:
        buf = torch.empty(max(32, need.value // 8 + need.value // 32), dtype=torch.float64, device='cuda')
        scratch_owner._proj_scratch = buf
    handle.check(handle.lib.lrbms_project_plan_create_ws(handle.h, len(descs), C.cast(arr, C.c_void_p), ptr(buf),
                                                         buf.numel() * 8, int(unit_rows_hint), C.byref(p)))
    return Plan(handle, p, list(keepalive) + [buf])


class Symbolic:
    """Host-only symbolic tile-Cholesky schedule (usable without a GPU)."""

    def __init__(self, basis_sizes, block_i, block_j):
        self.lib = load_library()
        sizes, bi, bj = host_i32(basis_sizes), host_i32(block_i), host_i32(block_j)
        s = C.c_void_p()
        rc = self.lib.lrbms_symbolic_create(len(sizes), ptr(sizes), len(bi), ptr(bi), ptr(bj), C.byref(s))
        if rc != 0:
            raise LrbmsError('lrbms_symbolic_create failed ({})'.format(rc))
        self.s = s
        self.n_sub = len(sizes)

    def info(self, what):
        out = C.c_int64()
        rc = self.lib.lrbms_symbolic_info(self.s, what, C.byref(out))
        if rc != 0:
            raise LrbmsError('lrbms_symbolic_info failed')
        return out.value

    n_red = property(lambda self: self.info(0))
    n_pad = property(lambda self: self.info(1))
    n_tile_cols = property(lambda self: self.info(2))
    n_tiles = property(lambda self: self.info(3))
    n_a_tiles = property(lambda self: self.info(4))
    n_pairs = property(lambda self: self.info(5))
    flops = property(lambda self: self.info(6))
    max_targets = property(lambda self: self.info(7))
    n_win_slots = property(lambda self: self.info(8))
    staggered = property(lambda self: self.info(11))
    order = property(lambda self: self.info(12))                 # 0 given, 1 Cuthill-McKee, 2 reverse Cuthill-McKee
    order_costs = property(lambda self: tuple(self.info(k) for k in (13, 14, 15)))

    def reorder(self, Q, smem_budget):
        """Re-plan in the cheapest subdomain order that fits ``smem_budget`` bytes (see lrbms_symbolic_reorder)."""
        rc = self.lib.lrbms_symbolic_reorder(self.s, int(Q), int(smem_budget))
        if rc != 0:
            raise LrbmsError('lrbms_symbolic_reorder failed ({})'.format(rc))
        return self.order

    def get(self, which):
        sizes = {0: self.n_tile_cols + 1, 1: self.n_tiles, 2: self.n_tiles + self.n_tile_cols + 1, 3: self.n_pairs,
                 4: self.n_pairs, 5: self.n_tiles, 6: self.n_tiles, 7: self.n_tiles + self.n_tile_cols, 8: self.n_pairs,
                 9: self.n_pairs, 10: self.n_tile_cols + 1, 11: self.n_tiles + self.n_tile_cols,
                 12: self.n_tiles + self.n_tile_cols, 13: self.n_tile_cols, 14: self.n_tiles + self.n_tile_cols,
                 15: self.n_sub, 16: self.n_sub, 17: self.n_red}
        out = np.zeros(sizes[which], dtype=np.int32)
        n = self.lib.lrbms_symbolic_get(self.s, which, ptr(out), out.size)
        if n != out.size:
            raise LrbmsError('lrbms_symbolic_get returned {}'.format(n))
        return out

    def __del__(self):
        try:
            if self.s is not None and self.s.value:
                self.lib.lrbms_symbolic_destroy(self.s)
                self.s = None
        except Exception:
            pass
