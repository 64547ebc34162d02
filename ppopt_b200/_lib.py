"""ctypes binding of libppgpu.so (include/ppgpu.h).  Fails loudly when the CUDA library is missing: there is no
CPU fallback anywhere in this package."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libppgpu.so')

NUM_COUNTERS = 27
NUM_FAMILIES = 10
FAMILY_NAMES = ('k1_rank', 'k2_feas_lp', 'k34_kkt_cheb', 'k5_emit', 'k6_count', 'k6_write', 'select', 'k2a_relax', 'k2w_walk', 'inherit')
COUNTER_NAMES = ('k1_candidates', 'k2_lps', 'k2_pivots', 'k2_work', 'k4_lps', 'k4_pivots', 'k4_work', 'k5_lps',
                 'k5_pivots', 'k5_work', 'numeric', 'border', 'k6_lookups', 'k2a_tried', 'k2a_certified', 'k2a_steps', 'k2a_work',
                 'k2w_certified', 'k2w_pivots', 'k2w_work', 'k2w_giveup', 'inherited', 'inherit_lookups',
                 'k2w_drop_reset', 'k2w_drop_giveup', 'k2w_infeasible', 'k2w_inf_band')

# status bits (csrc/tolerances.h)
ST_RANK, ST_FEAS, ST_OPT, ST_REGION, ST_BORDER, ST_NUMERIC, ST_THIN = 1, 2, 4, 8, 16, 32, 64
OPT_K2W_MIN = 0   # ppgpu_set_option (include/ppgpu.h)
OPT_K2W_REF = 1
OPT_K2W_INFEAS = 2
TREE_OPT_INHERIT = 0   # ppgpu_tree_set_option
WITNESS_SLOTS = 2  # PPGPU_WITNESS_SLOTS


class Dims(ctypes.Structure):
    _fields_ = [(k, ctypes.c_int32) for k in ('n', 't', 'm', 'q', 'n_eq', 'is_qp')]


class Info(ctypes.Structure):
    _fields_ = [(k, ctypes.c_int32) for k in
                ('words', 'n_ineq', 'region_rows', 'use_gram', 'max_depth', 'sm_count', 'lp_columns', 'reserved')]


# every symbol include/ppgpu.h declares: name -> (restype, argtypes)
_vp, _i32, _i64, _u8, _sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint8, ctypes.c_size_t
SYMBOLS = {
    'ppgpu_last_error': (ctypes.c_char_p, []),
    'ppgpu_version': (ctypes.c_int, []),
    'ppgpu_program_create': (ctypes.c_int, [ctypes.POINTER(Dims)] + [_vp] * 8 + [ctypes.c_int, ctypes.POINTER(_vp)]),
    'ppgpu_program_destroy': (ctypes.c_int, [_vp]),
    'ppgpu_program_info': (ctypes.c_int, [_vp, ctypes.POINTER(Info)]),
    'ppgpu_set_option': (ctypes.c_int, [_vp, _i32, _i64]),
    'ppgpu_root_level': (ctypes.c_int, [_vp, _vp, ctypes.POINTER(_i64), _vp]),
    'ppgpu_level_eval': (ctypes.c_int, [_vp, _vp, _i64, _i32, _vp, _i32, _vp]),
    'ppgpu_level_eval_w': (ctypes.c_int, [_vp, _vp, _i64, _i32, _vp, _i32, _vp, _vp, _i64, _vp, _vp, _vp]),
    'ppgpu_scan_workspace_bytes': (_sz, [_i64]),
    'ppgpu_select_workspace_bytes': (_sz, [_i64]),
    'ppgpu_level_select': (ctypes.c_int, [_vp, _vp, _i64, _u8, _u8, _vp, ctypes.POINTER(_i64), _vp, _sz, _vp]),
    'ppgpu_regions_emit': (ctypes.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    'ppgpu_children_count': (ctypes.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, ctypes.POINTER(_i64), _vp, _sz, _vp]),
    'ppgpu_children_prepare': (ctypes.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    'ppgpu_children_count_range': (ctypes.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _i64, _i64, _vp, _sz, _vp]),
    'ppgpu_children_scan': (ctypes.c_int, [_vp, _vp, _i64, ctypes.POINTER(_i64), _vp, _sz, _vp]),
    'ppgpu_children_write': (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, _vp]),
    'ppgpu_counters': (ctypes.c_int, [_vp, _vp, _i32, _vp]),
    'ppgpu_launch_count': (_i64, [_vp]),
    'ppgpu_profile_enable': (ctypes.c_int, [_vp, _i32]),
    'ppgpu_profile_read': (ctypes.c_int, [_vp, _vp, _vp, _i32]),
    'ppgpu_locate_points': (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp, _i64, _vp, _i32, _i32, ctypes.c_double, _i32, _vp, _vp, _vp,
                                           _vp, _vp, _vp]),
    'ppgpu_solve_theta_batch': (ctypes.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    'ppgpu_solve_theta_lp_batch': (ctypes.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    'ppgpu_chebyshev_batch': (ctypes.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp]),
    'ppgpu_facet_chebyshev_batch': (ctypes.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _i64, _vp, _vp, _vp, _vp]),
    'ppgpu_program_param_maps': (ctypes.c_int, [_vp, _i32, _vp, _vp, _vp, ctypes.POINTER(_i32)]),
    'ppgpu_mi_offsets': (ctypes.c_int, [_vp, _vp, _i32, _i32, _vp, _i64, _vp, _i32, _vp, _vp]),
    'ppgpu_solve_pairs_qp': (ctypes.c_int, [_vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'ppgpu_solve_pairs_lp': (ctypes.c_int, [_vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'ppgpu_mi_select': (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp, _i64, _i32, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp,
                                       _vp, _vp]),
    'ppgpu_tree_create': (ctypes.c_int, [ctypes.POINTER(Dims), _vp, _i32] + [_vp] * 5 + [ctypes.c_int, ctypes.POINTER(_vp)]),
    'ppgpu_tree_destroy': (ctypes.c_int, [_vp]),
    'ppgpu_tree_set_option': (ctypes.c_int, [_vp, _i32, _i64]),
    'ppgpu_tree_eval': (ctypes.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    'ppgpu_tree_children': (ctypes.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, ctypes.POINTER(_i64), _vp, _sz, _vp]),
    'ppgpu_measure_fp64_peak': (ctypes.c_int, [_i32, ctypes.POINTER(ctypes.c_double), _vp]),
}

_lib = None


def load():
    """Returns the loaded library; raises RuntimeError if it has not been built (python __graft_entry__.py)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f'{LIB_PATH} is missing - build it with `make -C ppopt_b200/csrc` '
                           f'(or __graft_entry__.build()); ppopt_b200 has no CPU fallback')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=''):
    if rc != 0:
        msg = load().ppgpu_last_error()
        raise RuntimeError(f'libppgpu {what} failed ({rc}): {msg.decode() if msg else "?"}')
