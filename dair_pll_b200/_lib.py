"""ctypes binding of ``libdair_pll_b200.so`` (C ABI: ``include/dair_pll_b200.h``).

There is deliberately no fallback: if the CUDA library is missing or a call fails, the
caller gets an exception.  The library is built in-tree by ``dair_pll_b200.build``.
"""
import ctypes
import os

from dair_pll_b200 import build as _build

_LIB = None
ABI_VERSION = 214        # DPLL_VERSION of include/dair_pll_b200.h this binding was written against

_c_void_p = ctypes.c_void_p
_i64, _i32, _f64, _f32, _sz = ctypes.c_int64, ctypes.c_int32, ctypes.c_double, ctypes.c_float, ctypes.c_size_t

EXPORTS = {
    'dpll_version': ([], ctypes.c_int),
    'dpll_workspace_bytes': ([], _sz),
    'dpll_set_loss_variant': ([ctypes.c_int], ctypes.c_int),
    'dpll_cube_loss_f64': ([_c_void_p] * 6 + [_f64, _f64, _i64] + [_c_void_p] * 6 + [_c_void_p, _sz, _c_void_p],
                           ctypes.c_int),
    'dpll_cube_loss_f32': ([_c_void_p] * 6 + [_f32, _f32, _i64] + [_c_void_p] * 6 + [_c_void_p, _sz, _c_void_p],
                           ctypes.c_int),
    'dpll_cube_loss_leaf_f64': ([_c_void_p] * 6 + [_f64, _f64, _i64] + [_c_void_p] * 6 + [_c_void_p, _sz, _c_void_p],
                                ctypes.c_int),
    'dpll_cube_loss_leaf_f32': ([_c_void_p] * 6 + [_f32, _f32, _i64] + [_c_void_p] * 6 + [_c_void_p, _sz, _c_void_p],
                                ctypes.c_int),
    'dpll_cube_rollout_f64': ([_c_void_p] * 4 + [_f64, _f64, _i64, _i32] + [_c_void_p] * 4, ctypes.c_int),
    'dpll_cube_rollout_f32': ([_c_void_p] * 4 + [_f32, _f32, _i64, _i32] + [_c_void_p] * 4, ctypes.c_int),
    'dpll_cube_terms_f64': ([_c_void_p] * 5 + [_i64] + [_c_void_p] * 6, ctypes.c_int),
    'dpll_body_loss_pts_f64': ([_c_void_p] * 6 + [_i32, _f64, _f64, _i64, _i32] + [_c_void_p] * 7 + [_c_void_p, _sz, _c_void_p],
                               ctypes.c_int),
    'dpll_body_step_pts_f64': ([_c_void_p] * 4 + [_i32, _f64, _f64, _i64] + [_c_void_p] * 3, ctypes.c_int),
    'dpll_chain_loss_f64': ([_i32] + [_c_void_p] * 7 + [_f64, _f64, _i64] + [_c_void_p] * 5 + [_c_void_p, _sz, _c_void_p],
                            ctypes.c_int),
    'dpll_chain_rollout_f64': ([_i32] + [_c_void_p] * 5 + [_f64, _f64, _i64, _i32] + [_c_void_p] * 2, ctypes.c_int),
    'dpll_elbow_terms_f64': ([_c_void_p] * 6 + [_i64] + [_c_void_p] * 6, ctypes.c_int),
    'dpll_chain_loss_pts_f64': ([ctypes.c_int32] + [_c_void_p] * 7 + [ctypes.c_uint32, ctypes.c_double, ctypes.c_double, _i64]
                                + [_c_void_p] * 5 + [ctypes.c_size_t, _c_void_p], ctypes.c_int),
    'dpll_chain_terms_f64': ([ctypes.c_int32] * 2 + [_c_void_p] * 6 + [_i64] + [_c_void_p] * 6, ctypes.c_int),
    'dpll_cube_rollout_grad_f64': ([_c_void_p] * 4 + [_f64, _f64, _i64, _i32] + [_c_void_p] * 4, ctypes.c_int),
    'dpll_cube_rollout_saved_f64': ([_c_void_p] * 4 + [_f64, _f64, _i64, _i32] + [_c_void_p] * 3, ctypes.c_int),
    'dpll_cube_rollout_backward_f64': ([_c_void_p] * 5 + [_f64, _f64, _i64, _i32] + [_c_void_p] * 4, ctypes.c_int),
    'dpll_elbow_loss_f64': ([_c_void_p] * 8 + [_f64, _f64, _i64, _i32] + [_c_void_p] * 7 + [_c_void_p, _sz, _c_void_p], ctypes.c_int),
    'dpll_elbow_loss_f32': ([_c_void_p] * 8 + [_f32, _f32, _i64, _i32] + [_c_void_p] * 7 + [_c_void_p, _sz, _c_void_p], ctypes.c_int),
    'dpll_elbow_rollout_f64': ([_c_void_p] * 6 + [_f64, _f64, _i64, _i32] + [_c_void_p] * 4, ctypes.c_int),
    'dpll_elbow_rollout_f32': ([_c_void_p] * 6 + [_f32, _f32, _i64, _i32] + [_c_void_p] * 4, ctypes.c_int),
    'dpll_icnn_input_f64': ([_c_void_p, _c_void_p, _i64, _i32, _f64, _c_void_p, _c_void_p], ctypes.c_int),
    'dpll_icnn_mask_f64': ([_c_void_p, _i64, _f64, _c_void_p], ctypes.c_int),
    'dpll_icnn_output_f64': ([_c_void_p] * 5 + [_i64, _i32, _f64, _c_void_p, _c_void_p], ctypes.c_int),
    'dpll_elbow_support_directions_f64': ([_c_void_p, _i64] + [_c_void_p] * 3 + [_i32, _i64] + [_c_void_p] * 3, ctypes.c_int),
    'dpll_body_support_directions_f64': ([_c_void_p, _i64, _c_void_p, _i32, _i64, _c_void_p, _c_void_p], ctypes.c_int),
    'dpll_icnn_tc_image_bytes': ([], ctypes.c_size_t),
    'dpll_icnn_tc_const_bytes': ([], ctypes.c_size_t),
    'dpll_icnn_tc_prepare_f64': ([_c_void_p] * 4 + [_i32, _f64, _c_void_p, _c_void_p, _c_void_p], ctypes.c_int),
    'dpll_icnn_tc_support_f64': ([_c_void_p, _i64, _c_void_p, _c_void_p, _c_void_p, _i32, _f64, _c_void_p, _c_void_p],
                                 ctypes.c_int),
    'dpll_icnn_tc_bwd_partial_bytes': ([], ctypes.c_size_t),
    'dpll_icnn_tc_bwd_planes': ([], ctypes.c_int32),
    'dpll_icnn_tc_record_f64': ([_c_void_p, _i64, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _i32, _f64, _c_void_p, _c_void_p,
                                 _i64, _c_void_p], ctypes.c_int),
    'dpll_icnn_tc_bwd_f64': ([_c_void_p] * 5 + [_i64, _f64] + [_c_void_p] * 5, ctypes.c_int),
    'dpll_icnn_backward_blocks': ([_i64], ctypes.c_int),
    'dpll_icnn_backward_f64': ([_c_void_p] * 5 + [_i64, _i32, _f64, _c_void_p, _c_void_p, _c_void_p], ctypes.c_int),
    'dpll_cube_loss_leaf_dp_f64': ([_c_void_p, _i64, _c_void_p, _i64] + [_c_void_p] * 3 + [_f64, _f64, _i64, _i32] +
                                   [_c_void_p] * 8 + [_c_void_p, _sz, _c_void_p], ctypes.c_int),
    'dpll_cube_loss_leaf_dp_f32': ([_c_void_p, _i64, _c_void_p, _i64] + [_c_void_p] * 3 + [_f32, _f32, _i64, _i32] +
                                   [_c_void_p] * 8 + [_c_void_p, _sz, _c_void_p], ctypes.c_int),
    'dpll_comm_handle_bytes': ([], _sz),
    'dpll_comm_create': ([_i32, _i32, ctypes.POINTER(_c_void_p), _c_void_p], ctypes.c_int),
    'dpll_comm_connect': ([_c_void_p, _c_void_p], ctypes.c_int),
    'dpll_comm_destroy': ([_c_void_p], ctypes.c_int),
    'dpll_comm_device_state': ([_c_void_p], _c_void_p),
    'dpll_comm_error': ([_c_void_p], ctypes.c_int),
    'dpll_comm_allreduce_f64': ([_c_void_p, _c_void_p, _i32, _f64, _c_void_p], ctypes.c_int),
    'dpll_elbow_step_pts_grad_f64': ([_c_void_p] * 6 + [_f64, _f64, _i64] + [_c_void_p] * 5, ctypes.c_int),
    'dpll_elbow_rollout_saved_f64': ([_c_void_p] * 6 + [_f64, _f64, _i64, _i32] + [_c_void_p] * 3, ctypes.c_int),
    'dpll_elbow_rollout_grad_saved_f64': ([_c_void_p] * 6 + [_f64, _f64, _i64, _i32] + [_c_void_p] * 4, ctypes.c_int),
    'dpll_body_step_pts_grad_f64': ([_c_void_p] * 4 + [_i32, _f64, _f64, _i64] + [_c_void_p] * 5, ctypes.c_int),
    'dpll_chain_rollout_grad_f64': ([_i32] + [_c_void_p] * 5 + [_f64, _f64, _i64, _i32] + [_c_void_p] * 4, ctypes.c_int),
    'dpll_leaf_prepare_f64': ([_c_void_p, _i32, _c_void_p, _c_void_p, _c_void_p, _i32, _c_void_p, _i32] + [_c_void_p] * 4, ctypes.c_int),
    'dpll_leaf_backward_f64': ([_c_void_p, _i32, _c_void_p, _i32, _c_void_p, _c_void_p, _i32, _c_void_p, _i32] + [_c_void_p] * 7,
                               ctypes.c_int),
    'dpll_fma_peak_f64': ([_c_void_p, _i32, _i64, _c_void_p], ctypes.c_int),
    'dpll_fma_peak_f32': ([_c_void_p, _i32, _i64, _c_void_p], ctypes.c_int),
}


def lib_path() -> str:
    """In-tree library; DAIR_PLL_B200_LIB overrides it (A/B builds during kernel development)."""
    return os.environ.get('DAIR_PLL_B200_LIB', _build.LIB_PATH)


def load() -> ctypes.CDLL:
    """Load the CUDA library; raises if it has not been built (no CPU fallback exists)."""
    global _LIB
    if _LIB is None:
        path = lib_path()
        if not os.path.exists(path):
            raise RuntimeError(
                f'{path} not found: build it with `python -m dair_pll_b200.build` '
                '(nvcc, sm_100a). dair_pll_b200 has no CPU or PyTorch fallback.')
        if path == _build.LIB_PATH and _build.sources_present() and _build.is_stale():
            # argtypes are positional: a library older than its sources could take shifted pointers
            raise RuntimeError(f'{path} is older than csrc/ or include/: rebuild it with `python -m dair_pll_b200.build`')
        lib = ctypes.CDLL(path)
        for name, (argtypes, restype) in EXPORTS.items():
            fn = getattr(lib, name)      # AttributeError if the symbol is missing
            fn.argtypes = argtypes
            fn.restype = restype
        version = lib.dpll_version()
        if version != ABI_VERSION:
            raise RuntimeError(f'{path} reports ABI version {version}, this binding expects {ABI_VERSION}: rebuild it')
        _LIB = lib
    return _LIB


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    if rc > 0:
        raise RuntimeError(f'{what}: CUDA error {rc}')
    if rc == -3:
        raise RuntimeError(f'{what}: a peer rank did not arrive at the gradient exchange (timeout)')
    raise RuntimeError(f'{what}: argument error {rc} (see include/dair_pll_b200.h)')
