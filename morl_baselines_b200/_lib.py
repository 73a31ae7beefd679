"""ctypes loader for libmorl_b200.so (the C-ABI of include/morl_b200.h).

There is NO CPU fallback: if the shared library is missing, or a compute entry point is called without a CUDA device,
the call raises.  The library is built in-tree by ``python -m morl_baselines_b200.csrc.build`` (nvcc, sm_100a) and
travels with the repo snapshot to the GPU box.
"""

from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libmorl_b200.so")

# constants of include/morl_b200.h
DOT_UNFUSED, DOT_FMA, DOT_PAIRFMA = 0, 1, 2
MAP_TILE, MAP_BLOCK = 0, 1
ROWS_REFERENCE, ROWS_BMAJOR = 0, 1
AC_ELEMENTWISE_MIN, AC_SCALAR_MIN, AC_ARGMIN_GATHER = 0, 1, 2
MAX_D = 8
FMT_BF16X3, FMT_F16X2 = 0, 1

_vp, _i, _f, _d, _i64, _sz = C.c_void_p, C.c_int, C.c_float, C.c_double, C.c_int64, C.c_size_t

# name -> (restype, argtypes); mirrors include/morl_b200.h one to one (checked by tests/test_abi.py)
SIGNATURES = {
    "morl_version": (_i, []),
    "morl_last_error": (C.c_char_p, []),
    "morl_device_sm_count": (_i, []),
    "morl_envelope_td_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "morl_greedy_td_f32": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _i, _i, _f, _i, _i, _i, _i, _vp, _vp, _vp]),
    "morl_critic_min_td_f32": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp, _i, _i, _f, _i, _i, _i, _i, _vp, _vp, _vp]),
    "morl_gpi_envelope_f32": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp, _i, _i, _f, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "morl_actor_critic_td_f32": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp, _vp, _f, _f, _i, _i, _i, _vp, _vp]),
    "morl_td_workspace_bytes": (_sz, [_i]),
    "morl_td_mse_priority_f32": (_i, [_vp, _vp, _vp, _vp, _f, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "morl_td_huber_priority_f32": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _f, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "morl_host_sumtree_walk": (_i, [_vp, _i, _vp, _i, _vp]),
    "morl_host_sumtree_batch_set": (_i, [_vp, _i, _vp, _vp, _i]),
    "morl_host_gather_rows": (_i, [_vp, C.c_longlong, _vp, _i, _vp]),
    "morl_host_gather_u8_to_i32": (_i, [_vp, C.c_longlong, _vp, _i, _vp]),
    "morl_sumtree_walk_f64": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp]),
    "morl_sumtree_batch_set_f64": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp]),
    "morl_sumtree_set_f64": (_i, [_vp, _i, C.c_longlong, _d, _i, _vp, _vp, _vp]),
    "morl_per_priority_f32": (_i, [_vp, _i, _f, _vp, _vp, _vp, _vp]),
    "morl_replay_gather": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "morl_pareto_mask_f32": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "morl_pareto_mask_f64": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "morl_front_pack_f64": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _vp, _vp]),
    "morl_front_unpack_f64": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "morl_hypervolume_f64": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "morl_polyak_f32": (_i, [_vp, _vp, _vp, _i, _i64, _d, _vp]),
    "morl_plane_overflow_count": (_i, [_i]),
    "morl_amax_scale_f32": (_i, [_vp, C.c_longlong, _i, _vp, _vp, _vp]),
    "morl_split_planes_multi": (_i, [_i, _vp, _i, _vp]),
    "morl_split_planes": (_i, [_i, _vp, _i, _i, _i, _i, _vp, _i, _i, C.c_longlong, _vp, _vp]),
    "morl_gemm_planes_f32": (_i, [_i, _vp, C.c_longlong, _vp, _vp, C.c_longlong, _vp, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, C.c_longlong,
                                  _vp, _i, _i, _vp, _vp, _vp]),
    "morl_gemm_chain_supported": (_i, [_i, _i, _i]),
    "morl_gemm_chain_f32": (_i, [_i, _i, _i, _vp, C.c_longlong, _vp, _vp, C.c_longlong, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _vp]),
    "morl_debug_gemm_stats": (_i, [_vp, _i]),
    "morl_ensemble_sample_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "morl_qhead_envelope_supported": (_i, [_i, _i, _i, _i, _i, _i]),
    "morl_qhead_gemm_supported": (_i, [_i, _i, _i, _i]),
    "morl_qhead_gemm_f32": (_i, [_i, _vp, C.c_longlong, _vp, _vp, C.c_longlong, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "morl_qhead_envelope_td_f32": (_i, [_i, _vp, _vp, C.c_longlong, _vp, _vp, _vp, _vp, C.c_longlong, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _f, _i, _i,
                                        _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "morl_pairs_relu_split_planes": (_i, [_i, _vp, _vp, _i, _i, _i, _vp, C.c_longlong, _vp, _vp, _vp]),
    "morl_gemm_mn_workspace_bytes": (_sz, [_i, _i, _i]),
    "morl_gemm_planes_mn_f32": (_i, [_i, _vp, C.c_longlong, _i, _i, _vp, _vp, C.c_longlong, _i, _i, _vp, _i, _i, _vp, _i, _vp, _vp, _vp]),
    "morl_gemm_mn_multi_workspace_bytes": (_sz, [_vp, _i, _i]),
    "morl_gemm_planes_mn_multi_f32": (_i, [_i, _vp, _i, _i, _vp, _vp]),
    "morl_colsum_planes": (_i, [_i, _vp, C.c_longlong, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "morl_pairs_grad_reduce_planes": (_i, [_i, _vp, C.c_longlong, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "morl_pair_layer1_uv_f32": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "morl_pair_layer1_grad_workspace_bytes": (_sz, [_i, _i, _i]),
    "morl_pair_layer1_grad_f32": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "morl_adam_workspace_bytes": (_sz, [_i, _i64]),
    "morl_adam_clip_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _f, _f, _f, _f, _f, _vp, _vp]),
}

SPLIT_MAX_JOBS = 16


class SplitJob(C.Structure):
    """MorlSplitJob of include/morl_b200.h"""

    _fields_ = [("src", _vp), ("dst_planes", _vp), ("plane_stride", C.c_longlong), ("scale", _vp), ("rows", _i), ("cols", _i), ("ld_src", _i),
                ("transpose", _i), ("rows_pad", _i), ("ldp", _i), ("auto_scale", _i), ("target_exp", _i)]


MN_MAX_JOBS = 4


class MnJob(C.Structure):
    """MorlMnJob of include/morl_b200.h"""

    _fields_ = [("g_planes", _vp), ("g_plane_stride", C.c_longlong), ("g_scale", _vp), ("h_planes", _vp), ("h_plane_stride", C.c_longlong),
                ("h_scale", _vp), ("out", _vp), ("colsum_out", _vp), ("ldg", _i), ("g_cols", _i), ("ldh", _i), ("h_cols", _i), ("ld_out", _i)]


_lib = None


class MorlB200Error(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built -- there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MorlB200Error(
            f"{LIB_PATH} not found: build it with `python -m morl_baselines_b200.csrc.build` (nvcc, sm_100a). "
            "morl_baselines_b200 has no CPU / eager fallback for its CUDA operators."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == ABI drift between header and library
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().morl_last_error().decode("utf-8", "replace")
        raise MorlB200Error(f"{what} failed (code {rc}): {msg}")
