"""ctypes binding of libvc_b200.so (C ABI: include/vc_b200.h).

There is NO fallback: if the shared library is missing or a call fails this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VC_B200_LIB") or os.path.join(_HERE, "libvc_b200.so")   # override: A/B builds of the kernels

ABI_VERSION = 7


class VcError(RuntimeError):
    pass


class GemmDesc(C.Structure):
    _fields_ = [("a", C.c_void_p), ("lda", C.c_int32), ("a2", C.c_void_p), ("lda2", C.c_int32),
                ("X", C.c_int32), ("Y", C.c_int32), ("Z", C.c_int32), ("bx", C.c_int32), ("by", C.c_int32),
                ("K", C.c_int32), ("K1", C.c_int32), ("w", C.c_void_p), ("ldw", C.c_int32), ("N", C.c_int32), ("num_taps", C.c_int32),
                ("tap_dx", C.c_int32 * 9), ("tap_dy", C.c_int32 * 9),
                ("out", C.c_void_p), ("out_f32", C.c_void_p), ("ldo", C.c_int32),
                ("bias", C.c_void_p), ("bias_z_div", C.c_int32), ("res", C.c_void_p), ("ldr", C.c_int32),
                ("geglu", C.c_int32), ("ln_stats", C.c_void_p), ("ln_colsum", C.c_void_p), ("ln_part", C.c_void_p),
                ("ldo_y", C.c_int64), ("ldo_z", C.c_int64), ("gn_part", C.c_void_p), ("gn_sub", C.c_int32),
                ("peer", C.c_void_p)]


class GemmPeer(C.Structure):
    _fields_ = [("mode", C.c_int32), ("world", C.c_int32), ("rank", C.c_int32), ("B", C.c_int32), ("T", C.c_int32), ("HW", C.c_int32),
                ("f0", C.c_int32 * 9), ("dst", C.c_void_p * 8)]


class GnPartGeom(C.Structure):
    _fields_ = [("part", C.c_void_p), ("n_chunks", C.c_int32), ("sub", C.c_int32), ("rb_per_z", C.c_int64),
                ("samples_per_z", C.c_int32), ("rb_per_sample", C.c_int64)]


class AttnDesc(C.Structure):
    _fields_ = [("q", C.c_void_p), ("ldq", C.c_int32), ("k", C.c_void_p), ("ldk", C.c_int32),
                ("v", C.c_void_p), ("ldv", C.c_int32), ("out", C.c_void_p), ("ldo", C.c_int32),
                ("B", C.c_int32), ("heads", C.c_int32), ("Nq", C.c_int32), ("Nk", C.c_int32),
                ("kv_batch_stride", C.c_int64), ("scale", C.c_float), ("accumulate", C.c_int32)]


class DdimScalars(C.Structure):
    _fields_ = [("cfg_scale", C.c_float), ("guidance_rescale", C.c_float), ("sqrt_ac_t", C.c_float),
                ("sqrt_1mac_t", C.c_float), ("a_prev", C.c_float), ("sigma_t", C.c_float),
                ("scale_t", C.c_float), ("prev_scale_t", C.c_float), ("use_cfg", C.c_int32)]


class PeerComm(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("flags", C.c_void_p), ("peer_flags", C.c_void_p * 8),
                ("seq", C.c_void_p), ("done", C.c_void_p), ("stats_slots", C.c_void_p * 8), ("cur_stats", C.c_void_p),
                ("Bmax", C.c_int32)]


_vp, _i32, _i64, _f32, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/vc_b200.h declares (tests check this)
SIGNATURES = {
    "vc_abi_version": (C.c_int, []),
    "vc_last_error": (C.c_char_p, []),
    "vc_launch_count": (C.c_longlong, []),
    "vc_reset_launch_count": (None, []),
    "vc_gemm_tap": (C.c_int, [C.POINTER(GemmDesc), _vp]),
    "vc_gemm_tile_n": (C.c_int, [_i32, _i32]),
    "vc_flash_attn_d64": (C.c_int, [C.POINTER(AttnDesc), _vp]),
    "vc_temporal_attn": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _i32, _i32, _i64, _i32, _f32, _vp]),
    "vc_groupnorm_ws_bytes": (_sz, [_i32]),
    "vc_groupnorm_nhwc": (C.c_int, [_vp, _i32, _vp, _i32, _i32, _i64, _vp, _vp, _f32, _i32, _vp, _vp, _sz, _vp]),
    "vc_groupnorm_stats": (C.c_int, [_vp, _i32, _vp, _i32, _i32, _i64, _vp, _vp, _sz, _vp]),
    "vc_groupnorm_apply": (C.c_int, [_vp, _i32, _vp, _i32, _i32, _i64, _vp, _i64, _vp, _vp, _f32, _i32, _vp, _vp]),
    "vc_groupnorm_parts_ws_bytes": (_sz, [_i32]),
    "vc_groupnorm_from_parts": (C.c_int, [_vp, _i32, C.POINTER(GnPartGeom), _vp, _i32, C.POINTER(GnPartGeom), _i32, _i64, _vp, _vp, _f32, _i32,
                                          _vp, _vp, _sz, _vp]),
    "vc_groupnorm_apply_parts": (C.c_int, [_vp, _i32, _i32, _i64, _vp, _i32, _i64, _vp, _vp, _f32, _i32, _vp, _vp]),
    "vc_enable_peer_access": (C.c_int, [_i32]),
    "vc_peer_alloc": (C.c_int, [_sz, C.POINTER(C.c_void_p), _vp]),
    "vc_peer_open": (C.c_int, [_vp, C.POINTER(C.c_void_p)]),
    "vc_peer_close": (C.c_int, [_vp]),
    "vc_peer_free": (C.c_int, [_vp]),
    "vc_peer_exchange": (C.c_int, [C.POINTER(PeerComm), _vp, C.POINTER(C.c_void_p), _i32, _i32, _i32, _i32, _i32, C.POINTER(C.c_int32), _i32,
                                   _vp, _sz, _vp]),
    "vc_peer_finish_scatter": (C.c_int, [C.POINTER(PeerComm), _vp, _i32, _i32, _vp, _sz, _vp]),
    "vc_peer_groupnorm_stats": (C.c_int, [C.POINTER(PeerComm), _vp, _i32, _i32, _i64, _vp, _sz, _vp]),
    "vc_layernorm_stats": (C.c_int, [_vp, _i64, _i32, _f32, _vp, _vp]),
    "vc_layernorm_stats_from_parts": (C.c_int, [_vp, _i64, _i32, _f32, _vp, _vp]),
    "vc_layernorm": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _f32, _vp, _vp]),
    "vc_softmax_rows_f32": (C.c_int, [_vp, _i64, _i64, _f32, _vp, _vp]),
    "vc_upsample2x_nhwc": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "vc_im2col3x3_s2": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "vc_ncthw_f32_to_rows_f16": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i64, _i32, _i32, _vp]),
    "vc_rows_f32_to_ncthw": (C.c_int, [_vp, _i32, _vp, _i32, _i32, _i32, _i64, _vp]),
    "vc_rows_f16_to_nchw_f32": (C.c_int, [_vp, _i32, _vp, _i32, _i32, _i64, _vp]),
    "vc_cast_f32_to_f16": (C.c_int, [_vp, _vp, _i64, _vp]),
    "vc_add_f16": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "vc_gelu_f16": (C.c_int, [_vp, _vp, _i64, _vp]),
    "vc_timestep_embedding": (C.c_int, [_vp, _i32, _i32, _vp, _vp]),
    "vc_small_linear_f32": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "vc_ddim_update": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, C.POINTER(DdimScalars), _vp, _vp]),
    "vc_ddim_update3": (C.c_int, [_vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _i64, C.POINTER(DdimScalars), _vp, _vp]),
}

_lib = None


def load():
    """Load the library and bind every symbol; raises VcError if it is missing (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VcError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                      f"(or viewcrafter_b200/csrc/build.sh). There is no non-CUDA fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.vc_abi_version() != ABI_VERSION:
        raise VcError(f"libvc_b200.so ABI {lib.vc_abi_version()} != binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().vc_last_error()
        raise VcError(f"{what} failed (status {rc}): {msg.decode() if msg else '?'}")
