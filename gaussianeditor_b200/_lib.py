"""ctypes binding of ``csrc/libgsr_b200.so`` (C ABI declared in ``include/gsr_b200.h``).

There is deliberately NO fallback: if the shared library is missing or fails to load, every
entry point of this package raises.  (The CPU oracle under ``oracle/`` is test infrastructure
and is never imported from here.)
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libgsr_b200.so")

# every symbol include/gsr_b200.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "gsr_abi_version", "gsr_last_error", "gsr_geometry_bytes", "gsr_image_bytes", "gsr_binning_bytes",
    "gsr_backward_scratch_bytes", "gsr_forward_preprocess", "gsr_forward_render",
    "gsr_forward_render_speculative", "gsr_backward",
    "gsr_mark_visible", "gsr_apply_weights", "gsr_view_geometry", "gsr_view_binning", "gsr_view_image",
    "gsr_set_option", "gsr_get_option", "gsr_launch_count", "gsr_profile_read", "gsr_host_create", "gsr_host_destroy",
    "gsr_host_upload_cloud", "gsr_host_step",
    "gsr_view_exchange", "gsr_shard_preprocess", "gsr_shard_order", "gsr_shard_render", "gsr_shard_backward_render",
    "gsr_shard_backward_preprocess",
    "gsr_peer_alloc", "gsr_peer_open", "gsr_peer_close", "gsr_peer_free", "gsr_shard_preprocess_p2p",
    "gsr_forward_preprocess_raw", "gsr_backward_raw",
    "gsr_alpha_image", "gsr_backward_alpha", "gsr_camera_scratch_bytes", "gsr_backward_camera",
    "gsr_sparse_local_bytes", "gsr_sparse_candidate_bytes", "gsr_sparse_view", "gsr_sparse_preprocess", "gsr_sparse_order",
    "gsr_sparse_return", "gsr_sparse_backward_preprocess", "gsr_frame_broadcast", "gsr_peer_barrier",
    "gsr_backward_depth", "gsr_backward_raw_depth",
]


class Settings(C.Structure):
    _fields_ = [
        ("image_height", C.c_int32), ("image_width", C.c_int32), ("tanfovx", C.c_float), ("tanfovy", C.c_float),
        ("scale_modifier", C.c_float), ("sh_degree", C.c_int32), ("sh_coeffs", C.c_int32),
        ("prefiltered", C.c_int32), ("debug", C.c_int32),
        ("bg", C.c_void_p), ("viewmatrix", C.c_void_p), ("projmatrix", C.c_void_p), ("campos", C.c_void_p),
    ]


class Cloud(C.Structure):
    _fields_ = [
        ("P", C.c_int32), ("means3D", C.c_void_p), ("opacities", C.c_void_p), ("shs", C.c_void_p),
        ("colors_precomp", C.c_void_p), ("scales", C.c_void_p), ("rotations", C.c_void_p),
        ("cov3D_precomp", C.c_void_p),
    ]


class Grads(C.Structure):
    _fields_ = [
        ("dL_dmeans3D", C.c_void_p), ("dL_dmeans2D", C.c_void_p), ("dL_dcolors", C.c_void_p),
        ("dL_dopacity", C.c_void_p), ("dL_dcov3D", C.c_void_p), ("dL_dsh", C.c_void_p),
        ("dL_dscales", C.c_void_p), ("dL_drotations", C.c_void_p),
    ]


class CameraGrads(C.Structure):
    _fields_ = [("dL_dviewmatrix", C.c_void_p), ("dL_dprojmatrix", C.c_void_p), ("dL_dcampos", C.c_void_p),
                ("scratch", C.c_void_p), ("scratch_bytes", C.c_size_t)]


class GeometryView(C.Structure):
    _fields_ = [("records", C.c_void_p), ("tiles_touched", C.c_void_p), ("clamped", C.c_void_p),
                ("depth_order", C.c_void_p)]


class BinningView(C.Structure):
    _fields_ = [("point_list", C.c_void_p), ("tile_keys", C.c_void_p), ("tile_key_bytes", C.c_int32)]


class ImageView(C.Structure):
    _fields_ = [("final_T", C.c_void_p), ("n_contrib", C.c_void_p), ("ranges", C.c_void_p)]


class RawCloud(C.Structure):
    _fields_ = [("P", C.c_int32), ("means3D", C.c_void_p), ("opacity_logits", C.c_void_p), ("features_dc", C.c_void_p),
                ("features_rest", C.c_void_p), ("log_scales", C.c_void_p), ("raw_rotations", C.c_void_p)]


class RawGrads(C.Structure):
    _fields_ = [("dL_dmeans3D", C.c_void_p), ("dL_dmeans2D", C.c_void_p), ("dL_dopacity_logits", C.c_void_p),
                ("dL_dfeatures_dc", C.c_void_p), ("dL_dfeatures_rest", C.c_void_p), ("dL_dlog_scales", C.c_void_p),
                ("dL_draw_rotations", C.c_void_p)]


class TileOwner(C.Structure):
    _fields_ = [("row_stride", C.c_int32), ("row_phase", C.c_int32)]


class ExchangeView(C.Structure):
    _fields_ = [("records", C.c_void_p)]


class SparsePlan(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("slice_len", C.c_int32), ("seg_cap", C.c_int32)]


class SparseView(C.Structure):
    _fields_ = [("records", C.c_void_p), ("ret", C.c_void_p), ("geometry_bytes", C.c_size_t)]


_lib = None


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into csrc/libgsr_b200.so (nvcc cross-compiles without a GPU)."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc"), "-j8"], stdout=out)
    return LIB_PATH


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU or PyTorch fallback for the rasterizer)")
    lib = C.CDLL(LIB_PATH)
    for name in SYMBOLS:
        if not hasattr(lib, name):
            raise RuntimeError(f"{LIB_PATH} does not export {name}")
    sz, vp, i32, i64 = C.c_size_t, C.c_void_p, C.c_int32, C.c_int64
    lib.gsr_abi_version.restype = C.c_int
    lib.gsr_last_error.restype = C.c_char_p
    lib.gsr_geometry_bytes.restype = sz; lib.gsr_geometry_bytes.argtypes = [i32]
    lib.gsr_image_bytes.restype = sz; lib.gsr_image_bytes.argtypes = [i32, i32]
    lib.gsr_binning_bytes.restype = sz; lib.gsr_binning_bytes.argtypes = [i32, i64, i32, i32]
    lib.gsr_backward_scratch_bytes.restype = sz; lib.gsr_backward_scratch_bytes.argtypes = [i32]
    lib.gsr_forward_preprocess.restype = C.c_int
    lib.gsr_forward_preprocess.argtypes = [C.POINTER(Settings), C.POINTER(Cloud), vp, sz, vp, vp, vp]
    lib.gsr_forward_render.restype = C.c_int
    lib.gsr_forward_render.argtypes = [C.POINTER(Settings), C.POINTER(Cloud), i32, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp]
    lib.gsr_forward_render_speculative.restype = C.c_int
    lib.gsr_forward_render_speculative.argtypes = lib.gsr_forward_render.argtypes
    lib.gsr_backward.restype = C.c_int
    lib.gsr_backward.argtypes = [C.POINTER(Settings), C.POINTER(Cloud), i32, vp, sz, vp, sz, vp, sz, vp, vp, vp, sz,
                                 C.POINTER(Grads), vp]
    lib.gsr_backward_alpha.restype = C.c_int
    lib.gsr_backward_alpha.argtypes = [C.POINTER(Settings), C.POINTER(Cloud), i32, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp,
                                       sz, C.POINTER(Grads), vp]
    lib.gsr_camera_scratch_bytes.restype = sz; lib.gsr_camera_scratch_bytes.argtypes = [i32]
    lib.gsr_backward_camera.restype = C.c_int
    lib.gsr_backward_camera.argtypes = [C.POINTER(Settings), C.POINTER(Cloud), i32, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp,
                                        sz, C.POINTER(Grads), C.POINTER(CameraGrads), vp]
    lib.gsr_backward_depth.restype = C.c_int
    lib.gsr_backward_depth.argtypes = [C.POINTER(Settings), C.POINTER(Cloud), i32, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp,
                                       vp, sz, C.POINTER(Grads), C.POINTER(CameraGrads), vp]
    lib.gsr_alpha_image.restype = C.c_int
    lib.gsr_alpha_image.argtypes = [vp, sz, i32, i32, vp, vp]
    lib.gsr_mark_visible.restype = C.c_int
    lib.gsr_mark_visible.argtypes = [i32, vp, vp, vp, vp, vp]
    lib.gsr_apply_weights.restype = C.c_int
    lib.gsr_apply_weights.argtypes = [C.POINTER(Settings), C.POINTER(Cloud), i32, vp, sz, vp, sz, vp, sz, vp, vp, i32,
                                      vp, vp, vp]
    lib.gsr_view_geometry.restype = C.c_int; lib.gsr_view_geometry.argtypes = [vp, i32, C.POINTER(GeometryView)]
    lib.gsr_view_binning.restype = C.c_int
    lib.gsr_view_binning.argtypes = [vp, i32, i64, i32, i32, C.POINTER(BinningView)]
    lib.gsr_view_image.restype = C.c_int; lib.gsr_view_image.argtypes = [vp, i32, i32, C.POINTER(ImageView)]
    lib.gsr_set_option.restype = C.c_int; lib.gsr_set_option.argtypes = [C.c_char_p, i64]
    lib.gsr_get_option.restype = i64; lib.gsr_get_option.argtypes = [C.c_char_p]
    lib.gsr_launch_count.restype = i64
    lib.gsr_host_create.restype = vp
    lib.gsr_host_destroy.argtypes = [vp]
    lib.gsr_host_upload_cloud.restype = C.c_int
    lib.gsr_host_upload_cloud.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp]
    lib.gsr_host_step.restype = i64
    lib.gsr_host_step.argtypes = [vp, C.POINTER(Settings), vp, vp, vp, vp]
    S, Cl, TO = C.POINTER(Settings), C.POINTER(Cloud), C.POINTER(TileOwner)
    lib.gsr_view_exchange.restype = C.c_int; lib.gsr_view_exchange.argtypes = [vp, i32, C.POINTER(ExchangeView)]
    lib.gsr_shard_preprocess.restype = C.c_int
    lib.gsr_shard_preprocess.argtypes = [S, Cl, i32, i32, i32, vp, sz, vp, vp]
    lib.gsr_shard_order.restype = C.c_int
    lib.gsr_shard_order.argtypes = [S, TO, i32, vp, sz, vp, vp, vp]
    lib.gsr_shard_render.restype = C.c_int
    lib.gsr_shard_render.argtypes = [S, TO, i32, i32, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp]
    lib.gsr_shard_backward_render.restype = C.c_int
    lib.gsr_shard_backward_render.argtypes = [S, TO, i32, i32, vp, sz, vp, sz, vp, sz, vp, vp, sz, vp]
    lib.gsr_shard_backward_preprocess.restype = C.c_int
    lib.gsr_shard_backward_preprocess.argtypes = [S, Cl, i32, i32, vp, sz, vp, vp, C.POINTER(Grads), vp]
    lib.gsr_peer_alloc.restype = C.c_int; lib.gsr_peer_alloc.argtypes = [sz, C.POINTER(vp), vp]
    lib.gsr_peer_open.restype = C.c_int; lib.gsr_peer_open.argtypes = [vp, C.POINTER(vp)]
    lib.gsr_peer_close.restype = C.c_int; lib.gsr_peer_close.argtypes = [vp]
    lib.gsr_peer_free.restype = C.c_int; lib.gsr_peer_free.argtypes = [vp]
    lib.gsr_shard_preprocess_p2p.restype = C.c_int
    lib.gsr_shard_preprocess_p2p.argtypes = [S, Cl, i32, i32, i32, C.POINTER(vp), i32, i32, sz, vp, vp]
    lib.gsr_forward_preprocess_raw.restype = C.c_int
    lib.gsr_forward_preprocess_raw.argtypes = [S, C.POINTER(RawCloud), vp, sz, vp, vp, vp]
    lib.gsr_backward_raw.restype = C.c_int
    lib.gsr_backward_raw.argtypes = [S, C.POINTER(RawCloud), i32, vp, sz, vp, sz, vp, sz, vp, vp, vp, sz,
                                     C.POINTER(RawGrads), vp]
    lib.gsr_backward_raw_depth.restype = C.c_int
    lib.gsr_backward_raw_depth.argtypes = [S, C.POINTER(RawCloud), i32, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp, sz,
                                           C.POINTER(RawGrads), vp]
    SP = C.POINTER(SparsePlan)
    lib.gsr_sparse_local_bytes.restype = sz; lib.gsr_sparse_local_bytes.argtypes = [i32]
    lib.gsr_sparse_candidate_bytes.restype = sz; lib.gsr_sparse_candidate_bytes.argtypes = [i32, i32]
    lib.gsr_sparse_view.restype = C.c_int; lib.gsr_sparse_view.argtypes = [vp, i32, i32, C.POINTER(SparseView)]
    lib.gsr_sparse_preprocess.restype = C.c_int
    lib.gsr_sparse_preprocess.argtypes = [S, Cl, SP, vp, sz, vp, C.POINTER(vp), sz, vp, vp]
    lib.gsr_sparse_order.restype = C.c_int
    lib.gsr_sparse_order.argtypes = [S, SP, vp, sz, vp, vp, vp, vp]
    lib.gsr_sparse_return.restype = C.c_int
    lib.gsr_sparse_return.argtypes = [SP, vp, vp, C.POINTER(vp), vp]
    lib.gsr_sparse_backward_preprocess.restype = C.c_int
    lib.gsr_sparse_backward_preprocess.argtypes = [S, Cl, SP, vp, sz, vp, vp, sz, vp, sz, C.POINTER(Grads), vp]
    lib.gsr_peer_barrier.restype = C.c_int
    lib.gsr_peer_barrier.argtypes = [i32, i32, C.POINTER(vp), C.c_uint32, i32, vp]
    lib.gsr_frame_broadcast.restype = C.c_int
    lib.gsr_frame_broadcast.argtypes = [TO, i32, i32, vp, C.POINTER(vp), vp]
    if lib.gsr_abi_version() != 2:
        raise RuntimeError("libgsr_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().gsr_last_error().decode(errors="replace")
        raise RuntimeError(f"{what} failed ({rc}): {msg}")


def set_option(name: str, value: int):
    check(load().gsr_set_option(name.encode(), int(value)), f"gsr_set_option({name})")


STAGES = ("preprocess_fwd,depth_order_scan,emit_instances,tile_sort,tile_ranges,render_fwd,render_bwd,"
          "preprocess_bwd,apply_weights").split(",")


def profile_read():
    """{stage: (total_ms, calls)} since the last read (option "profile" must be 1 while the work is issued)."""
    lib = load()
    ms = (C.c_double * len(STAGES))()
    calls = (C.c_int64 * len(STAGES))()
    check(lib.gsr_profile_read(ms, calls), "gsr_profile_read")
    return {n: (ms[i], calls[i]) for i, n in enumerate(STAGES)}


def launch_count() -> int:
    return int(load().gsr_launch_count())
