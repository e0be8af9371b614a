"""ctypes binding of libvtgs_cuda.so (include/vtgs.h).  No CPU fallback: `lib()` raises
if the library has not been built, and every op raises on non-CUDA tensors."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# VTGS_LIB_PATH: load another build of the same library (kernel experiments: csrc/Makefile OUT= / EXTRA=)
LIB_PATH = os.environ.get("VTGS_LIB_PATH") or os.path.join(_HERE, "lib", "libvtgs_cuda.so")
CSRC = os.path.join(_HERE, "csrc")

ABI_VERSION = 4
MEDIAN_STATE_WORDS = 264
MEDIAN_SUMMABLE_WORDS = 257
TRACK_BOOK_POST_STEP = 1
TRACK_CALLER_METRIC = 2
GEOM_RECORD_BYTES = 64
GRAD_GEOM_FLOATS = 32
BUF_DETERMINISTIC = 1
BA_RECORD_WORDS = 20


class VtgsCamera(C.Structure):
    _fields_ = [
        ("image_width", C.c_int32), ("image_height", C.c_int32),
        ("tanfovx", C.c_float), ("tanfovy", C.c_float),
        ("viewmatrix", C.c_float * 16), ("projmatrix", C.c_float * 16),
        ("bg", C.c_float * 3), ("scale_modifier", C.c_float),
        ("radius_sigma_mult", C.c_float),
        ("tile_row_begin", C.c_int32), ("tile_row_end", C.c_int32),
    ]


class VtgsCounters(C.Structure):
    _fields_ = [
        ("num_rendered", C.c_uint32), ("overflow", C.c_uint32), ("max_tile_pairs", C.c_uint32),
        ("reserved0", C.c_uint32),
        ("pose_R", C.c_float * 9), ("pose_t", C.c_float * 3), ("pose_q", C.c_float * 4),
        ("pose_qnorm", C.c_float * 2), ("reserved1", C.c_float * 10),
    ]


class VtgsBuffers(C.Structure):
    _fields_ = [
        ("geom", C.c_void_p), ("tiles_touched", C.c_void_p), ("tile_counts", C.c_void_p),
        ("tile_ranges", C.c_void_p), ("pair_keys", C.c_void_p), ("point_list", C.c_void_p),
        ("final_T", C.c_void_p), ("n_contrib", C.c_void_p), ("grad_geom", C.c_void_p),
        ("counters", C.c_void_p), ("region_pairs", C.c_void_p), ("region_cnt", C.c_void_p),
        ("region_masks", C.c_void_p), ("region_done", C.c_void_p), ("pair_capacity", C.c_uint64),
        ("band_flags", C.c_void_p), ("band_cand", C.c_void_p), ("tile_order", C.c_void_p),
        ("flags", C.c_uint32), ("reserved", C.c_uint32),
    ]


class VtgsWorkspaceSizes(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "geom_bytes", "tiles_touched_bytes", "tile_counts_bytes", "tile_ranges_bytes", "pair_keys_bytes",
        "point_list_bytes", "final_T_bytes", "n_contrib_bytes", "grad_geom_bytes", "counters_bytes",
        "region_pairs_bytes", "region_cnt_bytes", "region_masks_bytes", "region_done_bytes", "band_flags_bytes", "band_cand_bytes", "tile_order_bytes")] + \
        [("tiles_x", C.c_uint32), ("tiles_y", C.c_uint32)]


class VtgsParams(C.Structure):
    _fields_ = [
        ("means3D", C.c_void_p), ("rgb_colors", C.c_void_p), ("unnorm_rotations", C.c_void_p),
        ("logit_opacities", C.c_void_p), ("log_scales", C.c_void_p),
        ("log_scales_dim", C.c_int32), ("pad_", C.c_int32), ("num_gaussians", C.c_int64),
    ]


class VtgsPose(C.Structure):
    _fields_ = [("cam_unnorm_rot", C.c_void_p), ("cam_trans", C.c_void_p), ("depth_row", C.c_float * 4)]


class VtgsLossConfig(C.Structure):
    _fields_ = [
        ("mode", C.c_int32), ("use_sil_for_loss", C.c_int32), ("ignore_outlier_depth", C.c_int32),
        ("use_l1", C.c_int32), ("sil_thres", C.c_float), ("w_im", C.c_float), ("w_depth", C.c_float),
        ("far_depth_thres", C.c_float), ("pixel_mask", C.c_void_p),
        ("sil_thres_dev", C.c_void_p), ("median_state", C.c_void_p),
    ]


class VtgsParamGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "means3D", "rgb_colors", "unnorm_rotations", "logit_opacities", "log_scales", "means2D",
        "cam_unnorm_rot", "cam_trans", "pose_scratch", "pose_scale", "dL_abs_bound")]


# every symbol include/vtgs.h declares: (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "vtgs_abi_version": (C.c_int, []),
    "vtgs_last_error": (C.c_char_p, []),
    "vtgs_build_info": (C.c_char_p, []),
    "vtgs_workspace_query": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_uint64, C.POINTER(VtgsWorkspaceSizes)]),
    "vtgs_forward": (C.c_int, [C.POINTER(VtgsCamera), C.c_int64] + [_P] * 5 + [_P, _P, _P, C.POINTER(VtgsBuffers), _P]),
    "vtgs_backward": (C.c_int, [C.POINTER(VtgsCamera), C.c_int64] + [_P] * 5 + [_P] + [_P] * 6 + [C.POINTER(VtgsBuffers), _P]),
    "vtgs_mark_visible": (C.c_int, [C.POINTER(VtgsCamera), C.c_int64, _P, _P, _P]),
    "vtgs_export_sorted_keys": (C.c_int, [C.POINTER(VtgsCamera), C.c_int64, C.POINTER(VtgsBuffers), _P, C.c_uint64, _P]),
    "vtgs_export_geometry": (C.c_int, [C.c_int64, C.POINTER(VtgsBuffers), _P, _P, _P, _P]),
    "vtgs_fused_forward": (C.c_int, [C.POINTER(VtgsCamera), C.POINTER(VtgsParams), C.POINTER(VtgsPose), _P, _P, C.POINTER(VtgsBuffers), _P]),
    "vtgs_loss": (C.c_int, [C.POINTER(VtgsCamera), C.POINTER(VtgsLossConfig)] + [_P] * 6 + [_P]),
    "vtgs_loss_scratch_floats": (C.c_uint64, [C.c_int32, C.c_int32, C.c_int32]),
    "vtgs_pose_scratch_floats": (C.c_uint64, [C.c_int64]),
    "vtgs_fused_backward": (C.c_int, [C.POINTER(VtgsCamera), C.POINTER(VtgsParams), C.POINTER(VtgsPose), _P, C.c_int32,
                                      C.POINTER(VtgsParamGrads), C.POINTER(VtgsBuffers), _P]),
    "vtgs_fused_tracking_step": (C.c_int, [C.POINTER(VtgsCamera), C.POINTER(VtgsParams), C.POINTER(VtgsPose), C.POINTER(VtgsLossConfig)] +
                                 [_P] * 7 + [C.POINTER(VtgsParamGrads), _P, _P, C.POINTER(VtgsBuffers), _P]),
    "vtgs_sharded_adam": (C.c_int, [C.c_int32, C.c_int32, _P, C.c_uint64, C.c_int64, C.c_int64, C.c_int64, _P, _P, C.c_int64, C.c_int32, _P, _P,
                                    C.c_float, C.c_float, C.c_float, _P, _P, _P]),
    "vtgs_retie": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_float * 12), _P, _P, _P]),
    "vtgs_retie_dev": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, _P]),
    "vtgs_retie_records": (C.c_int, [C.c_int32, _P, C.c_int32, _P, C.c_int64, _P, _P]),
    "vtgs_tracking_update": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_float, C.c_float, C.c_float, C.c_int32, _P]),
    "vtgs_median_hist": (C.c_int, [C.POINTER(VtgsCamera), _P, _P, C.c_int32, _P, _P]),
    "vtgs_median_pick": (C.c_int, [C.c_int64, C.c_int32, _P, _P]),
    "vtgs_sil_ladder": (C.c_int, [C.POINTER(VtgsCamera), _P, _P, _P, _P, _P, _P]),
    "vtgs_sil_select": (C.c_int, [_P, _P, _P, _P]),
    "vtgs_nonpresence_mask": (C.c_int, [C.POINTER(VtgsCamera), _P, _P, C.c_float, _P, _P, _P, _P]),
    "vtgs_eval_scratch_floats": (C.c_uint64, []),
    "vtgs_eval_metrics": (C.c_int, [C.POINTER(VtgsCamera), _P, _P, _P, C.c_float, C.c_int32, _P, _P, _P]),
    "vtgs_p2p_prepare": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_float * 4), C.POINTER(C.c_float * 12), _P, _P, _P, _P, _P, _P, _P]),
    "vtgs_p2p_match": (C.c_int, [C.c_int64, _P, _P, _P, C.c_int64, _P, _P, C.c_float, _P, C.c_int64, _P, _P, _P, _P]),
    "vtgs_frame_convert": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, C.c_double, _P, _P, _P]),
    "vtgs_book_radii": (C.c_int, [C.c_int64, _P, _P, _P, _P]),
    "vtgs_ffma_probe": (C.c_int, [C.c_int64, _P, C.POINTER(C.c_uint64), _P]),
    "vtgs_profile_enable": (C.c_int, [C.c_int32]),
    "vtgs_profile_summary": (C.c_int, [C.c_char_p, C.c_uint64]),
    "vtgs_adam": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int32, _P, _P]),
}


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a with nvcc (csrc/Makefile) into lib/libvtgs_cuda.so."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    srcs.append(os.path.join(_HERE, "..", "include", "vtgs.h"))
    stale = (not os.path.exists(LIB_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        cmd = ["make", "-C", CSRC] + (["-B"] if force else [])
        subprocess.run(cmd, check=True, stdout=None if verbose else subprocess.DEVNULL)
    return LIB_PATH


_lib = None


def lib():
    """The loaded CUDA library.  Raises (loudly) if it is missing: there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C vtgaussian_slam_b200/csrc`). vtgaussian_slam_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)          # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        if L.vtgs_abi_version() != ABI_VERSION:
            raise RuntimeError("libvtgs_cuda.so ABI version mismatch")
        _lib = L
    return _lib


class VtgsError(RuntimeError):
    pass


def check(code: int):
    if code != 0:
        msg = lib().vtgs_last_error().decode()
        if code == -3:
            raise NotImplementedError(msg)
        raise VtgsError(f"vtgs error {code}: {msg}")


def profile_enable(on: bool):
    check(lib().vtgs_profile_enable(1 if on else 0))


def profile_summary():
    """-> {kernel name: (launches, total_ms)} of everything launched since profile_enable(True)."""
    buf = C.create_string_buffer(1 << 16)
    check(lib().vtgs_profile_summary(buf, len(buf)))
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms = line.split()
        out[name] = (int(n), float(ms))
    return out
