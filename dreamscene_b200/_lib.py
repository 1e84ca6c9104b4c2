"""ctypes binding of libb200gsr.so (include/b200gsr.h).  Fails loudly if the library is missing:
there is NO CPU or PyTorch fallback in the product path."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200GSR_LIB", os.path.join(HERE, "libb200gsr.so"))   # override: A/B builds only

EXPORTS = ["b200gsr_version", "b200gsr_last_error", "b200gsr_saved_layout_query",
           "b200gsr_scratch_layout_query", "b200gsr_forward", "b200gsr_backward", "b200gsr_backward_ex",
           "b200gsr_mark_visible", "b200gsr_profile_enable", "b200gsr_profile_counts",
           "b200gsr_profile_read", "b200gsr_debug_counters", "b200gsr_dist2_scratch_bytes", "b200gsr_dist2_knn3",
           "b200gsr_assemble_forward", "b200gsr_assemble_backward", "b200gsr_disparity_forward",
           "b200gsr_disparity_backward", "b200gsr_densify_stats", "b200gsr_densify_scratch_bytes",
           "b200gsr_densify_plan", "b200gsr_densify_map", "b200gsr_compact_plan", "b200gsr_gather_rows",
           "b200gsr_split_children", "b200gsr_kth_smallest", "b200gsr_views_geometry", "b200gsr_forward_views",
           "b200gsr_backward_views", "b200gsr_sh_grad_expand"]


class Params(C.Structure):
    _fields_ = [("P", C.c_int32), ("M", C.c_int32), ("sh_degree", C.c_int32),
                ("image_height", C.c_int32), ("image_width", C.c_int32),
                ("tanfovx", C.c_float), ("tanfovy", C.c_float), ("scale_modifier", C.c_float),
                ("prefiltered", C.c_int32), ("score_flag", C.c_int32),
                ("bg", C.c_void_p), ("viewmatrix", C.c_void_p), ("projmatrix", C.c_void_p),
                ("campos", C.c_void_p)]


class Group(C.Structure):           # == b200gsr_group
    _fields_ = [(n, C.c_void_p) for n in ("xyz", "opacity", "scaling", "rotation", "f_dc", "f_rest")] + [("n", C.c_int32)]


class GroupGrad(C.Structure):       # == b200gsr_group_grad
    _fields_ = [(n, C.c_void_p) for n in ("xyz", "opacity", "scaling", "rotation", "f_dc", "f_rest")]


MAX_GROUPS = 24
MAX_VIEWS = 16


class ViewInputs(C.Structure):      # == b200gsr_view_inputs
    _fields_ = [(n, C.c_void_p) for n in ("means3D", "shs", "colors_precomp", "opacities", "scales", "rotations", "cov3D_precomp")]


class ViewGrads(C.Structure):       # == b200gsr_view_grads
    _fields_ = [(n, C.c_void_p) for n in ("d_means3D", "d_means2D", "d_shs", "d_colors", "d_opacities", "d_scales",
                                          "d_rotations", "d_cov3D")] + [("accumulate", C.c_uint32)]


class SavedLayout(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in ("header", "tile_start", "work_order", "n_contrib",
                                          "keys", "geom", "dgeom", "bwd_items", "total")]


class ScratchLayout(C.Structure):
    _fields_ = [(n, C.c_size_t) for n in ("counters", "tile_count", "tile_cursor", "rectdepth",
                                          "ms_hist", "total")]


_lib = None
ABI_VERSION = 4
FWD_NO_BACKWARD = 1


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        # Not a fallback: the only thing ever attempted is compiling the same sm_100a sources in-tree.
        err = None
        if "B200GSR_LIB" not in os.environ and not os.environ.get("B200GSR_NO_AUTOBUILD"):
            try:
                from . import _build
                _build.build()
            except Exception as e:   # noqa: BLE001 - reported below
                err = e
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing and could not be built ({err}). Build it with "
                "`python -m dreamscene_b200._build` (needs nvcc; sm_100a only). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, sz, u64, u32, i32 = C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint32, C.c_int32
    lib.b200gsr_version.restype = C.c_int
    lib.b200gsr_last_error.restype = C.c_char_p
    lib.b200gsr_saved_layout_query.argtypes = [i32, i32, i32, u64, i32, C.POINTER(SavedLayout)]
    lib.b200gsr_scratch_layout_query.argtypes = [i32, i32, i32, u64, C.POINTER(ScratchLayout)]
    lib.b200gsr_forward.argtypes = [C.POINTER(Params)] + [vp] * 7 + [vp] * 4 + \
        [vp, sz, vp, sz, u64, u32, vp, u32, vp]
    lib.b200gsr_backward.argtypes = [C.POINTER(Params)] + [vp] * 7 + [vp] * 4 + \
        [vp, sz, vp, sz, u64] + [vp] * 8 + [vp]
    lib.b200gsr_backward_ex.argtypes = lib.b200gsr_backward.argtypes[:-1] + [i32, vp]
    lib.b200gsr_backward_ex.restype = C.c_int
    lib.b200gsr_mark_visible.argtypes = [i32, vp, vp, vp, vp, vp]
    lib.b200gsr_sh_grad_expand.argtypes = [i32, i32, i32, i32, vp, vp, sz, vp, vp]
    lib.b200gsr_sh_grad_expand.restype = C.c_int
    lib.b200gsr_dist2_scratch_bytes.argtypes = [i32]
    lib.b200gsr_dist2_scratch_bytes.restype = C.c_size_t
    lib.b200gsr_dist2_knn3.argtypes = [i32, vp, vp, vp, sz, vp]
    lib.b200gsr_dist2_knn3.restype = C.c_int
    lib.b200gsr_assemble_forward.argtypes = [i32, C.POINTER(Group), i32, i32, C.c_float, C.c_float, vp, vp, u64] + [vp] * 5 + [vp]
    lib.b200gsr_assemble_backward.argtypes = [i32, C.POINTER(Group), C.POINTER(GroupGrad), i32, i32, C.c_float, C.c_float,
                                              vp, vp, u64] + [vp] * 5 + [vp]
    lib.b200gsr_assemble_forward.restype = lib.b200gsr_assemble_backward.restype = C.c_int
    lib.b200gsr_disparity_forward.argtypes = [i32, i32, vp, vp, vp, vp, vp]
    lib.b200gsr_disparity_backward.argtypes = [i32, i32, vp, vp, vp, vp, vp, vp, vp]
    lib.b200gsr_disparity_forward.restype = lib.b200gsr_disparity_backward.restype = C.c_int
    f = C.c_float
    lib.b200gsr_densify_stats.argtypes = [i32, vp, vp, vp, vp, vp, vp]
    lib.b200gsr_densify_scratch_bytes.argtypes = [i32]
    lib.b200gsr_densify_scratch_bytes.restype = C.c_size_t
    lib.b200gsr_densify_plan.argtypes = [i32, vp, vp, vp, vp, f, f, f, f, f, vp, vp, vp]
    lib.b200gsr_densify_map.argtypes = [i32, i32, vp, vp, vp, vp, vp]
    lib.b200gsr_compact_plan.argtypes = [i32, vp, vp, vp, vp, vp]
    lib.b200gsr_gather_rows.argtypes = [i32, i32, vp, vp, vp, i32, vp]
    lib.b200gsr_split_children.argtypes = [i32, i32, f, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.b200gsr_kth_smallest.argtypes = [i32, vp, u32, vp, vp, vp]
    for fn in ("b200gsr_densify_stats", "b200gsr_densify_plan", "b200gsr_densify_map", "b200gsr_compact_plan",
               "b200gsr_gather_rows", "b200gsr_split_children", "b200gsr_kth_smallest"):
        getattr(lib, fn).restype = C.c_int
    lib.b200gsr_views_geometry.argtypes = [i32, i32, i32, C.POINTER(i32)]
    lib.b200gsr_forward_views.argtypes = [i32, C.POINTER(Params), C.POINTER(ViewInputs), vp, vp, vp, vp, vp, sz, vp, sz,
                                          u64, u32, vp, u32, vp]
    lib.b200gsr_backward_views.argtypes = [i32, C.POINTER(Params), C.POINTER(ViewInputs), vp, vp, vp, vp, vp, sz, u64,
                                           C.POINTER(ViewGrads), vp]
    for fn in ("b200gsr_views_geometry", "b200gsr_forward_views", "b200gsr_backward_views"):
        getattr(lib, fn).restype = C.c_int
    lib.b200gsr_debug_counters.argtypes = [vp]
    lib.b200gsr_debug_counters.restype = C.c_int
    lib.b200gsr_profile_enable.argtypes = [i32]
    lib.b200gsr_profile_counts.argtypes = [C.POINTER(i32), C.POINTER(i32)]
    lib.b200gsr_profile_read.argtypes = [i32, i32, C.POINTER(C.c_float)]
    for f in ("b200gsr_profile_enable", "b200gsr_profile_counts", "b200gsr_profile_read"):
        getattr(lib, f).restype = C.c_int
    for f in ("b200gsr_saved_layout_query", "b200gsr_scratch_layout_query", "b200gsr_forward",
              "b200gsr_backward", "b200gsr_mark_visible"):
        getattr(lib, f).restype = C.c_int
    if lib.b200gsr_version() != ABI_VERSION:
        raise RuntimeError(f"{LIB_PATH} has ABI version {lib.b200gsr_version()}, this package needs "
                           f"{ABI_VERSION}: rebuild with `python -m dreamscene_b200._build --force`")
    _lib = lib
    return lib


def last_error() -> str:
    return load().b200gsr_last_error().decode("utf-8", "replace")


def saved_layout(P: int, H: int, W: int, max_pairs: int, with_backward: bool = True) -> SavedLayout:
    out = SavedLayout()
    rc = load().b200gsr_saved_layout_query(P, H, W, max_pairs, int(bool(with_backward)), C.byref(out))
    if rc:
        raise RuntimeError(f"b200gsr_saved_layout_query failed ({rc}): {last_error()}")
    return out


def scratch_layout(P: int, H: int, W: int, max_pairs: int) -> ScratchLayout:
    out = ScratchLayout()
    rc = load().b200gsr_scratch_layout_query(P, H, W, max_pairs, C.byref(out))
    if rc:
        raise RuntimeError(f"b200gsr_scratch_layout_query failed ({rc}): {last_error()}")
    return out


FWD_STAGES = ("project_sh", "scan_order", "scatter", "tile_sort", "composite_fwd")
BWD_STAGES = ("composite_bwd", "project_bwd")


def profile_enable(max_calls: int) -> None:
    rc = load().b200gsr_profile_enable(int(max_calls))
    if rc:
        raise RuntimeError(f"b200gsr_profile_enable failed ({rc}): {last_error()}")


def profile_collect() -> dict:
    """-> {stage: [ms per recorded call]} for every call recorded since profile_enable."""
    lib = load()
    nf, nb = C.c_int32(0), C.c_int32(0)
    lib.b200gsr_profile_counts(C.byref(nf), C.byref(nb))
    out = {k: [] for k in FWD_STAGES + BWD_STAGES}
    buf = (C.c_float * 8)()
    for i in range(nf.value):
        if lib.b200gsr_profile_read(0, i, buf):
            raise RuntimeError(last_error())
        for k, name in enumerate(FWD_STAGES):
            out[name].append(float(buf[k]))
    for i in range(nb.value):
        if lib.b200gsr_profile_read(1, i, buf):
            raise RuntimeError(last_error())
        for k, name in enumerate(BWD_STAGES):
            out[name].append(float(buf[k]))
    return out


STAT_NAMES = ("bwd_pairs_evaluated", "bwd_pairs_contributing", "bwd_lane_contributions", "bwd_k1", "bwd_k2",
              "bwd_k3_4", "bwd_k5_8", "bwd_k9_16", "bwd_k17_32", "_9", "fwd_pairs_evaluated", "fwd_lane_blends",
              "_12", "_13", "_14", "_15",
              "fwd_busy_ns", "fwd_end_ns", "fwd_not_begin_ns", "fwd_workers", "fwd_max_item_ns",
              "bwd_busy_ns", "bwd_end_ns", "bwd_not_begin_ns", "bwd_workers", "bwd_max_item_evals", "bwd_max_item_ns")
STAT_WORDS = 32


def debug_counters(ptr) -> None:
    """ptr: device pointer to STAT_WORDS (32) zeroed uint64 (or None to switch the instrumented kernels off)."""
    rc = load().b200gsr_debug_counters(C.c_void_p(ptr) if ptr else None)
    if rc:
        raise RuntimeError(last_error())
