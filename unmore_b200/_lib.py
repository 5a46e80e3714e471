"""ctypes loader for the C-ABI library (include/unmore_b200.h).

There is deliberately no fallback: if ``libunmore_b200.so`` is missing or a symbol cannot be
resolved, importing the ops fails loudly (build with ``python -c 'import __graft_entry__ as g;
g.build()'`` or ``bash unmore_b200/csrc/build.sh``)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("UNMORE_B200_LIB", os.path.join(_HERE, "libunmore_b200.so"))  # override: A/B builds

_p = C.c_void_p
_i = C.c_int
_f = C.c_float
_d = C.c_double

# name -> argtypes; every function returns int except where noted
SIGNATURES = {
    "unmore_existence_scores": [_p, _i, _i, _i, _i, _i, _p, _i, _p, _i, _p, _p, _p],
    "unmore_existence_scores_aa": [_p, _i, _i, _i, _i, _i, _p, _i, _p, _i, _p, _p, _p],
    "unmore_crop_resize": [_p, _i, _i, _i, _i, _p, _i, _p, _i, _p, _i, _p, _p],
    "unmore_crop_resize_aa": [_p, _i, _i, _i, _i, _p, _i, _p, _i, _p, _i, _p, _p, C.c_size_t, _p],
    "unmore_mask_resize_aa": [_p, _i, _i, _i, _i, _i, _p, _p, C.c_size_t, _p],
    "unmore_tile_means": [_p, C.c_longlong, _i, _p, _p],
    "unmore_center_reasoning_from_tiles": [_p, _i, _i, _i, _p, _i, _p, _i, _d, _p, _p, _p, _p, _p, _p, _p, _p],
    "unmore_boundary_round_from_tiles": [_p, _i, _p, _i, _i, _i, _f, _f, _f, _p, _p, _p, _p, _p],
    "unmore_score_and_rasterise_from_tiles": [_p, _p, _i, _i, _i, _i, _p, _i, _p, _i, _p, _p, _p, _p, _p],
    "unmore_center_reasoning": [_p, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p, _i, _d, _p, _p, _p, _p, _p, _p, _p, _p],
    "unmore_center_reasoning_aa": [_p, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p, _i, _d, _p, _p, _p, _p, _p, _p, _p, _p],
    "unmore_boundary_refine": [_p, _i, _i, _i, _i, _i, _p, _i, _p, _i, _i, _i, _i, _f, _f, _f, _f, _p, _p, _p, _p, _p],
    "unmore_boundary_refine_aa": [_p, _i, _i, _i, _i, _i, _p, _i, _p, _i, _i, _i, _i, _f, _f, _f, _f, _p, _p, _p, _p, _p],
    "unmore_update_bbox_from_tiles": [_p, _i, _p, _p, _p],
    "unmore_compact_boxes": [_p, _i, _p, _i, _i, _i, _p, _f, _p, _i, _i, _p, _i, _p, _p, _p, _i, _p],
    "unmore_box_nms": [_p, _p, _p, _i, _i, _f, _p, _p, _p, _p, _p],
    "unmore_batch_erode": [_p, _i, _i, _i, _i, _i, _p, _p],
    "unmore_connected_components": [_p, _i, _i, _i, _p, _p, _p],
    "unmore_anti_center_map": [_p, _i, _i, _i, _i, _p, _p],
    "unmore_box_nms_matrix": [_p, _p, _i, _f, _p, _p, _p, _p, _p],
    "unmore_score_and_rasterise": [_p, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p, _i, _p, _p, _p, _p, _p],
    "unmore_mask_resize": [_p, _i, _i, _i, _i, _i, _p, _p],
    "unmore_final_scores": [_p, _p, _p, _p, _p, _i, _i, _d, _d, _d, _p, _p, _p, _p],
    "unmore_pack_detections": [_p, _p, _p, _p, _i, _i, _p, _i, _p],
    "unmore_sat_build": [_p, _i, _i, _i, _p, _p],
    "unmore_sat_build_fields": [_p, _i, _i, _i, _i, _p, _i, _p, _p],
    "unmore_box_sums": [_p, _i, _i, _i, _i, _i, _p, _i, _p, _i, _p, _p, _p],
    "unmore_mask_pack": [_p, C.c_size_t, _i, _i, _p, _p],
    "unmore_mask_stats": [_p, _i, _i, _i, _p, _p, _p],
    "unmore_mask_rle_counts": [_p, _i, _i, _i, _i, _p, _p, _p],
    "unmore_mask_nms": [_p, _i, _i, _i, _p, _p, _p, _f, _p, _p, _p, _p, _p],
    # padded stacks of images of different sizes: H, W are the pitch, the pointer after W is image_hw [n_img, 2]
    "unmore_existence_scores_hw": [_p, _i, _i, _i, _i, _p, _i, _p, _i, _p, _i, _p, _p, _p],
    "unmore_center_reasoning_hw": [_p, _i, _i, _i, _i, _p, _i, _i, _i, _p, _i, _p, _i, _d, _p, _p, _p, _p, _p, _p, _p, _p],
    "unmore_boundary_refine_hw": [_p, _i, _i, _i, _i, _p, _i, _p, _i, _p, _i, _i, _i, _i, _f, _f, _f, _f, _p, _p, _p, _p, _p],
    "unmore_score_and_rasterise_hw": [_p, _i, _i, _i, _i, _p, _i, _i, _i, _i, _p, _i, _p, _i, _p, _p, _p, _p, _p],
    "unmore_box_sums_hw": [_p, _i, _i, _i, _i, _i, _p, _p, _i, _p, _i, _p, _p, _p],
    "unmore_sat_build_fields_hw": [_p, _i, _i, _i, _i, _p, _p, _i, _p, _p],
    "unmore_existence_scores_aa_hw": [_p, _i, _i, _i, _i, _p, _i, _p, _i, _p, _i, _p, _p, _p],
    "unmore_boundary_refine_aa_hw": [_p, _i, _i, _i, _i, _p, _i, _p, _i, _p, _i, _i, _i, _i, _f, _f, _f, _f, _p, _p, _p, _p, _p],
    "unmore_center_reasoning_aa_hw": [_p, _i, _i, _i, _i, _p, _i, _i, _i, _p, _i, _p, _i, _d, _p, _p, _p, _p, _p, _p, _p, _p],
    "unmore_crop_resize_aa_hw": [_p, _i, _i, _i, _i, _p, _p, _i, _p, _i, _p, _i, _p, _p, C.c_size_t, _p],
    "unmore_center_reasoning_from_tiles_hw": [_p, _i, _i, _i, _p, _p, _i, _p, _i, _d, _p, _p, _p, _p, _p, _p, _p, _p],
    "unmore_score_and_rasterise_from_tiles_hw": [_p, _p, _i, _i, _i, _i, _p, _p, _i, _p, _i, _p, _p, _p, _p, _p],
}

_lib = None


class UnmoreError(RuntimeError):
    pass


def load():
    """Load the library once and bind every symbol the header declares."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise UnmoreError(f"{LIB_PATH} not built: run `bash unmore_b200/csrc/build.sh` (no CPU fallback exists)")
    lib = C.CDLL(LIB_PATH)
    lib.unmore_last_error.restype = C.c_char_p
    lib.unmore_last_error.argtypes = []
    lib.unmore_version.restype = _i
    lib.unmore_version.argtypes = []
    lib.unmore_workspace_bytes.restype = C.c_size_t
    lib.unmore_workspace_bytes.argtypes = [_i]
    lib.unmore_cc_cap.restype = _i
    lib.unmore_cc_cap.argtypes = []
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: intended
        fn.restype = _i
        fn.argtypes = args
    _lib = lib
    return lib


def call(name: str, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise UnmoreError(f"{name} failed (code {rc}): {lib.unmore_last_error().decode()}")
