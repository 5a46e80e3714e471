"""Tensor-level wrappers over the C ABI: pointer extraction, output allocation, stream.

PyTorch is only the allocator / stream provider here; all arithmetic runs in
``libunmore_b200.so``.  Inputs must be CUDA tensors; there is no CPU path."""
from __future__ import annotations

import threading
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import _lib
from .synth import CH_CCOL, CH_CROW, CH_EXIST, CH_SDF

CROP = 128
UnmoreError = _lib.UnmoreError


@dataclass(frozen=True)
class Channels:
    sdf: int = CH_SDF
    center_row: int = CH_CROW
    center_col: int = CH_CCOL
    exist: int = CH_EXIST


DEFAULT_CHANNELS = Channels()


_tls = threading.local()   # .device = device of the call being assembled on THIS thread: set by _on(), consumed by _stream() / _call()


def _on(t: torch.Tensor):
    """Pins the device of the call being assembled to the device of its first tensor (ADVICE r1: the C ABI
    launches on the CURRENT device; without this, tensors on cuda:1 under a current device of cuda:0 would be
    dereferenced by a kernel running on GPU 0).  Per thread, like the library's error string."""
    _tls.device = t.device
    return t


def _cur_device():
    return getattr(_tls, "device", None)


def _stream() -> int:
    return torch.cuda.current_stream(_cur_device()).cuda_stream


class StageTimer:
    """CUDA-event timing of every C-ABI call, on the stream the kernels are launched on.
    bench.py installs one (``ops.set_timer``) for the timed region; ``summary()`` synchronises."""

    def __init__(self):
        self.events = []   # (name, start, end, kernels)
        self.launches = 0

    def record(self, name, kernels, fn, *args):
        st = torch.cuda.current_stream(_cur_device())
        a = torch.cuda.Event(enable_timing=True)
        b = torch.cuda.Event(enable_timing=True)
        a.record(st)
        fn(name, *args)
        b.record(st)
        self.events.append((name, a, b))
        self.launches += kernels

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, a, b in self.events:
            d = out.setdefault(name, {"ms": 0.0, "calls": 0})
            d["ms"] += a.elapsed_time(b)
            d["calls"] += 1
        return out


_timer: Optional[StageTimer] = None
LAUNCHES = 0  # kernels launched through the C ABI since import (gpu_launches in bench.py)

# kernels per C-ABI call (memsets not counted); +1 when a counts prefix is built
_KERNELS = {"unmore_crop_resize": 1, "unmore_crop_resize_aa": 2, "unmore_mask_resize_aa": 2, "unmore_existence_scores": 1, "unmore_center_reasoning": 1, "unmore_boundary_refine": 1,
            "unmore_existence_scores_aa": 1, "unmore_boundary_refine_aa": 1, "unmore_center_reasoning_aa": 1,
            "unmore_update_bbox_from_tiles": 1, "unmore_compact_boxes": 1, "unmore_box_nms": 1,
            "unmore_batch_erode": 1, "unmore_anti_center_map": 1, "unmore_connected_components": 1, "unmore_box_nms_matrix": 3,
            "unmore_score_and_rasterise": 1, "unmore_mask_resize": 1, "unmore_final_scores": 1, "unmore_sat_build": 1, "unmore_sat_build_fields": 1, "unmore_box_sums": 1,
            "unmore_mask_pack": 1, "unmore_mask_stats": 1, "unmore_mask_nms": 3, "unmore_mask_rle_counts": 1,
            "unmore_pack_detections": 1, "unmore_tile_means": 1, "unmore_center_reasoning_from_tiles": 1,
            "unmore_boundary_round_from_tiles": 2, "unmore_score_and_rasterise_from_tiles": 1,
            "unmore_existence_scores_hw": 1, "unmore_center_reasoning_hw": 1, "unmore_boundary_refine_hw": 1,
            "unmore_score_and_rasterise_hw": 1, "unmore_box_sums_hw": 1, "unmore_sat_build_fields_hw": 1,
            "unmore_existence_scores_aa_hw": 1, "unmore_boundary_refine_aa_hw": 1, "unmore_center_reasoning_aa_hw": 1,
            "unmore_crop_resize_aa_hw": 2,
            "unmore_center_reasoning_from_tiles_hw": 1, "unmore_score_and_rasterise_from_tiles_hw": 1}


def set_timer(t: Optional[StageTimer]):
    global _timer
    _timer = t


def _call(name, *args, counts=None):
    global LAUNCHES
    k = _KERNELS[name] + (1 if counts is not None else 0)
    LAUNCHES += k
    dev = _cur_device()
    try:
        if dev is not None and dev.index is not None and dev.index != torch.cuda.current_device():
            with torch.cuda.device(dev):
                _lib.call(name, *args) if _timer is None else _timer.record(name, k, _lib.call, *args)
        elif _timer is not None:
            _timer.record(name, k, _lib.call, *args)
        else:
            _lib.call(name, *args)
    finally:
        _tls.device = None


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _check_fields(fields: torch.Tensor) -> Tuple[int, int, int, int]:
    if not fields.is_cuda:
        raise _lib.UnmoreError("fields must live on a CUDA device (no CPU path)")
    if fields.dtype != torch.float32 or fields.dim() != 4 or not fields.is_contiguous():
        raise _lib.UnmoreError("fields must be contiguous fp32 [n_img, C, H, W]")
    _on(fields)
    return tuple(fields.shape)  # type: ignore[return-value]


def _check_boxes(boxes: torch.Tensor, n_img: int) -> Tuple[int, int]:
    if boxes.dim() != 3 or boxes.shape[0] != n_img or boxes.shape[2] != 4 or not boxes.is_contiguous():
        raise _lib.UnmoreError("boxes must be contiguous [n_img, cap, 4]")
    if boxes.dtype not in (torch.float32, torch.float64):
        raise _lib.UnmoreError("boxes must be fp32 or fp64")
    return boxes.shape[1], int(boxes.dtype == torch.float64)


def _check_counts(counts: Optional[torch.Tensor], n_img: int):
    if counts is not None and (counts.dtype != torch.int32 or counts.numel() != n_img or not counts.is_cuda):
        raise _lib.UnmoreError("counts must be a CUDA int32 tensor of n_img entries")


def _check_extents(image_hw, n_img: int, device, what: str = "") -> torch.Tensor:
    """The (h, w) table of a padded stack: a CUDA int32 [n_img, 2] tensor on the fields' device, 8-byte aligned.  Its
    values are not read on the host (no sync); the kernels clamp them to [1, pitch]."""
    if not torch.is_tensor(image_hw) or not image_hw.is_cuda or image_hw.dtype != torch.int32 or \
            tuple(image_hw.shape) != (n_img, 2):
        raise _lib.UnmoreError(f"{what}: image_hw must be a CUDA int32 [n_img, 2] tensor of (h, w) per image")
    if image_hw.device != torch.device(device):
        raise _lib.UnmoreError(f"{what}: image_hw must live on the device of the fields")
    image_hw = image_hw.contiguous()
    return image_hw if image_hw.data_ptr() % 8 == 0 else image_hw.clone()


def pack_fields(images):
    """Pads a list of [C, h_i, w_i] fp32 field stacks with zeros into one stack of images of different sizes:
    -> (fields [B, C, Hp, Wp], image_hw [B, 2] int32 (h_i, w_i)), both on the device of the first image; (Hp, Wp), the
    pitch, is the largest h and w of the batch.  Image i is ``fields[i, :, :h_i, :w_i]``; no result of the ops that
    take ``image_hw`` depends on the padding."""
    images = list(images)
    if not images:
        raise _lib.UnmoreError("pack_fields: empty list")
    for im in images:
        if not torch.is_tensor(im) or im.dim() != 3:
            raise _lib.UnmoreError("pack_fields: every image must be a 3-D [C, h, w] tensor")
        if im.dtype != torch.float32:
            raise _lib.UnmoreError("pack_fields: every image must be fp32")
        if im.shape[1] < 1 or im.shape[2] < 1:
            raise _lib.UnmoreError("pack_fields: empty image")
    C = images[0].shape[0]
    if any(im.shape[0] != C for im in images):
        raise _lib.UnmoreError("pack_fields: all images must have the same number of channels")
    dev = images[0].device
    Hp, Wp = max(im.shape[1] for im in images), max(im.shape[2] for im in images)
    fields = torch.zeros((len(images), C, Hp, Wp), dtype=torch.float32, device=dev)
    for i, im in enumerate(images):
        fields[i, :, : im.shape[1], : im.shape[2]] = im.to(dev)
    hw = torch.tensor([[im.shape[1], im.shape[2]] for im in images], dtype=torch.int32).to(dev)
    return fields, hw


def stack_proposals(proposals, device=None):
    """Ragged proposal lists [n_i, 4] (tensors or arrays) -> (boxes [B, max n_i, 4], counts [B] int32), on ``device``
    (default: that of the first tensor).  fp64 unless every list is fp32; rows past a count are zero."""
    lists = [p if torch.is_tensor(p) else torch.as_tensor(p) for p in proposals]
    if not lists:
        raise _lib.UnmoreError("stack_proposals: empty list")
    if any(p.dim() != 2 or p.shape[1] != 4 for p in lists if p.numel()) or any(p.numel() % 4 for p in lists):
        raise _lib.UnmoreError("stack_proposals: every list must be [n, 4]")
    lists = [p.reshape(-1, 4) for p in lists]
    dev = torch.device(device) if device is not None else lists[0].device
    dtype = torch.float32 if all(p.dtype == torch.float32 for p in lists) else torch.float64
    n = max(p.shape[0] for p in lists)
    boxes = torch.zeros((len(lists), n, 4), dtype=dtype, device=dev)
    for i, p in enumerate(lists):
        if p.shape[0]:
            boxes[i, : p.shape[0]] = p.to(dev, dtype)
    counts = torch.tensor([p.shape[0] for p in lists], dtype=torch.int32).to(dev)
    return boxes, counts


def workspace(n_img: int, device) -> torch.Tensor:
    n = _lib.load().unmore_workspace_bytes(n_img)
    return torch.empty((n + 3) // 4, dtype=torch.int32, device=device)


def existence_scores(fields, boxes, counts=None, ch: Channels = DEFAULT_CHANNELS, ws=None, out=None,
                     antialias: bool = False, image_hw=None):
    """Existence score [n_img, cap] fp32 of every proposal: the mean of its resized crop of the existence channel
    (``antialias=True``: the second resize mode, equal to ``tile_means`` of ``crop_resize(..., antialias=True)``).
    ``image_hw`` [n_img, 2] int32: ``fields`` is a padded stack of images of different sizes (``pack_fields``)."""
    n_img, C, H, W = _check_fields(fields)
    cap, f64 = _check_boxes(boxes, n_img)
    _check_counts(counts, n_img)
    ws = workspace(n_img, fields.device) if ws is None else ws
    out = torch.zeros((n_img, cap), dtype=torch.float32, device=fields.device) if out is None else out
    if image_hw is not None:
        hw = _check_extents(image_hw, n_img, fields.device, "existence_scores")
        _on(fields)
        _call("unmore_existence_scores_aa_hw" if antialias else "unmore_existence_scores_hw", fields.data_ptr(), n_img, C, H, W, hw.data_ptr(), ch.exist, boxes.data_ptr(), f64,
              _ptr(counts), cap, out.data_ptr(), ws.data_ptr(), _stream(), counts=counts)
        return out
    _call("unmore_existence_scores_aa" if antialias else "unmore_existence_scores", fields.data_ptr(), n_img, C, H, W, ch.exist, boxes.data_ptr(), f64,
              _ptr(counts), cap, out.data_ptr(), ws.data_ptr(), _stream(), counts=counts)
    return out


def crop_resize(fields, boxes, channels, counts=None, antialias: bool = False, image_hw=None):
    """Resized crops [n_img, cap, len(channels), 128, 128] fp32 (a2 / a4 as a stand-alone op).
    ``antialias=True`` is the second resize mode (torchvision >= 0.17's default for transforms.Resize).
    ``image_hw`` [n_img, 2] int32, with ``antialias=True`` only: ``fields`` is a padded stack of images of different
    sizes (``pack_fields``) and every window snaps to its own image."""
    import ctypes
    n_img, C, H, W = _check_fields(fields)
    cap, f64 = _check_boxes(boxes, n_img)
    _check_counts(counts, n_img)
    hw = None
    if image_hw is not None:
        if not antialias:
            raise _lib.UnmoreError("crop_resize: image_hw (images of different sizes) needs antialias=True")
        hw = _check_extents(image_hw, n_img, fields.device, "crop_resize")
    ch = (ctypes.c_int * len(channels))(*[int(c) for c in channels])
    out = torch.zeros((n_img, cap, len(channels), CROP, CROP), dtype=torch.float32, device=fields.device)
    if cap and antialias:
        # the intermediate of the separable pass lives in scratch: bound it by walking the proposals in slices
        per_box = len(channels) * H * CROP * 4
        step = max(1, min(cap, (256 << 20) // max(1, per_box * n_img)))
        for c0 in range(0, cap, step):
            c1 = min(cap, c0 + step)
            bsl = boxes[:, c0:c1].contiguous()
            osl = torch.zeros((n_img, c1 - c0, len(channels), CROP, CROP), dtype=torch.float32, device=fields.device)
            cnt = None if counts is None else (counts - c0).clamp(0, c1 - c0).to(torch.int32)
            scratch = torch.empty((n_img * (c1 - c0) * per_box // 4,), dtype=torch.float32, device=fields.device)
            _on(fields)
            name, size = ("unmore_crop_resize_aa", (H, W)) if hw is None else ("unmore_crop_resize_aa_hw", (H, W, hw.data_ptr()))
            _call(name, fields.data_ptr(), n_img, C, *size, ctypes.cast(ch, ctypes.c_void_p), len(channels),
                  bsl.data_ptr(), f64, _ptr(cnt), c1 - c0, osl.data_ptr(), scratch.data_ptr(), scratch.numel() * 4, _stream())
            out[:, c0:c1] = osl
        return out
    if cap:
        _call("unmore_crop_resize", fields.data_ptr(), n_img, C, H, W, ctypes.cast(ch, ctypes.c_void_p), len(channels),
              boxes.data_ptr(), f64, _ptr(counts), cap, out.data_ptr(), _stream())
    return out


CENTER_AA_SLICE_BYTES = 1 << 30   # unused: center_reasoning(antialias=True) is one fused call, nothing is sliced


def center_reasoning(fields, boxes, counts=None, thr: float = 0.009, ch: Channels = DEFAULT_CHANNELS, ws=None,
                     want_splits: bool = True, analyze_cc: bool = False, antialias: bool = False, image_hw=None):
    """-> (max_values [n_img,cap] fp64, argmax [n_img,cap] int32 (-1 = passes), splits [n_img,cap,4,4] fp64 or None,
    cc) where cc is None or (cc_counts [n_img,cap] u8, cc_boxes [n_img,cap,CC_CAP,4] fp64, overflow [1] int32).
    ``antialias=True`` is the second resize mode: the fused kernel resamples every antialiased crop from the fields
    itself, bit-identical to ``center_reasoning_from_tiles`` on the tiles of ``crop_resize(..., antialias=True)``.
    ``image_hw`` [n_img, 2] int32: ``fields`` is a padded stack of images of different sizes (``pack_fields``); every
    window snaps to, and the --analyze_cc boxes are clipped against, each image's own size."""
    n_img, C, H, W = _check_fields(fields)
    cap, f64 = _check_boxes(boxes, n_img)
    _check_counts(counts, n_img)
    dev = fields.device
    ws = workspace(n_img, dev) if ws is None else ws
    hw = None if image_hw is None else _check_extents(image_hw, n_img, dev, "center_reasoning")
    maxv = torch.zeros((n_img, cap), dtype=torch.float64, device=dev)
    argmax = torch.full((n_img, cap), -1, dtype=torch.int32, device=dev)
    splits = torch.zeros((n_img, cap, 4, 4), dtype=torch.float64, device=dev) if want_splits else None
    cc = None
    if analyze_cc:
        cc_cap = _lib.load().unmore_cc_cap()
        cc = (torch.zeros((n_img, cap), dtype=torch.uint8, device=dev),
              torch.zeros((n_img, cap, cc_cap, 4), dtype=torch.float64, device=dev),
              torch.zeros((1,), dtype=torch.int32, device=dev))
    _on(fields)
    name = ("unmore_center_reasoning_aa" if antialias else "unmore_center_reasoning") + ("" if hw is None else "_hw")
    size = (H, W) if hw is None else (H, W, hw.data_ptr())
    _call(name, fields.data_ptr(), n_img, C, *size, ch.sdf, ch.center_row, ch.center_col,
          boxes.data_ptr(), f64, _ptr(counts), cap, float(thr), maxv.data_ptr(), argmax.data_ptr(),
          _ptr(splits), _ptr(cc[0]) if cc else None, _ptr(cc[1]) if cc else None, _ptr(cc[2]) if cc else None,
          ws.data_ptr(), _stream(), counts=counts)
    return maxv, argmax, splits, cc


def boundary_refine(fields, boxes, counts=None, n_round: int = 50, apply_small_filter: bool = True,
                    early_exit: bool = True, proposal_area_thres: float = 50.0, max_sdf_thres: float = 0.5,
                    max_shrink_threshold: float = 16.0, delta_ratio: float = 0.5, ch: Channels = DEFAULT_CHANNELS,
                    ws=None, want_rounds: bool = True, antialias: bool = False, image_hw=None):
    """Up to ``n_round`` rounds of boundary reasoning per proposal -> (boxes [n_img,cap,4] fp32, labels [n_img,cap]
    fp32 (-2 = removed by the area filter), rounds [n_img,cap] int32 or None); ``antialias=True``: the second
    resize mode.  ``image_hw`` [n_img, 2] int32: ``fields`` is a padded stack of images of different sizes
    (``pack_fields``); boxes are clipped against, and glued to, each image's own edges."""
    n_img, C, H, W = _check_fields(fields)
    cap, f64 = _check_boxes(boxes, n_img)
    _check_counts(counts, n_img)
    dev = fields.device
    ws = workspace(n_img, dev) if ws is None else ws
    hw = None if image_hw is None else _check_extents(image_hw, n_img, dev, "boundary_refine")
    out = torch.zeros((n_img, cap, 4), dtype=torch.float32, device=dev)
    labels = torch.full((n_img, cap), -2.0, dtype=torch.float32, device=dev)
    rounds = torch.zeros((n_img, cap), dtype=torch.int32, device=dev) if want_rounds else None
    _on(fields)
    name = ("unmore_boundary_refine_aa" if antialias else "unmore_boundary_refine") + ("" if hw is None else "_hw")
    _call(name, fields.data_ptr(), n_img, C, H, W, *(() if hw is None else (hw.data_ptr(),)), ch.sdf,
              boxes.data_ptr(), f64,
              _ptr(counts), cap, int(n_round), int(apply_small_filter), int(early_exit), float(proposal_area_thres),
              float(max_sdf_thres), float(max_shrink_threshold), float(delta_ratio), out.data_ptr(),
              labels.data_ptr(), _ptr(rounds), ws.data_ptr(), _stream(), counts=counts)
    return out, labels, rounds


def update_bbox_from_tiles(tiles: torch.Tensor):
    if not tiles.is_cuda or tiles.dtype != torch.float32 or tiles.dim() != 3 or tiles.shape[1:] != (CROP, CROP):
        raise _lib.UnmoreError("tiles must be CUDA fp32 [M, 128, 128]")
    tiles = _on(tiles.contiguous())
    m = tiles.shape[0]
    deltas = torch.zeros((m, 4), dtype=torch.float32, device=tiles.device)
    mx = torch.zeros((m,), dtype=torch.float32, device=tiles.device)
    _call("unmore_update_bbox_from_tiles", tiles.data_ptr(), m, deltas.data_ptr(), mx.data_ptr(), _stream())
    return deltas, mx


MODE_FLAGS, MODE_SCORE_GE, MODE_LABEL_EQ, MODE_ARGMAX_GE0, MODE_ARGMAX_LT0, MODE_U8_NONZERO = range(6)


def compact_boxes(inp, counts_in, mode, pred, thr=0.0, group=1, out=None, counts_out=None, cap_out=None,
                  out_dtype=None, append=False, want_index=False, group_counts=None, overflow=None):
    """Stable per-image selection; returns (out [n_img, cap_out, 4], counts_out [n_img], index or None)."""
    dev = _on(inp).device
    n_img, cap_in = inp.shape[0], inp.shape[1]
    if group != 1 and inp.shape[2] != group:
        raise _lib.UnmoreError("compact_boxes: input must be [n_img, cap, group, 4]")
    out_dtype = out_dtype or inp.dtype
    if cap_out is None:
        cap_out = out.shape[1] if out is not None else cap_in * group
    if out is None:
        out = torch.zeros((n_img, cap_out, 4), dtype=out_dtype, device=dev)
    if counts_out is None:
        counts_out = torch.zeros((n_img,), dtype=torch.int32, device=dev)
    index = torch.full((n_img, cap_out), -1, dtype=torch.int32, device=dev) if want_index else None
    _call("unmore_compact_boxes", inp.data_ptr(), int(inp.dtype == torch.float64), _ptr(counts_in), cap_in,
              group, mode, pred.data_ptr(), float(thr), out.data_ptr(), int(out.dtype == torch.float64), cap_out,
              counts_out.data_ptr(), int(append), _ptr(index), _ptr(group_counts), _ptr(overflow), n_img, _stream())
    return out, counts_out, index


def box_nms(boxes, scores=None, counts=None, iou_threshold: float = 0.5, want_boxes: bool = True):
    """boxes [n_img, cap, 4] fp32 -> (keep [n_img, cap] int32, keep_counts [n_img], kept boxes or None)."""
    if not boxes.is_cuda or boxes.dtype != torch.float32 or boxes.dim() != 3 or not boxes.is_contiguous():
        raise _lib.UnmoreError("boxes must be contiguous CUDA fp32 [n_img, cap, 4]")
    n_img, cap = boxes.shape[0], boxes.shape[1]
    dev = _on(boxes).device
    keep = torch.full((n_img, cap), -1, dtype=torch.int32, device=dev)
    kc = torch.zeros((n_img,), dtype=torch.int32, device=dev)
    order = torch.empty((n_img, max(cap, 1)), dtype=torch.int32, device=dev)
    kb = torch.zeros((n_img, cap, 4), dtype=torch.float32, device=dev) if want_boxes else None
    if scores is not None:
        scores = scores.contiguous().to(torch.float32)
    _call("unmore_box_nms", boxes.data_ptr(), _ptr(scores), _ptr(counts), cap, n_img, float(iou_threshold),
              keep.data_ptr(), kc.data_ptr(), _ptr(kb), order.data_ptr(), _stream())
    return keep, kc, kb


def box_nms_matrix(boxes, scores=None, iou_threshold: float = 0.5):
    """One list of K boxes [K,4] fp32 -> kept indices (int64, descending-score order)."""
    boxes = _on(boxes.contiguous().to(torch.float32))
    K = boxes.shape[0]
    dev = boxes.device
    nblk = (K + 63) // 64
    order = torch.empty((max(K, 1),), dtype=torch.int32, device=dev)
    matrix = torch.empty((max(K * nblk, 1),), dtype=torch.int64, device=dev)
    keep = torch.full((max(K, 1),), -1, dtype=torch.int32, device=dev)
    kc = torch.zeros((1,), dtype=torch.int32, device=dev)
    if scores is not None:
        scores = scores.contiguous().to(torch.float32)
    _call("unmore_box_nms_matrix", boxes.data_ptr(), _ptr(scores), K, float(iou_threshold), order.data_ptr(),
              matrix.data_ptr(), keep.data_ptr(), kc.data_ptr(), _stream())
    return keep[: int(kc.item())].to(torch.int64)


def batch_erode(masks_u8: torch.Tensor, kernel_size: int = 9, num_round: int = 3) -> torch.Tensor:
    m = _on(masks_u8.contiguous())
    B, H, W = m.shape
    out = torch.empty_like(m)
    _call("unmore_batch_erode", m.data_ptr(), B, H, W, int(kernel_size), int(num_round), out.data_ptr(), _stream())
    return out


def connected_components(masks_u8: torch.Tensor):
    """[B,128,128] u8 -> (counts [B] int32, boxes [B, CC_CAP, 4] int32 slice bounds) in scipy label order."""
    m = _on(masks_u8.contiguous())
    B, H, W = m.shape
    cap = _lib.load().unmore_cc_cap()
    counts = torch.zeros((B,), dtype=torch.int32, device=m.device)
    boxes = torch.zeros((B, cap, 4), dtype=torch.int32, device=m.device)
    _call("unmore_connected_components", m.data_ptr(), B, H, W, counts.data_ptr(), boxes.data_ptr(), _stream())
    return counts, boxes


def anti_center_map(vote_maps: torch.Tensor, kernel_size: int = 5) -> torch.Tensor:
    v = _on(vote_maps.contiguous().to(torch.float32))
    B, _, H, W = v.shape
    out = torch.empty((B, H, W), dtype=torch.float64, device=v.device)
    _call("unmore_anti_center_map", v.data_ptr(), B, H, W, int(kernel_size), out.data_ptr(), _stream())
    return out


def score_and_rasterise(fields, boxes, counts=None, ch: Channels = DEFAULT_CHANNELS, want_masks: bool = True,
                        image_hw=None):
    """-> scores [n_img,cap,4] (existence, center, boundary, 0), tight xyxy [n_img,cap,4], areas [n_img,cap],
    packed masks [n_img,cap,H,ceil(W/32)] int32 (or None).  ``image_hw`` [n_img, 2] int32: ``fields`` is a padded
    stack of images of different sizes (``pack_fields``); the masks stay on the pitched canvas, image i's mask is
    ``masks[i, :, :h_i, :ceil(w_i/32)]`` and every bit outside the image is 0."""
    n_img, C, H, W = _check_fields(fields)
    cap, f64 = _check_boxes(boxes, n_img)
    _check_counts(counts, n_img)
    dev = fields.device
    hw = None if image_hw is None else _check_extents(image_hw, n_img, dev, "score_and_rasterise")
    scores = torch.zeros((n_img, cap, 4), dtype=torch.float32, device=dev)
    tight = torch.zeros((n_img, cap, 4), dtype=torch.float32, device=dev)
    areas = torch.zeros((n_img, cap), dtype=torch.int32, device=dev)
    masks = torch.zeros((n_img, cap, H, (W + 31) // 32), dtype=torch.int32, device=dev) if want_masks else None
    if cap > 0:
        _on(fields)
        name, size = ("unmore_score_and_rasterise", (H, W)) if hw is None else ("unmore_score_and_rasterise_hw", (H, W, hw.data_ptr()))
        _call(name, fields.data_ptr(), n_img, C, *size, ch.sdf, ch.center_row, ch.center_col,
                  ch.exist, boxes.data_ptr(), f64, _ptr(counts), cap, scores.data_ptr(), tight.data_ptr(),
                  areas.data_ptr(), _ptr(masks), _stream())
    return scores, tight, areas, masks


def mask_resize(masks_u8: torch.Tensor, out_h: int, out_w: int, antialias: bool = False) -> torch.Tensor:
    """[B,128,128] u8 -> [B,out_h,out_w] u8: bilinear + round-half-even like the reference's Resize on int masks
    (``antialias=True``: the second resize mode)."""
    m = _on(masks_u8.contiguous())
    B, H, W = m.shape
    out = torch.zeros((B, out_h, out_w), dtype=torch.uint8, device=m.device)
    if B and out_h and out_w and antialias:
        scratch = torch.empty((B * CROP * out_w,), dtype=torch.float32, device=m.device)
        _call("unmore_mask_resize_aa", m.data_ptr(), B, H, W, int(out_h), int(out_w), out.data_ptr(), scratch.data_ptr(),
              scratch.numel() * 4, _stream())
        return out
    if B and out_h and out_w:
        _call("unmore_mask_resize", m.data_ptr(), B, H, W, int(out_h), int(out_w), out.data_ptr(), _stream())
    return out


def final_scores(scores, tight, areas, keep, keep_counts, existence_score_thres=0.5, center_score_thres=0.8,
                 boundary_score_thres=0.75):
    """-> out [n_img,cap,5] fp64 (score, existence, center, boundary, area_score), bbox xywh [n_img,cap,4],
    selected [n_img,cap] uint8 — all in NMS keep order."""
    n_img, cap = areas.shape
    dev = _on(areas).device
    out = torch.zeros((n_img, cap, 5), dtype=torch.float64, device=dev)
    bbox = torch.zeros((n_img, cap, 4), dtype=torch.float32, device=dev)
    sel = torch.zeros((n_img, cap), dtype=torch.uint8, device=dev)
    if cap > 0:
        _call("unmore_final_scores", scores.data_ptr(), tight.data_ptr(), areas.data_ptr(), keep.data_ptr(),
                  keep_counts.data_ptr(), cap, n_img, float(existence_score_thres), float(center_score_thres),
                  float(boundary_score_thres), out.data_ptr(), bbox.data_ptr(), sel.data_ptr(), _stream())
    return out, bbox, sel


def sat_build(planes: torch.Tensor) -> torch.Tensor:
    """[..., H, W] fp32 CUDA -> [..., H+1, W+1] fp64 exclusive 2-D prefix sums."""
    if not planes.is_cuda or planes.dtype != torch.float32:
        raise _lib.UnmoreError("sat_build needs a CUDA fp32 tensor")
    p = _on(planes.contiguous())
    H, W = p.shape[-2], p.shape[-1]
    n = p.numel() // (H * W) if H * W else 0
    out = torch.empty(p.shape[:-2] + (H + 1, W + 1), dtype=torch.float64, device=p.device)
    _call("unmore_sat_build", p.data_ptr(), n, H, W, out.data_ptr(), _stream())
    return out


def sat_build_fields(fields: torch.Tensor, channels, out: Optional[torch.Tensor] = None, image_hw=None) -> torch.Tensor:
    """Tables of selected channels straight from the field stack: [n_img, C, H, W] fp32 ->
    [n_img, len(channels), H+1, W+1] fp64 (no gather copy).  ``image_hw`` [n_img, 2] int32: ``fields`` is a padded
    stack (``pack_fields``) and the padding enters the sums as zeros, so entries [:h_i+1, :w_i+1] of image i's tables
    are those of the image alone."""
    import ctypes
    n_img, C, H, W = _check_fields(fields)
    ch = (ctypes.c_int * len(channels))(*[int(c) for c in channels])
    if out is None:
        out = torch.empty((n_img, len(channels), H + 1, W + 1), dtype=torch.float64, device=fields.device)
    if image_hw is not None:
        hw = _check_extents(image_hw, n_img, fields.device, "sat_build_fields")
        _on(fields)
        _call("unmore_sat_build_fields_hw", fields.data_ptr(), n_img, C, H, W, hw.data_ptr(), ctypes.cast(ch, ctypes.c_void_p),
              len(channels), out.data_ptr(), _stream())
        return out
    _call("unmore_sat_build_fields", fields.data_ptr(), n_img, C, H, W, ctypes.cast(ch, ctypes.c_void_p), len(channels),
          out.data_ptr(), _stream())
    return out


def box_sums(sat: torch.Tensor, plane: int, boxes: torch.Tensor, counts=None, image_hw=None):
    """sat [n_img, P, H+1, W+1] fp64, boxes [n_img, cap, 4] -> (sums, means) [n_img, cap] fp64.  ``image_hw``
    [n_img, 2] int32: the tables are those of a padded stack (``sat_build_fields(..., image_hw=)``); windows snap to
    each image's own size."""
    n_img, P, H1, W1 = _on(sat).shape
    cap, f64 = _check_boxes(boxes, n_img)
    sums = torch.zeros((n_img, cap), dtype=torch.float64, device=sat.device)
    means = torch.zeros((n_img, cap), dtype=torch.float64, device=sat.device)
    if image_hw is not None:
        hw = _check_extents(image_hw, n_img, sat.device, "box_sums")
        if cap > 0:
            _on(sat)
            _call("unmore_box_sums_hw", sat.data_ptr(), n_img, P, int(plane), H1 - 1, W1 - 1, hw.data_ptr(), boxes.data_ptr(), f64,
                  _ptr(counts), cap, sums.data_ptr(), means.data_ptr(), _stream())
        return sums, means
    if cap > 0:
        _call("unmore_box_sums", sat.data_ptr(), n_img, P, int(plane), H1 - 1, W1 - 1, boxes.data_ptr(), f64,
                  _ptr(counts), cap, sums.data_ptr(), means.data_ptr(), _stream())
    return sums, means


def mask_pack(dense_u8: torch.Tensor) -> torch.Tensor:
    """[K, H, W] uint8/bool CUDA -> [K, H, ceil(W/32)] int32 bit-packed (LSB = lowest x)."""
    d = dense_u8
    if d.dtype == torch.bool:
        d = d.view(torch.uint8)
    if not d.is_cuda or d.dtype != torch.uint8:
        raise _lib.UnmoreError("mask_pack needs a CUDA uint8/bool tensor")
    d = _on(d.contiguous())
    K, H, W = d.shape
    out = torch.empty((K, H, (W + 31) // 32), dtype=torch.int32, device=d.device)
    _call("unmore_mask_pack", d.data_ptr(), K, H, W, out.data_ptr(), _stream())
    return out


def mask_stats(packed: torch.Tensor, W: int):
    K, H, _ = _on(packed).shape
    areas = torch.zeros((K,), dtype=torch.int32, device=packed.device)
    tight = torch.zeros((K, 4), dtype=torch.int32, device=packed.device)
    _call("unmore_mask_stats", packed.data_ptr(), K, H, W, areas.data_ptr(), tight.data_ptr(), _stream())
    return areas, tight


def mask_nms(packed: torch.Tensor, W: int, scores: torch.Tensor, iou_threshold: float = 0.5, stats=None):
    """Mask-IoU NMS on packed masks [K, H, ceil(W/32)]: kept indices, descending-score order (int64)."""
    packed = packed.contiguous()
    K, H, _ = packed.shape
    dev = packed.device
    areas, tight = stats if stats is not None else mask_stats(packed, W)
    _on(packed)
    nblk = (K + 63) // 64
    order = torch.empty((max(K, 1),), dtype=torch.int32, device=dev)
    matrix = torch.empty((max(K * nblk, 1),), dtype=torch.int64, device=dev)
    keep = torch.full((max(K, 1),), -1, dtype=torch.int32, device=dev)
    kc = torch.zeros((1,), dtype=torch.int32, device=dev)
    scores = scores.contiguous().to(torch.float32)
    _call("unmore_mask_nms", packed.data_ptr(), K, H, W, scores.data_ptr(), areas.data_ptr(), tight.data_ptr(),
              float(iou_threshold), order.data_ptr(), matrix.data_ptr(), keep.data_ptr(), kc.data_ptr(), _stream())
    return keep[: int(kc.item())].to(torch.int64)


def mask_rle_counts(packed: torch.Tensor, W: int, max_runs: int = 4096):
    """Packed masks [K, H, ceil(W/32)] -> (counts [K, max_runs] int32 (as uint32), n_runs [K] int32):
    COCO column-major run lengths; rows with n_runs > max_runs are not filled."""
    packed = _on(packed.contiguous())
    K, H, _ = packed.shape
    counts = torch.zeros((K, max_runs), dtype=torch.int32, device=packed.device)
    n_runs = torch.zeros((K,), dtype=torch.int32, device=packed.device)
    if K:
        _call("unmore_mask_rle_counts", packed.data_ptr(), K, H, W, int(max_runs), counts.data_ptr(), n_runs.data_ptr(),
              _stream())
    return counts, n_runs


def detection_rows(max_rows: int, device) -> torch.Tensor:
    """Zeroed row buffer [max_rows + 1, 6] fp64 for ``pack_detections`` (row 0 is the header / append cursor)."""
    return torch.zeros((max_rows + 1, 6), dtype=torch.float64, device=device)


def pack_detections(image_ids: torch.Tensor, bbox: torch.Tensor, out5: torch.Tensor, keep_counts: torch.Tensor,
                    rows: torch.Tensor) -> torch.Tensor:
    """Appends (image_id, x, y, w, h, score) rows of a scored batch to ``rows`` (see ``detection_rows``) on the
    device, image-major in NMS keep order; no host round trip.  image_ids [B] int64, bbox [B,cap,4] fp32,
    out5 [B,cap,5] fp64, keep_counts [B] int32."""
    B, cap = bbox.shape[0], bbox.shape[1]
    if image_ids.dtype != torch.int64 or image_ids.numel() != B or not bbox.is_contiguous() or not out5.is_contiguous():
        raise _lib.UnmoreError("pack_detections: image_ids must be int64 [B]; bbox / out5 contiguous")
    if rows.dtype != torch.float64 or rows.dim() != 2 or rows.shape[1] != 6 or not rows.is_contiguous():
        raise _lib.UnmoreError("pack_detections: rows must be contiguous fp64 [max_rows + 1, 6]")
    _on(bbox)
    if B and cap:
        _call("unmore_pack_detections", image_ids.data_ptr(), bbox.data_ptr(), out5.data_ptr(), keep_counts.data_ptr(), cap, B,
              rows.data_ptr(), rows.shape[0] - 1, _stream())
    return rows


# ---- the tile path of the second resize mode (antialias=True): the stages on pre-resampled tiles ----------------------
def tile_means(tiles: torch.Tensor) -> torch.Tensor:
    """[M, 128, 128] fp32 tiles (dim-0 stride free, the tile itself contiguous) -> their means [M] (a3 on tiles)."""
    if not tiles.is_cuda or tiles.dtype != torch.float32 or tiles.dim() != 3 or tiles.shape[1:] != (CROP, CROP) or \
            tiles.stride(2) != 1 or tiles.stride(1) != CROP:
        raise _lib.UnmoreError("tile_means needs CUDA fp32 [M, 128, 128] with contiguous tiles")
    M = tiles.shape[0]
    out = torch.zeros((M,), dtype=torch.float32, device=tiles.device)
    _on(tiles)
    if M:
        _call("unmore_tile_means", tiles.data_ptr(), int(tiles.stride(0)), M, out.data_ptr(), _stream())
    return out


def center_reasoning_from_tiles(tiles, H, W, boxes, counts=None, thr: float = 0.009, ws=None, want_splits: bool = True,
                                analyze_cc: bool = False, image_hw=None):
    """center_reasoning on tiles [n_img, cap, 3, 128, 128] = (sdf, center_row, center_col); same returns as
    ``center_reasoning``.  H, W: image size (the --analyze_cc enlargement clips against it).  ``image_hw`` [n_img, 2]
    int32: the tiles come from a padded stack (``crop_resize(..., antialias=True, image_hw=)``), H, W are its pitch and
    each image's windows and clip use its own size."""
    tiles = _on(tiles.contiguous())
    n_img, cap = tiles.shape[0], tiles.shape[1]
    _, f64 = _check_boxes(boxes, n_img)
    _check_counts(counts, n_img)
    dev = tiles.device
    hw = None if image_hw is None else _check_extents(image_hw, n_img, dev, "center_reasoning_from_tiles")
    ws = workspace(n_img, dev) if ws is None else ws
    maxv = torch.zeros((n_img, cap), dtype=torch.float64, device=dev)
    argmax = torch.full((n_img, cap), -1, dtype=torch.int32, device=dev)
    splits = torch.zeros((n_img, cap, 4, 4), dtype=torch.float64, device=dev) if want_splits else None
    cc = None
    if analyze_cc:
        cc_cap = _lib.load().unmore_cc_cap()
        cc = (torch.zeros((n_img, cap), dtype=torch.uint8, device=dev),
              torch.zeros((n_img, cap, cc_cap, 4), dtype=torch.float64, device=dev),
              torch.zeros((1,), dtype=torch.int32, device=dev))
    _on(tiles)
    if cap:
        name, size = ("unmore_center_reasoning_from_tiles", (int(H), int(W))) if hw is None else \
            ("unmore_center_reasoning_from_tiles_hw", (int(H), int(W), hw.data_ptr()))
        _call(name, tiles.data_ptr(), n_img, *size, boxes.data_ptr(), f64, _ptr(counts), cap,
              float(thr), maxv.data_ptr(), argmax.data_ptr(), _ptr(splits), _ptr(cc[0]) if cc else None,
              _ptr(cc[1]) if cc else None, _ptr(cc[2]) if cc else None, ws.data_ptr(), _stream(), counts=counts)
    return maxv, argmax, splits, cc


def boundary_round_from_tiles(tiles, boxes, H, W, max_sdf_thres: float = 0.5, max_shrink_threshold: float = 16.0,
                              delta_ratio: float = 0.5):
    """One round of optimize_one_image_single_round on sdf tiles [M, 128, 128] and their boxes [M, 4] (fp64 or fp32):
    -> (updated boxes [M, 4] fp32, labels [M] fp32 in {-1, 0, 1})."""
    tiles = _on(tiles.contiguous())
    M = tiles.shape[0]
    boxes = boxes.contiguous()
    if boxes.shape != (M, 4) or boxes.dtype not in (torch.float32, torch.float64):
        raise _lib.UnmoreError("boundary_round_from_tiles: boxes must be [M, 4] fp32 / fp64")
    dev = tiles.device
    out = torch.zeros((M, 4), dtype=torch.float32, device=dev)
    lab = torch.full((M,), -1.0, dtype=torch.float32, device=dev)
    if M:
        dws = torch.empty((M, 4), dtype=torch.float32, device=dev)
        mws = torch.empty((M,), dtype=torch.float32, device=dev)
        _on(tiles)
        _call("unmore_boundary_round_from_tiles", tiles.data_ptr(), M, boxes.data_ptr(), int(boxes.dtype == torch.float64), int(H), int(W),
              float(max_sdf_thres), float(max_shrink_threshold), float(delta_ratio), out.data_ptr(), lab.data_ptr(),
              dws.data_ptr(), mws.data_ptr(), _stream())
    return out, lab


def score_and_rasterise_from_tiles(tiles, H, W, boxes, counts=None, want_masks: bool = True, antialias: bool = True,
                                   existence_scores: Optional[torch.Tensor] = None, image_hw=None):
    """score_and_rasterise on tiles [n_img, cap, 4, 128, 128] = (sdf, center_row, center_col, existence); the masks are
    resized back to the box with the antialiased kernel (``antialias``) or the plain one; ``existence_scores``
    [n_img, cap] fp32, when given, replaces the mean of the fourth tile.  Same returns as ``score_and_rasterise``.
    ``image_hw`` [n_img, 2] int32: the tiles come from a padded stack (``crop_resize(..., antialias=True, image_hw=)``)
    and H, W are its pitch; the masks stay on the pitched canvas as in ``score_and_rasterise``."""
    tiles = _on(tiles.contiguous())
    n_img, cap = tiles.shape[0], tiles.shape[1]
    _, f64 = _check_boxes(boxes, n_img)
    _check_counts(counts, n_img)
    dev = tiles.device
    hw = None if image_hw is None else _check_extents(image_hw, n_img, dev, "score_and_rasterise_from_tiles")
    scores = torch.zeros((n_img, cap, 4), dtype=torch.float32, device=dev)
    tight = torch.zeros((n_img, cap, 4), dtype=torch.float32, device=dev)
    areas = torch.zeros((n_img, cap), dtype=torch.int32, device=dev)
    masks = torch.zeros((n_img, cap, H, (W + 31) // 32), dtype=torch.int32, device=dev) if want_masks else None
    _on(tiles)
    if cap > 0:
        if existence_scores is not None:
            existence_scores = existence_scores.to(dev, torch.float32).reshape(n_img, cap).contiguous()
        name, size = ("unmore_score_and_rasterise_from_tiles", (int(H), int(W))) if hw is None else \
            ("unmore_score_and_rasterise_from_tiles_hw", (int(H), int(W), hw.data_ptr()))
        _call(name, tiles.data_ptr(), _ptr(existence_scores), int(antialias), n_img, *size,
              boxes.data_ptr(), f64, _ptr(counts), cap,
              scores.data_ptr(), tight.data_ptr(), areas.data_ptr(), _ptr(masks), _stream())
    return scores, tight, areas, masks
