"""Host-side mirror of the reference's ``object_reasoning.py`` (class ``Object_Discovery``).

Method names, argument order, return containers and dict keys follow the reference
(object_reasoning.py:43-665); the arithmetic runs in libunmore_b200.so on the GPU.  The
one deliberate difference is the producer boundary: the reference runs its nets on every
crop, every round (:398-417); here ``image`` is the per-image ``[4, H, W]`` field stack the
objectness net produced once ([sdf, center_row, center_col, existence]) and the kernels
resample it per proposal — SURVEY.md §0 "field-stub bridge".

``discover_batch`` is the batched, sync-free form of ``main_object_discovery``'s loop body
used by bench.py and the multi-GPU sharder: many images per launch, ragged lists with
device-side counts, no host round-trips between stages.
"""
from __future__ import annotations

import argparse
import json
import os
from typing import Dict, Optional

import numpy as np
import torch

from . import ops
from .synth import anchor_proposals

HYPER_DEFAULTS = dict(  # object_reasoning.py:700-707
    class_score_thres=0.1, center_score_max_thres=0.009, analyze_cc=False, max_sdf_thres=0.5,
    max_shrink_threshold=16, delta_ratio=0.5, n_round=50, proposal_area_thres=50, seed=0)


def default_args(**over) -> argparse.Namespace:
    d = dict(HYPER_DEFAULTS)
    d.update(over)
    return argparse.Namespace(**d)


def _label_boxes_host(mask_u8: np.ndarray):
    """8-connected components of one [128,128] mask on the host, in scipy's label order, as
    [x_start, y_start, x_stop, y_stop] slice bounds — the overflow path of separate_connected_components
    (more components than the kernels' per-proposal box buffer, unmore_cc_cap())."""
    from scipy.ndimage import find_objects, label
    lab, n = label(mask_u8, np.ones((3, 3), dtype=np.int64))
    return [[sl[1].start, sl[0].start, sl[1].stop, sl[0].stop] for sl in find_objects(lab)][:n]


class FieldDataset:
    """Duck-typed stand-in for the reference's ``COCO_Dataset`` on this path (datasets.py:441-453): the
    field stacks the producer made, addressed by position.  ``get_image_with_index(i)`` returns
    ``(fields [4,H,W] fp32, {'image_id': tensor})`` exactly like the reference's accessor returns the RGB
    image; ``start_idx`` / ``end_idx`` select a contiguous range like datasets.py:432-435."""

    def __init__(self, fields, image_ids=None, start_idx: int = -1, end_idx: int = -1):
        n = len(fields)
        ids = list(range(n)) if image_ids is None else [int(i) for i in image_ids]
        sel = range(n) if (start_idx == -1 or end_idx == -1) else range(n)[start_idx:end_idx]
        self.fields = fields
        self.index = list(sel)
        self.image_ids = ids

    def __len__(self):
        return len(self.index)

    def get_image_with_index(self, index):
        k = self.index[index]
        return self.fields[k], {"image_id": torch.tensor(self.image_ids[k])}


class Object_Discovery:
    def __init__(self, args: Optional[argparse.Namespace] = None, device=None, channels: ops.Channels = ops.DEFAULT_CHANNELS,
                 test_dataset=None, result_folder: Optional[str] = None, tile_provider=None):
        """Reference: ``Object_Discovery(args, device)`` (object_reasoning.py:44-107).  The reference builds its
        nets and a COCO_Dataset from ``args``; here the producer is outside the path, so the dataset of field
        stacks (anything with ``__len__`` / ``get_image_with_index``, e.g. ``FieldDataset``) and the result
        folder are handed in (or assigned to ``self.test_dataset`` / ``self.result_folder`` afterwards)."""
        self.args = args if args is not None else default_args()
        for k, v in HYPER_DEFAULTS.items():
            if not hasattr(self.args, k):
                setattr(self.args, k, v)
        self.device = torch.device(device if device is not None else "cuda:0")
        if self.device.type != "cuda":
            raise RuntimeError("unmore_b200 has no CPU path; pass a CUDA device")
        self.channels = channels
        self.height = None
        self.width = None
        self.test_dataset = test_dataset
        self.result_folder = result_folder
        # resize mode: False = torchvision 0.14.1 semantics (what the reference pins), True = ATen's antialiased kernel
        # (torchvision >= 0.17's default).  Both run batched on the device.  args.antialias, when present, sets it.
        self.antialias = bool(getattr(self.args, "antialias", False))
        # the reference's ORIGINAL mode: nets on every crop (producer.PerCropNets).  ``image`` is then the RGB image and
        # every stage runs on the tiles the provider makes (the tile path), in the provider's resize mode.
        self.tile_provider = tile_provider

    # ---- a1 ---------------------------------------------------------------------------
    @staticmethod
    def generate_random_proposal(height, width):
        """object_reasoning.py:110-137 — float64 [N,4] anchors (host side, negligible cost)."""
        return anchor_proposals(height, width)

    @staticmethod
    def unravel_index(index, shape):
        """object_reasoning.py:199-204 (host integer arithmetic; the kernel does the same split of the
        flat arg-max into (yc, xc), center.cu)."""
        out = []
        for dim in reversed(shape):
            out.append(index % dim)
            index = index // dim
        return tuple(reversed(out))

    def center_field_to_anti_center_map(self, vote_maps, kernel_size=5):
        """object_reasoning.py:360-377 — [B,2,H,W] center fields -> [B,H,W] float64 anti-center map
        (5x5 cross-correlation with the normalised offset filter, zero padding, / (k*k-1))."""
        if kernel_size != 5:
            raise ValueError("the CUDA anti-center map implements the reference's hard-coded kernel_size=5 (:533)")
        return ops.anti_center_map(torch.as_tensor(vote_maps).to(self.device), kernel_size)

    def get_prediction_with_proposal_images(self, proposal_images):
        """object_reasoning.py:339-358 under the field-stub bridge: ``proposal_images`` are already-cropped
        [N,C,128,128] field tiles, the 'net' selects channels -> (sdf_maps [N,128,128], center_fields [N,2,128,128])."""
        t = torch.as_tensor(proposal_images).to(self.device, torch.float32)
        ch = self.channels
        return t[:, ch.sdf], torch.stack((t[:, ch.center_row], t[:, ch.center_col]), dim=1)

    # ---- helpers ----------------------------------------------------------------------
    def _fields(self, image: torch.Tensor) -> torch.Tensor:
        f = image.to(self.device, torch.float32)
        if f.dim() == 3:
            f = f.unsqueeze(0)
        return f.contiguous()

    def _boxes(self, proposals) -> torch.Tensor:
        if not torch.is_tensor(proposals):
            proposals = torch.as_tensor(np.asarray(proposals))
        if proposals.numel() == 0:
            return torch.zeros((1, 0, 4), dtype=torch.float64, device=self.device)
        if proposals.dtype not in (torch.float32, torch.float64):
            proposals = proposals.to(torch.float64)
        return proposals.to(self.device).reshape(1, -1, 4).contiguous()

    @property
    def _tile_path(self) -> bool:
        """Per-crop nets (a tile provider) run every stage on the provider's tiles, image by image."""
        return self.tile_provider is not None

    def _field_tiles(self, f: torch.Tensor, boxes: torch.Tensor) -> torch.Tensor:
        """[1,K,3,128,128] (sdf, center_row, center_col) tiles of ``boxes`` [1,K,4] from the tile provider."""
        return self.tile_provider.fields(f[0], boxes[0])[None]

    # ---- a3 ---------------------------------------------------------------------------
    def existence_checking(self, image, proposals) -> Dict[str, torch.Tensor]:
        """object_reasoning.py:491-523 — {'existence_scores': [N] fp32 on CPU}."""
        boxes = self._boxes(proposals)
        if boxes.shape[1] == 0:
            return {"existence_scores": torch.zeros((0,), dtype=torch.float32)}
        if self.tile_provider is not None:   # the reference's original mode: one classifier output per crop
            return {"existence_scores": self.tile_provider.existence(self._fields(image)[0], boxes[0]).cpu()}
        scores = ops.existence_scores(self._fields(image), boxes, ch=self.channels, antialias=self.antialias)
        return {"existence_scores": scores[0].cpu()}

    # ---- a4 ---------------------------------------------------------------------------
    def get_prediction_with_proposals(self, proposals, image):
        """object_reasoning.py:301-337 (note the (proposals, image) order): the resized crops of the
        boundary-distance and center fields, (sdf_maps [N,128,128], center_fields [N,2,128,128])."""
        boxes = self._boxes(proposals)
        ch = self.channels
        if self.tile_provider is not None:
            crops = self.tile_provider.fields(self._fields(image)[0], boxes[0])
        else:
            crops = ops.crop_resize(self._fields(image), boxes, [ch.sdf, ch.center_row, ch.center_col], antialias=self.antialias)[0]
        return crops[:, 0], crops[:, 1:3]

    # ---- a7 ---------------------------------------------------------------------------
    def center_reasoning(self, image, proposals) -> Dict[str, torch.Tensor]:
        """object_reasoning.py:525-580 — {'proposals_pass_singularity', 'splited_new_proposals'}
        (an empty float64 [0,4] tensor where the reference leaves an empty list)."""
        boxes = self._boxes(proposals)
        if boxes.shape[1] == 0:
            e = torch.zeros((0, 4), dtype=torch.float64, device=self.device)
            return {"proposals_pass_singularity": e, "splited_new_proposals": e.clone()}
        cc_on = bool(getattr(self.args, "analyze_cc", False))
        if self._tile_path:
            f = self._fields(image)
            tiles = self._field_tiles(f, boxes)
            _, argmax, splits, cc = ops.center_reasoning_from_tiles(tiles, f.shape[-2], f.shape[-1], boxes,
                                                                    thr=self.args.center_score_max_thres, analyze_cc=cc_on)
        else:
            _, argmax, splits, cc = ops.center_reasoning(self._fields(image), boxes, thr=self.args.center_score_max_thres,
                                                         ch=self.channels, analyze_cc=cc_on, antialias=self.antialias)
        fail = argmax[0] >= 0
        new = splits[0][fail].reshape(-1, 4)
        if cc_on:
            # (:561-572) enlarged component boxes of passing multi-component masks, appended after the splits
            counts, cboxes, overflow = cc
            if int(overflow.item()):
                f = self._fields(image)
                extra = self._cc_boxes_with_overflow(f, boxes, torch.nonzero(~fail).flatten().tolist(), counts[0], cboxes[0],
                                                     f.shape[-2], f.shape[-1])
                new = torch.cat((new, torch.as_tensor(extra, device=self.device)), dim=0)
            else:
                valid = torch.arange(cboxes.shape[2], device=self.device)[None, :] < counts[0][:, None].to(torch.long)
                new = torch.cat((new, cboxes[0][valid]), dim=0)
        return {"proposals_pass_singularity": boxes[0][~fail], "splited_new_proposals": new}

    def _union_masks(self, fields: torch.Tensor, boxes: torch.Tensor) -> torch.Tensor:
        """Un-eroded union masks (object_reasoning.py:528-531) of ``boxes`` [1,K,4] as [K,128,128] u8, from the
        bit-exact resized crops and the same thresholds the center kernel applies (common.cuh)."""
        ch = self.channels
        crops = self._field_tiles(fields, boxes.contiguous())[0] if self.tile_provider is not None else \
            ops.crop_resize(fields, boxes.contiguous(), [ch.sdf, ch.center_row, ch.center_col], antialias=self.antialias)[0]
        sq = crops[:, 1] * crops[:, 1] + crops[:, 2] * crops[:, 2]
        return ((crops[:, 0] > 8.94069671630859375e-08) | (sq > 0.2500000298023223876953125)).to(torch.uint8)

    def _cc_boxes_with_overflow(self, fields, boxes, passing_idx, cc_counts, cc_boxes, H, W):
        """Component boxes (enlarged, :561-572) of the passing proposals ``passing_idx`` of ONE image, in
        proposal order.  Proposals whose component count reached the device buffer (unmore_cc_cap()) are
        re-labelled on the host without a limit, so any number of components is handled like the reference
        (object_reasoning.py:207-256) — only those rare proposals leave the device."""
        cap = cc_boxes.shape[1]
        counts = cc_counts.cpu().numpy()
        dev_boxes = cc_boxes.cpu().numpy()
        full = [int(k) for k in passing_idx if counts[k] >= cap]
        host = {}
        if full:
            masks = self._union_masks(fields, boxes[:, full]).cpu().numpy()
            for k, m in zip(full, masks):
                bb = _label_boxes_host(m)
                host[k] = np.asarray(self.enlarge_proposals(bb, (H, W), 1.5), dtype=np.float64).reshape(-1, 4)
        out = []
        for k in passing_idx:
            k = int(k)
            if k in host:
                if len(host[k]) >= 2:
                    out.append(host[k])
            elif counts[k]:
                out.append(dev_boxes[k, : counts[k]])
        return np.concatenate(out, axis=0) if out else np.zeros((0, 4), np.float64)

    @staticmethod
    def separate_connected_components(binary_masks):
        """object_reasoning.py:207-256 — ({'single': [...], 'multi': [...]}, indicators) with bboxes
        [x_start, y_start, x_stop, y_stop]; labelling on the GPU (8-connected, scipy label order)."""
        m8 = (binary_masks != 0).to(torch.uint8)
        counts, boxes = ops.connected_components(m8)
        counts, boxes = counts.cpu().tolist(), boxes.cpu().tolist()
        cap = len(boxes[0]) if boxes else 0
        combined = {"single": [], "multi": []}
        indicators = []
        for i, (n, bb) in enumerate(zip(counts, boxes)):
            if n > cap:   # more components than the device buffer holds: label this one mask on the host
                bb = _label_boxes_host(m8[i].cpu().numpy())
                n = len(bb)
            if n == 1:
                combined["single"].append(bb[0])
                indicators.append(1)
            else:
                indicators.append(0)
                combined["multi"].extend(bb[:n])
        return combined, indicators

    @staticmethod
    def enlarge_proposals(proposals, image_shape, ratio):
        """object_reasoning.py:259-291 (host arithmetic on a handful of boxes; fused on the device
        inside center_reasoning when args.analyze_cc is set)."""
        height, width = image_shape
        out = []
        for x1, y1, x2, y2 in proposals:
            cx, cy = (x1 + x2) / 2, (y1 + y2) / 2
            nw, nh = (x2 - x1) * ratio, (y2 - y1) * ratio
            out.append([int(max(cx - nw / 2, 0)), int(max(cy - nh / 2, 0)), int(min(cx + nw / 2, width)),
                        int(min(cy + nh / 2, height))])
        return out

    # ---- a9 ---------------------------------------------------------------------------
    def filter_small_proposal(self, proposals, labels):
        """object_reasoning.py:293-299 (plain tensor indexing; the fused loop does this on device)."""
        area = (proposals[:, 2] - proposals[:, 0]) * (proposals[:, 3] - proposals[:, 1])
        keep = area > self.args.proposal_area_thres
        return proposals[keep], labels[keep]

    # ---- a10 / a12 --------------------------------------------------------------------
    @staticmethod
    def update_bbox_with_boundary_fields(sdf_maps):
        """object_reasoning.py:140-174 on [B,128,128] CUDA tiles -> (dx1, dy1, dx2, dy2)."""
        deltas, _ = ops.update_bbox_from_tiles(sdf_maps)
        return deltas[:, 0], deltas[:, 1], deltas[:, 2], deltas[:, 3]

    @staticmethod
    def post_process_bbox_update(original_bboxes, delta_bboxes, delta_scale_x=128, delta_scale_y=128):
        """object_reasoning.py:177-196 — four elementwise ops; kept in torch (fused on device inside
        the refine kernel, this entry point exists for signature parity)."""
        xr = (original_bboxes[:, 2] - original_bboxes[:, 0]) / delta_scale_x
        yr = (original_bboxes[:, 3] - original_bboxes[:, 1]) / delta_scale_y
        out = original_bboxes.clone()
        out[:, 0] = original_bboxes[:, 0] + delta_bboxes[:, 0] * xr
        out[:, 1] = original_bboxes[:, 1] + delta_bboxes[:, 1] * yr
        out[:, 2] = original_bboxes[:, 2] + delta_bboxes[:, 2] * xr
        out[:, 3] = original_bboxes[:, 3] + delta_bboxes[:, 3] * yr
        return out

    # ---- a11 --------------------------------------------------------------------------
    def optimize_one_image_single_round(self, image, proposals, labels=None) -> Dict[str, torch.Tensor]:
        """object_reasoning.py:379-487 — {'updated_bboxes': [N,4] fp32, 'labels': [N] fp32}."""
        boxes = self._boxes(proposals)
        if boxes.shape[1] == 0:
            return {"updated_bboxes": torch.zeros((0, 4), dtype=torch.float32, device=self.device),
                    "labels": torch.zeros((0,), dtype=torch.float32, device=self.device)}
        a = self.args
        if self._tile_path:
            f = self._fields(image)
            tiles = self._sdf_tiles(f, boxes[0])
            out, lab = ops.boundary_round_from_tiles(tiles, boxes[0], f.shape[-2], f.shape[-1], max_sdf_thres=a.max_sdf_thres,
                                                     max_shrink_threshold=a.max_shrink_threshold, delta_ratio=a.delta_ratio)
            return {"updated_bboxes": out, "labels": lab}
        out, lab, _ = ops.boundary_refine(self._fields(image), boxes, n_round=1, apply_small_filter=False,
                                          early_exit=False, proposal_area_thres=a.proposal_area_thres,
                                          max_sdf_thres=a.max_sdf_thres, max_shrink_threshold=a.max_shrink_threshold,
                                          delta_ratio=a.delta_ratio, ch=self.channels, antialias=self.antialias)
        return {"updated_bboxes": out[0], "labels": lab[0]}

    # ---- a13 --------------------------------------------------------------------------
    def boundary_reasoning(self, image, proposals, n_round=50):
        """object_reasoning.py:582-612.  Like the reference the loop length is ``args.n_round``
        (the parameter is ignored there too, :592).  Returns the rows still in the list after
        the last round — label -1 rows of the last round included as zero boxes."""
        boxes = self._boxes(proposals)
        if boxes.shape[1] == 0:
            return {"proposals": [], "labels": []}
        a = self.args
        if self._tile_path:
            return self._boundary_reasoning_tiles(self._fields(image), boxes[0])
        out, lab, _ = ops.boundary_refine(self._fields(image), boxes, n_round=a.n_round, apply_small_filter=True,
                                          early_exit=True, proposal_area_thres=a.proposal_area_thres,
                                          max_sdf_thres=a.max_sdf_thres, max_shrink_threshold=a.max_shrink_threshold,
                                          delta_ratio=a.delta_ratio, ch=self.channels, antialias=self.antialias)
        in_list = lab[0] > -2
        if int(in_list.sum()) == 0:
            return {"proposals": [], "labels": []}
        return {"proposals": out[0][in_list], "labels": lab[0][in_list]}

    def _sdf_tiles(self, f: torch.Tensor, boxes: torch.Tensor) -> torch.Tensor:
        """[K,128,128] boundary-distance tiles of ``boxes`` [K,4]: the tile provider's, else antialiased crops (the
        tile-by-tile form of the second resize mode, kept as the reference of the fused antialiased refine)."""
        if self.tile_provider is not None:
            return self.tile_provider.fields(f[0], boxes)[:, 0].contiguous()
        return ops.crop_resize(f, boxes[None].contiguous(), [self.channels.sdf], antialias=True)[0, :, 0]

    def _boundary_reasoning_tiles(self, f: torch.Tensor, cur: torch.Tensor):
        """boundary_reasoning (object_reasoning.py:582-612) on tiles: the round loop runs on the host like the
        reference's, every round is crop (the tile provider's, else antialiased) -> tiles -> tile reductions -> box
        update on the device.  Rows that reached label 1 with an unchanged box are exact fixed points and are not recomputed."""
        a = self.args
        H, W = f.shape[-2], f.shape[-1]
        labels = torch.zeros((cur.shape[0],), dtype=torch.float32, device=self.device)
        fixed = torch.zeros((cur.shape[0],), dtype=torch.bool, device=self.device)
        for _ in range(a.n_round):
            area = (cur[:, 2] - cur[:, 0]) * (cur[:, 3] - cur[:, 1])          # filter_small_proposal (:293-299), in cur's dtype
            keep = area > a.proposal_area_thres
            cur, labels, fixed = cur[keep], labels[keep], fixed[keep]
            if cur.shape[0] == 0:
                return {"proposals": [], "labels": []}
            act = ~fixed
            new = cur.to(torch.float32).clone()
            newl = labels.clone()
            if bool(act.any()):
                boxes = cur[act].contiguous()
                tiles = self._sdf_tiles(f, boxes)
                out, lab = ops.boundary_round_from_tiles(tiles, boxes, H, W, max_sdf_thres=a.max_sdf_thres,
                                                         max_shrink_threshold=a.max_shrink_threshold, delta_ratio=a.delta_ratio)
                new[act] = out
                newl[act] = lab
                same = (out.to(cur.dtype) == boxes).all(dim=1) & (lab == 1)
                fx = fixed.clone()
                fx[act] = same
                fixed = fx
            cur, labels = new, newl
            if bool(fixed.all()):
                break
        return {"proposals": cur, "labels": labels}

    # ---- main loop body ---------------------------------------------------------------
    def discover_image(self, image, proposals=None) -> np.ndarray:
        """Loop body of main_object_discovery (object_reasoning.py:618-662) for one image:
        final [K,4] fp32 boxes (empty where the reference ``continue``s)."""
        f = self._fields(image)
        if proposals is None:
            proposals = self.generate_random_proposal(f.shape[-2], f.shape[-1])
        boxes = self._boxes(proposals)
        if self._tile_path:
            return self._discover_image_tiles(f[0], boxes[0])
        det, cnt = self.discover_batch(f, boxes)
        return det[0, : int(cnt[0])].cpu().numpy()

    def _discover_image_tiles(self, image: torch.Tensor, proposals: torch.Tensor) -> np.ndarray:
        """The loop body of main_object_discovery (:623-662) with per-crop nets, stage by stage through the
        reference-named methods (each one on the tile path); empty intermediate lists end the image like the
        reference's ``continue``s (and an empty split list is 'no splits' instead of the reference's crash)."""
        a = self.args
        empty = np.zeros((0, 4), dtype=np.float32)
        ex = self.existence_checking(image, proposals)["existence_scores"].to(self.device)
        proposals = proposals[ex >= a.class_score_thres]
        if len(proposals) == 0:
            return empty
        cr = self.center_reasoning(image, proposals)
        p_pass, split = cr["proposals_pass_singularity"], cr["splited_new_proposals"]
        if len(split) > 0:
            ex2 = self.existence_checking(image, split)["existence_scores"].to(self.device)
            split = split[ex2 >= a.class_score_thres]
        if len(split) > 0:
            cr2 = self.center_reasoning(image, split)
            proposals = torch.cat((p_pass, cr2["proposals_pass_singularity"]), dim=0)
        else:
            proposals = p_pass
        if len(proposals) == 0:
            return empty
        br = self.boundary_reasoning(image, proposals)
        if len(br["proposals"]) == 0:
            return empty
        final = br["proposals"][br["labels"] == 1]
        if len(final) == 0:
            return empty
        keep, kc, kb = ops.box_nms(final.to(torch.float32)[None].contiguous(), None, None, iou_threshold=0.5)
        return kb[0, : int(kc[0])].cpu().numpy()

    def discover_batch(self, fields: torch.Tensor, proposals: torch.Tensor, counts: Optional[torch.Tensor] = None,
                       stats: Optional[dict] = None, image_hw: Optional[torch.Tensor] = None):
        """Existence check -> center reasoning -> re-check of the splits -> boundary reasoning ->
        NMS for a batch of images, entirely on device.

        fields [B,4,H,W] fp32, proposals [B,N,4] fp64/fp32, counts [B] int32 or None.
        ``image_hw`` [B,2] int32 (device): ``fields`` is a padded stack of images of different sizes
        (``ops.pack_fields``); every image gets what it would get alone, in either resize mode.  Not with a tile provider.
        Returns (boxes [B, 5N (9N + 256 with --analyze_cc), 4] fp32, counts [B] int32) in the reference's output order."""
        a = self.args
        ch = self.channels
        B, N = proposals.shape[0], proposals.shape[1]
        dev = fields.device
        f64 = torch.float64
        if image_hw is not None and self._tile_path:
            raise ops.UnmoreError("discover_batch: image_hw (images of different sizes) is not supported with a tile provider")
        if self._tile_path:   # per-crop nets: image by image on the tile path (not the fused kernels)
            dets = [self._discover_image_tiles(fields[b], proposals[b] if counts is None else proposals[b, : int(counts[b])])
                    for b in range(B)]
            cap = max([len(d) for d in dets] + [1])
            kb = torch.zeros((B, cap, 4), dtype=torch.float32, device=dev)
            kc = torch.tensor([len(d) for d in dets], dtype=torch.int32, device=dev)
            for b, d in enumerate(dets):
                if len(d):
                    kb[b, : len(d)] = torch.as_tensor(d, device=dev)
            return kb, kc
        ws = ops.workspace(B, dev)
        # Step 1: existence checking (:627-630)
        aa = self.antialias
        hw = image_hw
        ex = ops.existence_scores(fields, proposals, counts, ch=ch, ws=ws, antialias=aa, image_hw=hw)
        p1, c1, _ = ops.compact_boxes(proposals, counts, ops.MODE_SCORE_GE, ex, thr=a.class_score_thres, out_dtype=f64)
        # Step 2: center reasoning (:634-637)
        cc_on = bool(getattr(a, "analyze_cc", False))
        _, am1, sp1, cc = ops.center_reasoning(fields, p1, c1, thr=a.center_score_max_thres, ch=ch, ws=ws,
                                               analyze_cc=cc_on, antialias=aa, image_hw=hw)
        # 4 split boxes per failing proposal; with --analyze_cc the component boxes of passing proposals follow
        # (a speckled mask can carry dozens: the reference has no limit, here the list holds 4N + 4N + 256 rows)
        split_cap = 8 * N + 256 if cc_on else 4 * N
        cap_out = N + split_cap
        refine_in = torch.zeros((B, cap_out, 4), dtype=f64, device=dev)
        rc = torch.zeros((B,), dtype=torch.int32, device=dev)
        ops.compact_boxes(p1, c1, ops.MODE_ARGMAX_LT0, am1, out=refine_in, counts_out=rc)
        split, sc, _ = ops.compact_boxes(sp1, c1, ops.MODE_ARGMAX_GE0, am1, group=4, out_dtype=f64, cap_out=split_cap)
        if cc_on:
            # (:561-572) component boxes of passing multi-component masks follow the split boxes
            cc_counts, cc_boxes, cc_over = cc
            lost = torch.zeros((1,), dtype=torch.int32, device=dev)
            ops.compact_boxes(cc_boxes, c1, ops.MODE_U8_NONZERO, cc_counts, group=cc_boxes.shape[2], out=split,
                              counts_out=sc, append=True, group_counts=cc_counts, overflow=lost)
            if int(lost.item()):   # one sync per batch, only with --analyze_cc
                raise RuntimeError("analyze_cc: component boxes exceeded the split-list capacity")
            if int(cc_over.item()):
                # a proposal with more components than the device buffer (unmore_cc_cap()): rebuild the component
                # part of the split list of the affected images with the unlimited host labelling (rare path)
                c1h = c1.cpu().tolist()
                hwh = None if hw is None else hw.cpu().tolist()
                capc = cc_boxes.shape[2]
                for b in range(B):
                    n = c1h[b]
                    if n == 0 or int((cc_counts[b, :n] >= capc).sum()) == 0:
                        continue
                    passing = torch.nonzero(am1[b, :n] < 0).flatten().tolist()
                    if hwh is None:
                        fb, (hb, wb) = fields[b:b + 1], fields.shape[-2:]
                    else:   # the image alone, at its own size (the kernels clamp the extents the same way)
                        hb, wb = (min(max(v, 1), p) for v, p in zip(hwh[b], fields.shape[-2:]))
                        fb = fields[b:b + 1, :, :hb, :wb].contiguous()
                    extra = self._cc_boxes_with_overflow(fb, p1[b:b + 1], passing, cc_counts[b], cc_boxes[b], hb, wb)
                    n_split = 4 * int((am1[b, :n] >= 0).sum())
                    if n_split + len(extra) > split_cap:
                        raise RuntimeError("analyze_cc: component boxes exceeded the split-list capacity")
                    split[b, n_split:n_split + len(extra)] = torch.as_tensor(extra, device=dev)
                    sc[b] = n_split + len(extra)
        # re-check the split proposals (:639-646)
        ex2 = ops.existence_scores(fields, split, sc, ch=ch, ws=ws, antialias=aa, image_hw=hw)
        p2, c2, _ = ops.compact_boxes(split, sc, ops.MODE_SCORE_GE, ex2, thr=a.class_score_thres, out_dtype=f64)
        _, am2, _, _ = ops.center_reasoning(fields, p2, c2, thr=a.center_score_max_thres, ch=ch, ws=ws, want_splits=False,
                                            antialias=aa, image_hw=hw)
        ops.compact_boxes(p2, c2, ops.MODE_ARGMAX_LT0, am2, out=refine_in, counts_out=rc, append=True)
        # Step 3: boundary reasoning (:650-658)
        rb, lab, rounds = ops.boundary_refine(fields, refine_in, rc, n_round=a.n_round, apply_small_filter=True,
                                              early_exit=True, proposal_area_thres=a.proposal_area_thres,
                                              max_sdf_thres=a.max_sdf_thres,
                                              max_shrink_threshold=a.max_shrink_threshold, delta_ratio=a.delta_ratio,
                                              ch=ch, ws=ws, want_rounds=stats is not None, antialias=aa, image_hw=hw)
        # label-1 survivors; the NMS kernel holds its alive set for at most 32768 boxes per image
        lost1 = torch.zeros((1,), dtype=torch.int32, device=dev) if cap_out > 32768 else None
        fin, fc, _ = ops.compact_boxes(rb, rc, ops.MODE_LABEL_EQ, lab, thr=1.0, out_dtype=torch.float32,
                                       cap_out=min(cap_out, 32768), overflow=lost1)
        if lost1 is not None and int(lost1.item()):
            raise RuntimeError("more than 32768 label-1 boxes in one image")
        # NMS with all-equal scores (:661): index order decides
        _, kc, kb = ops.box_nms(fin, None, fc, iou_threshold=0.5)
        if stats is not None:
            stats.update(existence_in=counts, pass1=c1, split=sc, split_kept=c2, refine_in=rc, refine_rounds=rounds,
                         label1=fc, kept=kc, existence_scores=ex, refine_boxes=rb, refine_labels=lab,
                         refine_in_boxes=refine_in, pass1_boxes=p1, argmax1=am1, pass2_boxes=p2, pass2=c2)
        return kb, kc

    def main_object_discovery(self, images=None, image_ids=None, proposals=None, batch_size: int = 1) -> Dict[int, np.ndarray]:
        """object_reasoning.py:615-665.  Called with no arguments like the reference: loops over
        ``self.test_dataset`` (``get_image_with_index`` -> field stack + ``{'image_id'}``), runs the loop body
        for every image and dumps ``results_dict`` {image_id: [[x1,y1,x2,y2], ...]} to
        ``<result_folder>/discovery_results.json`` (:664-665); images with no detection are absent, as in the
        reference.  ``images`` / ``image_ids`` (not in the reference) run the same loop over in-memory stacks
        without touching the disk.  Returns ``results_dict`` (the reference returns None).

        ``batch_size`` > 1 (not in the reference): consecutive dataset images of any sizes are padded into one stack
        (``ops.pack_fields``), each with its own anchors, and run through ``discover_batch`` together; the results and the
        file are identical to ``batch_size=1``, in either resize mode.  Ignored with a tile provider."""
        from . import rle
        results = {}
        if images is None and batch_size > 1 and not self._tile_path:
            if self.test_dataset is None:
                raise RuntimeError("main_object_discovery(): set self.test_dataset (e.g. FieldDataset) first")
            for start in range(0, len(self.test_dataset), batch_size):
                batch = [self.test_dataset.get_image_with_index(i)
                         for i in range(start, min(start + batch_size, len(self.test_dataset)))]
                ids = [int(lb["image_id"].item()) if torch.is_tensor(lb["image_id"]) else int(lb["image_id"]) for _, lb in batch]
                fields, hw = ops.pack_fields([im.to(self.device, torch.float32) for im, _ in batch])
                self.height, self.width = batch[-1][0].shape[-2], batch[-1][0].shape[-1]
                props = [proposals if proposals is not None else self.generate_random_proposal(im.shape[-2], im.shape[-1])
                         for im, _ in batch]
                boxes, counts = ops.stack_proposals([self._boxes(p)[0] for p in props], self.device)
                kb, kc = self.discover_batch(fields, boxes, counts, image_hw=hw)
                kb, kc = kb.cpu().numpy(), kc.cpu().tolist()
                for b, image_id in enumerate(ids):
                    if kc[b]:
                        results[image_id] = kb[b, : kc[b]].copy()
            return self._write_discovery(results)
        if images is not None:
            for img, iid in zip(images, image_ids):
                det = self.discover_image(img, proposals)
                if len(det):
                    results[int(iid)] = det
            return results
        if self.test_dataset is None:
            raise RuntimeError("main_object_discovery(): set self.test_dataset (e.g. FieldDataset) first")
        for image_idx in range(0, len(self.test_dataset)):
            image, label = self.test_dataset.get_image_with_index(image_idx)
            image_id = int(label["image_id"].item()) if torch.is_tensor(label["image_id"]) else int(label["image_id"])
            self.height, self.width = image.shape[-2], image.shape[-1]
            det = self.discover_image(image, proposals)
            if len(det):
                results[image_id] = det
        return self._write_discovery(results)

    def _write_discovery(self, results):
        from . import rle
        if self.result_folder is not None:
            os.makedirs(self.result_folder, exist_ok=True)
            with open(os.path.join(self.result_folder, "discovery_results.json"), "w") as f:
                f.write(rle.discovery_results_json(results))
        return results
