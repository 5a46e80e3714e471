"""Host-side mirror of the reference's ``object_scoring.py`` (class ``Object_Scoring``).

``main_object_scoring`` (object_scoring.py:172-272) scores every discovered box, rasterises
its union mask on the image canvas, takes the tight box, runs NMS on the tight boxes with
the boundary score, and emits one annotation per survivor.  Arithmetic runs in
libunmore_b200.so; masks stay bit-packed on the device ([H, ceil(W/32)] words, LSB = lowest
x) — the reference's dense [K, H, W] float canvases are never materialised."""
from __future__ import annotations

import argparse
import json
import os
from typing import Dict, List, Optional

import numpy as np
import torch

from . import ops

POST_DEFAULTS = dict(existence_score_thres=0.5, center_score_thres=0.8, boundary_score_thres=0.75)  # post_process.py:38-40


def unpack_masks(packed: torch.Tensor, width: int) -> np.ndarray:
    """[K, H, Wp] int32 packed -> uint8 [K, H, W] (host helper for JSON / tests)."""
    p = packed.cpu().numpy().view(np.uint32)
    bits = np.unpackbits(p.view(np.uint8), axis=-1, bitorder="little")
    return bits.reshape(p.shape[0], p.shape[1], -1)[:, :, :width]


class Object_Scoring:
    def __init__(self, args: Optional[argparse.Namespace] = None, device=None, raw_annotations: Optional[dict] = None,
                 channels: ops.Channels = ops.DEFAULT_CHANNELS, test_dataset=None, result_folder: Optional[str] = None,
                 tile_provider=None):
        """Reference: ``Object_Scoring(args, device)`` (object_scoring.py:45-104); dataset and result folder
        are handed in like in ``Object_Discovery``.  ``args.raw_annotations_path`` is read by
        ``load_raw_annotations`` when ``raw_annotations`` is not given."""
        self.args = args if args is not None else argparse.Namespace()
        for k, v in POST_DEFAULTS.items():
            if not hasattr(self.args, k):
                setattr(self.args, k, v)
        self.device = torch.device(device if device is not None else "cuda:0")
        if self.device.type != "cuda":
            raise RuntimeError("unmore_b200 has no CPU path; pass a CUDA device")
        self.channels = channels
        self.raw_annotations = raw_annotations if raw_annotations is not None else {}
        self.test_dataset = test_dataset
        self.result_folder = result_folder
        # resize mode (see Object_Discovery.antialias): True = the tile path with ATen's antialiased kernels
        self.antialias = bool(getattr(self.args, "antialias", False))
        self.tile_provider = tile_provider   # producer.PerCropNets: the reference's original per-crop mode (image = RGB)
        if raw_annotations is None and getattr(self.args, "raw_annotations_path", None):
            self.load_raw_annotations()

    def load_raw_annotations(self):
        """object_scoring.py:106-110 — reads ``discovery_results.json`` ({image_id: [[x1,y1,x2,y2], ...]})."""
        with open(self.args.raw_annotations_path) as f:
            self.raw_annotations = json.load(f)
        return self.raw_annotations

    def _fields(self, image):
        f = image.to(self.device, torch.float32)
        return (f.unsqueeze(0) if f.dim() == 3 else f).contiguous()

    def get_prediction_with_proposals(self, image, proposals) -> Dict[str, torch.Tensor]:
        """object_scoring.py:112-157 (note the (image, proposals) order): the resized crops of the
        boundary-distance and center fields and the per-crop existence score, under the reference's keys.
        ``score_batch`` never materialises these tiles; this is the signature-parity / inspection form."""
        boxes = torch.as_tensor(np.asarray(proposals, dtype=np.float64)).reshape(1, -1, 4).to(self.device)
        ch = self.channels
        f = self._fields(image)
        if self.tile_provider is not None:
            return {"pred_boundary_fields": (t := self.tile_provider.fields(f[0], boxes[0]))[:, 0], "pred_center_fields": t[:, 1:3],
                    "pred_existence_scores": self.tile_provider.existence(f[0], boxes[0])}
        if self.antialias:
            crops = ops.crop_resize(f, boxes, [ch.sdf, ch.center_row, ch.center_col, ch.exist], antialias=True)[0]
            return {"pred_boundary_fields": crops[:, 0], "pred_center_fields": crops[:, 1:3],
                    "pred_existence_scores": ops.tile_means(crops[:, 3])}
        crops = ops.crop_resize(f, boxes, [ch.sdf, ch.center_row, ch.center_col])[0]
        return {"pred_boundary_fields": crops[:, 0], "pred_center_fields": crops[:, 1:3],
                "pred_existence_scores": ops.existence_scores(f, boxes, ch=ch)[0]}

    def score_batch(self, fields: torch.Tensor, boxes: torch.Tensor, counts: Optional[torch.Tensor] = None,
                    want_masks: bool = True, image_hw: Optional[torch.Tensor] = None):
        """Steps 1-8 of main_object_scoring for a batch: returns a dict of device tensors in NMS keep
        order: out [B,cap,5] fp64 (score, existence, center, boundary, area_score), bbox [B,cap,4] xywh,
        selected [B,cap] (post_process predicate), keep [B,cap], keep_counts [B], masks (packed, indexed by
        the ORIGINAL proposal index: use keep to gather).  ``image_hw`` [B,2] int32 (device): ``fields`` is a padded
        stack of images of different sizes (``ops.pack_fields``); image b's masks are ``masks[b, :, :h_b,
        :ceil(w_b/32)]``.  In either resize mode; not with a tile provider."""
        if image_hw is not None and self.tile_provider is not None:
            raise ops.UnmoreError("score_batch: image_hw (images of different sizes) is not supported with a tile provider")
        if self.tile_provider is not None:   # per-crop nets: (sdf, center) tiles + one classifier scalar per crop
            B, cap = boxes.shape[0], boxes.shape[1]
            tiles = torch.zeros((B, cap, 4, ops.CROP, ops.CROP), dtype=torch.float32, device=fields.device)
            ex = torch.zeros((B, cap), dtype=torch.float32, device=fields.device)
            for b in range(B):
                n = cap if counts is None else int(counts[b])
                if n:
                    tiles[b, :n, 0:3] = self.tile_provider.fields(fields[b], boxes[b, :n])
                    ex[b, :n] = self.tile_provider.existence(fields[b], boxes[b, :n])
            scores, tight, areas, masks = ops.score_and_rasterise_from_tiles(
                tiles, fields.shape[-2], fields.shape[-1], boxes, counts, want_masks=want_masks,
                antialias=self.tile_provider.antialias, existence_scores=ex)
        elif self.antialias:
            ch = self.channels
            tiles = ops.crop_resize(fields, boxes, [ch.sdf, ch.center_row, ch.center_col, ch.exist], counts, antialias=True,
                                    image_hw=image_hw)
            scores, tight, areas, masks = ops.score_and_rasterise_from_tiles(tiles, fields.shape[-2], fields.shape[-1], boxes, counts,
                                                                             want_masks=want_masks, image_hw=image_hw)
        else:
            scores, tight, areas, masks = ops.score_and_rasterise(fields, boxes, counts, ch=self.channels, want_masks=want_masks,
                                                                  image_hw=image_hw)
        keep, kc, _ = ops.box_nms(tight, scores[:, :, 2].contiguous(), counts, iou_threshold=0.5, want_boxes=False)
        out, bbox, sel = ops.final_scores(scores, tight, areas, keep, kc, self.args.existence_score_thres,
                                          self.args.center_score_thres, self.args.boundary_score_thres)
        return dict(out=out, bbox=bbox, selected=sel, keep=keep, keep_counts=kc, masks=masks, areas=areas, tight=tight,
                    scores=scores)

    @staticmethod
    def binary_mask_to_tight_bbox_coco_style(binary_mask):
        """object_scoring.py:160-164 (pycocotools encode + toBbox) for one dense [H, W] mask:
        [xmin, ymin, xmax - xmin + 1, ymax - ymin + 1] as floats, zeros for an empty mask.  Packs the mask and
        takes the extent on the GPU (``unmore_mask_stats``: __ffs / __clz on the packed rows)."""
        m = torch.as_tensor(np.asarray(binary_mask.cpu() if torch.is_tensor(binary_mask) else binary_mask)).to(torch.uint8)
        packed = ops.mask_pack(m.cuda()[None].contiguous())
        areas, tight = ops.mask_stats(packed, m.shape[1])
        if int(areas[0]) == 0:
            return [0.0, 0.0, 0.0, 0.0]
        x1, y1, x2, y2 = (float(v) for v in tight[0].cpu().tolist())
        return [x1, y1, x2 - x1, y2 - y1]   # mask_stats reports exclusive upper bounds (xmax + 1, ymax + 1)

    @staticmethod
    def binary_mask_to_rle(binary_mask):
        """object_scoring.py:167-170 for one dense [H, W] mask (tensor or array): packs it, takes the
        run lengths on the GPU and returns {'size': [H, W], 'counts': ascii str}."""
        from . import rle
        m = torch.as_tensor(np.asarray(binary_mask.cpu() if torch.is_tensor(binary_mask) else binary_mask)).to(torch.uint8)
        packed = ops.mask_pack(m.cuda()[None].contiguous())
        return rle.encode_packed(packed, m.shape[1])[0]

    def score_image(self, image, raw_proposals, image_id=0, with_masks: bool = True, rle: bool = False) -> List[dict]:
        """Annotations of one image with the reference's keys (object_scoring.py:257-267).
        'segmentation' is {'size': [H, W], 'mask': uint8 [H, W]} (dense, for tests) or, with
        ``rle=True``, the reference's COCO RLE dict {'size': [H, W], 'counts': str}."""
        fields = self._fields(image)
        H, W = fields.shape[-2], fields.shape[-1]
        if len(raw_proposals) == 0:
            return []
        boxes = torch.as_tensor(np.asarray(raw_proposals, dtype=np.float64)).reshape(1, -1, 4).to(self.device)
        r = self.score_batch(fields, boxes, None, want_masks=with_masks)
        return self._annotations(r, 0, H, W, image_id, with_masks, rle)

    @staticmethod
    def _annotations(r, b, H, W, image_id, with_masks, rle):
        """Annotations of image ``b`` of a ``score_batch`` result, an (H, W) image; its masks are the [:H, :ceil(W/32)]
        corner of the (possibly pitched) mask canvas."""
        n = int(r["keep_counts"][b])
        keep = r["keep"][b, :n].long()
        out = r["out"][b, :n].cpu().numpy()
        bbox = r["bbox"][b, :n].cpu().numpy()
        masks = r["masks"][b][keep][:, :H, : (W + 31) // 32] if with_masks else None
        dense = unpack_masks(masks, W) if (with_masks and not rle) else None
        if with_masks and rle:
            from . import rle as rle_codec
            encoded = rle_codec.encode_packed(masks.contiguous(), W)
        anns = []
        for i in range(n):
            ann = {"image_id": image_id, "category_id": 1, "score": out[i, 0], "bbox": [v for v in bbox[i]],
                   "existence_score": np.float32(out[i, 1]), "center_score": np.float32(out[i, 2]),
                   "boundary_score": np.float32(out[i, 3]), "area_score": out[i, 4]}
            if with_masks:
                ann["segmentation"] = encoded[i] if rle else {"size": [H, W], "mask": dense[i]}
            anns.append(ann)
        return anns

    def main_object_scoring(self, images=None, image_ids=None, batch_size: int = 1) -> List[dict]:
        """object_scoring.py:172-272.  Called with no arguments like the reference: loops over
        ``self.test_dataset``, skips images without raw predictions (:177-179), and dumps ``out_annotations``
        (``segmentation`` = COCO RLE dicts, :257-268) to ``<result_folder>/object_discovery_with_scores.json``.
        ``images`` / ``image_ids`` (not in the reference) run the loop over in-memory stacks and keep the masks
        dense.  Returns ``out_annotations`` (the reference returns None).

        ``batch_size`` > 1 (not in the reference): consecutive dataset images of any sizes are padded into one stack
        (``ops.pack_fields``) and scored by one ``score_batch``; the annotations and the file are identical to
        ``batch_size=1``, in either resize mode.  Ignored with a tile provider."""
        out = []
        if images is None and batch_size > 1 and self.tile_provider is None:
            if self.test_dataset is None:
                raise RuntimeError("main_object_scoring(): set self.test_dataset (e.g. FieldDataset) first")
            for start in range(0, len(self.test_dataset), batch_size):
                batch = []
                for image_idx in range(start, min(start + batch_size, len(self.test_dataset))):
                    image, label = self.test_dataset.get_image_with_index(image_idx)
                    image_id = int(label["image_id"].item()) if torch.is_tensor(label["image_id"]) else int(label["image_id"])
                    if str(image_id) not in self.raw_annotations.keys():
                        print(image_id, "do not have raw predictions")
                        continue
                    batch.append((image, image_id, self.raw_annotations[str(image_id)]))
                if not batch:
                    continue
                fields, hw = ops.pack_fields([self._fields(im)[0] for im, _, _ in batch])
                boxes, counts = ops.stack_proposals(
                    [torch.as_tensor(np.asarray(raw, dtype=np.float64)).reshape(-1, 4) for _, _, raw in batch], self.device)
                r = self.score_batch(fields, boxes, counts, image_hw=hw)
                for b, (im, image_id, _) in enumerate(batch):
                    out.extend(self._annotations(r, b, im.shape[-2], im.shape[-1], image_id, True, True))
            return self._write_scoring(out)
        if images is not None:
            for img, iid in zip(images, image_ids):
                raw = self.raw_annotations.get(str(int(iid)))
                if raw is None:
                    continue
                out.extend(self.score_image(img, raw, image_id=int(iid)))
            return out
        if self.test_dataset is None:
            raise RuntimeError("main_object_scoring(): set self.test_dataset (e.g. FieldDataset) first")
        for image_idx in range(0, len(self.test_dataset)):
            image, label = self.test_dataset.get_image_with_index(image_idx)
            image_id = int(label["image_id"].item()) if torch.is_tensor(label["image_id"]) else int(label["image_id"])
            if str(image_id) not in self.raw_annotations.keys():
                print(image_id, "do not have raw predictions")
                continue
            out.extend(self.score_image(image, self.raw_annotations[str(image_id)], image_id=image_id, rle=True))
        return self._write_scoring(out)

    def _write_scoring(self, out):
        from . import rle
        if self.result_folder is not None:
            os.makedirs(self.result_folder, exist_ok=True)
            with open(os.path.join(self.result_folder, "object_discovery_with_scores.json"), "w") as f:
                f.write(rle.scored_annotations_json(out))
        return out
