"""Batched end-to-end reasoning over device-resident (or host-resident) field stacks:
discovery (object_reasoning.py:615-662) followed by scoring (object_scoring.py:172-268) and the
post_process predicate (post_process.py:61-74), many images per launch, no host round-trip
inside a stage.  This is what bench.py times and what the multi-GPU sharder drives."""
from __future__ import annotations

from typing import Optional

import torch

from . import ops
from .object_reasoning import Object_Discovery, default_args
from .object_scoring import Object_Scoring


def _pow2_at_least(n: int, lo: int = 8) -> int:
    c = lo
    while c < n:
        c *= 2
    return c


class ReasoningPipeline:
    def __init__(self, device, args=None, with_sat: bool = True, with_masks: bool = True):
        self.device = torch.device(device)
        self.args = args if args is not None else default_args()
        self.discovery = Object_Discovery(self.args, self.device)
        self.scoring = Object_Scoring(self.args, self.device)
        self.with_sat = with_sat
        self.with_masks = with_masks

    def build_sat(self, fields: torch.Tensor, out: Optional[torch.Tensor] = None,
                  image_hw: Optional[torch.Tensor] = None) -> torch.Tensor:
        """north-star op (a): summed-area tables of the existence and boundary-distance fields,
        [B, 2, H+1, W+1] fp64, built in place from the field stack (a padded one with ``image_hw``)."""
        ch = self.discovery.channels
        return ops.sat_build_fields(fields, [ch.exist, ch.sdf], out=out, image_hw=image_hw)

    def run_chunk(self, fields: torch.Tensor, proposals: torch.Tensor, counts: Optional[torch.Tensor] = None,
                  stats: Optional[dict] = None, sat: Optional[torch.Tensor] = None,
                  image_hw: Optional[torch.Tensor] = None) -> dict:
        """fields [B,4,H,W] fp32 (device), proposals [B,N,4] fp64/fp32 (device).
        Returns device tensors: ``boxes`` [B,cap,4] discovered boxes (xyxy) and ``box_counts``;
        ``out`` [B,cap,5] fp64 (score, existence, center, boundary, area_score), ``bbox`` xywh,
        ``selected`` and ``keep_counts`` in scoring-NMS order; ``masks`` packed; and, with
        ``with_sat``, the O(1) existence / boundary-distance box means of every input proposal.  ``image_hw`` [B,2]
        int32 (device): ``fields`` is a padded stack of images of different sizes (``ops.pack_fields``); a given ``sat``
        must then come from ``build_sat(fields, image_hw=image_hw)``."""
        ch = self.discovery.channels
        res = {}
        if self.with_sat:
            if sat is None:
                sat = self.build_sat(fields, image_hw=image_hw)
            res["exist_box_mean"] = ops.box_sums(sat, 0, proposals, counts, image_hw=image_hw)[1]
            res["sdf_box_mean"] = ops.box_sums(sat, 1, proposals, counts, image_hw=image_hw)[1]
        kb, kc = self.discovery.discover_batch(fields, proposals, counts, stats=stats, image_hw=image_hw)
        n_max = int(kc.max().item()) if kc.numel() else 0   # the one host sync of a chunk: sizes the mask arena
        cap = _pow2_at_least(max(n_max, 1))
        det = kb[:, :cap].contiguous()
        sc = self.scoring.score_batch(fields, det, kc, want_masks=self.with_masks, image_hw=image_hw)
        res.update(boxes=det, box_counts=kc, out=sc["out"], bbox=sc["bbox"], selected=sc["selected"],
                   keep=sc["keep"], keep_counts=sc["keep_counts"], masks=sc["masks"])
        return res
