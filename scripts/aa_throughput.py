"""Throughput of the second resize mode (antialias=True): the image-by-image tile path against the batched path, discovery
plus scoring, on the inputs of ``bench.py --config antialias`` (synth.make_fields(i), synth.make_proposals(i, 4096)).

* tile path: what this mode ran before the fused kernels, one image at a time: antialiased crops of the existence
  channel + tile_means, of the three center-stage channels + center_reasoning_from_tiles, of the boundary-distance
  channel alone in every round of the host loop _boundary_reasoning_tiles; then Object_Scoring.score_batch;
* batched path: ReasoningPipeline.run_chunk on all images (fused antialiased existence, center reasoning and refine,
  batched scoring).

Warm-up, then the two paths alternately, timed with CUDA events around synchronised runs; then one more run of each
with ops.StageTimer for the stage split, and the batched path's center stage once more with every count zero: its
time is what the stage costs with no work in it.  Peak device memory is that of one batched run.  Launches are the kernels of the
C-ABI calls (ops.LAUNCHES); the fills and copies torch launches around them are not counted.  Prints one JSON line and
asserts that both paths produced identical boxes, scores and masks.  usage: python scripts/aa_throughput.py [--images 16] [--repeats 3]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))   # repo root (scripts/..)
import numpy as np
import torch

from unmore_b200 import ops, synth
from unmore_b200.object_reasoning import Object_Discovery, default_args
from unmore_b200.object_scoring import Object_Scoring
from unmore_b200.pipeline import ReasoningPipeline

H, W, N = 480, 640, 4096


class AaTiles:
    """Tile provider of the tile path: antialiased crops of the field stack (center stage and existence)."""
    antialias = True

    def __init__(self, ch: ops.Channels):
        self.ch = ch

    def fields(self, f, boxes):
        return ops.crop_resize(f[None].contiguous(), boxes[None].contiguous(), [self.ch.sdf, self.ch.center_row,
                                                                                 self.ch.center_col], antialias=True)[0]

    def existence(self, f, boxes):
        tiles = ops.crop_resize(f[None].contiguous(), boxes[None].contiguous(), [self.ch.exist], antialias=True)
        return ops.tile_means(tiles[0, :, 0])


class TileDiscovery(Object_Discovery):
    """The refine rounds of the tile path crop the boundary-distance channel only, not the provider's three channels."""

    def _sdf_tiles(self, f, boxes):
        return ops.crop_resize(f, boxes[None].contiguous(), [self.channels.sdf], antialias=True)[0, :, 0]


class LabelledTimer(ops.StageTimer):
    """StageTimer whose entries are named after the stage being run (set by the wrappers below), not the C call."""
    stage = "other"

    def record(self, name, kernels, fn, *args):
        super().record(name, kernels, fn, *args)
        n, a, b = self.events[-1]
        self.events[-1] = (self.stage, a, b)


def _staged(fn, stage):
    def run(*a, **k):
        prev, LabelledTimer.stage = LabelledTimer.stage, stage
        try:
            return fn(*a, **k)
        finally:
            LabelledTimer.stage = prev
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=16)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    n = args.images
    fields = torch.stack([synth.make_fields(i, H, W) for i in range(n)]).to(dev)
    props = torch.stack([torch.from_numpy(synth.make_proposals(i, N, H, W)) for i in range(n)]).to(dev)
    rargs = default_args(antialias=True)
    tile_od = TileDiscovery(rargs, device=dev, tile_provider=AaTiles(ops.DEFAULT_CHANNELS))
    scoring = Object_Scoring(argparse.Namespace(antialias=True), device=dev)
    pipe = ReasoningPipeline(dev, rargs, with_sat=False)
    # stage labels for the split (the wrappers only name the timer's entries)
    ops.existence_scores = _staged(ops.existence_scores, "existence")
    ops.center_reasoning = _staged(ops.center_reasoning, "center")
    ops.boundary_refine = _staged(ops.boundary_refine, "refine")
    tile_od.existence_checking = _staged(tile_od.existence_checking, "existence")
    tile_od.center_reasoning = _staged(tile_od.center_reasoning, "center")
    tile_od.boundary_reasoning = _staged(tile_od.boundary_reasoning, "refine")
    scoring.score_batch = _staged(scoring.score_batch, "scoring")
    pipe.scoring.score_batch = _staged(pipe.scoring.score_batch, "scoring")

    def tile_path():
        res = []
        for b in range(n):
            det = tile_od.discover_image(fields[b], props[b])
            boxes = torch.as_tensor(det, device=dev).reshape(1, -1, 4).contiguous()
            res.append((det, scoring.score_batch(fields[b:b + 1], boxes) if len(det) else None))
        return res

    def batched_path():
        return pipe.run_chunk(fields, props)

    def timed(fn):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ops.LAUNCHES
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / 1e3, ops.LAUNCHES - l0, out

    for _ in range(args.warmup):
        timed(tile_path)
        timed(batched_path)
    t_tile, t_batch = [], []
    for _ in range(args.repeats):
        dt, l_tile, res_tile = timed(tile_path)
        t_tile.append(dt)
        dt, l_batch, res_batch = timed(batched_path)
        t_batch.append(dt)

    # identical outputs: discovered boxes, scoring outputs in NMS order and the kept masks
    r = res_batch
    n_det = n_ann = 0
    for b, (det, sc) in enumerate(res_tile):
        k = int(r["box_counts"][b])
        assert np.array_equal(r["boxes"][b, :k].cpu().numpy(), det), f"discovered boxes differ, image {b}"
        n_det += k
        kk = int(r["keep_counts"][b])
        if sc is None:
            assert kk == 0
            continue
        assert kk == int(sc["keep_counts"][0]), f"kept annotations differ, image {b}"
        assert torch.equal(r["out"][b, :kk], sc["out"][0, :kk]) and torch.equal(r["bbox"][b, :kk], sc["bbox"][0, :kk])
        assert torch.equal(r["keep"][b, :kk], sc["keep"][0, :kk])
        keep = r["keep"][b, :kk].long()
        assert torch.equal(r["masks"][b][keep], sc["masks"][0][keep]), f"masks differ, image {b}"
        n_ann += kk

    torch.cuda.reset_peak_memory_stats()
    batched_path()
    peak = torch.cuda.max_memory_allocated()
    split = {}
    for name, fn in (("tile", tile_path), ("batched", batched_path)):
        t = LabelledTimer()
        ops.set_timer(t)
        fn()
        ops.set_timer(None)
        split[name] = {k: round(v["ms"], 2) for k, v in sorted(t.summary().items())}

    # the batched center stage with no proposal in it: p1 (capacity N) and the split list (capacity 4N), as discover_batch
    ws = ops.workspace(n, dev)
    zero = torch.zeros((n,), dtype=torch.int32, device=dev)
    empty = [torch.zeros((n, cap, 4), dtype=torch.float64, device=dev) for cap in (N, 4 * N)]

    def empty_center():
        ops.center_reasoning(fields, empty[0], zero, ws=ws, antialias=True)
        ops.center_reasoning(fields, empty[1], zero, ws=ws, want_splits=False, antialias=True)

    timed(empty_center)
    t_empty, _, _ = timed(empty_center)

    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    med = lambda v: float(np.median(v))
    print(json.dumps({
        "gpu": torch.cuda.get_device_name(dev), "power_limit": power, "images": n, "proposals": N, "repeats": args.repeats,
        "tile_images_per_s": round(n / med(t_tile), 2), "batched_images_per_s": round(n / med(t_batch), 2),
        "speedup": round(med(t_tile) / med(t_batch), 2), "tile_s": [round(v, 3) for v in t_tile],
        "batched_s": [round(v, 3) for v in t_batch], "tile_launches_per_image": round(l_tile / n, 1),
        "batched_launches_per_image": round(l_batch / n, 1), "stage_ms": split,
        "center_empty_ms": round(t_empty * 1e3, 2), "batched_peak_device_memory_gb": round(peak / 1e9, 2),
        "launches_counted": "C-ABI kernels (ops.LAUNCHES); torch fills and copies not counted", "discovered": n_det, "annotations": n_ann,
        "outputs_identical": True}))


if __name__ == "__main__":
    main()
