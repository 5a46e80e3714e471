"""Discovery + scoring throughput over images of different sizes, three ways on the same images:
  (a) per_image  - one image per call, the loop the zero-argument mains run with batch_size=1;
  (b) same_size  - batches of identical size only, through the uniform path;
  (c) padded     - padded mixed batches (ops.pack_fields + image_hw) of --batch images.
Plus a uniform 480x640 batch with an image_hw table (the *_hw entry points) against the same batch without one.
Asserts that all ways give identical outputs and prints one JSON line.  --antialias runs all of it in the second resize mode (antialias=True).

The shape table below is a plausible mix of photo shapes with a 640-px longer side (4:3, 3:2, 16:9, portrait, square)
plus a few small images.  It is NOT COCO's measured size distribution.
usage: python scripts/mixed_size_throughput.py [--images 250] [--batch 250] [--proposals 4096] [--seed 0] [--antialias]"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from unmore_b200 import ops, synth  # noqa: E402
from unmore_b200.object_reasoning import Object_Discovery, default_args  # noqa: E402
from unmore_b200.object_scoring import Object_Scoring  # noqa: E402

SHAPES = [  # (h, w, weight)
    (480, 640, 30), (640, 480, 10), (427, 640, 15), (640, 427, 5), (360, 640, 12), (640, 360, 3),
    (640, 640, 8), (512, 512, 5), (240, 320, 5), (200, 300, 4), (128, 128, 3)]


def draw_shapes(n, seed):
    rng = np.random.default_rng(seed)
    w = np.array([s[2] for s in SHAPES], dtype=np.float64)
    idx = rng.choice(len(SHAPES), size=n, p=w / w.sum())
    return [SHAPES[i][:2] for i in idx]


def run_batch(od, osc, fields, boxes, counts, image_hw=None):
    kb, kc = od.discover_batch(fields, boxes, counts, image_hw=image_hw)
    n_max = int(kc.max().item()) if kc.numel() else 0
    cap = 8
    while cap < max(n_max, 1):
        cap *= 2
    det = kb[:, :cap].contiguous()
    sc = osc.score_batch(fields, det, kc, image_hw=image_hw)
    return kb, kc, sc


def outputs(kb, kc, sc, b, h, w):
    """Per-image results on the host: discovered boxes, scores, bbox and masks in keep order, cut to the image."""
    k, kk = int(kc[b]), int(sc["keep_counts"][b])
    keep = sc["keep"][b, :kk].long()
    return (kb[b, :k].cpu().numpy(), sc["out"][b, :kk].cpu().numpy(), sc["bbox"][b, :kk].cpu().numpy(),
            sc["masks"][b][keep][:, :h, : (w + 31) // 32].cpu().numpy())


def timed(fn, timer):
    ops.set_timer(timer)
    l0 = ops.LAUNCHES
    torch.cuda.synchronize()
    t = time.perf_counter()
    res = fn()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t
    ops.set_timer(None)
    return res, dt, ops.LAUNCHES - l0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=250)
    ap.add_argument("--batch", type=int, default=250)
    ap.add_argument("--proposals", type=int, default=4096)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--antialias", action="store_true", help="the second resize mode (antialias=True)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    shapes = draw_shapes(a.images, a.seed)
    images = [synth.make_fields(i, h, w).to(dev) for i, (h, w) in enumerate(shapes)]
    props = [torch.from_numpy(synth.make_proposals(i, a.proposals, h, w)).to(dev) for i, (h, w) in enumerate(shapes)]
    od = Object_Discovery(default_args(antialias=a.antialias), device=dev)
    osc = Object_Scoring(argparse.Namespace(antialias=a.antialias), device=dev)

    def per_image():
        return [outputs(*run_batch(od, osc, im[None].contiguous(), p[None].contiguous(), None), 0, *im.shape[1:])
                for im, p in zip(images, props)]

    def same_size():
        res = [None] * len(images)
        for hw in sorted(set(shapes)):
            idx = [i for i, s in enumerate(shapes) if s == hw]
            for s in range(0, len(idx), a.batch):
                sel = idx[s: s + a.batch]
                kb, kc, sc = run_batch(od, osc, torch.stack([images[i] for i in sel]), torch.stack([props[i] for i in sel]), None)
                for b, i in enumerate(sel):
                    res[i] = outputs(kb, kc, sc, b, *hw)
        return res

    pad_stats = {"pixels": 0, "padded": 0}

    def padded():
        res = []
        for s in range(0, len(images), a.batch):
            ims = images[s: s + a.batch]
            fields, hw = ops.pack_fields(ims)
            pad_stats["pixels"] += fields[:, 0].numel()
            pad_stats["padded"] += fields[:, 0].numel() - sum(im.shape[1] * im.shape[2] for im in ims)
            boxes, counts = ops.stack_proposals(props[s: s + a.batch], dev)
            kb, kc, sc = run_batch(od, osc, fields, boxes, counts, hw)
            res += [outputs(kb, kc, sc, b, *im.shape[1:]) for b, im in enumerate(ims)]
        return res

    # warm-up of every shape the timed runs use (first launches load modules)
    run_batch(od, osc, images[0][None].contiguous(), props[0][None].contiguous(), None)
    n_warm = min(4, len(images))
    f, hw = ops.pack_fields(images[:n_warm])
    bx, ct = ops.stack_proposals(props[:n_warm], dev)
    run_batch(od, osc, f, bx, ct, hw)

    result = {"images": a.images, "batch": a.batch, "proposals_per_image": a.proposals, "antialias": a.antialias, "ways": {}}
    outs = {}
    torch.cuda.reset_peak_memory_stats()
    for name, fn in (("per_image", per_image), ("same_size", same_size), ("padded", padded)):
        timer = ops.StageTimer()
        torch.cuda.reset_peak_memory_stats()
        outs[name], dt, launches = timed(fn, timer)
        stages = {k: round(v["ms"], 2) for k, v in timer.summary().items()}
        result["ways"][name] = {"images_per_s": round(a.images / dt, 2), "seconds": round(dt, 3),
                                "c_abi_launches_per_image": round(launches / a.images, 1), "stage_ms": stages,
                                "peak_device_memory_gb": round(torch.cuda.max_memory_allocated() / 1e9, 2)}
    for name in ("same_size", "padded"):
        for i, (x, y) in enumerate(zip(outs["per_image"], outs[name])):
            for u, v in zip(x, y):
                assert u.shape == v.shape and np.array_equal(u.view(np.uint8), v.view(np.uint8)), (name, i)
    result["padded_pixel_fraction"] = round(pad_stats["padded"] / max(pad_stats["pixels"], 1), 4)
    result["speedup_padded_vs_per_image"] = round(result["ways"]["padded"]["images_per_s"] / result["ways"]["per_image"]["images_per_s"], 2)

    # a uniform 480x640 batch (no padding) with an image_hw table against the same batch without one, alternating
    nu = min(a.batch, 64)
    uf = torch.stack([synth.make_fields(1000 + i) for i in range(nu)]).to(dev)
    up = torch.stack([torch.from_numpy(synth.make_proposals(1000 + i, a.proposals)) for i in range(nu)]).to(dev)
    uhw = torch.tensor([[480, 640]] * nu, dtype=torch.int32, device=dev)
    times = {"uniform": [], "sized": []}
    ref = run_batch(od, osc, uf, up, None)
    got = run_batch(od, osc, uf, up, None, uhw)
    assert torch.equal(ref[0], got[0]) and torch.equal(ref[2]["out"], got[2]["out"]) and torch.equal(ref[2]["masks"], got[2]["masks"])
    for _ in range(3):
        for key, hwarg in (("uniform", None), ("sized", uhw)):
            _, dt, _ = timed(lambda: run_batch(od, osc, uf, up, None, hwarg), None)
            times[key].append(dt)
    result["uniform_480x640"] = {"images": nu, "uniform_images_per_s": round(nu / min(times["uniform"]), 2),
                                 "sized_images_per_s": round(nu / min(times["sized"]), 2),
                                 "sized_over_uniform_time": round(min(times["sized"]) / min(times["uniform"]), 4),
                                 "runs_s": {k: [round(t, 4) for t in v] for k, v in times.items()}}
    try:
        import subprocess
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
    except OSError:
        q = ""
    result["card"] = q or torch.cuda.get_device_name(0)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
