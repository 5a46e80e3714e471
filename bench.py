#!/usr/bin/env python
"""Benchmark of the multi-object reasoning hot path.

    python bench.py --gpus N --steps K --warmup W                 # configs[1], our CUDA path
    python bench.py --impl reference ...                          # the CPU oracle port, bounded sample
    python bench.py --scaling strong ...                          # 5000 images TOTAL, interleaved over the ranks
    python bench.py --config producer [--producer-dtype fp32]     # configs[4]: DPT-L producer -> reasoning, 1024x1024
    python bench.py --config antialias [--images 16]              # the second resize mode (tile path), image by image
    python bench.py ... --dump-outputs DIR                        # also write the last timed step's result as .npy

configs[1] (default): a COCO-val-shaped synthetic batch — 5000 images of 480x640 fields, 4096 proposals per
image — through discovery (existence check, center reasoning, iterative boundary refinement, NMS), scoring +
mask rasterisation and the post-process predicate.  One "step" = one pass over the per-rank batch.  Prints ONE
JSON line (rank 0).  Default scaling is weak (every rank owns `--images` images, seeds = global image index);
the only collective is ONE all_gather_into_tensor of the fixed-capacity detection-row buffer at the end of a
step, inside the timed region, with no host synchronisation in front of it.

``--dump-outputs DIR`` writes what the last timed step delivered to its caller as ``DIR/<name>.npy``.  The inputs
are generated from fixed seeds, so two builds run with the same arguments can be compared output for output.
  * reasoning and producer configs: ``detections`` float64 ``[K, 6]`` rows ``(image_id, x, y, w, h, score)`` (COCO
    xywh boxes), image-sorted: the gathered detection rows.
  * antialias config: ``discovery`` float64 ``[D, 5]`` rows ``(image, x1, y1, x2, y2)``; ``annotations`` float64
    ``[A, 10]`` rows ``(image, x, y, w, h, score, existence_score, center_score, boundary_score, area_score)``;
    ``masks`` float32 ``[M, H, W]``, a seeded sample of at most DUMP_MASKS of the annotation masks, and
    ``mask_index`` float64 ``[M]``, the annotation rows they belong to.
Above DUMP_BYTES in all, every array keeps a fixed, seeded sample of its rows.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, N_PROP = 480, 640, 4096
WORKLOAD = "configs[1]: 5000 synthetic 480x640 field stacks x 4096 proposals/image, discovery + scoring"
XU_CYCLES_PER_ROW = 98.0   # 12.2 MUFU warp-instructions per output row (ex2, rcp, sqrt per pixel) x 8 cycles on the 4-lane XU pipe of one SM sub-partition
DUMP_BYTES = 64_000_000    # upper bound of what --dump-outputs writes
DUMP_MASKS = 16            # masks --dump-outputs keeps in the antialias config (1.2 MB each in float32 at 480x640)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="reasoning", choices=["reasoning", "producer", "antialias"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--images", type=int, default=None, help="images per rank (weak) or in total (strong); default 5000 (reasoning) / 16 (producer)")
    ap.add_argument("--proposals", type=int, default=N_PROP)
    ap.add_argument("--chunk", type=int, default=250, help="images per launch group")
    ap.add_argument("--cpu-sample-proposals", type=int, default=1536,
                    help="proposals of image 0 the CPU baseline / reference arm processes per sample (~7 s on 16 cores)")
    ap.add_argument("--producer-dtype", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--producer-batch", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """{name: float32 / float64 array (numpy or torch, any device)} -> out_dir/<name>.npy.  If the arrays hold
    more than DUMP_BYTES together, each one keeps a share of DUMP_BYTES in proportion to its size: a fixed,
    seeded choice of its rows (first axis), in their order."""
    import numpy as np
    arrs = {k: v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v) for k, v in arrays.items()}
    for k, a in arrs.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"{k}: {a.dtype} (dumps are float32 or float64)")
    total = sum(a.nbytes for a in arrs.values())
    budget = DUMP_BYTES - 4096 * len(arrs)   # 4096: room for each .npy header
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrs.items():
        if total > budget and a.ndim and a.shape[0]:
            cap = (budget * a.nbytes // total) // a[:1].nbytes
            if a.shape[0] > cap:
                a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], cap, replace=False))]
        np.save(os.path.join(out_dir, f"{k}.npy"), np.ascontiguousarray(a))


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
def cpu_sample(n_sample: int, n_prop: int, repeats: int = 1, keep_result: bool = False):
    """The oracle port (a bit-identical, faster restatement of the reference's CPU path, see
    oracle/oracle.py) on image 0 with a strided subset of its proposals; scaled to images/s.
    With ``keep_result`` also returns what the oracle produced (for the parity_sample of the bench line)."""
    import numpy as np
    import torch
    from oracle import oracle as O
    from unmore_b200 import synth

    torch.set_num_threads(os.cpu_count() or 1)
    img = synth.make_fields(0, H, W)
    props = synth.make_proposals(0, n_prop, H, W)
    sel = np.unique(np.linspace(0, n_prop - 1, n_sample).round().astype(np.int64))
    args = O.make_args()
    times, res = [], None
    for _ in range(repeats):
        t0 = time.perf_counter()
        det = O.discover_image(img, props[sel], args)
        sc = O.score_image(img, det.tolist(), args) if len(det) else None
        times.append(time.perf_counter() - t0)
        res = (props[sel], det, sc)
    t = statistics.median(times)
    scale = n_prop / len(sel)
    cb = {"value": 1.0 / (t * scale), "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
          "sample": f"image 0, {len(sel)} of {n_prop} proposals (strided), discovery+scoring in {t:.1f}s, "
                    f"scaled x{scale:.1f} to a full image; antialias=False"}
    return (cb, t, res) if keep_result else (cb, t)


def cpu_config0():
    """configs[0] timed in FULL on the CPU port (SURVEY.md section 8d): one 480x640 image, 512 proposals."""
    import torch
    from oracle import oracle as O
    from unmore_b200 import synth
    torch.set_num_threads(os.cpu_count() or 1)
    img = synth.make_fields(0, H, W)
    props = synth.make_proposals(0, 512, H, W)
    args = O.make_args()
    t0 = time.perf_counter()
    det = O.discover_image(img, props, args)
    if len(det):
        O.score_image(img, det.tolist(), args)
    t = time.perf_counter() - t0
    return {"workload": "configs[0]: one 480x640 image, 512 proposals, discovery + scoring, CPU port in full",
            "seconds": t, "images_per_s": 1.0 / t, "cores": torch.get_num_threads(), "detections": int(len(det))}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_img = args.images or 5000
    for _ in range(min(args.warmup, 1)):
        cpu_sample(args.cpu_sample_proposals, args.proposals)
    vals, ts = [], []
    for _ in range(args.steps):
        cb, t = cpu_sample(args.cpu_sample_proposals, args.proposals)
        vals.append(cb["value"]); ts.append(t)
    v = statistics.median(vals)
    cb["value"] = v
    line = {"impl": "reference", "metric": "object_reasoning_images_per_sec", "value": v, "unit": "images/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * statistics.median(ts), "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "images_per_rank": n_img, "proposals_per_image": args.proposals,
                       "field_hw": [H, W]},
            "proposals_per_sec": v * args.proposals, "cpu_baseline": cb,
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
def parity_sample(pipe, dev, oracle_res):
    """The GPU path on the SAME strided proposal subset of image 0 the CPU sample just processed, compared with
    what the oracle produced: list equality, worst relative box / score error, mask bit-equality."""
    import numpy as np
    import torch
    from unmore_b200 import synth
    from unmore_b200.object_scoring import unpack_masks
    props, det_ref, sc_ref = oracle_res
    f = synth.make_fields(0, H, W).to(dev)[None].contiguous()
    r = pipe.run_chunk(f, torch.tensor(props, device=dev)[None].contiguous())
    k = int(r["box_counts"][0])
    det = r["boxes"][0, :k].cpu().numpy()
    out = {"proposals": int(len(props)), "detections_ref": int(len(det_ref)), "detections_gpu": k,
           "lists_equal": bool(det.shape == det_ref.shape), "max_rel_err": None, "masks_equal": None, "scores_max_rel_err": None}
    if det.shape == det_ref.shape and len(det_ref):
        side = np.maximum(det_ref[:, 2] - det_ref[:, 0], det_ref[:, 3] - det_ref[:, 1])[:, None]
        out["max_rel_err"] = float((np.abs(det - det_ref) / np.maximum(np.abs(det_ref), side)).max())
        kk = int(r["keep_counts"][0])
        keep = r["keep"][0, :kk].long()
        same = kk == len(sc_ref["score"]) and np.array_equal(keep.cpu().numpy(), sc_ref["nms_index"])
        out["lists_equal"] = bool(out["lists_equal"] and same)
        if same:
            out["masks_equal"] = bool(np.array_equal(unpack_masks(r["masks"][0][keep], W), sc_ref["masks"]))
            s = r["out"][0, :kk, 0].cpu().numpy()
            out["scores_max_rel_err"] = float((np.abs(s - sc_ref["score"]) / np.abs(sc_ref["score"])).max())
            out["bbox_equal"] = bool(np.array_equal(r["bbox"][0, :kk].cpu().numpy(), sc_ref["bbox"]))
    return out


# ---------------------------------------------------------------------------------------------
def run_antialias(args):
    """The second resize mode (antialias=True, tile path) on a few benchmark images, image by image through the mirror
    classes: a labelled side figure, not the headline (the fused kernels implement the pinned antialias=False)."""
    import argparse as ap_
    import numpy as np
    import torch
    from unmore_b200 import ops, synth
    from unmore_b200.object_reasoning import Object_Discovery, default_args
    from unmore_b200.object_scoring import Object_Scoring
    if int(os.environ.get("RANK", "0")) != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    n_img = args.images or 16
    od = Object_Discovery(default_args(antialias=True), device=dev)
    sc = Object_Scoring(ap_.Namespace(antialias=True), device=dev)
    imgs = [synth.make_fields(i, H, W).to(dev) for i in range(n_img)]
    props = [synth.make_proposals(i, args.proposals, H, W) for i in range(n_img)]

    def step():
        """-> (annotations, [(image, discovered boxes)], [annotations with their masks])"""
        n, dets, anns = 0, [], []
        for k, (f, p) in enumerate(zip(imgs, props)):
            det = od.discover_image(f, p)
            dets.append((k, det))
            if len(det):
                a = sc.score_image(f, det.astype(np.float64).tolist(), image_id=k)
                n += len(a)
                anns += a
        return n, dets, anns

    for _ in range(max(1, min(args.warmup, 1))):
        step()
    torch.cuda.synchronize()
    l0 = ops.LAUNCHES
    t0 = time.perf_counter()
    for _ in range(args.steps):
        n_ann, dets, anns = step()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs is not None:
        keys = ("score", "existence_score", "center_score", "boundary_score", "area_score")
        masks = np.stack([a["segmentation"]["mask"] for a in anns]) if anns else np.zeros((0, H, W), np.uint8)
        pick = np.sort(np.random.default_rng(0).choice(len(anns), min(len(anns), DUMP_MASKS), replace=False))
        dump_outputs(args.dump_outputs, {
            "discovery": np.array([[k, *b] for k, det in dets for b in det], np.float64).reshape(-1, 5),
            "annotations": np.array([[a["image_id"], *a["bbox"], *(a[c] for c in keys)] for a in anns],
                                    np.float64).reshape(-1, 10),
            "masks": masks[pick].astype(np.float32), "mask_index": pick.astype(np.float64)})
    print(json.dumps({"metric": "object_reasoning_images_per_sec", "value": n_img / dt, "unit": "images/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": f"second resize mode (antialias=True, tile path, image by image): {n_img} synthetic 480x640 "
                                             f"field stacks x {args.proposals} proposals, discovery + scoring through the mirror classes",
                                 "resize": "bilinear, antialias=True (torchvision >= 0.17 default)"},
                      "annotations": n_ann, "gpu_launches": ops.LAUNCHES - l0, "timing": "wall clock around synchronised steps"}))


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    if args.config == "antialias":
        return run_antialias(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from unmore_b200 import ops, synth
    from unmore_b200.pipeline import ReasoningPipeline
    from unmore_b200.sharding import gather_rows, merge_rows, overflowed, rows_digest, shard_indices

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    producer_cfg = args.config == "producer"
    Hc, Wc = (1024, 1024) if producer_cfg else (H, W)
    n_total_arg = args.images if args.images is not None else (16 if producer_cfg else 5000)
    if args.scaling == "strong":
        my_ids = shard_indices(n_total_arg, rank, world, interleave=True)   # image i -> rank i mod G
        n_global = n_total_arg
    else:
        my_ids = list(range(rank * n_total_arg, (rank + 1) * n_total_arg))
        n_global = n_total_arg * world
    n_img = len(my_ids)
    n_prop = args.proposals
    chunk = max(1, min(args.chunk, n_img))
    px = Hc * Wc
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")

    # ---- synthetic inputs, generated on the device (seed = global image index)
    t_gen = time.time()
    producer = None
    if producer_cfg:
        from unmore_b200.producer import FieldProducer
        anchors = synth.anchor_proposals(Hc, Wc)
        n_prop = len(anchors)
        torch.manual_seed(0)   # identical weights on every rank
        producer = FieldProducer(autocast_dtype=torch.bfloat16 if args.producer_dtype == "bf16" else None).to(dev).eval()
        gen = torch.Generator(device=dev)

        def rgb_images(ids):
            out = torch.empty((len(ids), 3, Hc, Wc), device=dev)
            for k, i in enumerate(ids):
                gen.manual_seed(int(i))
                out[k] = torch.rand((3, Hc, Wc), generator=gen, device=dev)
            return out

        producer.calibrate_random_init(rgb_images([0]))
        rgb = rgb_images(my_ids)                                   # resident input of the producer config
        fields = torch.empty((n_img, 4, Hc, Wc), dtype=torch.float32, device=dev)
        props_np = np.ascontiguousarray(np.broadcast_to(anchors, (n_img,) + anchors.shape))
    else:
        fields = torch.empty((n_img, 4, Hc, Wc), dtype=torch.float32, device=dev)
        for k, i in enumerate(my_ids):
            fields[k] = synth.render_fields(synth.scene_params(i, Hc, Wc), Hc, Wc, device=dev)
        anchors = synth.anchor_proposals(Hc, Wc)
        props_np = np.empty((n_img, n_prop, 4), dtype=np.float64)
        for k, i in enumerate(my_ids):
            if n_prop >= len(anchors):
                props_np[k, : len(anchors)] = anchors
                props_np[k, len(anchors):] = synth.random_proposals(i, n_prop - len(anchors), Hc, Wc)
            else:
                props_np[k] = synth.make_proposals(i, n_prop, Hc, Wc)
    proposals = torch.from_numpy(props_np).to(dev)
    image_ids = torch.tensor(my_ids, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    t_gen = time.time() - t_gen

    pipe = ReasoningPipeline(dev, with_sat=not producer_cfg)
    sat_buf = None if producer_cfg else torch.empty((n_img, 2, Hc + 1, Wc + 1), dtype=torch.float64, device=dev)
    # one capacity on every rank (the collective has a fixed shape): 16 detection rows per image on average
    n_img_max = -(-n_global // world) if args.scaling == "strong" else n_total_arg
    max_rows = 16 * max(n_img_max, 1) + 64
    prod_ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def step(collect_stats=None):
        rows = ops.detection_rows(max_rows, dev)
        if producer is not None:
            prod_ev[0].record()
            for i0 in range(0, n_img, args.producer_batch):
                producer(rgb[i0:i0 + args.producer_batch], out=fields[i0:i0 + args.producer_batch])
            prod_ev[1].record()
        # north-star op (a): summed-area tables of the existence / boundary-distance fields for the
        # whole batch in one HBM-streaming launch; the chunks below read their slices
        sat = pipe.build_sat(fields, out=sat_buf) if sat_buf is not None else None
        for c0 in range(0, n_img, chunk):
            c1 = min(c0 + chunk, n_img)
            st = {} if collect_stats is not None else None
            r = pipe.run_chunk(fields[c0:c1], proposals[c0:c1], stats=st, sat=None if sat is None else sat[c0:c1])
            ops.pack_detections(image_ids[c0:c1], r["bbox"], r["out"], r["keep_counts"], rows)   # device-side append
            if collect_stats is not None:
                collect_stats["proposal_rounds"] = collect_stats.get("proposal_rounds", 0) + int(st["refine_rounds"].sum())
                collect_stats["refine_in"] = collect_stats.get("refine_in", 0) + int(st["refine_in"].sum())
                collect_stats["center_in"] = collect_stats.get("center_in", 0) + int(st["pass1"].sum()) + int(st["split_kept"].sum())
                collect_stats["exist_in"] = collect_stats.get("exist_in", 0) + (c1 - c0) * n_prop + int(st["split"].sum())
                collect_stats["detections"] = collect_stats.get("detections", 0) + int(r["keep_counts"].sum())
        g = gather_rows(rows)            # the single collective of the path (no-op at world 1), no host sync before it
        merged, total = merge_rows(g)    # image-sorted on the device; sliced when read
        return merged, total, g

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 0)):
        step()
    work = {}
    step(work)  # untimed: work counters for the roofline arithmetic (device syncs inside)

    # ---- timed region: K steps, device time, max over ranks
    sampler = ClockSampler(local_rank)
    timer = ops.StageTimer()
    barrier()
    sampler.start()
    launches0 = ops.LAUNCHES
    ops.set_timer(timer)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    prof_range = os.environ.get("UNMORE_PROFILE_RANGE") == "1"   # ncu --profile-from-start off: timed region only
    if prof_range:
        torch.cuda.profiler.start()
    producer_ms = 0.0
    ev0.record()
    for _ in range(args.steps):
        merged, total, g = step()
        if producer is not None:
            torch.cuda.synchronize()
            producer_ms += prod_ev[0].elapsed_time(prod_ev[1])
    ev1.record()
    barrier()
    if prof_range:
        torch.cuda.profiler.stop()
    ops.set_timer(None)
    clocks = sampler.stop()
    launches = ops.LAUNCHES - launches0
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    images_per_s = n_global / (ms_per_step / 1e3)
    stages = timer.summary()
    if bool(overflowed(g)):
        raise RuntimeError("detection row buffer overflowed: raise max_rows")
    result_rows = merged[: int(total.item())]
    digest = rows_digest(result_rows)
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, {"detections": result_rows})

    # ---- hardware equality: rank 0 recomputes, on its own, a slice of images that ANOTHER rank owned and
    # compares the rows the collective delivered for them, bit for bit (outside the timed region)
    gather_equal = None
    if world > 1 and not producer_cfg:
        n_chk = min(32, n_img)
        other = (rank + 1) % world
        oth_ids = (shard_indices(n_global, other, world, interleave=True) if args.scaling == "strong"
                   else list(range(other * n_total_arg, (other + 1) * n_total_arg)))[:n_chk]
        f2 = torch.stack([synth.render_fields(synth.scene_params(i, Hc, Wc), Hc, Wc, device=dev) for i in oth_ids])
        p2 = torch.from_numpy(np.stack([np.concatenate([anchors, synth.random_proposals(i, n_prop - len(anchors), Hc, Wc)])
                                        if n_prop >= len(anchors) else synth.make_proposals(i, n_prop, Hc, Wc)
                                        for i in oth_ids])).to(dev)
        r2 = pipe.run_chunk(f2, p2)
        rows2 = ops.pack_detections(torch.tensor(oth_ids, dtype=torch.int64, device=dev), r2["bbox"], r2["out"], r2["keep_counts"],
                                    ops.detection_rows(max_rows, dev))
        mine = rows2[1:1 + int(rows2[0, 0].item())]
        idset = torch.tensor(oth_ids, dtype=torch.float64, device=dev)
        theirs = result_rows[torch.isin(result_rows[:, 0], idset)]
        mine = mine[torch.sort(mine[:, 0], stable=True).indices]
        eq = torch.tensor([int(mine.shape == theirs.shape and torch.equal(mine, theirs))], device=dev)
        dist.all_reduce(eq, op=dist.ReduceOp.MIN)
        gather_equal = bool(eq.item())
        del f2, p2, r2

    # ---- roofline of every kernel from the live CUDA-event times (per launch averages)
    per_step = {k: v["ms"] / args.steps for k, v in stages.items()}
    alg = {  # algorithmic DRAM bytes per STEP (DESIGN.md section 4): fields read once per image + boxes in/out
        "unmore_boundary_refine": n_img * px * 4 + work["refine_in"] * (32 + 16 + 4 + 4),
        "unmore_center_reasoning": n_img * px * 12 + work["center_in"] * (32 + 8 + 4 + 128),
        "unmore_existence_scores": n_img * px * 4 + work["exist_in"] * (32 + 4),
        "unmore_sat_build_fields": n_img * 2 * (px * 4 + (Hc + 1) * (Wc + 1) * 8),
        "unmore_score_and_rasterise": n_img * px * 16 + work["detections"] * (Hc * ((Wc + 31) // 32) * 4),
    }
    kernels = {}
    for name, b in alg.items():
        if name in per_step and per_step[name] > 0:
            ach = b / (per_step[name] / 1e3) / 1e9
            kernels[name] = {"ms_per_step": per_step[name], "share": per_step[name] / ms_per_step,
                             "ms_per_launch": stages[name]["ms"] / stages[name]["calls"], "achieved_gbs": ach,
                             "bound": "hbm", "frac": ach / hbm_peak}
    # ncu figures per launch of exactly this shape, committed under profiles/ (dram bytes, issue-slot utilisation)
    prof = {}
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("images_per_launch") == chunk and tj.get("proposals_per_image") == n_prop and tj.get("field_hw") == [Hc, Wc]:
            prof = tj
    except Exception:
        pass
    for name, k in kernels.items():
        k["traffic"] = prof.get("dram_bytes_per_launch", {}).get(name)
        if name == "unmore_sat_build_fields" and n_img != 5000:
            k["traffic"] = None    # the SAT capture is of the whole 5000-image batch (one launch of 10 000 planes)
        if name in prof.get("issue_active", {}):
            k["issue_active"] = prof["issue_active"][name]
    # the on-chip roofline of the refine kernel: its fields are L2-resident by construction (HBM frac << 1%), the
    # binding unit is the XU (MUFU) pipe: 12.2 MUFU warp-instructions per output row of 128 pixels
    sm_mhz = clocks.get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
    n_sms = torch.cuda.get_device_properties(dev).multi_processor_count
    if "unmore_boundary_refine" in kernels and work.get("proposal_rounds"):
        rows_done = work["proposal_rounds"] * 128.0
        cyc = per_step["unmore_boundary_refine"] * 1e-3 * sm_mhz * 1e6 * n_sms * 4 / rows_done
        kernels["unmore_boundary_refine"]["onchip"] = {
            "bound": "xu", "unit": "cycles per output row per SM sub-partition", "achieved": cyc, "floor": XU_CYCLES_PER_ROW,
            "frac": XU_CYCLES_PER_ROW / cyc, "sm_mhz_used": sm_mhz,
            "note": "floor = 12.2 MUFU (ex2, rcp, sqrt per pixel, 4 pixels per lane) x 8 issue cycles on the 4-lane XU pipe"}
    dominant = max(per_step, key=per_step.get)
    dk = kernels.get(dominant, {"achieved_gbs": 0.0, "frac": 0.0})
    roofline = {"kernel": dominant, "bound": "hbm", "achieved": dk.get("achieved_gbs", 0.0), "peak": hbm_peak, "unit": "GB/s",
                "frac": dk.get("frac", 0.0), "traffic": dk.get("traffic"), "peak_source": peak_src,
                "onchip": dk.get("onchip"),
                "note": "the per-proposal kernels re-read L2-resident fields: their HBM fraction is << 1% by construction and "
                        "`onchip` is the roofline that binds the dominant kernel (XU pipe); the HBM-streaming kernels "
                        "(unmore_sat_build_fields, mask pack in extras) carry the HBM fractions — see `kernels`",
                "proposal_rounds_per_step": work.get("proposal_rounds"),
                "proposal_rounds_per_sec": (work.get("proposal_rounds", 0) / (per_step.get("unmore_boundary_refine", 1e9) / 1e3))}
    if producer is not None:
        per_step["producer_forward"] = producer_ms / args.steps

    # ---- end to end through the public API with HOST buffers (pinned), copies inside the timed region.
    # Result read back per step = the reference's output: the detection rows AND the COCO run lengths of every
    # kept mask (object_scoring.py:257-268 `segmentation`), produced on the device by unmore_mask_rle_counts.
    e2e = None
    if not args.no_e2e and not producer_cfg:
        import psutil
        pool = n_img
        avail = psutil.virtual_memory().available
        while pool > chunk and pool * 4 * px * 4 * world > avail // 4:   # every rank pins its own pool
            pool //= 2
        pool = max(chunk, (pool // chunk) * chunk)
        h_fields = torch.empty((pool, 4, Hc, Wc), dtype=torch.float32).pin_memory()
        for c0 in range(0, pool, chunk):
            n = min(chunk, n_img - c0)
            if n > 0:
                h_fields[c0:c0 + n].copy_(fields[c0:c0 + n])
        h_props = torch.from_numpy(props_np).pin_memory()
        torch.cuda.synchronize()
        copy_stream = torch.cuda.Stream()
        side_stream = torch.cuda.Stream()
        bufs = [(torch.empty((chunk, 4, Hc, Wc), dtype=torch.float32, device=dev),
                 torch.empty((chunk, n_prop, 4), dtype=torch.float64, device=dev)) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]
        MAX_RUNS = 2048   # a mask over all 640 columns has up to 1281 runs
        h2d = d2h = d2h_rows = 0
        n_rle = rle_off = rle_moff = 0
        from concurrent.futures import ThreadPoolExecutor
        reader = ThreadPoolExecutor(max_workers=1)   # the RLE read-back of chunk j overlaps the launches of chunk j + 1
        rle_len = torch.empty((max(1024, 12 * n_img),), dtype=torch.int32).pin_memory()   # ~7 kept masks per image here
        rle_arena = torch.empty((rle_len.shape[0] * 512,), dtype=torch.int32).pin_memory()   # ~200 runs per mask here

        def e2e_step(with_rle=True):
            nonlocal h2d, d2h, d2h_rows, n_rle, rle_off, rle_moff
            h2d = d2h = d2h_rows = n_rle = rle_off = rle_moff = 0
            rows = ops.detection_rows(max_rows, dev)
            host_rle = []
            # a short first chunk: its host -> device copy is the only one nothing overlaps
            chunks, c0 = [], 0
            while c0 < n_img:
                c1 = min(n_img, c0 + (max(1, chunk // 4) if c0 == 0 else chunk))
                chunks.append((c0, c1))
                c0 = c1

            def issue(j):
                c0, c1 = chunks[j]
                fb, pb = bufs[j % 2]
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(freed[j % 2])
                    p0 = min(c0 % pool, pool - (c1 - c0))   # the host pool may hold fewer images than the step (they repeat)
                    fb[: c1 - c0].copy_(h_fields[p0:p0 + (c1 - c0)], non_blocking=True)
                    pb[: c1 - c0].copy_(h_props[c0:c1], non_blocking=True)
                    ready[j % 2].record(copy_stream)
                return (c1 - c0) * (4 * px * 4 + n_prop * 32)

            rle_stream = side_stream
            done_ev = [torch.cuda.Event() for _ in chunks]
            futures = []

            def read_back(j, r):
                """COCO run lengths of the kept masks of chunk j (NMS order) on the SIDE stream, then their device -> host
                read into the pinned arena.  Runs on the reader thread: the thread that launches the chunks never waits for it."""
                nonlocal d2h, n_rle, rle_off, rle_moff
                torch.cuda.set_device(dev)
                with torch.cuda.stream(rle_stream):
                    rle_stream.wait_event(done_ev[j])
                    B, cap = r["keep"].shape
                    valid = torch.arange(cap, device=dev)[None, :] < r["keep_counts"][:, None]
                    flat = (torch.arange(B, device=dev)[:, None] * cap + r["keep"].clamp_min(0))[valid]
                    km = r["masks"].view(B * cap, Hc, -1).index_select(0, flat)
                    cnt, nr = ops.mask_rle_counts(km, Wc, MAX_RUNS)
                    K = int(nr.numel())
                    n_max = int(nr.max().item()) if K else 0
                    if n_max > MAX_RUNS:   # a ragged mask with more runs than the buffer holds: once more, large enough
                        cnt, nr = ops.mask_rle_counts(km, Wc, 1 << (n_max - 1).bit_length())
                    # only the run lengths that exist travel: [sum of n_runs] int32 + the K lengths
                    used = torch.arange(cnt.shape[1], device=dev)[None, :] < nr[:, None]
                    flat_counts = cnt[used]
                    T = int(flat_counts.numel())
                    if rle_off + T <= rle_arena.shape[0] and rle_moff + K <= rle_len.shape[0]:
                        hc, hn = rle_arena[rle_off:rle_off + T], rle_len[rle_moff:rle_moff + K]
                        hc.copy_(flat_counts, non_blocking=True)
                        hn.copy_(nr, non_blocking=True)
                        rle_off += T
                        rle_moff += K
                        rle_stream.synchronize()
                    else:   # more than the arena was sized for: pageable copies
                        hc, hn = flat_counts.cpu(), nr.cpu()
                    for t_ in (r["keep"], r["keep_counts"], r["masks"]):
                        t_.record_stream(rle_stream)
                d2h += hc.numel() * 4 + hn.numel() * 4
                n_rle += K
                host_rle.append((hc, hn))

            h2d += issue(0)
            for j, (c0, c1) in enumerate(chunks):
                if j + 1 < len(chunks):
                    h2d += issue(j + 1)
                torch.cuda.current_stream().wait_event(ready[j % 2])
                fb, pb = bufs[j % 2]
                r = pipe.run_chunk(fb[: c1 - c0], pb[: c1 - c0])
                ops.pack_detections(image_ids[c0:c1], r["bbox"], r["out"], r["keep_counts"], rows)
                freed[j % 2].record(torch.cuda.current_stream())
                done_ev[j].record(torch.cuda.current_stream())
                if with_rle:
                    futures.append(reader.submit(read_back, j, r))
            for f in futures:
                f.result()
            g2 = gather_rows(rows)
            m2, t2 = merge_rows(g2)
            hr = m2[: int(t2.item())].cpu()          # device -> host read of the detection rows
            d2h += hr.numel() * 8
            d2h_rows = hr.numel() * 8
            return hr, host_rle

        freed[0].record(); freed[1].record()
        e2e_step()
        barrier()
        reps = args.steps   # timed end-to-end steps, like the device-resident ones
        t0 = time.perf_counter()
        for _ in range(reps):
            last = e2e_step()
        barrier()
        dt = (time.perf_counter() - t0) / reps
        d2h_full, n_rle_full = d2h, n_rle
        # what was read back is a complete result: every mask's run lengths cover the image, one mask per detection row
        def _complete(hc, hn):
            n = hn.numpy().astype(np.int64)
            if n.size == 0:
                return True
            starts = np.concatenate([[0], np.cumsum(n)[:-1]])
            return int(n.sum()) == hc.numel() and bool((np.add.reduceat(hc.numpy().astype(np.int64), starts) == Hc * Wc).all())
        rle_ok = all(_complete(hc, hn) for hc, hn in last[1])
        rle_ok = rle_ok and sum(int(hn.numel()) for _, hn in last[1]) == (int(last[0].shape[0]) if world == 1 else n_rle)
        e2e_step(with_rle=False)
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            e2e_step(with_rle=False)
        barrier()
        dt_rows = (time.perf_counter() - t0) / reps
        if world > 1:
            t = torch.tensor([dt, dt_rows], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt, dt_rows = float(t[0].item()), float(t[1].item())
        e2e = {"value": n_global / dt, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_full,
               "host_pool_images": pool, "ms_per_step": dt * 1e3, "steps": reps,
               "result": "detection rows (image_id, x, y, w, h, score) fp64 + COCO RLE run lengths of every kept mask "
                         "(unmore_mask_rle_counts; the existing run lengths of each mask + its length, int32)",
               "masks_rle_per_step": n_rle_full, "rle_complete": bool(rle_ok),
               "rows_only": {"value": n_global / dt_rows, "ms_per_step": dt_rows * 1e3, "d2h_bytes_per_step": d2h_rows}}
        reader.shutdown()
        del h_fields, bufs, rle_arena, rle_len

    # ---- configs[2] side measurement (outside the step): mask bit-pack (HBM streaming) and the
    # mask-IoU / box NMS sweep at 1k - 16k masks per image, 480x640
    extras = {}
    if rank == 0 and not args.no_extras and not producer_cfg:
        sat_buf = None
        torch.cuda.empty_cache()

        def timed(fn, reps=5):
            fn(); torch.cuda.synchronize()
            best = 1e30
            for _ in range(reps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); fn(); b.record(); torch.cuda.synchronize()
                best = min(best, a.elapsed_time(b))
            return best

        g_ = torch.Generator(device=dev).manual_seed(0)
        ys = torch.arange(H, device=dev).view(1, H, 1); xs = torch.arange(W, device=dev).view(1, 1, W)
        sweep = []
        for K in (1024, 4096, 16384):
            dense = torch.empty((K, H, W), dtype=torch.uint8, device=dev)
            cx = torch.rand(K, generator=g_, device=dev) * W; cy = torch.rand(K, generator=g_, device=dev) * H
            rx = 20 + torch.rand(K, generator=g_, device=dev) * 120; ry = 20 + torch.rand(K, generator=g_, device=dev) * 120
            for k0 in range(0, K, 256):
                sl = slice(k0, k0 + 256)
                dense[sl] = ((((ys - cy[sl].view(-1, 1, 1)) / ry[sl].view(-1, 1, 1)) ** 2 +
                              ((xs - cx[sl].view(-1, 1, 1)) / rx[sl].view(-1, 1, 1)) ** 2) < 1).to(torch.uint8)
            msc = torch.rand(K, generator=g_, device=dev)
            t_pack = timed(lambda: ops.mask_pack(dense))
            packed = ops.mask_pack(dense)
            del dense
            pack_bytes = K * H * W + K * H * ((W + 31) // 32) * 4
            stats_ = ops.mask_stats(packed, W)
            t_nms = timed(lambda: ops.mask_nms(packed, W, msc, 0.5, stats=stats_), reps=3)
            kept = int(ops.mask_nms(packed, W, msc, 0.5, stats=stats_).numel())
            boxes = stats_[1].to(torch.float32)
            t_box = timed(lambda: ops.box_nms_matrix(boxes, msc, 0.5), reps=3)
            sweep.append({"masks": K, "pack_ms": t_pack, "pack_gbs": pack_bytes / t_pack / 1e6,
                          "pack_frac_of_hbm_peak": pack_bytes / t_pack / 1e6 / hbm_peak,
                          "mask_nms_ms": t_nms, "mask_nms_kept": kept, "box_nms_matrix_ms": t_box})
            del packed
        # CPU side of the sweep: the dense-mask greedy restatement (oracle, north-star op C) on 256 masks
        cpu_nms = None
        if world == 1 and not args.no_cpu_baseline:
            from oracle import oracle as O
            Kc = 256
            dense = torch.empty((Kc, H, W), dtype=torch.uint8, device=dev)
            cx = torch.rand(Kc, generator=g_, device=dev) * W; cy = torch.rand(Kc, generator=g_, device=dev) * H
            rx = 20 + torch.rand(Kc, generator=g_, device=dev) * 120; ry = 20 + torch.rand(Kc, generator=g_, device=dev) * 120
            dense[:] = ((((ys - cy.view(-1, 1, 1)) / ry.view(-1, 1, 1)) ** 2 + ((xs - cx.view(-1, 1, 1)) / rx.view(-1, 1, 1)) ** 2) < 1).to(torch.uint8)
            msc = torch.rand(Kc, generator=g_, device=dev)
            packed = ops.mask_pack(dense)
            t_gpu = timed(lambda: ops.mask_nms(packed, W, msc, 0.5), reps=3)
            keep_gpu = ops.mask_nms(packed, W, msc, 0.5).cpu().numpy()
            dn, sn = dense.cpu().numpy(), msc.cpu().numpy()
            t0 = time.perf_counter()
            keep_cpu = O.mask_nms_dense(dn, sn, 0.5)
            t_cpu = (time.perf_counter() - t0) * 1e3
            cpu_nms = {"masks": Kc, "cpu_dense_ms": t_cpu, "gpu_ms_incl_stats": t_gpu, "keep_sets_equal": bool(np.array_equal(keep_gpu, keep_cpu)),
                       "kind": "port (numpy, 1 core)"}
            del dense, packed
        extras = {"cpu_mask_nms": cpu_nms, "nms_sweep_480x640": sweep,
                  "note": "configs[2]; mask_nms = rank sort + 64-wide IoU bit-matrix (popc on packed masks) + greedy scan"}

    cpu_baseline = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not producer_cfg:
        cpu_baseline, _, ores = cpu_sample(args.cpu_sample_proposals, n_prop, keep_result=True)
        parity = parity_sample(pipe, dev, ores)
        extras["cpu_config0"] = cpu_config0()

    if rank == 0:
        workload = (f"configs[4]: random-init DPT-L objectness net ({args.producer_dtype}, PyTorch producer) -> CUDA reasoning, "
                    f"{Hc}x{Wc}, {n_prop} anchors/image" if producer_cfg else WORKLOAD)
        line = {"metric": "object_reasoning_images_per_sec", "value": images_per_s, "unit": "images/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload, "images_per_rank": n_img, "images_total": n_global, "proposals_per_image": n_prop,
                           "field_hw": [Hc, Wc], "chunk_images": chunk, "n_round": 50, "resize": "bilinear, antialias=False",
                           "sharding": ("image i -> rank i mod G (strong: fixed total)" if args.scaling == "strong"
                                        else "rank r owns images [r*n, (r+1)*n) (weak: fixed per rank)"),
                           "l2": f"inputs ({n_img * 4 * px * 4 / 1e9:.1f} GB of fields per rank) exceed the 126 MB L2; no flush needed",
                           "input_generation_s": round(t_gen, 1)},
                "proposals_per_sec": images_per_s * n_prop, "detections": int(result_rows.shape[0]),
                "detections_sha256": digest, "gather_equal": gather_equal,
                "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "kernels": kernels,
                "stage_ms_per_step": per_step, "e2e": e2e, "cpu_baseline": cpu_baseline, "parity_sample": parity, "extras": extras}
        if producer_cfg:
            line["config"]["producer"] = {"dtype": args.producer_dtype, "batch": args.producer_batch,
                                          "weights": "random-init, head output layers rescaled (FieldProducer.calibrate_random_init)"}
            line["dtype"] = "f32 reasoning; producer " + args.producer_dtype
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
