"""TEST INFRASTRUCTURE ONLY — generates tests/golden/*.npz by executing the UNMODIFIED
reference (/root/reference) on CPU through oracle/ref_harness.py.

Run in the build container (the reference does not exist on the GPU box):

    python -m oracle.gen_golden            # writes tests/golden/
    python -m oracle.gen_golden signatures # only tests/golden/reference_signatures.json

Everything stored is an output of reference code (or a library op the reference calls
at the cited line), never of this repo's oracle or CUDA path.
"""
from __future__ import annotations

import io
import json
import os
import runpy
import sys
import tempfile
import time
from contextlib import redirect_stdout

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_harness as rh  # noqa: E402
from unmore_b200 import synth  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def _quiet(fn, *a, **k):
    with redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def _ast_params(path, class_name=None):
    """{function name: [positional parameter names]} of a module (or one class of it), read with ``ast``."""
    import ast
    with open(path) as f:
        tree = ast.parse(f.read())
    body = tree.body
    if class_name is not None:
        body = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == class_name).body
    return {n.name: [x.arg for x in n.args.posonlyargs + n.args.args] for n in body if isinstance(n, ast.FunctionDef)}


def reference_signatures(root):
    """Parameter lists of the reference's Object_Discovery / Object_Scoring methods, batch_erode and
    convert_pred_annotations_to_training_format (what tests/test_cpu_host.py pins the mirrors against)."""
    misc = _ast_params(os.path.join(root, "utils", "misc.py"))
    post = _ast_params(os.path.join(root, "post_process.py"))
    return {"Object_Discovery": _ast_params(os.path.join(root, "object_reasoning.py"), "Object_Discovery"),
            "Object_Scoring": _ast_params(os.path.join(root, "object_scoring.py"), "Object_Scoring"),
            "functions": {"batch_erode": misc["batch_erode"],
                          "convert_pred_annotations_to_training_format": post["convert_pred_annotations_to_training_format"]}}


def gen_signatures():
    with open(os.path.join(GOLD, "reference_signatures.json"), "w") as f:
        json.dump(reference_signatures(rh.REFERENCE_ROOT), f, indent=1)
    print("reference_signatures.json written")


def gen_units(od):
    """Unit-level vectors for the static / free functions."""
    import torchvision
    from utils.misc import batch_erode

    g = torch.Generator().manual_seed(1234)
    out = {}
    # a2 crop+resize through the reference's own Resize call pattern (object_reasoning.py:404-408)
    img = synth.make_fields(3)
    boxes = np.array([[0, 0, 32, 32], [10.3, 20.7, 200.2, 300.9], [0, 0, 640, 480], [600.5, 400.25, 640, 480],
                      [123.0, 45.0, 131.0, 52.0], [5.5, 5.5, 517.5, 261.5], [300.1, 100.9, 364.1, 228.9]])
    from torchvision import transforms
    import math
    crops = []
    for b in boxes:
        x1, y1, x2, y2 = int(math.floor(b[0])), int(math.floor(b[1])), int(math.ceil(b[2])), int(math.ceil(b[3]))
        resize = transforms.Resize((128, 128), interpolation=torchvision.transforms.InterpolationMode.BILINEAR)
        crops.append(resize(img[:, y1:y2, x1:x2]))
    out["crop_boxes"] = boxes
    out["crop_out"] = torch.stack(crops).numpy()
    # a10 update_bbox_with_boundary_fields on smooth-ish tiles
    tiles = torch.tanh(torch.randn(24, 128, 128, generator=g).cumsum(1).cumsum(2) / 60.0)
    d = od.update_bbox_with_boundary_fields(tiles)
    out["a10_tiles"] = tiles.numpy()
    out["a10_deltas"] = torch.stack(d, dim=1).numpy()
    # a12 post_process_bbox_update: fp64 boxes (round 0) and fp32 boxes (later rounds)
    ob = torch.rand(64, 4, generator=g, dtype=torch.float64) * 300
    ob[:, 2:] += ob[:, :2] + 5
    dl = torch.randn(64, 4, generator=g) * 20
    out["a12_boxes64"] = ob.numpy()
    out["a12_delta"] = dl.numpy()
    out["a12_out64"] = od.post_process_bbox_update(ob, dl).numpy()
    out["a12_out32"] = od.post_process_bbox_update(ob.float(), dl).numpy()
    # a5 batch_erode
    m = (torch.rand(6, 128, 128, generator=g) > 0.02).long()
    m[0, 30:100, 20:90] = 1
    out["a5_masks"] = m.numpy().astype(np.uint8)
    out["a5_out"] = batch_erode(m, kernel_size=9, num_round=3).numpy().astype(np.uint8)
    # a6 anti-center map
    v = torch.randn(4, 2, 128, 128, generator=g)
    out["a6_in"] = v.numpy()
    out["a6_out"] = _quiet(od.center_field_to_anti_center_map, v, 5).numpy()
    # a14 torchvision.ops.nms incl. exact ties in score and threshold-straddling IoUs
    nb = 400
    c = torch.rand(nb, 2, generator=g) * 300
    wh = torch.rand(nb, 2, generator=g) * 120 + 4
    b = torch.cat([c, c + wh], dim=1)
    b[50:60] = b[40:50]  # duplicates
    s = torch.rand(nb, generator=g)
    s[100:200] = 0.5     # tied scores -> index order decides
    out["a14_boxes"] = b.numpy()
    out["a14_scores"] = s.numpy()
    out["a14_keep"] = torchvision.ops.nms(b, s, 0.5).numpy()
    out["a14_keep_allones"] = torchvision.ops.nms(b, torch.ones(nb), 0.5).numpy()
    # a9 filter_small_proposal
    sb = torch.tensor([[0, 0, 10, 5], [0, 0, 10, 5.0001], [3, 3, 3, 50], [0, 0, 7.2, 7.2], [1, 1, 8.1, 8.05]],
                      dtype=torch.float64)
    fo, fl = od.filter_small_proposal(sb, torch.arange(5).float())
    out["a9_in"] = sb.numpy()
    out["a9_keep_index"] = fl.numpy()
    # N2: mask resize with round-half-even (object_scoring.py:206-207)
    masks = (torch.rand(3, 128, 128, generator=g) > 0.5).long()
    yy, xx = torch.meshgrid(torch.arange(128), torch.arange(128), indexing="ij")
    masks[1] = (((yy - 60) ** 2 + (xx - 70) ** 2) < 45 ** 2).long()
    sizes = [(64, 64), (256, 256), (32, 32), (100, 300), (480, 640), (13, 17), (127, 129), (61, 67), (1, 1), (3, 200)]
    out["n2_masks"] = masks.numpy().astype(np.uint8)
    out["n2_sizes"] = np.array(sizes)
    for k, (h, w) in enumerate(sizes):
        rs = transforms.Resize((h, w), interpolation=torchvision.transforms.InterpolationMode.BILINEAR)
        out[f"n2_out_{k}"] = np.stack([rs(masks[i].unsqueeze(0))[0].numpy() for i in range(3)]).astype(np.uint8)
    np.savez_compressed(os.path.join(GOLD, "units.npz"), **out)
    print("units.npz written")


def gen_units_aa(od):
    """Second resize mode (torchvision default antialias=True; run with UNMORE_REF_ANTIALIAS=1): the reference's own
    Resize call pattern on crops and on int masks, its get_prediction_with_proposals tiles, and one round of
    optimize_one_image_single_round on them."""
    import math
    import torchvision
    from torchvision import transforms
    assert os.environ.get("UNMORE_REF_ANTIALIAS") == "1", "run as: UNMORE_REF_ANTIALIAS=1 python -m oracle.gen_golden units_aa"
    g = torch.Generator().manual_seed(4321)
    out = {}
    img = synth.make_fields(3)
    boxes = np.array([[0, 0, 32, 32], [10.3, 20.7, 200.2, 300.9], [0, 0, 640, 480], [600.5, 400.25, 640, 480],
                      [123.0, 45.0, 131.0, 52.0], [5.5, 5.5, 517.5, 261.5], [300.1, 100.9, 364.1, 228.9],
                      [100.0, 50.0, 357.0, 179.0], [17.2, 300.4, 500.9, 460.0]])
    crops = []
    for b in boxes:
        x1, y1, x2, y2 = int(math.floor(b[0])), int(math.floor(b[1])), int(math.ceil(b[2])), int(math.ceil(b[3]))
        resize = transforms.Resize((128, 128), interpolation=torchvision.transforms.InterpolationMode.BILINEAR)
        crops.append(resize(img[:, y1:y2, x1:x2]))
    out["crop_boxes"] = boxes
    out["crop_out"] = torch.stack(crops).numpy()
    sdf, cen = _quiet(od.get_prediction_with_proposals, torch.tensor(boxes), img)
    out["pred_sdf"] = sdf.cpu().numpy()
    out["pred_center"] = cen.cpu().numpy()
    d = od.update_bbox_with_boundary_fields(sdf.cpu())
    out["a10_deltas"] = torch.stack(d, dim=1).numpy()
    r = _quiet(od.optimize_one_image_single_round, img, torch.tensor(boxes), torch.zeros(len(boxes)))
    out["round_boxes"] = r["updated_bboxes"].cpu().numpy()
    out["round_labels"] = r["labels"].cpu().numpy()
    masks = (torch.rand(3, 128, 128, generator=g) > 0.5).long()
    yy, xx = torch.meshgrid(torch.arange(128), torch.arange(128), indexing="ij")
    masks[1] = (((yy - 60) ** 2 + (xx - 70) ** 2) < 45 ** 2).long()
    sizes = [(64, 64), (256, 256), (32, 32), (100, 300), (480, 640), (13, 17), (127, 129), (61, 67), (1, 1), (3, 200)]
    out["n2_masks"] = masks.numpy().astype(np.uint8)
    out["n2_sizes"] = np.array(sizes)
    for k, (h, w) in enumerate(sizes):
        rs = transforms.Resize((h, w), interpolation=torchvision.transforms.InterpolationMode.BILINEAR)
        out[f"n2_out_{k}"] = np.stack([rs(masks[i].unsqueeze(0))[0].numpy() for i in range(3)]).astype(np.uint8)
    np.savez_compressed(os.path.join(GOLD, "units_aa.npz"), **out)
    print("units_aa.npz written")


def gen_scene(od, index, n_prop, tag, n_round=50):
    """Stage-by-stage vectors of main_object_discovery's body on one synthetic image."""
    H, W = 480, 640
    img = synth.make_fields(index, H, W)
    props = torch.tensor(synth.make_proposals(index, n_prop, H, W))
    od.height, od.width = H, W
    od.args.n_round = n_round
    out = {"index": index, "n_prop": n_prop, "n_round": n_round}
    t0 = time.time()
    ex = _quiet(od.existence_checking, img, props)["existence_scores"]
    out["existence_scores"] = ex.numpy()
    p1 = props[ex >= od.args.class_score_thres]
    cr = _quiet(od.center_reasoning, img, p1)
    out["pass1"] = cr["proposals_pass_singularity"].numpy()
    split = cr["splited_new_proposals"]
    out["split"] = split.numpy() if torch.is_tensor(split) else np.zeros((0, 4))
    if torch.is_tensor(split) and len(split):
        ex2 = _quiet(od.existence_checking, img, split)["existence_scores"]
        out["split_existence"] = ex2.numpy()
        split2 = split[ex2 >= od.args.class_score_thres]
        cr2 = _quiet(od.center_reasoning, img, split2)
        out["pass2"] = cr2["proposals_pass_singularity"].numpy()
        refine_in = torch.cat((cr["proposals_pass_singularity"], cr2["proposals_pass_singularity"]), dim=0)
    else:
        out["pass2"] = np.zeros((0, 4))
        refine_in = cr["proposals_pass_singularity"]
    out["refine_in"] = refine_in.numpy()
    print(f"[{tag}] exist+center {time.time()-t0:.1f}s: {len(props)} -> {len(p1)} -> pass {len(out['pass1'])}"
          f" split {len(out['split'])} pass2 {len(out['pass2'])}")

    # boundary reasoning with a per-round recorder around the unmodified method
    trace = []
    orig = od.optimize_one_image_single_round

    def recorder(image, proposals, labels):
        res = orig(image, proposals, labels)
        trace.append((proposals.clone(), res["updated_bboxes"].clone(), res["labels"].clone()))
        return res

    od.optimize_one_image_single_round = recorder
    t0 = time.time()
    try:
        import tqdm as _tq
        br = _quiet(od.boundary_reasoning, img, refine_in, od.args.n_round)
    finally:
        del od.optimize_one_image_single_round
    print(f"[{tag}] boundary_reasoning {time.time()-t0:.1f}s, rounds recorded {len(trace)}")
    out["n_trace"] = len(trace)
    for r, (pin, pout, lab) in enumerate(trace):
        out[f"r{r}_in"] = pin.numpy()
        out[f"r{r}_out"] = pout.numpy()
        out[f"r{r}_labels"] = lab.numpy()
    if len(br["proposals"]):
        fp, fl = br["proposals"], br["labels"]
        out["final_proposals"] = fp.numpy()
        out["final_labels"] = fl.numpy()
        sel = fp[fl == 1]
        import torchvision
        if len(sel):
            keep = torchvision.ops.nms(sel.to(torch.float32), fl[fl == 1], iou_threshold=0.5)
            out["nms_keep"] = keep.numpy()
            out["discovered"] = sel[keep].numpy()
        else:
            out["nms_keep"] = np.zeros((0,), np.int64)
            out["discovered"] = np.zeros((0, 4), np.float32)
    else:
        out["final_proposals"] = np.zeros((0, 4), np.float32)
        out["final_labels"] = np.zeros((0,), np.float32)
        out["nms_keep"] = np.zeros((0,), np.int64)
        out["discovered"] = np.zeros((0, 4), np.float32)
    print(f"[{tag}] discovered {len(out['discovered'])}")

    # scoring of the discovered boxes through main_object_scoring (object_scoring.py:172-272)
    if len(out["discovered"]):
        raw = {str(index): [[float(v) for v in b] for b in out["discovered"]]}
        sc = rh.make_scoring([img], [index], raw)
        t0 = time.time()
        anns = _quiet(rh.run_scoring_capture, sc)
        print(f"[{tag}] scoring {time.time()-t0:.1f}s -> {len(anns)} annotations")
        out["score_bbox"] = np.array([a["bbox"] for a in anns], dtype=np.float32).reshape(-1, 4)
        for key in ("score", "existence_score", "center_score", "boundary_score", "area_score"):
            out["score_" + key] = np.array([a[key] for a in anns], dtype=np.float64)
        masks = np.stack([a["segmentation"]["_mask"] for a in anns]).astype(np.uint8)
        out["score_masks_packed"] = np.packbits(masks.reshape(len(anns), -1), axis=1, bitorder="little")
    np.savez_compressed(os.path.join(GOLD, f"scene_{tag}.npz"), **out)
    print(f"scene_{tag}.npz written")
    return out


def gen_scene_cc(od):
    """center_reasoning and the whole discovery loop body with --analyze_cc (README.md:176)."""
    import torchvision
    H, W = 480, 640
    out = {}
    od.height, od.width = H, W
    od.args.analyze_cc = True
    od.args.n_round = 50
    try:
        done = []
        for index, n_prop in [(0, 512), (4, 300), (8, 200), (12, 300), (16, 300)]:
            if len(done) == 3:
                break
            img = synth.make_fields(index, H, W)
            props = torch.tensor(synth.make_proposals(index, n_prop, H, W))
            ex = _quiet(od.existence_checking, img, props)["existence_scores"]
            p1 = props[ex >= od.args.class_score_thres]
            try:
                cr = _quiet(od.center_reasoning, img, p1)
            except AttributeError as e:  # the reference crashes when nothing fails singularity (:571)
                print(f"[cc] image {index}: reference crashed ({e}); skipped")
                continue
            done.append(index)
            out[f"i{index}_n_prop"] = n_prop
            out[f"i{index}_pass1"] = cr["proposals_pass_singularity"].numpy()
            out[f"i{index}_split"] = cr["splited_new_proposals"].numpy()
            print(f"[cc] image {index}: {len(p1)} -> pass {len(out[f'i{index}_pass1'])}, split+cc {len(out[f'i{index}_split'])}")
        out["indices"] = np.array(done)
        # full loop body for image 0 (the second center_reasoning must see a failing split too)
        index, n_prop = 0, 512
        img = synth.make_fields(index, H, W)
        od.test_dataset = rh._OneImageDataset([img], [index])
        od.result_folder = tempfile.mkdtemp()
        import object_reasoning as ref_or
        captured = {}
        orig_dump = ref_or.json.dump
        orig_gen = od.generate_random_proposal
        ref_or.json.dump = lambda obj, f, *a, **k: (captured.__setitem__("results", obj), f.write("{}"))
        od.generate_random_proposal = lambda height, width: synth.make_proposals(index, n_prop, height, width)
        try:
            _quiet(od.main_object_discovery)
        finally:
            ref_or.json.dump = orig_dump
            del od.generate_random_proposal
        out["disc_index"], out["disc_n_prop"] = index, n_prop
        out["disc"] = np.asarray(captured["results"].get(index, np.zeros((0, 4), np.float32)), np.float32).reshape(-1, 4)
        print(f"[cc] discovery with analyze_cc: {len(out['disc'])} boxes")
    finally:
        od.args.analyze_cc = False
    np.savez_compressed(os.path.join(GOLD, "scene_cc.npz"), **out)
    print("scene_cc.npz written")


def gen_main_loop(od):
    """main_object_discovery (object_reasoning.py:615-665) over a 3-image in-memory dataset,
    results_dict captured at json.dump; then post_process.py's __main__ on scored output."""
    import object_reasoning as ref_or

    ids = [11, 12, 13]
    H, W = 256, 320
    imgs = [synth.make_fields(i, H, W) for i in ids]
    od.test_dataset = rh._OneImageDataset(imgs, ids)
    od.result_folder = tempfile.mkdtemp()
    od.args.n_round = 50
    captured = {}
    orig_dump = ref_or.json.dump

    def dump_capture(obj, f, *a, **k):
        captured["results"] = obj
        f.write("{}")

    ref_or.json.dump = dump_capture
    t0 = time.time()
    try:
        _quiet(od.main_object_discovery)
    finally:
        ref_or.json.dump = orig_dump
    res = captured["results"]
    print(f"[main] main_object_discovery {time.time()-t0:.1f}s: " + ", ".join(f"{k}:{len(v)}" for k, v in res.items()))
    out = {"ids": np.array(ids), "H": H, "W": W}
    for i in ids:
        out[f"disc_{i}"] = np.asarray(res.get(i, np.zeros((0, 4), np.float32)), dtype=np.float32).reshape(-1, 4)
    # scoring over all three images
    raw = {str(i): [[float(v) for v in b] for b in out[f"disc_{i}"]] for i in ids if len(out[f"disc_{i}"])}
    sc = rh.make_scoring(imgs, ids, raw)
    anns = _quiet(rh.run_scoring_capture, sc)
    out["ann_image_id"] = np.array([a["image_id"] for a in anns])
    out["ann_bbox"] = np.array([a["bbox"] for a in anns], dtype=np.float32).reshape(-1, 4)
    for key in ("score", "existence_score", "center_score", "boundary_score", "area_score"):
        out["ann_" + key] = np.array([a[key] for a in anns], dtype=np.float64)
    # post_process.py __main__ (post_process.py:35-77) run as a script on these annotations
    tmp = tempfile.mkdtemp()
    plain = [{k: (float(v) if k.endswith("score") else v) for k, v in a.items() if k != "segmentation"} for a in anns]
    for a, src in zip(plain, anns):
        a["bbox"] = [float(x) for x in src["bbox"]]
        a["segmentation"] = {"size": src["segmentation"]["size"], "counts": ""}
    with open(os.path.join(tmp, "object_discovery_with_scores.json"), "w") as f:
        json.dump(plain, f)
    with open(os.path.join(tmp, "path to coco_cls_agnostic_instances_val2017.json"), "w") as f:
        json.dump({"images": []}, f)
    argv, cwd = sys.argv, os.getcwd()
    try:
        os.chdir(tmp)
        sys.argv = ["post_process.py", "--pred_annotations_path", os.path.join(tmp, "object_discovery_with_scores.json")]
        _quiet(runpy.run_path, os.path.join(rh.REFERENCE_ROOT, "post_process.py"), run_name="__main__")
    finally:
        os.chdir(cwd)
        sys.argv = argv
    with open(os.path.join(tmp, "selected_training_annotations.json")) as f:
        sel = json.load(f)["annotations"]
    out["pp_ids"] = np.array([a["id"] for a in sel], dtype=np.int64)
    out["pp_score"] = np.array([a["score"] for a in sel], dtype=np.float64)
    out["pp_bbox"] = np.array([a["bbox"] for a in sel], dtype=np.float64).reshape(-1, 4)
    out["pp_image_id"] = np.array([a["image_id"] for a in sel], dtype=np.int64)
    print(f"[main] scoring {len(anns)} annotations, post_process kept {len(sel)}")
    np.savez_compressed(os.path.join(GOLD, "main_loop.npz"), **out)
    print("main_loop.npz written")


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 1)
    od = rh.make_discovery(480, 640)
    which = sys.argv[1:] or ["signatures", "units", "scene_a", "scene_b", "main", "scene_cc"]
    if "signatures" in which:
        gen_signatures()
        if which == ["signatures"]:
            return
    if "units" in which:
        gen_units(od)
    if "units_aa" in which:
        gen_units_aa(od)
    if "scene_a" in which:
        gen_scene(od, index=0, n_prop=512, tag="a")          # BASELINE.json configs[0]
    if "scene_b" in which:
        gen_scene(od, index=5, n_prop=160, tag="b", n_round=50)
    if "scene_aa" in which:   # second resize mode: UNMORE_REF_ANTIALIAS=1 python -m oracle.gen_golden scene_aa
        assert os.environ.get("UNMORE_REF_ANTIALIAS") == "1"
        gen_scene(od, index=5, n_prop=160, tag="aa", n_round=50)
    if "main" in which:
        gen_main_loop(od)
    if "scene_cc" in which:
        gen_scene_cc(od)


if __name__ == "__main__":
    main()
