"""The fused kernels of the second resize mode (antialias=True): antialiased existence and boundary refine resample
every crop inside the kernel.  They must equal, bit for bit, the tile path they replace: antialiased tiles from
``crop_resize(..., antialias=True)`` fed to the tile stages (``tile_means``, ``boundary_round_from_tiles``, the host
round loop ``Object_Discovery._boundary_reasoning_tiles``, ``center_reasoning_from_tiles``)."""
import ctypes

import numpy as np
import pytest
import torch

from unmore_b200 import synth

H, W = 480, 640
N = 4096


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int64) if t.dtype == torch.float64 else t


def _assert_bit_equal(a, b, what=""):
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert torch.equal(_bits(a.contiguous()), _bits(b.contiguous())), what


def _tile_scores(ops, fields, boxes, counts=None):
    tiles = ops.crop_resize(fields, boxes, [ops.DEFAULT_CHANNELS.exist], counts, antialias=True)
    return ops.tile_means(tiles.reshape(-1, 1, 128, 128)[:, 0]).reshape(boxes.shape[:2])


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def bench_image(dev):
    return synth.make_fields(0, H, W).to(dev), torch.from_numpy(synth.make_proposals(0, N, H, W)).to(dev)


@pytest.fixture(scope="module")
def oda(dev):
    from unmore_b200.object_reasoning import Object_Discovery, default_args
    return Object_Discovery(default_args(antialias=True), device=dev)


def _extreme_windows(dev):
    """A 1024x1024 field and the windows of the stand-alone resize's extreme-window test: 1x1, 2x3, 1-px strips,
    up-sampled windows, and windows whose 16-17 taps per axis exceed the kernels' tables (the fallback path)."""
    g = torch.Generator().manual_seed(11)
    f = torch.randn((1, 4, 1024, 1024), generator=g)
    boxes = [[10.0, 20.0, 11.0, 21.0], [100.2, 200.7, 101.9, 203.1], [5.0, 5.0, 6.0, 400.0], [5.0, 700.0, 900.0, 701.0],
             [12.3, 7.9, 1011.5, 1007.2], [0.0, 0.0, 1024.0, 1024.0], [500.0, 500.0, 628.0, 628.0], [40.5, 60.2, 97.0, 90.9],
             [0.0, 0.0, 700.0, 300.0], [300.0, 10.0, 400.0, 1000.0], [3.0, 3.0, 3.0, 9.0]]
    return f.to(dev), torch.tensor(boxes, dtype=torch.float64, device=dev)[None].contiguous()


# ---- existence -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_existence_benchmark_image_and_its_split_lists(bench_image, oda):
    from unmore_b200 import ops
    f, props = bench_image
    fields, boxes = f[None].contiguous(), props[None].contiguous()
    got = ops.existence_scores(fields, boxes, antialias=True)
    _assert_bit_equal(got, _tile_scores(ops, fields, boxes), "benchmark proposals")
    assert not torch.equal(got, ops.existence_scores(fields, boxes))   # the modes differ
    p1 = props[got[0] >= 0.1]
    split = oda.center_reasoning(f, p1)["splited_new_proposals"]
    assert len(split) > 0
    split = split[None].contiguous()
    _assert_bit_equal(ops.existence_scores(fields, split, antialias=True), _tile_scores(ops, fields, split), "splits")


@pytest.mark.gpu
def test_existence_fp32_ragged_counts_and_empty_image(dev):
    from unmore_b200 import ops
    fields = torch.stack([synth.make_fields(i, H, W) for i in (1, 2, 3)]).to(dev)
    boxes = torch.stack([torch.from_numpy(synth.make_proposals(i, 700, H, W)) for i in (1, 2, 3)]).to(dev, torch.float32)
    counts = torch.tensor([512, 0, 700], dtype=torch.int32, device=dev)
    got = ops.existence_scores(fields, boxes.contiguous(), counts, antialias=True)
    ref = _tile_scores(ops, fields, boxes.contiguous(), counts)
    for b, n in enumerate(counts.tolist()):
        _assert_bit_equal(got[b, :n], ref[b, :n], f"image {b}")
        assert float(got[b, n:].abs().sum()) == 0.0


@pytest.mark.gpu
def test_existence_extreme_windows_and_tap_fallback(dev):
    from unmore_b200 import ops
    f, boxes = _extreme_windows(dev)
    _assert_bit_equal(ops.existence_scores(f, boxes, antialias=True), _tile_scores(ops, f, boxes), "extreme windows")


@pytest.mark.gpu
def test_existence_other_field_width(dev):
    from unmore_b200 import ops
    h, w = 300, 517
    f = torch.stack([synth.make_fields(i, h, w) for i in (4, 5)]).to(dev)
    boxes = torch.stack([torch.from_numpy(synth.make_proposals(i, 600, h, w)) for i in (4, 5)]).to(dev).contiguous()
    _assert_bit_equal(ops.existence_scores(f, boxes, antialias=True), _tile_scores(ops, f, boxes), "517 px wide")


# ---- one refine round ------------------------------------------------------------------------------------------
def _one_round(ops, fields, boxes):
    out, lab, _ = ops.boundary_refine(fields, boxes, n_round=1, apply_small_filter=False, early_exit=False, antialias=True)
    tiles = ops.crop_resize(fields, boxes, [ops.DEFAULT_CHANNELS.sdf], antialias=True)
    ref_out, ref_lab = ops.boundary_round_from_tiles(tiles.reshape(-1, 128, 128), boxes.reshape(-1, 4),
                                                     fields.shape[-2], fields.shape[-1])
    _assert_bit_equal(out.reshape(-1, 4), ref_out, "boxes")
    _assert_bit_equal(lab.reshape(-1), ref_lab, "labels")
    return lab


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_one_round_equals_tile_round(bench_image, dev, dtype):
    from unmore_b200 import ops
    f, props = bench_image
    lab = _one_round(ops, f[None].contiguous(), props.to(dtype)[None].contiguous())
    assert len(torch.unique(lab)) >= 2
    fx, bx = _extreme_windows(dev)
    _one_round(ops, fx, bx.to(dtype).contiguous())


# ---- the 50-round loop ---------------------------------------------------------------------------------------
def _fused_loop(ops, oda, f, boxes, early_exit=True):
    a = oda.args
    out, lab, rounds = ops.boundary_refine(f[None].contiguous(), boxes[None].contiguous(), n_round=a.n_round,
                                           apply_small_filter=True, early_exit=early_exit,
                                           proposal_area_thres=a.proposal_area_thres, max_sdf_thres=a.max_sdf_thres,
                                           max_shrink_threshold=a.max_shrink_threshold, delta_ratio=a.delta_ratio,
                                           antialias=True)
    keep = lab[0] > -2
    return out[0][keep], lab[0][keep], rounds


@pytest.mark.gpu
@pytest.mark.parametrize("index", [0, 1])
def test_full_loop_equals_host_tile_loop(oda, dev, index):
    from unmore_b200 import ops
    f = synth.make_fields(index, H, W).to(dev)
    boxes = torch.from_numpy(synth.make_proposals(index, N, H, W)).to(dev)
    ref = oda._boundary_reasoning_tiles(f[None].contiguous(), boxes)
    runs = [_fused_loop(ops, oda, f, boxes, early_exit=e) for e in (True, False)]
    assert int(runs[0][2].sum()) < int(runs[1][2].sum())    # early exit does skip rounds
    for out, lab, _ in runs:
        _assert_bit_equal(out, ref["proposals"], "proposals")
        _assert_bit_equal(lab, ref["labels"], "labels")
    assert int((ref["labels"] == 1).sum()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("early_exit", [True, False])
def test_window_cache_sharing_is_invisible(bench_image, early_exit):
    """All proposals in one image (the window cache shared between them) against one proposal per image."""
    from unmore_b200 import ops
    f, props = bench_image
    plane = f[:1]
    kw = dict(ch=ops.Channels(sdf=0), early_exit=early_exit, antialias=True)
    shared = ops.boundary_refine(plane[None].contiguous(), props[None].contiguous(), **kw)
    chunk = 512
    fields = plane[None].expand(chunk, -1, -1, -1).contiguous()
    parts = [ops.boundary_refine(fields[: len(b)], b[:, None].contiguous(), **kw) for b in props.split(chunk)]
    for i, what in enumerate(("boxes", "labels", "rounds")):
        _assert_bit_equal(shared[i][0], torch.cat([p[i][:, 0] for p in parts]), what)


# ---- batched discovery -----------------------------------------------------------------------------------------
def _tile_discovery(ops, oda, f, boxes, cc_on):
    """main_object_discovery's loop body for one image composed from the tile ops (antialiased tiles throughout)."""
    a, ch = oda.args, ops.DEFAULT_CHANNELS
    fields = f[None].contiguous()
    empty = np.zeros((0, 4), np.float32)
    thr = a.class_score_thres

    def exist(b):
        return _tile_scores(ops, fields, b[None].contiguous())[0]

    def center(b, cc):
        tiles = ops.crop_resize(fields, b[None].contiguous(), [ch.sdf, ch.center_row, ch.center_col], antialias=True)
        return ops.center_reasoning_from_tiles(tiles, H, W, b[None].contiguous(), thr=a.center_score_max_thres, analyze_cc=cc)

    p = boxes[exist(boxes) >= thr]
    if len(p) == 0:
        return empty
    _, am, sp, cc = center(p, cc_on)
    fail = am[0] >= 0
    split = sp[0][fail].reshape(-1, 4)
    if cc_on:
        counts, cboxes, overflow = cc
        if int(overflow.item()):
            extra = oda._cc_boxes_with_overflow(fields, p[None], torch.nonzero(~fail).flatten().tolist(), counts[0],
                                                cboxes[0], H, W)
            split = torch.cat((split, torch.as_tensor(extra, device=f.device)))
        else:
            valid = torch.arange(cboxes.shape[2], device=f.device)[None, :] < counts[0][:, None].to(torch.long)
            split = torch.cat((split, cboxes[0][valid]))
    p = p[~fail]
    if len(split):
        split = split[exist(split) >= thr]
    if len(split):
        _, am2, _, _ = center(split, False)
        p = torch.cat((p, split[am2[0] < 0]))
    if len(p) == 0:
        return empty
    br = oda._boundary_reasoning_tiles(fields, p)
    if len(br["proposals"]) == 0:
        return empty
    final = br["proposals"][br["labels"] == 1]
    if len(final) == 0:
        return empty
    _, kc, kb = ops.box_nms(final.to(torch.float32)[None].contiguous(), None, None, iou_threshold=0.5)
    return kb[0, : int(kc[0])].cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("cc_on", [False, True])
def test_discover_batch_equals_tile_composition(dev, monkeypatch, cc_on):
    from unmore_b200 import ops
    from unmore_b200.object_reasoning import Object_Discovery, default_args
    ids, counts = [0, 1, 2, 3], [N, 2900, 1, 3333]
    fields = torch.stack([synth.make_fields(i, H, W) for i in ids]).to(dev)
    props = torch.stack([torch.from_numpy(synth.make_proposals(i, N, H, W)) for i in ids]).to(dev)
    cnt = torch.tensor(counts, dtype=torch.int32, device=dev)
    # slices of 613 proposals in the center stage: the slice boundaries cut through every list
    per_box = 3 * (128 * 128 + H * 128) * 4 * len(ids)
    monkeypatch.setattr(ops, "CENTER_AA_SLICE_BYTES", per_box * 613)
    od = Object_Discovery(default_args(antialias=True, analyze_cc=cc_on), device=dev)
    st = {}
    kb, kc = od.discover_batch(fields, props, cnt, stats=st)
    assert int(st["pass1"].max()) > 613
    for b, n in enumerate(counts):
        ref = _tile_discovery(ops, od, fields[b], props[b, :n], cc_on)
        got = kb[b, : int(kc[b])].cpu().numpy()
        assert got.shape == ref.shape and np.array_equal(got, ref), (b, got.shape, ref.shape)
    assert int(kc.sum()) > 0


@pytest.mark.gpu
def test_pipeline_equals_per_image_mirror_path(dev):
    import argparse
    from unmore_b200.object_reasoning import default_args
    from unmore_b200.object_scoring import Object_Scoring, unpack_masks
    from unmore_b200.pipeline import ReasoningPipeline
    ids = [5, 6, 7, 8]
    fields = torch.stack([synth.make_fields(i, H, W) for i in ids]).to(dev)
    props = torch.stack([torch.from_numpy(synth.make_proposals(i, 1024, H, W)) for i in ids]).to(dev)
    pipe = ReasoningPipeline(dev, default_args(antialias=True))
    r = pipe.run_chunk(fields, props)
    sc = Object_Scoring(argparse.Namespace(antialias=True), device=dev)
    n_ann = 0
    for b in range(len(ids)):
        det = pipe.discovery.discover_image(fields[b], props[b])
        k = int(r["box_counts"][b])
        assert np.array_equal(r["boxes"][b, :k].cpu().numpy(), det)
        anns = sc.score_image(fields[b], det.astype(np.float64).tolist()) if len(det) else []
        kk = int(r["keep_counts"][b])
        assert kk == len(anns)
        n_ann += kk
        if kk:
            assert np.array_equal(r["bbox"][b, :kk].cpu().numpy(), np.array([a["bbox"] for a in anns], np.float32))
            assert np.array_equal(r["out"][b, :kk, 0].cpu().numpy(), np.array([a["score"] for a in anns]))
            keep = r["keep"][b, :kk].long()
            assert np.array_equal(unpack_masks(r["masks"][b][keep], W), np.stack([a["segmentation"]["mask"] for a in anns]))
    assert n_ann > 0


# ---- C ABI -------------------------------------------------------------------------------------------------------
def test_aa_entry_points_reject_bad_arguments():
    """The antialiased entry points validate their arguments like their antialias=False counterparts (no GPU
    needed: the checks run before anything is launched)."""
    from unmore_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(0x1000)
    for name in ("unmore_existence_scores", "unmore_existence_scores_aa"):
        fn = getattr(lib, name)
        assert fn(None, 1, 4, 8, 8, 3, fake, 1, None, 4, fake, fake, None) == -1            # no fields
        assert fn(fake, 1, 4, 8, 8, 4, fake, 1, None, 4, fake, fake, None) == -1            # channel out of range
        assert fn(fake, 1, 4, 8, 8, 3, None, 1, None, 4, fake, fake, None) == -1            # no boxes
        assert fn(fake, 1, 4, 8, 8, 3, fake, 1, None, -1, fake, fake, None) == -1           # negative capacity
        assert fn(fake, 1, 4, 8, 8, 3, fake, 1, None, 4, fake, None, None) == -1            # no workspace
        assert name.encode() in lib.unmore_last_error()
    for name in ("unmore_boundary_refine", "unmore_boundary_refine_aa"):
        fn = getattr(lib, name)
        ok = [fake, 1, 4, 8, 8, 0, fake, 1, None, 4, 50, 1, 1, 50.0, 0.5, 16.0, 0.5, fake, fake, None, fake, None]
        for i, bad in ((0, None), (5, 4), (6, None), (9, -1), (10, 0), (17, None), (18, None), (20, None)):
            args = list(ok)
            args[i] = bad
            assert fn(*args) == -1, (name, i)
            assert i == 0 or name.encode() in lib.unmore_last_error()
