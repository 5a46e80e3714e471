"""Batches of images of different sizes in the second resize mode (antialias=True): a padded field stack with per-image
extents (``ops.pack_fields``, ``image_hw``).  Every op, and discovery / scoring end to end, must give each image of a
padded batch exactly, bit for bit, what the same antialiased op gives that image alone.  The padding is filled with NaN
(and, once, left at zero): a kernel that read it would show it in its results, and since the padding lies inside the
allocation nothing can fault."""
import argparse
import ctypes
import json
import math

import numpy as np
import pytest
import torch

from unmore_b200 import synth

# (pitch, [(h, w, proposals)]): the first batch has the 480x640 pitch of the specialised kernels and an image that fills
# it; the second a pitch no kernel is specialised for.  Both hold an image without proposals and a tiny image.  At most
# 700 proposals per image: the antialiased kernels run at tens of images per second.
BATCHES = [
    ((480, 640), [(480, 640, 700), (300, 400, 500), (200, 360, 0), (37, 53, 64), (411, 517, 600)]),
    ((640, 612), [(640, 480, 700), (612, 612, 600), (200, 360, 300), (9, 14, 16), (333, 97, 0)]),
]
CASES = [(0, math.nan), (1, math.nan), (0, 0.0)]
ALL_CH = [0, 1, 2, 3]


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int64) if t.dtype == torch.float64 else t


def _eq(a, b, what=""):
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert torch.equal(_bits(a.contiguous()), _bits(b.contiguous())), what


def _pad(fields, shapes, value):
    if value != 0.0:
        for i, (h, w) in enumerate(shapes):
            fields[i, :, h:, :] = value
            fields[i, :, :, w:] = value
    return fields


def _batch(k, pad, dev):
    from unmore_b200 import ops
    _, spec = BATCHES[k]
    images = [synth.make_fields(10 * k + i, h, w).to(dev) for i, (h, w, _) in enumerate(spec)]
    props = [torch.from_numpy(synth.make_proposals(10 * k + i, n, h, w)[:n]) for i, (h, w, n) in enumerate(spec)]
    fields, hw = ops.pack_fields(images)
    _pad(fields, [(h, w) for h, w, _ in spec], pad)
    boxes, counts = ops.stack_proposals(props, dev)
    return images, props, fields, hw, boxes, counts


def _alone(im, p, dev):
    return im[None].contiguous(), p[None].to(dev).contiguous()


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


# ---- per op ------------------------------------------------------------------------------------------------------
def _check_ops(images, props, fields, hw, boxes, counts, dev, n_round=50):
    """existence, antialiased tiles, center reasoning (three ways) and refine (early exit on and off) of every image of a
    padded batch against the same op on the image alone."""
    from unmore_b200 import ops
    ex = ops.existence_scores(fields, boxes, counts, antialias=True, image_hw=hw)
    tiles = ops.crop_resize(fields, boxes, ALL_CH, counts, antialias=True, image_hw=hw)
    center = {(s, cc): ops.center_reasoning(fields, boxes, counts, want_splits=s, analyze_cc=cc, antialias=True, image_hw=hw)
              for s, cc in ((True, False), (False, False), (True, True))}
    refine = {ee: ops.boundary_refine(fields, boxes, counts, n_round=n_round, early_exit=ee, antialias=True, image_hw=hw)
              for ee in (True, False)}
    for i, (im, p) in enumerate(zip(images, props)):
        n = p.shape[0]
        if not n:
            continue
        f1, b1 = _alone(im, p, dev)
        _eq(ex[i, :n], ops.existence_scores(f1, b1, antialias=True)[0], ("existence", i))
        _eq(tiles[i, :n], ops.crop_resize(f1, b1, ALL_CH, antialias=True)[0], ("tiles", i))
        for (s, cc), (mv, am, sp, cs) in center.items():
            rmv, ram, rsp, rcs = ops.center_reasoning(f1, b1, want_splits=s, analyze_cc=cc, antialias=True)
            _eq(mv[i, :n], rmv[0], ("center max", s, cc, i))
            _eq(am[i, :n], ram[0], ("center argmax", s, cc, i))
            if s:
                _eq(sp[i, :n], rsp[0], ("splits", cc, i))
            if cc:
                _eq(cs[0][i, :n], rcs[0][0], ("cc counts", i))
                _eq(cs[1][i, :n], rcs[1][0], ("cc boxes", i))
        for ee, (rb, lab, rounds) in refine.items():
            rrb, rlab, rrounds = ops.boundary_refine(f1, b1, n_round=n_round, early_exit=ee, antialias=True)
            _eq(rb[i, :n], rrb[0], ("refine boxes", ee, i))
            _eq(lab[i, :n], rlab[0], ("refine labels", ee, i))
            _eq(rounds[i, :n], rrounds[0], ("refine rounds", ee, i))
    return ex, refine


@pytest.mark.gpu
@pytest.mark.parametrize("k,pad", CASES)
def test_ops_per_image(dev, k, pad):
    images, props, fields, hw, boxes, counts = _batch(k, pad, dev)
    ex, refine = _check_ops(images, props, fields, hw, boxes, counts, dev)
    assert float(ex.sum()) > 0 and int((refine[True][1] == 1).sum()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("k,pad", CASES)
def test_score_batch_per_image(dev, k, pad):
    from unmore_b200.object_scoring import Object_Scoring
    images, props, fields, hw, boxes, counts = _batch(k, pad, dev)
    osc = Object_Scoring(argparse.Namespace(antialias=True), device=dev)
    r = osc.score_batch(fields, boxes, counts, image_hw=hw)
    for i, (im, p) in enumerate(zip(images, props)):
        n, h, w = p.shape[0], im.shape[1], im.shape[2]
        if not n:
            continue
        ref = osc.score_batch(*_alone(im, p, dev))
        for key in ("scores", "tight", "areas"):
            _eq(r[key][i, :n], ref[key][0], (key, i))
        kk = int(ref["keep_counts"][0])
        assert int(r["keep_counts"][i]) == kk
        for key in ("out", "bbox", "selected", "keep"):
            _eq(r[key][i, :kk], ref[key][0, :kk], (key, i))
        wp = (w + 31) // 32
        _eq(r["masks"][i, :n, :h, :wp], ref["masks"][0], ("masks", i))
        outside = r["masks"][i, :n].clone()
        outside[:, :h, :wp] = 0
        assert int(outside.abs().sum()) == 0, ("mask bits outside the image", i)
    assert int(r["areas"].sum()) > 0


# ---- edge windows ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_boxes_past_the_image_edge_snap_to_the_image(dev):
    """Boxes that run past w_i / h_i into the padding: every window must snap to the image's own edge (the refine glue
    and clip too), so each image gets what it gets alone, and nothing reads the NaN padding."""
    from unmore_b200 import ops
    shapes = [(200, 300), (480, 640), (120, 95)]
    images = [synth.make_fields(70 + i, h, w).to(dev) for i, (h, w) in enumerate(shapes)]
    past = lambda h, w: [[w - 80.5, h - 60.2, w + 200.0, h + 150.0], [-10.0, -5.0, w + 20.0, h + 10.0],
                         [w * 0.5, 0.0, 640.0, 480.0], [0.0, h * 0.4, w + 0.5, h - 1.0], [w - 3.0, h - 3.0, w + 40.0, h + 40.0],
                         [w - 0.5, 2.0, w + 90.0, h * 0.7], [5.0, 5.0, w * 0.8, h * 0.8]]
    props = [torch.tensor(past(h, w), dtype=torch.float64) for h, w in shapes]
    fields, hw = ops.pack_fields(images)
    _pad(fields, shapes, math.nan)
    boxes, counts = ops.stack_proposals(props, dev)
    _check_ops(images, props, fields, hw, boxes, counts, dev)


def _extreme_windows():
    """Windows of the stand-alone resize's extreme-window test for a 1024x1024 field: 1x1, 2x3, 1-px strips, up-sampled
    windows, and windows whose 16-17 taps per axis exceed the fused kernels' 12-tap tables (they take aa_dot)."""
    return [[10.0, 20.0, 11.0, 21.0], [100.2, 200.7, 101.9, 203.1], [5.0, 5.0, 6.0, 400.0], [5.0, 700.0, 900.0, 701.0],
            [12.3, 7.9, 1011.5, 1007.2], [0.0, 0.0, 1024.0, 1024.0], [500.0, 500.0, 628.0, 628.0], [40.5, 60.2, 97.0, 90.9],
            [0.0, 0.0, 700.0, 300.0], [300.0, 10.0, 400.0, 1000.0], [3.0, 3.0, 3.0, 9.0]]


@pytest.mark.gpu
@pytest.mark.parametrize("n_round", [1, 50])
def test_extreme_windows_in_a_padded_batch(dev, n_round):
    """The extreme windows on a 1024x1024 field batched with a small image (whose boxes run past its edge)."""
    from unmore_b200 import ops
    g = torch.Generator().manual_seed(11)
    big = torch.randn((4, 1024, 1024), generator=g).to(dev)
    small = synth.make_fields(77, 37, 53).to(dev)
    props = [torch.tensor(_extreme_windows(), dtype=torch.float64),
             torch.tensor([[0.0, 0.0, 53.0, 37.0], [10.0, 5.0, 1000.0, 1000.0], [2.0, 2.0, 3.0, 3.0], [20.0, 30.0, 53.0, 37.0]],
                          dtype=torch.float64)]
    fields, hw = ops.pack_fields([big, small])
    _pad(fields, [(1024, 1024), (37, 53)], math.nan)
    boxes, counts = ops.stack_proposals(props, dev)
    _check_ops([big, small], props, fields, hw, boxes, counts, dev, n_round=n_round)


# ---- end to end --------------------------------------------------------------------------------------------------
def _oda(dev, **over):
    from unmore_b200.object_reasoning import Object_Discovery, default_args
    return Object_Discovery(default_args(antialias=True, **over), device=dev)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 1])
@pytest.mark.parametrize("cc_on", [False, True])
def test_discover_batch_per_image(dev, k, cc_on):
    images, props, fields, hw, boxes, counts = _batch(k, math.nan, dev)
    od = _oda(dev, analyze_cc=cc_on)
    kb, kc = od.discover_batch(fields, boxes, counts, image_hw=hw)
    for i, (im, p) in enumerate(zip(images, props)):
        ref = od.discover_image(im, p.numpy()) if p.shape[0] else np.zeros((0, 4), np.float32)
        got = kb[i, : int(kc[i])].cpu().numpy()
        assert got.shape == ref.shape and np.array_equal(got, ref), (i, got.shape, ref.shape)
    assert int(kc.sum()) > 0


def _speckled(h, w, dev):
    """A field whose union mask is a lattice of isolated dots: every proposal over it passes the center test with more
    connected components than the device buffer holds, so --analyze_cc takes the host re-labelling path."""
    f = torch.full((4, h, w), -4.0)
    f[0, 2::6, 2::6] = 4.0
    f[1:3] = 0.0
    f[3] = 1.0
    return f.to(dev)


@pytest.mark.gpu
def test_discover_batch_cc_overflow_per_image(dev):
    from unmore_b200 import ops
    shapes = [(100, 90), (120, 150), (64, 70)]
    images = [_speckled(h, w, dev) for h, w in shapes]
    props = [torch.tensor([[5.0, 5.0, 60.0, 55.0], [10.0, 20.0, 80.0, 60.0]], dtype=torch.float64)[: 2 - (i == 2)]
             for i in range(len(shapes))]
    fields, hw = ops.pack_fields(images)
    _pad(fields, shapes, math.nan)
    boxes, counts = ops.stack_proposals(props, dev)
    cc = ops.center_reasoning(fields, boxes, counts, analyze_cc=True, antialias=True, image_hw=hw)[3]
    assert int(cc[2]) > 0   # the overflow path is taken
    od = _oda(dev, analyze_cc=True)
    kb, kc = od.discover_batch(fields, boxes, counts, image_hw=hw)
    for i, (im, p) in enumerate(zip(images, props)):
        ref = od.discover_image(im, p.numpy())
        got = kb[i, : int(kc[i])].cpu().numpy()
        assert got.shape == ref.shape and np.array_equal(got, ref), (i, got.shape, ref.shape)


def _pipe(dev):
    from unmore_b200.object_reasoning import default_args
    from unmore_b200.pipeline import ReasoningPipeline
    return ReasoningPipeline(dev, args=default_args(antialias=True))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 1])
def test_run_chunk_per_image(dev, k):
    images, props, fields, hw, boxes, counts = _batch(k, math.nan, dev)
    pipe = _pipe(dev)
    r = pipe.run_chunk(fields, boxes, counts, image_hw=hw)
    for i, (im, p) in enumerate(zip(images, props)):
        if not p.shape[0]:
            continue
        ref = pipe.run_chunk(*_alone(im, p, dev))
        h, w = im.shape[1], im.shape[2]
        nk = int(ref["box_counts"][0])
        assert int(r["box_counts"][i]) == nk
        _eq(r["boxes"][i, :nk], ref["boxes"][0, :nk], "boxes")
        kk = int(ref["keep_counts"][0])
        assert int(r["keep_counts"][i]) == kk
        for key in ("out", "bbox", "selected", "keep"):
            _eq(r[key][i, :kk], ref[key][0, :kk], key)
        _eq(r["masks"][i, :nk, :h, :(w + 31) // 32], ref["masks"][0, :nk], "masks")
        for key in ("exist_box_mean", "sdf_box_mean"):
            _eq(r[key][i, :p.shape[0]], ref[key][0], key)


@pytest.mark.gpu
def test_uniform_batch_through_image_hw_equals_uniform_path(dev):
    """Two bench.py images (480x640, 4096 proposals): the sized antialiased kernels on a batch without padding give what
    the uniform antialiased kernels give."""
    fields = torch.stack([synth.make_fields(i) for i in (0, 1)]).to(dev)
    props = torch.stack([torch.from_numpy(synth.make_proposals(i, 4096)) for i in (0, 1)]).to(dev)
    hw = torch.tensor([[480, 640]] * 2, dtype=torch.int32, device=dev)
    pipe = _pipe(dev)
    a, b = pipe.run_chunk(fields, props), pipe.run_chunk(fields, props, image_hw=hw)
    assert a.keys() == b.keys()
    for key in a:
        _eq(a[key], b[key], key)
    assert int(a["keep_counts"].sum()) > 0


@pytest.mark.gpu
def test_mains_batch_size_write_identical_files(dev, tmp_path):
    from unmore_b200.object_reasoning import FieldDataset, Object_Discovery, default_args
    from unmore_b200.object_scoring import Object_Scoring
    shapes = [(480, 640), (427, 640), (640, 480), (360, 640), (500, 375), (256, 256), (120, 90), (640, 612), (333, 500),
              (480, 640), (90, 160)]
    ds = FieldDataset([synth.make_fields(50 + i, h, w) for i, (h, w) in enumerate(shapes)], image_ids=[5 + 2 * i for i in range(len(shapes))])
    files = {}
    for bs in (1, 8):
        od = Object_Discovery(default_args(antialias=True), device=dev, test_dataset=ds, result_folder=str(tmp_path / f"d{bs}"))
        res = od.main_object_discovery(batch_size=bs)
        with open(tmp_path / f"d{bs}" / "discovery_results.json") as f:
            raw = f.read()
        osc = Object_Scoring(argparse.Namespace(antialias=True), device=dev, raw_annotations=json.loads(raw), test_dataset=ds,
                             result_folder=str(tmp_path / f"s{bs}"))
        anns = osc.main_object_scoring(batch_size=bs)
        with open(tmp_path / f"s{bs}" / "object_discovery_with_scores.json") as f:
            files[bs] = (res, raw, anns, f.read())
    (r1, d1, a1, s1), (r8, d8, a8, s8) = files[1], files[8]
    assert list(r1) == list(r8) and all(np.array_equal(r1[k], r8[k]) for k in r1)
    assert d1 == d8 and s1 == s8
    assert len(a1) == len(a8) > 0


@pytest.mark.gpu
def test_off_size_image_in_padded_batch_against_oracle(dev):
    """One 300x400 image between two others in a NaN-padded batch, against the CPU oracle in the antialiased mode, with
    the tolerances of the antialiased fuzz test (boxes and scores 1e-5 relative, masks bit-exact)."""
    from oracle import oracle as O
    from unmore_b200 import ops
    from unmore_b200.object_scoring import Object_Scoring
    shapes = [(480, 640), (300, 400), (250, 180)]
    images = [synth.make_fields(4100 + i, h, w) for i, (h, w) in enumerate(shapes)]
    props = [torch.from_numpy(synth.make_proposals(4100 + i, 120, h, w)) for i, (h, w) in enumerate(shapes)]
    fields, hw = ops.pack_fields([im.to(dev) for im in images])
    _pad(fields, shapes, math.nan)
    boxes, counts = ops.stack_proposals(props, dev)
    args = O.make_args()
    with O.antialias_mode(True):
        ref = O.discover_image(images[1], props[1].numpy(), args)
        s_ref = O.score_image(images[1], ref.tolist(), args) if len(ref) else None
    kb, kc = _oda(dev).discover_batch(fields, boxes, counts, image_hw=hw)
    det = kb[1, : int(kc[1])].cpu().numpy().astype(np.float64)
    assert det.shape == ref.shape and len(ref) > 0, (det.shape, ref.shape)
    side = np.maximum(ref[:, 2] - ref[:, 0], ref[:, 3] - ref[:, 1])[:, None]
    assert (np.abs(det - ref) <= 1e-5 * np.maximum(np.abs(ref), side)).all()
    # score the oracle's boxes in the padded batch (the other images score their own discoveries)
    dets = [kb[i, : int(kc[i])].to(torch.float64) for i in range(3)]
    dets[1] = torch.as_tensor(ref, dtype=torch.float64)
    sb, sc = ops.stack_proposals(dets, dev)
    r = Object_Scoring(argparse.Namespace(antialias=True), device=dev).score_batch(fields, sb, sc, image_hw=hw)
    anns = Object_Scoring._annotations(r, 1, 300, 400, 0, True, False)
    assert len(anns) == len(s_ref["score"])
    assert np.array_equal(np.stack([a["segmentation"]["mask"] for a in anns]), s_ref["masks"])
    got = np.array([a["score"] for a in anns], np.float64)
    assert (np.abs(got - s_ref["score"]) <= 1e-5 * np.abs(s_ref["score"])).all()


@pytest.mark.gpu
def test_host_image_hw_is_rejected(dev):
    from unmore_b200 import _lib, ops
    lib = _lib.load()
    fields = torch.zeros((1, 4, 8, 8), device=dev)
    boxes = torch.zeros((1, 4, 4), device=dev)
    out = torch.zeros((1, 4), device=dev)
    ws = torch.zeros((1 << 20,), dtype=torch.int32, device=dev)
    host = np.array([[8, 8]], dtype=np.int32)
    rc = lib.unmore_existence_scores_aa_hw(fields.data_ptr(), 1, 4, 8, 8, host.ctypes.data, 3, boxes.data_ptr(), 0, None, 4,
                                           out.data_ptr(), ws.data_ptr(), None)
    assert rc == -1 and b"host memory" in lib.unmore_last_error()
    with pytest.raises(ops.UnmoreError):   # no sized plain crop
        ops.crop_resize(fields, boxes, [0], image_hw=torch.tensor([[8, 8]], dtype=torch.int32, device=dev))


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_aa_hw_entry_points_reject_bad_arguments():
    """The sized entry points of the second resize mode check their arguments, the extents table included, before
    anything is launched."""
    from unmore_b200 import _lib
    lib = _lib.load()
    fake, hw, odd = ctypes.c_void_p(0x1000), ctypes.c_void_p(0x2000), ctypes.c_void_p(0x2004)
    chans = ctypes.cast((ctypes.c_int * 2)(3, 0), ctypes.c_void_p)
    bad_chans = ctypes.cast((ctypes.c_int * 2)(3, 4), ctypes.c_void_p)
    calls = {   # name: (valid arguments, index of image_hw, [(index, bad value)])
        "unmore_existence_scores_aa_hw": ([fake, 1, 4, 8, 8, hw, 3, fake, 1, None, 4, fake, fake, None], 5,
                                          [(0, None), (4, 0), (5, odd), (6, 4), (7, None), (9, -1), (11, None), (12, None)]),
        "unmore_boundary_refine_aa_hw": ([fake, 1, 4, 8, 8, hw, 0, fake, 1, None, 4, 50, 1, 1, 50.0, 0.5, 16.0, 0.5, fake, fake,
                                          None, fake, None], 5,
                                         [(0, None), (4, -3), (5, odd), (6, 4), (7, None), (10, -1), (11, 0), (18, None),
                                          (19, None), (21, None)]),
        "unmore_crop_resize_aa_hw": ([fake, 1, 4, 8, 8, hw, chans, 2, fake, 1, None, 4, fake, fake, 1 << 20, None], 5,
                                     [(0, None), (3, 0), (5, odd), (6, None), (6, bad_chans), (7, 0), (7, 5), (8, None),
                                      (11, -1), (12, None), (13, None), (14, 16)]),
        "unmore_center_reasoning_from_tiles_hw": ([fake, 1, 8, 8, hw, fake, 1, None, 4, 0.009, fake, fake, fake, None, None,
                                                   None, fake, None], 4,
                                                  [(0, None), (1, 0), (2, 0), (4, odd), (5, None), (8, -1), (10, None),
                                                   (11, None), (13, fake), (16, None)]),
        "unmore_score_and_rasterise_from_tiles_hw": ([fake, None, 1, 1, 8, 8, hw, fake, 1, None, 4, fake, fake, fake, None,
                                                      None], 6,
                                                     [(0, None), (3, 0), (4, 0), (6, odd), (7, None), (10, -1), (11, None),
                                                      (12, None), (13, None), (3, 70000)]),
    }
    assert set(calls) <= set(_lib.SIGNATURES)
    for name, (ok, at, bads) in calls.items():
        fn = getattr(lib, name)
        for i, bad in bads:
            args = list(ok)
            args[i] = bad
            assert fn(*args) != 0, (name, i)
        args = list(ok)
        args[at] = None
        assert fn(*args) == -1 and b"image_hw is null" in lib.unmore_last_error(), name
        args[at] = odd
        assert fn(*args) == -1 and b"8-byte aligned" in lib.unmore_last_error(), name


def test_image_hw_with_a_tile_provider_still_raises():
    """Mixed sizes with per-crop nets are not supported: discover_batch and score_batch refuse image_hw before any work."""
    from unmore_b200 import ops
    from unmore_b200.object_reasoning import Object_Discovery, default_args
    from unmore_b200.object_scoring import Object_Scoring
    fields, boxes = torch.zeros((1, 4, 8, 8)), torch.zeros((1, 2, 4))
    hw = torch.tensor([[8, 8]], dtype=torch.int32)
    od = Object_Discovery.__new__(Object_Discovery)   # the constructors want a CUDA device; the check runs before any
    od.args, od.channels, od.antialias, od.tile_provider = default_args(antialias=True), ops.DEFAULT_CHANNELS, True, object()
    with pytest.raises(ops.UnmoreError, match="tile provider"):
        od.discover_batch(fields, boxes, image_hw=hw)
    osc = Object_Scoring.__new__(Object_Scoring)
    osc.args, osc.channels, osc.antialias, osc.tile_provider = argparse.Namespace(antialias=True), ops.DEFAULT_CHANNELS, True, object()
    with pytest.raises(ops.UnmoreError, match="tile provider"):
        osc.score_batch(fields, boxes, image_hw=hw)
