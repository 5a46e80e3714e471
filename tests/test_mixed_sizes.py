"""Batches of images of different sizes: a padded field stack with per-image extents (``ops.pack_fields``, ``image_hw``).
Every op, and discovery / scoring end to end, must give each image of a padded batch exactly, bit for bit, what the
uniform path gives that image alone.  The padding is filled with NaN (and, once, left at zero): a kernel that read it
would show it in its results, and since the padding lies inside the allocation nothing can fault."""
import ctypes
import json
import math

import numpy as np
import pytest
import torch

from unmore_b200 import synth

# (pitch, [(h, w, proposals)]): the first batch has the 480x640 pitch of the specialised kernels and an image that fills
# it; the second a pitch no kernel is specialised for.  Both hold an image without proposals and a tiny image.
BATCHES = [
    ((480, 640), [(480, 640, 700), (300, 400, 500), (200, 360, 0), (37, 53, 64), (411, 517, 600)]),
    ((640, 612), [(640, 480, 700), (612, 612, 600), (200, 360, 300), (9, 14, 16), (333, 97, 0)]),
]


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int64) if t.dtype == torch.float64 else t


def _eq(a, b, what=""):
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert torch.equal(_bits(a.contiguous()), _bits(b.contiguous())), what


def _batch(k, pad, dev):
    from unmore_b200 import ops
    _, spec = BATCHES[k]
    images = [synth.make_fields(10 * k + i, h, w).to(dev) for i, (h, w, _) in enumerate(spec)]
    props = [torch.from_numpy(synth.make_proposals(10 * k + i, n, h, w)[:n]) for i, (h, w, n) in enumerate(spec)]
    fields, hw = ops.pack_fields(images)
    if pad != 0.0:
        for i, (h, w, _) in enumerate(spec):
            fields[i, :, h:, :] = pad
            fields[i, :, :, w:] = pad
    boxes, counts = ops.stack_proposals(props, dev)
    return images, props, fields, hw, boxes, counts


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


CASES = [(0, math.nan), (1, math.nan), (0, 0.0)]


# ---- per op ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k,pad", CASES)
def test_existence_per_image(dev, k, pad):
    from unmore_b200 import ops
    images, props, fields, hw, boxes, counts = _batch(k, pad, dev)
    got = ops.existence_scores(fields, boxes, counts, image_hw=hw)
    for i, (im, p) in enumerate(zip(images, props)):
        n = p.shape[0]
        if n:
            _eq(got[i, :n], ops.existence_scores(im[None].contiguous(), p[None].to(dev).contiguous())[0], ("existence", i))


@pytest.mark.gpu
@pytest.mark.parametrize("k,pad", CASES)
@pytest.mark.parametrize("splits,cc", [(True, False), (False, False), (True, True)])
def test_center_per_image(dev, k, pad, splits, cc):
    from unmore_b200 import ops
    images, props, fields, hw, boxes, counts = _batch(k, pad, dev)
    mv, am, sp, cs = ops.center_reasoning(fields, boxes, counts, want_splits=splits, analyze_cc=cc, image_hw=hw)
    for i, (im, p) in enumerate(zip(images, props)):
        n = p.shape[0]
        if not n:
            continue
        rmv, ram, rsp, rcs = ops.center_reasoning(im[None].contiguous(), p[None].to(dev).contiguous(), want_splits=splits,
                                                  analyze_cc=cc)
        _eq(mv[i, :n], rmv[0], ("max", i))
        _eq(am[i, :n], ram[0], ("argmax", i))
        if splits:
            _eq(sp[i, :n], rsp[0], ("splits", i))
        if cc:
            _eq(cs[0][i, :n], rcs[0][0], ("cc counts", i))
            _eq(cs[1][i, :n], rcs[1][0], ("cc boxes", i))


@pytest.mark.gpu
@pytest.mark.parametrize("k,pad", CASES)
@pytest.mark.parametrize("early_exit", [True, False])
def test_refine_per_image(dev, k, pad, early_exit):
    from unmore_b200 import ops
    images, props, fields, hw, boxes, counts = _batch(k, pad, dev)
    rb, lab, rounds = ops.boundary_refine(fields, boxes, counts, early_exit=early_exit, image_hw=hw)
    for i, (im, p) in enumerate(zip(images, props)):
        n = p.shape[0]
        if not n:
            continue
        rrb, rlab, rrounds = ops.boundary_refine(im[None].contiguous(), p[None].to(dev).contiguous(), early_exit=early_exit)
        _eq(rb[i, :n], rrb[0], ("boxes", i))
        _eq(lab[i, :n], rlab[0], ("labels", i))
        _eq(rounds[i, :n], rrounds[0], ("rounds", i))


@pytest.mark.gpu
@pytest.mark.parametrize("k,pad", CASES)
def test_scoring_per_image(dev, k, pad):
    from unmore_b200 import ops
    images, props, fields, hw, boxes, counts = _batch(k, pad, dev)
    sc, tight, areas, masks = ops.score_and_rasterise(fields, boxes, counts, image_hw=hw)
    for i, (im, p) in enumerate(zip(images, props)):
        n, h, w = p.shape[0], im.shape[1], im.shape[2]
        if not n:
            continue
        rsc, rtight, rareas, rmasks = ops.score_and_rasterise(im[None].contiguous(), p[None].to(dev).contiguous())
        _eq(sc[i, :n], rsc[0], ("scores", i))
        _eq(tight[i, :n], rtight[0], ("tight", i))
        _eq(areas[i, :n], rareas[0], ("areas", i))
        wp = (w + 31) // 32
        _eq(masks[i, :n, :h, :wp], rmasks[0], ("masks", i))
        outside = masks[i, :n].clone()
        outside[:, :h, :wp] = 0
        assert int(outside.abs().sum()) == 0, ("mask bits outside the image", i)
    assert int(areas.sum()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("k,pad", CASES)
def test_box_sums_per_image(dev, k, pad):
    from unmore_b200 import ops
    images, props, fields, hw, boxes, counts = _batch(k, pad, dev)
    sat = ops.sat_build_fields(fields, [3, 0], image_hw=hw)
    for plane in (0, 1):
        s, m = ops.box_sums(sat, plane, boxes, counts, image_hw=hw)
        for i, (im, p) in enumerate(zip(images, props)):
            n = p.shape[0]
            if not n:
                continue
            rs, rm = ops.box_sums(ops.sat_build_fields(im[None].contiguous(), [3, 0]), plane, p[None].to(dev).contiguous())
            _eq(s[i, :n], rs[0], ("sums", plane, i))
            _eq(m[i, :n], rm[0], ("means", plane, i))


# ---- end to end --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 1])
@pytest.mark.parametrize("cc_on", [False, True])
def test_discover_batch_per_image(dev, k, cc_on):
    from unmore_b200.object_reasoning import Object_Discovery, default_args
    images, props, fields, hw, boxes, counts = _batch(k, math.nan, dev)
    od = Object_Discovery(default_args(analyze_cc=cc_on), device=dev)
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
    from unmore_b200.object_reasoning import Object_Discovery, default_args
    shapes = [(100, 90), (120, 150), (64, 70)]
    images = [_speckled(h, w, dev) for h, w in shapes]
    props = [torch.tensor([[5.0, 5.0, 60.0, 55.0], [10.0, 20.0, 80.0, 60.0]], dtype=torch.float64)[: 2 - (i == 2)]
             for i in range(len(shapes))]
    fields, hw = ops.pack_fields(images)
    for i, (h, w) in enumerate(shapes):
        fields[i, :, h:, :] = math.nan
        fields[i, :, :, w:] = math.nan
    boxes, counts = ops.stack_proposals(props, dev)
    cc = ops.center_reasoning(fields, boxes, counts, analyze_cc=True, image_hw=hw)[3]
    assert int(cc[2]) > 0   # the overflow path is taken
    od = Object_Discovery(default_args(analyze_cc=True), device=dev)
    kb, kc = od.discover_batch(fields, boxes, counts, image_hw=hw)
    for i, (im, p) in enumerate(zip(images, props)):
        ref = od.discover_image(im, p.numpy())
        got = kb[i, : int(kc[i])].cpu().numpy()
        assert got.shape == ref.shape and np.array_equal(got, ref), (i, got.shape, ref.shape)


def _run_chunk_equal(r, ref, b, n_props, h, w):
    k = int(ref["box_counts"][0])
    assert int(r["box_counts"][b]) == k
    _eq(r["boxes"][b, :k], ref["boxes"][0, :k], "boxes")
    kk = int(ref["keep_counts"][0])
    assert int(r["keep_counts"][b]) == kk
    for key in ("out", "bbox", "selected", "keep"):
        _eq(r[key][b, :kk], ref[key][0, :kk], key)
    wp = (w + 31) // 32
    _eq(r["masks"][b, :k, :h, :wp], ref["masks"][0, :k], "masks")
    for key in ("exist_box_mean", "sdf_box_mean"):
        _eq(r[key][b, :n_props], ref[key][0], key)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 1])
def test_run_chunk_per_image(dev, k):
    from unmore_b200.pipeline import ReasoningPipeline
    images, props, fields, hw, boxes, counts = _batch(k, math.nan, dev)
    pipe = ReasoningPipeline(dev)
    r = pipe.run_chunk(fields, boxes, counts, image_hw=hw)
    for i, (im, p) in enumerate(zip(images, props)):
        if p.shape[0]:
            ref = pipe.run_chunk(im[None].contiguous(), p[None].to(dev).contiguous())
            _run_chunk_equal(r, ref, i, p.shape[0], im.shape[1], im.shape[2])


@pytest.mark.gpu
def test_uniform_batch_through_image_hw_equals_uniform_path(dev):
    """Two bench.py images (480x640, 4096 proposals): the sized kernels on a batch without padding give what the
    uniform kernels give."""
    from unmore_b200.pipeline import ReasoningPipeline
    fields = torch.stack([synth.make_fields(i) for i in (0, 1)]).to(dev)
    props = torch.stack([torch.from_numpy(synth.make_proposals(i, 4096)) for i in (0, 1)]).to(dev)
    hw = torch.tensor([[480, 640]] * 2, dtype=torch.int32, device=dev)
    pipe = ReasoningPipeline(dev)
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
    ds = FieldDataset([synth.make_fields(30 + i, h, w) for i, (h, w) in enumerate(shapes)], image_ids=[7 + 3 * i for i in range(len(shapes))])
    files = {}
    for bs in (1, 8):
        od = Object_Discovery(default_args(), device=dev, test_dataset=ds, result_folder=str(tmp_path / f"d{bs}"))
        res = od.main_object_discovery(batch_size=bs)
        with open(tmp_path / f"d{bs}" / "discovery_results.json") as f:
            raw = f.read()
        osc = Object_Scoring(device=dev, raw_annotations=json.loads(raw), test_dataset=ds, result_folder=str(tmp_path / f"s{bs}"))
        anns = osc.main_object_scoring(batch_size=bs)
        with open(tmp_path / f"s{bs}" / "object_discovery_with_scores.json") as f:
            files[bs] = (res, raw, anns, f.read())
    (r1, d1, a1, s1), (r8, d8, a8, s8) = files[1], files[8]
    assert list(r1) == list(r8) and all(np.array_equal(r1[k], r8[k]) for k in r1)
    assert d1 == d8 and s1 == s8
    assert len(a1) == len(a8) > 0


@pytest.mark.gpu
def test_host_image_hw_is_rejected(dev):
    from unmore_b200 import _lib
    lib = _lib.load()
    fields = torch.zeros((1, 4, 8, 8), device=dev)
    boxes = torch.zeros((1, 4, 4), device=dev)
    out = torch.zeros((1, 4), device=dev)
    ws = torch.zeros((1 << 20,), dtype=torch.int32, device=dev)
    host = np.array([[8, 8]], dtype=np.int32)
    rc = lib.unmore_existence_scores_hw(fields.data_ptr(), 1, 4, 8, 8, host.ctypes.data, 3, boxes.data_ptr(), 0, None, 4,
                                        out.data_ptr(), ws.data_ptr(), None)
    assert rc == -1 and b"host memory" in lib.unmore_last_error()


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_pack_fields_and_stack_proposals():
    from unmore_b200 import ops
    a, b = torch.rand(4, 5, 7), torch.rand(4, 9, 3)
    f, hw = ops.pack_fields([a, b])
    assert f.shape == (2, 4, 9, 7) and f.dtype == torch.float32
    assert hw.dtype == torch.int32 and hw.tolist() == [[5, 7], [9, 3]]
    assert torch.equal(f[0, :, :5, :7], a) and torch.equal(f[1, :, :9, :3], b)
    assert int(f[0, :, 5:].abs().sum()) == 0 and int(f[1, :, :, 3:].abs().sum()) == 0
    boxes, counts = ops.stack_proposals([np.ones((3, 4)), torch.zeros((0, 4)), torch.full((5, 4), 2.0)], "cpu")
    assert boxes.shape == (3, 5, 4) and boxes.dtype == torch.float64 and counts.tolist() == [3, 0, 5]
    assert float(boxes[0, :3].sum()) == 12.0 and float(boxes[0, 3:].abs().sum()) == 0.0 and float(boxes[1].abs().sum()) == 0.0
    b32, _ = ops.stack_proposals([torch.ones((2, 4))], "cpu")
    assert b32.dtype == torch.float32
    for bad in ([], [torch.rand(4, 5, 7), torch.rand(3, 5, 7)], [torch.rand(4, 5, 7, dtype=torch.float64)], [torch.rand(5, 7)],
                [torch.rand(1, 4, 5, 7)]):
        with pytest.raises(ops.UnmoreError):
            ops.pack_fields(bad)
    with pytest.raises(ops.UnmoreError):
        ops.stack_proposals([torch.ones((2, 3))])


def test_hw_entry_points_reject_bad_arguments():
    """The sized entry points check their arguments, the extents table included, before anything is launched."""
    from unmore_b200 import _lib
    lib = _lib.load()
    assert lib.unmore_version() == 102
    fake, hw = ctypes.c_void_p(0x1000), ctypes.c_void_p(0x2000)
    calls = {
        "unmore_existence_scores_hw": ([fake, 1, 4, 8, 8, hw, 3, fake, 1, None, 4, fake, fake, None],
                                       [(0, None), (4, 0), (5, None), (5, ctypes.c_void_p(0x2004)), (6, 4), (7, None), (9, -1), (11, None)]),
        "unmore_center_reasoning_hw": ([fake, 1, 4, 8, 8, hw, 0, 1, 2, fake, 1, None, 4, 0.009, fake, fake, fake, None, None, None, fake, None],
                                       [(0, None), (3, 0), (5, None), (6, 4), (9, None), (12, -1), (14, None), (17, fake), (20, None)]),
        "unmore_boundary_refine_hw": ([fake, 1, 4, 8, 8, hw, 0, fake, 1, None, 4, 50, 1, 1, 50.0, 0.5, 16.0, 0.5, fake, fake, None, fake, None],
                                      [(0, None), (4, -3), (5, None), (6, 4), (7, None), (10, -1), (11, 0), (18, None), (21, None)]),
        "unmore_score_and_rasterise_hw": ([fake, 1, 4, 8, 8, hw, 0, 1, 2, 3, fake, 1, None, 4, fake, fake, fake, None, None],
                                          [(0, None), (3, 0), (5, None), (9, 4), (10, None), (13, -1), (16, None), (1, 70000)]),
        "unmore_box_sums_hw": ([fake, 1, 2, 0, 8, 8, hw, fake, 1, None, 4, fake, None, None],
                               [(0, None), (4, 0), (5, 0), (6, None), (3, 2), (7, None), (10, -1), (11, None)]),
        "unmore_sat_build_fields_hw": ([fake, 1, 4, 8, 8, hw, None, 2, fake, None],
                                       [(0, None), (3, 0), (5, None), (6, None), (7, 0), (8, None), (4, 4096)]),
    }
    chans = (ctypes.c_int * 2)(3, 0)
    for name, (ok, bads) in calls.items():
        fn = getattr(lib, name)
        if name == "unmore_sat_build_fields_hw":
            ok[6] = ctypes.cast(chans, ctypes.c_void_p)
        for i, bad in bads:
            args = list(ok)
            args[i] = bad
            assert fn(*args) != 0, (name, i)
        args = list(ok)
        args[5 if name != "unmore_box_sums_hw" else 6] = None
        assert fn(*args) == -1 and b"image_hw is null" in lib.unmore_last_error(), name


def test_mains_accept_batch_size():
    import inspect
    from unmore_b200.object_reasoning import Object_Discovery
    from unmore_b200.object_scoring import Object_Scoring
    for fn in (Object_Discovery.main_object_discovery, Object_Scoring.main_object_scoring):
        p = inspect.signature(fn).parameters["batch_size"]
        assert p.default == 1
