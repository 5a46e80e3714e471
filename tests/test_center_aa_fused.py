"""Center reasoning in the second resize mode (antialias=True) in one fused call: the kernel resamples the antialiased
crops of the three center-stage planes straight from the fields.  It must equal, bit for bit, the tile composition it
replaces: ``crop_resize(..., antialias=True)`` of (sdf, center_row, center_col) followed by
``center_reasoning_from_tiles`` (both with ``image_hw`` on a padded stack).  Compared: max values, arg-max, split boxes,
the --analyze_cc counts and boxes and the overflow count."""
import ctypes
import math

import pytest
import torch

from unmore_b200 import synth

H, W = 480, 640
N = 4096
MODES = [dict(want_splits=True), dict(want_splits=False), dict(want_splits=True, analyze_cc=True)]


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int64) if t.dtype == torch.float64 else t


def _eq(a, b, what=""):
    assert (a is None) == (b is None), what
    if a is None:
        return
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert torch.equal(_bits(a.contiguous()), _bits(b.contiguous())), what


def _eq_result(got, ref, what=""):
    for name, a, b in zip(("max_values", "argmax", "splits"), got[:3], ref[:3]):
        _eq(a, b, f"{what} {name}")
    assert (got[3] is None) == (ref[3] is None), what
    if got[3] is not None:
        for name, a, b in zip(("cc_counts", "cc_boxes", "cc_overflow"), got[3], ref[3]):
            _eq(a, b, f"{what} {name}")


def _tiles_ref(fields, boxes, counts=None, image_hw=None, **kw):
    from unmore_b200 import ops
    ch = ops.DEFAULT_CHANNELS
    tiles = ops.crop_resize(fields, boxes, [ch.sdf, ch.center_row, ch.center_col], counts, antialias=True, image_hw=image_hw)
    return ops.center_reasoning_from_tiles(tiles, fields.shape[-2], fields.shape[-1], boxes, counts, image_hw=image_hw, **kw)


def _check(fields, boxes, counts=None, image_hw=None, modes=MODES, what=""):
    """The fused call against the tile composition in every pass; returns the fused results by mode index."""
    from unmore_b200 import ops
    out = []
    for kw in modes:
        got = ops.center_reasoning(fields, boxes, counts, antialias=True, image_hw=image_hw, **kw)
        _eq_result(got, _tiles_ref(fields, boxes, counts, image_hw, **kw), f"{what} {kw}")
        out.append(got)
    return out


def _extreme_windows(dev):
    """A 1024x1024 field and the windows of the stand-alone resize's extreme-window test: 1x1, 2x3, 1-px strips,
    up-sampled windows, and windows whose 16-17 taps per axis exceed the kernels' tables (the fallback path)."""
    g = torch.Generator().manual_seed(11)
    f = torch.randn((1, 4, 1024, 1024), generator=g)
    boxes = [[10.0, 20.0, 11.0, 21.0], [100.2, 200.7, 101.9, 203.1], [5.0, 5.0, 6.0, 400.0], [5.0, 700.0, 900.0, 701.0],
             [12.3, 7.9, 1011.5, 1007.2], [0.0, 0.0, 1024.0, 1024.0], [500.0, 500.0, 628.0, 628.0], [40.5, 60.2, 97.0, 90.9],
             [0.0, 0.0, 700.0, 300.0], [300.0, 10.0, 400.0, 1000.0], [3.0, 3.0, 3.0, 9.0]]
    return f.to(dev), torch.tensor(boxes, dtype=torch.float64, device=dev)[None].contiguous()


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def bench_image(dev):
    """The benchmark image and its proposals kept at existence >= 0.1 (the first pass of discovery)."""
    from unmore_b200 import ops
    f = synth.make_fields(0, H, W).to(dev)
    props = torch.from_numpy(synth.make_proposals(0, N, H, W)).to(dev)
    ex = ops.existence_scores(f[None].contiguous(), props[None].contiguous(), antialias=True)[0]
    return f[None].contiguous(), props[ex >= 0.1]


# ---- the benchmark image -----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_benchmark_image_first_and_second_pass(bench_image, dtype):
    from unmore_b200 import ops
    fields, p1 = bench_image
    boxes = p1.to(dtype)[None].contiguous()
    first = _check(fields, boxes, modes=[dict(want_splits=True)], what="first pass")[0]
    fail = first[1][0] >= 0
    assert 0 < int(fail.sum()) < boxes.shape[1]   # proposals both pass and split
    assert not torch.equal(first[0], ops.center_reasoning(fields, boxes)[0])   # the resize modes differ
    split = first[2][0][fail].reshape(1, -1, 4).contiguous()
    _check(fields, split, modes=[dict(want_splits=False)], what="second pass")


# ---- counts, field sizes, windows --------------------------------------------------------------------------------
@pytest.mark.gpu
def test_ragged_counts_empty_image_and_other_field_width(dev):
    h, w = 300, 517
    fields = torch.stack([synth.make_fields(i, h, w) for i in (4, 5, 6)]).to(dev)
    boxes = torch.stack([torch.from_numpy(synth.make_proposals(i, 600, h, w)) for i in (4, 5, 6)]).to(dev).contiguous()
    counts = torch.tensor([600, 0, 257], dtype=torch.int32, device=dev)
    got = _check(fields, boxes, counts, what="ragged")
    for r in got:   # rows past the counts keep their initial values
        assert float(r[0][1:2].abs().sum()) == 0.0 and bool((r[1][1:2] == -1).all())
    _check(fields, boxes, None, what="counts=None")


@pytest.mark.gpu
def test_extreme_windows_and_tap_fallbacks(dev):
    f, boxes = _extreme_windows(dev)
    _check(f, boxes, what="extreme windows")
    # 2304 rows, one window over all of them: scale 18, about 36 vertical taps per output row, more than a warp's lanes
    g = torch.Generator().manual_seed(12)
    tall = torch.randn((1, 4, 2304, 200), generator=g).to(dev)
    tb = torch.tensor([[[0.0, 0.0, 200.0, 2304.0], [7.5, 1.0, 190.2, 2300.5], [0.0, 100.0, 1.0, 2304.0]]],
                      dtype=torch.float64, device=dev)
    _check(tall, tb, what="2304 rows")


def _flat(dev, center, h=160, w=200):
    """A field whose union mask covers everything (sdf > 0) and whose center field is `center` [2, h, w]."""
    f = torch.empty((1, 4, h, w))
    f[0, 0] = 1.0
    f[0, 1:3] = center
    f[0, 3] = 0.5
    return f.to(dev)


@pytest.mark.gpu
def test_plateaus_and_ties(dev):
    """Constant, two-valued and zero center fields: more screening candidates than the queue holds (the plateau path),
    and ties of the exact maximum broken by the first flat index."""
    h, w = 160, 200
    two = torch.full((2, h, w), 0.3)
    two[:, :, w // 2:] = -0.3
    boxes = torch.tensor([[[0.0, 0.0, 200.0, 160.0], [10.5, 3.2, 170.0, 150.8], [50.0, 40.0, 90.0, 80.0],
                           [99.0, 20.0, 101.0, 140.0], [30.0, 30.0, 190.0, 60.0]]], dtype=torch.float64, device=dev)
    for what, center in (("constant", torch.full((2, h, w), 0.7)), ("two-valued", two), ("zero", torch.zeros((2, h, w)))):
        _check(_flat(dev, center, h, w), boxes, what=what)


# ---- --analyze_cc ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_analyze_cc_components_and_overflow(dev):
    from unmore_b200 import _lib
    h, w = 100, 90
    blobs = torch.full((1, 4, h, w), -4.0)
    blobs[0, 0, 10:30, 10:30] = 4.0
    blobs[0, 0, 50:80, 45:85] = 4.0
    blobs[0, 1:3] = 0.0
    speckled = torch.full((1, 4, h, w), -4.0)
    speckled[0, 0, 2::6, 2::6] = 4.0
    speckled[0, 1:3] = 0.0
    boxes = torch.tensor([[[0.0, 0.0, 90.0, 100.0], [5.0, 5.0, 60.0, 55.0], [10.0, 20.0, 80.0, 60.0]]],
                         dtype=torch.float64, device=dev)
    kw = [dict(want_splits=True, analyze_cc=True)]
    two = _check(blobs.to(dev), boxes, modes=kw, what="two components")[0]
    assert int(two[3][0][0, 0]) == 2 and int(two[3][2]) == 0
    many = _check(speckled.to(dev), boxes, modes=kw, what="more than the cap")[0]
    assert int(many[3][2]) > 0 and int(many[3][0].max()) == _lib.load().unmore_cc_cap()


# ---- padded stacks -----------------------------------------------------------------------------------------------
def _past(h, w):
    return [[w - 80.5, h - 60.2, w + 200.0, h + 150.0], [-10.0, -5.0, w + 20.0, h + 10.0], [w * 0.5, 0.0, 640.0, 480.0],
            [0.0, h * 0.4, w + 0.5, h - 1.0], [w - 3.0, h - 3.0, w + 40.0, h + 40.0], [5.0, 5.0, w * 0.8, h * 0.8]]


@pytest.mark.gpu
@pytest.mark.parametrize("pad", [math.nan, 0.0])
def test_padded_stack_per_image(dev, pad):
    """Images of two sizes plus one at the full pitch, boxes past the image edges and an image without proposals: the
    sized call equals the sized tile composition, and gives every image what the uniform fused call gives it alone."""
    from unmore_b200 import ops
    shapes, n = [(300, 400), (480, 640), (211, 517), (120, 95)], [300, 250, 0, 40]
    images = [synth.make_fields(40 + i, h, w).to(dev) for i, (h, w) in enumerate(shapes)]
    props = [torch.cat((torch.from_numpy(synth.make_proposals(40 + i, k, h, w)[:k]), torch.tensor(_past(h, w), dtype=torch.float64)))
             if k else torch.zeros((0, 4), dtype=torch.float64) for i, ((h, w), k) in enumerate(zip(shapes, n))]
    fields, hw = ops.pack_fields(images)
    for i, (h, w) in enumerate(shapes):
        fields[i, :, h:, :] = pad
        fields[i, :, :, w:] = pad
    boxes, counts = ops.stack_proposals(props, dev)
    got = _check(fields, boxes, counts, hw, what="padded")
    for i, (im, p) in enumerate(zip(images, props)):
        k = p.shape[0]
        if not k:
            assert float(got[0][0][i].abs().sum()) == 0.0
            continue
        for kw, g in zip(MODES, got):
            alone = ops.center_reasoning(im[None].contiguous(), p[None].to(dev).contiguous(), antialias=True, **kw)
            for a, b, name in zip(g[:3], alone[:3], ("max_values", "argmax", "splits")):
                if a is not None:
                    _eq(a[i, :k], b[0], f"image {i} {kw} {name}")
            if g[3] is not None:
                _eq(g[3][0][i, :k], alone[3][0][0], f"image {i} cc_counts")
                _eq(g[3][1][i, :k], alone[3][1][0], f"image {i} cc_boxes (clipped to the image)")


# ---- one call ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cap", [8, 50000])
def test_one_call_at_any_capacity(dev, cap):
    """No slicing: one kernel plus the counts prefix, whatever the capacity."""
    from unmore_b200 import ops
    fields = torch.stack([synth.make_fields(i, H, W) for i in (0, 1)]).to(dev)
    boxes = torch.zeros((2, cap, 4), dtype=torch.float64, device=dev)
    boxes[:, :8] = torch.stack([torch.from_numpy(synth.make_proposals(i, 8, H, W)) for i in (0, 1)]).to(dev)
    counts = torch.tensor([8, 5], dtype=torch.int32, device=dev)
    for kw in MODES:
        l0 = ops.LAUNCHES
        ops.center_reasoning(fields, boxes, counts, antialias=True, **kw)
        assert ops.LAUNCHES - l0 == 2, kw
    if cap == 8:
        _check(fields, boxes, counts, what="8 proposals")


# ---- C ABI (no GPU) ----------------------------------------------------------------------------------------------
def test_center_aa_entry_points_reject_bad_arguments():
    """Both entry points check their arguments like unmore_center_reasoning[_hw] before anything is launched."""
    from unmore_b200 import _lib
    lib = _lib.load()
    fake, hw, odd = ctypes.c_void_p(0x1000), ctypes.c_void_p(0x2000), ctypes.c_void_p(0x2004)
    ok = [fake, 1, 4, 8, 8, 0, 1, 2, fake, 1, None, 4, 0.009, fake, fake, None, None, None, None, fake, None]
    # null fields, channel out of range (each of the three), null boxes, negative capacity, null workspace
    bads = [(0, None), (5, 4), (6, -1), (7, 4), (8, None), (11, -1), (19, None)]
    for name, sized in (("unmore_center_reasoning_aa", False), ("unmore_center_reasoning_aa_hw", True)):
        assert name in _lib.SIGNATURES
        fn = getattr(lib, name)
        base = ok[:5] + [hw] + ok[5:] if sized else ok
        shift = 1 if sized else 0
        for i, bad in bads:
            args = list(base)
            args[i + shift if i >= 5 else i] = bad
            assert fn(*args) == -1, (name, i)
            assert i == 0 or name.encode() in lib.unmore_last_error(), (name, i)
        if sized:
            for bad, msg in ((None, b"image_hw is null"), (odd, b"8-byte aligned")):
                args = list(base)
                args[5] = bad
                assert fn(*args) == -1 and msg in lib.unmore_last_error(), name
