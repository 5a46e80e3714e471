"""The refine kernel's per-image window cache: proposals of one image share the boundary terms of a crop window
that another proposal already evaluated.  Sharing must be invisible: every result is compared bit for bit with the
same proposals laid out one per image, where nothing can be shared."""
import numpy as np
import pytest
import torch

from unmore_b200 import synth

H, W = 480, 640
CHUNK = 512   # proposals (= single-proposal images) per call of the unshared layout


def _slots_per_image(lib):
    # the workspace grows by the worklist offset (one int) and one table of 32-byte slots per image
    return (lib.unmore_workspace_bytes(2) - lib.unmore_workspace_bytes(1) - 4) // 32


def test_workspace_covers_worklist_and_aligned_tables():
    from unmore_b200 import _lib
    lib = _lib.load()
    slots = _slots_per_image(lib)
    assert slots >= 1024 and slots & (slots - 1) == 0
    assert lib.unmore_workspace_bytes(0) >= 4 * 2
    for n in (1, 3, 250, 4096):
        # counter + n + 1 offsets, up to 31 bytes to the first 32-byte boundary, n tables
        assert lib.unmore_workspace_bytes(n) >= 4 * (n + 2) + 31 + 32 * slots * n


def _refine_shared(ops, plane, boxes, **kw):
    """All proposals in one image: the window cache is shared between them."""
    return ops.boundary_refine(plane[None].contiguous(), boxes[None].contiguous(), ch=ops.Channels(sdf=0), **kw)


def _refine_unshared(ops, plane, boxes, **kw):
    """One proposal per image (the field repeated): no two proposals can share a table."""
    n = boxes.shape[0]
    fields = plane[None].expand(min(n, CHUNK), -1, -1, -1).contiguous()
    outs = []
    for s in range(0, n, CHUNK):
        b = boxes[s:s + CHUNK]
        o = ops.boundary_refine(fields[: len(b)], b[:, None].contiguous(), ch=ops.Channels(sdf=0), **kw)
        outs.append([t[:, 0] if t is not None else None for t in o])
    return [torch.cat([o[i] for o in outs]) if outs[0][i] is not None else None for i in range(3)]


def _assert_bit_equal(a, b):
    for x, y in zip(a, b):
        if x is None:
            assert y is None
            continue
        assert torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                           y.view(torch.int32) if y.dtype == torch.float32 else y)


def _sdf_plane(index, dev):
    return synth.make_fields(index, H, W)[:1].to(dev)   # channel 0: the boundary-distance field


@pytest.mark.gpu
@pytest.mark.parametrize("early_exit", [True, False])
def test_sharing_is_invisible_on_a_benchmark_image(early_exit):
    from unmore_b200 import ops
    dev = torch.device("cuda:0")
    plane = _sdf_plane(0, dev)
    boxes = torch.from_numpy(synth.make_proposals(0, 4096, H, W)).to(dev)
    a = _refine_shared(ops, plane, boxes, early_exit=early_exit)
    b = _refine_unshared(ops, plane, boxes, early_exit=early_exit)
    assert int(a[2].sum()) > 4096   # proposals do run several rounds
    _assert_bit_equal([t[0] for t in a], b)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_forced_collisions(dtype):
    """Many sub-pixel jittered copies of a few boxes: all copies snap to the same window in round 0, so warps
    race for the same slots (claim, wait, read) from the first round on."""
    from unmore_b200 import ops
    dev = torch.device("cuda:0")
    plane = _sdf_plane(1, dev)
    rng = np.random.default_rng(7)
    base = np.array([[100, 80, 260, 240], [0, 0, 640, 480], [300, 200, 420, 330], [20, 300, 90, 470],
                     [500, 10, 639, 120], [230, 150, 250, 170], [50, 50, 400, 400], [400, 250, 600, 470]], np.float64)
    copies = 512
    j = rng.uniform(0.0, 0.99, size=(len(base), copies, 4))
    boxes = np.repeat(base[:, None], copies, axis=1)
    boxes[..., :2] += j[..., :2]   # floor(x1) unchanged
    boxes[..., 2:] -= j[..., 2:]   # ceil(x2) unchanged
    boxes = torch.from_numpy(boxes.reshape(-1, 4)).to(dev, dtype)
    perm = torch.from_numpy(rng.permutation(len(boxes))).to(dev)   # interleave the copies across warps
    boxes = boxes[perm].contiguous()
    a = _refine_shared(ops, plane, boxes)
    b = _refine_unshared(ops, plane, boxes)
    _assert_bit_equal([t[0] for t in a], b)


@pytest.mark.gpu
def test_full_table():
    """More distinct windows in one image than its table has slots: the probe bound runs out and rounds compute
    their terms without publishing them."""
    from unmore_b200 import ops, _lib
    dev = torch.device("cuda:0")
    slots = _slots_per_image(_lib.load())
    plane = _sdf_plane(2, dev)
    rng = np.random.default_rng(11)
    n = slots + slots // 4
    x1 = rng.uniform(0, W - 8, n)
    y1 = rng.uniform(0, H - 8, n)
    boxes = np.stack([x1, y1, x1 + rng.uniform(4, W - x1), y1 + rng.uniform(4, H - y1)], 1)
    snapped = np.stack([np.floor(boxes[:, 0]), np.floor(boxes[:, 1]), np.ceil(boxes[:, 2]), np.ceil(boxes[:, 3])], 1)
    assert len(np.unique(snapped, axis=0)) > slots
    boxes = torch.from_numpy(boxes).to(dev, torch.float32)
    kw = dict(n_round=1, apply_small_filter=False)
    a = _refine_shared(ops, plane, boxes, **kw)
    b = _refine_unshared(ops, plane, boxes, **kw)
    _assert_bit_equal([t[0] for t in a], b)
