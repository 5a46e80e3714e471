"""CPU-side checks: the C-ABI library loads and exports every symbol the header declares (no
compute without a GPU), host logic of the mirrors, and the multi-rank gather on gloo."""
import os
import re
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "unmore_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(unmore_[a-z0-9_]+)\s*\(", src)) - {"unmore_stream_t"})


def test_library_exports_every_declared_symbol():
    from unmore_b200 import _lib
    lib = _lib.load()
    names = _header_functions()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/unmore_b200.h but not exported"
    bound = set(_lib.SIGNATURES) | {"unmore_last_error", "unmore_version", "unmore_workspace_bytes", "unmore_cc_cap"}
    assert set(names) == bound, set(names) ^ bound
    assert lib.unmore_version() >= 100
    assert lib.unmore_workspace_bytes(10) >= 4 * 12


def test_no_cpu_fallback():
    """The product path must fail loudly without a GPU tensor instead of routing to the oracle."""
    from unmore_b200 import ops, _lib
    with pytest.raises(_lib.UnmoreError):
        ops.existence_scores(torch.zeros((1, 4, 8, 8)), torch.zeros((1, 1, 4)))
    from unmore_b200.object_reasoning import Object_Discovery
    with pytest.raises(RuntimeError):
        Object_Discovery(device="cpu")
    # nothing under unmore_b200/ imports the oracle
    for dirpath, _, files in os.walk(os.path.join(ROOT, "unmore_b200")):
        for f in files:
            if f.endswith(".py"):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, f


def test_synth_is_deterministic_and_shaped():
    from unmore_b200 import synth
    a, b = synth.make_fields(17), synth.make_fields(17)
    assert a.shape == (4, 480, 640) and a.dtype == torch.float32 and torch.equal(a, b)
    assert not torch.equal(a, synth.make_fields(18))
    nrm = torch.sqrt(a[1] ** 2 + a[2] ** 2)
    inside = a[0] > 0
    assert torch.allclose(nrm[inside], torch.ones_like(nrm[inside]), atol=1e-5) or inside.sum() == 0
    assert float(nrm[~inside].max()) == 0.0
    p = synth.make_proposals(17, 4096)
    assert p.shape == (4096, 4) and p.dtype == np.float64
    assert (p[:, 0] >= 0).all() and (p[:, 2] <= 640).all() and (p[:, 3] <= 480).all()
    assert np.array_equal(p[:1225], synth.anchor_proposals(480, 640))


def test_post_process_mirror():
    from unmore_b200.post_process import select_annotations
    anns = [dict(existence_score=0.6, center_score=0.9, boundary_score=0.8, area_score=0.5, score=0.1, bbox=[0, 0, 1, 1]),
            dict(existence_score=0.4, center_score=0.9, boundary_score=0.8, area_score=0.6, score=0.2, bbox=[0, 0, 1, 1]),
            dict(existence_score=0.5, center_score=0.8, boundary_score=0.75, area_score=0.7, score=0.3, bbox=[0, 0, 1, 1]),
            dict(existence_score=0.9, center_score=0.79, boundary_score=0.9, area_score=0.8, score=0.4, bbox=[0, 0, 1, 1])]
    sel = select_annotations(anns)
    assert [a["id"] for a in sel] == [0, 1] and [a["score"] for a in sel] == [0.5, 0.7]  # thresholds are strict '<'


def test_rle_codec_known_answers_and_round_trip():
    """COCO RLE (a16).  pycocotools is absent, so the anchors are answers derived by hand from the
    published maskApi.c (rleEncode / rleToString) plus the decode round trip — parity unpinned."""
    from oracle import oracle as O
    from unmore_b200 import rle
    # column-major [0,1,1,1] -> counts [1,3]; all ones -> leading zero-length run
    assert O.rle_counts(np.array([[0, 1], [1, 1]])) == [1, 3] and O.rle_to_string([1, 3]) == "13"
    assert O.rle_counts(np.ones((2, 2))) == [0, 4] and O.rle_to_string([0, 4]) == "04"
    assert O.rle_counts(np.zeros((3, 2))) == [6] and O.rle_to_string([6]) == "6"
    # 5-bit groups: 31 = 0b11111 has bit 4 set, so a continuation group follows ('o' = 63+48, then '0');
    # 32 -> low group 0 with continuation ('P' = 32+48) then '1'; third+ counts are deltas
    assert rle.counts_to_string([31]) == "o0" and rle.counts_to_string([32]) == "P1"
    assert rle.counts_to_string([5, 7, 9, 3]) == "579" + rle.counts_to_string([3 - 7])   # delta -4, sign-extended
    rng = np.random.default_rng(0)
    for _ in range(40):
        h, w = (int(v) for v in rng.integers(1, 90, 2))
        m = (rng.random((h, w)) < rng.random()).astype(np.uint8)
        c = O.rle_counts(m)
        assert c == O.rle_counts_np(m) and sum(c) == h * w
        s = O.rle_to_string(c)
        assert s == rle.counts_to_string(c) and rle.string_to_counts(s) == c
        assert np.array_equal(rle.decode({"size": [h, w], "counts": s}), m)
        assert all(48 <= ord(ch) <= 111 for ch in s)


def test_shard_ranges_cover_everything():
    from unmore_b200.sharding import shard_indices, shard_range
    for n, w in [(5000, 8), (7, 3), (2, 4), (0, 2)]:
        got = sum((shard_indices(n, r, w) for r in range(w)), [])
        assert got == list(range(n))
        assert sorted(sum((shard_indices(n, r, w, interleave=True) for r in range(w)), [])) == list(range(n))
        assert shard_range(n, w - 1, w)[1] == n


def test_merge_rows_properties():
    """merge_rows on stacked per-rank buffers (what the collective delivers), seeded random shapes: the valid rows
    come first, stably sorted by image id (rank order, then arrival order inside an image), the padding never leaks,
    the total is the sum of the headers, and an overflow flag on any rank is seen."""
    from hypothesis import given, settings, strategies as st
    from unmore_b200.sharding import merge_rows, overflowed, pack_rows_host

    @settings(max_examples=60, deadline=None)
    @given(st.integers(1, 5), st.integers(0, 6), st.integers(1, 4), st.integers(0, 2 ** 31 - 1))
    def check(world, n_img, cap, seed):
        g = torch.Generator().manual_seed(seed)
        bufs, ref = [], []
        for r in range(world):
            ids = torch.randint(0, 9, (n_img,), generator=g).sort().values + 2 ** 30      # ranks may even share an image id
            counts = torch.randint(0, cap + 1, (n_img,), generator=g).to(torch.int32)
            boxes = torch.rand((n_img, cap, 4), generator=g, dtype=torch.float64)
            scores = torch.rand((n_img, cap), generator=g, dtype=torch.float64)
            bufs.append(pack_rows_host(ids, boxes, counts, scores, max_rows=n_img * cap + 3))
            for j in range(n_img):
                for k in range(int(counts[j])):
                    ref.append((int(ids[j]), r, len(ref), torch.cat([ids[j:j + 1].double(), boxes[j, k], scores[j, k:k + 1]])))
        gathered = torch.stack(bufs)
        rows, total = merge_rows(gathered)
        assert int(total) == len(ref) and not bool(overflowed(gathered))
        ref.sort(key=lambda t: (t[0], t[1], t[2]))
        if ref:
            assert torch.equal(rows[: len(ref)], torch.stack([t[3] for t in ref]))
        gathered[world - 1, 0, 1] = 1
        assert bool(overflowed(gathered))

    check()


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from unmore_b200.sharding import shard_indices, pack_rows_host, gather_rows, merge_rows, overflowed, rows_digest
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo")
n_images = 7
def fake(i):   # deterministic ragged "detections" of image i
    g = torch.Generator().manual_seed(i)
    k = int(torch.randint(0, 5, (1,), generator=g))
    return torch.rand((k, 4), generator=g), torch.rand((k,), generator=g)
mine = shard_indices(n_images, rank, world, interleave=True)
cap = 4
boxes = torch.zeros((len(mine), cap, 4)); scores = torch.zeros((len(mine), cap)); counts = torch.zeros(len(mine), dtype=torch.int32)
for j, i in enumerate(mine):
    b, s = fake(i); boxes[j, :len(b)] = b; scores[j, :len(b)] = s; counts[j] = len(b)
big = 2 ** 40   # image ids beyond float32's 2^24 must survive the gather (ADVICE r1)
rows = pack_rows_host(torch.tensor(mine) + big, boxes, counts, scores, max_rows=16)   # same capacity on every rank
g = gather_rows(rows)                    # ONE all_gather_into_tensor
assert g.shape == (world, 17, 6) and not bool(overflowed(g))
merged, total = merge_rows(g)
allrows = merged[: int(total)]
allrows[:, 0] -= big
ref = []
for i in range(n_images):
    b, s = fake(i)
    for k in range(len(b)):
        ref.append(torch.cat([torch.tensor([float(i)]), b[k], s[k:k+1]]))
ref = torch.stack(ref).to(torch.float64)
assert allrows.shape == ref.shape and torch.equal(allrows, ref), (rank, allrows, ref)
digests = [None] * world
dist.all_gather_object(digests, rows_digest(allrows))
assert len(set(digests)) == 1
dist.destroy_process_group()
print("ok", rank)
"""


def test_gather_detections_world2_gloo(tmp_path):
    """N>1 path on CPU: two gloo ranks, interleaved sharding, gathered result == single process."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script), ROOT], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=120)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs


def test_header_is_plain_c_and_links(tmp_path):
    """include/unmore_b200.h is the drop-in boundary: it must compile as C (no C++ or torch types in the
    signatures) and a C program must link against the library and call its non-compute entry points."""
    import shutil
    import subprocess
    from unmore_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "t.c"
    src.write_text('#include <stdio.h>\n#include "unmore_b200.h"\n'
                   'int main(void) { printf("%d %d %zu\\n", unmore_version(), unmore_cc_cap(), (size_t)unmore_workspace_bytes(3));\n'
                   '  const char* e = unmore_last_error(); return e == 0; }\n')
    inc = os.path.join(ROOT, "include")
    libdir = os.path.dirname(_lib.LIB_PATH)
    exe = tmp_path / "t"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", inc, str(src), "-o", str(exe),
                    "-L", libdir, "-l:" + os.path.basename(_lib.LIB_PATH), "-Wl,-rpath," + libdir], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert int(out[0]) >= 100 and int(out[1]) >= 1 and int(out[2]) > 0
    # and as C++ (extern "C" guards)
    cpp = tmp_path / "t.cpp"
    cpp.write_text('#include "unmore_b200.h"\nint main() { return unmore_version() < 0; }\n')
    subprocess.run(["g++", "-std=c++17", "-Wall", "-Werror", "-I", inc, "-c", str(cpp), "-o", str(tmp_path / "t.o")], check=True)


GOLDEN_SIGNATURES = os.path.join(ROOT, "tests", "golden", "reference_signatures.json")
REFERENCE_ROOT = os.environ.get("UNMORE_REFERENCE_ROOT", "")


def _reference_signatures():
    """Parameter lists of the reference's public entry points: the stored ones (``python -m oracle.gen_golden
    signatures`` with UNMORE_REFERENCE_ROOT set writes them), else read from a reference checkout."""
    import json
    if os.path.isfile(GOLDEN_SIGNATURES):
        with open(GOLDEN_SIGNATURES) as f:
            return json.load(f)
    if os.path.isdir(REFERENCE_ROOT):
        from oracle.gen_golden import reference_signatures
        return reference_signatures(REFERENCE_ROOT)
    pytest.skip("the reference's signatures are not stored in tests/golden/reference_signatures.json "
                "and UNMORE_REFERENCE_ROOT names no checkout of the original vLAR-group/unMORE sources")


def test_mirror_signatures_match_the_reference():
    """Every public method of the reference's Object_Discovery / Object_Scoring, batch_erode and
    convert_pred_annotations_to_training_format exists here under the same name, with the reference's
    parameters as a prefix in the same order, and can be called with exactly the reference's required
    arguments (extra parameters here must be optional).  The reference is read with ``ast``: nothing is imported."""
    import inspect
    from unmore_b200 import object_reasoning, object_scoring, post_process
    from unmore_b200.utils import misc
    refsig = _reference_signatures()
    checked = 0
    for cname, cls in [("Object_Discovery", object_reasoning.Object_Discovery),
                       ("Object_Scoring", object_scoring.Object_Scoring)]:
        for name, params in refsig[cname].items():
            assert hasattr(cls, name), f"{cname}.{name} missing"
            sig = inspect.signature(getattr(cls, name))
            ours = list(sig.parameters)
            ref = [p for p in params if p != "self"]   # also the @staticmethod get_prediction_with_proposal_images,
            mine = [p for p in ours if p != "self"]     # which still lists self in the reference
            assert mine[: len(ref)] == ref, f"{cname}.{name}: {mine} vs reference {ref}"
            for p in mine[len(ref):]:
                assert sig.parameters[p].default is not inspect.Parameter.empty, f"{cname}.{name}: extra required parameter {p}"
            checked += 1
    for fn, ours in [("batch_erode", misc.batch_erode),
                     ("convert_pred_annotations_to_training_format", post_process.convert_pred_annotations_to_training_format)]:
        params = refsig["functions"][fn]
        assert list(inspect.signature(ours).parameters)[: len(params)] == params, fn
        checked += 1
    assert checked >= 24
