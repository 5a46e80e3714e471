"""Time of unmore_mask_rle_counts on one chunk worth of kept masks (1750 x 480x640): 0.34 ms on one B200, where the
bit-serial round-1 kernel took 1.60 ms."""
import os, sys, torch, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from unmore_b200 import ops
dev = torch.device("cuda:0")
H, W, K = 480, 640, 1750
rng = np.random.default_rng(0)
yy, xx = np.mgrid[0:H, 0:W]
m = np.zeros((K, H, W), np.uint8)
for i in range(K):
    cy, cx, ry, rx = rng.uniform(0, H), rng.uniform(0, W), rng.uniform(20, 200), rng.uniform(20, 250)
    m[i] = (((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2) < 1
packed = ops.mask_pack(torch.tensor(m, device=dev))
cnt, nr = ops.mask_rle_counts(packed, W, 1024); torch.cuda.synchronize()
ts = []
for _ in range(5):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); ops.mask_rle_counts(packed, W, 1024); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b))
print(f"rle_counts {K} masks {H}x{W}: {min(ts):.3f} ms  ({min(ts)*1e3/K:.2f} us per mask)  checksum {int(cnt.sum())} {int(nr.sum())}")
