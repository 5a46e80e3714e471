"""Share of refine proposal-rounds whose snapped crop window was already evaluated for the same image
(CPU oracle, bench images, kernel early exit emulated).  usage: python scripts/window_repeats.py 0 1 2 3"""
import sys, time, math, collections
import os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))   # repo root (scripts/..)
import numpy as np, torch
from oracle import oracle as O
from unmore_b200 import synth
torch.set_num_threads(16)
args = O.make_args()
H, W = 480, 640
def snap(b):
    return (math.floor(float(b[0])), math.floor(float(b[1])), math.ceil(float(b[2])), math.ceil(float(b[3])))
tot_N = tot_D = tot_D_round = 0
for i in [int(a) for a in sys.argv[1:]]:
    t0 = time.time()
    img = synth.make_fields(i, H, W)
    props = torch.as_tensor(synth.make_proposals(i, 4096, H, W), dtype=torch.float64)
    ex = O.existence_checking(img, props)["existence_scores"]
    props = props[ex >= args.class_score_thres]
    cr = O.center_reasoning(img, props, args)
    p_pass, split = cr["proposals_pass_singularity"], cr["splited_new_proposals"]
    if len(split):
        ex2 = O.existence_checking(img, split)["existence_scores"]
        split = split[ex2 >= args.class_score_thres]
    if len(split):
        props = torch.cat((p_pass, O.center_reasoning(img, split, args)["proposals_pass_singularity"]), 0)
    else:
        props = p_pass
    n_in = len(props)
    trace = []
    O.boundary_reasoning(img, props, args, trace=trace)
    exited = set()
    keys = []          # (round, proposal, window) computed with early exit
    per_round_distinct = 0
    for r, (idx, cin, cout, lab) in enumerate(trace):
        seen_r = set()
        for j in range(len(idx)):
            p = int(idx[j])
            if p in exited:
                continue
            w = snap(cin[j])
            if w[2] > w[0] and w[3] > w[1]:
                keys.append((r, p, w)); seen_r.add(w)
            l = float(lab[j])
            if l < 0 or (l == 1 and torch.equal(cout[j], cin[j].to(torch.float32))):
                exited.add(p)
        per_round_distinct += len(seen_r)
    N = len(keys); D = len({k[2] for k in keys})
    first = {}
    for r, p, w in keys:
        first.setdefault(w, p)
    self_hits = sum(1 for r, p, w in keys if first[w] == p) - D   # repeats of a window the same proposal computed first
    rounds_per_prop = collections.Counter(p for _, p, _ in keys)
    print(f"image {i}: refine_in {n_in}, proposal-rounds {N}, distinct windows {D} ({1 - D / max(N,1):.1%} repeats), "
          f"within-round distinct {per_round_distinct} ({1 - per_round_distinct / max(N,1):.1%}), repeats of own window {self_hits}, "
          f"max rounds {max(rounds_per_prop.values()) if keys else 0}, {time.time()-t0:.0f}s", flush=True)
    tot_N += N; tot_D += D; tot_D_round += per_round_distinct
print(f"total: proposal-rounds {tot_N}, distinct {tot_D} ({1 - tot_D / tot_N:.1%} repeats), within-round repeats {1 - tot_D_round / tot_N:.1%}")
