#!/usr/bin/env python
"""Small end-to-end run for compute-sanitizer (memcheck / racecheck / initcheck / synccheck):
every kernel of the path at sizes that exercise partial tiles, partial TMA stages and the
split (atomic) epilogue, in every scoring variant family member used by default."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry

pkg = entry.load_package()
O = pkg.synthetic          # scenes + intrinsics only: no checker code in these tools
K, Kinv = O.reference_K()
for n, H, pairs, variant in ((700, 300, 1, -1), (1100, 2500, 2, -1), (520, 1030, 1, 0), (2049, 700, 1, 6), (600, 2100, 1, 3), (5000, 1500, 1, 10), (300, 40, 2, 10)):
    px = np.stack([O.synthetic_pair(n, seed=3 + b)["px"] for b in range(pairs)])
    h = pkg.BatchedPairs(K, Kinv, pairs, n, H)
    h.set_option(2, variant)
    out = h.run_host(px, H, 11, 1e-6)
    h.set_option(1, 0)
    h.set_option(3, 1)
    out2 = h.run_host(px, H, 11, 1e-6)
    pos = torch.empty((n, 4), device="cuda")
    col = torch.empty((n, 4), device="cuda")
    h.copy_to_vbo(pos, col)
    h.get_E_candidates(); h.get_inlier_counts(); h.get_inlier_mask(); h.get_X(0)
    lo, hi = pkg.sharding.shard_range(H, 1, 2)
    h.estimate_e(hi - lo, 11, 1e-6, H_total=H, h_begin=lo)
    h.adopt_best(H, 11)
    h.synchronize()
    print(n, H, pairs, variant, "inliers", out["inliers"].tolist(), out2["inliers"].tolist(), h.score_plan())
    h.close()
# the 8f stages: filtered ingest is covered by its test; here refit, adaptive termination, homography,
# bundle adjustment and N-view chaining at sizes with partial CTAs
seq = O.synthetic_sequence(3, 1300, seed=8)
h = pkg.BatchedPairs(K, Kinv, 2, 1300, 2048)
h.set_option(1, 0)
h.set_points_xy(torch.from_numpy(seq["px_pairs"]).cuda())
used = h.estimate_e_adaptive(2048, 5, 1e-6, 0.99, 256, 2)
acc = h.refine_e(3)
h.pose_candidates(); h.choose_pose(); h.triangulate()
st = h.bundle_adjust(2, 4)
ch = h.chain_views()
gst = h.bundle_adjust_global(ch, iterations=3)
Hm, cnt = h.find_homography(1500, 3, 5.0)
h.synchronize()
print("8f stages: used", used, "refits", acc.tolist(), "ba inliers", st[:, 6].tolist(), "scales", ch["scales"].tolist(), "global ba", gst[:3].tolist(),
      "h matches", cnt.tolist())
h.close()
# round 2: fused small-problem path (forced on and off), symmetric-epipolar metric, disjoint sampler, batched pipeline, peer exchange
for n, H, pairs in ((2153, 269, 1), (900, 100, 3), (4100, 600, 1)):
    px = np.stack([O.synthetic_pair(n, seed=20 + b)["px"] for b in range(pairs)])
    h = pkg.BatchedPairs(K, Kinv, pairs, n, H)
    for small in (1, 0):
        h.set_option(7, small)
        out = h.run_host(px, H, 5, 1e-6)
        h.set_points_xy(torch.from_numpy(px).cuda())
        h.estimate_e(H, 5, 1e-6)
    h.set_option(9, 1)
    h.run_device(torch.from_numpy(px).cuda(), H, 5, 1e-6)
    h.set_option(9, 0)
    h.set_option(10, 1)
    h.estimate_e(min(H, n // 8), 5, 1e-6)
    h.set_option(10, 0)
    pkg.sharding.connect_peers(h, 0, 1)
    pkg.sharding.estimate_e_p2p(h, H, 5, 1e-6)
    pkg.sharding.estimate_e_p2p(h, H, 6, 1e-6)
    h.synchronize()
    print("round-2 paths", n, H, pairs, "inliers", out["inliers"].tolist(), "timeouts", pkg.sharding.p2p_timeouts(h))
    h.close()
print("sanitize run done")
