#!/usr/bin/env python
"""Device time of batches with a count per pair (the *_ragged entry points) on one GPU.

(a) Overhead of the per-pair walk: config 4 (4,096 pairs x 4,096 correspondences x 4,096 hypotheses) through run_device
    against the same data through run_device_ragged with every count 4,096, alternated.
(b) A ragged batch: 4,096 pairs with counts uniform in [1,024, 7,168], H = 4,096, through run_device_ragged.
(c) What a caller without ragged batches can do: one-pair run_device calls over the first 256 pairs of (b).
Whole-path calls between CUDA events, warm-ups first, the L2 overwritten (256 MiB) before each timed call, as bench.py
does.  Prints one JSON object (and writes it to --out): card name and power limit read in the same process."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

THR, SEED = 1e-6, 99
SEED_STEP = 0x632BE59BD9B4E019


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn, flush, reps, busy=False):
    """Event-pair times of fn.  busy: a ~2 ms spin kernel ahead of the first event keeps the stream occupied while the host
    submits, so the pair holds device time only; otherwise the pair also holds the host's time to submit the call."""
    ts = []
    for i in range(reps):
        flush.fill_(i & 0xFF)
        if busy:
            torch.cuda._sleep(4_000_000)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--single", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = entry.load_package()
    S = pkg.synthetic
    K, Kinv = S.reference_K()
    B, n4, H = args.pairs, 4096, 4096
    res = {"card": card(), "pairs": B, "H": H}
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")      # > 126 MB L2

    # (a) config 4, uniform vs ragged with equal counts (same inputs as bench.py's c4: pair p = scene p mod 8)
    base = np.stack([S.synthetic_pair(7168, seed=500 + i)["px"].astype(np.float32) for i in range(8)])
    d_base = torch.from_numpy(base).cuda()
    d_px4 = d_base[torch.arange(B, device="cuda") % 8, :n4].contiguous()
    off4 = (np.arange(B + 1) * n4).astype(np.int32)
    hu = pkg.BatchedPairs(K, Kinv, B, n4, H)
    hr = pkg.BatchedPairs(K, Kinv, B, n4, H)
    run_u = lambda: hu.run_device(d_px4, H, SEED, THR)                                   # noqa: E731
    run_r = lambda: hr.run_device_ragged(d_px4.view(-1, 4), H, SEED, THR, offsets=off4)  # noqa: E731
    for _ in range(2):
        run_u(); run_r()
    torch.cuda.synchronize()
    tu, tr, du, dr = [], [], [], []
    for _ in range(args.reps):            # alternated: the two share whatever else the host is doing
        tu += timed(run_u, flush, 1)
        tr += timed(run_r, flush, 1)
        du += timed(run_u, flush, 1, busy=True)
        dr += timed(run_r, flush, 1, busy=True)
    same = bool(np.array_equal(hu.get_best()[1], hr.get_best()[1]) and np.array_equal(hu.get_E(), hr.get_E()))
    ev4 = B * n4 * H
    res["a"] = {"uniform_ms": tu, "ragged_ms": tr, "uniform_evals_per_s": ev4 / (min(tu) * 1e-3),
                "ragged_evals_per_s": ev4 / (min(tr) * 1e-3), "overhead_pct_min": 100 * (min(tr) / min(tu) - 1),
                "overhead_pct_median": 100 * (float(np.median(tr)) / float(np.median(tu)) - 1),
                "device_only_uniform_ms": du, "device_only_ragged_ms": dr, "device_only_overhead_pct_min": 100 * (min(dr) / min(du) - 1),
                "same_results": same,
                "plan_uniform": hu.score_plan(), "plan_ragged": hr.score_plan()}
    hu.close(); hr.close()
    del d_px4

    # (b) counts uniform in [1024, 7168]
    rng = np.random.default_rng(7)
    counts = rng.integers(1024, 7169, B).astype(np.int64)
    offb = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    d_pxb = torch.cat([d_base[p % 8, :counts[p]] for p in range(B)]).contiguous()
    hb = pkg.BatchedPairs(K, Kinv, B, 7168, H)
    run_b = lambda: hb.run_device_ragged(d_pxb, H, SEED, THR, offsets=offb)               # noqa: E731
    for _ in range(2):
        run_b()
    tb = timed(run_b, flush, args.reps)
    db = timed(run_b, flush, args.reps, busy=True)
    evb = int(counts.sum()) * H
    res["b"] = {"counts_sum": int(counts.sum()), "counts_min": int(counts.min()), "counts_max": int(counts.max()), "ms": tb,
                "evals_per_s": evb / (min(tb) * 1e-3), "vs_a_uniform_pct": 100 * (evb / min(tb)) / (ev4 / min(tu)) - 100,
                "device_only_ms": db, "device_only_evals_per_s": evb / (min(db) * 1e-3),
                "device_only_vs_a_uniform_pct": 100 * (evb / min(db)) / (ev4 / min(du)) - 100,
                "plan": hb.score_plan()}
    best_b = hb.get_best()[1][: args.single].copy()
    hb.close()

    # (c) one-pair run_device calls over the first pairs of (b), each with that pair's batch seed
    h1 = pkg.BatchedPairs(K, Kinv, 1, 7168, H)
    singles = [d_base[p % 8, :counts[p]][None].contiguous() for p in range(args.single)]
    seeds = [(SEED + SEED_STEP * p) % (1 << 64) for p in range(args.single)]

    def run_c():
        for p in range(args.single):
            h1.run_device(singles[p], H, seeds[p], THR)
    run_c()
    tc = timed(run_c, flush, 3)
    h1.run_device(singles[-1], H, seeds[-1], THR)
    evc = int(counts[: args.single].sum()) * H
    res["c"] = {"pairs": args.single, "ms": tc, "ms_per_pair": min(tc) / args.single, "evals_per_s": evc / (min(tc) * 1e-3),
                "b_ms_per_pair": min(tb) / B, "last_pair_matches_batch": int(h1.get_best()[1][0]) == int(best_b[-1])}
    h1.close()
    del flush
    out = json.dumps(res)
    print(out)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
