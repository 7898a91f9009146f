#!/usr/bin/env python
"""Benchmark of the hot path on BASELINE.json's metric: RANSAC hyp x corr evals/s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A step = one pass of the whole hot path over one synthetic image pair of
BASELINE config 2 (10,000 correspondences, 30 % outliers, 1 px noise, 65,536
hypotheses): ingest (fillXU) -> hypothesis generation -> Sampson scoring + fused
arg-max -> 4 pose candidates -> cheirality -> linear triangulation.  `value` is
H*N evaluations per second of device time with the pixel correspondences
already in HBM; `e2e` is the same through the C-ABI host entry point
(sfmb200_run_host) with pinned host buffers, copies inside the timed region.
N > 1: one process per GPU (torchrun), pairs sharded across ranks, no data-path
collective (weak scaling); the barrier + max over ranks follows the contract.

The same JSON line also carries, each measured outside the headline region and
bounded to a few seconds: `sustained` (config 2 back to back for >= 2 s with its
own clock samples), `c1` (the reference's dino pair with its own CudaSift matches,
tests/golden/dino_cudasift_000_001.npz), `c3` (1M x 1M, HYPOTHESES sharded over the
N ranks, the (count, index) exchange once through NVLink peer memory -
sfmb200_estimate_e_mg - and once through an NCCL all-reduce; strong scaling),
`c4` (4,096 pairs x 4k x 4k, PAIRS sharded over the N ranks; strong scaling) and
`c5` (full path with 1M triangulated points; the triangulation roofline).

--dump-outputs DIR writes, after the K timed steps, what the last of them left for the caller
(rank 0's pair: the outputs of sfmb200_run_host, read from the device-path handle) as DIR/<name>.npy
in float32 (E, P, points) or float64 (the integer outputs, exact), so that two builds can be compared
output for output: the inputs depend on the arguments only.

--impl reference times the reference's OWN implementation of the path, which is
CUDA (it has no CPU path): its unmodified sources rebuilt for sm_100a as
oracle/_ref/libsfm_ref.so, same config, rank 0 only.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

N_CORR, N_HYP, THR, SEED = 10_000, 65_536, 1e-6, 1237
WORKLOAD = ("BASELINE config 2: synthetic two-view scene, 10,000 correspondences, 30% outliers, 1 px noise, 65,536 hypotheses, "
            "full hot path per pair (ingest, hypgen, scoring+arg-max, pose candidates, cheirality, triangulation)")
FLOP_PER_EVAL = 34.0              # SURVEY.md 8d: 15 FFMA x2 + 3 FMUL + 1 compare
# dram__bytes_read.sum + dram__bytes_write.sum of one score_kernel launch at this config,
# from the ncu --set full capture summarised in profiles/r01_ncu_summary.md
SCORE_TRAFFIC_BYTES_NCU = 2_972_416


def ncu_traffic():
    """DRAM bytes per score_kernel launch from the committed ncu capture (profiles/ncu_traffic.json, written by
    tools/make_profiles.py from the `ncu --set full` report of `python bench.py`); a profiler counter cannot be
    read inside an unprofiled run, so the line names the capture it comes from."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        return int(d["score_kernel_dram_bytes_per_launch"]), d.get("source", "profiles/ncu_traffic.json")
    except Exception:
        return SCORE_TRAFFIC_BYTES_NCU, "profiles/r01_ncu_summary.md"
FP32_NOMINAL_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12     # 74.4


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows, self.proc = [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def dist_setup(gpus: int):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def barrier(world):
    import torch
    import torch.distributed as dist

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def cpu_baseline(O, x, full: bool = True) -> dict:
    """The oracle's C port on the host cores: hypothesis generation (fp64 one-sided
    Jacobi) + fp32 Sampson scoring + arg-max for the whole config-2 step."""
    path = os.path.join(ROOT, "oracle", "_ref", "liboracle_c.so")
    L = C.CDLL(path)
    L.oracle_threads.restype = C.c_int
    cores = L.oracle_threads()
    H = N_HYP if full else N_HYP // 8
    idx = O.sample_indices(SEED, H, len(x))
    fp, ip, dp = C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_double)
    E = np.zeros((H, 9))
    cnt = np.zeros(H, np.int32)
    t0 = time.perf_counter()
    L.oracle_hypotheses_f64(x.ctypes.data_as(fp), len(x), idx.ctypes.data_as(ip), H, E.ctypes.data_as(dp))
    t1 = time.perf_counter()
    E32 = E.astype(np.float32)
    L.oracle_counts_f32(E32.ctypes.data_as(fp), H, x.ctypes.data_as(fp), len(x), C.c_float(THR), cnt.ctypes.data_as(ip))
    best = L.oracle_argmax_first(cnt.ctypes.data_as(ip), H)
    t2 = time.perf_counter()
    return {"value": H * len(x) / (t2 - t0), "unit": "hyp*corr evals/s", "cores": cores, "kind": "port",
            "sample": f"one config-2 estimateE step: {H} hypotheses x {len(x)} correspondences "
                      f"(hypgen {t1 - t0:.2f} s + scoring/arg-max {t2 - t1:.2f} s), oracle/oracle_c.c with OpenMP",
            "best_inliers": int(cnt[best])}


def cv2_baseline(scene, K) -> dict | None:
    """OpenCV findEssentialMat(RANSAC) + recoverPose + triangulatePoints on the host
    cores (BASELINE.md 2b): ms/pair only - its iteration count is not observable."""
    try:
        import cv2
    except Exception:
        return None
    p1 = scene["px"][:, :2].astype(np.float64)
    p2 = scene["px"][:, 2:].astype(np.float64)
    Kd = K.astype(np.float64)
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        E, mask = cv2.findEssentialMat(p1, p2, Kd, method=cv2.RANSAC, prob=1 - 1e-12, threshold=2.36, maxIters=N_HYP)
        _, R, t, mask2 = cv2.recoverPose(E, p1, p2, Kd, mask=mask)
        P1 = Kd @ np.eye(3, 4)
        P2 = Kd @ np.hstack([R, t])
        cv2.triangulatePoints(P1, P2, p1.T, p2.T)
        ts.append(time.perf_counter() - t0)
    return {"ms_per_pair": 1e3 * min(ts), "threads": cv2.getNumThreads(), "cores": os.cpu_count(),
            "what": "cv2 4.x findEssentialMat(RANSAC, 5-point, adaptive stop) + recoverPose + triangulatePoints, best of 3",
            "inliers": int(mask.sum())}


def _timed(torch, dist, world, fn, reps):
    """ms per call: barrier + synchronise, CUDA events on the launching stream around ONE call, max over ranks; min over reps."""
    out = []
    for _ in range(reps):
        barrier(world)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out.append(float(t.item()))
    return out


def dump_outputs(out_dir: str, h) -> None:
    """The arrays sfmb200_run_host returns for pair 0 (E, selected pose P, pose index, inlier count, points) plus the
    winning hypothesis' index and the inlier mask, as the last whole-path call left them on the handle."""
    best_idx, best_cnt = h.get_best()
    ind = h.get_pose_index()
    arrays = {"E": h.get_E().reshape(h.pairs, 9), "P": h.get_poses()[np.arange(h.pairs), ind].reshape(h.pairs, 16),
              "pose_index": ind, "inliers": best_cnt, "best_hypothesis": best_idx, "points": h.get_points_host(0)[None],
              "inlier_mask": h.get_inlier_mask().cpu().numpy()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def run_configs(pkg, torch, dist, rank, world, K, Kinv, args) -> dict:
    """BASELINE configs 1, 3, 4, 5 (config 2 is the headline).  Bounded: a few launches each."""
    S = pkg.synthetic
    sh = pkg.sharding
    res = {}
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    scale = float(os.environ.get("SFMB200_BENCH_SCALE", "1.0"))        # < 1 shrinks configs 3-5 (CPU-side dry runs of this file)

    # ---- c3: one pair, 1M correspondences x 1M hypotheses, hypotheses sharded over the ranks (strong scaling) ----
    n3 = H3 = max(int((1 << 20) * scale), 4096)
    sc3 = S.synthetic_pair(n3, seed=1234)                   # replicated: every rank builds the same pair
    d_px3 = torch.from_numpy(sc3["px"]).cuda()
    lo, hi = sh.shard_range(H3, rank, world)
    h = pkg.BatchedPairs(K, Kinv, 1, n3, hi - lo)
    h.set_points_xy(d_px3)
    c3 = {"workload": f"1 pair, {n3} correspondences x {H3} hypotheses, hypotheses sharded over {world} GPU(s): rank r generates and scores "
                      "its contiguous slice against the replicated correspondences; one 8-byte (count, index) key per pair is exchanged",
          "n": n3, "H": H3, "scaling": "strong", "evals": n3 * H3}
    winners = {}
    for name in ("p2p", "nccl"):
        try:
            if name == "p2p":
                sh.connect_peers(h, rank, world)
                step = lambda: sh.estimate_e_p2p(h, H3, SEED, THR)          # noqa: E731
            else:
                step = lambda: sh.estimate_e_sharded(h, H3, SEED, THR, rank, world)   # noqa: E731
            step()
            ms = _timed(torch, dist, world, step, 2)
            idx, cnt = h.get_best()
            E = torch.from_numpy(h.get_E()).cuda()
            same = True
            if world > 1:                                   # every rank must hold the same winner and the same E bits
                Es = [torch.empty_like(E) for _ in range(world)]
                dist.all_gather(Es, E)
                same = all(torch.equal(Es[0], e) for e in Es)
            winners[name] = (int(idx[0]), int(cnt[0]))
            c3[name] = {"ms": min(ms), "ms_all": ms, "evals_per_s": n3 * H3 / (min(ms) * 1e-3), "winner_index": int(idx[0]),
                        "winner_inliers": int(cnt[0]), "all_ranks_same_E_bits": bool(same),
                        "exchange": "keys + E pushed into every peer's buffer by system-scope atomics over NVLink peer memory (csrc/mg.cu), no collective call"
                        if name == "p2p" else "dist.all_reduce(MAX) of the 8-byte packed key over NCCL, winner regenerated locally from its index",
                        "timeouts": sh.p2p_timeouts(h) if name == "p2p" else None}
        except Exception as e:  # noqa: BLE001
            c3[name] = {"error": repr(e)}
    c3["same_winner_both_exchanges"] = len(set(winners.values())) == 1 if len(winners) == 2 else None
    c3["plan"] = h.score_plan()
    res["c3"] = c3
    h.close()

    # ---- c5: full path on one pair with 1M correspondences, all triangulated (replicas: rank 0's number is reported) ----
    H5 = 65536
    h = pkg.BatchedPairs(K, Kinv, 1, n3, H5)
    h.run_device(d_px3, H5, SEED, THR)
    step_ms = _timed(torch, dist, world, lambda: h.run_device(d_px3, H5, SEED, THR), 3)
    tri = []
    for i in range(24):                                     # the triangulation launch alone, L2 flushed before each
        flush.fill_(i & 0xFF)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        h.triangulate()
        b.record()
        torch.cuda.synchronize()
        tri.append(a.elapsed_time(b))
    tri = sorted(tri[4:])
    tri_iso_ms = tri[len(tri) // 2]
    # what the same event pair reads around the smallest possible launch (its floor is inside the isolated figure above)
    tiny = torch.zeros(32, device="cuda")
    floor = []
    for i in range(24):
        torch.cuda._sleep(100000)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        tiny.fill_(1.0)
        b.record()
        torch.cuda.synchronize()
        floor.append(a.elapsed_time(b))
    floor_ms = sorted(floor)[len(floor) // 2]
    # the launch duration proper: launches back to back inside ONE event pair, rotating over 12 point sets of the same size -
    # a set is touched again after 11 x 32 MB of other traffic (inputs larger than L2, no flush kernel in between); a spin kernel
    # in front keeps the host ahead of the device
    SETS, LAUNCHES = 12, 120
    hs = [h]
    for k in range(SETS - 1):
        hk = pkg.BatchedPairs(K, Kinv, 1, n3, 4096)
        hk.run_device(d_px3, 4096, SEED + 1 + k, THR)
        hs.append(hk)
    for hk in hs:
        hk.triangulate()
    torch.cuda.synchronize()
    b2b = []
    for rep in range(5):
        torch.cuda._sleep(2000000)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(LAUNCHES):
            hs[i % SETS].triangulate()
        b.record()
        torch.cuda.synchronize()
        b2b.append(a.elapsed_time(b) / LAUNCHES)
    tri_ms = sorted(b2b)[len(b2b) // 2]
    for hk in hs[1:]:
        hk.close()
    pts = h.get_points_host()
    inl = h.get_inlier_mask().cpu().numpy().astype(bool)
    res["c5"] = {"workload": f"full path, 1 pair, {n3} correspondences, {H5} hypotheses, all {n3} points triangulated", "n": n3, "H": H5,
                 "ms_per_pair": min(step_ms), "tri_ms": tri_ms, "tri_ms_runs": b2b, "tri_points_per_s": n3 / (tri_ms * 1e-3),
                 "tri_gbs": 32.0 * n3 / (tri_ms * 1e-3) / 1e9,
                 "tri_method": f"{LAUNCHES} launches back to back in one CUDA-event pair, rotating over {SETS} point sets "
                               f"({SETS} x {32 * n3 / 1e6:.1f} MB, {'larger' if SETS * 32 * n3 > 126e6 else 'NOT larger'} than the 126 MB L2)",
                 "tri_isolated_ms": tri_iso_ms, "tri_isolated_ms_min": tri[0], "tri_isolated_gbs": 32.0 * n3 / (tri_iso_ms * 1e-3) / 1e9,
                 "tri_isolated_method": "one launch per event pair, L2 flushed (256 MiB write) before each",
                 "event_pair_floor_ms": floor_ms, "inliers": int(inl.sum()),
                 "inliers_in_front_of_camera_1": float(np.mean(pts[2][inl] > 0)) if inl.any() else None}
    h.close()
    del d_px3

    # ---- c4: 4,096 pairs x 4,096 correspondences x 4,096 hypotheses, pairs sharded over the ranks (strong scaling) ----
    pairs, n4, H4 = max(int(4096 * scale), world), 4096, 4096
    lo, hi = sh.shard_range(pairs, rank, world)
    mine = hi - lo
    base = [S.synthetic_pair(n4, seed=500 + i)["px"] for i in range(8)]
    d_base = torch.from_numpy(np.stack(base)).cuda()
    d_px4 = d_base[torch.arange(lo, hi, device="cuda") % 8].contiguous()        # pair p = scene p mod 8, its own sample seed
    h = pkg.BatchedPairs(K, Kinv, mine, n4, H4)
    step = lambda: h.run_device(d_px4, H4, 99 + lo, THR, n=n4)                  # noqa: E731
    step()
    ms = _timed(torch, dist, world, step, 3)
    t = min(ms)
    res["c4"] = {"workload": f"{pairs} pairs x {n4} correspondences x {H4} hypotheses, full path per pair, pairs sharded over {world} GPU(s), "
                             "no data-path collective", "pairs": pairs, "n": n4, "H": H4, "scaling": "strong", "ms": t, "ms_all": ms,
                 "pairs_per_s": pairs / (t * 1e-3), "evals_per_s": pairs * n4 * H4 / (t * 1e-3), "hypotheses_per_s_whole_path": pairs * H4 / (t * 1e-3),
                 "inliers_first_pairs_rank0": [int(v) for v in h.get_best()[1][:4]], "plan": h.score_plan()}
    h.close()
    del d_px4, d_base

    # ---- c1: the reference's dino pair with its own CudaSift matches (rank 0 only; ~2k correspondences, H = N/8) ----
    fx = os.path.join(ROOT, "tests", "golden", "dino_cudasift_000_001.npz")
    if rank == 0 and os.path.exists(fx):
        g = np.load(fx)
        px1 = np.ascontiguousarray(g["px"])
        n1, H1 = len(px1), len(g["idx"])
        K1, K1inv = S.reference_K(int(g["image_wh"][0]), int(g["image_wh"][1]))
        d_px1 = torch.from_numpy(px1).cuda()
        d_idx1 = torch.from_numpy(np.ascontiguousarray(g["idx"])).cuda()
        h = pkg.BatchedPairs(K1, K1inv, 1, n1, H1)

        def staged():                                       # the five calls main.cpp makes (src/main.cpp:298-307), exported rows
            h.set_points_xy(d_px1)
            h.estimate_e(H1, 0, THR, d_idx=d_idx1)
            h.pose_candidates()
            h.choose_pose()
            h.triangulate()
        dev = {}
        for name, fn in (("staged_calls_fixture_rows", staged), ("run_device", lambda: h.run_device(d_px1, H1, SEED, THR))):
            for _ in range(5):
                fn()
            ts = []
            for i in range(40):
                flush[: 1 << 20].fill_(i & 0xFF)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            dev[name] = sorted(ts)[len(ts) // 2]
        # the same single-launch call with the stream kept busy by a ~100 us spin kernel while the host submits: the event pair then
        # holds device time only (above, an idle GPU waits for the host to get from record() to the launch: ~10 us of Python + driver)
        ts = []
        for i in range(40):
            flush[: 1 << 20].fill_(i & 0xFF)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(200000)
            a.record()
            h.run_device(d_px1, H1, SEED, THR)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        dev["run_device_stream_busy"] = sorted(ts)[len(ts) // 2]
        staged()
        bi, bc = h.get_best()
        hp1 = torch.from_numpy(px1).pin_memory().numpy()
        out1 = {"E": np.empty((1, 9), np.float32), "P": np.empty((1, 16), np.float32), "pose_index": np.empty(1, np.int32),
                "inliers": np.empty(1, np.int32), "points": torch.empty((1, 4, n1), dtype=torch.float32).pin_memory().numpy()}
        run1, _ = h.prepare_run_host(hp1, H1, SEED, THR, out=out1)
        for _ in range(5):
            run1()
        ts = []
        for _ in range(40):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run1()
            ts.append(time.perf_counter() - t0)
        ref_ms = [float(v) for v in g["ref_ms"]]
        res["c1"] = {"workload": f"data/dino viff.000/001, the reference's own CudaSift matches: {n1} correspondences, {H1} hypotheses (N/8), 1 GPU",
                     "n": n1, "H": H1, "device_ms_per_pair": dev, "e2e_ms_per_pair": 1e3 * sorted(ts)[len(ts) // 2],
                     "winner": [int(bi[0]), int(bc[0])], "winner_fixture_fp64": [int(g["best"]), int(g["counts"].max())],
                     "reference_rebuilt_b200_ms": {"estimateE": ref_ms[0], "computePosecandidates": ref_ms[1], "choosePose_first_call": ref_ms[2],
                                                   "linear_triangulation": ref_ms[3], "source": "tests/golden/make_dino_cudasift_fixture.py (oracle/_ref/libsfm_ref.so on a B200)"},
                     "reference_published_1080ti_ms": {"hot_path_total": 38.92, "estimateE": 24.12, "source": "BASELINE.md section 1"}}
        h.close()
    del flush
    torch.cuda.empty_cache()
    return res


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank, world, local = dist_setup(args.gpus)
    pkg = entry.load_package()           # the checker (oracle/) is loaded by the baseline legs only
    K, Kinv = pkg.synthetic.reference_K()
    # pairs sharded across ranks: each rank owns its own synthetic pair (weak scaling)
    scene = pkg.synthetic.synthetic_pair(N_CORR, 0.3, 1.0, seed=1234 + 10 * rank)
    px = scene["px"]
    d_px = torch.from_numpy(px).cuda()
    h_px = torch.from_numpy(px).pin_memory()
    h = pkg.BatchedPairs(K, Kinv, 1, N_CORR, N_HYP)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")     # > 126 MB L2

    def step():
        h.run_device(d_px, N_HYP, SEED, THR)

    def timed_region(steps):
        """K steps, each bracketed by CUDA events on the launching stream, L2 flushed between steps
        (outside the events); returns the summed device time in ms, max over ranks."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier(world)
        for i in range(steps):
            ev[i][0].record()
            step()
            ev[i][1].record()
            flush.fill_(i & 0xFF)
        barrier(world)
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    h.set_option(4, 0)           # the timed region runs WITHOUT the per-stage events: 8 event records per step
                                 # between the kernels cost ~25 us of a 0.42 ms step (tools/event_overhead.py)
    for _ in range(max(args.warmup, 3)):
        step()
        flush.fill_(1)
    launches0 = h.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    wall0 = time.perf_counter()
    total_ms = timed_region(args.steps)
    wall = time.perf_counter() - wall0
    launches = h.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, h)
    ms_per_step = total_ms / args.steps
    value = world * N_HYP * N_CORR / (ms_per_step * 1e-3)
    # second region, same K steps of the same workload, WITH the per-stage CUDA events (recorded on the
    # handle's stream = torch's current stream): per-kernel durations for the roofline and stage_ms
    h.set_option(4, 1)
    for _ in range(3):
        step()
        flush.fill_(1)
    h.set_option(4, 1)           # reset the stage ring
    staged_ms = timed_region(args.steps) / args.steps
    clocks = sampler.stop()
    stage = h.stage_times()
    stage_ms = stage.mean(axis=0) if len(stage) else np.zeros(7)
    best_idx, best_cnt = h.get_best()
    plan_main = h.score_plan()
    # hypothesis generation with the other null-vector solver (9x9 Jacobi eigensolve), outside the timed region
    h.set_option(5, 0)
    h.set_option(4, 1)
    for _ in range(10):
        step()
        flush.fill_(3)
    jac = h.stage_times()
    hypgen_jacobi_ms = float(jac[2:, 1].mean()) if len(jac) > 2 else None
    h.set_option(5, 1)
    h.set_option(4, 0)

    # ---- end to end through the C-ABI host call: pinned H2D + D2H inside ----
    out = {"E": np.empty((1, 9), np.float32), "P": np.empty((1, 16), np.float32), "pose_index": np.empty(1, np.int32),
           "inliers": np.empty(1, np.int32), "points": torch.empty((1, 4, N_CORR), dtype=torch.float32).pin_memory().numpy()}
    hp = h_px.numpy()
    run_host, _ = h.prepare_run_host(hp, N_HYP, SEED, THR, out=out)     # same C-ABI call, argument marshalling done once
    for _ in range(3):
        run_host()
    barrier(world)
    e2e_t = []
    for i in range(args.steps):
        flush.fill_(i & 0xFF)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run_host()                                    # sfmb200_run_host: returns after its own stream sync
        e2e_t.append(time.perf_counter() - t0)
    e2e_total = torch.tensor([sum(e2e_t)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_total, op=dist.ReduceOp.MAX)
    e2e_ms = float(e2e_total.item()) * 1e3 / args.steps
    h2d = px.nbytes
    d2h = 9 * 4 + 16 * 4 + 4 + 4 + 4 * N_CORR * 4

    h2d_pageable = None
    if rank == 0:
        # the same call with PAGEABLE caller buffers: staged through the copy engines (api.cu: ingest_xy_host + pack)
        hp_pg = np.array(px, copy=True)
        out_pg = {"E": np.empty((1, 9), np.float32), "P": np.empty((1, 16), np.float32), "pose_index": np.empty(1, np.int32),
                  "inliers": np.empty(1, np.int32), "points": np.empty((1, 4, N_CORR), np.float32)}
        run_pg, _ = h.prepare_run_host(hp_pg, N_HYP, SEED, THR, out=out_pg)
        for _ in range(3):
            run_pg()
        ts = []
        for i in range(min(args.steps, 50)):
            flush.fill_(i & 0xFF)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run_pg()
            ts.append(time.perf_counter() - t0)
        h2d_pageable = 1e3 * sum(ts) / len(ts)

    # ---- sustained: config 2 back to back for >= 2 s (same step, same flush, same events), its own clock samples ----
    sus_steps = int(min(max(2000.0 / max(ms_per_step + 0.06, 1e-3), args.steps), 20000))
    sus_sampler = ClockSampler(local)
    sus_sampler.start()
    sus_wall0 = time.perf_counter()
    sus_ms = timed_region(sus_steps) / sus_steps
    sus_wall = time.perf_counter() - sus_wall0
    sus_clocks = sus_sampler.stop()
    h.close()
    del flush
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs (all ranks take part; rank 0 reports) ----
    extra = {} if args.no_extras else run_configs(pkg, torch, dist, rank, world, K, Kinv, args)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    # ---- rank 0: roofline, probes, CPU baselines, JSON line ----
    lib = pkg.load_library()
    build_info = lib.raw("sfmb200_build_info")().decode()
    try:
        import importlib.util as _ilu
        _sp = _ilu.spec_from_file_location("sfmb200_build", os.path.join(ROOT, "cuda-sfm_b200", "build.py"))
        _b = _ilu.module_from_spec(_sp)
        _sp.loader.exec_module(_b)
        tree_hash = _b.source_hash()
    except Exception:
        tree_hash = None
    score_plan = plan_main
    probe = {}
    for mode, name in ((0, "ffma"), (1, "ffma2")):
        fmas, ms = C.c_double(), C.c_float()
        lib.call("sfmb200_fma_probe", mode, 2000, C.byref(fmas), C.byref(ms))
        probe[name + "_tflops"] = 2 * fmas.value / (ms.value * 1e-3) / 1e12
    peaks = measured_peaks()
    traffic, traffic_src = ncu_traffic()
    score_ms = float(stage_ms[2])
    achieved = FLOP_PER_EVAL * N_HYP * N_CORR / (score_ms * 1e-3) / 1e12 if score_ms > 0 else None
    fp32_probe = max(probe.values())
    roofline = {
        "kernel": "score_kernel (Sampson scoring + fused arg-max)", "bound": "fp32",
        "achieved": achieved, "peak": FP32_NOMINAL_TFLOPS, "unit": "TFLOP/s",
        "frac": achieved / FP32_NOMINAL_TFLOPS if achieved else None,
        "peak_source": "nominal 148 SM x 128 lanes x 2 x 1.965 GHz (MEASURED_PEAKS.json has HBM and bf16 only; "
                       "this kernel is FP32 CUDA-core bound, not hbm/tensor)",
        "peak_measured_probe": fp32_probe, "frac_of_measured_probe": achieved / fp32_probe if achieved else None,
        "probe": probe, "flop_per_eval": FLOP_PER_EVAL, "evals_per_launch": N_HYP * N_CORR,
        "kernel_ms": score_ms, "kernel_share_of_step": score_ms / ms_per_step if ms_per_step else None, "evals_per_s_kernel": N_HYP * N_CORR / (score_ms * 1e-3) if score_ms > 0 else None,
        "traffic": traffic, "traffic_unit": "bytes per launch: dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the ncu --set full "
                                             "capture of this command (" + traffic_src + "); algorithmic input 2.36 MB of E candidates + 0.32 MB of points",
    }
    hbm = peaks.get("hbm_gbs", 6650.0)
    c5 = extra.get("c5") or {}
    tri_ms = c5.get("tri_ms")
    tri = {"kernel": "triangulate_kernel", "bound": "hbm", "achieved": c5.get("tri_gbs"),
           "peak": hbm, "unit": "GB/s", "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback",
           "bytes_per_point": 32, "points_per_launch": c5.get("n"), "kernel_ms": tri_ms,
           "method": c5.get("tri_method"),
           "isolated_launch": {"kernel_ms": c5.get("tri_isolated_ms"), "achieved": c5.get("tri_isolated_gbs"),
                               "frac": (c5.get("tri_isolated_gbs") / hbm) if c5.get("tri_isolated_gbs") else None,
                               "method": c5.get("tri_isolated_method"), "event_pair_floor_ms": c5.get("event_pair_floor_ms")},
           "note": "BASELINE config 5: 1,048,576 points per launch (32 MB of traffic). kernel_ms is the average launch duration of a "
                   "stream of such launches over inputs larger than L2; isolated_launch is ONE launch between its own two events after an "
                   "L2 flush - that figure contains event_pair_floor_ms, what the same event pair reads around an empty launch. "
                   f"The 10k-point launch inside a config-2 step is launch-latency bound ({float(stage_ms[6]) * 1e3:.1f} us)"}
    tri["frac"] = tri["achieved"] / hbm if tri["achieved"] else None
    cpu = cv2b = None
    if world == 1:                       # CPU baselines: N = 1 only (at N > 1 the other ranks would idle behind them)
        O = entry.load_oracle()          # cpu_baseline leg: the oracle port timed on the host cores
        x = O.normalise_points(px, Kinv)
        cpu = cpu_baseline(O, x)
        cv2b = cv2_baseline(scene, K)
    line = {
        "metric": "RANSAC hyp*corr evals/s", "value": value, "unit": "hyp*corr evals/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "pairs_per_step_per_gpu": 1,
                   "parallelism": f"pairs sharded over {world} GPU(s), no data-path collective",
                   "l2": "flushed between timed iterations (256 MiB write)", "threshold": THR, "seed": SEED,
                   "score_plan": score_plan},
        "e2e": {"value": world * N_HYP * N_CORR / (e2e_ms * 1e-3), "unit": "hyp*corr evals/s", "ms_per_pair": e2e_ms,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "sfmb200_run_host (C ABI), pinned host buffers (read and written by the kernels through their "
                       "device-visible aliases: the bytes cross PCIe inside the timed call), host wall clock around the call"},
        "gpu_launches": int(launches), "launches_per_step": launches / args.steps,
        "stage_ms": {k: float(v) for k, v in zip(pkg.BatchedPairs.STAGES, stage_ms)},
        "stage_timing": {"how": "second region of the same K steps with 8 CUDA events per step on the launching stream "
                                "(the timed region for `value` runs without them: they cost ~25 us per step)",
                         "ms_per_step_with_stage_events": staged_ms},
        "hypotheses_per_s": N_HYP / (float(stage_ms[1]) * 1e-3) if stage_ms[1] > 0 else None,
        "hypgen_solvers": {"default": "8x8 Cholesky projector", "projector_ms": float(stage_ms[1]), "jacobi_9x9_ms": hypgen_jacobi_ms,
                           "jacobi_hypotheses_per_s": N_HYP / (hypgen_jacobi_ms * 1e-3) if hypgen_jacobi_ms else None},
        "e_estimate_ms_per_pair": float(stage_ms[1] + stage_ms[2] + stage_ms[3]),
        "pairs_per_s": world / (ms_per_step * 1e-3),
        "result": {"best_hypothesis": int(best_idx[0]), "inliers": int(best_cnt[0]), "pose_index": int(out["pose_index"][0])},
        "roofline": roofline, "roofline_triangulation": tri, "cpu_baseline": cpu, "cv2_baseline": cv2b,
        "clocks": clocks, "wall_s_timed_region": wall,
        "library": {"path": os.path.relpath(lib.path, ROOT), "build_info": build_info, "source_tree_hash": tree_hash,
                    "built_from_this_tree": bool(tree_hash and tree_hash in build_info)},
        "sustained": {"what": "the same config-2 step back to back (L2 flushed between steps, CUDA events per step, max over ranks)",
                      "steps": sus_steps, "ms_per_step": sus_ms, "value": world * N_HYP * N_CORR / (sus_ms * 1e-3), "unit": "hyp*corr evals/s",
                      "wall_s": sus_wall, "clocks": sus_clocks},
        **extra,
    }
    line["e2e"]["ms_per_pair_pageable_buffers"] = h2d_pageable
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    O = entry.load_oracle()
    K, Kinv = O.reference_K()
    scene = O.synthetic_pair(N_CORR, 0.3, 1.0, seed=1234)
    px = scene["px"]
    # n_gpus = the N of this launch; the reference is single-GPU, so rank 0 alone runs it (gpus_used = 1)
    base = {"impl": "reference", "metric": "RANSAC hyp*corr evals/s", "unit": "hyp*corr evals/s", "n_gpus": max(args.gpus, 1),
            "gpus_used": 1, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    path = os.path.join(ROOT, "oracle", "_ref", "libsfm_ref.so")
    if not (os.path.exists(path) and torch.cuda.is_available()):
        # no rebuilt reference (or no GPU for its CUDA-only path): time the oracle port instead
        x = O.normalise_points(px, Kinv)
        cpu = cpu_baseline(O, x)
        line = dict(base, value=cpu["value"], steps=1, warmup=0, ms_per_step=1e3 * N_HYP * N_CORR / cpu["value"],
                    config={"workload": WORKLOAD, "pairs_per_step_per_gpu": 1, "threshold": THR, "seed": SEED,
                            "note": "estimateE on the host cores (oracle port; oracle/_ref/libsfm_ref.so or GPU missing)"},
                    cpu_baseline=cpu, e2e={"value": cpu["value"], "unit": base["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
        emit(line)
        return
    if not args.ref_child:
        # The reference exit()s the process on any CUDA error (common.cu:14) and its as-built path reads uninitialised memory
        # (SURVEY Q9-Q13), so a run of it can die: it runs in a child process, is retried, and only then replaced by the port.
        import subprocess
        last = ""
        ATTEMPTS = 6
        for attempt in range(ATTEMPTS):
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--ref-child", "--gpus", str(args.gpus),
                                "--steps", str(args.steps), "--warmup", str(args.warmup)], capture_output=True, text=True,
                               env=dict(os.environ, RANK="0", WORLD_SIZE="1"))
            rows = [l for l in r.stdout.splitlines() if l.startswith("{")]
            if r.returncode == 0 and rows:
                line = json.loads(rows[-1])
                line["attempts"] = attempt + 1          # attempts - 1 children died in the reference's own code (see stderr)
                if attempt:
                    line["died_before"] = last
                emit(line)
                return
            last = (r.stderr.strip().splitlines() or ["no output"])[-1][:200]
            sys.stderr.write(f"[bench] reference child attempt {attempt + 1} failed (rc {r.returncode}): {last}\n")
        x = O.normalise_points(px, Kinv)
        cpu = cpu_baseline(O, x)
        line = dict(base, value=cpu["value"], steps=1, warmup=0, ms_per_step=1e3 * N_HYP * N_CORR / cpu["value"],
                    config={"workload": WORKLOAD, "pairs_per_step_per_gpu": 1, "threshold": THR, "seed": SEED,
                            "note": f"estimateE on the host cores (oracle port): the reference's CUDA path died {ATTEMPTS} times in a row on this box ({last})"},
                    cpu_baseline=cpu, e2e={"value": cpu["value"], "unit": base["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
        emit(line)
        return
    if os.environ.get("SFMB200_BENCH_REF_CRASH"):       # test hook: the child dies the way the reference's checkCUDAError does
        sys.stderr.write("CUDA error (test hook): simulated\n")
        os._exit(1)
    torch.cuda.set_device(0)
    L = C.CDLL(path)
    L.ref_create.restype = C.c_void_p
    for name in ("ref_estimateE_injected", "ref_computePosecandidates", "ref_choosePose", "ref_linear_triangulation"):
        getattr(L, name).restype = C.c_float
    fp, ip = C.POINTER(C.c_float), C.POINTER(C.c_int32)
    r = C.c_void_p(L.ref_create(K.reshape(9).ctypes.data_as(fp), Kinv.reshape(9).ctypes.data_as(fp), N_CORR))
    H = N_HYP
    idx = O.sample_indices(SEED, H, N_CORR)

    def step(Hs):
        t0 = time.perf_counter()
        L.ref_fillXU(r, px.ctypes.data_as(fp))
        t_e = L.ref_estimateE_injected(r, idx.ctypes.data_as(ip), Hs, None)
        t_pc = L.ref_computePosecandidates(r)
        t_cp = L.ref_choosePose(r)
        t_tr = L.ref_linear_triangulation(r)
        return time.perf_counter() - t0, (t_e, t_pc, t_cp, t_tr)

    # bound the run: first step at full size, then shrink the hypothesis sample if K steps would not fit
    t_first, _ = step(H)
    budget = 150.0
    Hs = H
    if t_first * (args.steps + max(args.warmup, 1)) > budget:
        Hs = max(1024, int(H * budget / (t_first * (args.steps + max(args.warmup, 1)))) // 1024 * 1024)
    for _ in range(max(args.warmup, 1)):
        step(Hs)
    ts, stages = [], []
    for _ in range(args.steps):
        t, st = step(Hs)
        ts.append(t)
        stages.append(st)
    ms = 1e3 * sum(ts) / len(ts)
    value = Hs * N_CORR / (ms * 1e-3)
    st = np.mean(np.array(stages), axis=0)
    sample = (f"reference's own CUDA path (SfM/sfm.cu rebuilt unmodified for sm_100a, oracle/ref_harness.cu) on the GPU: "
              f"fillXU + estimateE body with {Hs} of {H} injected hypotheses x {N_CORR} correspondences + "
              f"computePosecandidates + choosePose + linear_triangulation; host wall clock incl. its cudaMalloc/syncs")
    line = dict(base, value=value, steps=args.steps, warmup=max(args.warmup, 1), ms_per_step=ms,
                config={"workload": WORKLOAD, "pairs_per_step_per_gpu": 1, "threshold": THR, "seed": SEED,
                        "hypotheses_per_step": Hs, "first_full_size_step_s": t_first},
                stage_ms={"estimateE": float(st[0]), "computePosecandidates": float(st[1]), "choosePose": float(st[2]),
                          "linear_triangulation": float(st[3])},
                cpu_baseline={"value": value, "unit": base["unit"], "cores": 1, "kind": "reference", "sample": sample,
                              "note": "the reference has no CPU path (README.md:12); this is its CUDA path on the same B200"},
                e2e={"value": value, "unit": base["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    emit(line)
    L.ref_destroy(r)


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line of the contract, written to the process's real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # stdout carries exactly one JSON line.  Libraries write there too (NCCL prints its version banner to stdout at
    # NCCL_DEBUG >= VERSION): from here on file descriptor 1 points at stderr and emit() writes to the saved real stdout.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-extras", action="store_true",
                    help="headline config-2 regions only (for profiler captures: skips the sustained run's companions c1, c3, c4, c5)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (--impl ours only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this project's path: use it with --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
