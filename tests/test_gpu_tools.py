"""GPU tier: the multi-config tool (tools/configs.py) runs at reduced scale in one process."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_configs_tool_small_scale():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "configs.py"), "c3", "c4", "c5", "--scale", "0.004", "--reps", "1"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [json.loads(l) for l in r.stdout.strip().splitlines() if l.startswith("{")]
    assert [l["config"] for l in lines] == ["c3", "c4", "c5"]
    assert lines[0]["inliers"] > 0 and lines[1]["pairs"] == 16 and lines[2]["tri_points_per_s"] > 0


def test_coloured_vbo(pkg, O):
    """Egress with colours (SURVEY 8f rank 4): positions as copyBoidsToVBO (scaled), colours by inlier status or depth."""
    import numpy as np
    import torch

    K, Kinv = O.reference_K()
    n = 1500
    sc = O.synthetic_pair(n, seed=21)
    h = pkg.BatchedPairs(K, Kinv, 1, n, 2048)
    h.set_option(1, 0)
    h.run_device(torch.from_numpy(sc["px"][None]).cuda(), 2048, 4, 1e-6)
    pos, col = torch.empty((n, 4), device="cuda"), torch.empty((n, 4), device="cuda")
    X = h.get_points_host(0)
    mask = h.get_inlier_mask().cpu().numpy().astype(bool)
    h.copy_to_vbo_coloured(pos, col, scale=2.0, mode=1)
    assert np.array_equal(pos.cpu().numpy(), np.c_[2.0 * X[:3].T, np.ones(n, np.float32)])
    c = col.cpu().numpy()
    assert np.all(c[mask] == [0, 1, 0, 1]) and np.all(c[~mask] == [1, 0, 0, 1])
    h.copy_to_vbo_coloured(pos, col, mode=2, z_near=4.0, z_far=8.0)
    c = col.cpu().numpy()
    front = X[2] > 0
    t = np.clip((X[2] - 4.0) / 4.0, 0, 1).astype(np.float32)
    assert np.allclose(c[front], np.c_[t, np.zeros(n), 1 - t, np.ones(n)][front], atol=1e-6)
    assert np.all(c[~front] == [0.5, 0.5, 0.5, 1])
    h.copy_to_vbo_coloured(pos, col, mode=0)
    ref_pos, ref_col = torch.empty((n, 4), device="cuda"), torch.empty((n, 4), device="cuda")
    h.copy_to_vbo(ref_pos, ref_col)
    assert torch.equal(pos, ref_pos) and torch.equal(col, ref_col)
    with pytest.raises(Exception):
        h.copy_to_vbo_coloured(pos, col, mode=3)
    h.close()


def test_run_host_pinned_zero_copy_equals_staged(pkg, O):
    """sfmb200_run_host reads / writes page-locked buffers through their device aliases and stages pageable ones:
    both routes give the same bits, and the prepared call equals the plain one."""
    import numpy as np
    import torch

    K, Kinv = O.reference_K()
    n, H = 3000, 2048
    px = np.stack([O.synthetic_pair(n, seed=70 + b)["px"] for b in range(2)])
    h = pkg.BatchedPairs(K, Kinv, 2, n, H)
    a = h.run_host(px.copy(), H, 9, 1e-6)                                   # pageable in, pageable out
    pin_in = torch.from_numpy(px).pin_memory()
    out = {"E": np.empty((2, 9), np.float32), "P": np.empty((2, 16), np.float32), "pose_index": np.empty(2, np.int32),
           "inliers": np.empty(2, np.int32), "points": torch.zeros((2, 4, n), dtype=torch.float32).pin_memory().numpy()}
    b = h.run_host(pin_in.numpy(), H, 9, 1e-6, out=out)                     # pinned in, pinned out (zero copy)
    for k in ("E", "P", "pose_index", "inliers", "points"):
        assert np.array_equal(a[k], b[k]), k
    call, out2 = h.prepare_run_host(pin_in.numpy(), H, 9, 1e-6)             # pinned in, pageable out
    call(); call()
    for k in ("E", "P", "pose_index", "inliers", "points"):
        assert np.array_equal(a[k], out2[k]), k
    h.close()


def test_whole_path_is_cuda_graph_capturable(pkg, O):
    """run_device only enqueues kernels on the handle's stream (no allocation, no synchronisation), so a caller can
    capture it in a CUDA graph; replay gives the same bits (tools/graph_check.py: -19 % at config-1 sizes)."""
    import numpy as np
    import torch

    K, Kinv = O.reference_K()
    n, H = 2000, 250
    d_px = torch.from_numpy(O.synthetic_pair(n, seed=5)["px"][None]).cuda()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        h = pkg.BatchedPairs(K, Kinv, 1, n, H)
        for _ in range(2):
            h.run_device(d_px, H, 7, 1e-6)
        s.synchronize()
        ref = (h.get_best()[0].copy(), h.get_E().copy(), h.get_points_host(0).copy())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            h.run_device(d_px, H, 7, 1e-6)
        h.set_E(np.zeros((1, 9), np.float32))          # perturb the state, then let the replay restore it
        for _ in range(3):
            g.replay()
        s.synchronize()
        got = (h.get_best()[0], h.get_E(), h.get_points_host(0))
        assert all(np.array_equal(a, b) for a, b in zip(ref, got))
        h.close()


def test_bench_json_contract_reduced_extras(tmp_path):
    """bench.py prints ONE JSON line with the contract's keys; the extra configs run at a reduced scale here
    (SFMB200_BENCH_SCALE shrinks configs 3-5 only: the headline config 2 is always full size).  --dump-outputs writes
    the last timed step's outputs, and they agree with what the line reports."""
    import numpy as np

    env = dict(os.environ, SFMB200_BENCH_SCALE="0.01")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "5", "--warmup", "3", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    out = [l for l in r.stdout.strip().splitlines() if l.strip()]
    assert len(out) == 1, out[:3]
    d = json.loads(out[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks", "sustained", "c1", "c3", "c4", "c5", "library"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 5 and d["dtype"] == "f32" and "workload" in d["config"] and d["vs_baseline"] is None
    assert d["value"] > 1e12 and d["e2e"]["value"] > 1e12 and d["e2e"]["h2d_bytes_per_step"] == 160000 and d["gpu_launches"] == 25
    rf = d["roofline"]
    assert 0.5 < rf["frac"] < 1.0 and rf["traffic"] > 2e6 and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] > 0
    assert d["library"]["built_from_this_tree"] is True
    assert d["c3"]["same_winner_both_exchanges"] is True and d["c3"]["p2p"]["timeouts"] == 0
    assert d["c1"]["winner"] == d["c1"]["winner_fixture_fp64"] or abs(d["c1"]["winner"][1] - d["c1"]["winner_fixture_fp64"][1]) <= 3
    assert d["roofline_triangulation"]["frac"] is not None and d["c4"]["pairs"] >= 1
    assert d["sustained"]["wall_s"] >= 1.5 and not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    o = {k: np.load(tmp_path / f"{k}.npy") for k in ("E", "P", "pose_index", "inliers", "best_hypothesis", "points", "inlier_mask")}
    assert all(a.dtype in (np.float32, np.float64) for a in o.values())
    assert o["E"].shape == (1, 9) and o["P"].shape == (1, 16) and o["points"].shape == (1, 4, 10000) and o["inlier_mask"].shape == (10000,)
    res = d["result"]
    assert int(o["inliers"][0]) == int(o["inlier_mask"].sum()) == res["inliers"]
    assert int(o["best_hypothesis"][0]) == res["best_hypothesis"] and int(o["pose_index"][0]) == res["pose_index"]
    assert np.all(o["points"][0, 3] == 1)
    # the same arguments again (the companion configs run after the dump, so they are left out): the same outputs, bit for bit
    again = tmp_path / "again"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "5", "--warmup", "3", "--no-extras", "--dump-outputs", str(again)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    for k, a in o.items():
        assert np.array_equal(np.load(again / f"{k}.npy"), a), k


def test_bench_reference_arm_survives_a_dying_reference():
    """bench.py --impl reference: the reference's CUDA path exit()s its process on any CUDA error (common.cu:14), so it runs in a
    child that is retried; when every attempt dies the arm still prints its ONE line, from the oracle port, and says why."""
    ref = os.path.join(ROOT, "oracle", "_ref", "libsfm_ref.so")
    if not os.path.exists(ref):
        pytest.skip("oracle/_ref/libsfm_ref.so not built")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900, env=dict(os.environ, SFMB200_BENCH_REF_CRASH="1"))
    assert r.returncode == 0, r.stderr[-2000:]
    out = [l for l in r.stdout.strip().splitlines() if l.strip()]
    assert len(out) == 1, out[:3]
    d = json.loads(out[0])
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["value"] > 0
    assert "times in a row" in d["config"]["note"] and r.stderr.count("reference child attempt") == 6
    # and the healthy path: one line, the reference itself, first or second attempt
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    out = [l for l in r.stdout.strip().splitlines() if l.strip()]
    assert len(out) == 1, out[:3]
    d = json.loads(out[0])
    assert d["impl"] == "reference" and d["value"] > 0 and d["e2e"]["value"] == d["value"]
    if d["cpu_baseline"]["kind"] == "reference":
        assert 1 <= d["attempts"] <= 6 and d["config"]["workload"].startswith("BASELINE config 2")
