"""GPU tier: degenerate inputs through the 8f stages (adaptive termination, refit, bundle adjustment,
chaining): nothing may crash, hang or produce non-finite state; no-op cases must be no-ops."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
THR = 1e-6


def test_all_outliers_and_tiny_inputs(pkg, O):
    import torch

    K, Kinv = O.reference_K()
    rng = np.random.default_rng(0)
    # pure noise: uniform pixels in both views, two pairs
    n = 900
    px = np.stack([np.c_[rng.uniform(0, 720, n), rng.uniform(0, 576, n), rng.uniform(0, 720, n), rng.uniform(0, 576, n)]
                   for _ in range(2)]).astype(np.float32)
    h = pkg.BatchedPairs(K, Kinv, 2, n, 1024)
    h.set_option(1, 0)
    h.set_points_xy(torch.from_numpy(px).cuda())
    used = h.estimate_e_adaptive(1024, 1, THR, 0.99, 128, 2)
    assert used == 1024                                   # no consensus: never stops early
    h.refine_e(3)
    h.pose_candidates(); h.choose_pose(); h.triangulate()
    E0, P0 = h.get_E().copy(), h.get_poses().copy()
    st = h.bundle_adjust(2, 5)
    assert np.all(np.isfinite(st)) and np.all(st[:, 2] <= st[:, 1] + 1e-12)
    assert np.all(np.isfinite(h.get_E())) and np.all(np.isfinite(h.get_poses()))
    for b in range(2):
        assert np.all(np.isfinite(h.get_points_host(b)))
        if st[b, 0] < 8:                                  # fewer than 8 active points: the pair is left alone
            assert np.array_equal(h.get_E()[b], E0[b]) and np.array_equal(h.get_poses()[b], P0[b])
    ch = h.chain_views()
    assert np.all(np.isfinite(ch["cameras"])) and np.all(np.isfinite(ch["scales"])) and np.all(ch["scales"] > 0)
    assert np.all(np.isfinite(ch["cloud"].cpu().numpy()))
    if ch["used"][1] == 0:
        assert ch["scales"][1] == 1.0                     # no linking track: scale stays 1
    h.close()
    # the smallest input the handle accepts: 8 correspondences
    sc = O.synthetic_pair(8, outlier_frac=0.0, noise_px=0.0, seed=2)
    h = pkg.BatchedPairs(K, Kinv, 1, 8, 64)
    h.set_option(1, 0)
    h.set_points_xy(torch.from_numpy(sc["px"][None]).cuda())
    assert h.estimate_e_adaptive(64, 1, THR, 0.999, 8, 2) in (8, 16, 32, 64)
    h.refine_e(2)
    h.pose_candidates(); h.choose_pose(); h.triangulate()
    st = h.bundle_adjust(1, 3)
    assert np.all(np.isfinite(st)) and np.all(np.isfinite(h.get_points_host(0)))
    ch = h.chain_views()
    assert np.array_equal(ch["used"], [0]) and np.all(np.isfinite(ch["cameras"]))
    h.close()


def test_bundle_adjust_then_rest_of_the_api_still_consistent(pkg, O):
    """After BA the handle's E / pose / points / count describe ONE model: re-running the downstream getters and
    a second adjustment from that state is idempotent up to LM's own progress (cost never increases)."""
    import torch

    K, Kinv = O.reference_K()
    n = 2500
    sc = O.synthetic_pair(n, noise_px=0.5, seed=17)
    h = pkg.BatchedPairs(K, Kinv, 1, n, 4096)
    h.set_option(1, 0)
    h.set_points_xy(torch.from_numpy(sc["px"][None]).cuda())
    h.estimate_e(4096, 2, THR); h.refine_e(4); h.pose_candidates(); h.choose_pose(); h.triangulate()
    s1 = h.bundle_adjust(4, 40)[0]
    c1 = int(h.get_best()[1][0])
    s2 = h.bundle_adjust(1, 40)[0]
    c2 = int(h.get_best()[1][0])
    # a new round re-selects the active set with the refined E and restarts from DLT points, so its entry cost may
    # exceed the previous exit cost; per active point it ends where the first run ended
    assert s2[2] <= s2[1] and s2[2] / s2[0] <= 1.1 * s1[2] / s1[0]
    assert c2 >= 0.95 * c1                                         # commit guard: a round that collapses the consensus is dropped
    x = O.normalise_points(sc["px"], Kinv)
    assert c2 == int(O.sampson_mask_f32(h.get_E()[0], x, THR).sum())
    # the adjusted pose can be handed back through set_E + the pose stages: same pose index, same camera up to rounding
    M = h.get_poses()[0][int(h.get_pose_index()[0])].copy()
    h.set_E(h.get_E())
    h.pose_candidates(); h.choose_pose()
    M2 = h.get_poses()[0][int(h.get_pose_index()[0])]
    assert np.linalg.norm(M2[:3, :3] - M[:3, :3]) < 1e-3 and np.linalg.norm(M2[:3, 3] - M[:3, 3]) < 1e-3
    h.close()


def test_failed_run_does_not_corrupt_the_threshold_scale(pkg, O):
    """ADVICE r1: run_device / run_host used to commit the new threshold scale before the ingest was validated; a
    failing call then left corr_s / corr_dup at the old scale while pt_scale claimed the new one, and the next
    estimate at that threshold scored mis-scaled points.  Every argument is validated before anything is enqueued,
    so a failing call leaves the handle as it was."""
    import torch

    K, Kinv = O.reference_K()
    n, H = 2000, 1024
    px = O.synthetic_pair(n, seed=3)["px"]
    d_px = torch.from_numpy(px).cuda()
    h = pkg.BatchedPairs(K, Kinv, 1, n, H)
    h.run_device(d_px, H, 7, 1e-6)
    want = h.get_inlier_counts().cpu().numpy().copy()
    fresh = pkg.BatchedPairs(K, Kinv, 1, n, H)
    fresh.run_device(d_px, H, 7, 4e-6)
    want4 = fresh.get_inlier_counts().cpu().numpy().copy()
    launches = h.launch_count()
    big = torch.zeros((n + 100, 4), device="cuda")
    with pytest.raises(pkg.SfmError):
        h.run_device(big, H, 7, 4e-6)                       # n above max_points: must leave the handle untouched
    with pytest.raises(pkg.SfmError):
        h.lib.call("sfmb200_run_host", h._h, None, n, H, __import__("ctypes").c_uint64(7), __import__("ctypes").c_float(4e-6),
                   None, None, None, None, None)            # null input
    with pytest.raises(pkg.SfmError):
        h.run_device(d_px, H + 1, 7, 4e-6)                  # H above max_hypotheses, with a valid input
    with pytest.raises(pkg.SfmError):
        h.run_host(px, H + 1, 7, 4e-6)
    assert h.launch_count() == launches                     # nothing was enqueued
    assert np.array_equal(h.get_inlier_counts().cpu().numpy(), want)
    h.estimate_e(H, 7, 4e-6)                                # re-materialises the scaled copies for the new threshold
    assert np.array_equal(h.get_inlier_counts().cpu().numpy(), want4)
    h.estimate_e(H, 7, 1e-6)
    assert np.array_equal(h.get_inlier_counts().cpu().numpy(), want)
    h.close(); fresh.close()


def test_python_mirror_validates_buffers(pkg, O):
    """ADVICE r1: dtype / shape of every buffer whose raw pointer crosses the C ABI is checked first."""
    import torch

    K, Kinv = O.reference_K()
    n, H = 1000, 256
    px = O.synthetic_pair(n, seed=4)["px"]
    h = pkg.BatchedPairs(K, Kinv, 1, n, H)
    out = h.run_host(px.astype(np.float64), H, 1, 1e-6)      # float64 input is coerced, not reinterpreted
    ref = h.run_host(px, H, 1, 1e-6)
    assert np.array_equal(out["E"], ref["E"]) and np.array_equal(out["points"], ref["points"])
    bad = {k: v.copy() if v is not None else None for k, v in ref.items()}
    bad["points"] = np.empty((1, 4, n // 2), np.float32)
    with pytest.raises(ValueError):
        h.run_host(px, H, 1, 1e-6, out=bad)
    bad["points"] = np.empty((1, 4, n), np.float64)
    with pytest.raises(TypeError):
        h.run_host(px, H, 1, 1e-6, out=bad)
    with pytest.raises(TypeError):
        h.prepare_run_host(px, H, 1, 1e-6, out=dict(ref, inliers=np.empty(1, np.int64)))
    with pytest.raises(TypeError):
        h.set_points_xy(torch.zeros((n, 4), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        h.set_points_xy(torch.zeros((n // 2, 4), device="cuda"), n)
    with pytest.raises(TypeError):
        h.estimate_e(H, 1, 1e-6, d_idx=torch.zeros((H, 8), dtype=torch.int64, device="cuda"))
    h.close()


def test_handle_keeps_its_device_when_another_is_current(pkg, O):
    """ADVICE r1: a handle belongs to the device that was current at create; every entry point makes that device current for
    the call and restores the caller's.  Needs two GPUs (skipped on a one-GPU box)."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    K, Kinv = O.reference_K()
    n, H = 3000, 4096
    px = O.synthetic_pair(n, seed=31)["px"]
    torch.cuda.set_device(0)
    ref = pkg.BatchedPairs(K, Kinv, 1, n, H)
    want = ref.run_host(px, H, 3, THR)
    torch.cuda.set_device(1)
    h1 = pkg.BatchedPairs(K, Kinv, 1, n, H)              # lives on device 1
    torch.cuda.set_device(0)                               # ... and is driven while device 0 is current
    got = h1.run_host(px, H, 3, THR)
    assert torch.cuda.current_device() == 0
    for k in ("E", "P", "pose_index", "inliers", "points"):
        assert np.array_equal(got[k], want[k]), k
    d_px1 = torch.from_numpy(px).to("cuda:1")
    h1.set_points_xy(d_px1)
    h1.estimate_e(H, 3, THR)
    h1.pose_candidates(); h1.choose_pose(); h1.triangulate()
    assert np.array_equal(h1.get_points_host(0), want["points"][0])
    h1.close(); ref.close()


@pytest.mark.parametrize("n,H", [(1200, 150), (5000, 1024)])        # fused small-problem path / general five-launch path
def test_dirty_handle_equals_fresh_handle(pkg, O, n, H):
    """Whatever ran on a handle before - homography, adaptive estimate, refit, bundle adjustment, chaining, another threshold,
    another metric or sampler (reset afterwards), a slice estimate - a whole-path run gives the bits a fresh handle gives, and
    the stages that follow it are accepted."""
    import torch

    K, Kinv = O.reference_K()
    px = np.ascontiguousarray(pkg.synthetic.synthetic_sequence(3, n, seed=51)["px_pairs"])       # 3 views = 2 consecutive pairs
    d_px = torch.from_numpy(px).cuda()
    cap = max(H, 4096)
    fresh = pkg.BatchedPairs(K, Kinv, 2, n, cap)
    fresh.run_device(d_px, H, 21, 1e-6)
    want = (fresh.get_E(), fresh.get_best()[0], fresh.get_best()[1], fresh.get_poses(), fresh.get_pose_index(),
            fresh.get_points_host(0), fresh.get_points_host(1))

    def check(h, what):
        h.run_device(d_px, H, 21, 1e-6)
        got = (h.get_E(), h.get_best()[0], h.get_best()[1], h.get_poses(), h.get_pose_index(), h.get_points_host(0), h.get_points_host(1))
        for a, b in zip(want, got):
            assert np.array_equal(a, b), what
        h.get_inlier_mask(); h.refine_e(1)                       # accepted: the handle holds an essential-matrix estimate again

    h = pkg.BatchedPairs(K, Kinv, 2, n, cap)
    h.set_points_xy(d_px)
    h.find_homography(1024, 3, 5.0)
    check(h, "after find_homography")
    h.estimate_e_adaptive(4096, 5, 4e-6, 0.99)                   # another threshold: the scaled copies are re-materialised
    h.refine_e(2)
    h.pose_candidates(); h.choose_pose(); h.triangulate()
    h.bundle_adjust(1, 3)
    check(h, "after adaptive + refit + bundle adjustment at another threshold")
    h.run_device(d_px, H, 21, 1e-6)                              # (the refit inside check() invalidated the poses)
    ch = h.chain_views()
    h.bundle_adjust_global(ch, iterations=2)
    check(h, "after chaining + global bundle adjustment")
    for opt, val, back in ((9, 1, 0), (10, 1, 0), (5, 0, 1), (1, 0, 1), (3, 1, 0)):     # metric, sampler, solver, pose mode, inliers-only
        h.set_option(opt, val)
        h.run_device(d_px, H, 21, 1e-6)
        h.set_option(opt, back)
        check(h, f"after option {opt} = {val} and back")
    lo, hi = pkg.sharding.shard_range(H, 1, 2)
    h.estimate_e(hi - lo, 21, 1e-6, H_total=H, h_begin=lo)
    check(h, "after a slice estimate")
    h.close(); fresh.close()
