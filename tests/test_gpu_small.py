"""GPU tier: the fused single-launch path for small problems (csrc/small.cu: one thread-block cluster per pair runs
ingest, hypothesis generation, scoring + arg-max, pose candidates, cheirality and triangulation) against the general
five-launch path.  Both call the same device functions, so everything - candidates, counts, winner, E, poses, pose
index, points - must agree BIT FOR BIT; the general path is itself pinned by the oracle (test_gpu_parity.py)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
THR = 1e-6
OPT_SMALL = 7


def results(h, B):
    out = {"best": h.get_best(), "E": h.get_E().copy()}
    out["cand"] = [h.get_E_candidates(b).cpu().numpy() for b in range(B)]
    out["counts"] = [h.get_inlier_counts(b).cpu().numpy() for b in range(B)]
    return out


def same(a, b):
    return (np.array_equal(a["best"][0], b["best"][0]) and np.array_equal(a["best"][1], b["best"][1]) and np.array_equal(a["E"], b["E"])
            and all(np.array_equal(x, y) for x, y in zip(a["cand"], b["cand"])) and all(np.array_equal(x, y) for x, y in zip(a["counts"], b["counts"])))


@pytest.mark.parametrize("B,n,H", [(1, 8, 1), (1, 100, 7), (1, 2153, 269), (2, 1000, 33), (3, 1500, 700), (1, 4000, 1500), (1, 3000, 2048)])
def test_fused_path_equals_general_path(pkg, O, B, n, H):
    import torch

    K, Kinv = O.reference_K()
    px = np.stack([O.synthetic_pair(max(n, 64), seed=40 + b)["px"][:n] for b in range(B)])
    d_px = torch.from_numpy(np.ascontiguousarray(px)).cuda()
    hs, hg = pkg.BatchedPairs(K, Kinv, B, n, H), pkg.BatchedPairs(K, Kinv, B, n, H)
    hs.set_option(OPT_SMALL, 1)
    hg.set_option(OPT_SMALL, 0)
    # whole path, device-drawn rows
    for tri_only in (0, 1):
        for h in (hs, hg):
            h.set_option(3, tri_only)
            h.run_device(d_px, H, 77, THR)
        assert hs.score_plan()["variant"] == -2 and hg.score_plan()["variant"] >= 0
        assert hs.launch_count() < hg.launch_count()
        assert same(results(hs, B), results(hg, B))
        assert np.array_equal(hs.get_poses(), hg.get_poses()) and np.array_equal(hs.get_pose_index(), hg.get_pose_index())
        for b in range(B):
            assert np.array_equal(hs.get_points_host(b), hg.get_points_host(b))
    # estimate only, caller-supplied rows (incl. a degenerate one), then the staged pose calls
    idx = np.stack([O.sample_indices(5 + b, H, n) for b in range(B)]).astype(np.int32)
    if H > 3:
        idx[0, 2, 1] = idx[0, 2, 0]
    d_idx = torch.from_numpy(idx).cuda()
    for h in (hs, hg):
        h.set_points_xy(d_px)
        h.estimate_e(H, 0, THR, d_idx=d_idx)
        h.pose_candidates(); h.choose_pose(); h.triangulate()
    assert same(results(hs, B), results(hg, B))
    assert np.array_equal(hs.get_poses(), hg.get_poses()) and np.array_equal(hs.get_points_host(B - 1), hg.get_points_host(B - 1))
    # a hypothesis slice (multi-GPU shape): global indices and the packed key carry the offset
    if H >= 8:
        for h in (hs, hg):
            h.estimate_e(H // 2, 9, THR, H_total=3 * H, h_begin=H)
        assert same(results(hs, B), results(hg, B))
        assert np.all(hs.get_best()[0] >= H) and np.all(hs.get_best()[0] < H + H // 2)
    hs.close(); hg.close()


def test_fused_path_host_entry_and_dispatch(pkg, O):
    import torch

    K, Kinv = O.reference_K()
    n, H = 2153, 269
    px = O.synthetic_pair(n, seed=8)["px"]
    ref = pkg.BatchedPairs(K, Kinv, 1, n, H)
    ref.set_option(OPT_SMALL, 0)
    want = ref.run_host(px, H, 3, THR)
    h = pkg.BatchedPairs(K, Kinv, 1, n, 65536)
    for src in (px, torch.from_numpy(px).pin_memory().numpy()):          # pageable and pinned (zero-copy) input
        got = h.run_host(src, H, 3, THR)
        assert h.score_plan()["variant"] == -2                              # automatic choice at this size
        for k in ("E", "P", "pose_index", "inliers", "points"):
            assert np.array_equal(got[k], want[k]), k
    # above the evaluation limit the automatic choice is the general path; the limit is an option
    big = O.synthetic_pair(n, seed=8)["px"]
    h.run_host(big, 65536, 3, THR)
    assert h.score_plan()["variant"] >= 0
    h.set_option(8, 1000)
    h.run_host(px, H, 3, THR)
    assert h.score_plan()["variant"] >= 0
    h.set_option(8, 2500000)
    # the automatic choice is for a handful of pairs: a 16-CTA cluster per pair fills a GPC, many pairs queue up behind each other
    for pairs, fused in ((4, True), (8, False)):
        hb = pkg.BatchedPairs(K, Kinv, pairs, n, H)
        hb.run_host(np.stack([px] * pairs), H, 3, THR)
        assert (hb.score_plan()["variant"] == -2) == fused, pairs
        hb.close()
    # not eligible: Jacobi solver, explicit scoring variant, textbook pose mode, more hypotheses than a cluster holds
    for opt, val in ((5, 0), (2, 0), (1, 0)):
        h.set_option(opt, val)
        h.run_host(px, H, 3, THR)
        assert h.score_plan()["variant"] >= 0, (opt, val)
        h.set_option(opt, {5: 1, 2: -1, 1: 1}[opt])
    h.set_option(OPT_SMALL, 1)
    h.run_host(px, 4096, 3, THR)
    assert h.score_plan()["variant"] >= 0
    h.close(); ref.close()


def test_batched_pair_equals_single_pair_with_its_seed(pkg, O):
    """Pairs of a batch are seeded by their absolute index: pair 33 of a batch, alone on a handle with that pair's seed,
    reproduces its batched result."""
    import torch

    K, Kinv = O.reference_K()
    B, n, H = 70, 1200, 900
    px = np.stack([O.synthetic_pair(n, seed=300 + (b % 5))["px"] for b in range(B)])
    ref = pkg.BatchedPairs(K, Kinv, B, n, H)
    ref.set_option(OPT_SMALL, 0)
    ref.run_device(torch.from_numpy(px).cuda(), H, 42, THR)
    one = pkg.BatchedPairs(K, Kinv, 1, n, H)
    one.set_option(OPT_SMALL, 0)
    one.run_device(torch.from_numpy(px[33]).cuda(), H, (42 + 0x632BE59BD9B4E019 * 33) % (1 << 64), THR)
    assert np.array_equal(one.get_inlier_counts(0).cpu().numpy(), ref.get_inlier_counts(33).cpu().numpy())
    with pytest.raises(pkg.SfmError) as e:
        ref.set_option(11, 2)                              # the retired batch-pipeline option
    assert e.value.code == -1
    one.close(); ref.close()
