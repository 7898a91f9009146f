"""GPU tier: the CUDA path through the C ABI against the oracle on the same
seeded inputs.  Bars: sample indices / inlier counts / arg-max / pose index are
integer work -> bit-exact (counts: bit-exact against the fp32 port of the same
fma tree, and inside the borderline band of the fp64 truth); floating-point
stages carry their tolerance in the test."""
import ctypes as C
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

fp = C.POINTER(C.c_float)
ip = C.POINTER(C.c_int32)
THR = 1e-6


def P(a, t=fp):
    return a.ctypes.data_as(t)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "GPU tier needs a CUDA device"
    torch.cuda.set_device(0)
    return torch


def counts_f32(oracle_c, E32, x, thr=THR):
    out = np.zeros(len(E32), np.int32)
    oracle_c.oracle_counts_f32(P(np.ascontiguousarray(E32)), len(E32), P(x), len(x), C.c_float(thr), P(out, ip))
    return out


# Borderline band of the fp64 comparison.  north_star asks for exact counts except
# for correspondences "within 1e-6 of the threshold"; read as a relative band on
# num^2 - thr*den that is unreachable for ANY fp32 evaluation: x1^T E x2 is a
# cancelling sum of O(0.1..1) terms that equals ~1e-3 at the threshold, so fp32
# rounding alone moves num^2 by ~1e-5 relative there.  The exact-equality check
# is the fp32 port (same fma tree, bit for bit); against fp64 the band is 1e-4.
BAND = 1e-4


def counts_f64(oracle_c, E32, x, thr=THR):
    cnt = np.zeros(len(E32), np.int32)
    amb = np.zeros(len(E32), np.int32)
    oracle_c.oracle_counts_f64(P(np.ascontiguousarray(E32)), len(E32), P(x), len(x), C.c_double(thr), C.c_double(BAND),
                               P(cnt, ip), P(amb, ip))
    return cnt, amb


def gpu_x(h, pair=0):
    """(n,4) normalised correspondences exactly as the device holds them."""
    X0, X1 = h.get_X(0, pair).cpu().numpy(), h.get_X(1, pair).cpu().numpy()
    return np.ascontiguousarray(np.stack([X0[0], X0[1], X1[0], X1[1]], 1))


def make_handle(pkg, sc, H, pairs=1, n=None):
    return pkg.BatchedPairs(sc["K"], sc["Kinv"], pairs, n or len(sc["px"]), H)


# --------------------------------------------------------------------------
def test_ingest_matches_oracle(pkg, O, torch_cuda, scene_small):
    torch = torch_cuda
    h = make_handle(pkg, scene_small, 16)
    h.set_points_xy(torch.from_numpy(scene_small["px"]).cuda())
    X0, X1 = h.get_X(0).cpu().numpy(), h.get_X(1).cpu().numpy()
    x = scene_small["x"]
    # fp32 K^-1 [u v 1]: 1-2 ulp of the fp64-accumulated restatement
    assert np.abs(X0[0] - x[:, 0]).max() < 3e-8 and np.abs(X0[1] - x[:, 1]).max() < 3e-8
    assert np.abs(X1[0] - x[:, 2]).max() < 3e-8 and np.abs(X1[1] - x[:, 3]).max() < 3e-8
    assert np.all(X0[2] == 1) and np.all(X1[2] == 1)
    # host path and SiftPoint path give the same bits
    h2 = make_handle(pkg, scene_small, 16)
    h2.set_points_xy_host(scene_small["px"])
    assert np.array_equal(h2.get_X(1).cpu().numpy(), X1)
    n = len(x)
    sift = np.zeros((n, 144), np.float32)          # 576-byte SiftPoint records
    sift[:, 0], sift[:, 1], sift[:, 9], sift[:, 10] = scene_small["px"].T
    sift[:, 2:9] = 7.0                               # other fields are ignored
    ipair = pkg.ImagePair(scene_small["K"], scene_small["Kinv"], 2, n)
    ipair.fillXU(torch.from_numpy(sift).cuda())
    assert np.array_equal(ipair.get_X(0).cpu().numpy(), X0)
    assert np.array_equal(ipair.get_X(1).cpu().numpy(), X1)


@pytest.mark.parametrize("variant,solver", [(0, 0), (1, 0), (4, 0), (4, 1), (9, 1), (10, 1), (-1, 1)])
def test_estimate_e_against_oracle(pkg, O, oracle_c, torch_cuda, scene_small, variant, solver):
    torch = torch_cuda
    x, n = scene_small["x"], len(scene_small["x"])
    H, seed = 3000, 1237          # H not a multiple of any tile size
    h = make_handle(pkg, scene_small, H)
    h.set_option(2, variant)
    h.set_option(5, solver)       # 0: 9x9 Jacobi eigensolve, 1: 8x8 Cholesky projector
    h.set_points_xy(torch.from_numpy(scene_small["px"]).cuda())
    h.estimate_e(H, seed, THR)
    Eg = h.get_E_candidates().cpu().numpy()
    # (1) hypotheses: device-generated indices == oracle generator; E within 1e-4
    idx = O.sample_indices(seed, H, n)
    E64 = O.hypotheses(x, idx)
    d = O.e_distance(Eg, E64)
    assert np.mean(d < 1e-4) >= 0.995, f"{np.mean(d < 1e-4)} of hypotheses within 1e-4"
    assert np.median(d) < 1e-6
    # (2) counts: bit-exact vs the fp32 port, banded vs fp64
    got = h.get_inlier_counts().cpu().numpy()
    xg = gpu_x(h)
    assert np.array_equal(got, counts_f32(oracle_c, Eg, xg))
    c64, amb = counts_f64(oracle_c, Eg, xg)
    assert np.all(np.abs(got - c64) <= amb)
    # (3) arg-max: highest count, lowest index
    bi, bc = h.get_best()
    assert bc[0] == got.max() and bi[0] == int(np.argmax(got))
    assert np.array_equal(h.get_E()[0].reshape(9), Eg[bi[0]])
    plan = h.score_plan()
    assert variant < 0 or plan["variant"] == variant
    h.close()


def test_scalar_and_packed_kernels_are_bit_identical(pkg, torch_cuda, scene_small):
    torch = torch_cuda
    res = []
    for variant in (0, 1, 10):
        h = make_handle(pkg, scene_small, 5000)
        h.set_option(2, variant)
        h.set_points_xy(torch.from_numpy(scene_small["px"]).cuda())
        h.estimate_e(5000, 99, THR)
        res.append((h.get_inlier_counts().cpu().numpy(), h.get_best(), h.get_E()))
        h.close()
    for r in res[1:]:
        assert np.array_equal(res[0][0], r[0])
        assert res[0][1][0][0] == r[1][0][0] and res[0][1][1][0] == r[1][1][0]
        assert np.array_equal(res[0][2], r[2])


@pytest.mark.parametrize("n,H", [(8, 1), (9, 7), (511, 513), (512, 1024), (513, 1025), (2049, 300), (3000, 2)])
def test_ragged_shapes_and_split_paths(pkg, O, oracle_c, torch_cuda, scene_small, n, H):
    """Covers splits == 1 and splits > 1 (atomic partial counts + last-CTA arg-max),
    partial TMA stages, partial hypothesis tiles, minimum sizes."""
    torch = torch_cuda
    px = np.ascontiguousarray(scene_small["px"][:n])
    for variant in (0, 1, 10):
        h = pkg.BatchedPairs(scene_small["K"], scene_small["Kinv"], 1, max(n, 8), H)
        h.set_option(2, variant)
        h.set_points_xy(torch.from_numpy(px).cuda())
        h.estimate_e(H, 5, THR)
        Eg = h.get_E_candidates().cpu().numpy()
        got = h.get_inlier_counts().cpu().numpy()
        assert np.array_equal(got, counts_f32(oracle_c, Eg, gpu_x(h))), (n, H, variant, h.score_plan())
        bi, bc = h.get_best()
        assert bc[0] == got.max() and bi[0] == int(np.argmax(got))
        h.close()


def test_user_supplied_indices_and_degenerate_rows(pkg, O, oracle_c, torch_cuda, scene_small):
    torch = torch_cuda
    x, n = scene_small["x"], len(scene_small["x"])
    H = 700
    idx = O.sample_indices(31337, H, n)
    idx[5, 3] = idx[5, 0]            # repeated index -> degenerate
    idx[6, 7] = n + 10               # out of range   -> degenerate
    idx[7, 2] = -1
    h = make_handle(pkg, scene_small, H)
    h.set_points_xy(torch.from_numpy(scene_small["px"]).cuda())
    h.estimate_e(H, 0, THR, d_idx=torch.from_numpy(idx).cuda())
    Eg = h.get_E_candidates().cpu().numpy()
    got = h.get_inlier_counts().cpu().numpy()
    assert np.all(Eg[[5, 6, 7]] == 0) and np.all(got[[5, 6, 7]] == 0)
    good = np.ones(H, bool)
    good[[5, 6, 7]] = False
    d = O.e_distance(Eg[good], O.hypotheses(x, idx[good]))
    assert np.mean(d < 1e-4) >= 0.99
    assert np.array_equal(got, counts_f32(oracle_c, Eg, gpu_x(h)))
    # same rows through the generator path give the same bits as explicit rows
    idx2 = O.sample_indices(8, H, n)
    h.estimate_e(H, 0, THR, d_idx=torch.from_numpy(idx2).cuda())
    a = (h.get_E_candidates().cpu().numpy(), h.get_inlier_counts().cpu().numpy())
    h.estimate_e(H, 8, THR)
    b = (h.get_E_candidates().cpu().numpy(), h.get_inlier_counts().cpu().numpy())
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    h.close()


def test_hypothesis_slices_reproduce_the_full_run(pkg, torch_cuda, scene_small):
    """Multi-GPU hypothesis sharding on one device: slices [lo,hi) of H_total give
    the same E / counts as the single run, and MAX over the packed keys followed
    by adopt_best reproduces the single-run winner bit for bit."""
    torch = torch_cuda
    H, seed = 4100, 77
    dpx = torch.from_numpy(scene_small["px"]).cuda()
    full = make_handle(pkg, scene_small, H)
    full.set_points_xy(dpx)
    full.estimate_e(H, seed, THR)
    # the other solver reproduces itself through adopt_best as well
    alt = make_handle(pkg, scene_small, H)
    alt.set_option(5, 1)
    alt.set_points_xy(dpx)
    alt.estimate_e(H, seed, THR)
    E_alt, best_alt = alt.get_E().copy(), alt.get_best()
    alt.adopt_best(H, seed)
    assert np.array_equal(alt.get_E(), E_alt) and alt.get_best()[0][0] == best_alt[0][0]
    alt.close()
    Ef, cf = full.get_E_candidates().cpu().numpy(), full.get_inlier_counts().cpu().numpy()
    keys = []
    for world in (2, 3):
        keys.clear()
        for r in range(world):
            lo, hi = pkg.sharding.shard_range(H, r, world)
            hs = make_handle(pkg, scene_small, hi - lo)
            hs.set_points_xy(dpx)
            hs.estimate_e(hi - lo, seed, THR, H_total=H, h_begin=lo)
            assert np.array_equal(hs.get_E_candidates().cpu().numpy(), Ef[lo:hi])
            assert np.array_equal(hs.get_inlier_counts().cpu().numpy(), cf[lo:hi])
            hs.synchronize()
            keys.append(int(hs.best_buffer().cpu()[0]))
            if r == world - 1:
                best = hs.best_buffer()
                best.fill_(max(keys))
                torch.cuda.synchronize()
                hs.adopt_best(H, seed)
                assert np.array_equal(hs.get_E(), full.get_E())
                assert hs.get_best()[0][0] == full.get_best()[0][0]
                assert hs.get_best()[1][0] == full.get_best()[1][0]
            hs.close()
    full.close()


def test_poses_cheirality_triangulation_compat(pkg, O, torch_cuda, scene_small):
    torch = torch_cuda
    x = scene_small["x"]
    h = make_handle(pkg, scene_small, 4096)
    h.set_points_xy(torch.from_numpy(scene_small["px"]).cuda())
    h.estimate_e(4096, 3, THR)
    E = h.get_E()[0].astype(np.float64)
    h.pose_candidates()
    Pg = h.get_poses()[0]
    Po = O.pose_candidates(E, compat=True)
    perm = O.match_candidates(Pg, Po, tol=2e-5)      # fp32 3x3 SVD vs fp64
    assert perm is not None, np.abs(Pg - Po).max()
    h.choose_pose()
    # cheirality on OUR candidates through the oracle's restatement: exact index
    ind_o, Pinv_o = O.choose_pose(x, Pg.astype(np.float64), compat=True)
    assert h.get_pose_index()[0] == ind_o
    assert np.abs(h.get_poses()[0] - Pinv_o).max() < 5e-5      # side effect: inverses (Q18)
    h.triangulate()
    pts = h.get_points_host()
    ref = O.triangulate(x, Pinv_o[ind_o])
    assert np.all(pts[3] == 1)
    # fp32 DLT null vector vs fp64: relative to the point's depth; the tail are
    # outlier correspondences whose two smallest singular values nearly coincide
    rel = np.abs(pts[:3] - ref[:3]).max(axis=0) / np.maximum(np.abs(ref[:3]).max(axis=0), 1e-3)
    inl = ~scene_small["is_outlier"]
    assert np.median(rel[inl]) < 1e-4 and np.mean(rel[inl] < 1e-3) > 0.99
    assert np.mean(rel < 1e-3) > 0.97
    # egress: N x 4 AoS (x, y, z, 1), colours all ones
    pos = torch.empty((len(x), 4), device="cuda")
    col = torch.zeros((len(x), 4), device="cuda")
    h.copy_to_vbo(pos, col)
    assert np.array_equal(pos.cpu().numpy(), O.to_vbo(pts).astype(np.float32))
    assert torch.all(col == 1)
    h.close()


def test_correct_mode_recovers_ground_truth_pose(pkg, O, torch_cuda):
    torch = torch_cuda
    K, Kinv = O.reference_K()
    sc = O.synthetic_pair(4000, outlier_frac=0.3, noise_px=0.3, seed=21)
    h = pkg.BatchedPairs(K, Kinv, 1, 4000, 16384)
    h.set_option(1, 0)               # textbook geometry + inlier vote
    h.set_option(3, 1)               # triangulate inliers only
    out = h.run_host(sc["px"], 16384, 1, THR)
    Psel = out["P"][0].reshape(4, 4)
    assert np.abs(Psel[:3, :3] - sc["R"]).max() < 0.1
    t = Psel[:3, 3]
    assert np.dot(t, sc["t"]) > 0.8
    mask = h.get_inlier_mask().cpu().numpy().astype(bool)
    assert mask.sum() == out["inliers"][0]
    assert np.mean(mask[~sc["is_outlier"]]) > 0.6 and np.mean(mask[sc["is_outlier"]]) < 0.1
    pts = out["points"][0]
    assert np.all(pts[:3, ~mask] == 0)
    err = np.linalg.norm(pts[:3, mask].T - sc["X"][mask], axis=1) / np.linalg.norm(sc["X"][mask], axis=1)
    assert np.median(err) < 0.25
    h.close()


@pytest.mark.parametrize("seed", [5, 61])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("n", [700, 5000])
def test_vote_mode_poses_against_oracle(pkg, O, torch_cuda, seed, B, n):
    """SFMB200_OPT_COMPAT = 0 (textbook candidates + inlier vote) and inliers-only triangulation against the oracle:
    the four candidates equal the fp64 ones as a set (the SVD's orientation, hence their order, is free), the selected
    pose equals the oracle's vote winner over the device's inlier mask, and points outside the mask are (0, 0, 0, 1)."""
    torch = torch_cuda
    K, Kinv = O.reference_K()
    H = 2048
    scenes = [O.synthetic_pair(n, seed=1000 * seed + b) for b in range(B)]
    h = pkg.BatchedPairs(K, Kinv, B, n, H)
    h.set_option(1, 0)
    h.set_option(3, 1)
    h.run_device(torch.from_numpy(np.stack([s["px"] for s in scenes])).cuda(), H, seed, THR)
    E, Pg, ind = h.get_E(), h.get_poses(), h.get_pose_index()
    for b in range(B):
        xg = gpu_x(h, b)
        mask = h.get_inlier_mask(b).cpu().numpy().astype(bool)
        assert np.array_equal(mask, O.sampson_mask_f32(E[b], xg, THR))
        Po = O.pose_candidates(E[b].astype(np.float64), compat=False)
        assert O.match_candidate_set(Pg[b], Po, tol=1e-4) is not None, (b, np.abs(Pg[b] - Po).max())
        votes = O.cheirality_votes(xg, Po, mask)
        top = sorted(votes)
        assert top[3] - top[2] > 0.01 * sum(votes), votes          # a clear winner, so the pose is pinned below
        assert np.abs(Pg[b][ind[b]] - Po[int(np.argmax(votes))]).max() < 1e-4, (b, int(ind[b]), votes)
        pts = h.get_points_host(b)
        assert np.all(pts[:3, ~mask] == 0) and np.all(pts[3] == 1)
        ref = O.triangulate(xg[mask], Pg[b][ind[b]].astype(np.float64))
        rel = np.abs(pts[:3, mask] - ref[:3]).max(axis=0) / np.maximum(np.abs(ref[:3]).max(axis=0), 1e-3)
        assert np.median(rel) <= 1e-6 and np.mean(rel < 1e-3) >= 0.99, (b, np.median(rel), np.mean(rel < 1e-3))
    h.close()


def test_batched_pairs_equal_single_pairs(pkg, O, torch_cuda):
    torch = torch_cuda
    K, Kinv = O.reference_K()
    B, n, H, seed = 5, 700, 1100, 17
    scenes = [O.synthetic_pair(n, seed=100 + b) for b in range(B)]
    px = np.stack([s["px"] for s in scenes])
    hb = pkg.BatchedPairs(K, Kinv, B, n, H)
    out = hb.run_host(px, H, seed, THR)
    for b in range(B):
        hs = pkg.BatchedPairs(K, Kinv, 1, n, H)
        pair_seed = (seed + 0x632BE59BD9B4E019 * b) % (1 << 64)
        o1 = hs.run_host(px[b], H, pair_seed, THR)
        assert np.array_equal(o1["E"][0], out["E"][b])
        assert o1["inliers"][0] == out["inliers"][b] and o1["pose_index"][0] == out["pose_index"][b]
        assert np.array_equal(o1["P"][0], out["P"][b])
        assert np.array_equal(o1["points"][0], out["points"][b])
        assert np.array_equal(hs.get_inlier_counts().cpu().numpy(), hb.get_inlier_counts(b).cpu().numpy())
        hs.close()
    hb.close()


def test_run_host_is_deterministic_and_matches_staged_calls(pkg, torch_cuda, scene_small):
    torch = torch_cuda
    H = 2048
    h = make_handle(pkg, scene_small, H)
    a = h.run_host(scene_small["px"], H, 4, THR)
    b = h.run_host(scene_small["px"], H, 4, THR)
    for k in ("E", "P", "pose_index", "inliers", "points"):
        assert np.array_equal(a[k], b[k]), k
    h2 = make_handle(pkg, scene_small, H)
    h2.set_points_xy(torch.from_numpy(scene_small["px"]).cuda())
    h2.estimate_e(H, 4, THR)
    h2.pose_candidates()
    h2.choose_pose()
    h2.triangulate()
    assert np.array_equal(h2.get_E()[0].reshape(9), a["E"][0])
    assert np.array_equal(h2.get_points_host(), a["points"][0])
    assert h2.get_pose_index()[0] == a["pose_index"][0]
    assert np.array_equal(h2.get_poses()[0][a["pose_index"][0]].reshape(16), a["P"][0])
    h.close()
    h2.close()


def test_error_paths(pkg, O, torch_cuda, scene_small):
    torch = torch_cuda
    h = make_handle(pkg, scene_small, 100)
    with pytest.raises(pkg.SfmError) as e:
        h.estimate_e(10, 0, THR)                     # before points
    assert e.value.code == -3
    dpx = torch.from_numpy(scene_small["px"]).cuda()
    with pytest.raises(pkg.SfmError):
        h.set_points_xy(dpx, n=7)                    # fewer than 8 correspondences
    with pytest.raises(ValueError):
        h.set_points_xy(dpx, n=len(scene_small["px"]) + 1)   # tensor smaller than n says (caught by the Python mirror)
    with pytest.raises(pkg.SfmError):
        h.set_points_xy(torch.zeros((len(scene_small["px"]) + 1, 4), device="cuda"))   # above capacity (caught by the C ABI)
    h.set_points_xy(dpx)
    with pytest.raises(pkg.SfmError):
        h.estimate_e(101, 0, THR)                    # above max_hypotheses
    with pytest.raises(pkg.SfmError):
        h.estimate_e(10, 0, 0.0)                     # non-positive threshold
    with pytest.raises(pkg.SfmError) as e:
        h.pose_candidates()                          # no E yet
    assert e.value.code == -3
    h.estimate_e(100, 0, THR)
    with pytest.raises(pkg.SfmError):
        h.triangulate()                              # before pose_candidates
    h.close()


def test_full_size_properties_config2(pkg, O, oracle_c, torch_cuda):
    """BASELINE config 2 (10k correspondences, 30 % outliers, 65,536 hypotheses):
    size-independent properties instead of an oracle run."""
    torch = torch_cuda
    K, Kinv = O.reference_K()
    n, H = 10000, 65536
    sc = O.synthetic_pair(n, seed=1234)
    dpx = torch.from_numpy(sc["px"]).cuda()
    h = pkg.BatchedPairs(K, Kinv, 1, n, H)
    h.set_points_xy(dpx)
    h.estimate_e(H, 1237, THR)
    c = h.get_inlier_counts()
    E = h.get_E_candidates()
    bi, bc = h.get_best()
    assert int(c.max()) == bc[0] and int((c == c.max()).nonzero()[0]) == bi[0]
    assert 0 <= int(c.min()) and int(c.max()) <= n
    # every non-degenerate candidate is a projected essential matrix: |E|_F = sqrt 2, det ~ 0
    nrm = torch.linalg.norm(E, dim=1)
    assert torch.all(((nrm - 2 ** 0.5).abs() < 1e-3) | (nrm == 0))
    assert float(torch.linalg.det(E.view(-1, 3, 3)).abs().max()) < 1e-3
    # the winner is a good model: most true inliers satisfy it
    mask = h.get_inlier_mask().cpu().numpy().astype(bool)
    assert mask.sum() == bc[0]
    assert np.mean(mask[~sc["is_outlier"]]) > 0.5 and np.mean(mask[sc["is_outlier"]]) < 0.1
    # checksum of checksums: two variants, two runs, same total and same per-hypothesis counts
    h.set_option(2, 0)
    h.estimate_e(H, 1237, THR)
    c0 = h.get_inlier_counts()
    assert torch.equal(c, c0) and h.get_best()[0][0] == bi[0]
    # ALL 65,536 hypotheses: bit-exact against the fp32 port of the same fma tree, and against the fp64 truth inside
    # the borderline band; how much of the band is actually used is recorded (profiles/r02_count_parity.md)
    Enp, got = E.cpu().numpy(), c.cpu().numpy()
    xg = gpu_x(h)
    assert np.array_equal(got, counts_f32(oracle_c, Enp, xg))
    c64, amb = counts_f64(oracle_c, Enp, xg)
    diff = np.abs(got - c64)
    assert np.all(diff <= amb)
    # ALL 65,536 candidates against the fp64 null vectors of the same rows
    d = O.e_distance(Enp, O.hypotheses(xg, O.sample_indices(1237, H, n)))
    assert np.mean(d < 1e-4) >= 0.995, f"{np.mean(d < 1e-4)} of hypotheses within 1e-4"
    assert np.median(d) < 1e-6
    rec = {"config": "BASELINE config 2: 10,000 correspondences x 65,536 hypotheses, seed 1237, thr 1e-6", "band_rel": BAND,
           "E_within_1e-4": float(np.mean(d < 1e-4)), "E_within_1e-6": float(np.mean(d < 1e-6)),
           "E_median_distance": float(np.median(d)),
           "hypotheses": int(H), "evaluations": int(H) * n, "sum_borderline": int(amb.sum()), "sum_abs_diff_vs_fp64": int(diff.sum()),
           "max_abs_diff_vs_fp64": int(diff.max()), "hypotheses_with_any_diff": int((diff > 0).sum()),
           "fp32_port_bit_exact": True, "winner_fp32": [int(bi[0]), int(bc[0])],
           "winner_fp64": [int(np.argmax(c64)), int(c64.max())]}
    for band in (1e-5, 1e-6):            # the band north_star's wording would imply: how many decisions fall outside it
        cb, ab = np.zeros(H, np.int32), np.zeros(H, np.int32)
        oracle_c.oracle_counts_f64(P(np.ascontiguousarray(Enp)), H, P(xg), n, C.c_double(THR), C.c_double(band), P(cb, ip), P(ab, ip))
        rec[f"hypotheses_outside_band_{band:g}"] = int((np.abs(got - cb) > ab).sum())
        rec[f"sum_borderline_band_{band:g}"] = int(ab.sum())
    print("\ncount parity record:", json.dumps(rec))
    out_dir = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "count_parity_config2.json"), "w") as f:
        json.dump(rec, f, indent=1)
    h.close()


def test_filtered_sift_ingest(pkg, O, torch_cuda, scene_small):
    """SURVEY 8f rank 1: match filtering fused into ingest, ordered compaction."""
    torch = torch_cuda
    n = len(scene_small["px"])
    rng = np.random.default_rng(7)
    sift = np.zeros((n, 144), np.float32)
    sift[:, 0], sift[:, 1], sift[:, 9], sift[:, 10] = scene_small["px"].T
    sift[:, 6] = rng.uniform(0.5, 1.0, n)           # score
    sift[:, 7] = rng.uniform(0.5, 1.0, n)           # ambiguity
    d_sift = torch.from_numpy(sift).cuda()
    for min_score, max_amb in ((0.85, 0.95), (0.0, 2.0), (0.5, 0.75)):
        keep = (sift[:, 6] > np.float32(min_score)) & (sift[:, 7] < np.float32(max_amb))
        ip_f = pkg.ImagePair(scene_small["K"], scene_small["Kinv"], 2, n)
        kept_idx = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        kept = ip_f.set_points_sift_filtered(d_sift, n, min_score, max_amb, kept_idx)
        assert kept == int(keep.sum())
        assert np.array_equal(kept_idx.cpu().numpy()[:kept], np.flatnonzero(keep).astype(np.int32))
        # same bits as an unfiltered ingest of the surviving records
        ip_u = pkg.ImagePair(scene_small["K"], scene_small["Kinv"], 2, n)
        ip_u.fillXU(torch.from_numpy(np.ascontiguousarray(sift[keep])).cuda(), n=kept)
        for image in (0, 1):
            assert np.array_equal(ip_f.get_X(image).cpu().numpy(), ip_u.get_X(image).cpu().numpy())
        ip_f.estimateE(256, 3, THR)
        ip_u.estimateE(256, 3, THR)
        assert np.array_equal(ip_f.get_E(), ip_u.get_E()) and ip_f.get_best()[1][0] == ip_u.get_best()[1][0]
        ip_f.close(); ip_u.close()
    ip_f = pkg.ImagePair(scene_small["K"], scene_small["Kinv"], 2, n)
    with pytest.raises(pkg.SfmError) as e:
        ip_f.set_points_sift_filtered(d_sift, n, 2.0, 0.0)       # nothing survives
    assert e.value.code == -3


def test_random_shapes_fuzz(pkg, O, oracle_c, torch_cuda):
    """Random (pairs, n, H, variant, solver) shapes: the stream-K partition, the split /
    atomic epilogue and the fused arg-max against the fp32 port, bit for bit."""
    torch = torch_cuda
    K, Kinv = O.reference_K()
    rng = np.random.default_rng(2024)
    base = O.synthetic_pair(6000, seed=77)["px"]
    for trial in range(24):
        B = int(rng.integers(1, 4))
        n = int(rng.integers(8, 6000))
        H = int(rng.integers(1, 5000))
        variant = int(rng.integers(-1, 11))          # 10 = constant-bank kernel
        solver = int(rng.integers(0, 2))
        px = np.stack([np.ascontiguousarray(base[rng.permutation(6000)[:n]]) for _ in range(B)])
        h = pkg.BatchedPairs(K, Kinv, B, n, H)
        h.set_option(2, variant)
        h.set_option(5, solver)
        h.set_points_xy(torch.from_numpy(px).cuda())
        seed = int(rng.integers(0, 2**62))
        h.estimate_e(H, seed, THR)
        bi, bc = h.get_best()
        for b in range(B):
            Eg = h.get_E_candidates(b).cpu().numpy()
            got = h.get_inlier_counts(b).cpu().numpy()
            want = counts_f32(oracle_c, Eg, gpu_x(h, b))
            assert np.array_equal(got, want), (trial, B, n, H, variant, solver, h.score_plan())
            assert bc[b] == got.max() and bi[b] == int(np.argmax(got)), (trial, B, n, H, variant)
            assert np.array_equal(h.get_E()[b].reshape(9), Eg[bi[b]])
        h.close()


@pytest.mark.parametrize("H", [200, 700, 3000])
def test_symmetric_epipolar_metric(pkg, O, oracle_c, torch_cuda, scene_small, H):
    """SFMB200_OPT_SCORE_METRIC = 1: the symmetric epipolar distance the reference's calculateInliers was written to compute
    (sfm.cu:155-221, SURVEY Q14), on the same kernel skeleton (three tile sizes), bit-exact against the fp32 port of its
    fma tree, banded against fp64, and consistent through the later classifiers."""
    torch = torch_cuda
    x, n = scene_small["x"], len(scene_small["x"])
    h = make_handle(pkg, scene_small, H)
    h.set_option(9, 1)
    h.set_points_xy(torch.from_numpy(scene_small["px"]).cuda())
    h.estimate_e(H, 1237, THR)
    assert h.score_plan()["variant"] >= 0                      # the fused small path is Sampson-only
    Eg = h.get_E_candidates().cpu().numpy()
    got = h.get_inlier_counts().cpu().numpy()
    xg = gpu_x(h)
    c32 = np.zeros(H, np.int32)
    oracle_c.oracle_counts_sym_f32(P(np.ascontiguousarray(Eg)), H, P(xg), n, C.c_float(THR), P(c32, ip))
    assert np.array_equal(got, c32)
    c64, amb = np.zeros(H, np.int32), np.zeros(H, np.int32)
    oracle_c.oracle_counts_sym_f64(P(np.ascontiguousarray(Eg)), H, P(xg), n, C.c_double(THR), C.c_double(BAND), P(c64, ip), P(amb, ip))
    assert np.all(np.abs(got - c64) <= amb)
    cpy, _ = O.symmetric_counts(Eg.astype(np.float64), xg, THR, band=BAND)
    assert np.array_equal(cpy, c64)
    bi, bc = h.get_best()
    assert bc[0] == got.max() and bi[0] == int(np.argmax(got))
    mask = h.get_inlier_mask().cpu().numpy().astype(bool)
    assert mask.sum() == bc[0]
    # d_sym = n^2 (1/A + 1/B) >= 4 n^2 / (A + B) = 4 x Sampson: an inlier of the symmetric test at thr is a Sampson inlier at
    # thr / 4 (up to a borderline decision), let alone at thr
    hs = make_handle(pkg, scene_small, H)
    hs.set_points_xy(torch.from_numpy(scene_small["px"]).cuda())
    hs.estimate_e(H, 1237, THR)
    assert np.array_equal(hs.get_E_candidates().cpu().numpy(), Eg)
    samp = hs.get_inlier_counts().cpu().numpy()
    hs.estimate_e(H, 1237, THR / 4)
    samp4 = hs.get_inlier_counts().cpu().numpy()
    assert np.all(got <= samp) and np.all(got <= samp4 + 2) and got.sum() < samp.sum()
    # downstream: inliers-only triangulation keeps exactly the metric's inliers
    h.set_option(3, 1)
    h.pose_candidates(); h.choose_pose(); h.triangulate()
    pts = h.get_points_host()
    assert np.all(pts[:3, ~mask] == 0) and np.all(pts[3] == 1)
    with pytest.raises(pkg.SfmError):
        h.set_option(9, 2)
    h.close(); hs.close()


def test_disjoint_permutation_sampler_on_device(pkg, O, torch_cuda, scene_small):
    """estimateE() with no arguments means what sfm.cu:95-104 means: H = N/8 rows from ONE permutation, drawn on the device;
    identical to feeding the oracle's rows explicitly, on the general and on the fused small path."""
    torch = torch_cuda
    n = len(scene_small["px"])
    d_px = torch.from_numpy(scene_small["px"]).cuda()
    H = n // 8
    rows = O.sample_indices_disjoint(77, H, n)
    for small in (0, 1):
        a, b = make_handle(pkg, scene_small, H), make_handle(pkg, scene_small, H)
        for h in (a, b):
            h.set_option(7, small)
            h.set_points_xy(d_px)
        a.set_option(10, 1)
        a.estimate_e(H, 77, THR)
        b.estimate_e(H, 0, THR, d_idx=torch.from_numpy(rows).cuda())
        assert np.array_equal(a.get_E_candidates().cpu().numpy(), b.get_E_candidates().cpu().numpy())
        assert np.array_equal(a.get_inlier_counts().cpu().numpy(), b.get_inlier_counts().cpu().numpy())
        assert np.array_equal(a.get_E(), b.get_E())
        with pytest.raises(pkg.SfmError):
            a.estimate_e(H + 1, 77, THR)                       # 8 H > n: not a permutation any more
        a.close(); b.close()
    ipair = pkg.ImagePair(scene_small["K"], scene_small["Kinv"], 2, n)
    ipair.set_points_xy(d_px)
    ipair.estimateE()                                          # the reference's call
    ref = make_handle(pkg, scene_small, H)
    ref.set_points_xy(d_px)
    ref.estimate_e(H, 0, THR, d_idx=torch.from_numpy(O.sample_indices_disjoint(0, H, n)).cuda())
    assert np.array_equal(ipair.get_E(), ref.get_E()) and ipair.H == H
    ipair.close(); ref.close()
