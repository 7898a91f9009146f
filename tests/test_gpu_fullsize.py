"""GPU tier: BASELINE.json configs 3, 4 and 5 at FULL size.  Size-independent properties (sharded arg-max == single-launch
arg-max, batched == single for sampled pairs, published count == size of the published mask, triangulated inliers
reproject onto their observations), and the fp64 / fp32-port oracle on samples the CPU can afford: hypotheses at tile and
shard edges, whole pairs of the batch, a 65,536-point sample of the triangulation."""
import ctypes as C
import json

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
THR = 1e-6
BAND = 1e-4          # borderline band of the fp64 comparison (tests/test_gpu_parity.py explains the value)
PAIR_SEED_STEP = 0x632BE59BD9B4E019

fp = C.POINTER(C.c_float)
ip = C.POINTER(C.c_int32)
dp = C.POINTER(C.c_double)


def P(a, t=fp):
    return a.ctypes.data_as(t)


def counts_f32(oracle_c, E32, x, thr=THR):
    out = np.zeros(len(E32), np.int32)
    oracle_c.oracle_counts_f32(P(np.ascontiguousarray(E32)), len(E32), P(x), len(x), C.c_float(thr), P(out, ip))
    return out


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


def tri_c(oracle_c, x, M):
    """O.triangulate through the threaded C port (same fp64 null vector, (4,n) SoA)."""
    x = np.ascontiguousarray(x, np.float32)
    out = np.empty((4, len(x)))
    oracle_c.oracle_triangulate_f64(P(x), len(x), P(np.ascontiguousarray(M, np.float64), dp), P(out, dp))
    return out


def check_e_candidates(O, Eg, E64):
    """Device E candidates against the fp64 null vectors of the same rows: the bar of test_estimate_e_against_oracle."""
    d = O.e_distance(Eg, E64)
    within = float(np.mean(d < 1e-4))
    assert within >= 0.995, f"{within} of hypotheses within 1e-4"
    assert np.median(d) < 1e-6, np.median(d)
    return within, float(np.median(d))


def rel_error(pts, ref):
    """Per point: max |xyz - ref| relative to the point's size (test_poses_cheirality_triangulation_compat)."""
    return np.abs(pts[:3] - ref[:3]).max(axis=0) / np.maximum(np.abs(ref[:3]).max(axis=0), 1e-3)


def check_vote_pose(O, x, E, Pg, ind, mask, tri=None):
    """compat = 0 against the oracle: the textbook candidates as a set, and the pose the inlier vote selects equals the
    oracle's vote winner over the device's mask.  Returns the oracle's vote margin as a fraction of the votes; the
    selected pose is only pinned (and the margin must allow it) when the margin exceeds 1 %."""
    Po = O.pose_candidates(np.asarray(E, np.float64).reshape(3, 3), compat=False)
    perm = O.match_candidate_set(Pg, Po, tol=1e-4)
    assert perm is not None, np.abs(Pg - Po).max()
    votes = O.cheirality_votes(x, Po, mask, tri=tri or O.triangulate)
    top = sorted(votes)
    margin = (top[3] - top[2]) / max(sum(votes), 1)
    assert margin > 0.01, votes
    assert np.abs(Pg[int(ind)] - Po[int(np.argmax(votes))]).max() < 1e-4, (int(ind), votes)
    return margin


def sample_hypotheses(rng, H, winner, tile, edges, total=2048):
    """Winner, both ends, both sides of the hypothesis-tile edges around the winner and at random tiles, both sides of
    the shard edges, then random indices up to `total`."""
    s = {winner, 0, H - 1}
    k = winner // tile
    tiles = list(range(max(k - 2, 0), k + 4)) + [int(t) for t in rng.integers(1, H // tile, 120)]
    for e in [t * tile for t in tiles] + list(edges):
        s.update(i for i in (e - 1, e) if 0 <= i < H)
    while len(s) < total:
        s.add(int(rng.integers(0, H)))
    return np.array(sorted(s))


def test_config3_one_million_by_one_million_slices_agree(pkg, O, oracle_c):
    """C3: 1M correspondences x 1M hypotheses.  Hypothesis slices (the multi-GPU decomposition) scored one after
    the other on one GPU and merged by MAX of the packed key select the same hypothesis with the same count as a
    single launch over all of them, and the regenerated E is bit-identical.  The single launch is pinned to the
    oracle on ~2,048 hypotheses (tile and shard edges, the winner): E candidates against fp64, counts bit-exact
    against the fp32 port over all 1,048,576 points; the published (index, count) is the first maximum of all counts
    and the published mask is the fp32 Sampson mask of the winner, point by point."""
    import torch

    K, Kinv = O.reference_K()
    n = H = 1 << 20
    sc = O.synthetic_pair(n, seed=1234)
    h = pkg.BatchedPairs(K, Kinv, 1, n, H)
    h.set_points_xy(torch.from_numpy(sc["px"]).cuda())
    h.estimate_e(H, 1237, THR)
    idx_all, cnt_all = (int(v[0]) for v in h.get_best())
    E_all = h.get_E().copy()
    assert 0 < cnt_all <= n and 0 <= idx_all < H
    counts = h.get_inlier_counts().cpu().numpy()
    Ecand = h.get_E_candidates().cpu().numpy()
    tile = h.score_plan()["hyp_per_cta"]
    xg = gpu_x(h)
    assert (idx_all, cnt_all) == (int(np.argmax(counts)), int(counts.max()))
    assert np.array_equal(E_all[0].reshape(9), Ecand[idx_all])
    keys = []
    parts = 4
    for r in range(parts):
        lo, hi = pkg.sharding.shard_range(H, r, parts)
        h.estimate_e(hi - lo, 1237, THR, H_total=H, h_begin=lo)
        keys.append(h.best_buffer().clone())
        i, c = h.get_best()
        assert lo <= int(i[0]) < hi
    best = torch.stack(keys).max(dim=0).values
    h.best_buffer().copy_(best)
    h.adopt_best(H, 1237)
    idx_m, cnt_m = (int(v[0]) for v in h.get_best())
    assert (idx_m, cnt_m) == (idx_all, cnt_all) and pkg.sharding.unpack_key(int(best[0])) == (cnt_all, idx_all)
    assert np.array_equal(h.get_E(), E_all)
    mask = h.get_inlier_mask()
    assert int(mask.sum()) == cnt_all
    m = mask.cpu().numpy().astype(bool)
    assert m[~sc["is_outlier"]].mean() > 0.5 and m[sc["is_outlier"]].mean() < 0.1
    assert np.array_equal(m, O.sampson_mask_f32(E_all[0], xg, THR))
    h.close()

    # oracle on sampled hypotheses
    rng = np.random.default_rng(3)
    edges = [e for r in range(parts) for e in pkg.sharding.shard_range(H, r, parts)]
    S = sample_hypotheses(rng, H, idx_all, tile, edges)
    rows = np.concatenate([O.sample_indices(1237, 1, n, h0=int(s)) for s in S])
    within, med = check_e_candidates(O, Ecand[S], O.hypotheses(xg, rows))
    c32 = counts_f32(oracle_c, Ecand[S], xg)
    bad = np.flatnonzero(c32 != counts[S])
    assert len(bad) == 0, [(int(S[i]), int(counts[S[i]]), int(c32[i])) for i in bad[:8]]
    sub = np.concatenate([[idx_all], rng.choice(S[S != idx_all], 127, replace=False)])
    c64, amb = counts_f64(oracle_c, Ecand[sub], xg)
    assert np.all(np.abs(counts[sub] - c64) <= amb)
    rec = {"leg": "C3", "sampled": int(len(S)), "tile": int(tile), "E_within_1e-4": within, "E_median_distance": med,
           "winner": idx_all, "winner_count_gpu": cnt_all, "winner_count_fp32_port": int(c32[np.searchsorted(S, idx_all)]),
           "winner_count_fp64": int(c64[0]), "winner_borderline": int(amb[0]),
           "sub128_max_abs_diff_vs_fp64": int(np.abs(counts[sub] - c64).max())}
    print("\noracle pin record:", json.dumps(rec))


def test_config4_4096_pairs_batched_equals_single(pkg, O, oracle_c):
    """C4: 4,096 pairs x 4,096 correspondences x 4,096 hypotheses in one batched run; sampled pairs re-run alone
    give the same bits (pair b draws its samples from seed + pair offset, so the single run injects the batch's
    E and compares the downstream stages), and every published count is the size of the published mask.  Sixteen
    pairs run the whole path through the oracle with their own sample stream: E candidates, counts and arg-max; the
    reference-semantics poses, cheirality index and points of the batch as run; then the same handle in inlier-vote
    mode, which runs the vote kernel with one CTA per pair."""
    import torch

    K, Kinv = O.reference_K()
    pairs, n, H, seed = 4096, 4096, 4096, 99
    scenes = [O.synthetic_pair(n, seed=500 + i) for i in range(8)]
    px = np.stack([scenes[b % 8]["px"] for b in range(pairs)])
    h = pkg.BatchedPairs(K, Kinv, pairs, n, H)
    h.run_device(torch.from_numpy(px).cuda(), H, seed, THR)
    idx, cnt = h.get_best()
    E, Pp, ind = h.get_E(), h.get_poses(), h.get_pose_index()
    assert np.all(cnt > 0) and np.all(cnt <= n) and np.all((idx >= 0) & (idx < H)) and np.all(np.isfinite(E))
    # pairs 0 and 8 see the same correspondences but different sample streams: same scene, (almost surely) different winner index
    assert np.array_equal(px[0], px[8])
    for b in (0, 1, 777, 4095):
        assert int(h.get_inlier_mask(b).sum()) == int(cnt[b])
        x = O.normalise_points(px[b], Kinv)
        assert int(O.sampson_mask_f32(E[b], x, THR).sum()) == int(cnt[b])
        pts = h.get_points_host(b)
        s1 = pkg.BatchedPairs(K, Kinv, 1, n, 64)
        s1.set_points_xy(torch.from_numpy(px[b][None]).cuda())
        s1.set_E(E[b][None])
        s1.pose_candidates(); s1.choose_pose(); s1.triangulate()
        assert np.array_equal(s1.get_poses()[0], Pp[b]) and int(s1.get_pose_index()[0]) == int(ind[b])
        assert np.array_equal(s1.get_points_host(0), pts)
        s1.close()

    rng = np.random.default_rng(4)
    sampled = [0, 1, 7, 8, 511, 512, 2047, 2048, 4095]
    sampled += sorted(int(b) for b in rng.choice(np.setdiff1d(np.arange(pairs), sampled), 7, replace=False))
    within_all, xs, pts_c = [], {}, {}
    for b in sampled:
        xg = xs[b] = gpu_x(h, b)
        pair_seed = (seed + PAIR_SEED_STEP * b) % (1 << 64)
        Ec = h.get_E_candidates(b).cpu().numpy()
        got = h.get_inlier_counts(b).cpu().numpy()
        within_all.append(check_e_candidates(O, Ec, O.hypotheses(xg, O.sample_indices(pair_seed, H, n)))[0])
        assert np.array_equal(got, counts_f32(oracle_c, Ec, xg)), b
        c64, amb = counts_f64(oracle_c, Ec, xg)
        assert np.all(np.abs(got - c64) <= amb), b
        assert (int(idx[b]), int(cnt[b])) == (int(np.argmax(got)), int(got.max())), b
        assert np.array_equal(E[b].reshape(9), Ec[idx[b]]), b
        # reference semantics: the candidates in the reference's order (choosePose leaves their inverses in place),
        # cheirality of correspondence 0, points under the selected pose
        E64 = E[b].astype(np.float64)
        Pcand = np.stack([np.linalg.inv(Pp[b][i].astype(np.float64)) for i in range(4)])
        Po = O.pose_candidates(E64, compat=True)
        assert np.abs(Pcand - Po).max() < 2e-5, (b, np.abs(Pcand - Po).max())
        ind_o, Pinv_o = O.choose_pose(xg, Pcand, compat=True)
        assert int(ind[b]) == ind_o, b
        assert np.abs(Pp[b] - Pinv_o).max() < 5e-5, b
        pts_c[b] = h.get_points_host(b)
        rel = rel_error(pts_c[b], O.triangulate(xg, Pp[b][ind[b]].astype(np.float64)))
        inl = ~scenes[b % 8]["is_outlier"]
        assert np.median(rel[inl]) < 1e-4 and np.mean(rel[inl] < 1e-3) > 0.99, b
        assert np.mean(rel < 1e-3) > 0.97, b

    # inlier-vote semantics on the same batch: the vote kernel at 4,096 pairs
    h.set_option(1, 0)
    h.pose_candidates(); h.choose_pose(); h.triangulate()
    Pv, indv = h.get_poses(), h.get_pose_index()
    margins = []
    for b in sampled:
        xg = xs[b]
        mask = h.get_inlier_mask(b).cpu().numpy().astype(bool)
        margins.append(check_vote_pose(O, xg, E[b], Pv[b], indv[b], mask))
        rel = rel_error(h.get_points_host(b), O.triangulate(xg, Pv[b][indv[b]].astype(np.float64)))
        inl = ~scenes[b % 8]["is_outlier"]
        assert np.median(rel[inl]) < 1e-4 and np.mean(rel[inl] < 1e-3) > 0.99, b
        assert np.mean(rel < 1e-3) > 0.97, b
    h.close()
    rec = {"leg": "C4", "pairs_checked": len(sampled), "E_within_1e-4_min": min(within_all),
           "vote_margin_min": min(margins)}
    print("\noracle pin record:", json.dumps(rec))


def test_config5_one_million_points_triangulated(pkg, O, oracle_c):
    """C5: estimation + poses + cheirality + triangulation of 1,048,576 points: inliers of the selected E (vote
    mode) triangulate in front of both cameras and reproject within the inlier threshold's scale.  Against the
    oracle: the candidate set and the vote winner over the device's ~700 k inliers, and a 65,536-point sample of the
    triangulation (random points, both ends, both sides of the first point of the persistent grid's second pass).
    A second handle with the correspondences rotated by one (each point gets another FFMA2 partner, CTA and pass)
    reproduces every point bit for bit."""
    import torch

    K, Kinv = O.reference_K()
    n, H = 1 << 20, 65536
    sc = O.synthetic_pair(n, seed=77)
    h = pkg.BatchedPairs(K, Kinv, 1, n, H)
    h.set_option(1, 0)
    h.run_device(torch.from_numpy(sc["px"]).cuda(), H, 1237, THR)
    X = h.get_points_host(0).astype(np.float64)
    Pg, ind = h.get_poses()[0], int(h.get_pose_index()[0])
    M = Pg[ind].astype(np.float64)
    E = h.get_E()[0]
    m = h.get_inlier_mask().cpu().numpy().astype(bool)
    assert int(m.sum()) == int(h.get_best()[1][0]) and np.all(np.isfinite(X)) and np.all(X[3] == 1)
    x = O.normalise_points(sc["px"], Kinv)
    Y = X[:3].T @ M[:3, :3].T + M[:3, 3]
    front = (X[2] > 0) & (Y[:, 2] > 0)
    assert front[m].mean() > 0.99
    sel = m & front
    r1 = X[:2].T[sel] / X[2][sel, None] - x[sel, :2]
    r2 = Y[sel, :2] / Y[sel, 2:3] - x[sel, 2:]
    rms = np.sqrt(((r1 ** 2).sum(1) + (r2 ** 2).sum(1)).mean() / 2)
    print(f"\nC5: {int(m.sum())} inliers of {n}, {sel.sum()} in front of both cameras, reprojection rms {rms * 2360:.3f} px")
    assert rms < 1.5e-3            # the Sampson threshold is 1e-3 in these units (2.36 px)

    xg = gpu_x(h)
    margin = check_vote_pose(O, xg, E, Pg, ind, m, tri=lambda xs, Mc: tri_c(oracle_c, xs, Mc))
    # triangulation on a sample: min(ceil(n / 256), 148 * 16) CTAs stride over 256-point chunks
    second_pass = min(-(-n // 256), 148 * 16) * 256
    rng = np.random.default_rng(5)
    S = np.unique(np.concatenate([[0, 1, n - 2, n - 1], np.arange(second_pass - 256, second_pass + 256),
                                  rng.choice(n, 65536 - 516, replace=False)]))
    ref = O.triangulate(xg[S], M)
    rel = rel_error(X[:, S], ref)
    inl = m[S]
    assert np.median(rel[inl]) <= 1e-6 and rel[inl].max() <= 1e-3, (np.median(rel[inl]), rel[inl].max())
    assert np.mean(rel <= 1e-3) >= 0.999, np.mean(rel <= 1e-3)
    # every point outside 1e-3 must be ill-conditioned in fp64: the two smallest singular values of its DLT matrix nearly
    # coincide (sigma4 / sigma3 > 0.5), or the point lies so close to infinity that an fp32 solve cannot place it: the
    # first-order error of the de-homogenised point, 2^-24 sigma1 / ((sigma3 - sigma4) |w|) for the unit null vector, is
    # above 1e-5 (a hundredth of the bar).  The tail of this scene is all of the second kind: outliers near infinity.
    off = rel > 1e-3
    near_inf = 0
    if off.any():
        _, sv, Vt = np.linalg.svd(O.dlt_rows(xg[S][off], M))
        kappa = 2.0 ** -24 * sv[:, 0] / ((sv[:, 2] - sv[:, 3]) * np.abs(Vt[:, 3, 3]))
        flat = sv[:, 3] > 0.5 * sv[:, 2]
        assert np.all(flat | (kappa > 1e-5)), np.c_[S[off], rel[off], sv, kappa][~(flat | (kappa > 1e-5))]
        near_inf = int((~flat).sum())
    rec = {"leg": "C5", "inliers": int(m.sum()), "vote_margin": margin, "sampled_points": int(len(S)),
           "sampled_inliers": int(inl.sum()), "rel_inlier_median": float(np.median(rel[inl])),
           "rel_inlier_p99": float(np.quantile(rel[inl], 0.99)), "rel_inlier_max": float(rel[inl].max()),
           "rel_all_p99": float(np.quantile(rel, 0.99)), "outside_1e-3": int(off.sum()), "outside_1e-3_near_infinity": near_inf}
    print("\noracle pin record:", json.dumps(rec))

    # lane independence: index 0 stays, the rest rotate by one
    order = np.concatenate([[0], np.arange(2, n), [1]])
    h2 = pkg.BatchedPairs(K, Kinv, 1, n, 64)
    h2.set_option(1, 0)
    h2.set_points_xy(torch.from_numpy(np.ascontiguousarray(sc["px"][order])).cuda())
    h2.set_E(E[None])
    h2.pose_candidates(); h2.choose_pose(); h2.triangulate()
    assert np.array_equal(h2.get_poses()[0], Pg) and int(h2.get_pose_index()[0]) == ind
    X2 = np.empty((4, n), np.float32)
    X2[:, order] = h2.get_points_host(0)
    assert np.array_equal(X2, h.get_points_host(0)), int((X2 != h.get_points_host(0)).any(0).sum())
    h2.close()
    h.close()
