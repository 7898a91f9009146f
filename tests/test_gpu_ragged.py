"""Batches with a different number of correspondences per pair (the *_ragged entry points of include/sfmb200.h).

The contract: pair b of a ragged batch gives the same bits as a one-pair handle holding only pair b's rows (n = count_b)
with the batch's per-pair seed.  The GPU tests compare every pair against such a handle; the CPU tests cover the pack /
unpack helper and the Python-side argument checks."""
import ctypes as C
import math

import numpy as np
import pytest

THR = 1e-6
SEED_STEP = 0x632BE59BD9B4E019
OPT_COMPAT, OPT_VARIANT, OPT_TRI, OPT_SMALL, OPT_SAMPLER, OPT_METRIC = 1, 2, 3, 7, 10, 9


def pair_seed(seed, b):
    return (seed + SEED_STEP * b) % (1 << 64)


# ---------------------------------------------------------------------------------------------------------------------
# CPU tier
# ---------------------------------------------------------------------------------------------------------------------
def test_pack_unpack_round_trip(pkg):
    rng = np.random.default_rng(3)
    parts = [rng.standard_normal((c, 4)).astype(np.float32) for c in (8, 9, 64, 513, 8)]
    packed, offsets = pkg.pack_ragged(parts)
    assert packed.dtype == np.float32 and packed.shape == (sum(len(p) for p in parts), 4) and packed.flags["C_CONTIGUOUS"]
    assert offsets.dtype == np.int32 and offsets.tolist() == [0, 8, 17, 81, 594, 602]
    back = pkg.unpack_ragged(packed, offsets)
    assert len(back) == len(parts) and all(np.array_equal(a, b) for a, b in zip(parts, back))
    # the packed SoA output layout of run_host_ragged: pair b's [4][count_b] block at float 4 * offsets[b]
    flat = np.arange(4 * offsets[-1], dtype=np.float32)
    blocks = [p.reshape(4, -1) for p in pkg.unpack_ragged(flat.reshape(-1, 4), offsets)]
    for b, blk in enumerate(blocks):
        c = offsets[b + 1] - offsets[b]
        assert blk.shape == (4, c) and np.array_equal(blk.reshape(-1), flat[4 * offsets[b]:4 * offsets[b + 1]])


def test_pack_torch_tensors(pkg):
    import torch

    parts = [torch.arange(4 * c, dtype=torch.float64).reshape(c, 4) for c in (8, 20)]
    packed, offsets = pkg.pack_ragged(parts)
    assert packed.dtype == torch.float32 and tuple(packed.shape) == (28, 4) and offsets.tolist() == [0, 8, 28]
    assert all(torch.equal(a.float(), b) for a, b in zip(parts, pkg.unpack_ragged(packed, offsets)))


@pytest.mark.parametrize("offsets,rows,msg", [
    ([0, 8], 8, "pairs \\+ 1"),                     # wrong length
    ([1, 9, 17], 16, "offsets\\[0\\]"),
    ([0, 20, 12], 12, "must not decrease"),
    ([0, 7, 20], 20, "\\[8, max_points"),
    ([0, 8, 109], 109, "\\[8, max_points"),         # 101 > max_points = 100
    ([0, 8, 20], 21, "rows"),
])
def test_offsets_checks(pkg, offsets, rows, msg):
    with pytest.raises(ValueError, match=msg):
        pkg.check_offsets(np.array(offsets, np.int32), 2, 100, rows)


def test_offsets_checks_accept_and_convert(pkg):
    o = pkg.check_offsets([0, 8, 108], 2, 100, 108)
    assert o.dtype == np.int32 and o.tolist() == [0, 8, 108]
    with pytest.raises(TypeError):
        pkg.check_offsets(np.array([0.0, 8.0, 16.0]), 2, 100)


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier
# ---------------------------------------------------------------------------------------------------------------------
MAXP = 1100
H = 2300          # several tiles for every variant: 2048 (4), 512 (6), 256 (9), 1024 (10) hypotheses per tile


def _counts(B=40, seed=5):
    fixed = [8, 9, 63, 64, 65, 511, 512, 513, MAXP, MAXP - 1, 10, 11]
    rng = np.random.default_rng(seed)
    return fixed + [int(c) for c in rng.integers(8, MAXP + 1, B - len(fixed))]


def _scene(O, counts, seed0=100):
    return [np.ascontiguousarray(O.synthetic_pair(c, seed=seed0 + b)["px"], dtype=np.float32) for b, c in enumerate(counts)]


def _opts(h, variant=-1, metric=0, compat=1, tri=0):
    h.set_option(OPT_VARIANT, variant)
    h.set_option(OPT_METRIC, metric)
    h.set_option(OPT_COMPAT, compat)
    h.set_option(OPT_TRI, tri)
    h.set_option(OPT_SMALL, 0)


def _pair_results(h, b):
    """Per-pair results of a handle after estimate + poses + triangulation."""
    idx, cnt = h.get_best()
    return {"counts": h.get_inlier_counts(b).cpu().numpy(), "best": (int(idx[b]), int(cnt[b])), "E": h.get_E()[b].copy(),
            "P": h.get_poses()[b].copy(), "pose": int(h.get_pose_index()[b]), "points": h.get_points_host(b),
            "mask": h.get_inlier_mask(b).cpu().numpy()}


def _assert_same(got, want, where):
    for k in want:
        a, b = got[k], want[k]
        ok = a == b if isinstance(b, (int, tuple)) else (a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)))
        assert ok, f"{where}: {k} differs"


def _staged(h, Hh, seed, d_idx=None):
    h.estimate_e(Hh, seed, THR, d_idx)
    h.pose_candidates()
    h.choose_pose()
    h.triangulate()


@pytest.fixture(scope="module")
def ragged_scene(O):
    counts = _counts()
    return counts, _scene(O, counts)


def _single(pkg, O, px_b, seed_b, d_idx_b, opts, Hh=H):
    import torch

    K, Kinv = O.reference_K()
    one = pkg.BatchedPairs(K, Kinv, 1, max(MAXP, len(px_b)), Hh)
    _opts(one, **opts)
    one.set_points_xy(torch.from_numpy(px_b[None]).cuda())
    _staged(one, Hh, seed_b, None if d_idx_b is None else torch.from_numpy(np.ascontiguousarray(d_idx_b[None])).cuda())
    r = _pair_results(one, 0)
    one.close()
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("metric", [0, 1])
@pytest.mark.parametrize("variant", [4, 6, 9, 10, -1])
def test_each_pair_equals_its_one_pair_handle(pkg, O, ragged_scene, variant, metric):
    import torch

    counts, px = ragged_scene
    B, seed = len(counts), 77
    K, Kinv = O.reference_K()
    rng = np.random.default_rng(variant + 10 * metric + 20)
    rows = {"caller": np.stack([rng.integers(0, c, (H, 8)) for c in counts]).astype(np.int32),
            "caller_oob": rng.integers(0, MAXP, (B, H, 8)).astype(np.int32)}
    h = pkg.BatchedPairs(K, Kinv, B, MAXP, H)
    h.set_points_xy_ragged([torch.from_numpy(p).cuda() for p in px])
    assert h.point_counts().tolist() == counts
    for compat, tri, src in [(1, 0, "device"), (0, 1, "caller"), (1, 1, "caller_oob"), (0, 0, "device")]:
        opts = dict(variant=variant, metric=metric, compat=compat, tri=tri)
        _opts(h, **opts)
        d_idx = rows.get(src)
        _staged(h, H, seed, None if d_idx is None else torch.from_numpy(d_idx).cuda())
        if variant >= 0 and metric == 0:
            assert h.score_plan()["variant"] == variant
        for b in range(B):
            want = _single(pkg, O, px[b], pair_seed(seed, b), None if d_idx is None else d_idx[b], opts)
            _assert_same(_pair_results(h, b), want, f"pair {b} (count {counts[b]}) {opts} rows {src}")
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("compat", [1, 0])
def test_run_device_ragged_equals_one_pair_run_device(pkg, O, ragged_scene, compat):
    import torch

    counts, px = ragged_scene
    B, seed = len(counts), 9
    K, Kinv = O.reference_K()
    h = pkg.BatchedPairs(K, Kinv, B, MAXP, H)
    _opts(h, compat=compat)
    h.set_option(OPT_SMALL, 1)          # never taken in per-pair-count mode
    before = h.launch_count()
    packed, offsets = pkg.pack_ragged(px)
    h.run_device_ragged(torch.from_numpy(packed).cuda(), H, seed, THR, offsets=offsets)
    assert h.launch_count() - before >= 5 and h.score_plan()["variant"] >= 0          # the general path ran
    one = pkg.BatchedPairs(K, Kinv, 1, MAXP, H)
    _opts(one, compat=compat)
    for b in range(B):
        one.run_device(torch.from_numpy(px[b][None]).cuda(), H, pair_seed(seed, b), THR)
        want = _pair_results(one, 0)
        _assert_same(_pair_results(h, b), want, f"pair {b} (count {counts[b]}) compat {compat}")
    h.close(); one.close()


@pytest.mark.gpu
def test_uneven_split_crosses_pair_boundaries(pkg, O):
    import torch

    rng = np.random.default_rng(8)
    counts = [200000] + [int(c) for c in rng.integers(8, 65, 300)]
    px = _scene(O, counts, seed0=500)
    B, Hh, seed = len(counts), 4096, 31
    K, Kinv = O.reference_K()
    h = pkg.BatchedPairs(K, Kinv, B, counts[0], Hh)
    _opts(h)
    h.set_points_xy_ragged(px)
    _staged(h, Hh, seed)
    plan = h.score_plan()
    # the work split of the scoring kernel (score.cu: ChunkWalk): CTA c owns units [c U / G, (c + 1) U / G) of the
    # pair-major space, pair b's units being [T goff[b], T goff[b + 1])
    goff = np.concatenate([[0], np.cumsum([(c + 63) // 64 for c in counts])]).astype(np.int64) * plan["tiles"]
    U, G = int(goff[-1]), plan["ctas"]
    lo = np.array([c * U // G for c in range(G)]), np.array([(c + 1) * U // G for c in range(G)])
    first_pair = np.searchsorted(goff, lo[0], side="right") - 1
    last_pair = np.searchsorted(goff, lo[1] - 1, side="right") - 1
    assert np.any(first_pair != last_pair), "no share crosses a pair boundary"
    assert np.sum(first_pair == 0) > G // 2, "the large pair is not spread over the CTAs"
    for b in range(B):
        want = _single(pkg, O, px[b], pair_seed(seed, b), None, {}, Hh)
        _assert_same(_pair_results(h, b), want, f"pair {b} (count {counts[b]})")
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("tri", [0, 1])
def test_equal_counts_equal_the_uniform_ingest(pkg, O, tri):
    import torch

    B, n, seed = 12, 700, 5
    px = np.stack(_scene(O, [n] * B, seed0=900))
    K, Kinv = O.reference_K()
    res = []
    for ragged in (False, True):
        h = pkg.BatchedPairs(K, Kinv, B, MAXP, H)
        _opts(h, tri=tri)
        if ragged:
            h.set_points_xy_ragged(list(px))
        else:
            h.set_points_xy(torch.from_numpy(px).cuda())
        _staged(h, H, seed)
        res.append([_pair_results(h, b) for b in range(B)])
        if ragged:
            h.run_device_ragged(list(px), H, seed + 1, THR)
        else:
            h.run_device(torch.from_numpy(px).cuda(), H, seed + 1, THR)
        res.append([_pair_results(h, b) for b in range(B)])
        h.close()
    for b in range(B):
        _assert_same(res[2][b], res[0][b], f"staged pair {b}")
        _assert_same(res[3][b], res[1][b], f"run_device pair {b}")


# fp32 port of the scoring test (bit-exact bar) and the fp64 truth with its borderline band, as in test_gpu_parity.py
BAND = 1e-4
_fp, _ip = C.POINTER(C.c_float), C.POINTER(C.c_int32)


def counts_f32(oracle_c, E32, x):
    out = np.zeros(len(E32), np.int32)
    oracle_c.oracle_counts_f32(np.ascontiguousarray(E32).ctypes.data_as(_fp), len(E32), x.ctypes.data_as(_fp), len(x),
                               C.c_float(THR), out.ctypes.data_as(_ip))
    return out


def counts_f64(oracle_c, E32, x):
    cnt, amb = np.zeros(len(E32), np.int32), np.zeros(len(E32), np.int32)
    oracle_c.oracle_counts_f64(np.ascontiguousarray(E32).ctypes.data_as(_fp), len(E32), x.ctypes.data_as(_fp), len(x),
                               C.c_double(THR), C.c_double(BAND), cnt.ctypes.data_as(_ip), amb.ctypes.data_as(_ip))
    return cnt, amb


def gpu_x(h, pair):
    """(count_b, 4) normalised correspondences exactly as the device holds them."""
    X0, X1 = h.get_X(0, pair).cpu().numpy(), h.get_X(1, pair).cpu().numpy()
    return np.ascontiguousarray(np.stack([X0[0], X0[1], X1[0], X1[1]], 1))


@pytest.mark.gpu
def test_counts_and_winner_against_the_oracle(pkg, O, oracle_c):
    counts, Hh, seed = [900, 1500, 333, 2048], 3000, 1237
    px = _scene(O, counts, seed0=4321)
    K, Kinv = O.reference_K()
    h = pkg.BatchedPairs(K, Kinv, len(counts), max(counts), Hh)
    h.set_points_xy_ragged(px)
    h.estimate_e(Hh, seed, THR)
    bi, bc = h.get_best()
    E = h.get_E()
    for b, n in enumerate(counts):
        Eg = h.get_E_candidates(b).cpu().numpy()
        xg = gpu_x(h, b)
        assert xg.shape == (n, 4)
        got = h.get_inlier_counts(b).cpu().numpy()
        assert np.array_equal(got, counts_f32(oracle_c, Eg, xg)), f"pair {b}"
        c64, amb = counts_f64(oracle_c, Eg, xg)
        assert np.all(np.abs(got - c64) <= amb), f"pair {b}"
        assert bc[b] == got.max() and bi[b] == int(np.argmax(got))
        assert np.array_equal(E[b].reshape(9), Eg[bi[b]])
        x = O.normalise_points(px[b], Kinv)
        d = O.e_distance(Eg, O.hypotheses(x, O.sample_indices(pair_seed(seed, b), Hh, n)))
        assert np.mean(d < 1e-4) >= 0.995 and np.median(d) < 1e-6, f"pair {b}"
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["pinned_small", "pinned_large", "pageable"])
def test_run_host_ragged_equals_device_path(pkg, O, kind):
    import torch

    counts = {"pinned_small": [8, 9, 640, 3001, 1200, 65], "pinned_large": [60000, 8, 70001, 55555, 64, 90000],
              "pageable": [500, 8, 7000, 513, 64, 9]}[kind]
    px = _scene(O, counts, seed0=70)
    packed, offsets = pkg.pack_ragged(px)
    if kind.startswith("pinned"):           # both sides of the 4 MB zero-copy limit
        assert (packed.nbytes <= 4 << 20) == (kind == "pinned_small")
    if kind.startswith("pinned"):
        pinned = torch.empty(packed.shape, dtype=torch.float32, pin_memory=True)
        pinned.numpy()[:] = packed
        host_in = pinned.numpy()
    else:
        host_in = packed
    K, Kinv = O.reference_K()
    B, Hh, seed = len(counts), 1500, 3
    h = pkg.BatchedPairs(K, Kinv, B, max(counts), Hh)
    out = h.run_host_ragged(host_in, Hh, seed, THR, offsets=offsets)
    dev = pkg.BatchedPairs(K, Kinv, B, max(counts), Hh)
    dev.run_device_ragged(torch.from_numpy(packed).cuda(), Hh, seed, THR, offsets=offsets)
    idx, cnt = dev.get_best()
    E, P, pose = dev.get_E().reshape(B, 9), dev.get_poses(), dev.get_pose_index()
    assert np.array_equal(out["E"], E) and np.array_equal(out["pose_index"], pose) and np.array_equal(out["inliers"], cnt)
    for b, n in enumerate(counts):
        assert np.array_equal(out["P"][b], P[b, pose[b]].reshape(16))
        pts = dev.get_points_host(b)
        assert pts.shape == (4, n) and np.array_equal(out["points"][b], pts)
        assert np.array_equal(out["points_packed"][4 * offsets[b]:4 * offsets[b + 1]].reshape(4, n), pts)
    assert h.point_counts().tolist() == counts
    h.close(); dev.close()


@pytest.mark.gpu
def test_adaptive_on_a_ragged_batch(pkg, O):
    counts = [3000, 800, 5000, 64, 1999]
    px = [np.ascontiguousarray(O.synthetic_pair(c, outlier_frac=0.45, noise_px=0.5, seed=40 + b)["px"], dtype=np.float32)
          for b, c in enumerate(counts)]
    K, Kinv = O.reference_K()
    B, H_max, first, growth, seed, conf = len(counts), 16384, 256, 2, 13, 0.99
    h = pkg.BatchedPairs(K, Kinv, B, max(counts), H_max)
    h.set_points_xy_ragged(px)
    h.estimate_e(H_max, seed, THR)
    all_counts = np.stack([h.get_inlier_counts(b).cpu().numpy() for b in range(B)])
    # the rule with w = best / count_b per pair, every pair satisfied
    bounds, want = O.adaptive_rounds(H_max, first, growth), None
    for done in bounds:
        ok = True
        for b, n in enumerate(counts):
            w8 = (all_counts[b, :done].max() / n) ** 8
            ok &= w8 >= 1.0 or (w8 > 0.0 and done >= math.log1p(-float(np.float32(conf))) / math.log1p(-w8))
        if ok:
            want = done
            break
    want = want or bounds[-1]
    used = h.estimate_e_adaptive(H_max, seed, THR, conf, first, growth)
    E_a, (idx_a, cnt_a) = h.get_E().copy(), h.get_best()
    assert used == want
    h.estimate_e(used, seed, THR)
    idx_p, cnt_p = h.get_best()
    assert np.array_equal(idx_a, idx_p) and np.array_equal(cnt_a, cnt_p) and np.array_equal(E_a, h.get_E())
    h.close()


def _raw(h, name, *args):
    return h.lib.raw(name)(h._h, *args)


def _snapshot(h):
    idx, cnt = h.get_best()
    return (h.launch_count(), idx.tolist(), cnt.tolist(), h.point_counts().tolist(),
            [h.get_inlier_counts(b).cpu().numpy().tolist() for b in range(h.pairs)], h.get_points_host(1).tobytes())


@pytest.mark.gpu
def test_bad_arguments_change_nothing(pkg, O):
    import torch

    counts = [40, 100, 64]
    px = _scene(O, counts, seed0=11)
    packed, offsets = pkg.pack_ragged(px)
    K, Kinv = O.reference_K()
    h = pkg.BatchedPairs(K, Kinv, 3, 100, 500)
    d_px = torch.from_numpy(packed).cuda()
    h.run_device_ragged(d_px, 500, 1, THR, offsets=offsets)
    before = _snapshot(h)
    p, null = C.c_void_p(d_px.data_ptr()), C.c_void_p(0)
    hp = C.c_void_p(packed.ctypes.data)
    o = lambda a: np.array(a, np.int32)            # noqa: E731
    bad_offsets = [o([1, 41, 141, 205]), o([0, 100, 40, 204]), o([0, 7, 107, 171]), o([0, 40, 141, 205])]
    keep = []
    for offs in bad_offsets:
        keep.append(offs)
        op = C.c_void_p(offs.ctypes.data)
        assert _raw(h, "sfmb200_set_points_xy_ragged", p, op) == -1
        assert _raw(h, "sfmb200_run_device_ragged", p, op, 500, C.c_uint64(1), C.c_float(THR)) == -1
        assert _raw(h, "sfmb200_run_host_ragged", hp, op, 500, C.c_uint64(1), C.c_float(THR), null, null, null, null, null) == -1
    op = C.c_void_p(offsets.ctypes.data)
    assert _raw(h, "sfmb200_set_points_xy_ragged", null, op) == -1
    assert _raw(h, "sfmb200_set_points_xy_ragged", p, null) == -1
    for Hh, thr in [(0, THR), (501, THR), (500, 0.0), (500, float("nan")), (500, -1.0)]:
        assert _raw(h, "sfmb200_run_device_ragged", p, op, Hh, C.c_uint64(1), C.c_float(thr)) == -1
        assert _raw(h, "sfmb200_run_host_ragged", hp, op, Hh, C.c_uint64(1), C.c_float(thr), null, null, null, null, null) == -1
    assert _raw(h, "sfmb200_get_point_counts", null) == -1
    assert _snapshot(h) == before
    h.close()


@pytest.mark.gpu
def test_stages_that_refuse_per_pair_counts(pkg, O):
    import torch

    counts = [300, 500]
    px = _scene(O, counts, seed0=61)
    K, Kinv = O.reference_K()
    h = pkg.BatchedPairs(K, Kinv, 2, 500, 256)
    h.set_points_xy_ragged(px)
    h.estimate_e(256, 3, THR)
    h.pose_candidates(); h.choose_pose(); h.triangulate()
    cloud = torch.zeros((4, 500), dtype=torch.float32, device="cuda")
    cnt = torch.zeros(500, dtype=torch.int32, device="cuda")
    cp, kp, null = C.c_void_p(cloud.data_ptr()), C.c_void_p(cnt.data_ptr()), C.c_void_p(0)
    calls = {
        "refine_e": lambda: _raw(h, "sfmb200_refine_e", 2),
        "bundle_adjust": lambda: _raw(h, "sfmb200_bundle_adjust", 1, 2, null),
        "chain_views": lambda: _raw(h, "sfmb200_chain_views", cp, kp, null, null, null),
        "bundle_adjust_global": lambda: _raw(h, "sfmb200_bundle_adjust_global", cp, kp, 2, null, null),
        "find_homography": lambda: _raw(h, "sfmb200_find_homography", 64, C.c_uint64(1), C.c_float(5.0), null, null),
        "estimate_e_mg": lambda: _raw(h, "sfmb200_estimate_e_mg", null, 256, C.c_uint64(3), C.c_float(THR)),
        "adopt_best": lambda: _raw(h, "sfmb200_adopt_best", null, 256, C.c_uint64(3)),
    }
    for name, call in calls.items():
        launches = h.launch_count()
        assert call() == -3, name
        assert "_ragged" in h.lib.last_error() and name in h.lib.last_error()
        assert h.launch_count() == launches
    # the disjoint sampler needs 8 * H_total <= the smallest count (300)
    h.set_option(OPT_SAMPLER, 1)
    assert _raw(h, "sfmb200_estimate_e", null, 38, C.c_uint64(1), C.c_float(THR)) == -1
    assert _raw(h, "sfmb200_estimate_e", null, 37, C.c_uint64(1), C.c_float(THR)) == 0
    h.set_option(OPT_SAMPLER, 0)
    # a uniform ingest returns the handle to uniform mode: every stage works again
    h.set_points_xy(torch.from_numpy(np.stack([px[0][:300], px[1][:300]])).cuda())
    assert h.point_counts().tolist() == [300, 300]
    h.estimate_e(256, 3, THR)
    h.pose_candidates(); h.choose_pose(); h.triangulate()
    ok = ["bundle_adjust", "chain_views", "bundle_adjust_global", "refine_e", "adopt_best", "find_homography"]
    for name in ok:
        assert calls[name]() == 0, (name, h.lib.last_error())
    assert calls["estimate_e_mg"]() == -3 and "_ragged" not in h.lib.last_error()      # now only mg_init is missing
    h.close()
