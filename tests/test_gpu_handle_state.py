"""GPU tier: what each call needs from the handle and what it leaves there (include/sfmb200.h, "handle state").

One small handle (one pair, n = 1,500, H = 512) is brought into every state a caller can leave it in.  In each state
every guarded entry point is called on a handle of its own: it either runs or is refused with SFMB200_ERR_STATE, and
the kernel launches it enqueues (sfmb200_launch_count, which bench.py reports) are pinned, on the fused single-launch
path and on the general five-launch path."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
N, H, SEED, THR = 1500, 512, 11, 1e-6
OPT_SMALL = 7
ERR_STATE = -3
E_SET = np.array([[0, 0, 0], [0, 0, -1], [0, 1, 0]], np.float32).reshape(1, 9)   # [t]x R with t = x, R = I


class Io:
    """Inputs and output buffers shared by every handle of the test."""

    def __init__(self, O):
        import torch

        self.K, self.Kinv = O.reference_K()
        self.h_px = np.ascontiguousarray(O.synthetic_pair(N, seed=77)["px"].reshape(1, N, 4), dtype=np.float32)
        self.d_px = torch.from_numpy(self.h_px).cuda()
        sift = np.zeros((N, 144), np.float32)                  # 576-byte SiftPoint records
        sift[:, 0], sift[:, 1], sift[:, 9], sift[:, 10] = self.h_px[0].T
        sift[:, 6] = sift[:, 7] = 1.0                          # score, ambiguity
        self.d_sift = torch.from_numpy(sift).cuda()
        self.out = {"E": np.empty((1, 9), np.float32), "P": np.empty((1, 16), np.float32), "idx": np.empty(1, np.int32),
                    "inl": np.empty(1, np.int32), "pts": np.empty((1, 4, N), np.float32)}
        self.counts = torch.empty(H, dtype=torch.int32, device="cuda")
        self.ecand = torch.empty((H, 9), dtype=torch.float32, device="cuda")
        self.X = torch.empty((3, N), dtype=torch.float32, device="cuda")
        self.mask = torch.empty(N, dtype=torch.uint8, device="cuda")
        self.pos = torch.empty((N, 4), dtype=torch.float32, device="cuda")
        self.col = torch.empty((N, 4), dtype=torch.float32, device="cuda")
        self.cloud = torch.empty((4, N), dtype=torch.float32, device="cuda")
        self.count = torch.empty(N, dtype=torch.int32, device="cuda")


def _points(h, io):
    h.set_points_xy(io.d_px)


def _estimate(h, io):
    _points(h, io)
    h.estimate_e(H, SEED, THR)


def _run(h, io):
    h.run_device(io.d_px, H, SEED, THR)


def _state_mg(h, io, pkg):
    _points(h, io)
    pkg.sharding.connect_peers(h, 0, 1)                  # a world of one rank: the exchange runs against itself
    pkg.sharding.estimate_e_p2p(h, H, SEED, THR)


def _state_chain(h, io, pkg):
    _run(h, io)
    h.chain = h.chain_views()              # the cloud and count that bundle_adjust_global takes


def _state_filtered_none(h, io, pkg):
    _run(h, io)
    with pytest.raises(pkg.SfmError) as e:
        h.set_points_sift_filtered(io.d_sift, N, 2.0, 0.0)      # no record passes: fewer than 8 survive
    assert e.value.code == ERR_STATE


# state -> setup(h, io, pkg)
STATES = {
    "fresh": lambda h, io, pkg: None,
    "points": lambda h, io, pkg: _points(h, io),
    "estimate_e": lambda h, io, pkg: _estimate(h, io),
    "estimate_e_slice": lambda h, io, pkg: (_points(h, io), h.estimate_e(H // 2, SEED, THR, H_total=H, h_begin=H // 4)),
    "estimate_e_adaptive": lambda h, io, pkg: (_points(h, io), h.estimate_e_adaptive(H, SEED, THR, 0.99, 128, 2)),
    "estimate_e_mg": _state_mg,
    "homography": lambda h, io, pkg: (_points(h, io), h.find_homography(H, SEED, 5.0)),
    "set_E": lambda h, io, pkg: (_points(h, io), h.set_E(E_SET)),
    "pose_candidates": lambda h, io, pkg: (_estimate(h, io), h.pose_candidates()),
    "refine_e": lambda h, io, pkg: (_estimate(h, io), h.pose_candidates(), h.refine_e(2)),
    "run_device": lambda h, io, pkg: _run(h, io),
    "bundle_adjust": lambda h, io, pkg: (_run(h, io), h.bundle_adjust(1, 5)),
    "chain_views": _state_chain,
    "filtered_none": _state_filtered_none,
}


def _p(t):
    return C.c_void_p(t.data_ptr())


def _a(a):
    return a.ctypes.data_as(C.c_void_p)


def _call(h, name, *args):
    return h.lib.raw("sfmb200_" + name)(h._h, *args)


def _gba(h, io):
    chain = getattr(h, "chain", {"cloud": io.cloud, "count": io.count})
    cloud, count = chain["cloud"], chain["count"]
    return _call(h, "bundle_adjust_global", _p(cloud), _p(count), 3, None, None)


S, T = C.c_uint64(SEED), C.c_float(THR)
PROBES = {
    "set_points_xy": lambda h, io: _call(h, "set_points_xy", _p(io.d_px), N),
    "estimate_e": lambda h, io: _call(h, "estimate_e", None, H, S, T),
    "estimate_e_slice": lambda h, io: _call(h, "estimate_e_slice", None, H, H // 4, H // 2, S, T),
    "estimate_e_adaptive": lambda h, io: _call(h, "estimate_e_adaptive", None, H, 128, 2, S, T, C.c_float(0.99), None),
    "find_homography": lambda h, io: _call(h, "find_homography", H, S, C.c_float(5.0), None, None),
    "adopt_best": lambda h, io: _call(h, "adopt_best", None, H, S),
    "set_E": lambda h, io: _call(h, "set_E", _a(E_SET)),
    "refine_e": lambda h, io: _call(h, "refine_e", 2),
    "pose_candidates": lambda h, io: _call(h, "pose_candidates"),
    "choose_pose": lambda h, io: _call(h, "choose_pose"),
    "triangulate": lambda h, io: _call(h, "triangulate"),
    "run_device": lambda h, io: _call(h, "run_device", _p(io.d_px), N, H, S, T),
    "run_host": lambda h, io: _call(h, "run_host", _a(io.h_px), N, H, S, T, *(_a(v) for v in io.out.values())),
    "bundle_adjust": lambda h, io: _call(h, "bundle_adjust", 1, 5, None),
    "chain_views": lambda h, io: _call(h, "chain_views", None, None, None, None, None),
    "bundle_adjust_global": _gba,
    "get_inlier_counts": lambda h, io: _call(h, "get_inlier_counts", 0, _p(io.counts)),
    "get_E_candidates": lambda h, io: _call(h, "get_E_candidates", 0, _p(io.ecand)),
    "get_X": lambda h, io: _call(h, "get_X", 0, 0, _p(io.X)),
    "get_inlier_mask": lambda h, io: _call(h, "get_inlier_mask", 0, _p(io.mask)),
    "copy_to_vbo_coloured": lambda h, io: _call(h, "copy_to_vbo_coloured", 0, _p(io.pos), _p(io.col), 1.0, 1, 0.0, 1.0),
}

# calls refused with SFMB200_ERR_STATE in each state; every other call succeeds
NEED_POSE = "choose_pose triangulate bundle_adjust chain_views bundle_adjust_global"
REFUSED = {
    "fresh": "estimate_e estimate_e_slice estimate_e_adaptive find_homography adopt_best refine_e pose_candidates "
             f"{NEED_POSE} get_inlier_counts get_E_candidates get_X get_inlier_mask copy_to_vbo_coloured",
    "points": f"adopt_best refine_e pose_candidates {NEED_POSE} get_inlier_counts get_E_candidates get_inlier_mask "
              "copy_to_vbo_coloured",
    "estimate_e": NEED_POSE,
    "estimate_e_slice": NEED_POSE,
    "estimate_e_adaptive": f"{NEED_POSE} get_inlier_counts get_E_candidates",
    "estimate_e_mg": f"{NEED_POSE} get_inlier_counts get_E_candidates",
    "homography": f"adopt_best refine_e pose_candidates {NEED_POSE} copy_to_vbo_coloured",
    "set_E": f"{NEED_POSE} get_inlier_counts get_E_candidates",
    "pose_candidates": "bundle_adjust_global",
    "refine_e": NEED_POSE,
    "run_device": "bundle_adjust_global",
    "bundle_adjust": "bundle_adjust_global",
    "chain_views": "",
    "filtered_none": "estimate_e estimate_e_slice estimate_e_adaptive find_homography adopt_best refine_e "
                     f"{NEED_POSE} get_X get_inlier_mask",
}

# launches of each call that runs: the general path's count, and where the fused path differs, its count
LAUNCHES = {
    "set_points_xy": 1, "estimate_e": 3, "estimate_e_slice": 3, "estimate_e_adaptive": 9, "find_homography": 3,
    "adopt_best": 1, "set_E": 0, "refine_e": 6, "pose_candidates": 1, "choose_pose": 1, "triangulate": 1,
    "run_device": 5, "run_host": 6, "bundle_adjust": 9, "chain_views": 1, "bundle_adjust_global": 8,
    "get_inlier_counts": 0, "get_E_candidates": 1, "get_X": 1, "get_inlier_mask": 1, "copy_to_vbo_coloured": 1,
}
LAUNCHES_FUSED = {"estimate_e": 1, "estimate_e_slice": 1, "run_device": 1, "run_host": 2}


def _expected(path):
    want = {}
    for state, refused in REFUSED.items():
        for probe in PROBES:
            if probe in refused.split():
                want[state, probe] = "refused"
                continue
            n = (LAUNCHES_FUSED if path == "fused" else {}).get(probe, LAUNCHES[probe])
            # one more launch re-materialises the scaled copies of the points when an estimate switches between the
            # homography's unscaled coordinates and the essential-matrix threshold
            if probe == "find_homography" and state != "homography":
                n += 1
            if probe.startswith("estimate_e") and state == "homography":
                n += 1
            want[state, probe] = n
    return want


@pytest.mark.parametrize("path", ["fused", "general"])
def test_state_table(pkg, O, path):
    io = Io(O)
    got = {}
    for state, setup in STATES.items():
        for probe, call in PROBES.items():
            h = pkg.BatchedPairs(io.K, io.Kinv, 1, N, H)
            if path == "general":
                h.set_option(OPT_SMALL, 0)
            setup(h, io, pkg)
            before = h.launch_count()
            rc = call(h, io)
            h.synchronize()
            delta = h.launch_count() - before
            got[state, probe] = delta if rc == 0 else "refused" if rc == ERR_STATE and delta == 0 else (rc, delta, h.lib.last_error())
            h.close()
    want = _expected(path)
    diff = [(k, want[k], got[k]) for k in want if want[k] != got[k]]
    assert not diff, "(state, call), expected, observed:\n" + "\n".join(map(str, diff))
