"""Python mirror of the reference's operator surface, SfM::Image_pair
(SfM/sfm.h:20-60), over the C ABI.  Same method names and argument meaning as
the C++ class (and as the C++ facade in cuda-sfm_b200/SfM/sfm.h); torch is used
only for device memory and streams.  No algorithmic code lives here.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from .binding import Lib, SfmError, load_library

OPT_COMPAT, OPT_SCORE_VARIANT, OPT_TRI_INLIERS_ONLY = 1, 2, 3


def _torch():
    import torch

    return torch


def _dptr(t, dtype: str | None = None, min_elems: int = 0) -> C.c_void_p:
    """Device pointer of a torch CUDA tensor (or a raw int address, taken on trust).  dtype ("float32", "int32",
    "uint8") and min_elems, when given, are checked: the C ABI reads / writes raw memory of that type and size."""
    if t is None:
        return C.c_void_p(0)
    if isinstance(t, int):
        return C.c_void_p(t)
    if not (t.is_cuda and t.is_contiguous()):
        raise ValueError("expected a contiguous CUDA tensor")
    if dtype is not None and str(t.dtype) != "torch." + dtype:
        raise TypeError(f"expected a {dtype} tensor, got {t.dtype}")
    if t.numel() < min_elems:
        raise ValueError(f"tensor too small: {t.numel()} elements, need {min_elems}")
    return C.c_void_p(t.data_ptr())


def _hptr(a: np.ndarray, dtype=None, shape: tuple | None = None) -> C.c_void_p:
    """Host pointer of a C-contiguous numpy array; dtype / exact shape are checked when given (the C ABI writes
    raw float32 / int32 of a fixed size through it)."""
    if not isinstance(a, np.ndarray) or not a.flags["C_CONTIGUOUS"]:
        raise ValueError("expected a C-contiguous numpy array")
    if dtype is not None and a.dtype != np.dtype(dtype):
        raise TypeError(f"expected a {np.dtype(dtype)} array, got {a.dtype}")
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError(f"expected shape {tuple(shape)}, got {tuple(a.shape)}")
    return C.c_void_p(a.ctypes.data)


def pack_ragged(parts):
    """Per-pair (count_b, 4) rows -> (packed rows [sum count_b][4], offsets int32 [pairs + 1]), the layout of the
    *_ragged entry points.  numpy arrays stay numpy (float32); torch tensors are concatenated by torch (same device)."""
    if len(parts) == 0:
        raise ValueError("no pairs")
    counts = [int(p.shape[0]) for p in parts]
    offsets = np.zeros(len(parts) + 1, np.int32)
    offsets[1:] = np.cumsum(counts)
    if hasattr(parts[0], "is_cuda"):
        torch = _torch()
        packed = torch.cat([p.reshape(-1, 4).to(torch.float32) for p in parts]).contiguous()
    else:
        packed = np.ascontiguousarray(np.concatenate([np.asarray(p, np.float32).reshape(-1, 4) for p in parts]))
    return packed, offsets


def unpack_ragged(packed, offsets) -> list:
    """Inverse of pack_ragged: the views packed[offsets[b]:offsets[b + 1]].  For a packed [4][count_b] SoA output (points
    of run_host_ragged) pass it viewed as rows of 4 floats and reshape each part to (4, -1)."""
    return [packed[int(offsets[b]):int(offsets[b + 1])] for b in range(len(offsets) - 1)]


def check_offsets(offsets, pairs: int, max_points: int, rows: int | None = None) -> np.ndarray:
    """The C ABI's checks of a ragged batch's offsets, done before any call: int32 [pairs + 1], offsets[0] == 0, every
    count in [8, max_points] and, when given, rows == offsets[pairs].  Returns the offsets as a C-contiguous int32 array."""
    o = np.asarray(offsets)
    if o.ndim != 1 or o.shape[0] != pairs + 1:
        raise ValueError(f"offsets must have pairs + 1 = {pairs + 1} entries, got shape {o.shape}")
    if not np.issubdtype(o.dtype, np.integer):
        raise TypeError(f"offsets must be integers, got {o.dtype}")
    o = o.astype(np.int64)
    if o[0] != 0:
        raise ValueError("offsets[0] must be 0")
    c = np.diff(o)
    if np.any(c < 0):
        raise ValueError("offsets must not decrease")
    if np.any(c < 8) or np.any(c > max_points):
        raise ValueError(f"every count offsets[b+1] - offsets[b] must be in [8, max_points={max_points}]")
    if rows is not None and rows != o[-1]:
        raise ValueError(f"the packed input has {rows} rows, offsets[-1] = {o[-1]}")
    return np.ascontiguousarray(o.astype(np.int32))


class BatchedPairs:
    """A handle over `pairs` image pairs with n correspondences each, or count_b for pair b (the *_ragged methods)."""

    def __init__(self, K, Kinv, pairs: int, max_points: int, max_hypotheses: int, lib: Lib | None = None):
        self.lib = lib or load_library()
        self.K = np.ascontiguousarray(K, dtype=np.float32).reshape(9)
        self.Kinv = np.ascontiguousarray(Kinv, dtype=np.float32).reshape(9)
        self.pairs, self.max_points, self.max_hypotheses = pairs, max_points, max_hypotheses
        self.n = 0
        self.H = 0
        self.counts = None        # per-pair counts after a *_ragged ingest, None while every pair holds n
        h = C.c_void_p()
        fp = C.POINTER(C.c_float)
        self.lib.call("sfmb200_create", self.K.ctypes.data_as(fp), self.Kinv.ctypes.data_as(fp), pairs, max_points,
                      max_hypotheses, C.byref(h))
        self._h = h
        # Enqueue on torch's current stream so that tensors produced / consumed by
        # torch around these calls are ordered without extra synchronisation.
        self.use_torch_stream()

    # ---- lifetime ----
    def close(self):
        if getattr(self, "_h", None):
            self.lib.call("sfmb200_destroy", self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, option: int, value: int):
        self.lib.call("sfmb200_set_option", self._h, option, value)

    def use_torch_stream(self, stream=None):
        torch = _torch()
        stream = stream or torch.cuda.current_stream()
        self.lib.call("sfmb200_set_stream", self._h, C.c_void_p(stream.cuda_stream))

    def synchronize(self):
        self.lib.call("sfmb200_synchronize", self._h)

    # ---- ingest ----
    def set_points_sift(self, d_sift, n: int):
        self.lib.call("sfmb200_set_points_sift", self._h, _dptr(d_sift), n)
        self.n, self.counts = n, None

    def set_points_sift_filtered(self, d_sift, n: int, min_score: float, max_ambiguity: float, d_kept_index=None) -> int:
        kept = C.c_int32(0)
        try:
            self.lib.call("sfmb200_set_points_sift_filtered", self._h, _dptr(d_sift), n, C.c_float(min_score),
                          C.c_float(max_ambiguity), _dptr(d_kept_index), C.byref(kept))
        finally:
            self.n, self.counts = kept.value, None
        return kept.value

    def set_points_xy(self, d_px, n: int | None = None):
        n = n if n is not None else d_px.shape[-2]
        self.lib.call("sfmb200_set_points_xy", self._h, _dptr(d_px, "float32", self.pairs * n * 4), n)
        self.n, self.counts = n, None

    def set_points_xy_host(self, h_px: np.ndarray):
        h_px = np.ascontiguousarray(h_px, dtype=np.float32)
        n = h_px.shape[-2]
        self.lib.call("sfmb200_set_points_xy_host", self._h, _hptr(h_px), n)
        self.synchronize()   # h_px may be pageable and die with the caller
        self.n, self.counts = n, None

    def set_points_normalised(self, d_x, n: int | None = None):
        n = n if n is not None else d_x.shape[-2]
        self.lib.call("sfmb200_set_points_normalised", self._h, _dptr(d_x, "float32", self.pairs * n * 4), n)
        self.n, self.counts = n, None

    # ---- batches with a count per pair ----
    def _ragged(self, px, offsets, device: bool):
        """(packed rows, offsets) of a ragged input: a list of per-pair (count_b, 4) arrays / tensors, or packed rows with
        their offsets.  device: a contiguous float32 CUDA tensor; else a C-contiguous float32 numpy array (a pinned one
        is passed through untouched)."""
        if offsets is None:
            if not isinstance(px, (list, tuple)):
                raise ValueError("pass a list of per-pair (count_b, 4) arrays, or packed rows with offsets")
            px, offsets = pack_ragged(px)
        torch = _torch() if device else None
        if device:
            if not hasattr(px, "is_cuda"):
                px = torch.from_numpy(np.ascontiguousarray(px, dtype=np.float32))
            px = px.to(device="cuda", dtype=torch.float32).contiguous()
        elif not (isinstance(px, np.ndarray) and px.dtype == np.float32 and px.flags["C_CONTIGUOUS"]):
            px = np.ascontiguousarray(px.cpu().numpy() if hasattr(px, "is_cuda") else px, dtype=np.float32)
        if px.shape[-1] != 4 or px.ndim != 2:
            raise ValueError(f"packed rows must be [rows][4], got {tuple(px.shape)}")
        offsets = check_offsets(offsets, self.pairs, self.max_points, int(px.shape[0]))
        return px, offsets

    def _set_counts(self, offsets: np.ndarray):
        self.counts = np.diff(offsets).astype(np.int32)
        self.n = int(self.counts.max())

    def set_points_xy_ragged(self, px, offsets=None):
        """Pixel correspondences with a count per pair (include/sfmb200.h: sfmb200_set_points_xy_ragged)."""
        px, offsets = self._ragged(px, offsets, True)
        self.lib.call("sfmb200_set_points_xy_ragged", self._h, _dptr(px), _hptr(offsets))
        self._set_counts(offsets)

    def run_device_ragged(self, px, H: int, seed: int = 0, thr: float = 1e-6, offsets=None):
        px, offsets = self._ragged(px, offsets, True)
        self.lib.call("sfmb200_run_device_ragged", self._h, _dptr(px), _hptr(offsets), H, C.c_uint64(seed), C.c_float(thr))
        self._set_counts(offsets)
        self.H = H

    def run_host_ragged(self, px, H: int, seed: int = 0, thr: float = 1e-6, offsets=None, want_points: bool = True) -> dict:
        """Whole path from host pixel correspondences with a count per pair.  Returns E [pairs,9], P [pairs,16],
        pose_index / inliers [pairs], points: a list of per-pair (4, count_b) arrays (views of points_packed, the
        packed buffer the C ABI wrote) or None."""
        px, offsets = self._ragged(px, offsets, False)
        B = self.pairs
        out = {"E": np.empty((B, 9), np.float32), "P": np.empty((B, 16), np.float32), "pose_index": np.empty(B, np.int32),
               "inliers": np.empty(B, np.int32)}
        packed = np.empty(4 * int(offsets[-1]), np.float32) if want_points else None
        self.lib.call("sfmb200_run_host_ragged", self._h, _hptr(px), _hptr(offsets), H, C.c_uint64(seed), C.c_float(thr),
                      _hptr(out["E"]), _hptr(out["P"]), _hptr(out["pose_index"]), _hptr(out["inliers"]),
                      _hptr(packed) if want_points else C.c_void_p(0))
        self._set_counts(offsets)
        self.H = H
        out["points_packed"] = packed
        out["points"] = [p.reshape(4, -1) for p in unpack_ragged(packed.reshape(-1, 4), offsets)] if want_points else None
        return out

    def point_counts(self) -> np.ndarray:
        """Correspondences per pair of the current points (n for every pair after a uniform ingest)."""
        out = np.empty(self.pairs, np.int32)
        self.lib.call("sfmb200_get_point_counts", self._h, _hptr(out))
        return out

    def _count(self, pair: int) -> int:
        """Rows the per-pair getters return for `pair`."""
        return int(self.counts[pair]) if self.counts is not None else self.n

    # ---- stages ----
    def estimate_e(self, H: int, seed: int = 0, thr: float = 1e-6, d_idx=None, H_total: int | None = None, h_begin: int = 0):
        idx = _dptr(d_idx, "int32", self.pairs * (H_total or H) * 8)
        if H_total is None:
            self.lib.call("sfmb200_estimate_e", self._h, idx, H, C.c_uint64(seed), C.c_float(thr))
        else:
            self.lib.call("sfmb200_estimate_e_slice", self._h, idx, H_total, h_begin, H, C.c_uint64(seed), C.c_float(thr))
        self.H = H

    def estimate_e_adaptive(self, H_max: int, seed: int = 0, thr: float = 1e-6, confidence: float = 0.99,
                            first_round: int = 4096, growth: int = 4, d_idx=None) -> int:
        """RANSAC with adaptive termination, rounds skipped on the device; returns the hypotheses tried.  Defaults: rounds
        [0, 4096), [4096, 16384), [16384, 65536), ... - every round costs three dependent launches and a small round fills
        the GPU badly, so few and large ones (profiles/r02_adaptive.md)."""
        used = C.c_int32(0)
        self.lib.call("sfmb200_estimate_e_adaptive", self._h, _dptr(d_idx), H_max, first_round, growth, C.c_uint64(seed),
                      C.c_float(thr), C.c_float(confidence), C.byref(used))
        self.H = used.value
        return used.value

    def best_buffer(self):
        """torch int64 view [pairs] of the packed winners (for dist.all_reduce MAX)."""
        torch = _torch()
        p = C.c_void_p()
        self.lib.call("sfmb200_best_buffer", self._h, C.byref(p))
        return _tensor_from_ptr(p.value, (self.pairs,), torch.int64)

    def adopt_best(self, H_total: int, seed: int = 0, d_idx=None):
        self.lib.call("sfmb200_adopt_best", self._h, _dptr(d_idx), H_total, C.c_uint64(seed))

    def find_homography(self, loops: int, seed: int = 0, thresh: float = 5.0):
        """CudaSift FindHomography semantics on this handle's correspondences: `thresh` in PIXELS, H maps image-1 pixels
        to image-2 pixels (needs K = [f 0 cx; 0 f cy; 0 0 1]); returns (H [pairs,3,3], matches [pairs])."""
        Hm = np.empty((self.pairs, 3, 3), np.float32)
        cnt = np.empty(self.pairs, np.int32)
        self.lib.call("sfmb200_find_homography", self._h, loops, C.c_uint64(seed), C.c_float(thresh), _hptr(Hm), _hptr(cnt))
        self.H = loops
        return Hm, cnt

    def refine_e(self, iterations: int = 4) -> np.ndarray:
        """LO-RANSAC refit on the inlier set; returns accepted refits per pair."""
        self.lib.call("sfmb200_refine_e", self._h, iterations)
        out = np.empty(self.pairs, np.int32)
        self.lib.call("sfmb200_get_refit_iterations", self._h, _hptr(out))
        return out

    BA_STATS = ("active", "cost_entry", "cost", "accepted", "lambda", "gauge_scale", "inliers", "committed")

    def bundle_adjust(self, outer_rounds: int = 4, iterations: int = 40) -> np.ndarray:
        """Two-view bundle adjustment with inlier re-selection; returns the [pairs, 8] statistics of the last round (BA_STATS)."""
        st = np.empty((self.pairs, 8), np.float32)
        self.lib.call("sfmb200_bundle_adjust", self._h, outer_rounds, iterations, _hptr(st))
        return st

    def chain_views(self, want_cloud: bool = True):
        """N-view chaining over consecutive pairs with index-aligned tracks; returns dict(cameras [pairs+1,3,4],
        scales [pairs], used [pairs], cloud torch [4,n] or None, count torch [n] or None)."""
        torch = _torch()
        cams = np.empty((self.pairs + 1, 3, 4), np.float32)
        scales = np.empty(self.pairs, np.float32)
        used = np.empty(self.pairs, np.int32)
        cloud = torch.empty((4, self.n), dtype=torch.float32, device="cuda") if want_cloud else None
        count = torch.empty(self.n, dtype=torch.int32, device="cuda") if want_cloud else None
        self.lib.call("sfmb200_chain_views", self._h, _dptr(cloud), _dptr(count), _hptr(cams), _hptr(scales), _hptr(used))
        return dict(cameras=cams, scales=scales, used=used, cloud=cloud, count=count)

    GBA_STATS = ("cost_entry", "cost", "accepted", "lambda", "gauge_scale", "iterations", "spare0", "spare1")

    def bundle_adjust_global(self, chain: dict, iterations: int = 30):
        """Global bundle adjustment of all cameras and points of the chained reconstruction (after chain_views(want_cloud=True),
        whose dict is passed in and updated: cloud in place, cameras replaced).  Returns the [8] statistics (GBA_STATS)."""
        if chain.get("cloud") is None or chain.get("count") is None:
            raise ValueError("bundle_adjust_global needs the cloud and count of chain_views(want_cloud=True)")
        cams = np.empty((self.pairs + 1, 3, 4), np.float32)
        st = np.empty(8, np.float32)
        self.lib.call("sfmb200_bundle_adjust_global", self._h, _dptr(chain["cloud"], "float32", 4 * self.n), _dptr(chain["count"], "int32", self.n),
                      iterations, _hptr(cams), _hptr(st))
        chain["cameras"] = cams
        return st

    def pose_candidates(self):
        self.lib.call("sfmb200_pose_candidates", self._h)

    def choose_pose(self):
        self.lib.call("sfmb200_choose_pose", self._h)

    def triangulate(self):
        self.lib.call("sfmb200_triangulate", self._h)

    def run_device(self, d_px, H: int, seed: int = 0, thr: float = 1e-6, n: int | None = None):
        n = n if n is not None else d_px.shape[-2]
        self.lib.call("sfmb200_run_device", self._h, _dptr(d_px, "float32", self.pairs * n * 4), n, H, C.c_uint64(seed), C.c_float(thr))
        self.n, self.H, self.counts = n, H, None

    def _host_io(self, h_px: np.ndarray, want_points: bool, out: dict | None):
        """Validated host buffers of the e2e call: h_px float32 [pairs][n][4] (coerced like set_points_xy_host unless it
        already is - a pinned buffer is passed through untouched), out[...] float32 / int32 of the exact shapes."""
        if not (isinstance(h_px, np.ndarray) and h_px.dtype == np.float32 and h_px.flags["C_CONTIGUOUS"]):
            h_px = np.ascontiguousarray(h_px, dtype=np.float32)
        if h_px.shape[-1] != 4 or h_px.size % 4 or h_px.size // 4 % self.pairs:
            raise ValueError(f"h_px must be [pairs={self.pairs}][n][4], got {h_px.shape}")
        n = h_px.size // 4 // self.pairs
        B = self.pairs
        if out is None:
            out = {"E": np.empty((B, 9), np.float32), "P": np.empty((B, 16), np.float32), "pose_index": np.empty(B, np.int32),
                   "inliers": np.empty(B, np.int32), "points": np.empty((B, 4, n), np.float32) if want_points else None}
        pts = out.get("points")
        ptrs = (_hptr(out["E"], np.float32, (B, 9)), _hptr(out["P"], np.float32, (B, 16)), _hptr(out["pose_index"], np.int32, (B,)),
                _hptr(out["inliers"], np.int32, (B,)), _hptr(pts, np.float32, (B, 4, n)) if pts is not None else C.c_void_p(0))
        return h_px, n, out, ptrs

    def run_host(self, h_px: np.ndarray, H: int, seed: int = 0, thr: float = 1e-6, want_points: bool = True, out: dict | None = None):
        """Whole path from host pixel correspondences to host results (the e2e call)."""
        h_px, n, out, ptrs = self._host_io(h_px, want_points, out)
        self.lib.call("sfmb200_run_host", self._h, _hptr(h_px), n, H, C.c_uint64(seed), C.c_float(thr), *ptrs)
        self.n, self.H, self.counts = n, H, None
        return out

    def prepare_run_host(self, h_px: np.ndarray, H: int, seed: int = 0, thr: float = 1e-6, out: dict | None = None):
        """run_host with the argument marshalling done once: returns (call, out); call() runs the whole path on the
        buffers captured here (a caller that processes a stream of pairs through the same buffers pays the ctypes
        conversions once, not ~10 us per call)."""
        h_px, n, out, ptrs = self._host_io(h_px, True, out)
        args = (self._h, _hptr(h_px), n, H, C.c_uint64(seed), C.c_float(thr), *ptrs)
        fn = self.lib.raw("sfmb200_run_host")
        lib = self.lib
        self.n, self.H, self.counts = n, H, None

        def call():
            rc = fn(*args)
            if rc != 0:
                raise SfmError(rc, lib.last_error())
        call.keepalive = (h_px, out)          # the captured pointers must outlive the closure's users
        return call, out

    # ---- getters ----
    def get_E(self) -> np.ndarray:
        out = np.empty((self.pairs, 3, 3), np.float32)
        self.lib.call("sfmb200_get_E", self._h, _hptr(out))
        return out

    def set_E(self, E: np.ndarray):
        E = np.ascontiguousarray(E, dtype=np.float32).reshape(self.pairs, 9)
        self.lib.call("sfmb200_set_E", self._h, _hptr(E))

    def get_best(self):
        idx = np.empty(self.pairs, np.int32)
        cnt = np.empty(self.pairs, np.int32)
        self.lib.call("sfmb200_get_best", self._h, _hptr(idx), _hptr(cnt))
        return idx, cnt

    def get_poses(self) -> np.ndarray:
        out = np.empty((self.pairs, 4, 4, 4), np.float32)
        self.lib.call("sfmb200_get_poses", self._h, _hptr(out))
        return out

    def get_pose_index(self) -> np.ndarray:
        out = np.empty(self.pairs, np.int32)
        self.lib.call("sfmb200_get_pose_index", self._h, _hptr(out))
        return out

    def get_points_host(self, pair: int = 0) -> np.ndarray:
        out = np.empty((4, self._count(pair)), np.float32)
        self.lib.call("sfmb200_get_points_host", self._h, pair, _hptr(out))
        return out

    def get_points(self, pair: int = 0):
        torch = _torch()
        out = torch.empty((4, self._count(pair)), dtype=torch.float32, device="cuda")
        self.lib.call("sfmb200_get_points", self._h, pair, _dptr(out))
        self.synchronize()
        return out

    def get_inlier_counts(self, pair: int = 0):
        torch = _torch()
        out = torch.empty(self.H, dtype=torch.int32, device="cuda")
        self.lib.call("sfmb200_get_inlier_counts", self._h, pair, _dptr(out))
        self.synchronize()
        return out

    def get_E_candidates(self, pair: int = 0):
        torch = _torch()
        out = torch.empty((self.H, 9), dtype=torch.float32, device="cuda")
        self.lib.call("sfmb200_get_E_candidates", self._h, pair, _dptr(out))
        self.synchronize()
        return out

    def get_X(self, image: int, pair: int = 0):
        torch = _torch()
        out = torch.empty((3, self._count(pair)), dtype=torch.float32, device="cuda")
        self.lib.call("sfmb200_get_X", self._h, pair, image, _dptr(out))
        self.synchronize()
        return out

    def get_inlier_mask(self, pair: int = 0):
        torch = _torch()
        out = torch.empty(self._count(pair), dtype=torch.uint8, device="cuda")
        self.lib.call("sfmb200_get_inlier_mask", self._h, pair, _dptr(out))
        self.synchronize()
        return out

    def copy_to_vbo(self, d_pos, d_col, pair: int = 0):
        n = self._count(pair)
        self.lib.call("sfmb200_copy_to_vbo", self._h, pair, _dptr(d_pos, "float32", 4 * n), _dptr(d_col, "float32", 4 * n))

    def copy_to_vbo_coloured(self, d_pos, d_col, pair: int = 0, scale: float = 1.0, mode: int = 1, z_near: float = 0.0, z_far: float = 1.0):
        """mode 0 ones, 1 inlier green / outlier red, 2 depth ramp blue -> red between z_near and z_far."""
        n = self._count(pair)
        self.lib.call("sfmb200_copy_to_vbo_coloured", self._h, pair, _dptr(d_pos, "float32", 4 * n), _dptr(d_col, "float32", 4 * n),
                      C.c_float(scale), mode,
                      C.c_float(z_near), C.c_float(z_far))

    def score_plan(self) -> dict:
        out = (C.c_int32 * 4)()
        self.lib.call("sfmb200_score_plan", self._h, out)
        return {"variant": out[0], "tiles": out[1], "ctas": out[2], "hyp_per_cta": out[3]}

    STAGES = ("ingest", "hypgen", "score", "select", "pose_candidates", "choose_pose", "triangulate")

    def stage_times(self, max_sets: int = 256) -> np.ndarray:
        """ms [sets][7] of the most recent profiled run_* calls (option 4)."""
        ms = np.zeros((max_sets, 7), np.float32)
        sets = C.c_int(0)
        self.lib.call("sfmb200_stage_times", self._h, max_sets, _hptr(ms), C.byref(sets))
        return ms[: sets.value]

    def launch_count(self) -> int:
        return int(self.lib.raw("sfmb200_launch_count")(self._h))


def _tensor_from_ptr(ptr: int, shape, dtype):
    """Zero-copy torch view of device memory owned by the handle."""
    torch = _torch()
    n = int(np.prod(shape))
    itemsize = torch.empty((), dtype=dtype).element_size()

    class _Holder:
        __cuda_array_interface__ = {
            "shape": (n * itemsize,), "typestr": "|u1", "data": (ptr, False), "version": 3, "strides": None,
        }

    raw = torch.as_tensor(_Holder(), device="cuda")
    return raw.view(dtype).view(*shape)


class ImagePair(BatchedPairs):
    """SfM::Image_pair (SfM/sfm.h:20-60): same constructor arguments and method
    names; `image_count` is accepted and must be 2 like the reference's only use
    (src/main.cpp:298).  The reference's estimateE() draws H = N/8 disjoint
    samples from a host shuffle (sfm.cu:95-104); here H, the seed and the
    threshold are explicit (defaults reproduce H = N/8 and 1e-6)."""

    def __init__(self, k, k_inv, image_count: int, num_points: int, max_hypotheses: int | None = None, lib: Lib | None = None):
        if image_count != 2:
            raise ValueError("Image_pair handles exactly two images (like the reference)")
        self.image_count, self.num_points = image_count, num_points
        super().__init__(k, k_inv, 1, num_points, max_hypotheses or max(num_points // 8, 1), lib)

    def fillXU(self, data, n: int | None = None, min_score: float | None = None, max_ambiguity: float | None = None):
        """data: device SiftPoint array (raw address or CUDA tensor).  With
        min_score / max_ambiguity: keep only matches passing CudaSift's own test."""
        if min_score is None and max_ambiguity is None:
            self.set_points_sift(data, n or self.num_points)
            return self.n
        return self.set_points_sift_filtered(data, n or self.num_points, min_score if min_score is not None else -np.inf,
                                             max_ambiguity if max_ambiguity is not None else np.inf)

    def estimateE(self, H: int | None = None, seed: int = 0, thr: float = 1e-6, d_idx=None):
        """No H and no rows = the reference's estimateE(): one permutation of the point indices cut into N/8 disjoint rows
        (drawn on the device, option 10 = 1).  With H or rows: independent rows / the caller's rows."""
        if H is None and d_idx is None:
            self.set_option(10, 1)
            try:
                self.estimate_e(max(self.n // 8, 1), seed, thr)
            finally:
                self.set_option(10, 0)
            return
        self.estimate_e(H or max(self.n // 8, 1), seed, thr, d_idx)

    def computePosecandidates(self):
        self.pose_candidates()

    def choosePose(self):
        self.choose_pose()

    def linear_triangulation(self):
        self.triangulate()

    def copyBoidsToVBO(self, vbodptr_positions, vbodptr_velocities):
        self.copy_to_vbo(vbodptr_positions, vbodptr_velocities)
