"""fp64 CPU restatement of the reference hot path (TEST INFRASTRUCTURE ONLY).

Only tests/ (including the checker-side diagnostics under tests/diag/),
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product path (cuda-sfm_b200/) never does: it fails
loudly when the CUDA library is missing.

Reference: Black-Phoenix/CUDA-SfM, files under SfM/.  Each function cites the
file:line whose *stated* algorithm it restates.  Where the reference's code is
undefined behaviour (inlier scoring reads uninitialised memory, sfm.cu:208-215;
arg-max off by one, sfm.cu:137) the restatement follows BASELINE.json's
north_star definition instead (Sampson error, true arg-max, lowest index on
ties) - see SURVEY.md section 2.3.

PARITY PINNING: the reference ships no asserting tests and no golden vectors
(SURVEY.md section 4), so the pins are (1) the literals of its print-only tests
and its own host svd()/det() compiled from svd.h (tests/test_cpu_oracle.py,
tests/test_cpu_hostlogic.py, tests/test_gpu_la_wrappers.py), (2) the reference's
own CUDA code rebuilt unmodified as oracle/_ref/libsfm_ref.so and run stage by
stage on the GPU box (tests/test_gpu_reference_parity.py), (3) the committed
fixture of the reference's own image pair (tests/golden/dino_000_001.npz,
tests/test_golden_dino.py).  What the reference cannot pin because its code is
undefined behaviour there (inlier counts, arg-max) and everything it does not
have (refit, adaptive termination, homography model, bundle adjustment,
chaining) is pinned by fp64 math and ground truth only.
"""
from __future__ import annotations

import math

import numpy as np

MASK64 = (1 << 64) - 1

# --------------------------------------------------------------------------
# Camera + synthetic scene: input generation lives with the host code
# (cuda-sfm_b200/synthetic.py) so that the measured arm of bench.py never imports
# this checker; re-exported here for the tests.
# --------------------------------------------------------------------------
import importlib.util as _ilu
import os as _os

_spec = _ilu.spec_from_file_location(
    "sfm_synthetic", _os.path.join(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))), "cuda-sfm_b200", "synthetic.py"))
_synthetic = _ilu.module_from_spec(_spec)
_spec.loader.exec_module(_synthetic)
F_REF, W_REF, H_REF = _synthetic.F_REF, _synthetic.W_REF, _synthetic.H_REF
reference_K = _synthetic.reference_K
synthetic_pair = _synthetic.synthetic_pair
planar_pair = _synthetic.planar_pair
synthetic_sequence = _synthetic.synthetic_sequence
synthetic_orbit = _synthetic.synthetic_orbit


def normalise_points(px: np.ndarray, Kinv: np.ndarray) -> np.ndarray:
    """fillXU (SfM/sfm.cu:80-92, kernels.h:261-279): X = K^-1 [u v 1]^T for both
    images.  Returns (n,4) fp32 (x1,y1,x2,y2); evaluated in fp32 with the same
    operation order as the CUDA ingest kernel (fma(k01,v, fma(k00,u, k02)) is
    within 1 ulp of this; tests use a 2-ulp tolerance)."""
    px = px.astype(np.float32)
    k = Kinv.astype(np.float32)
    out = np.empty_like(px)
    for c, (iu, iv) in enumerate(((0, 1), (2, 3))):
        u, v = px[:, iu].astype(np.float64), px[:, iv].astype(np.float64)
        out[:, 2 * c + 0] = (k[0, 0] * u + k[0, 1] * v + k[0, 2]).astype(np.float32)
        out[:, 2 * c + 1] = (k[1, 0] * u + k[1, 1] * v + k[1, 2]).astype(np.float32)
    return out


# --------------------------------------------------------------------------
# Sample indices: counter-based generator, bit-exact mirror of
# cuda-sfm_b200/csrc/hyp_solver.cuh: sample_indices().  The reference draws
# H = N/8 disjoint samples from one host std::shuffle seeded by random_device
# (sfm.cu:95-104) - nondeterministic, so the new API takes explicit indices or
# this generator (SURVEY Q4).
# --------------------------------------------------------------------------
def _splitmix64(z: int) -> int:
    z = (z + 0x9E3779B97F4A7C15) & MASK64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK64
    return z ^ (z >> 31)


def sample_indices_one(seed: int, h: int, n: int) -> list[int]:
    key = _splitmix64((seed ^ ((h * 0xD1342543DE82EF95) & MASK64)) & MASK64)
    ctr, idx = 0, []
    for _ in range(8):
        while True:
            r = _splitmix64((key + ctr) & MASK64)
            ctr += 1
            cand = ((r >> 32) * n) >> 32
            if cand not in idx:
                break
        idx.append(cand)
    return idx


def sample_indices(seed: int, H: int, n: int, h0: int = 0) -> np.ndarray:
    """Vectorised version of sample_indices_one for rows h0..h0+H-1."""
    def sm(z):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))

    with np.errstate(over="ignore"):
        h = np.arange(h0, h0 + H, dtype=np.uint64)
        key = sm(np.uint64(seed) ^ (h * np.uint64(0xD1342543DE82EF95)))
        ctr = np.zeros(H, dtype=np.uint64)
        out = np.full((H, 8), -1, dtype=np.int64)
        for j in range(8):
            todo = np.ones(H, dtype=bool)
            while todo.any():
                r = sm(key[todo] + ctr[todo])
                ctr[todo] += np.uint64(1)
                cand = (((r >> np.uint64(32)) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)
                dup = (out[todo, :j] == cand[:, None]).any(axis=1) if j else np.zeros(cand.shape, bool)
                rows = np.flatnonzero(todo)
                okrows = rows[~dup]
                out[okrows, j] = cand[~dup]
                todo[okrows] = False
    return out.astype(np.int32)


# --------------------------------------------------------------------------
# Hypothesis generation (K3-K7)
# --------------------------------------------------------------------------
def sample_indices_disjoint(seed: int, H: int, n: int, h0: int = 0) -> np.ndarray:
    """The reference's sampling scheme (sfm.cu:95-104: one shuffle of the point indices cut into H = N/8 disjoint groups of
    8), as the device draws it for SFMB200_OPT_SAMPLER = 1: row h = perm(8h .. 8h+7) with perm a keyed 4-round Feistel
    permutation of [0, n) with cycle walking.  Bit-exact mirror of hyp_solver.cuh: sample_indices_disjoint."""
    assert 8 * (h0 + H) <= n
    k0 = _splitmix64(seed ^ 0xA5A5A5A5A5A5A5A5)
    k1 = _splitmix64(k0)
    keys = [k0 & 0xFFFFFFFF, k0 >> 32, k1 & 0xFFFFFFFF, k1 >> 32]
    bits = 1
    while (1 << bits) < n:
        bits += 1
    half = (bits + 1) // 2
    mask = np.uint32((1 << half) - 1)

    def mix(v, key):
        v = v ^ np.uint32(key)
        v = (v * np.uint32(0x85EBCA6B)).astype(np.uint32)
        v = v ^ (v >> np.uint32(13))
        v = (v * np.uint32(0xC2B2AE35)).astype(np.uint32)
        return v ^ (v >> np.uint32(16))

    x = np.arange(8 * h0, 8 * (h0 + H), dtype=np.uint32)
    todo = np.ones(len(x), bool)
    with np.errstate(over="ignore"):
        while todo.any():
            L, R = x[todo] >> np.uint32(half), x[todo] & mask
            for r in range(4):
                L, R = R, L ^ (mix(R, keys[r]) & mask)
            x[todo] = (L << np.uint32(half)) | R
            todo = x >= n
    return x.astype(np.int32).reshape(H, 8)


def design_matrix(x: np.ndarray) -> np.ndarray:
    """kernels::kernels (SfM/kernels.h:247-257): row = kron((x1,y1,1),(x2,y2,1))
    so that the null vector reshaped row-major satisfies x1^T E x2 = 0."""
    x1, y1, x2, y2 = (x[..., i].astype(np.float64) for i in range(4))
    o = np.ones_like(x1)
    return np.stack([x1 * x2, x1 * y2, x1, y1 * x2, y1 * y2, y1, x2, y2, o], -1)


def project_essential(E: np.ndarray) -> np.ndarray:
    """normalizeE (SfM/kernels.h:281-295): E <- U diag(1,1,0) V^T."""
    U, _, Vt = np.linalg.svd(E)
    return U[..., :, :2] @ Vt[..., :2, :]


def hypotheses(x: np.ndarray, idx: np.ndarray) -> np.ndarray:
    """E candidates (H,3,3) in fp64 for sample rows idx (H,8) over points x (n,4).
    Null vector of the 8x9 design matrix (regular_svd + row_extraction_kernel,
    kernels.h:211-234, 452-458), then rank-2 projection.  Sign is arbitrary."""
    A = design_matrix(x[idx])                       # (H,8,9)
    _, _, Vt = np.linalg.svd(A)                     # full: (H,9,9)
    E = Vt[:, -1, :].reshape(-1, 3, 3)
    return project_essential(E)


def e_distance(Ea: np.ndarray, Eb: np.ndarray) -> np.ndarray:
    """Relative Frobenius distance up to sign and scale (north_star tolerance 1e-4)."""
    a = Ea.reshape(len(Ea), -1).astype(np.float64)
    b = Eb.reshape(len(Eb), -1).astype(np.float64)
    na = np.linalg.norm(a, axis=1, keepdims=True)
    nb = np.linalg.norm(b, axis=1, keepdims=True)
    with np.errstate(invalid="ignore", divide="ignore"):
        a, b = a / na, b / nb
    return np.minimum(np.linalg.norm(a - b, axis=1), np.linalg.norm(a + b, axis=1))


# --------------------------------------------------------------------------
# Inlier scoring (calculateInliers' stated intent, sfm.cu:155-221, with the
# Sampson error north_star mandates; threshold literal 1e-6 from sfm.cu:220)
# --------------------------------------------------------------------------
def sampson_terms(E: np.ndarray, x: np.ndarray):
    """num^2 and den of the Sampson error for every (hypothesis, point), fp64.
    Convention x1^T E x2 = 0: l = E x2, m = E^T x1,
    err = (x1.l)^2 / (l0^2 + l1^2 + m0^2 + m1^2)."""
    E = E.reshape(-1, 3, 3).astype(np.float64)
    x1 = np.stack([x[:, 0], x[:, 1], np.ones(len(x))], 0).astype(np.float64)   # (3,n)
    x2 = np.stack([x[:, 2], x[:, 3], np.ones(len(x))], 0).astype(np.float64)
    l = E @ x2                                        # (H,3,n)
    m = np.transpose(E, (0, 2, 1)) @ x1               # (H,3,n)
    num = (x1[None] * l).sum(1)
    den = l[:, 0] ** 2 + l[:, 1] ** 2 + m[:, 0] ** 2 + m[:, 1] ** 2
    return num * num, den


def inlier_counts(E: np.ndarray, x: np.ndarray, thr: float = 1e-6, band: float = 1e-6, chunk: int = 256):
    """Counts (H,) of points with num^2 < thr*den, plus the number of borderline
    points per hypothesis (|num^2 - thr*den| <= band*thr*den + tiny): the CUDA
    fp32 count must lie in [count - borderline, count + borderline]."""
    E = E.reshape(-1, 3, 3)
    cnt = np.zeros(len(E), np.int64)
    amb = np.zeros(len(E), np.int64)
    for s in range(0, len(E), chunk):
        n2, den = sampson_terms(E[s:s + chunk], x)
        d = n2 - thr * den
        cnt[s:s + chunk] = (d < 0).sum(1)
        amb[s:s + chunk] = (np.abs(d) <= band * thr * den + 1e-300).sum(1)
    return cnt, amb


def symmetric_counts(E: np.ndarray, x: np.ndarray, thr: float = 1e-6, band: float = 1e-4, chunk: int = 256):
    """Symmetric epipolar distance, the stated intent of calculateInliers (sfm.cu:155-221; SURVEY Q14):
    n^2 / (l0^2 + l1^2) + n^2 / (m0^2 + m1^2) < thr with n = x1^T E x2, l = E x2, m = E^T x1, evaluated division-free as
    n^2 (A + B) < thr A B.  Returns (counts, borderline) like inlier_counts."""
    E = E.reshape(-1, 3, 3).astype(np.float64)
    x1 = np.stack([x[:, 0], x[:, 1], np.ones(len(x))], 0).astype(np.float64)
    x2 = np.stack([x[:, 2], x[:, 3], np.ones(len(x))], 0).astype(np.float64)
    cnt = np.zeros(len(E), np.int64)
    amb = np.zeros(len(E), np.int64)
    for s in range(0, len(E), chunk):
        Ec = E[s:s + chunk]
        l = Ec @ x2
        m = np.transpose(Ec, (0, 2, 1)) @ x1
        num = (x1[None] * l).sum(1)
        A, B = l[:, 0] ** 2 + l[:, 1] ** 2, m[:, 0] ** 2 + m[:, 1] ** 2
        d = num * num * (A + B) - thr * A * B
        cnt[s:s + chunk] = (d < 0).sum(1)
        amb[s:s + chunk] = (np.abs(d) <= band * thr * A * B + 1e-300).sum(1)
    return cnt, amb


def sampson_mask_f32(E: np.ndarray, x: np.ndarray, thr: float = 1e-6) -> np.ndarray:
    """Inlier mask with the SAME fp32 fma tree as the CUDA kernels (sampson.cuh: sampson_d),
    emulated with exactly-rounded fp64 products: every fp32 fma(a,b,c) is computed as
    float32(float64(a)*float64(b) + float64(c)), which is correctly rounded because the
    fp64 product of two fp32 numbers is exact.  (The sum can still double-round in rare
    half-way cases; tests allow for a handful of such points.)"""
    f32, f64 = np.float32, np.float64
    # threshold folded into the coordinates (sampson.cuh): k = sqrt(thr), points * 1/k, E~ = D E D, D = diag(k,k,1)
    k = np.sqrt(f32(thr)).astype(f32)
    ik = (f32(1.0) / k).astype(f32)
    k2 = (k * k).astype(f32)
    fac = np.array([k2, k2, k, k2, k2, k, k, k, f32(1.0)], f32)
    e = E.reshape(9).astype(f32)
    e = np.where(np.arange(9) == 8, e, (e * fac).astype(f32)).astype(f32)
    x1, y1, x2, y2 = ((x[:, i].astype(f32) * ik).astype(f32) for i in range(4))

    def fma(a, b, c):
        return (a.astype(f64) * np.asarray(b, f64) + np.asarray(c, f64)).astype(f32)

    l0 = fma(x2, e[0], fma(y2, e[1], np.full_like(x1, e[2])))
    l1 = fma(x2, e[3], fma(y2, e[4], np.full_like(x1, e[5])))
    l2 = fma(x2, e[6], fma(y2, e[7], np.full_like(x1, e[8])))
    num = fma(x1, l0, fma(y1, l1, l2))
    m0 = fma(x1, e[0], fma(y1, e[3], np.full_like(x1, e[6])))
    m1 = fma(x1, e[1], fma(y1, e[4], np.full_like(x1, e[7])))
    den = fma(l0, l0, fma(l1, l1, fma(m0, m0, (m1 * m1).astype(f32))))
    d = fma(num, num, -den)
    return d < 0


def refit_on_inliers(x: np.ndarray, E0: np.ndarray, thr: float = 1e-6, iterations: int = 4):
    """LO-RANSAC local optimisation (README.md:65-69 future work; SURVEY 8f rank 2),
    restating cuda-sfm_b200/csrc/refit.cu in fp64.  A chain of models m_0 = E0,
    m_{k+1} = fit(inliers of m_k at mult_k * thr), mult = 4, 2, 1, 1, ...; fit =
    Hartley-normalise (centroid, sqrt(2)/RMS scale), null vector of the Gram matrix
    of the design rows kron(x1h, x2h), E = T1^T Eh T2, rank-2 projection.  The
    incumbent is the chain member with strictly the most inliers at thr.
    Returns (E, count, accepted)."""
    mult = lambda k: 4.0 if k == 0 else (2.0 if k == 1 else 1.0)
    model = np.asarray(E0, np.float64).reshape(3, 3)
    E, count, accepted = model, int(sampson_mask_f32(model, x, thr).sum()), 0
    for k in range(iterations):
        fit_mask = sampson_mask_f32(model, x, np.float32(thr) * np.float32(mult(k)))
        if int(fit_mask.sum()) < 8:
            break
        xi = x[fit_mask].astype(np.float64)
        T = []
        xh = np.empty_like(xi)
        for c in (0, 2):
            cen = xi[:, c:c + 2].mean(0)
            var = (xi[:, c:c + 2] ** 2).sum(1).mean() - (cen ** 2).sum()
            sc = np.sqrt(2.0 / var) if var > 0 else 1.0
            xh[:, c:c + 2] = sc * (xi[:, c:c + 2] - cen)
            T.append(np.array([[sc, 0, -sc * cen[0]], [0, sc, -sc * cen[1]], [0, 0, 1]]))
        A = design_matrix(xh)
        w, V = np.linalg.eigh(A.T @ A)
        model = project_essential(T[0].T @ V[:, 0].reshape(3, 3) @ T[1])
        c = int(sampson_mask_f32(model.astype(np.float32), x, thr).sum())
        if c > count:
            E, count, accepted = model, c, accepted + 1
    return E, count, accepted


# --------------------------------------------------------------------------
# Homography RANSAC (CudaSift FindHomography: ComputeHomographies matching.cu:907-948,
# TestHomographies 953-996, selection 1063-1071) - SURVEY.md 8f rank 3
# --------------------------------------------------------------------------
def homography_hypotheses(x: np.ndarray, idx4: np.ndarray) -> np.ndarray:
    """H candidates (L,3,3) in fp64 mapping image-1 to image-2 points, from 4
    correspondences each (idx4: (L,4)); exact 4-point DLT null vector, unit
    Frobenius norm (CudaSift solves the same system with h8 = 1)."""
    p = x[idx4].astype(np.float64)                       # (L,4,4)
    X, Y, U, V = p[..., 0], p[..., 1], p[..., 2], p[..., 3]
    Z, O1 = np.zeros_like(X), np.ones_like(X)
    r0 = np.stack([-X, -Y, -O1, Z, Z, Z, U * X, U * Y, U], -1)
    r1 = np.stack([Z, Z, Z, -X, -Y, -O1, V * X, V * Y, V], -1)
    A = np.concatenate([r0, r1], 1)                      # (L,8,9)
    _, _, Vt = np.linalg.svd(A)
    Hm = Vt[:, -1, :]
    return (Hm / np.linalg.norm(Hm, axis=1, keepdims=True)).reshape(-1, 3, 3)


def homography_mask_f32(Hm: np.ndarray, x: np.ndarray, thresh: float) -> np.ndarray:
    """Inliers under the transfer-error test with the kernels' fp32 fma tree
    (csrc/sampson.cuh: homography_d), emulated like sampson_mask_f32."""
    f32, f64 = np.float32, np.float64
    e = Hm.reshape(9).astype(f32)
    x1, y1, x2, y2 = (x[:, i].astype(f32) for i in range(4))

    def fma(a, b, c):
        return (a.astype(f64) * np.asarray(b, f64) + np.asarray(c, f64)).astype(f32)

    X = fma(x1, e[0], fma(y1, e[1], np.full_like(x1, e[2])))
    Y = fma(x1, e[3], fma(y1, e[4], np.full_like(x1, e[5])))
    W = fma(x1, e[6], fma(y1, e[7], np.full_like(x1, e[8])))
    ex = fma(x2, W, -X)
    ey = fma(y2, W, -Y)
    err2 = fma(ex, ex, (ey * ey).astype(f32))
    nthr = -(f32(thresh) * f32(thresh))
    d = fma((W * W).astype(f32), nthr, err2)
    return d < 0


def homography_counts(Hm: np.ndarray, x: np.ndarray, thresh: float, band: float = 1e-4):
    """fp64 counts of the same test + borderline counts (|d| <= band * thr^2 W^2)."""
    Hm = Hm.reshape(-1, 3, 3).astype(np.float64)
    x1 = np.stack([x[:, 0], x[:, 1], np.ones(len(x))], 0).astype(np.float64)
    q = Hm @ x1                                           # (L,3,n)
    ex = x[:, 2][None] * q[:, 2] - q[:, 0]
    ey = x[:, 3][None] * q[:, 2] - q[:, 1]
    t = thresh * thresh * q[:, 2] ** 2
    d = ex * ex + ey * ey - t
    return (d < 0).sum(1), (np.abs(d) <= band * t + 1e-300).sum(1)


def argmax_first(counts: np.ndarray) -> int:
    """thrust::max_element semantics (sfm.cu:135-136): first maximum.  The
    reference then subtracts one (sfm.cu:137, SURVEY Q13: a bug); we do not."""
    return int(np.argmax(counts))


def adaptive_rounds(H_max: int, first_round: int, growth: int) -> list[int]:
    """Round boundaries of the adaptive RANSAC: hypotheses tried after each round."""
    out, hi = [], first_round
    while True:
        out.append(min(hi, H_max))
        if hi >= H_max:
            return out
        hi *= growth


def adaptive_used(best_after_round, n: int, confidence: float, bounds: list[int]) -> int:
    """Adaptive termination (new functionality; the reference lists "limit on RANSAC
    iterations" as future work, README.md:65-69): the textbook bound
    needed = log(1 - p) / log(1 - w^8), w = best inlier ratio so far.  best_after_round[r] =
    best inlier count (per pair: min over pairs decides) over hypotheses [0, bounds[r])."""
    for r, done in enumerate(bounds):
        w8 = (np.min(best_after_round[r]) / n) ** 8
        if w8 >= 1.0 or (w8 > 0.0 and done >= math.log1p(-confidence) / math.log1p(-w8)):
            return done
    return bounds[-1]


# --------------------------------------------------------------------------
# Pose candidates and cheirality (computePosecandidates sfm.cu:238-252,
# candidate_kernels kernels.h:357-385, choosePose sfm.cu:254-307)
# --------------------------------------------------------------------------
def svd_rot(E: np.ndarray):
    """SVD with the reference svd()'s contract (svd.h:311-335): U, V proper
    rotations, singular values sorted, the last one carries the sign."""
    U, S, Vt = np.linalg.svd(E.astype(np.float64))
    V = Vt.T
    if np.linalg.det(U) < 0:
        U[:, 2] = -U[:, 2]
        S[2] = -S[2]
    if np.linalg.det(V) < 0:
        V[:, 2] = -V[:, 2]
        S[2] = -S[2]
    return U, S, V


def reference_null_direction(E: np.ndarray) -> np.ndarray:
    """Third column of V as the reference's svd() (svd.h:311-335) ORIENTS it.  The SO(3) contract leaves one
    discrete freedom - the sign of v3 (together with u3 and one in-plane column) - which permutes the pose
    candidates 0<->3, 1<->2.  The reference's choice is decided by the rotation path of its algorithm (McAdams et
    al. 2011): cyclic Jacobi on E^T E from the identity over the pairs (0,1), (1,2), (2,0), 4 sweeps, half-angle
    estimate (ch, sh) ~ (2 (s_pp - s_qq), s_pq) or the fixed angle pi/8 when gamma sh^2 >= ch^2 (svd.h:120-215),
    then columns ordered by decreasing |E v_i| with negating swaps (svd.h:217-241).  Replayed here in fp32 on plain
    matrices for that one bit only; pinned against the reference's own host svd() in tests/test_cpu_oracle.py."""
    f = np.float32
    gamma, cstar, sstar = f(5.828427124746190), f(0.923879532511287), f(0.382683432365090)
    A = np.asarray(E, f).reshape(3, 3)
    S = (A.T @ A).astype(f)
    V = np.eye(3, dtype=f)
    for _ in range(4):
        for p, q in ((0, 1), (1, 2), (2, 0)):
            ch, sh = f(2) * (S[p, p] - S[q, q]), S[p, q]
            if gamma * sh * sh < ch * ch:
                w = f(1) / np.sqrt(ch * ch + sh * sh)
                ch, sh = w * ch, w * sh
            else:
                ch, sh = cstar, sstar
            c, sn = ch * ch - sh * sh, f(2) * sh * ch
            Q = np.eye(3, dtype=f)
            Q[p, p], Q[q, q], Q[p, q], Q[q, p] = c, c, -sn, sn
            S = (Q.T @ S @ Q).astype(f)
            V = (V @ Q).astype(f)
    rho = list(((A @ V) ** 2).sum(axis=0))
    for i, j in ((0, 1), (0, 2), (1, 2)):
        if rho[i] < rho[j]:
            rho[i], rho[j] = rho[j], rho[i]
            vi = V[:, i].copy()
            V[:, i], V[:, j] = V[:, j], -vi
    return V[:, 2].astype(np.float64)


def svd_reference_orientation(E: np.ndarray):
    """svd_rot with v3 (and u3, and column 0 of both) oriented as the reference's svd() orients them."""
    U, S, V = svd_rot(E)
    if reference_null_direction(E) @ V[:, 2] < 0:
        U[:, [0, 2]] = -U[:, [0, 2]]
        V[:, [0, 2]] = -V[:, [0, 2]]
    return U, S, V


def det_reference_typo(a: np.ndarray) -> float:
    """det() exactly as written at svd.h:337-341 (third term a0*a3*a8, SURVEY Q15)."""
    a = a.reshape(9)
    return float(a[0] * a[4] * a[8] - a[0] * a[5] * a[7] - a[0] * a[3] * a[8] + a[1] * a[5] * a[6] + a[2] * a[3] * a[7] - a[2] * a[4] * a[6])


def pose_candidates(E: np.ndarray, compat: bool = True) -> np.ndarray:
    """Four 4x4 candidates.  compat=True replicates the reference
    (SURVEY Appendix A.4): P_i = [ (U W(^T) V^T)^T | +-u3 ; 0 0 0 1 ],
    W for i<2, W^T for i>=2, sign - for i in {0,2}, with the det-typo sign fix
    applied to V.  compat=False is textbook geometry for the x1^T E x2 = 0
    convention: X2 = R X1 + t with E^T = [t]x R.  In compat mode the candidates also come in the reference's ORDER
    (svd_reference_orientation); match_candidates remains for comparing against arbitrary SVDs."""
    U, _, V = svd_reference_orientation(E) if compat else svd_rot(E)
    W = np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1]], float)
    P = np.zeros((4, 4, 4))
    if compat:
        tmp = U @ V.T
        if det_reference_typo(tmp) < 0:
            V = -V
        for i in range(4):
            Rm = U @ (W if i < 2 else W.T) @ V.T
            s = -1.0 if i in (0, 2) else 1.0
            P[i, :3, :3] = Rm.T
            P[i, :3, 3] = s * U[:, 2]
            P[i, 3, 3] = 1.0
    else:
        # x1^T E x2 = 0  <=>  x2^T E^T x1 = 0, so F := E^T = [t]x R maps cam1->cam2.
        # svd(E) = U S V^T  =>  E^T = V S U^T: R = V W(^T) U^T, t = +-v3.
        for i in range(4):
            Rm = V @ (W if i < 2 else W.T) @ U.T
            if np.linalg.det(Rm) < 0:
                Rm = -Rm
            s = -1.0 if i in (0, 2) else 1.0
            P[i, :3, :3] = Rm
            P[i, :3, 3] = s * V[:, 2]
            P[i, 3, 3] = 1.0
    return P


def match_candidates(Pa: np.ndarray, Pb: np.ndarray, tol: float = 1e-3):
    """Pose-candidate sets are defined up to ONE discrete freedom of the SVD of a
    rank-2 E under the reference's U, V in SO(3) contract: negating (u1, v1, u3, v3)
    leaves E, U V^T and the det test unchanged but swaps W <-> W^T and the sign of
    u3, i.e. permutes the candidates 0<->3, 1<->2.  Which of the two an SVD returns
    is an artefact of its rotation sequence (for sigma1 == sigma2 it is decided by
    rounding), so parity of candidates means: equal under the identity or under
    that permutation.  Returns the permutation perm with Pa[i] ~ Pb[perm[i]], or None."""
    Pa, Pb = np.asarray(Pa, float).reshape(4, 4, 4), np.asarray(Pb, float).reshape(4, 4, 4)
    for perm in ((0, 1, 2, 3), (3, 2, 1, 0)):
        if all(np.abs(Pa[i] - Pb[perm[i]]).max() < tol for i in range(4)):
            return perm
    return None


def match_candidate_set(Pa: np.ndarray, Pb: np.ndarray, tol: float = 1e-4):
    """Textbook candidates (compat=False) come from an SVD whose orientation is free, so their order is too: parity
    means equal as a SET.  Returns a bijection perm with |Pa[i] - Pb[perm[i]]| < tol, or None."""
    import itertools

    Pa, Pb = np.asarray(Pa, float).reshape(4, 4, 4), np.asarray(Pb, float).reshape(4, 4, 4)
    for perm in itertools.permutations(range(4)):
        if all(np.abs(Pa[i] - Pb[perm[i]]).max() < tol for i in range(4)):
            return perm
    return None


def dlt_rows(x: np.ndarray, M: np.ndarray) -> np.ndarray:
    """compute_linear_triangulation_A (kernels.h:387-431): per point the 4x4
    [x1*I[2]-I[0]; y1*I[2]-I[1]; x2*M[2]-M[0]; y2*M[2]-M[1]] with camera 1 = I4."""
    x = np.atleast_2d(x).astype(np.float64)
    n = len(x)
    I4 = np.eye(4)
    A = np.empty((n, 4, 4))
    A[:, 0] = x[:, 0:1] * I4[2] - I4[0]
    A[:, 1] = x[:, 1:2] * I4[2] - I4[1]
    A[:, 2] = x[:, 2:3] * M[2] - M[0]
    A[:, 3] = x[:, 3:4] * M[2] - M[1]
    return A


def triangulate(x: np.ndarray, M: np.ndarray) -> np.ndarray:
    """linear_triangulation (sfm.cu:309-336) + normalize_pt_kernal
    (kernels.h:433-450): null vector of each A, de-homogenised; (0,0,0,1) when
    w == 0.  Returns (4,n) SoA like d_final_points."""
    A = dlt_rows(x, M)
    _, _, Vt = np.linalg.svd(A)
    v = Vt[:, -1, :]
    w = v[:, 3]
    out = np.zeros((4, len(v)))
    ok = w != 0
    out[:3, ok] = (v[ok, :3] / w[ok, None]).T
    out[3] = 1.0
    return out


def choose_pose(x: np.ndarray, P: np.ndarray, compat: bool = True, mask: np.ndarray | None = None):
    """choosePose (sfm.cu:254-297).  compat: cheirality of correspondence 0 only,
    each candidate inverted in place, depth tested in both frames, the LAST
    passing index wins (default 0); returns (P_ind, P_after) where P_after holds
    the inverses (SURVEY Q17-Q19).  correct mode: vote over (masked) points with
    X2 = P_i X, arg-max of votes (first max), P unchanged."""
    if compat:
        Pinv = np.stack([np.linalg.inv(P[i]) for i in range(4)])
        ind = 0
        for i in range(4):
            X = triangulate(x[0:1], P[i])[:, 0]
            z1 = X[2]
            z2 = (Pinv[i] @ X)[2]
            if z1 > 0 and z2 > 0:
                ind = i
        return ind, Pinv
    return int(np.argmax(cheirality_votes(x, P, mask))), P.copy()


def cheirality_votes(x: np.ndarray, P: np.ndarray, mask: np.ndarray | None = None, tri=triangulate) -> list[int]:
    """Votes of choosePose's correct mode: per candidate, the (masked) points whose triangulation lies in front of both
    cameras.  tri(x, M) -> (4,n) is the triangulation to use (default: this module's fp64 SVD)."""
    xs = x if mask is None else x[mask]
    votes = []
    for i in range(4):
        X = tri(xs, P[i])
        z2 = (P[i] @ X)[2]
        votes.append(int(((X[2] > 0) & (z2 > 0)).sum()))
    return votes


# --------------------------------------------------------------------------
# Two-view bundle adjustment (new functionality: "bundle adjustment" is the
# reference's listed future work, README.md:65-69; SURVEY.md 8f rank 4).
# Restated in fp64 with the same parameterisation, damping schedule and
# accept rule as cuda-sfm_b200/csrc/bundle.cu.
# --------------------------------------------------------------------------
def ba_active(x: np.ndarray, M: np.ndarray, X: np.ndarray, mask: np.ndarray) -> np.ndarray:
    """Points that take part: inliers of the selected E (mask) whose triangulated
    point is finite and in front of both cameras (x1 ~ X, x2 ~ M X)."""
    Xc = X[:3].T
    Y = Xc @ M[:3, :3].T + M[:3, 3]
    return mask.astype(bool) & np.isfinite(Xc).all(1) & (Xc[:, 2] > 0) & (Y[:, 2] > 0)


def ba_cost(x: np.ndarray, R: np.ndarray, t: np.ndarray, Xc: np.ndarray) -> float:
    """Sum of squared reprojection errors in normalised coordinates, both views."""
    Y = Xc @ R.T + t
    r1 = Xc[:, :2] / Xc[:, 2:3] - x[:, 0:2]
    r2 = Y[:, :2] / Y[:, 2:3] - x[:, 2:4]
    return float((r1 * r1).sum() + (r2 * r2).sum())


def _rodrigues(w: np.ndarray) -> np.ndarray:
    th = float(np.linalg.norm(w))
    Kx = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    if th < 1e-12:
        return np.eye(3) + Kx
    return np.eye(3) + (math.sin(th) / th) * Kx + ((1 - math.cos(th)) / (th * th)) * (Kx @ Kx)


def bundle_adjust(x: np.ndarray, M: np.ndarray, X: np.ndarray, active: np.ndarray, iterations: int = 10,
                  lambda0: float = 1e-3):
    """Levenberg-Marquardt over (R, t) of camera 2 and the active 3-D points; camera 1 = [I|0].
    Left-multiplicative rotation update R <- exp([dw]x) R; Marquardt damping lambda*diag on the
    point blocks and on the reduced 6x6 camera system (Schur complement); a step is accepted iff
    the cost decreases strictly (lambda /= 3, floor 1e-9), else rejected (lambda *= 4, cap 1e6).
    Finally the gauge is fixed to |t| = 1 (points scaled alike).  Returns dict(M, X, cost0, cost,
    accepted, n_active)."""
    x = np.asarray(x, np.float64)
    R, t = M[:3, :3].astype(np.float64).copy(), M[:3, 3].astype(np.float64).copy()
    Xall = X[:3].T.astype(np.float64).copy()
    act = np.flatnonzero(active)
    xa = x[act]
    Xc = Xall[act].copy()
    lam, accepted = lambda0, 0
    cost0 = cost = ba_cost(xa, R, t, Xc) if len(act) else 0.0
    if len(act) >= 8:
        for _ in range(iterations):
            n = len(Xc)
            iz = 1.0 / Xc[:, 2]
            u, v = Xc[:, 0] * iz, Xc[:, 1] * iz
            r1 = np.stack([u - xa[:, 0], v - xa[:, 1]], 1)
            Jp1 = np.zeros((n, 2, 3))
            Jp1[:, 0, 0] = iz; Jp1[:, 0, 2] = -u * iz
            Jp1[:, 1, 1] = iz; Jp1[:, 1, 2] = -v * iz
            Q = Xc @ R.T
            Y = Q + t
            iz2 = 1.0 / Y[:, 2]
            u2, v2 = Y[:, 0] * iz2, Y[:, 1] * iz2
            r2 = np.stack([u2 - xa[:, 2], v2 - xa[:, 3]], 1)
            Jpi = np.zeros((n, 2, 3))
            Jpi[:, 0, 0] = iz2; Jpi[:, 0, 2] = -u2 * iz2
            Jpi[:, 1, 1] = iz2; Jpi[:, 1, 2] = -v2 * iz2
            Jp2 = Jpi @ R
            nQx = np.zeros((n, 3, 3))                      # -[Q]x
            nQx[:, 0, 1] = Q[:, 2]; nQx[:, 0, 2] = -Q[:, 1]
            nQx[:, 1, 0] = -Q[:, 2]; nQx[:, 1, 2] = Q[:, 0]
            nQx[:, 2, 0] = Q[:, 1]; nQx[:, 2, 1] = -Q[:, 0]
            Jc = np.concatenate([Jpi @ nQx, Jpi], axis=2)  # (n,2,6)
            V = Jp1.transpose(0, 2, 1) @ Jp1 + Jp2.transpose(0, 2, 1) @ Jp2
            gp = (Jp1.transpose(0, 2, 1) @ r1[:, :, None] + Jp2.transpose(0, 2, 1) @ r2[:, :, None])[:, :, 0]
            Vd = V + lam * np.einsum("nii->ni", V)[:, :, None] * np.eye(3)
            Vinv = np.linalg.inv(Vd)
            W = Jc.transpose(0, 2, 1) @ Jp2                # (n,6,3)
            U = Jc.transpose(0, 2, 1) @ Jc
            gc = (Jc.transpose(0, 2, 1) @ r2[:, :, None])[:, :, 0]
            Yw = W @ Vinv
            A = (U - Yw @ W.transpose(0, 2, 1)).sum(0)
            D = np.einsum("nii->i", U)
            g = (gc - (Yw @ gp[:, :, None])[:, :, 0]).sum(0)
            try:
                dc = np.linalg.solve(A + lam * np.diag(D), -g)
            except np.linalg.LinAlgError:
                lam = min(lam * 4, 1e6)
                continue
            dp = -(Vinv @ (gp + (W.transpose(0, 2, 1) @ dc))[:, :, None])[:, :, 0]
            Rn, tn, Xn = _rodrigues(dc[:3]) @ R, t + dc[3:], Xc + dp
            Yn = Xn @ Rn.T + tn
            ok = bool(np.all(Xn[:, 2] > 0) and np.all(Yn[:, 2] > 0))
            cn = ba_cost(xa, Rn, tn, Xn) if ok else np.inf
            if cn < cost:
                R, t, Xc, cost = Rn, tn, Xn, cn
                lam = max(lam / 3, 1e-9)
                accepted += 1
            else:
                lam = min(lam * 4, 1e6)
    sc = 1.0 / np.linalg.norm(t) if np.linalg.norm(t) > 0 else 1.0
    Mo = np.eye(4)
    Mo[:3, :3], Mo[:3, 3] = R, t * sc
    Xo = triangulate(x, Mo)     # whole cloud under the refined camera; adjusted points for the active set
    Xo[:3, act] = (Xc * sc).T
    return dict(M=Mo, X=Xo, cost0=cost0, cost=cost, accepted=accepted, n_active=len(act), gauge_scale=sc)


def essential_from_pose(M: np.ndarray) -> np.ndarray:
    """E with x1^T E x2 = 0 for x1 ~ X, x2 ~ R X + t: E = ([t]x R)^T."""
    R, t = M[:3, :3], M[:3, 3]
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    return (tx @ R).T


def bundle_adjust_rounds(x: np.ndarray, M: np.ndarray, E: np.ndarray, thr: float = 1e-6, outer_rounds: int = 3,
                         iterations: int = 10):
    """Outer loop of sfmb200_bundle_adjust: inliers of the current E -> LM -> E from the
    refined camera -> recount -> commit unless the consensus collapsed.  Returns dict(M, E, X, inliers, rounds=[per-round results])."""
    M, E = np.asarray(M, np.float64), np.asarray(E, np.float64)
    rounds = []
    X = None
    base_count = int(sampson_mask_f32(E, x, thr).sum())
    for _ in range(outer_rounds):
        mask = sampson_mask_f32(E, x, thr)
        X0 = triangulate(x, M)
        act = ba_active(x, M, X0, mask)
        if act.sum() < 8:
            X = X0
            rounds.append(dict(M=M, X=X0, cost0=0.0, cost=0.0, accepted=0, n_active=int(act.sum())))
            continue
        r = bundle_adjust(x, M, X0, act, iterations)
        # commit guard: the adjusted model replaces the incumbent only if its E still explains >= 95 % of the
        # correspondences the model had when the call started
        E_new = essential_from_pose(r["M"])
        r["inliers"] = int(sampson_mask_f32(E_new, x, thr).sum())
        r["committed"] = 20 * r["inliers"] >= 19 * base_count
        if r["committed"]:
            M, X, E = r["M"], r["X"], E_new
        else:
            X = triangulate(x, M)
        rounds.append(r)
    return dict(M=M, E=E, X=X, inliers=int(sampson_mask_f32(E, x, thr).sum()), rounds=rounds)


# --------------------------------------------------------------------------
# N-view chaining of consecutive pairs (new functionality, SURVEY.md 8f rank 4:
# the reference shapes Image_pair for image_count views, sfm.h:23,30-31, but only
# ever handles two).  Pair b = (view b, view b+1); correspondence i is the same
# track in every pair.  Restates cuda-sfm_b200/csrc/chain.cu.
# --------------------------------------------------------------------------
CHAIN_BINS = 2048
CHAIN_LOG_RANGE = math.log(16.0)      # ratios in [1/16, 16]


def chain_valid(x: np.ndarray, M: np.ndarray, X: np.ndarray, mask: np.ndarray) -> np.ndarray:
    """A track contributes from a pair when it is an inlier of the pair's E and its point is finite and in
    front of both cameras."""
    return ba_active(x, M, X, mask)


def chain_scales(Ms, Xs, valids):
    """scale[b] (b >= 1) = robust central value of depth_in_camera_b(pair b-1) / depth_in_camera_b(pair b)
    over the tracks valid in both pairs: median bin of a 2048-bin histogram of the log ratio over
    [ln 1/16, ln 16], refined to the mean log ratio of the entries of that bin.  scale[0] = 1.
    Also returns the number of tracks used."""
    B = len(Ms)
    scales, used = np.ones(B), np.zeros(B, int)
    for b in range(1, B):
        both = valids[b - 1] & valids[b]
        Xp = Xs[b - 1][:3].T[both]
        zprev = Xp @ Ms[b - 1][2, :3] + Ms[b - 1][2, 3]
        zcur = Xs[b][2][both]
        lr = np.log(zprev / zcur)
        ok = np.isfinite(lr) & (np.abs(lr) < CHAIN_LOG_RANGE)
        lr = lr[ok]
        used[b] = len(lr)
        if len(lr) == 0:
            continue
        bins = np.minimum(((lr + CHAIN_LOG_RANGE) * (CHAIN_BINS / (2 * CHAIN_LOG_RANGE))).astype(int), CHAIN_BINS - 1)
        hist = np.bincount(bins, minlength=CHAIN_BINS)
        cum = np.cumsum(hist)
        mb = int(np.searchsorted(cum, (len(lr) + 1) // 2))
        scales[b] = math.exp(lr[bins == mb].mean())
    return scales, used


def chain_cameras(Ms, scales):
    """Global world(camera 0) -> camera k matrices in units of the first baseline:
    G_0 = I, G_{b+1} = [R_b | S_b t_b] G_b with S_b = prod_{j<=b} scale[j]."""
    G = [np.eye(4)]
    S = np.cumprod(scales)
    for b, M in enumerate(Ms):
        T = np.eye(4)
        T[:3, :3], T[:3, 3] = M[:3, :3], S[b] * M[:3, 3]
        G.append(T @ G[-1])
    return np.stack(G), S


def chain_merge(Xs, valids, G, S):
    """Global position of every track: mean over the pairs where it is valid of G_b^-1 (S_b X_b);
    (0,0,0,1) and count 0 when no pair sees it."""
    n = Xs[0].shape[1]
    acc, cnt = np.zeros((3, n)), np.zeros(n, int)
    for b, X in enumerate(Xs):
        R, t = G[b][:3, :3], G[b][:3, 3]
        W = R.T @ (S[b] * X[:3] - t[:, None])
        acc[:, valids[b]] += W[:, valids[b]]
        cnt += valids[b]
    out = np.zeros((4, n))
    out[:3, cnt > 0] = acc[:, cnt > 0] / cnt[cnt > 0]
    out[3] = 1.0
    return out, cnt


GBA_GATE = 25.0


def gba_observations(xs, valids, G=None, X=None, thr: float = 1e-6):
    """Observation set of the global adjustment (chain.cu: gba_prepare_kernel): view k sees track i when the track is valid in
    a pair that contains view k and - when the chained start (G, X) is given - its reprojection error there is at most
    GBA_GATE x thr squared (a match can pass a pair's epipolar test and still be wrong along the epipolar line).
    xs: per pair (n,4) normalised correspondences; valids: per pair (n,) bool.
    Returns uv (V, n, 2) and obs (V, n) bool; tracks seen by fewer than two views are dropped."""
    B, n = len(xs), len(xs[0])
    V = B + 1
    uv = np.zeros((V, n, 2))
    obs = np.zeros((V, n), bool)
    uv[0] = xs[0][:, :2]
    for b in range(B):
        uv[b + 1] = xs[b][:, 2:]
        obs[b] |= valids[b]
        obs[b + 1] |= valids[b]
    if G is not None:
        Xc = np.asarray(X, float)[:3]
        for k in range(V):
            Y = Xc.T @ G[k][:3, :3].T + G[k][:3, 3]
            with np.errstate(divide="ignore", invalid="ignore"):
                d2 = ((Y[:, :2] / Y[:, 2:3] - uv[k]) ** 2).sum(1)
            obs[k] &= (Y[:, 2] > 0) & (d2 <= GBA_GATE * thr)
    obs[:, obs.sum(0) < 2] = False
    return uv, obs


def gba_cost(uv, obs, G, X):
    c = 0.0
    for k in range(len(G)):
        Y = X[:, obs[k]].T @ G[k][:3, :3].T + G[k][:3, 3]
        if np.any(Y[:, 2] <= 0):
            return np.inf
        c += (((Y[:, :2] / Y[:, 2:3]) - uv[k][obs[k]]) ** 2).sum()
    return float(c)


def bundle_adjust_global(uv, obs, G, X, iterations: int = 30, lam0: float = 1e-3):
    """Global bundle adjustment over the chained reconstruction (chain.cu, sfmb200_bundle_adjust_global) in fp64 with the same
    parameterisation (cameras 1..V-1: left-multiplicative so(3) update + translation; camera 0 fixed; one point per active
    track), the same multiplicative LM damping, accept rule (strict decrease, every observation in front of its camera:
    lambda / 3, else 4 lambda) and final gauge (|t_1| restored).  The step is taken from the explicit damped normal
    equations - identical to the Schur-complement step of the CUDA code.  G: (V,4,4); X: (3,n) or (4,n).
    Returns G, X, stats dict."""
    V, n = obs.shape
    G = np.array(G, float).copy()
    X = np.array(X, float)[:3].copy()
    act = np.flatnonzero(obs.any(0))
    pid = -np.ones(n, int)
    pid[act] = np.arange(len(act))
    ncam = 6 * (V - 1)
    t1 = np.linalg.norm(G[1][:3, 3]) if V > 1 else 1.0
    lam = lam0
    cost = gba_cost(uv, obs, G, X)
    cost0, accepted = cost, 0
    for _ in range(iterations):
        rows = int(obs.sum()) * 2
        J = np.zeros((rows, ncam + 3 * len(act)))
        r = np.zeros(rows)
        q = 0
        for k in range(V):
            R, t = G[k][:3, :3], G[k][:3, 3]
            for i in np.flatnonzero(obs[k]):
                Q = R @ X[:, i]
                Y = Q + t
                iz = 1.0 / Y[2]
                u, v = Y[0] * iz, Y[1] * iz
                bp = np.array([[iz, 0, -u * iz], [0, iz, -v * iz]])
                r[q:q + 2] = [u - uv[k][i, 0], v - uv[k][i, 1]]
                J[q:q + 2, ncam + 3 * pid[i]: ncam + 3 * pid[i] + 3] = bp @ R
                if k > 0:
                    N = np.array([[0, Q[2], -Q[1]], [-Q[2], 0, Q[0]], [Q[1], -Q[0], 0]])
                    J[q:q + 2, 6 * (k - 1): 6 * (k - 1) + 3] = bp @ N
                    J[q:q + 2, 6 * (k - 1) + 3: 6 * (k - 1) + 6] = bp
                q += 2
        H = J.T @ J
        H[np.diag_indices_from(H)] *= 1.0 + lam
        try:
            d = np.linalg.solve(H, -J.T @ r)
        except np.linalg.LinAlgError:
            lam = min(4 * lam, 1e6)
            continue
        Gn = G.copy()
        for k in range(1, V):
            w, dt = d[6 * (k - 1): 6 * (k - 1) + 3], d[6 * (k - 1) + 3: 6 * (k - 1) + 6]
            Gn[k][:3, :3] = _rodrigues(w) @ G[k][:3, :3]
            Gn[k][:3, 3] = G[k][:3, 3] + dt
        Xn = X.copy()
        Xn[:, act] += d[ncam:].reshape(-1, 3).T
        cn = gba_cost(uv, obs, Gn, Xn)
        if np.isfinite(cn) and cn < cost:
            G, X, cost, accepted = Gn, Xn, cn, accepted + 1
            lam = max(lam / 3, 1e-9)
        else:
            lam = min(4 * lam, 1e6)
    sc = t1 / np.linalg.norm(G[1][:3, 3]) if V > 1 else 1.0
    G[:, :3, 3] *= sc
    X[:, act] *= sc
    return G, X, {"cost_entry": cost0, "cost": cost, "accepted": accepted, "lambda": lam, "gauge_scale": sc}


def bundle_adjust_global_schur(uv, obs, G, X, iterations: int = 30, lam0: float = 1e-3):
    """bundle_adjust_global restated the way chain.cu computes the step, for sequences and track counts where the dense
    Jacobian is too large: per view the residuals and Jacobians of all its observations at once, the damped 3x3 point
    blocks inverted as a batch, the reduced camera system S dc = -rhs of 6 (V-1) unknowns assembled from them and solved
    densely, then the back-substitution dX_i = -V_i*^-1 (g_p,i + sum_k W_ki^T dc_k).  Same damping (diagonal x (1 + lambda)),
    accept rule, lambda schedule and gauge as the dense version; same returns."""
    V, n = obs.shape
    G = np.array(G, float).copy()
    X = np.array(X, float)[:3].copy()
    act = np.flatnonzero(obs.any(0))
    P, K = len(act), V - 1
    ob = obs[:, act]
    t1 = np.linalg.norm(G[1][:3, 3]) if V > 1 else 1.0
    lam = lam0
    cost = gba_cost(uv, obs, G, X)
    cost0, accepted = cost, 0
    for _ in range(iterations):
        Vp = np.zeros((P, 3, 3))
        gp = np.zeros((P, 3))
        W = np.zeros((P, K, 6, 3))                          # W_ki = Jc^T Jp, zero where view k does not see track i
        U = np.zeros((K, 6, 6))
        gc = np.zeros((K, 6))
        Xa = X[:, act].T
        for k in range(V):
            j = np.flatnonzero(ob[k])
            R, t = G[k][:3, :3], G[k][:3, 3]
            Q = Xa[j] @ R.T
            Y = Q + t
            iz = 1.0 / Y[:, 2]
            u, v = Y[:, 0] * iz, Y[:, 1] * iz
            r = np.stack([u - uv[k][act[j], 0], v - uv[k][act[j], 1]], 1)
            bp = np.zeros((len(j), 2, 3))
            bp[:, 0, 0] = iz; bp[:, 0, 2] = -u * iz
            bp[:, 1, 1] = iz; bp[:, 1, 2] = -v * iz
            Jp = bp @ R
            Vp[j] += Jp.transpose(0, 2, 1) @ Jp
            gp[j] += (Jp.transpose(0, 2, 1) @ r[:, :, None])[:, :, 0]
            if k == 0:
                continue
            N = np.zeros((len(j), 3, 3))                      # -[Q]x
            N[:, 0, 1] = Q[:, 2]; N[:, 0, 2] = -Q[:, 1]
            N[:, 1, 0] = -Q[:, 2]; N[:, 1, 2] = Q[:, 0]
            N[:, 2, 0] = Q[:, 1]; N[:, 2, 1] = -Q[:, 0]
            Jc = np.concatenate([bp @ N, bp], axis=2)
            U[k - 1] = np.einsum("mra,mrb->ab", Jc, Jc)
            gc[k - 1] = np.einsum("mra,mr->a", Jc, r)
            W[j, k - 1] = Jc.transpose(0, 2, 1) @ Jp
        Vp[:, np.arange(3), np.arange(3)] *= 1.0 + lam
        U[:, np.arange(6), np.arange(6)] *= 1.0 + lam
        Vinv = np.linalg.inv(Vp)
        T = np.einsum("pkac,pcd->pkad", W, Vinv)            # W_ki V_i*^-1
        S = -np.einsum("pkad,plbd->kalb", T, W).reshape(6 * K, 6 * K)
        for k in range(K):
            S[6 * k: 6 * k + 6, 6 * k: 6 * k + 6] += U[k]
        rhs = (gc - np.einsum("pkad,pd->ka", T, gp)).reshape(-1)
        try:
            dc = np.linalg.solve(S, -rhs)
        except np.linalg.LinAlgError:
            lam = min(4 * lam, 1e6)
            continue
        dX = -np.einsum("pcd,pd->pc", Vinv, gp + np.einsum("pkac,ka->pc", W, dc.reshape(K, 6)))
        Gn = G.copy()
        for k in range(1, V):
            w, dt = dc[6 * (k - 1): 6 * (k - 1) + 3], dc[6 * (k - 1) + 3: 6 * (k - 1) + 6]
            Gn[k][:3, :3] = _rodrigues(w) @ G[k][:3, :3]
            Gn[k][:3, 3] = G[k][:3, 3] + dt
        Xn = X.copy()
        Xn[:, act] += dX.T
        cn = gba_cost(uv, obs, Gn, Xn)
        if np.isfinite(cn) and cn < cost:
            G, X, cost, accepted = Gn, Xn, cn, accepted + 1
            lam = max(lam / 3, 1e-9)
        else:
            lam = min(4 * lam, 1e6)
    sc = t1 / np.linalg.norm(G[1][:3, 3]) if V > 1 else 1.0
    G[:, :3, 3] *= sc
    X[:, act] *= sc
    return G, X, {"cost_entry": cost0, "cost": cost, "accepted": accepted, "lambda": lam, "gauge_scale": sc}


def to_vbo(points_soa: np.ndarray) -> np.ndarray:
    """kernCopyPositionsToVBO (kernels.h:471-483): 4xN SoA -> Nx4 AoS (x,y,z,1)."""
    out = points_soa.T.copy()
    out[:, 3] = 1.0
    return out
