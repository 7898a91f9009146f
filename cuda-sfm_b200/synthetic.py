"""Synthetic two-view scenes for BASELINE.json configs 2-5 and the reference's
camera intrinsics (src/main.cpp:292-297).  Pure numpy host code: input generation
for bench.py, the tools and the tests - not part of the checker, not a compute path.
"""
from __future__ import annotations

import numpy as np

F_REF = 2360.0
W_REF, H_REF = 720, 576


def reference_K(w: int = W_REF, h: int = H_REF):
    """K and K^-1 exactly as src/main.cpp:292-297 builds them (fp32)."""
    K = np.array([[F_REF, 0, w / 2.0], [0, F_REF, h / 2.0], [0, 0, 1]], dtype=np.float32)
    Kinv = np.array(
        [[1.0 / F_REF, 0, -(w / 2.0) / F_REF], [0, 1.0 / F_REF, -(h / 2.0) / F_REF], [0, 0, 1]],
        dtype=np.float32,
    )
    return K, Kinv


def _rot(axis, deg):
    a = np.asarray(axis, float)
    a = a / np.linalg.norm(a)
    t = np.deg2rad(deg)
    Kx = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(t) * Kx + (1 - np.cos(t)) * Kx @ Kx


def synthetic_pair(n: int, outlier_frac: float = 0.3, noise_px: float = 1.0, seed: int = 1234):
    """Two-view scene of BASELINE.json configs 2-5.

    Camera 1 = [I|0]; camera 2: X2 = R X + t with R = 10 degrees about
    (0.1, 1, 0.05) verging towards the scene (negative angle: with the positive
    one the two 720x576 views do not overlap) and unit baseline along
    (1, 0.05, 0.1).  Depth U[4, 8] baselines.  Gaussian pixel noise on both
    views; outliers replace the image-2 point by a uniform pixel.

    Returns dict: px (n,4) float32 pixel coords (u1,v1,u2,v2), R, t, is_outlier,
    X (n,3) ground-truth 3-D points in camera-1 frame.
    """
    rng_scene = np.random.Generator(np.random.PCG64(seed))
    rng_out = np.random.Generator(np.random.PCG64(seed + 1))
    rng_noise = np.random.Generator(np.random.PCG64(seed + 2))
    f, cx, cy = F_REF, W_REF / 2.0, H_REF / 2.0
    R = _rot([0.1, 1.0, 0.05], -10.0)
    t = np.array([1.0, 0.05, 0.1])
    t = t / np.linalg.norm(t)
    chunks, Xs, have = [], [], 0
    while have < n:
        m = max(4 * (n - have), 1024)
        z = rng_scene.uniform(4.0, 8.0, m)
        x = rng_scene.uniform(-1.2, 1.2, m) * z * (cx / f)
        y = rng_scene.uniform(-1.2, 1.2, m) * z * (cy / f)
        X = np.stack([x, y, z], 1)
        X2 = X @ R.T + t
        u1 = f * X[:, 0] / X[:, 2] + cx
        v1 = f * X[:, 1] / X[:, 2] + cy
        u2 = f * X2[:, 0] / X2[:, 2] + cx
        v2 = f * X2[:, 1] / X2[:, 2] + cy
        ok = (u1 >= 0) & (u1 < W_REF) & (v1 >= 0) & (v1 < H_REF) & (u2 >= 0) & (u2 < W_REF) & (v2 >= 0) & (v2 < H_REF) & (X2[:, 2] > 0)
        chunks.append(np.stack([u1, v1, u2, v2], 1)[ok])
        Xs.append(X[ok])
        have += int(ok.sum())
    px = np.concatenate(chunks)[:n]
    X = np.concatenate(Xs)[:n]
    px = px + rng_noise.normal(0.0, noise_px, px.shape)
    is_out = rng_out.random(n) < outlier_frac
    k = int(is_out.sum())
    px[is_out, 2] = rng_out.uniform(0, W_REF, k)
    px[is_out, 3] = rng_out.uniform(0, H_REF, k)
    return {"px": px.astype(np.float32), "R": R, "t": t, "is_outlier": is_out, "X": X}


def synthetic_sequence(views: int, n: int, outlier_frac: float = 0.2, noise_px: float = 0.5, seed: int = 4321,
                       step_deg: float = -6.0, depth=(4.0, 8.0)):
    """N-view scene for the pose-chaining stage (SURVEY 8f rank 4): camera 0 = [I|0], camera k+1 =
    [R_s | t_k] * camera k with R_s = step_deg about (0.1, 1, 0.05) verging towards the scene and
    baselines of DIFFERENT lengths along (1, 0.05, 0.1), so that the relative scales are not all 1.
    Every one of the n tracks is visible in every view (index-aligned tracks); per view k >= 1 a fraction
    of the observations is replaced by uniform pixels.

    Returns dict: px_views (views, n, 2) float32, px_pairs (views-1, n, 4) float32 = (view b, view b+1),
    G (views, 4, 4) world(camera 0)->camera k, X (n, 3), is_outlier (views, n), baselines (views-1,)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    f, cx, cy = F_REF, W_REF / 2.0, H_REF / 2.0
    Rs = _rot([0.1, 1.0, 0.05], step_deg)
    tdir = np.array([1.0, 0.05, 0.1])
    tdir = tdir / np.linalg.norm(tdir)
    baselines = 0.5 + 0.5 * rng.random(views - 1)
    G = [np.eye(4)]
    for k in range(views - 1):
        S = np.eye(4)
        S[:3, :3], S[:3, 3] = Rs, tdir * baselines[k]
        G.append(S @ G[-1])
    G = np.stack(G)
    Xs, have = [], 0
    while have < n:
        m = max(4 * (n - have), 1024)
        z = rng.uniform(depth[0], depth[1], m)
        X = np.stack([rng.uniform(-1.2, 1.2, m) * z * (cx / f), rng.uniform(-1.2, 1.2, m) * z * (cy / f), z], 1)
        ok = np.ones(m, bool)
        for k in range(views):
            Y = X @ G[k, :3, :3].T + G[k, :3, 3]
            u, v = f * Y[:, 0] / Y[:, 2] + cx, f * Y[:, 1] / Y[:, 2] + cy
            ok &= (Y[:, 2] > 0) & (u >= 0) & (u < W_REF) & (v >= 0) & (v < H_REF)
        Xs.append(X[ok])
        have += int(ok.sum())
    X = np.concatenate(Xs)[:n]
    px = np.empty((views, n, 2))
    for k in range(views):
        Y = X @ G[k, :3, :3].T + G[k, :3, 3]
        px[k, :, 0], px[k, :, 1] = f * Y[:, 0] / Y[:, 2] + cx, f * Y[:, 1] / Y[:, 2] + cy
    px += rng.normal(0.0, noise_px, px.shape)
    is_out = np.zeros((views, n), bool)
    for k in range(1, views):
        is_out[k] = rng.random(n) < outlier_frac
        c = int(is_out[k].sum())
        px[k, is_out[k], 0] = rng.uniform(0, W_REF, c)
        px[k, is_out[k], 1] = rng.uniform(0, H_REF, c)
    px = px.astype(np.float32)
    pairs = np.stack([np.concatenate([px[b], px[b + 1]], 1) for b in range(views - 1)])
    return {"px_views": px, "px_pairs": pairs, "G": G, "X": X, "is_outlier": is_out, "baselines": baselines}


def synthetic_orbit(views: int, n: int, noise_px: float = 0.5, seed: int = 2468, radius: float = 6.0,
                    step_deg=(0.8, 2.0), window=(2, 10), dropout: float = 0.1):
    """Long N-view sequence (up to a full turn) for the chaining and global-adjustment stages: camera k sits on a circle of
    the given radius about the scene centre (0, 0, radius), turned by a random step in step_deg degrees per view about the
    vertical axis and looking at the centre, so baselines (and the relative scales of consecutive pairs) differ.  Camera 0
    = [I|0].  Each track is seen by a window of consecutive views whose length is drawn from window (inclusive) and which
    the ends of the sequence may cut short; each view strictly inside the window drops it with probability dropout.  A view that does not see a track holds a uniform pixel
    for it, one per view: pair k-1's second image and pair k's first image carry the same pixel.

    Returns dict: px_views (views, n, 2) float32, px_pairs (views-1, n, 4) float32 = (view b, view b+1), G (views, 4, 4)
    world(camera 0)->camera k, X (n, 3), visible (views, n) bool, baselines (views-1,)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    f, cx, cy = F_REF, W_REF / 2.0, H_REF / 2.0
    theta = np.concatenate([[0.0], np.cumsum(np.deg2rad(rng.uniform(step_deg[0], step_deg[1], views - 1)))])
    C = np.array([0.0, 0.0, radius])
    G = np.tile(np.eye(4), (views, 1, 1))
    for k, th in enumerate(theta):
        Rc = _rot([0.0, 1.0, 0.0], np.rad2deg(th))                 # camera -> world; optical axis towards the centre
        G[k, :3, :3] = Rc.T
        G[k, :3, 3] = -Rc.T @ (C - radius * Rc[:, 2])
    baselines = np.linalg.norm(np.diff([-G[k, :3, :3].T @ G[k, :3, 3] for k in range(views)], axis=0), axis=1)
    lo, hi = window[0], min(window[1], views)
    length = rng.integers(lo, hi + 1, n)
    start = (rng.random(n) * (views + length - 1)).astype(int) - (length - 1)     # windows cut by the ends: even coverage
    k_ = np.arange(views)[:, None]
    in_window = (k_ >= start) & (k_ < start + length)
    visible = in_window & ~((k_ > start) & (k_ < start + length - 1) & (rng.random((views, n)) < dropout))
    X = np.empty((n, 3))
    todo = np.arange(n)
    while len(todo):                                               # a point must project into every view of its window
        P = C + np.stack([rng.uniform(-1, 1, len(todo)), rng.uniform(-0.6, 0.6, len(todo)), rng.uniform(-1, 1, len(todo))], 1)
        ok = np.ones(len(todo), bool)
        for k in range(views):
            w = in_window[k, todo]
            if not w.any():
                continue
            Y = P[w] @ G[k, :3, :3].T + G[k, :3, 3]
            u, v = f * Y[:, 0] / Y[:, 2] + cx, f * Y[:, 1] / Y[:, 2] + cy
            ok[np.flatnonzero(w)[~((Y[:, 2] > 0) & (u >= 0) & (u < W_REF) & (v >= 0) & (v < H_REF))]] = False
        X[todo[ok]] = P[ok]
        todo = todo[~ok]
    px = np.empty((views, n, 2))
    for k in range(views):
        Y = X @ G[k, :3, :3].T + G[k, :3, 3]
        px[k, :, 0], px[k, :, 1] = f * Y[:, 0] / Y[:, 2] + cx, f * Y[:, 1] / Y[:, 2] + cy
    px += rng.normal(0.0, noise_px, px.shape)
    hidden = ~visible
    px[hidden, 0] = rng.uniform(0, W_REF, int(hidden.sum()))
    px[hidden, 1] = rng.uniform(0, H_REF, int(hidden.sum()))
    px = px.astype(np.float32)
    pairs = np.concatenate([px[:-1], px[1:]], axis=2)
    return {"px_views": px, "px_pairs": pairs, "G": G, "X": X, "visible": visible, "baselines": baselines}


def planar_pair(n: int, outlier_frac: float = 0.3, noise_px: float = 0.5, seed: int = 7):
    """Correspondences of a planar scene (points on a slanted plane seen by the same two
    cameras as synthetic_pair): image 2 = H(image 1) + noise, plus uniform outliers.
    Returns dict: px (n,4) float32, H (3,3) pixel-space ground-truth homography (h8 = 1), is_outlier."""
    rng = np.random.Generator(np.random.PCG64(seed))
    f, cx, cy = F_REF, W_REF / 2.0, H_REF / 2.0
    K = np.array([[f, 0, cx], [0, f, cy], [0, 0, 1.0]])
    R = _rot([0.1, 1.0, 0.05], -10.0)
    t = np.array([1.0, 0.05, 0.1])
    t = t / np.linalg.norm(t)
    nrm = np.array([0.15, -0.1, 1.0])
    nrm = nrm / np.linalg.norm(nrm)
    d = 6.0                                               # plane n.X = d in camera-1 frame
    Hm = K @ (R + np.outer(t, nrm) / d) @ np.linalg.inv(K)
    Hm = Hm / Hm[2, 2]
    pts = []
    while sum(len(p) for p in pts) < n:
        u = rng.uniform(0, W_REF, 4 * n)
        v = rng.uniform(0, H_REF, 4 * n)
        q = Hm @ np.stack([u, v, np.ones_like(u)])
        u2, v2 = q[0] / q[2], q[1] / q[2]
        ok = (u2 >= 0) & (u2 < W_REF) & (v2 >= 0) & (v2 < H_REF)
        pts.append(np.stack([u, v, u2, v2], 1)[ok])
    px = np.concatenate(pts)[:n]
    px[:, 2:] += rng.normal(0.0, noise_px, (n, 2))
    is_out = rng.random(n) < outlier_frac
    k = int(is_out.sum())
    px[is_out, 2] = rng.uniform(0, W_REF, k)
    px[is_out, 3] = rng.uniform(0, H_REF, k)
    return {"px": px.astype(np.float32), "H": Hm, "is_outlier": is_out}
