"""CPU tier: host logic of the product (C-ABI surface, host small-matrix code,
sharding) - no compute calls that need a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
fp = C.POINTER(C.c_float)


def P(a):
    return a.ctypes.data_as(fp)


def _declared_symbols():
    names = set()
    for hdr in ("sfmb200.h", "sfmb200_la.h"):
        text = open(os.path.join(ROOT, "include", hdr)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names |= set(re.findall(r"\b(sfmb200_\w+)\s*\(", text))
    return names


def test_library_exports_every_declared_symbol(lib, pkg):
    declared = _declared_symbols()
    assert len(declared) > 45
    for name in declared:
        assert hasattr(lib.cdll, name), f"{name} declared in include/ but not exported"
    # and the ctypes table binds exactly the declared surface
    from cuda_sfm_b200.binding import SIGNATURES

    assert set(SIGNATURES) == declared


def test_missing_library_fails_loudly(pkg):
    from cuda_sfm_b200.binding import Lib

    with pytest.raises(FileNotFoundError, match="no CPU fallback"):
        Lib("/nonexistent/libsfmb200.so")


def test_create_without_gpu_is_an_error_not_a_fallback(pkg, O):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    K, Kinv = O.reference_K()
    with pytest.raises(pkg.SfmError) as e:
        pkg.BatchedPairs(K, Kinv, 1, 100, 100)
    assert e.value.code == -4 and "no CPU fallback" in str(e.value)


def test_host_sample_indices_match_oracle(lib, O):
    out = np.zeros(8, np.int32)
    for seed, h, n in ((1237, 0, 10000), (1237, 65535, 10000), (2**63 + 5, 123456789, 1 << 20), (0, 3, 8)):
        lib.raw("sfmb200_host_sample_indices")(C.c_uint64(seed), C.c_uint64(h), n, out.ctypes.data_as(C.POINTER(C.c_int32)))
        assert list(out) == O.sample_indices_one(seed, h, n)


@pytest.mark.parametrize("entry_point", ["sfmb200_host_solve_hypothesis", "sfmb200_host_solve_hypothesis_projector"])
def test_host_hypothesis_solver_matches_fp64_oracle(lib, O, scene_small, entry_point):
    """Both null-vector solvers (9x9 Jacobi eigensolve, 8x8 Cholesky projector)."""
    x = scene_small["x"]
    H = 1500
    idx = O.sample_indices(1237, H, len(x))
    E64 = O.hypotheses(x, idx)
    E32 = np.zeros((H, 9), np.float32)
    solve = lib.raw(entry_point)
    for h in range(H):
        p = np.ascontiguousarray(x[idx[h]], dtype=np.float32)
        solve(P(p), P(E32[h]))
    d = O.e_distance(E32, E64)
    # north_star tolerance: 1e-4 relative Frobenius up to sign/scale.  The
    # remainder are samples whose design matrix has condition number > 1e5.
    assert np.mean(d < 1e-4) >= 0.995, np.mean(d < 1e-4)
    assert np.median(d) < 1e-6
    assert np.allclose(np.linalg.norm(E32, axis=1), np.sqrt(2), atol=1e-4)


def test_host_hypothesis_degenerate_sample_is_zero(lib):
    # eight identical points (dyadic, so the centroid is exact): Hartley scale is
    # 1/0 -> non-finite -> the solver must return the all-zero matrix (count 0)
    p = np.tile(np.array([[0.5, 0.25, 0.125, 0.75]], np.float32), (8, 1))
    for name in ("sfmb200_host_solve_hypothesis", "sfmb200_host_solve_hypothesis_projector"):
        E = np.ones(9, np.float32)
        lib.raw(name)(P(p), P(E))
        assert np.all(E == 0)
    E = np.ones(9, np.float32)
    # rank-deficient but finite samples stay finite (never NaN into the scorer)
    p = np.tile(np.array([[0.1, 0.2, 0.3, 0.4]], np.float32), (8, 1))
    p[:, 0] += np.arange(8, dtype=np.float32) * 1e-3
    lib.raw("sfmb200_host_solve_hypothesis")(P(p), P(E))
    assert np.all(np.isfinite(E))


def test_host_svd3_contract(lib):
    rng = np.random.default_rng(0)
    f = lib.raw("sfmb200_host_svd3")
    for k in range(500):
        a = rng.normal(size=9).astype(np.float32)
        if k % 5 == 0:      # rank deficient like an essential matrix
            A = a.reshape(3, 3).astype(np.float64)
            U, S, Vt = np.linalg.svd(A)
            a = (U @ np.diag([S[0], S[1], 0]) @ Vt).astype(np.float32).reshape(9)
        u, s, v = (np.zeros(9, np.float32) for _ in range(3))
        f(P(a), P(u), P(s), P(v))
        A, U, S, V = (m.reshape(3, 3).astype(np.float64) for m in (a, u, s, v))
        assert np.abs(U @ S @ V.T - A).max() < 5e-6 * max(1, np.abs(A).max())
        assert abs(np.linalg.det(U) - 1) < 1e-5 and abs(np.linalg.det(V) - 1) < 1e-5
        assert S[0, 0] >= S[1, 1] >= abs(S[2, 2]) - 1e-6
        assert np.abs(S - np.diag(np.diag(S))).max() < 5e-6 * max(1, np.abs(A).max())
        sv = np.linalg.svd(A, compute_uv=False)
        assert np.abs(np.abs(np.diag(S)) - sv).max() < 5e-6 * max(1, sv[0])


def test_host_svd3_agrees_with_reference_host_svd(lib, ref_lib):
    """Same contract => same U V^T and same rank-2 projection as svd.h's svd()."""
    rng = np.random.default_rng(3)
    for _ in range(200):
        a = rng.normal(size=9).astype(np.float32)
        u, s, v = (np.zeros(9, np.float32) for _ in range(3))
        ur, sr, vr = (np.zeros(9, np.float32) for _ in range(3))
        lib.raw("sfmb200_host_svd3")(P(a), P(u), P(s), P(v))
        ref_lib.ref_host_svd(P(a), P(ur), P(sr), P(vr))
        sv = np.abs(np.diag(s.reshape(3, 3)))
        if sv[1] + sv[2] < 0.5 or sv[1] - sv[2] < 0.1:
            continue
        U, V, Ur, Vr = (m.reshape(3, 3) for m in (u, v, ur, vr))
        assert np.abs(U @ V.T - Ur @ Vr.T).max() < 2e-2
        proj = U[:, :2] @ V[:, :2].T
        projr = Ur[:, :2] @ Vr[:, :2].T
        assert np.abs(proj - projr).max() < 2e-2


def test_host_null4_and_inv4(lib):
    rng = np.random.default_rng(4)
    for _ in range(300):
        A = rng.normal(size=(4, 4)).astype(np.float32)
        x = np.zeros(4, np.float32)
        lib.raw("sfmb200_host_null4")(P(A), P(x))
        v = np.linalg.svd(A.astype(np.float64))[2][-1]
        s = np.linalg.svd(A.astype(np.float64), compute_uv=False)
        if s[2] - s[3] > 0.05:
            assert min(np.linalg.norm(v - x), np.linalg.norm(v + x)) < 1e-4
        inv = np.zeros(16, np.float32)
        assert lib.raw("sfmb200_host_inv4")(P(A), P(inv)) == 0
        assert np.abs(inv.reshape(4, 4) @ A - np.eye(4)).max() < 1e-2 * np.linalg.cond(A) / 10
    Z = np.zeros(16, np.float32)
    assert lib.raw("sfmb200_host_inv4")(P(Z), P(np.zeros(16, np.float32))) != 0


def test_host_null4_fast_path_matches_jacobi_on_dlt_matrices(lib, O):
    """Triangulation's inverse-iteration solve vs the Jacobi solve vs fp64, on real
    DLT matrices (inliers and outliers, true and inverted pose)."""
    K, Kinv = O.reference_K()
    sc = O.synthetic_pair(1500, seed=5, noise_px=2.0)
    x = O.normalise_points(sc["px"], Kinv)
    M = np.eye(4)
    M[:3, :3], M[:3, 3] = sc["R"], sc["t"]
    for MM in (M, np.linalg.inv(M)):
        A = O.dlt_rows(x, MM).astype(np.float32)
        ref = O.triangulate(x, MM)
        fast = np.zeros((len(x), 4), np.float32)
        fails = 0
        for i in range(len(x)):
            f = lib.raw("sfmb200_host_null4_fast")(P(A[i]), P(fast[i]))
            fails += f
            if f:
                lib.raw("sfmb200_host_null4")(P(A[i]), P(fast[i]))
        X = fast[:, :3] / fast[:, 3:4]
        rel = np.abs(X.T - ref[:3]).max(0) / np.maximum(np.abs(ref[:3]).max(0), 1e-3)
        assert fails <= 2                       # the fallback exists for pathological geometry only
        assert np.median(rel) < 1e-6 and np.percentile(rel, 99) < 1e-4 and rel.max() < 5e-3
    # a matrix with a repeated smallest singular value must report non-convergence or a valid null vector
    A = np.diag([1.0, 1.0, 1e-3, 1e-3]).astype(np.float32)
    v = np.zeros(4, np.float32)
    f = lib.raw("sfmb200_host_null4_fast")(P(A), P(v))
    assert f == 1 or abs(np.linalg.norm(A @ v)) < 2e-3


def test_host_dlt_null_adjugate_matches_fp64_on_dlt_matrices(lib, O):
    """The triangulation kernel's solve (adjugate power iteration exploiting camera 1 = I4, smallmat.cuh) vs the
    fp64 SVD null vector on real DLT matrices: inliers and outliers, true and inverted pose."""
    K, Kinv = O.reference_K()
    sc = O.synthetic_pair(3000, seed=5, noise_px=2.0)
    x = O.normalise_points(sc["px"], Kinv)
    M = np.eye(4)
    M[:3, :3], M[:3, 3] = sc["R"], sc["t"]
    for MM in (M, np.linalg.inv(M)):
        A = O.dlt_rows(x, MM).astype(np.float32)
        ref = O.triangulate(x, MM)
        out = np.zeros((len(x), 4), np.float32)
        fails = 0
        for i in range(len(x)):
            f = lib.raw("sfmb200_host_dlt_null")(P(A[i]), P(out[i]))
            fails += f
            if f:
                lib.raw("sfmb200_host_null4")(P(A[i]), P(out[i]))
        X = out[:, :3] / out[:, 3:4]
        rel = np.abs(X.T - ref[:3]).max(0) / np.maximum(np.abs(ref[:3]).max(0), 1e-3)
        inl = ~sc["is_outlier"]
        assert fails <= 3                       # the fallback exists for pathological geometry only
        assert np.median(rel) < 1e-6 and np.percentile(rel[inl], 99) < 1e-5 and np.percentile(rel, 99) < 1e-4 and rel.max() < 5e-3
    # pixel-sized coordinates (K = I): no overflow in the cofactors
    A = O.dlt_rows(sc["px"], M).astype(np.float32)
    v = np.zeros(4, np.float32)
    ok = 0
    for i in range(200):
        f = lib.raw("sfmb200_host_dlt_null")(P(A[i]), P(v))
        assert np.all(np.isfinite(v))
        if not f:
            t = np.linalg.svd(A[i].astype(np.float64))[2][-1]
            ok += min(np.linalg.norm(t - v), np.linalg.norm(t + v)) < 1e-3
    assert ok >= 150


def test_disjoint_permutation_sampler_matches_oracle(lib, O):
    """SFMB200_OPT_SAMPLER = 1 (the reference's scheme, sfm.cu:95-104: one permutation cut into disjoint groups of 8):
    the device / host code and the oracle mirror agree bit for bit, rows are disjoint and cover distinct indices."""
    for n, seed in ((2153, 5), (8, 0), (17, 3), (65536, 99), (1000003, 7)):
        H = min(n // 8, 1500)
        want = O.sample_indices_disjoint(seed, H, n)
        got = np.zeros((H, 8), np.int32)
        for h in range(H):
            lib.raw("sfmb200_host_sample_indices_disjoint")(C.c_uint64(seed), C.c_uint64(h), n, got[h].ctypes.data_as(C.POINTER(C.c_int32)))
        assert np.array_equal(want, got)
        flat = want.reshape(-1)
        assert len(set(flat.tolist())) == len(flat) and flat.min() >= 0 and flat.max() < n
        # a slice regenerates without the rows before it
        assert np.array_equal(O.sample_indices_disjoint(seed, H - H // 2, n, h0=H // 2), want[H // 2:])
    # a full permutation when n is a multiple of 8
    full = O.sample_indices_disjoint(11, 64, 512).reshape(-1)
    assert sorted(full.tolist()) == list(range(512))


def test_shard_range_and_keys(pkg):
    sh = pkg.sharding
    for total in (0, 1, 7, 8, 65536, 1000003):
        for world in (1, 2, 3, 4, 8):
            spans = [sh.shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
    assert sh.unpack_key(sh.pack_key(7001, 123)) == (7001, 123)
    # higher count wins; on ties the lower index wins
    assert sh.pack_key(10, 500) > sh.pack_key(9, 0)
    assert sh.pack_key(10, 3) > sh.pack_key(10, 4)
    assert sh.pack_key(2**31 - 1, 0) < 2**63


def test_headers_are_plain_c_and_a_c_program_links(tmp_path):
    """The boundary is a C ABI: include/*.h compile as strict C99, and a C program that includes them links
    against the shared library with nothing but gcc (no CUDA headers, no C++)."""
    import shutil
    import subprocess

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    src = tmp_path / "abi.c"
    src.write_text(
        '#include <stdio.h>\n#include "sfmb200.h"\n#include "sfmb200_la.h"\n'
        "int main(void) {\n"
        "    float K[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};\n"
        "    sfmb200_t* h = NULL;\n"
        "    int rc = sfmb200_create(K, K, 1, 64, 64, &h);\n"
        '    printf("%d %d %s\\n", sfmb200_version(), rc, sfmb200_last_error());\n'
        "    if (rc == 0) sfmb200_destroy(h);\n"
        "    return 0;\n}\n")
    libdir = os.path.join(ROOT, "cuda-sfm_b200")
    exe = tmp_path / "abi"
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                        "-o", str(exe), "-L", libdir, "-lsfmb200", f"-Wl,-rpath,{libdir}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0, out.stderr
    ver, rc, *msg = out.stdout.split()
    assert int(ver) >= 100
    # without a GPU the create call must fail with the "no CUDA device" status, never fall back
    import torch
    if not torch.cuda.is_available():
        assert int(rc) != 0 and "no CUDA device" in out.stdout


def test_svd_h_facade_surface_host_and_device(tmp_path):
    """SfM/svd.h facade: every name of the reference's header (svd.h:33-501), including its six internal steps, is there
    with its meaning (tests/src/svd_surface_check.cpp asserts the maths on the host, g++), and all of it is
    __host__ __device__ like the reference's: the same file compiles as CUDA with a kernel that calls it (nvcc -c)."""
    import shutil
    import subprocess

    src = os.path.join(ROOT, "tests", "src", "svd_surface_check.cpp")
    inc = os.path.join(ROOT, "cuda-sfm_b200", "SfM")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    exe = tmp_path / "svdchk"
    r = subprocess.run(["g++", "-O1", "-std=c++17", f"-I{cuda}/include", f"-I{inc}", "-o", str(exe), src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "svd.h surface ok" in r.stdout, (r.returncode, r.stdout, r.stderr)
    nvcc = os.path.join(cuda, "bin", "nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    cu = tmp_path / "svdchk.cu"
    shutil.copy(src, cu)
    r = subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", f"-I{inc}", "-c", "-o", str(tmp_path / "svdchk.o"), str(cu)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]])
def test_bench_rejects_arguments_it_cannot_honour(args, tmp_path):
    """Checked before anything runs: no step count below 1, and --dump-outputs only for this project's path (the
    reference arm has nothing to dump, and an empty directory must not pass for a comparable run)."""
    import subprocess
    import sys

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=120, cwd=tmp_path)
    assert r.returncode == 2 and "error" in r.stderr and not r.stdout.strip()
    assert not (tmp_path / "unused").exists()
