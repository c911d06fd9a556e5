"""CPU checks of the pre-processing oracle (oracle/ghicp_prep_oracle.cpp: voxel filter, radius PCA, keypoint pruning +
non-maximum suppression) against independent numpy formulations, and of the product's pre-processing KERNELS run on the
CPU through the host emulation shim (tests/harness) against that oracle — bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import reference_golden as rg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
fp, ip, dp = C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_double)


def scan_like_cloud(n, seed, extent=(20.0, 20.0, 5.0)):
    """A crude 'scan': a ground plane, two walls, a box edge and clutter (float32 like PCL points)."""
    rng = np.random.default_rng(seed)
    P = rng.random((n, 3)) * np.asarray(extent)
    q = n // 8
    P[:3 * q, 2] = 0.02 * rng.standard_normal(3 * q)                        # ground
    P[3 * q:5 * q, 0] = extent[0] * 0.5 + 0.02 * rng.standard_normal(2 * q)  # wall x = const
    P[5 * q:6 * q, 1] = extent[1] * 0.25 + 0.02 * rng.standard_normal(q)     # wall y = const
    P[6 * q:7 * q, 0] = 3.0 + 0.01 * rng.standard_normal(q)                  # a pole-like edge
    P[6 * q:7 * q, 1] = 4.0 + 0.01 * rng.standard_normal(q)
    return P.astype(np.float32)


# ---- oracle vs independent numpy ---------------------------------------------------------------------------------------
def test_voxel_filter_one_point_per_voxel_smallest_index_plus_phantom(orc):
    P = scan_like_cloud(6000, 1)
    v = np.float32(0.4)
    idx = orc.voxel_downsample(P, float(v))
    inv = np.float32(1.0) / v
    mn = P.min(axis=0)
    vox = np.floor((P - mn) * inv).astype(np.int64)                       # float32 arithmetic like include/filter.hpp:56-58
    gap = P.max(axis=0) - mn
    my, mz = int(np.ceil(gap[1] * inv) + 1), int(np.ceil(gap[2] * inv) + 1)
    key = vox[:, 0] * (my * mz) + vox[:, 1] * mz + vox[:, 2]
    assert idx[0] == 0                                                    # the reference's phantom voxel-0 entry
    rest = idx[1:]
    uk, first = np.unique(key, return_index=True)                         # np.unique: first occurrence = smallest index
    keep = uk != 0
    assert np.array_equal(rest, first[keep].astype(np.int32))             # ascending voxel id, smallest index per voxel
    assert np.all(np.diff(key[rest]) > 0)


VOXEL_CASES = [(6000, 0.4, 1), (20000, 0.1, 2), (500, 5.0, 3), (3000, 0.02, 4)]
KEYPOINT_CASES = [(4000, 1.0, 1.5, 8), (1500, 0.6, 0.6, 9), (600, 3.0, 0.3, 10), (6000, 0.8, 1.0, 12)]


@pytest.mark.parametrize("n,voxel,seed", VOXEL_CASES)
def test_voxel_filter_against_the_reference_build(orc, n, voxel, seed):
    """The REFERENCE's own CFilter::voxelfilter (include/filter.hpp compiled verbatim; its outputs are stored): same number of
    output points, the phantom point 0 first, the same voxel at every output position.  WHICH point of a voxel is kept is
    implementation-defined there (an unstable std::sort on the voxel id alone, :71); the oracle / CUDA path keep the smallest
    index."""
    P = scan_like_cloud(n, seed)
    ref = P[rg.load("voxel")[rg.key(n, voxel, seed)]]          # stored as the rows of P the reference kept
    mine = P[orc.voxel_downsample(P, voxel)]
    assert len(ref) == len(mine)
    assert np.array_equal(ref[0], P[0]) and np.array_equal(mine[0], P[0])
    inv = np.float32(1.0) / np.float32(voxel)
    mn = P.min(axis=0)
    vr, vm = np.floor((ref - mn) * inv), np.floor((mine - mn) * inv)
    assert np.array_equal(vr[1:], vm[1:])                      # same voxel, position by position (position 0 is the phantom)


@pytest.mark.parametrize("n,radius,nms,seed", KEYPOINT_CASES)
def test_keypoint_detection_against_the_reference_build(orc, n, radius, nms, seed):
    """The REFERENCE's own keypointDetectionBasedOnCurvature (keypoint_detect.hpp + pca.h compiled verbatim: its PCA driver,
    pruneUnstablePoints, the curvature sort and the std::set based greedy suppression; KD-tree / PCA numerics from the
    stand-ins; its outputs are stored): normally the same number of keypoints with the same curvature at every output
    position, indices differing only between points of EXACTLY equal curvature that suppress each other — the reference
    orders such ties through an unstable std::sort (:151), the oracle / CUDA path by index."""
    P = scan_like_cloud(n, seed)
    ref = rg.load("keypoints")[rg.key(n, radius, nms, seed)]
    kp, lam, curv, cnt = orc.detect_keypoints(P, radius, 0.65, 20, nms)
    assert len(kp) > 0
    if np.array_equal(curv[ref], curv[kp]):
        for a, b in zip(ref, kp):          # index differences: exact-tie twins only
            if a != b:
                assert curv[a] == curv[b] and np.linalg.norm(P[a].astype(np.float64) - P[b].astype(np.float64)) < nms
    else:
        # the stand-in PCA sums the neighbours in KD-tree (distance) order, the oracle in grid order: the double sums differ in
        # the last bit now and then, which can move a point across the 0.65 ratio threshold or swap two near-equal curvatures
        # (seen with the 3.0 m neighbourhoods of several hundred points).  The two keypoint sets must still nearly coincide.
        inter = len(set(ref.tolist()) & set(kp.tolist()))
        assert abs(len(ref) - len(kp)) <= max(2, len(kp) // 50)
        assert inter >= 0.9 * max(len(ref), len(kp))


def test_pca_eigenvalues_and_counts_match_numpy(orc):
    P = scan_like_cloud(3000, 2)
    r = 0.9
    lam, curv, cnt = orc.pca_curvature(P, r)
    Pd = P.astype(np.float64)
    rng = np.random.default_rng(0)
    for i in rng.integers(0, len(P), 60):
        d = P - P[i]                                                       # float32 differences, like the KD-tree's metric
        d2 = d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2]
        nb = np.nonzero(d2 < np.float32(r) * np.float32(r))[0]
        assert cnt[i] == len(nb)
        if len(nb) >= 3:
            w = np.linalg.eigvalsh(np.cov(Pd[nb].T))[::-1]
            assert np.allclose(lam[i], w, rtol=2e-4, atol=2e-6)
            assert curv[i] == pytest.approx(w[2] / w.sum(), rel=2e-3, abs=2e-6)


def test_keypoints_satisfy_the_greedy_nms_definition(orc):
    P = scan_like_cloud(5000, 3)
    kp, lam, curv, cnt = orc.detect_keypoints(P, 1.0, 0.65, 20, 1.5)
    assert len(kp) > 10
    with np.errstate(invalid="ignore", divide="ignore"):
        ok = (lam[:, 1] / lam[:, 0] < 0.65) & (lam[:, 2] / lam[:, 1] < 0.65) & (cnt > 20)
    assert ok[kp].all()
    assert np.all(np.diff(curv[kp]) <= 0)                                  # emitted best first
    K = P[kp].astype(np.float64)
    D = np.linalg.norm(K[:, None] - K[None], axis=2) + 10 * np.eye(len(kp))
    assert D.min() >= 1.5 - 1e-5                                           # no two keypoints within the NMS radius
    cand = np.nonzero(ok)[0]
    rest = np.setdiff1d(cand, kp)
    for i in rest[:300]:                                                   # every rejected candidate lost to a better keypoint
        d = np.linalg.norm(P[kp].astype(np.float64) - P[i].astype(np.float64), axis=1)
        near = kp[d < 1.5 + 1e-6]
        assert len(near) and curv[near].max() >= curv[i]


# ---- product kernels on the CPU (emulation) vs the oracle: bit for bit -----------------------------------------------------
@pytest.fixture(scope="module")
def emu(emu_harness_path):
    L = C.CDLL(emu_harness_path)
    L.emu_voxel_downsample.argtypes = [fp, C.c_int, C.c_float, ip, ip]
    L.emu_detect_keypoints.argtypes = [fp, C.c_int, C.c_float, C.c_float, C.c_int, C.c_float, ip, ip, fp, dp, ip, ip]
    return L


@pytest.mark.parametrize("n,voxel,seed", [(5000, 0.4, 4), (777, 0.05, 5), (1, 1.0, 6), (300, 50.0, 7)])
def test_emulated_voxel_filter_equals_oracle(orc, emu, n, voxel, seed):
    P = scan_like_cloud(max(n, 8), seed)[:n]
    out, m = np.zeros(n + 1, np.int32), C.c_int(0)
    assert emu.emu_voxel_downsample(P.ctypes.data_as(fp), n, voxel, out.ctypes.data_as(ip), C.byref(m)) == 0
    assert np.array_equal(out[:m.value], orc.voxel_downsample(P, voxel))


@pytest.mark.parametrize("n,radius,nms,seed", [(4000, 1.0, 1.5, 8), (1500, 0.6, 0.6, 9), (600, 3.0, 0.3, 10)])
def test_emulated_keypoint_detection_equals_oracle(orc, emu, n, radius, nms, seed):
    P = scan_like_cloud(n, seed)
    kp, m, rounds = np.zeros(n, np.int32), C.c_int(0), C.c_int(0)
    lam, curv, cnt = np.zeros((n, 3), np.float32), np.zeros(n), np.zeros(n, np.int32)
    rc = emu.emu_detect_keypoints(P.ctypes.data_as(fp), n, radius, 0.65, 20, nms, kp.ctypes.data_as(ip), C.byref(m),
                                  lam.ctypes.data_as(fp), curv.ctypes.data_as(dp), cnt.ctypes.data_as(ip), C.byref(rounds))
    assert rc == 0
    okp, olam, ocurv, ocnt = orc.detect_keypoints(P, radius, 0.65, 20, nms)
    assert np.array_equal(cnt, ocnt)
    assert np.array_equal(lam, olam) and np.array_equal(curv, ocurv)      # same sums, same Jacobi: identical bits
    assert np.array_equal(kp[:m.value], okp)
    assert 1 <= rounds.value <= 64


def test_emulated_pipeline_downsample_then_keypoints(orc, emu):
    P = scan_like_cloud(20000, 11)
    out, m = np.zeros(len(P) + 1, np.int32), C.c_int(0)
    emu.emu_voxel_downsample(P.ctypes.data_as(fp), len(P), 0.3, out.ctypes.data_as(ip), C.byref(m))
    D = np.ascontiguousarray(P[out[:m.value]])
    n = len(D)
    kp, k, rounds = np.zeros(n, np.int32), C.c_int(0), C.c_int(0)
    lam, curv, cnt = np.zeros((n, 3), np.float32), np.zeros(n), np.zeros(n, np.int32)
    emu.emu_detect_keypoints(D.ctypes.data_as(fp), n, 1.0, 0.65, 20, 1.5, kp.ctypes.data_as(ip), C.byref(k),
                             lam.ctypes.data_as(fp), curv.ctypes.data_as(dp), cnt.ctypes.data_as(ip), C.byref(rounds))
    okp, _, _, _ = orc.detect_keypoints(D, 1.0, 0.65, 20, 1.5)
    assert np.array_equal(kp[:k.value], okp) and len(okp) > 20
