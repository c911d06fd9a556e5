"""Regenerates tests/golden/reference_golden.npz: what the reference's own code (oracle/_ref, built by oracle/Makefile from
the reference's sources) returns on the inputs of the parity tests that compare the oracle or the product with it.  The
inputs are not stored: every test rebuilds them from the same seeds (see tests/reference_golden.py).

    python tests/golden/make_reference_golden.py        # needs oracle/_ref, i.e. the reference's sources at build time
"""
import ctypes as C
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ghicp_b200 as g  # noqa: E402  (only its seeded synthetic generator is used here)
import oracle  # noqa: E402
import reference_golden as rg  # noqa: E402
import test_bsc_encoder as tb  # noqa: E402
import test_gpu_km_freerun as tf  # noqa: E402
import test_oracle_golden as to  # noqa: E402
import test_prep_oracle as tp  # noqa: E402
import test_reference_loop as tl  # noqa: E402

out = {}
K = rg.key


def bsc(prefix, xyz, kp, radius, dofs, store=lambda a: a):
    for dof in dofs:
        bits, lrf = oracle.ref_bsc_extract(xyz, kp, radius, pairs, 7, dof)
        out[K(prefix, f"dof{dof}", "bits")], out[K(prefix, f"dof{dof}", "lrf")] = store(bits), store(lrf)


def rows_of(P, Q):
    """Index into P of every row of Q (Q's rows are rows of P)."""
    first = {}
    for i, r in enumerate(map(bytes, P)):
        first.setdefault(r, i)
    idx = np.array([first[bytes(r)] for r in Q])
    assert len(P) <= 65536 and np.array_equal(P[idx], Q)
    return idx.astype(np.uint16)


def loop_reference(sc, ft, ct, dof):
    ref = tl.build(oracle, oracle.Reference, sc, ft, ct, dof)
    rows = {f: [] for f in ("cd", "penalty", "cor", "rt", "rmse", "fdm", "fdstd", "Rt", "rmse_after", "iou", "para1", "para2",
                            "Rt_tillnow", "source", "energy", "converged")}
    for _ in range(tl.MAX_ITER):
        a = ref.iterate()
        rows["cd"].append(rg.digest(ref.cd()))
        rows["rt"].append(rg.digest(ref.pairs_xyz()[1]))
        rows["source"].append(rg.digest(ref.source()))
        for f in ("penalty", "cor", "rmse", "fdm", "fdstd", "rmse_after", "iou", "para1", "para2", "energy", "converged"):
            rows[f].append(getattr(a, f))
        rows["Rt"].append(np.array(a.Rt)); rows["Rt_tillnow"].append(np.array(a.Rt_tillnow))
        if a.converged:
            break
    d = {f: np.array(v) for f, v in rows.items()}
    d["fd"] = rg.digest(ref.fd()) if ft != "none" else np.zeros(0, np.uint8)
    return d


def main():
    global pairs
    assert oracle.ref_ghreg_lib() is not None and oracle.ref_bsc_lib() is not None, "oracle/_ref not built"
    os.chdir(tempfile.mkdtemp())                    # the reference writes Corres.txt and ./sample_pattern.txt
    pairs = oracle.ref_bsc_pattern(7)
    assert np.array_equal(pairs, g.capi.bsc_default_pattern(7))

    for n, nkp, radius, seed in tb.FRESH_CASES:
        xyz, kp = tb.fresh_scene(n, nkp, seed)
        bsc(K("bsc_fresh", n, nkp, radius, seed), xyz, kp, radius, (0, 4, 6), rg.digest)
    for name, xyz in tb._degenerate_clouds().items():
        radius, kp = tb.degenerate_case(name, xyz)
        bsc(K("bsc_degenerate", name), xyz, kp, radius, (0, 6), rg.digest)
    rng = np.random.default_rng(2024)               # the cases of test_oracle_equals_the_reference_build_randomised
    params = np.array([[rng.integers(0, 2 ** 31 - 1), rng.integers(30, 501), rng.integers(0, 3), rng.uniform(0.2, 3.0),
                        rng.choice([0, 2, 4, 6])] for _ in range(tb.RANDOM_CASES)])
    out["bsc_random/params"] = params
    for i, (seed, n, kind, radius, dof) in enumerate(params):
        xyz, kp = tb.random_scene(int(seed), int(n), int(kind))
        bsc(K("bsc_random", i), xyz, kp, float(radius), (int(dof),))

    for n, seed in to.KM_CASES:
        out[K("km", n, seed, "match")] = oracle.km_solve(to.km_case(oracle, n, seed), 0.01, "ref")
    R = oracle.ref_feat_lib()
    x = to.feature_code_inputs()
    for bits in to.FEATURE_BITS:
        out[K("feat", f"hamming{bits}")] = np.array([R.featref_hamming(a.ctypes.data, b.ctypes.data, bits)
                                                     for a, b in x[f"pairs{bits}"]], np.int32)
        pos = np.nonzero(x[f"bits{bits}"])[0].astype(np.int32)
        packed = np.zeros((bits + 7) // 8, np.uint8)
        R.featref_set_bits(bits, pos.ctypes.data_as(C.POINTER(C.c_int)), len(pos), packed.ctypes.data)
        out[K("feat", f"set_bits{bits}")] = packed
        out[K("feat", f"get_bit{bits}")] = np.array([R.featref_get_bit(packed.ctypes.data, bits, k) for k in range(bits)], np.int32)
    out[K("feat", "fpfh_distance")] = np.array([R.featref_fpfh_distance(h1.ctypes.data, h2.ctypes.data) for h1, h2 in x["fpfh"]],
                                               np.float32)

    for n, voxel, seed in tp.VOXEL_CASES:            # the filter keeps input points: stored as their rows in the input
        P = tp.scan_like_cloud(n, seed)
        out[K("voxel", n, voxel, seed)] = rows_of(P, oracle.ref_voxelfilter(P, voxel))
    for n, radius, nms, seed in tp.KEYPOINT_CASES:
        out[K("keypoints", n, radius, nms, seed)] = oracle.ref_detect_keypoints(tp.scan_like_cloud(n, seed), radius, 0.65, 20, nms)

    for ft, ct, dof in tl.CASES:
        for f, v in loop_reference(tl.loop_scene(ft, ct), ft, ct, dof).items():
            out[K("loop", ft, ct, dof, f)] = v
    for ft, ct in tl.RUN_CASES:
        sc = tl.run_scene(ft)
        ref = oracle.Reference(tl.FT(oracle, ft), tl.CT(oracle, ct), bbx_magnitude=sc.bbx_magnitude, solve_mode=0)
        ref.set_keypoints(sc.S, sc.T)
        tl.set_inputs(ref, sc, ft)
        out[K("run", ft, ct, "Rt")], out[K("run", ft, ct, "iterations")] = ref.run()

    for N, M, seed, dof, overlap, noise in tf.CASES:
        sc = tf.scene(g, N, M, seed, overlap, noise)
        r = oracle.Reference(oracle.FT_BSC, oracle.CT_KM, dof=dof, bbx_magnitude=sc.bbx_magnitude, solve_mode=0)
        Rt, its = tf.free_run(r, sc)
        out[K("freerun", N, M, seed, dof, "Rt")], out[K("freerun", N, M, seed, dof, "iterations")] = Rt, its

    np.savez_compressed(rg.PATH, **out)
    print(f"wrote {rg.PATH}: {len(out)} arrays, {os.path.getsize(rg.PATH)} bytes")


if __name__ == "__main__":
    main()
