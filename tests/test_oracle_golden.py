"""Pins the CPU oracle against every golden vector the reference holds for the hot path
(SURVEY.md §4: G1, G2, G4) and against the stored outputs of the reference's own src/km.cpp compiled verbatim
(oracle/_ref/libkm_ref.so, tests/golden/reference_golden.npz), plus independent numpy/scipy cross-checks."""
import json
import math
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

import reference_golden as rg  # noqa: E402
from golden_vectors import G1_W, G2_CD, G2_PAIRS  # noqa: E402


def backends(orc):
    return ["port", "ref"] if orc.ref_km_lib() is not None else ["port"]


def test_g1_km_known_answer(orc, scratch_cwd):
    for be in backends(orc):
        m = orc.km_solve(G1_W, 0.01, be)
        assert list(m) == [0, 2, 1]
        assert -sum(G1_W[m[y], y] for y in range(3)) == 12.0


def test_g2_workflow_figure(orc, scratch_cwd):
    G = orc.km_graph(G2_CD, 30.0)
    assert G.shape == (7, 7)
    for be in backends(orc):
        m = orc.km_solve(G, 0.01, be)
        SP, TP, SPo, TPo, e = orc.km_output(G, 7, 6, 30.0, m)
        assert list(zip(SP.tolist(), TP.tolist())) == [(0, 0), (1, 1), (6, 2), (4, 3), (2, 4)]
        assert sorted(SPo.tolist()) == [3, 5] and TPo.tolist() == [5]
        assert e == 106.0


def test_golden_fixture_file_matches(orc, scratch_cwd):
    with open(os.path.join(GOLD, "km_golden.json")) as f:
        gold = json.load(f)
    for case in gold["cases"]:
        W = np.array(case["W"], dtype=np.float64)
        m = orc.km_solve(W, case["eps"], "port")
        assert m.tolist() == case["match"], case["name"]


KM_CASES = [(8, 0), (40, 1), (150, 2), (300, 3)]


def km_case(orc, n, seed):
    rng = np.random.default_rng(seed)
    return orc.km_graph(rng.random((n, n - n // 5)) * 60.0, 25.0)


@pytest.mark.parametrize("n,seed", KM_CASES)
def test_port_equals_reference_km_bitwise(orc, scratch_cwd, n, seed):
    a = orc.km_solve(km_case(orc, n, seed), 0.01, "port")
    assert np.array_equal(a, rg.load(rg.key("km", n, seed))["match"])


@pytest.mark.parametrize("n,seed", [(30, 5), (120, 6)])
def test_km_within_n_eps_of_optimum(orc, scratch_cwd, n, seed):
    from scipy.optimize import linear_sum_assignment
    rng = np.random.default_rng(seed)
    CD = rng.random((n, n)) * 50.0
    G = orc.km_graph(CD, 20.0)
    m = orc.km_solve(G, 0.01, "port")
    ours = sum(G[m[y], y] for y in range(n))
    r, c = linear_sum_assignment(-G)
    opt = G[r, c].sum()
    assert ours <= opt + 1e-9 and ours >= opt - n * 0.01


def test_constants_g4(orc):
    """Energyfunction::init / ctor constants (include/ghicp_reg.h:32-40, 80-81, 98)."""
    sc = np.float32(0.005 * np.float32(220.0))
    o = orc.Oracle(orc.FT_NONE, orc.CT_NN, bbx_magnitude=220.0)
    S = np.array([[0.0, 0, 0], [1, 0, 0], [0, 2, 0]])
    T = np.array([[0.0, 0, 0.5], [1, 0, 0.5], [0, 2, 0.5]])
    o.set_keypoints(S, T)
    st = o.iterate()
    assert st.iteration == 0
    # CD = scale * dist; penalty = max(CDmean, 1.0) (src/ghicp_reg.cpp:239)
    d = np.linalg.norm(S[:, None, :] - T[None, :, :], axis=2)
    assert np.allclose(o.cd(), float(sc) * d, rtol=0, atol=1e-12)
    assert st.penalty == max(st.cd_mean, 1.0)
    assert st.cor == 3 and st.converged == 1 and st.warn_few_pairs == 1  # cor < min_cor = 10
    assert st.para1 == pytest.approx(1.0 + np.float32(0.1)) or st.para1 == pytest.approx(1.0 - np.float32(0.1)) or st.para1 == 1.0


def test_hamming_matches_numpy(orc):
    rng = np.random.default_rng(0)
    a = rng.integers(0, 256, 56, dtype=np.uint8)
    b = rng.integers(0, 256, 56, dtype=np.uint8)
    L = orc.lib()
    assert L.orc_hamming(a.ctypes.data, b.ctypes.data, 56) == int(np.unpackbits(a ^ b).sum())


def test_fpfh_distance_is_abs_pearson(orc):
    rng = np.random.default_rng(1)
    a = (rng.random(33) * 100).astype(np.float32)
    b = (rng.random(33) * 100).astype(np.float32)
    d = orc.lib().orc_fpfh_distance(a.ctypes.data, b.ctypes.data)
    ref = abs(np.corrcoef(a.astype(np.float64), b.astype(np.float64))[0, 1])
    assert abs(d - ref) < 1e-5


def kabsch(S, T):
    ms, mt = S.mean(0), T.mean(0)
    H = (T - mt).T @ (S - ms)
    U, _, Vt = np.linalg.svd(H)
    D = np.diag([1, 1, np.sign(np.linalg.det(U) * np.linalg.det(Vt))])
    R = U @ D @ Vt
    return R, mt - R @ ms


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("n,planar", [(3, False), (50, False), (5000, False), (400, True)])
def test_rigid_fit_against_numpy_kabsch(orc, mode, n, planar):
    from ghicp_b200.synth import rot_xyz_deg, rot_angle
    rng = np.random.default_rng(n)
    S = rng.random((n, 3)) * [100, 100, 0.0 if planar else 20]
    R = rot_xyz_deg(2.0, -1.0, 4.0)
    t = np.array([0.5, -0.25, 0.1])
    T = S @ R.T + t + rng.normal(0, 0.01, (n, 3))
    Rt = orc.rigid_fit(S, T, mode)
    Rk, tk = kabsch(S, T)
    assert rot_angle(Rt[:3, :3], Rk) < 1e-5          # float32 solve vs float64 Kabsch
    assert np.linalg.norm(Rt[:3, 3] - tk) < 2e-3 if mode == 0 else np.linalg.norm(Rt[:3, 3] - tk) < 5e-4
    assert abs(np.linalg.det(Rt[:3, :3]) - 1) < 1e-5


def test_rigid_fit_reflection_case(orc):
    """Coplanar, noisy points whose unconstrained optimum is a reflection: S(2) = -1 branch of Umeyama."""
    rng = np.random.default_rng(3)
    S = rng.random((30, 3)) * [10, 10, 0.0]
    T = S.copy()
    T[:, 2] = rng.normal(0, 1e-3, 30)
    T[:, 0] *= 1.0
    Rt = orc.rigid_fit(S, T, 0)
    assert np.linalg.det(Rt[:3, :3]) > 0.999


def test_loop_converges_to_ground_truth(orc):
    from ghicp_b200 import synth
    sc = synth.config1(400, 400, seed=11)
    o = orc.Oracle(orc.FT_NONE, orc.CT_NN, bbx_magnitude=sc.bbx_magnitude, max_iter=60)
    o.set_keypoints(sc.S, sc.T)
    Rt, it, rc = o.run()
    assert rc == 0 and it < 60
    assert synth.rot_angle(Rt[:3, :3], sc.R_gt) < 2e-3
    assert np.linalg.norm(Rt[:3, 3] - sc.t_gt) < 0.5  # plain ICP with 10 % outliers: near, not exact


# ---- loop-level fixtures (tests/golden/loop_golden.npz, generated by tests/golden/make_loop_golden.py) --------------
LOOP_CASES = ["none_nn", "none_nnr", "bsc_nn", "bsc_nnr", "bsc_km", "bsc_nn_dof4", "fpfh_nn", "fpfh_nnr"]


def load_loop_case(name):
    z = np.load(os.path.join(GOLD, "loop_golden.npz"))
    pre = name + "/"
    return {k[len(pre):]: z[k] for k in z.files if k.startswith(pre)}


@pytest.mark.parametrize("name", LOOP_CASES)
def test_oracle_reproduces_loop_fixture(orc, scratch_cwd, name):
    """Guards the oracle against drift: the committed loops (inputs, per-iteration pair lists, transforms) replay."""
    c = load_loop_case(name)
    ft, ct, dof, max_it, n_it = (int(v) for v in c["meta"])
    o = orc.Oracle(ft, ct, dof=dof, bbx_magnitude=float(c["bbx"]), solve_mode=1, max_iter=max_it,
                   use_ref_km=(ct == orc.CT_KM and orc.ref_km_lib() is not None))
    o.set_keypoints(c["S"], c["T"])
    if "bsc_s" in c:
        o.set_bsc(c["bsc_s"], c["bsc_t"], 441)
    if "fpfh_s" in c:
        o.set_fpfh(c["fpfh_s"], c["fpfh_t"])
    o.build_fd()
    for it in range(n_it):
        st = o.iterate()
        sp, tp = o.pairs()
        b, e = c["off"][it], c["off"][it + 1]
        assert np.array_equal(sp, c["sp"][b:e]) and np.array_equal(tp, c["tp"][b:e]), (name, it)
        assert np.allclose(np.array(st.Rt), c["Rt"][it], atol=1e-12)
        assert st.penalty == pytest.approx(float(c["penalty"][it]), rel=1e-12)
    assert st.converged == 1
    assert np.allclose(np.array(st.Rt_tillnow), c["Rt_final"], atol=1e-12)


# ---- the reference's own per-pair feature-distance code (oracle/_ref/libfeat_ref.so) and its committed outputs ---------------
def load_feat_golden():
    return np.load(os.path.join(GOLD, "feat_golden.npz"))


@pytest.mark.parametrize("bits", [441, 672, 9, 64, 2048])
def test_oracle_fd_bsc_equals_reference_hamming_fixture(orc, bits):
    """calFD_BSC (src/ghicp_reg.cpp:143-200) of the oracle == min over variants of the Hamming distances the REFERENCE's own
    StereoBinaryFeature::hammingDistance produced (fixture generated by tests/golden/make_feat_golden.py)."""
    z = load_feat_golden()
    S, T, H = z[f"bsc{bits}/S"], z[f"bsc{bits}/T"], z[f"bsc{bits}/H"]
    _, V, N, M = (int(v) for v in z[f"bsc{bits}/meta"])
    for i in range(N):
        for j in range(M):
            for v in range(V):
                assert orc.hamming(S[v, i], T[j]) == H[v, i, j]
    for dof, nv in ((6, min(V, 4)), (4, 2)):
        if V < (4 if dof == 6 else 2):
            continue
        o = orc.Oracle(orc.FT_BSC, orc.CT_NN, dof=dof, bbx_magnitude=10.0)
        o.set_keypoints(np.zeros((N, 3)), np.zeros((M, 3)))
        o.set_bsc(S, T, bits)
        o.build_fd()
        assert np.array_equal(o.fd(), H[:nv].min(axis=0).astype(np.float64))


def test_oracle_fd_fpfh_equals_reference_fixture(orc):
    z = load_feat_golden()
    fs, ft, D = z["fpfh/S"], z["fpfh/T"], z["fpfh/D"]
    o = orc.Oracle(orc.FT_FPFH, orc.CT_NN, bbx_magnitude=10.0)
    o.set_keypoints(np.zeros((len(fs), 3)), np.zeros((len(ft), 3)))
    o.set_fpfh(fs, ft)
    o.build_fd()
    assert np.array_equal(o.fd().astype(np.float32), D, equal_nan=True)     # bit-identical floats, NaN where the reference gives 0/0
    assert np.isnan(D[:, 12]).all() and D[10, 11] == pytest.approx(1.0, abs=1e-6)


FEATURE_BITS = (441, 672, 13)


def feature_code_inputs():
    """Random descriptor pairs, bit sets and FPFH histogram pairs (fixed seed) the reference's feature code was run on."""
    rng = np.random.default_rng(5)
    d = {}
    for bits in FEATURE_BITS:
        B = (bits + 7) // 8
        d[f"pairs{bits}"] = [(rng.integers(0, 256, B, dtype=np.uint8), rng.integers(0, 256, B, dtype=np.uint8)) for _ in range(50)]
        d[f"bits{bits}"] = rng.random(bits) < 0.4
    d["fpfh"] = [((rng.gamma(0.6, 1.0, 33) * 20).astype(np.float32), (rng.gamma(0.6, 1.0, 33) * 20).astype(np.float32))
                 for _ in range(200)]
    return d


def test_reference_feature_code_live(orc):
    """The oracle against the stored outputs of the reference's own functions (StereoBinaryFeature::hammingDistance,
    setNthBitValue / getNthBitValue, compute_fpfh_distance) on random inputs, and the descriptor bit layout (setNthBitValue:
    bit k -> byte k/8, bit k%8) the synthetic generator assumes."""
    import ghicp_b200 as g
    ref = rg.load("feat")
    x = feature_code_inputs()
    for bits in FEATURE_BITS:
        assert [orc.hamming(a, b) for a, b in x[f"pairs{bits}"]] == ref[f"hamming{bits}"].tolist()
        bits01 = x[f"bits{bits}"]
        assert np.array_equal(ref[f"set_bits{bits}"], g.synth.pack_bits(bits01))
        assert np.array_equal(ref[f"get_bit{bits}"], bits01.astype(np.int32))
    a = np.array([orc.fpfh_distance(h1, h2) for h1, h2 in x["fpfh"]], np.float32)
    assert np.array_equal(a, ref["fpfh_distance"])
