"""BSC descriptor encoder (SURVEY.md §8f row N2) without a GPU:
  * the oracle restatement (oracle/ghicp_bsc_oracle.cpp) against the outputs of the reference's own header compiled
    verbatim (oracle/_ref/libbsc_ref.so), stored in tests/golden/reference_golden.npz and tests/golden/bsc_golden.npz;
  * structural properties of the reference's descriptor (bit layout, the re-arranged variants' quirk, rigid invariance);
  * the product's kernel (k_bsc in gh-icp_b200/csrc/ghicp_prep.cu) run on the CPU through the host emulation shim, against
    the oracle.  TOLERANCE: the kernel holds exact sums where the reference accumulates in float32 in KD-tree order
    (covariance, depth sums), so a comparison closer to its threshold than float32 accumulation error may fall the other way:
    at least 98 % of the descriptors must be bit-identical and the mean Hamming distance at most 0.05 bits of 441
    (measured on these scenes: 100 % and 0)."""
import ctypes as C
import os

import numpy as np
import pytest

import reference_golden as rg
from test_prep_oracle import scan_like_cloud

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "bsc_golden.npz")


def hamming(a, b):
    return np.unpackbits(a ^ b, axis=-1).sum(axis=-1)


def bits01(feat, nbits=441):
    return np.unpackbits(feat, axis=-1, bitorder="little")[..., :nbits]


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.fixture(scope="module")
def emu(emu_harness_path):
    L = C.CDLL(emu_harness_path)
    L.emu_bsc_extract.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                  C.c_void_p, C.c_void_p]
    return L


def emu_extract(emu, xyz, kp, radius, pairs, side=7, dof=6):
    xyz = np.ascontiguousarray(xyz, np.float32); kp = np.ascontiguousarray(kp, np.int32); pairs = np.ascontiguousarray(pairs, np.int32)
    V = 4 if dof > 4 else (2 if dof > 0 else 1)
    nb = (9 * side * side + 7) // 8
    bits = np.full((V, len(kp), nb), 0xAA, np.uint8); lrf = np.zeros((len(kp), 12), np.float32); st = np.full(len(kp), -1, np.int32)
    rc = emu.emu_bsc_extract(xyz.ctypes.data, len(xyz), kp.ctypes.data, len(kp), radius, side, pairs.ctypes.data, dof,
                             bits.ctypes.data, lrf.ctypes.data, st.ctypes.data)
    assert rc == 0
    return bits, lrf, st


# ---- the oracle is the reference ------------------------------------------------------------------------------------------
def test_oracle_reproduces_the_golden_vectors_of_the_reference_build(orc, gold):
    bits, lrf, status = orc.bsc_extract(gold["xyz"], gold["kp"], float(gold["radius"]), gold["pairs"], 7, 6)
    assert status.sum() == 0
    assert np.array_equal(bits, gold["bits"])
    assert np.array_equal(lrf, gold["lrf"])
    for dof, V in ((0, 1), (3, 2)):
        b, _, _ = orc.bsc_extract(gold["xyz"], gold["kp"], float(gold["radius"]), gold["pairs"], 7, dof)
        assert b.shape[0] == V and np.array_equal(b, gold["bits"][:V])


FRESH_CASES = [(3000, 40, 1.0, 1), (5000, 30, 0.6, 2), (1500, 25, 2.0, 3)]


def fresh_scene(n, nkp, seed):
    xyz = scan_like_cloud(n, seed, extent=(10.0, 10.0, 4.0))
    return xyz, np.random.default_rng(seed).choice(n, nkp, replace=False).astype(np.int32)


@pytest.mark.parametrize("n,nkp,radius,seed", FRESH_CASES)
def test_oracle_equals_the_reference_build_on_fresh_scenes(orc, gold, n, nkp, radius, seed):
    ref = rg.load(rg.key("bsc_fresh", n, nkp, radius, seed))
    xyz, kp = fresh_scene(n, nkp, seed)
    for dof in (0, 4, 6):
        bits, lrf, _ = orc.bsc_extract(xyz, kp, radius, gold["pairs"], 7, dof)
        assert np.array_equal(rg.digest(bits), ref[f"dof{dof}/bits"])
        assert np.array_equal(rg.digest(lrf), ref[f"dof{dof}/lrf"])


def test_shipped_pattern_is_what_the_reference_constructor_generates(orc, scratch_cwd, gold):
    """ghicp_bsc_default_pattern (compiled into the library; no GPU needed to read it) = glibc rand() from the default seed
    through the reference's own constructor = the golden file's pattern."""
    import ghicp_b200 as g
    shipped = g.capi.bsc_default_pattern(7)
    assert np.array_equal(shipped, gold["pairs"])
    assert shipped.shape == (49, 2) and shipped.min() >= 0 and shipped.max() < 49
    assert all(a != b for a, b in shipped.tolist())
    assert len({(min(a, b), max(a, b)) for a, b in shipped.tolist()}) == 49       # contain2DPair: no repeated pair
    if orc.ref_bsc_lib() is not None:
        assert np.array_equal(orc.ref_bsc_pattern(7), shipped)
        with open("sample_pattern.txt") as f:                                      # the side effect a reference user sees
            assert np.array_equal(np.loadtxt(f, dtype=np.int32).reshape(-1, 2), shipped)
        assert np.array_equal(g.capi.read_sample_pattern("sample_pattern.txt"), shipped)


# ---- what the descriptor is -----------------------------------------------------------------------------------------------
def test_descriptor_layout_and_the_rearranged_variants_quirk(orc, gold):
    """Variant 0: 147 occupancy bits then 3 x 49 x (depth bit, density bit).  Variants 1-3 (ReArrangeGrid appends to a
    pre-sized vector): nothing but the occupancy bits of the re-arranged grid, at bit offset 147."""
    b = bits01(gold["bits"])
    occ0 = b[0][:, :147]
    num, dep, npw = orc.bsc_grid(gold["xyz"], int(gold["kp"][0]), float(gold["radius"]), 7)
    assert np.array_equal(occ0[0], (npw > np.float32(0.1)).astype(np.uint8))
    assert b[0][:, 147:].sum() > 0
    for v in (1, 2, 3):
        assert b[v][:, :147].sum() == 0 and b[v][:, 294:].sum() == 0
        assert np.array_equal(b[v][:, 147:294].sum(axis=1), occ0.sum(axis=1))     # a permutation of the same cells
    k = np.arange(49)
    i, j = k // 7, k % 7
    rev_all, sym2, sym1 = 48 - k, (6 - i) * 7 + j, i * 7 + 6 - j
    plan = {1: (rev_all, sym2, sym2), 2: (sym1, sym2, rev_all), 3: (sym2, rev_all, sym1)}   # :789, :804, :813
    for v, maps in plan.items():
        for pl in range(3):
            assert np.array_equal(b[v][:, 147 + 49 * pl:147 + 49 * (pl + 1)], occ0[:, 49 * pl:49 * (pl + 1)][:, maps[pl]])


def test_grid_weights_are_gaussian_sums_of_the_projected_neighbours(orc, gold):
    """Independent numpy formulation of one cell row: sum over the neighbours within 1.5 cells of exp(-d^2 / 2 delta^2)."""
    xyz, p, R = gold["xyz"].astype(np.float64), int(gold["kp"][3]), float(gold["radius"])
    num, dep, npw = orc.bsc_grid(gold["xyz"], p, R, 7)
    _, lrf, _ = orc.bsc_extract(gold["xyz"], gold["kp"][3:4], R, gold["pairs"], 7, 0)
    ax, ay, az = lrf[0, 0:3].astype(np.float64), lrf[0, 3:6].astype(np.float64), lrf[0, 6:9].astype(np.float64)
    d = xyz - xyz[p]
    nb = d[(d ** 2).sum(axis=1) < 3.0 * R * R]
    loc = np.stack([nb @ ax, nb @ ay, nb @ az], axis=1)          # orthonormal frame: the inverse is the transpose
    unit = 2 * R / 7
    delta = unit / 2
    centres = (np.arange(7) + 0.5) * unit - R
    for pl, (u, v, w) in enumerate([(0, 1, 2), (0, 2, 1), (1, 2, 0)]):
        for i in range(7):
            for j in range(7):
                dd = (loc[:, u] - centres[i]) ** 2 + (loc[:, v] - centres[j]) ** 2
                m = dd < (1.5 * unit) ** 2
                wgt = np.exp(-dd[m] / (2 * delta * delta))
                assert num[i + 7 * j + 49 * pl] == pytest.approx(wgt.sum(), rel=2e-4, abs=2e-4)
                if wgt.sum() > 1e-3:
                    assert dep[i + 7 * j + 49 * pl] == pytest.approx(((loc[m, w] + R) * wgt).sum() / wgt.sum(), rel=5e-4, abs=5e-4)
    area = np.pi * R * R
    assert np.allclose(npw, (num / unit ** 2) / (len(nb) / area), rtol=1e-4, atol=1e-6)


def test_descriptor_is_invariant_to_a_rigid_motion_of_the_cloud_up_to_the_frame_sign(orc, gold):
    """The local frame turns with the cloud, so the descriptor of a keypoint barely changes — except that an eigenvector's
    sign is a convention (the reference's variants exist for that): compare modulo the sign flips that keep a right-handed
    frame, on the occupancy bits the variants carry."""
    import ghicp_b200 as g
    xyz, kp, R = gold["xyz"], gold["kp"], float(gold["radius"])
    Rm = g.synth.rot_xyz_deg(20.0, -35.0, 50.0)
    moved = (xyz.astype(np.float64) @ Rm.T + [3.0, -2.0, 1.0]).astype(np.float32)
    a, _, _ = orc.bsc_extract(xyz, kp, R, gold["pairs"], 7, 6)
    b, _, _ = orc.bsc_extract(moved, kp, R, gold["pairs"], 7, 6)
    A, B = bits01(a), bits01(b)
    occ = lambda X, v: X[v][:, :147] if v == 0 else X[v][:, 147:294]
    best = np.min([np.abs(occ(A, 0).astype(int) - occ(B, v).astype(int)).sum(axis=1) for v in range(4)], axis=0)
    other = np.abs(occ(A, 0).astype(int) - np.roll(occ(B, 0), 7, axis=0).astype(int)).sum(axis=1)   # a different keypoint
    assert np.median(best) <= 6 and np.median(other) >= 3 * max(np.median(best), 1)


def test_keypoints_with_fewer_than_three_neighbours_are_flagged(orc, gold):
    xyz = np.concatenate([gold["xyz"], np.array([[500.0, 500.0, 500.0], [500.1, 500.0, 500.0]], np.float32)])
    kp = np.array([len(xyz) - 1, int(gold["kp"][0])], np.int32)
    bits, lrf, status = orc.bsc_extract(xyz, kp, float(gold["radius"]), gold["pairs"], 7, 6)
    assert status.tolist() == [1, 0]
    assert bits[:, 0].sum() == 0 and bits[0, 1].sum() > 0


# ---- the product's kernel, emulated --------------------------------------------------------------------------------------
def check_against_oracle(got, want, what):
    h = hamming(got, want)
    identical = float((h == 0).mean())
    assert identical >= 0.98 and h.mean() <= 0.05, f"{what}: {identical:.4f} identical, mean Hamming {h.mean():.4f}, max {h.max()}"
    return identical, h


@pytest.mark.parametrize("dof", [0, 4, 6])
def test_emulated_kernel_reproduces_the_golden_vectors(emu, gold, dof):
    V = 4 if dof > 4 else (2 if dof > 0 else 1)
    bits, lrf, st = emu_extract(emu, gold["xyz"], gold["kp"], float(gold["radius"]), gold["pairs"], 7, dof)
    assert (st == 0).all()
    check_against_oracle(bits, gold["bits"][:V], f"dof {dof}")
    assert np.abs(lrf - gold["lrf"]).max() < 2e-5


@pytest.mark.parametrize("n,nkp,radius,side,seed", [(3000, 40, 1.0, 7, 1), (6000, 24, 0.5, 7, 2), (1500, 25, 2.0, 7, 3),
                                                    (2500, 20, 1.2, 5, 4), (2500, 16, 1.2, 9, 5)])
def test_emulated_kernel_equals_oracle(orc, emu, gold, n, nkp, radius, side, seed):
    xyz = scan_like_cloud(n, seed, extent=(10.0, 10.0, 4.0))
    rng = np.random.default_rng(seed)
    kp = rng.choice(n, nkp, replace=False).astype(np.int32)
    if side == 7:
        pairs = gold["pairs"]
    else:                                             # other grid sizes: any valid pattern
        pairs = np.stack([rng.permutation(side * side), np.roll(rng.permutation(side * side), 1)], axis=1).astype(np.int32)
        pairs[pairs[:, 0] == pairs[:, 1], 1] = (pairs[pairs[:, 0] == pairs[:, 1], 1] + 1) % (side * side)
    want, wlrf, wst = orc.bsc_extract(xyz, kp, radius, pairs, side, 6)
    got, lrf, st = emu_extract(emu, xyz, kp, radius, pairs, side, 6)
    assert np.array_equal(st, wst)
    check_against_oracle(got, want, f"n {n} side {side}")
    assert np.abs(lrf - wlrf).max() < 5e-5


def test_emulated_kernel_flags_isolated_keypoints_and_handles_cloud_borders(orc, emu, gold):
    """Keypoints on the bounding box (neighbour cells outside the grid) and an isolated pair of points."""
    xyz = np.concatenate([gold["xyz"], np.array([[500.0, 500.0, 500.0], [500.1, 500.0, 500.0]], np.float32)])
    lo, hi = int(np.argmin(xyz[:-2].sum(axis=1))), int(np.argmax(xyz[:-2].sum(axis=1)))
    kp = np.array([len(xyz) - 1, lo, hi, int(np.argmin(xyz[:-2, 0])), int(gold["kp"][0])], np.int32)
    want, wlrf, wst = orc.bsc_extract(xyz, kp, float(gold["radius"]), gold["pairs"], 7, 6)
    got, lrf, st = emu_extract(emu, xyz, kp, float(gold["radius"]), gold["pairs"], 7, 6)
    assert st.tolist() == wst.tolist() == [1, 0, 0, 0, 0]
    assert got[:, 0].sum() == 0
    check_against_oracle(got[:, 1:], want[:, 1:], "border keypoints")


# ---- randomised and degenerate geometry: the restatement against the reference build ------------------------------------
def _degenerate_clouds():
    rng = np.random.default_rng(99)
    base = (rng.random((300, 3)) * [4.0, 4.0, 2.0]).astype(np.float32)
    plane = base.copy(); plane[:, 2] = 1.0                                     # exactly planar: smallest eigenvalue 0
    line = base.copy(); line[:, 1] = 2.0; line[:, 2] = 1.0                      # collinear: two zero eigenvalues
    dup = np.repeat(base[:60], 5, axis=0)                                      # every point five times
    lattice = np.stack(np.meshgrid(np.arange(8), np.arange(8), np.arange(4), indexing="ij"), -1).reshape(-1, 3).astype(np.float32) * 0.5
    tiny = (base * 1e-3).astype(np.float32)                                    # millimetre scale
    far = (base + np.float32(5000.0)).astype(np.float32)                       # large coordinates: float32 cancellation
    return {"plane": plane, "line": line, "duplicates": dup, "lattice": lattice, "tiny": tiny, "far": far}


def degenerate_case(name, xyz):
    """(radius, keypoints) of the degenerate cloud `name`."""
    return {"tiny": 1e-3, "lattice": 0.9}.get(name, 1.0), np.arange(0, len(xyz), max(1, len(xyz) // 24), dtype=np.int32)


@pytest.mark.parametrize("name", ["plane", "line", "duplicates", "lattice", "tiny", "far"])
def test_oracle_equals_the_reference_build_on_degenerate_geometry(orc, gold, name):
    """Zero and repeated eigenvalues, coincident points, symmetric lattices (masses of exactly equal distances: the tie order of
    the neighbour search matters), very small and very large coordinates."""
    ref = rg.load(rg.key("bsc_degenerate", name))
    xyz = _degenerate_clouds()[name]
    radius, kp = degenerate_case(name, xyz)
    for dof in (0, 6):
        bits, lrf, status = orc.bsc_extract(xyz, kp, radius, gold["pairs"], 7, dof)
        assert status.sum() == 0
        assert np.array_equal(rg.digest(bits), ref[f"dof{dof}/bits"]), name
        assert np.array_equal(rg.digest(lrf), ref[f"dof{dof}/lrf"]), name                 # NaN equal to NaN


RANDOM_CASES = 40
RANDOM_KINDS = ["uniform", "clustered", "layered"]


def random_scene(seed, n, kind):
    rng = np.random.default_rng(seed)
    P = rng.random((n, 3)) * [5.0, 5.0, 2.0]
    if RANDOM_KINDS[kind] == "clustered":
        P = P[rng.integers(0, max(3, n // 20), n)] + 0.05 * rng.standard_normal((n, 3))
    elif RANDOM_KINDS[kind] == "layered":
        P[:, 2] = np.round(P[:, 2] * 2) / 2
    return P.astype(np.float32), rng.choice(n, min(n, 12), replace=False).astype(np.int32)


def test_oracle_equals_the_reference_build_randomised(orc, gold):
    """40 random small clouds (uniform, clustered or layered), radii, keypoints and dof types, drawn once from a fixed seed
    (the parameters are stored with the reference's outputs)."""
    params = rg.load("bsc_random")["params"]
    assert len(params) == RANDOM_CASES
    for i, (seed, n, kind, radius, dof) in enumerate(params):
        ref = rg.load(rg.key("bsc_random", i))
        xyz, kp = random_scene(int(seed), int(n), int(kind))
        bits, lrf, status = orc.bsc_extract(xyz, kp, float(radius), gold["pairs"], 7, int(dof))
        ok = status == 0                      # < 3 neighbours: the reference reads uninitialised axes; not comparable
        assert np.array_equal(bits[:, ok], ref[f"dof{int(dof)}/bits"][:, ok]), i
        assert np.array_equal(lrf[ok], ref[f"dof{int(dof)}/lrf"][ok], equal_nan=True), i


@pytest.mark.parametrize("name", ["line", "duplicates", "tiny", "far", "plane"])
def test_emulated_kernel_on_degenerate_geometry(orc, emu, gold, name):
    """Collinear / coincident points and extreme coordinate scales meet the usual bar.  On an EXACTLY planar cloud the depth
    of every cell is the same number up to rounding noise, so the depth-comparison bits (`|d - mean| > sigma` on differences
    that are mathematically zero) are decided by the accumulation order in the reference itself: only the other bits —
    occupancy, density comparisons, all variants — are comparable, and must be identical.  (A perfectly symmetric lattice has
    repeated eigenvalues: its frame is arbitrary in the reference too, and is not compared.)"""
    xyz = _degenerate_clouds()[name]
    radius = 1e-3 if name == "tiny" else 1.0
    kp = np.arange(0, len(xyz), max(1, len(xyz) // 24), dtype=np.int32)
    want, wlrf, wst = orc.bsc_extract(xyz, kp, radius, gold["pairs"], 7, 6)
    got, lrf, st = emu_extract(emu, xyz, kp, radius, gold["pairs"], 7, 6)
    assert np.array_equal(st, wst)
    if name != "plane":
        check_against_oracle(got, want, name)
        return
    A, B = bits01(want), bits01(got)
    depth_bits = np.zeros(441, bool)
    depth_bits[147::2] = True                          # 147 + 98 pl + 2 i
    assert np.array_equal(A[:, :, ~depth_bits], B[:, :, ~depth_bits])
    assert np.abs(lrf - wlrf).max() < 1e-5
