"""The oracle against the REFERENCE's own GHRegistration (src/ghicp_reg.cpp + km.cpp + stereo_binary_feature.cpp compiled
VERBATIM into oracle/_ref/libghreg_ref.so; Eigen / PCL / VTK replaced by declaration-level stubs, the PCL SVD call delegated
to the oracle — see oracle/ghreg_ref_shim.cpp).  What that build computed on these seeded scenes is stored in
tests/golden/reference_golden.npz (tests/golden/make_reference_golden.py); the planes and keypoint sets as digests.

Everything compared here is produced by the reference's own statements: calED, calFD_BSC / calFD_FPFH, calCD_NF / calCD_BSC /
calCD_FPFH with the penalty rules, findcorrespondenceNN / NNR / KM, the pair statistics, the update of the keypoints, the
Euler-angle convergence test, adjustweight and the accumulated transform — and the oracle must agree BIT FOR BIT.  In KM mode
the oracle runs its restatement of src/km.cpp, which tests/test_oracle_golden.py pins to the reference's bit for bit."""
import numpy as np
import pytest

import ghicp_b200 as g
import reference_golden as rg

CASES = [("none", "nn", 6), ("none", "nnr", 6), ("none", "km", 6), ("bsc", "nn", 6), ("bsc", "nnr", 6), ("bsc", "km", 6),
         ("bsc", "nn", 4), ("bsc", "km", 4), ("fpfh", "nn", 6), ("fpfh", "nnr", 6), ("fpfh", "km", 6)]


MAX_ITER = 40
RUN_CASES = [("none", "nn"), ("bsc", "nnr"), ("fpfh", "nn")]


def FT(orc, ft):
    return {"none": orc.FT_NONE, "bsc": orc.FT_BSC, "fpfh": orc.FT_FPFH}[ft]


def CT(orc, ct):
    return {"nn": orc.CT_NN, "nnr": orc.CT_NNR, "km": orc.CT_KM}[ct]


def set_inputs(o, sc, ft):
    if ft == "bsc":
        o.set_bsc(sc.bsc_s, sc.bsc_t, sc.bits)
    if ft == "fpfh":
        o.set_fpfh(sc.fpfh_s, sc.fpfh_t)


def build(orc, cls, sc, ft, ct, dof, **kw):
    o = cls(FT(orc, ft), CT(orc, ct), dof=dof, bbx_magnitude=sc.bbx_magnitude, solve_mode=0, **kw)
    o.set_keypoints(sc.S, sc.T)
    set_inputs(o, sc, ft)
    o.build_fd()
    return o


def with_features(sc, ft):
    if ft == "bsc":
        g.synth.add_bsc(sc, bits=441, V=4)
    if ft == "fpfh":
        g.synth.add_fpfh(sc)
    return sc


def loop_scene(ft, ct):
    N, M = (90, 100) if ct == "km" else (230, 250)
    return with_features(g.synth.gen_points(N, M, overlap=0.7, extent=(50, 50, 10), noise=0.03, seed=7 + N), ft)


def run_scene(ft):
    return with_features(g.synth.gen_points(200, 210, overlap=0.7, extent=(50, 50, 10), noise=0.03, seed=3), ft)


@pytest.mark.parametrize("ft,ct,dof", CASES)
def test_oracle_equals_reference_loop_bit_for_bit(orc, scratch_cwd, ft, ct, dof):
    ref = rg.load(rg.key("loop", ft, ct, dof))
    sc = loop_scene(ft, ct)
    orac = build(orc, orc.Oracle, sc, ft, ct, dof)
    if ft != "none":
        assert np.array_equal(rg.digest(orac.fd()), ref["fd"])                           # calFD_* (:143-214)
    n_it = len(ref["converged"])
    for it in range(n_it):
        b = orac.iterate()
        assert np.array_equal(rg.digest(orac.cd()), ref["cd"][it]), it                   # calED + calCD_* (:114-341)
        assert b.penalty == ref["penalty"][it] and b.cor == ref["cor"][it], it
        osp, otp = orac.pairs()
        # the target points of this iteration's pairs, before the update (Tpoint: :446-452, 664-675, 735-746)
        assert np.array_equal(rg.digest(np.asarray(sc.T)[otp]), ref["rt"][it]), it
        assert b.rmse == ref["rmse"][it] and b.fdm == ref["fdm"][it] and b.fdstd == ref["fdstd"][it], it   # :549-578, 676-766
        assert np.array_equal(np.array(b.Rt), ref["Rt"][it]), it                            # glue around the (delegated) SVD
        assert b.rmse_after == ref["rmse_after"][it] and b.iou == ref["iou"][it], it         # :889-907, 799
        assert b.para1 == ref["para1"][it] and b.para2 == ref["para2"][it], it               # adjustweight :771-789
        assert np.array_equal(np.array(b.Rt_tillnow), ref["Rt_tillnow"][it]), it            # :93
        assert np.array_equal(rg.digest(orac.source()), ref["source"][it]), it               # update of KP.kpSXYZ :891-894
        if ct == "km":
            assert b.km_energy == ref["energy"][it], it                                      # Km::Calenergy via the loop (:442-443)
        assert b.converged == ref["converged"][it], it                                       # :796-797, 909-914
    assert b.converged == 1


@pytest.mark.parametrize("ft,ct", RUN_CASES)
def test_reference_ghicp_reg_function_equals_stepped_loop(orc, scratch_cwd, ft, ct):
    """GHRegistration::ghicp_reg itself (src/ghicp_reg.cpp:24-112), start to finish, against the oracle's run()."""
    ref = rg.load(rg.key("run", ft, ct))
    sc = run_scene(ft)
    o = orc.Oracle(FT(orc, ft), CT(orc, ct), bbx_magnitude=sc.bbx_magnitude, solve_mode=0)
    o.set_keypoints(sc.S, sc.T)
    set_inputs(o, sc, ft)
    Ro, ito, rc = o.run()          # calFD_* + the whole while loop, like the reference's own function
    assert rc == 0 and ito == ref["iterations"]
    assert np.array_equal(Ro, ref["Rt"])
