"""KM-mode OUTPUT-TRANSFORM parity (BASELINE.json north_star: <= 1e-4 rad / <= 1e-3 m against the reference CPU path).

The CUDA path (eps-scaled auction) and the REFERENCE's own GHRegistration (src/ghicp_reg.cpp + src/km.cpp compiled verbatim,
oracle/_ref/libghreg_ref.so; its final transforms and iteration counts on these scenes are stored in
tests/golden/reference_golden.npz) are both run FREE from iteration 0 to convergence on the same seeded scene: nothing
re-synchronises the two trajectories.  eps-optimal matchings are not unique (the reference's depends on DFS order, ours on
bid order), so the pair lists may differ in weak pairs; what the test pins is what north_star pins: the accumulated
transform.  Measured gap (emulated ABI vs the reference build, 300-500 keypoints): <= 1e-7 rad, <= 2e-5 m.
Also: a stand-alone 4000 x 4000 KM instance against the exact optimum (scipy) — the benchmark's regime, 4x the largest
instance of tests/test_gpu_parity.py."""
import numpy as np
import pytest

import reference_golden as rg

pytestmark = pytest.mark.gpu

ROT_TOL = 1e-4    # rad   (BASELINE.json north_star)
TRANS_TOL = 1e-3  # m
MAX_ITER = 80
CASES = [
    (300, 300, 5, 6, 0.6, 0.03),
    (420, 360, 6, 6, 0.6, 0.03),
    (500, 500, 7, 4, 0.6, 0.03),
    (640, 700, 8, 6, 0.5, 0.05),
    (1000, 1000, 9, 6, 0.6, 0.05),
    (1500, 1300, 10, 4, 0.7, 0.04),
    (2000, 2000, 11, 6, 0.6, 0.05),
]


def scene(g, N, M, seed, overlap, noise):
    f = (max(N, M) / 300.0) ** (1.0 / 3.0)
    return g.synth.add_bsc(g.synth.gen_points(N, M, overlap=overlap, extent=(40 * f, 40 * f, 8 * f), noise=noise, seed=seed),
                           bits=441, V=4)


def free_run(r, sc):
    """The reference's loop (oracle.Reference) from iteration 0 to convergence: (accumulated transform, iterations)."""
    r.set_keypoints(sc.S, sc.T)
    r.set_bsc(sc.bsc_s, sc.bsc_t, sc.bits)
    r.build_fd()
    Rt = np.eye(4)
    its = 0
    for _ in range(MAX_ITER):
        st = r.iterate()
        its += 1
        Rt = np.array(st.Rt).reshape(4, 4).T @ Rt        # Rt_tillnow = Rt_temp * Rt_tillnow (src/ghicp_reg.cpp:93)
        if st.converged:
            break
    return Rt, its


@pytest.mark.parametrize("N,M,seed,dof,overlap,noise", CASES)
def test_km_free_running_final_transform(g, scratch_cwd, N, M, seed, dof, overlap, noise):
    ref = rg.load(rg.key("freerun", N, M, seed, dof))
    sc = scene(g, N, M, seed, overlap, noise)
    reg = g.registration.from_scene(sc, g.FT_BSC, g.CT_KM, dof=dof, max_iter=MAX_ITER)
    its = 0
    for _ in range(MAX_ITER):
        a = reg.iterate()
        its += 1
        if a.converged:
            break
    Rt = reg.Rt_tillnow()
    Rt_ref, its_ref = ref["Rt"], int(ref["iterations"])
    ang = g.synth.rot_angle(Rt[:3, :3], Rt_ref[:3, :3])
    dt = float(np.linalg.norm(Rt[:3, 3] - Rt_ref[:3, 3]))
    print(f"KM free run {N}x{M} dof {dof}: {its} / {its_ref} iterations (ours / reference), gap {ang:.2e} rad {dt:.2e} m")
    assert its == its_ref
    assert ang <= ROT_TOL and dt <= TRANS_TOL, (ang, dt)
    assert g.synth.rot_angle(Rt[:3, :3], sc.R_gt) < 5e-3       # and the registration itself succeeded


def test_km_4000_objective_against_exact_optimum(g, orc):
    """Stand-alone KM at 4000 x 4000 on a config-2-like cost (integer Hamming part + metric part, ~2 % candidate edges):
    total energy within n*KM_eps of the exact optimum (scipy's Jonker-Volgenant), matching valid."""
    from scipy.optimize import linear_sum_assignment
    n = 4000
    rng = np.random.default_rng(40)
    CD = rng.integers(150, 230, size=(n, n)).astype(np.float64) * 0.8 + rng.random((n, n)) * 12.0
    perm = rng.permutation(n)
    CD[np.arange(n), perm] -= rng.random(n) * 90.0                 # true matches stand out, like the BSC ground truth
    pen = float(np.quantile(CD, 0.02))
    G = orc.km_graph(CD, pen)
    match, energy, rounds = g.km_solve(G, sp=n, tp=n, eps=0.01, penalty=pen)
    used = [x for x in match if x >= 0]
    assert len(used) == len(set(used))
    for y, x in enumerate(match):
        if x >= 0:
            assert CD[x, y] < pen
    r, c = linear_sum_assignment(-G)
    e_opt = -G[r, c].sum()
    print(f"KM 4000: energy {energy:.3f}, optimum {e_opt:.3f}, gap {energy - e_opt:.3f} (bound {n * 0.01}), rounds {rounds}")
    assert e_opt - 1e-6 <= energy <= e_opt + n * 0.01
