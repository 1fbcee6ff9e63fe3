"""ORACLE (test infrastructure - never imported by the product).

numpy restatement of the level-0 part of the Levenberg-Marquardt driver CoarseTracker::trackNewestCoarse
(tandem/src/FullSystem/CoarseTracker.cpp:761-916) on top of a tracker object with the CudaCoarseTracker call surface
(calcRes / calcG).  SURVEY.md section 8(f) row n3 moves this loop onto the device (tdm_tracker_track); this file is what
the device loop is checked against.  PINNED (round 2): the reference driver as a whole needs Eigen + Sophus (absent here),
but its level loop (CoarseTracker.cpp:750-916) is cut out of the file where it lies by oracle/ref_build.mk and compiled,
unmodified, against a stand-in Eigen / SE3 (tests/cpp/eigen_stub, oracle/ref_wrap_lm.cpp) into oracle/_ref/liblm_ref.so;
tests/test_oracle_cpu.py::test_lm_driver_pinned_to_reference_trackNewestCoarse drives that loop and this restatement with the
SAME tracker object and requires the same number of evaluations (= the same accept / reject sequence, cutoff doublings, stop
iteration and level repeat) and the same pose / affine parameters, for free, fixed-a, fixed-b and fixed-a-b optimisation and
a saturating start; what that loop returned is stored in tests/golden/ref_lm.npz (oracle/ref_golden.py), so the test runs
without the reference.  The restatement follows
the listed lines statement by statement: cutoff doubling while the saturated ratio exceeds 0.6
(:779-790), lambda = 0.01 (:798), H diagonal *(1+lambda) and LDLT solve on the free parameters (:814-840), the
extrapolation factor (:843-845), SCALE_* (:847-851, cuda_coarse_tracker.cpp:12-19), left-multiplicative SE3 update
(:855), accept iff the mean energy drops (:868), lambda *0.5 / *4 with the extrapolation limit as floor (:887-900), stop
when |inc| <= 1e-3 (:903-907).
"""
import numpy as np

SCALE = np.array([1.0, 1.0, 1.0, 0.5, 0.5, 0.5, 10.0, 1000.0])   # SCALE_XI_ROT x3, SCALE_XI_TRANS x3, SCALE_A, SCALE_B


def hat(w):
    return np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]], np.float64)


def se3_exp(xi):
    """Sophus convention: xi = (upsilon, omega); returns the 4x4 matrix of exp(xi)."""
    xi = np.asarray(xi, np.float64)
    ups, om = xi[:3], xi[3:]
    th = np.linalg.norm(om)
    Om = hat(om)
    if th < 1e-8:
        A, B, C = 1.0 - th * th / 6, 0.5 - th * th / 24, 1.0 / 6 - th * th / 120
    else:
        A, B, C = np.sin(th) / th, (1 - np.cos(th)) / th ** 2, (th - np.sin(th)) / th ** 3
    R = np.eye(3) + A * Om + B * Om @ Om
    V = np.eye(3) + B * Om + C * Om @ Om
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = V @ ups
    return T


def track_level0(trk, refToNew, aff, new_exposure, coarse_cutoff=20.0, max_iterations=10,
                 lambda_extrapolation_limit=0.001, fix_a=False, fix_b=False):
    """Returns dict(refToNew, aff, res (6,), iterations, cutoff_repeat, evaluations)."""
    T = np.array(refToNew, np.float64)
    aff = np.array(aff, np.float64)
    repeat = 1.0
    evals = 1
    res_old = trk.calcRes(T, new_exposure, aff, coarse_cutoff * repeat)
    while res_old[5] > 0.6 and repeat < 50:
        repeat *= 2
        res_old = trk.calcRes(T, new_exposure, aff, coarse_cutoff * repeat)
        evals += 1
    H, b = trk.calcG(new_exposure, aff)
    lam = 0.01
    free = [i for i in range(8) if not ((i == 6 and fix_a) or (i == 7 and fix_b))]
    it_done = 0
    for it in range(max_iterations):
        Hl = H.copy()
        Hl[np.diag_indices(8)] *= (1 + lam)
        inc = np.zeros(8)
        inc[free] = np.linalg.solve(Hl[np.ix_(free, free)], -b[free])
        extrap = 1.0
        if lam < lambda_extrapolation_limit:
            extrap = np.sqrt(np.sqrt(lambda_extrapolation_limit / lam))
        inc = inc * extrap
        inc_scaled = inc * SCALE
        if not np.isfinite(inc_scaled.sum()):
            inc_scaled[:] = 0
        T_new = se3_exp(inc_scaled[:6]) @ T
        aff_new = aff + inc_scaled[6:8]
        res_new = trk.calcRes(T_new, new_exposure, aff_new, coarse_cutoff * repeat)
        evals += 1
        it_done = it + 1
        if res_new[0] / res_new[1] < res_old[0] / res_old[1]:
            H, b = trk.calcG(new_exposure, aff_new)
            res_old, aff, T = res_new, aff_new, T_new
            lam *= 0.5
        else:
            lam *= 4
            if lam < lambda_extrapolation_limit:
                lam = lambda_extrapolation_limit
        if not (np.linalg.norm(inc) > 1e-3):
            break
    return dict(refToNew=T, aff=aff, res=np.array(res_old), iterations=it_done, cutoff_repeat=repeat, evaluations=evals)
