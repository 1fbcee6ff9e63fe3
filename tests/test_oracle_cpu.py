"""CPU tests that pin the oracles (no GPU needed)."""
import os

import numpy as np
import pytest
import torch

from oracle import mvsnet_oracle as O
from oracle.cpu import TrackerOracle, TsdfOracle
from oracle.ref_golden import (FRONT_DENSE_CASES, FRONT_PYRAMID_CASES, LM_CASES, assert_exact, front_dense_case,
                               front_pyramid_case, golden_path, lm_case, lm_key, lm_start, mvsnet_fresh_case)
from tandem_b200 import DrFusionOptions, default_weights
from tandem_b200.synthetic import RoomScene, look_at_pose, tracker_case
from tandem_b200.weights_io import load_tdmw


def _forward(g, weights):
    w, dn, va = load_tdmw(default_weights(weights))
    img, order = O.preprocess_bgr(g["bgr"], int(g["ref_index"]))
    Ks = [torch.from_numpy(g[f"K{s}"]) for s in (1, 2, 3)]
    with torch.no_grad():
        return O.forward(w, dn, img, Ks, torch.from_numpy(g["c2w"][order]), float(g["depth_min"]), float(g["depth_max"]),
                         float(g["discard"]), va)


def test_mvsnet_oracle_reproduces_shipped_goldens(golden_small):
    """tandem/exported/tandem_512x320/sample_inputs.pt outputs (abl04) - the reference's own known-answer data."""
    outs = _forward(golden_small, "abl04_fewer_depth_planes")
    for s in (1, 2, 3):
        ed = np.abs(outs[s - 1]["depth"].numpy() - golden_small[f"abl04_stage{s}_depth"]).mean()
        ec = np.abs(outs[s - 1]["confidence"].numpy() - golden_small[f"abl04_stage{s}_confidence"]).mean()
        assert ed < 2e-5 and ec < 2e-5, (s, ed, ec)


def test_mvsnet_oracle_matches_reference_abl03(golden_small):
    outs = _forward(golden_small, "abl03_view_aggregation")
    for s in (1, 2, 3):
        ed = np.abs(outs[s - 1]["depth_dense"].numpy() - golden_small[f"abl03_stage{s}_depth_dense"]).mean()
        assert ed < 2e-5, (s, ed)


def test_oracle_matches_reference_model_on_fresh_input():
    """The restatement equals the reference model (its stored outputs, oracle/ref_golden.py) on a seeded synthetic window."""
    img, Ks, c2w, dmin, dmax, disc = mvsnet_fresh_case()
    g = np.load(golden_path("ref_mvsnet_fresh.npz"))
    assert np.array_equal(img.reshape(-1)[::997].numpy(), g["input_probe"]), "the seeded input window changed"
    with torch.no_grad():
        w, dn, va = load_tdmw(default_weights("abl03_view_aggregation"))
        ours = O.forward(w, dn, img, Ks, c2w, dmin, dmax, disc, va)
    for s in range(3):
        dense = g[f"stage{s + 1}_depth_dense"]
        zero = np.unpackbits(g[f"stage{s + 1}_depth_zero"], count=dense.size).reshape(dense.shape).astype(bool)
        depth = np.where(zero, np.float32(0), dense)
        assert np.abs(dense - ours[s]["depth_dense"].numpy()).max() < 1e-4
        assert np.abs(depth - ours[s]["depth"].numpy()).max() < 1e-4
        assert np.abs(g[f"stage{s + 1}_confidence"] - ours[s]["confidence"].numpy()).max() < 1e-4


def test_tsdf_oracle_basic_properties():
    H, W = 60, 80
    opt = DrFusionOptions(height=H, width=W, fx=40.0, fy=40.0, cx=39.5, cy=29.5, num_buckets=50021, num_blocks=40000)
    scene = RoomScene(half=1.0, spheres=((0.4, 0.0, 0.5, 0.25),))
    pose = look_at_pose((0.0, 0.0, -0.2), (0.3, 0.05, 1.0))
    bgr, depth = scene.render(pose, H, W, 40.0, 40.0, 39.5, 29.5)
    o = TsdfOracle(opt)
    o.integrate(bgr, depth, pose)
    n1 = o.stats()["allocated_blocks"]
    assert n1 > 100 and o.stats()["dropped_blocks"] == 0
    o.integrate(bgr, depth, pose)
    assert o.stats()["allocated_blocks"] == n1 and o.stats()["candidate_blocks"] == 0   # idempotent block set
    coords, vox = o.dump_blocks()
    assert vox["weight"].max() == 2
    assert np.all(np.abs(vox["sdf"]) <= opt.truncation_distance + 1e-6)
    rb, rd = o.render(pose)
    ok = (rd > 0) & (depth > 0.1)
    assert ok.mean() > 0.8 and np.median(np.abs(rd[ok] - depth[ok])) < 0.01
    assert o.stats()["render_distinct_voxels"] > 0


def test_tracker_oracle_gauss_newton_descends():
    """The normal equations must point downhill: one damped GN step on the affine+pose parameters lowers E."""
    c = tracker_case(H=120, W=160, fx=80.0, fy=80.0, cx=79.5, cy=59.5)
    t = TrackerOracle(c["w"], c["h"])
    t.setK(c["w"], c["h"], c["fx"], c["fy"], c["cx"], c["cy"])
    t.setReference(c["n"], c["pc_u"], c["pc_v"], c["pc_idepth"], c["pc_color"], 1.0, np.zeros(2))
    t.setNew(c["dInew"])
    r0 = t.calcRes(np.eye(4), 1.0, np.zeros(2), 1e9)
    r1 = t.calcRes(c["refToNew"], 1.0, np.zeros(2), 1e9)
    assert r1[0] / r1[1] < r0[0] / r0[1], "true relative pose must explain the new image better than identity"
    H, b = t.calcG(1.0, np.zeros(2))
    assert np.allclose(H, H.T) and np.all(np.linalg.eigvalsh(H[:6, :6]) > -1e-6)


def test_front_oracle_pyramid_and_dense_reference():
    """Sanity of the n2 / n1 restatements (oracle/front_oracle.c) on cases whose answer is known in closed form."""
    from oracle.cpu import FrontOracle
    f = FrontOracle()
    h, w = 48, 64
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    gray = 3.0 * xx + 5.0 * yy                                    # a plane: gradients are the slopes, 2x2 means stay planar
    lv = f.make_images(gray, 3)
    assert [l[0].shape for l in lv] == [(48, 64, 3), (24, 32, 3), (12, 16, 3)]
    assert np.allclose(lv[0][0][2:-2, 2:-2, 1], 3.0) and np.allclose(lv[0][0][2:-2, 2:-2, 2], 5.0)
    assert np.allclose(lv[1][0][2:-2, 2:-2, 1], 6.0) and np.allclose(lv[1][0][2:-2, 2:-2, 2], 10.0)
    assert np.allclose(lv[1][0][..., 0], 0.25 * (gray[0::2, 0::2] + gray[0::2, 1::2] + gray[1::2, 0::2] + gray[1::2, 1::2]))
    assert np.all(lv[0][0][0, :, 1:] == 0) and np.all(lv[0][0][-1, :, 1:] == 0)       # first / last row: no gradients
    assert np.allclose(lv[0][1][3, 3], 3.0 ** 2 + 5.0 ** 2)
    # identity transform: every valid interior pixel maps onto itself
    depth = np.full((h, w), 2.0, np.float32)
    depth[10, 10] = 0.0
    K4 = (40.0, 40.0, 31.5, 23.5)
    n, arrs, proj = f.dense_reference(depth, np.eye(4), K4, 1, True, None, None, gray)
    interior = (w - 6) * (h - 6) - 1                              # 3 <= u <= w-4, 3 <= v <= h-4, minus the hole
    assert n == interior and proj[10, 10] == -1 and proj[5, 5] == 2.0
    assert arrs[0][0] == 0 and arrs[0][1] == 3 and arrs[1][1] == 3          # slot 0 = the skipped slot; first point (3,3)
    assert np.allclose(arrs[2][1:n + 1], 0.5) and arrs[3][1] == gray[3, 3]
    # nearest depth wins when two source pixels land on one target pixel
    T = np.eye(4)
    d2 = depth.copy()
    d2[20, 20], d2[20, 21] = 1.0, 2.0
    T[0, 3] = 0.0
    _, _, proj2 = f.dense_reference(d2, T, K4, 1, True, None, None, gray)
    assert proj2[20, 20] == 1.0
    # sparse points stay in front, dense points skip pixels that already carry a sparse inverse depth
    sparse = [np.array([7, 9, 0], np.float32), np.array([8, 8, 0], np.float32), np.array([0.4, 0.6, 0], np.float32),
              np.array([10, 20, 0], np.float32)]
    id0 = np.zeros((h, w), np.float32)
    id0[8, 7], id0[8, 9] = 0.4, 0.6
    n3, arrs3, _ = f.dense_reference(depth, np.eye(4), K4, 1, False, sparse, id0, gray)
    assert n3 == 2 + interior - 2 and arrs3[0][0] == 7 and arrs3[0][1] == 9


@pytest.mark.parametrize("size,levels", FRONT_PYRAMID_CASES)
def test_front_oracle_pyramid_pinned_to_reference_makeImages(size, levels):
    """n2 pin: oracle/front_oracle.c == the reference's own FrameHessian::makeImages body (HessianBlocks.cpp:128-191,
    compiled unmodified by oracle/ref_build.mk; its outputs are stored by oracle/ref_golden.py), bit for bit, incl. a
    non-finite input pixel."""
    from oracle.cpu import FrontOracle
    g = np.load(golden_path("ref_front.npz"))
    a = FrontOracle().make_images(front_pyramid_case(size), levels)
    for lvl in range(levels):
        key = f"pyr/{size[0]}x{size[1]}/{lvl}"
        assert_exact(g, key + "/dI", a[lvl][0], f"level {lvl} (I,dx,dy)")
        assert_exact(g, key + "/absSquaredGrad", a[lvl][1], f"level {lvl} absSquaredGrad")


@pytest.mark.parametrize("step,with_sparse,size", FRONT_DENSE_CASES)
def test_front_oracle_dense_reference_pinned_to_reference_setCoarseTrackingRef(step, with_sparse, size):
    """n1 pin: forward warp + nearest-depth test + raster-order append (incl. the ++pc_n quirk) of oracle/front_oracle.c ==
    the reference's own dense block of CoarseTracker::setCoarseTrackingRef (CoarseTracker.cpp:655-725, outputs stored by
    oracle/ref_golden.py), bit for bit: pc_n, all four point arrays and the stale / uncounted slots."""
    from oracle.cpu import FrontOracle
    g = np.load(golden_path("ref_front.npz"))
    key = f"dense/{step}/{int(with_sparse)}/{size[0]}x{size[1]}"
    depth, pose_d, pose_r, K4, sparse, idepth0, gray_r = front_dense_case(step, with_sparse, size)
    n_ref, T = int(g[key + "/n"]), g[key + "/T"]
    # the transform the reference derives (SE3 inverse * SE3) is the one the oracle / the device path is handed
    assert np.allclose(T, np.linalg.inv(pose_r.astype(np.float64)) @ pose_d.astype(np.float64), atol=1e-12)
    n, arrs, _ = FrontOracle().dense_reference(depth, T, K4, step, not with_sparse, sparse, idepth0, gray_r)
    assert n == n_ref and n > 1000
    for a, name in zip(arrs, ("u", "v", "idepth", "color")):
        assert_exact(g, f"{key}/{name}", a, name)


def test_lm_driver_converges_with_oracle_tracker():
    """The host restatement of trackNewestCoarse's level loop (oracle/lm_driver.py) reduces the pose error and the energy."""
    from oracle.lm_driver import se3_exp, track_level0
    c = tracker_case(H=120, W=160, fx=80.0, fy=80.0, cx=79.5, cy=59.5)
    t = TrackerOracle(c["w"], c["h"])
    t.setK(c["w"], c["h"], c["fx"], c["fy"], c["cx"], c["cy"])
    t.setReference(c["n"], c["pc_u"], c["pc_v"], c["pc_idepth"], c["pc_color"], c["ref_exposure"], c["ref_aff"])
    t.setNew(c["dInew"])
    r0 = t.calcRes(np.eye(4), c["new_exposure"], c["ref_aff"], 20.0)
    r = track_level0(t, np.eye(4), c["ref_aff"], c["new_exposure"], max_iterations=10)
    assert r["iterations"] >= 3 and r["res"][0] / r["res"][1] < 0.5 * r0[0] / r0[1]
    D0 = np.linalg.inv(c["refToNew"])
    D1 = np.linalg.inv(c["refToNew"]) @ r["refToNew"]
    assert np.linalg.norm(D1[:3, 3]) < 0.5 * np.linalg.norm(D0[:3, 3])
    E = se3_exp([0.1, -0.2, 0.3, 0.02, -0.01, 0.03])
    assert np.allclose(E[:3, :3] @ E[:3, :3].T, np.eye(3), atol=1e-12) and abs(np.linalg.det(E[:3, :3]) - 1) < 1e-12
    assert np.allclose(se3_exp(np.zeros(6)), np.eye(4))


@pytest.mark.parametrize("start,fix_a,fix_b,cutoff", LM_CASES)
def test_lm_driver_pinned_to_reference_trackNewestCoarse(start, fix_a, fix_b, cutoff):
    """n3 pin: oracle/lm_driver.py == the reference's own level loop (CoarseTracker.cpp:750-916 compiled unmodified by
    oracle/ref_build.mk; oracle/ref_golden.py stores what it returned) when both drive the SAME tracker object: same number
    of residual / normal-equation evaluations (i.e. same accept / reject sequence, cutoff doublings and stop iteration), same
    pose and affine parameters.  The last case starts with a cutoff so small that > 60 % of the points saturate: the
    cutoff-doubling and REPEAT-LEVEL rules run."""
    from oracle.lm_driver import track_level0
    g = np.load(golden_path("ref_lm.npz"))
    k = lm_key(start, fix_a, fix_b, cutoff)
    ok, counts, T, aff, out5 = int(g[k + "/ok"]), g[k + "/counts"], g[k + "/T"], g[k + "/aff"], g[k + "/out5"]
    assert ok == 1
    c, t = lm_case()
    T0 = lm_start(c, start)
    # the restatement: one pass, plus the reference's single REPEAT of the level when the cutoff had to be raised (:911-915)
    r = track_level0(t, T0, c["ref_aff"], c["new_exposure"], coarse_cutoff=cutoff, max_iterations=10, fix_a=fix_a, fix_b=fix_b)
    evals, passes = r["evaluations"], 1
    if r["cutoff_repeat"] > 1:
        r2 = track_level0(t, r["refToNew"], r["aff"], c["new_exposure"], coarse_cutoff=cutoff, max_iterations=10, fix_a=fix_a, fix_b=fix_b)
        evals += r2["evaluations"]
        passes, r = 2, r2
    print(f"{start} fix_a={fix_a} fix_b={fix_b} cutoff={cutoff}: reference loop {counts[0]} calcRes / {counts[1]} calcG, restatement {evals} "
          f"evaluations in {passes} pass(es); |dT| {np.abs(T - r['refToNew']).max():.2e}, |daff| {np.abs(aff - r['aff']).max():.2e}")
    assert counts[0] == evals
    assert np.abs(T - r["refToNew"]).max() < 1e-6 and np.abs(aff - r["aff"]).max() < 1e-4   # fp32 evaluations amplify the 1e-16 difference of the two linear solvers
    with np.errstate(invalid="ignore"):   # cutoff 0.8 < huber / 2 makes maxEnergy negative: sqrtf(E / n) is NaN in the reference too
        rms = np.sqrt(np.float32(r["res"][0] / r["res"][1]))
    assert (np.isnan(out5[0]) and np.isnan(rms)) or abs(out5[0] - rms) < 1e-5
    if cutoff < 1.0:
        assert passes == 2, "the small-cutoff case must exercise cutoff doubling + REPEAT LEVEL"
    if fix_a:
        assert aff[0] == c["ref_aff"][0]
    if fix_b:
        assert aff[1] == c["ref_aff"][1]


# ---------------------------------------------------------------------------------------------------------------------
# marching cubes oracle (SURVEY.md 8f n4): properties on the CPU (the reference has no mesh test or golden)
def _mesh_scene():
    from oracle.cpu import TsdfOracle
    from tandem_b200 import DrFusionOptions
    from tandem_b200.synthetic import RoomScene, look_at_pose
    H, W = 60, 80
    intr = dict(fx=40.0, fy=40.0, cx=39.5, cy=29.5)
    scene = RoomScene(half=0.6, spheres=((0.0, 0.0, 0.35, 0.15),))
    o = TsdfOracle(DrFusionOptions(height=H, width=W, num_buckets=50021, bucket_size=10, num_blocks=30000, **intr))
    for eye in ((0.0, 0.0, -0.3), (0.05, 0.02, -0.28), (-0.04, -0.03, -0.31)):
        pose = look_at_pose(eye, (0.0, 0.0, 0.6))
        bgr, depth = scene.render(pose, H, W, **intr)
        o.integrate(bgr, depth, pose)
    return o


def test_mesh_oracle_properties():
    o = _mesh_scene()
    lo, up = np.float32([-0.64, -0.64, -0.64]), np.float32([0.64, 0.64, 0.64])
    vert, cols = o.extract_mesh(lo, up)
    assert len(vert) % 3 == 0 and len(vert) > 3000
    assert np.isfinite(vert).all() and (cols >= 0).all() and (cols <= 1).all()
    assert (vert >= lo - 0.011).all() and (vert <= up + 0.011).all()
    # every vertex lies on the true surface (sphere r=0.15 at (0,0,0.35) or the z=+0.6 wall / side walls) within ~1.5 voxels
    d_sphere = np.abs(np.linalg.norm(vert - np.float32([0, 0, 0.35]), axis=1) - 0.15)
    d_walls = np.min(np.abs(np.abs(vert) - 0.6), axis=1)
    assert np.quantile(np.minimum(d_sphere, d_walls), 0.99) < 0.015
    # triangles are small (one cell) and non-degenerate on the whole
    tri = vert.reshape(-1, 3, 3)
    assert np.max(np.linalg.norm(tri[:, 0] - tri[:, 1], axis=1)) < 0.02
    # cell locality: the box split at a cell boundary yields exactly the two halves (same cells, same arithmetic)
    mid = np.float32(lo[0] + np.float32(64) * np.float32(0.01))
    va, _ = o.extract_mesh(lo, np.float32([mid, up[1], up[2]]))
    assert len(va) > 0
    whole_left = vert.reshape(-1, 9)[(vert.reshape(-1, 3, 3)[:, :, 0].max(1) <= mid + 0.0051)]
    assert abs(len(va) // 3 - len(whole_left)) <= 0.02 * len(whole_left) + 8
    # an empty / inverted-size box gives nothing; zero-extent axis gives nothing
    assert len(o.extract_mesh(lo, np.float32([lo[0], up[1], up[2]]))[0]) == 0
    assert len(o.extract_mesh(np.float32([3, 3, 3]), np.float32([3.5, 3.5, 3.5]))[0]) == 0


def test_marching_cubes_tables_are_consistent():
    """The committed nibble-packed case tables (product copy and oracle copy) are identical and internally consistent: the
    edges a case triangulates are exactly the edges whose two corners lie on different sides (so the crossed-edge mask the
    reference stores as `edgeTable` is implied), complementary cases use the same edges, at most five triangles per case."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def load(path):
        words = re.findall(r"0x([0-9a-f]{16})ull", open(path).read())
        assert len(words) == 256, path
        return [int(w, 16) for w in words]

    a = load(os.path.join(root, "tandem_b200", "csrc", "mc_tables.h"))
    b = load(os.path.join(root, "oracle", "mc_tables.h"))
    assert a == b
    ends = [(0, 1), (1, 2), (2, 3), (3, 0), (4, 5), (5, 6), (6, 7), (7, 4), (0, 4), (1, 5), (2, 6), (3, 7)]
    masks = []
    for case, w in enumerate(a):
        nib = [(w >> (4 * k)) & 0xF for k in range(16)]
        n = nib.index(0xF)
        assert n % 3 == 0 and n <= 15 and all(x == 0xF for x in nib[n:]) and all(x < 12 for x in nib[:n])
        used = 0
        for e in nib[:n]:
            used |= 1 << e
        topo = sum(1 << e for e, (p, q) in enumerate(ends) if ((case >> p) & 1) != ((case >> q) & 1))
        assert used == topo, case
        for t in range(0, n, 3):
            assert len({nib[t], nib[t + 1], nib[t + 2]}) == 3, case       # no degenerate triangle in the table
        masks.append(used)
    assert all(masks[c] == masks[255 - c] for c in range(256)) and masks[0] == 0 and masks[255] == 0


def test_host_homography_matches_oracle_and_reference_formula(golden_full):
    """Host logic of the cost-volume path (no GPU): the per-view homography the library uploads (double precision on the host,
    rounded to fp32) against the oracle's fp32 restatement of homo_warping (module.py:795-808) on the golden window's poses
    and intrinsics - they must agree to fp32 noise, and projecting a point through the homography must equal projecting it
    through the two cameras."""
    import ctypes
    from tandem_b200._lib import lib
    g = golden_full
    fp = ctypes.POINTER(ctypes.c_float)
    V = g["c2w"].shape[0]
    order = [int(g["ref_index"])] + [v for v in range(V) if v != int(g["ref_index"])]
    for s in (1, 2, 3):
        K = np.ascontiguousarray(g[f"K{s}"], np.float32)
        ref = np.ascontiguousarray(g["c2w"][order[0]], np.float32)
        for v in order[1:]:
            src = np.ascontiguousarray(g["c2w"][v], np.float32)
            rot = np.zeros(9, np.float32); tr = np.zeros(3, np.float32)
            assert lib().tdm_debug_homography(K.ctypes.data_as(fp), ref.ctypes.data_as(fp), src.ctypes.data_as(fp),
                                              rot.ctypes.data_as(fp), tr.ctypes.data_as(fp)) == 0
            M = O.homography(torch.from_numpy(K), torch.from_numpy(ref), torch.from_numpy(K), torch.from_numpy(src)).numpy()
            assert np.abs(rot.reshape(3, 3) - M[:3, :3]).max() < 2e-4 * max(1.0, np.abs(M[:3, :3]).max())
            assert np.abs(tr - M[:3, 3]).max() < 2e-3 * max(1.0, np.abs(M[:3, 3]).max())
            # geometric meaning, in double: a reference pixel at depth d, lifted to the world and projected into the source
            Kd, Rd, Sd = K.astype(np.float64), ref.astype(np.float64), src.astype(np.float64)
            x, y, d = 37.0, 21.0, 1.7
            Xw = Rd @ np.append(np.linalg.inv(Kd) @ np.array([x, y, 1.0]) * d, 1.0)
            q = Kd @ (np.linalg.inv(Sd) @ Xw)[:3]
            qh = rot.reshape(3, 3).astype(np.float64) @ np.array([x, y, 1.0]) * d + tr.astype(np.float64)
            assert np.abs(q - qh).max() < 1e-3 * max(1.0, np.abs(q).max())
