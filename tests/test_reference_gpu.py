"""Pins against the REAL reference: the reference's own dr_fusion class and tracker kernels, compiled unmodified for
sm_100a (oracle/ref_build.mk) and run on a B200, produced the known answers in tests/golden/ref_gpu.npz
(oracle/ref_golden.py); the same seeded inputs run here through the CUDA path and the CPU oracle.
These tests are what lifts the TSDF / tracker oracles from "parity unpinned" to "pinned against the reference's
CUDA code" (modulo the reference's documented races, SURVEY.md Appendix B).  Large reference outputs are stored as a
fixed seeded sample (see oracle/ref_golden.py for which parts are complete)."""
import numpy as np
import pytest

from oracle.ref_golden import (TRACKER_CASES, decode_depth, fusion_mesh_case, fusion_options, fusion_render_case, golden_path,
                               tracker_oracle, tracker_ref_case)
from oracle.cpu import TsdfOracle
from tandem_b200 import CudaCoarseTracker, DrFusion

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    return np.load(golden_path("ref_gpu.npz"))


def test_fusion_matches_reference_dr_fusion(ref):
    opt = fusion_options()
    H, W = opt.height, opt.width
    poses, frames, render_poses = fusion_render_case()
    ours, orc = DrFusion(opt), TsdfOracle(opt)
    for k, (pose, (bgr, depth), rp) in enumerate(zip(poses, frames, render_poses)):
        ours.IntegrateScanAsync(bgr, depth, pose)
        orc.integrate(bgr, depth, pose)
        ours.RenderAsync([rp])
        (ob,), (od,) = ours.GetRenderResult()
        cb, cd = orc.render(rp)
        rd = decode_depth(ref[f"render/{k}/depth_q"]).reshape(-1)
        idx, rb = ref[f"render/{k}/idx"], ref[f"render/{k}/bgr"]      # colour: a seeded sample of the pixels
        for name, xd, xb in (("cuda", od, ob), ("oracle", cd, cb)):
            xd, xb = xd.reshape(-1), xb.reshape(-1, 3)[idx]
            hit_r, hit_x = rd > 0, xd > 0
            mism = float(np.mean(hit_r != hit_x))
            both = hit_r & hit_x
            err = np.abs(rd[both] - xd[both])
            both_s = both[idx]
            print(f"frame {k} {name} vs reference: hit mismatch {mism:.5f}, depth mean-abs {err.mean():.2e}, "
                  f"max {err.max():.2e}, colour equal {np.mean(rb == xb):.5f} (on {idx.size} sampled pixels)")
            # the reference itself is FMA-contracted, uses a different 4x4 inverse and sphere-traces, so "same
            # surface to a small fraction of a voxel" is the strongest statement available (voxel = 1e-2 m)
            assert mism <= 3e-3
            assert err.mean() <= 3e-4 and np.quantile(err, 0.99) <= 5e-3
            assert np.mean(np.abs(rb[both_s].astype(int) - xb[both_s].astype(int)) <= 2) > 0.98


@pytest.mark.parametrize("size,step", TRACKER_CASES)
def test_tracker_matches_reference_kernels(ref, size, step):
    c = tracker_ref_case(size, step)
    n = c["n"]
    orc = tracker_oracle(c)
    ro = orc.calcRes(c["refToNew"], c["new_exposure"], c["new_aff"], c["cutoffTH"])
    Ho, bo = orc.calcG(c["new_exposure"], c["new_aff"])
    key = f"tracker/{size[0]}x{size[1]}/{step}"
    o7, o45 = ref[key + "/o7"], ref[key + "/o45"]
    # reference host post-processing (cuda_coarse_tracker.cpp:264-272, 335-355)
    rr = np.array([o7[0], o7[1], o7[4] / o7[6], 0, o7[5] / o7[6], o7[3] / o7[1]], np.float64)
    scale = np.array([1, 1, 1, .5, .5, .5, 10, 1000.0])
    tri = lambda r, q: min(r, q) * 9 + max(r, q) - min(r, q) * (min(r, q) + 1) // 2
    Hr = np.array([[o45[tri(r, q)] for q in range(8)] for r in range(8)], np.float64) / o7[2] * np.outer(scale, scale)
    br = np.array([o45[tri(r, 8)] for r in range(8)], np.float64) / o7[2] * scale
    w, h = c["w"], c["h"]
    g = CudaCoarseTracker(w, h)
    g.init()
    g.setK(w, h, c["fx"], c["fy"], c["cx"], c["cy"])
    g.setReference(n, c["pc_u"], c["pc_v"], c["pc_idepth"], c["pc_color"], c["ref_exposure"], c["ref_aff"])
    g.setNew(c["dInew"])
    rg, Hg, bg = g.calcResAndG(c["refToNew"], c["new_exposure"], c["new_aff"], c["cutoffTH"])
    rel = lambda a, b: np.max(np.abs(a - b)) / np.max(np.abs(b))
    for name, (r_, H_, b_) in (("cuda", (rg, Hg, bg)), ("oracle", (ro, Ho, bo))):
        print(f"{name} vs reference kernels: dE/E {abs(r_[0] - rr[0]) / rr[0]:.2e}, numE {r_[1]} vs {rr[1]}, "
              f"H rel {rel(H_, Hr):.2e}, b rel {rel(b_, br):.2e}")
        assert abs(r_[1] - rr[1]) <= 2          # the reference's own FMA contraction may flip a border point
        assert abs(r_[0] - rr[0]) <= 2e-4 * rr[0]
        assert abs(r_[2] - rr[2]) <= 1e-3 * rr[2] and abs(r_[4] - rr[4]) <= 1e-3 * rr[4]
        assert abs(r_[5] - rr[5]) <= 1e-4
        assert rel(H_, Hr) < 2e-3 and rel(b_, br) < 2e-3   # reference sums 3e5 fp32 terms with float atomics
    wo = orc.warped
    valid = np.unpackbits(ref[key + "/valid"], count=n).astype(bool)
    same = valid == (wo[6] != 0)
    assert same.mean() > 0.9999
    idx = ref[key + "/idx"]                 # residuals: a seeded sample of the points
    m = valid[idx] & (wo[6][idx] != 0)
    d = np.abs(ref[key + "/residual"][m] - wo[5][idx][m])
    assert np.quantile(d, 0.999) < 5e-3 and np.max(d) < 5e-2


def test_mesh_matches_reference_marching_cubes(ref):
    """DrFusion::GetMesh of the reference (brute-force ExtractMeshKernel, mesh_extractor.cu:244-265) vs ours and vs the
    oracle on volumes fused from the same scans.  The volumes themselves differ in the last bits (FMA contraction, 4x4
    inverse, allocation races - see the render test above), so the meshes are compared as surfaces: triangle counts
    within 2 %, inside a crop cube (where the reference mesh is stored in full) every vertex of ours has a reference vertex
    within a small fraction of a voxel, and so has every sampled vertex of the reference mesh one of ours."""
    from scipy.spatial import cKDTree
    opt = fusion_options()
    poses, frames, lo, up = fusion_mesh_case()
    ours, orc = DrFusion(opt), TsdfOracle(opt)
    for pose, (bgr, depth) in zip(poses, frames):
        ours.IntegrateScanAsync(bgr, depth, pose)
        ours.RenderAsync([pose]); ours.GetRenderResult()
        orc.integrate(bgr, depth, pose)
    n = int(ref["mesh/n"])
    sv = ref["mesh/sample_vert"]
    clo, cup = ref["mesh/crop_lo"], ref["mesh/crop_up"]
    cv, cc = ref["mesh/crop_vert"], ref["mesh/crop_color"].astype(np.float32)
    gv, gc = ours.GetMesh(lo, up)
    ov, oc = orc.extract_mesh(lo, up)
    tree = cKDTree(cv)
    margin = np.float32(0.01)           # one voxel: the nearest reference vertex of a vertex this far inside is in the crop
    for name, xv, xc in (("cuda", gv, gc), ("oracle", ov, oc)):
        inner = np.all((xv >= clo + margin) & (xv <= cup - margin), axis=1)
        assert inner.sum() > 100, (name, int(inner.sum()))
        dist, idx = tree.query(xv[inner])
        back, _ = cKDTree(xv).query(sv)
        exact = float(np.mean(dist == 0))
        print(f"{name} vs reference mesh: {len(xv) // 3} vs {n // 3} triangles, vertex NN distance median {np.median(dist):.2e} "
              f"p99 {np.quantile(dist, 0.99):.2e} ({int(inner.sum())} vertices in the crop; reverse p99 {np.quantile(back, 0.99):.2e} "
              f"over {len(sv)} sampled reference vertices), coincident vertices {exact:.4f}, "
              f"colour max diff at NN (median) {np.median(np.abs(xc[inner] - cc[idx]).max(1)):.3f}")
        assert abs(len(xv) - n) <= 0.02 * n
        assert np.median(dist) <= 1e-4 and np.quantile(dist, 0.99) <= 5e-3 and np.quantile(back, 0.99) <= 5e-3
        assert np.median(np.abs(xc[inner] - cc[idx]).max(1)) <= 2.5 / 255
