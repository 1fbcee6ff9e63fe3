"""Known answers of the REFERENCE implementation for the pin tests, stored under tests/golden/ so that the tests run without
the reference.  TEST INFRASTRUCTURE ONLY.

The case builders below construct the (seeded, synthetic) inputs; the tests call the same builders, so the inputs a test
feeds the oracle or the CUDA path are the ones the reference saw.  Regenerating the files needs the reference: its
Python model (cva_mvsnet) and the libraries oracle/ref_build.mk compiles from its sources into oracle/_ref/:

    python oracle/ref_golden.py cpu --reference DIR   # CPU pins: MVSNet model, makeImages, setCoarseTrackingRef, trackNewestCoarse
    python oracle/ref_golden.py gpu [--full OUT]      # needs a B200: dr_fusion render + mesh, tracker kernels

Bit-exact pins store a SHA-256 of each output array (with NaNs and signed zeros canonicalised, which is what
np.array_equal(..., equal_nan=True) ignores) plus a seeded sample of its values, which names the first differing
element when the digest does not match.  Tolerance pins store the reference's outputs in full where they are small,
and a fixed seeded sample otherwise (every file stays well below 1 MB).
"""
import argparse
import ctypes
import hashlib
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
GOLDEN = os.path.join(REPO, "tests", "golden")
REF_LIBS = os.path.join(REPO, "oracle", "_ref")
N_SAMPLE = 16


def golden_path(name):
    return os.path.join(GOLDEN, name)


# ---------------------------------------------------------------------------------------------------------------------
# bit-exact comparison through digests
def canonical(a):
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), a.dtype.type(np.nan), a + a.dtype.type(0))   # one NaN pattern, -0 -> +0
    return a


def digest(a):
    a = canonical(a)
    return hashlib.sha256(str(a.dtype).encode() + str(a.shape).encode() + a.tobytes()).hexdigest()


def sample_index(size, k=N_SAMPLE, seed=0):
    idx = np.sort(np.random.default_rng(seed).choice(size, min(k, size), replace=False))
    return idx.astype(np.uint16 if size <= 1 << 16 else np.int32)


def pin_exact(store, key, a):
    """Record digest + a seeded sample of `a` under `key`."""
    a = np.asarray(a)
    idx = sample_index(a.size)
    store[key + "/sha256"] = np.array(digest(a))
    store[key + "/shape"] = np.array(a.shape, np.int64)
    store[key + "/idx"] = idx
    store[key + "/val"] = canonical(a).reshape(-1)[idx]


def assert_exact(g, key, a, name=None):
    """a must equal, bit for bit up to NaN payloads and zero signs, the array pinned under `key`."""
    a = np.asarray(a)
    name = name or key
    assert tuple(a.shape) == tuple(g[key + "/shape"]), (name, a.shape, tuple(g[key + "/shape"]))
    got = canonical(a).reshape(-1)[g[key + "/idx"]]
    exp = g[key + "/val"]
    bad = np.flatnonzero(~((got == exp) | (np.isnan(got) & np.isnan(exp))))
    assert bad.size == 0, f"{name}: element {int(g[key + '/idx'][bad[0]])} is {got[bad[0]]!r}, reference {exp[bad[0]]!r}"
    assert digest(a) == str(g[key + "/sha256"]), f"{name}: differs from the reference (digest)"


# ---------------------------------------------------------------------------------------------------------------------
# case builders shared by the generator and the tests
def mvsnet_fresh_case():
    """A seeded synthetic 4-view window for abl03 (64x96); returns (img, Ks, c2w, dmin, dmax, discard)."""
    import torch
    torch.manual_seed(0)
    V, H, W = 4, 64, 96
    img = torch.rand(V, 3, H, W)
    img = torch.nn.functional.avg_pool2d(img, 5, 1, 2)
    K3 = torch.tensor([[100.0, 0, 47.5], [0, 100.0, 31.5], [0, 0, 1]])
    Ks = [torch.cat([K3[:2] * s, K3[2:]]) for s in (0.25, 0.5, 1.0)]
    c2w = torch.eye(4).repeat(V, 1, 1)
    c2w[:, 0, 3] = torch.arange(V) * 0.05
    return img, Ks, c2w, 0.5, 5.0, 10.0


FRONT_PYRAMID_CASES = [((480, 640), 4), ((96, 130), 2), ((60, 80), 3)]
FRONT_DENSE_CASES = [(1, False, (240, 320)), (2, True, (240, 320)), (1, True, (120, 160)), (3, False, (480, 640))]


def front_pyramid_case(size):
    h, w = size
    rng = np.random.default_rng(3)
    gray = (rng.random((h, w)) * 255).astype(np.float32)
    gray[5, 7] = np.inf
    return gray


def front_dense_case(step, with_sparse, size):
    """Inputs of setCoarseTrackingRef's dense block: (depth, pose_d, pose_r, K4, sparse, idepth0, gray_r)."""
    from tandem_b200.synthetic import RoomScene, look_at_pose
    h, w = size
    f = 160.0 * w / 320.0
    K4 = (f, f, (w - 1) / 2.0, (h - 1) / 2.0)
    scene = RoomScene()
    pose_d = look_at_pose((0.3, 0.0, -0.2), (2.5, 0.2, 0.5))
    pose_r = look_at_pose((0.34, 0.02, -0.17), (2.5, 0.25, 0.45))
    _, depth = scene.render(pose_d, h, w, *K4, dropout=0.02, seed=1)
    bgr_r, _ = scene.render(pose_r, h, w, *K4)
    gray_r = bgr_r.astype(np.float32) @ np.array([0.114, 0.587, 0.299], np.float32)
    rng = np.random.default_rng(5)
    sparse, idepth0 = None, None
    if with_sparse:
        ns = 500
        sparse = [rng.integers(3, w - 3, ns + 1).astype(np.float32), rng.integers(3, h - 3, ns + 1).astype(np.float32),
                  rng.uniform(0.2, 2.0, ns + 1).astype(np.float32), rng.uniform(0, 255, ns + 1).astype(np.float32)]
        idepth0 = np.zeros((h, w), np.float32)
        idepth0[sparse[1][:ns].astype(int), sparse[0][:ns].astype(int)] = sparse[2][:ns]
    return depth, pose_d, pose_r, K4, sparse, idepth0, gray_r


LM_CASES = [("identity", False, False, 20.0), ("near", False, False, 20.0), ("identity", True, True, 20.0),
            ("identity", False, True, 20.0), ("identity", True, False, 20.0), ("identity", False, False, 0.8)]


def lm_case():
    """The tracker case and an oracle tracker set up on it (both sides of the LM pin drive this same tracker)."""
    from tandem_b200.synthetic import tracker_case
    c = tracker_case(H=120, W=160, fx=80.0, fy=80.0, cx=79.5, cy=59.5)
    return c, tracker_oracle(c)


def lm_start(c, start):
    if start == "identity":
        return np.eye(4)
    return np.array(c["refToNew"], np.float64) @ np.linalg.inv(
        np.array([[1, 0, 0, 0.004], [0, 1, 0, -0.003], [0, 0, 1, 0.002], [0, 0, 0, 1.0]]))


def lm_key(start, fix_a, fix_b, cutoff):
    return f"lm/{start}/{int(fix_a)}{int(fix_b)}/{cutoff:g}"


FUSION_INTR = dict(fx=80.0, fy=80.0, cx=79.5, cy=59.5)
FUSION_HW = (120, 160)
# world shifted by +2.56 m (32 blocks): the reference also integrates its FREE hash entries, all aliased to block (0,0,0)
# (Appendix B.2 of SURVEY.md); keeping the origin far outside the map keeps that quirk out of the comparison.
FUSION_OFFSET = np.array([2.56, 2.56, 2.56], np.float32)


def fusion_options():
    from tandem_b200 import DrFusionOptions
    H, W = FUSION_HW
    return DrFusionOptions(height=H, width=W, num_buckets=200003, bucket_size=10, num_blocks=120000, **FUSION_INTR)


def _fusion_scene():
    from tandem_b200.synthetic import RoomScene
    return RoomScene(half=1.2, spheres=((0.5, 0.1, 0.4, 0.3), (-0.4, -0.2, 0.6, 0.25), (0.1, 0.4, -0.6, 0.3)))


def _fusion_frames(poses):
    H, W = FUSION_HW
    scene = _fusion_scene()
    frames = [scene.render(p, H, W, **FUSION_INTR, noise_sigma=0.002, dropout=0.02, seed=k) for k, p in enumerate(poses)]
    for p in poses:
        p[:3, 3] += FUSION_OFFSET
    return poses, frames


def fusion_render_case():
    """Four scans (two poses, each with a perturbed twin) and the pose each frame's render uses."""
    from tandem_b200.synthetic import circle_trajectory
    poses = circle_trajectory(2, radius=0.3)
    poses = [poses[0], poses[0].copy(), poses[1], poses[1].copy()]
    poses[1][:3, 3] += np.float32(0.03)
    poses[3][:3, 3] -= np.float32(0.02)
    poses, frames = _fusion_frames(poses)
    render_poses = [poses[max(k - 1, 0)] if k % 2 else p for k, p in enumerate(poses)]
    return poses, frames, render_poses


def fusion_mesh_case():
    from tandem_b200.synthetic import circle_trajectory
    poses, frames = _fusion_frames(circle_trajectory(3, radius=0.3))
    lo = (FUSION_OFFSET - np.float32(1.28)).astype(np.float32)
    up = (FUSION_OFFSET + np.float32(1.28)).astype(np.float32)
    return poses, frames, lo, up


TRACKER_CASES = [((120, 160), 1), ((480, 640), 1)]


def tracker_ref_case(size, step):
    from tandem_b200.synthetic import tracker_case
    h, w = size
    s = w / 640.0
    return tracker_case(H=h, W=w, fx=320.0 * s, fy=320.0 * s, cx=319.5 * s, cy=239.5 * s, step=step)


def tracker_oracle(c):
    from oracle.cpu import TrackerOracle
    o = TrackerOracle(c["w"], c["h"])
    o.setK(c["w"], c["h"], c["fx"], c["fy"], c["cx"], c["cy"])
    o.setReference(c["n"], c["pc_u"], c["pc_v"], c["pc_idepth"], c["pc_color"], c["ref_exposure"], c["ref_aff"])
    o.setNew(c["dInew"])
    return o


# sampling of the large GPU-side outputs
RENDER_SAMPLE = 1024           # pixels per rendered frame whose reference colour is stored (depth: all pixels)
TRACKER_SAMPLE = 2048          # points per case whose reference residual is stored
MESH_SAMPLE = 1024             # reference mesh vertices stored, drawn over the whole mesh
MESH_CROP_MAX = 2000           # the reference vertices inside one crop cube are stored in full (for the forward query)


def mesh_crop_box(rv):
    """A cube around a seeded vertex of the reference mesh, halved until it holds at most MESH_CROP_MAX vertices."""
    c = rv[sample_index(len(rv), 1, seed=1)[0]]
    half = np.float32(0.4)
    while True:
        lo, up = (c - half).astype(np.float32), (c + half).astype(np.float32)
        if np.all((rv >= lo) & (rv <= up), axis=1).sum() <= MESH_CROP_MAX:
            return lo, up
        half = np.float32(half * 0.75)


# ---------------------------------------------------------------------------------------------------------------------
# generation (needs the reference)
def _ref_lib(name):
    p = os.path.join(REF_LIBS, name)
    if not os.path.exists(p):
        sys.exit(f"{p} missing: build it with `make -C oracle -f ref_build.mk` (needs the reference sources)")
    return ctypes.CDLL(p)


def gen_mvsnet(ref_root):
    import types
    import torch
    sys.path.insert(0, os.path.join(ref_root, "cva_mvsnet"))
    pkg = types.ModuleType("models")
    pkg.__path__ = [os.path.join(ref_root, "cva_mvsnet", "models")]
    sys.modules["models"] = pkg           # bypasses models/__init__.py (needs pytorch_lightning)
    from models.cva_mvsnet import CvaMVSNet, StageTensor
    ck = torch.load(os.path.join(ref_root, "cva_mvsnet", "pretrained", "ablation", "abl03_view_aggregation.ckpt"),
                    map_location="cpu", weights_only=False)
    net = CvaMVSNet(depth_num=ck["hparams"]["MODEL.DEPTH_NUM"], view_aggregation=True).eval()
    net.load_state_dict({k[len("cva_mvsnet."):]: v for k, v in ck["state_dict"].items()})
    img, Ks, c2w, dmin, dmax, disc = mvsnet_fresh_case()
    with torch.no_grad():
        ref = net(img[None], StageTensor(*[k[None] for k in Ks]), c2w[None], torch.tensor([dmin]), torch.tensor([dmax]),
                  torch.tensor([disc]))
    d = {"input_probe": img.reshape(-1)[::997].numpy()}
    for s in range(3):
        dense, depth = ref[s].depth_dense[0].numpy(), ref[s].depth[0].numpy()
        # the filtered depth is the dense depth with the low-confidence pixels zeroed: stored as that mask
        assert np.array_equal(depth, np.where(depth == 0, 0, dense))
        d[f"stage{s + 1}_depth_dense"] = dense
        d[f"stage{s + 1}_depth_zero"] = np.packbits(depth == 0)
        d[f"stage{s + 1}_confidence"] = ref[s].confidence[0].numpy()
    return d


def gen_front():
    from oracle.cpu import FrontRef
    ref = FrontRef()
    d = {}
    for size, levels in FRONT_PYRAMID_CASES:
        out = ref.make_images(front_pyramid_case(size), levels)
        for lvl in range(levels):
            pin_exact(d, f"pyr/{size[0]}x{size[1]}/{lvl}/dI", out[lvl][0])
            pin_exact(d, f"pyr/{size[0]}x{size[1]}/{lvl}/absSquaredGrad", out[lvl][1])
    for step, with_sparse, size in FRONT_DENSE_CASES:
        depth, pose_d, pose_r, K4, sparse, idepth0, gray_r = front_dense_case(step, with_sparse, size)
        n, arrs, T = ref.dense_reference(depth, pose_d, pose_r.astype(np.float64), K4, step, not with_sparse, sparse, idepth0,
                                         gray_r)
        key = f"dense/{step}/{int(with_sparse)}/{size[0]}x{size[1]}"
        d[key + "/n"] = np.int64(n)
        d[key + "/T"] = T
        for a, name in zip(arrs, ("u", "v", "idepth", "color")):
            pin_exact(d, f"{key}/{name}", a)
    return d


def gen_lm():
    lib = _ref_lib("liblm_ref.so")
    lib.ref_lm_track_level0.restype = ctypes.c_int
    dp = ctypes.POINTER(ctypes.c_double)
    RES = ctypes.CFUNCTYPE(None, ctypes.c_void_p, dp, ctypes.c_float, dp, ctypes.c_float, dp)
    G = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_float, dp, dp, dp)
    d = {}
    for start, fix_a, fix_b, cutoff in LM_CASES:
        c, t = lm_case()

        def res_cb(_, T16, expo, aff2, cut, out6):
            r = t.calcRes(np.array([T16[i] for i in range(16)]).reshape(4, 4), expo, np.array([aff2[0], aff2[1]]), cut)
            for i in range(6):
                out6[i] = r[i]

        def g_cb(_, expo, aff2, H64, b8):
            H, b = t.calcG(expo, np.array([aff2[0], aff2[1]]))
            for i in range(8):
                b8[i] = b[i]
                for j in range(8):
                    H64[8 * i + j] = H[i, j]
        T = np.ascontiguousarray(lm_start(c, start), np.float64).copy()
        aff = np.array(c["ref_aff"], np.float64).copy()
        out5 = np.zeros(5)
        counts = (ctypes.c_int * 2)()
        ok = lib.ref_lm_track_level0(None, RES(res_cb), G(g_cb), T.ctypes.data_as(dp), aff.ctypes.data_as(dp),
                                     ctypes.c_float(c["new_exposure"]), ctypes.c_float(c["ref_exposure"]),
                                     np.array(c["ref_aff"], np.float64).ctypes.data_as(dp), ctypes.c_float(cutoff), int(fix_a),
                                     int(fix_b), out5.ctypes.data_as(dp), counts)
        k = lm_key(start, fix_a, fix_b, cutoff)
        d[k + "/ok"], d[k + "/counts"] = np.int64(ok), np.array(counts[:], np.int64)
        d[k + "/T"], d[k + "/aff"], d[k + "/out5"] = T, aff, out5
    return d


def _fusion_ref():
    lib = _ref_lib("libdr_fusion_ref.so")
    lib.ref_fusion_create.restype = ctypes.c_void_p
    lib.ref_fusion_get_mesh.restype = ctypes.c_longlong
    return lib


def gen_gpu(full=None):
    fp = ctypes.POINTER(ctypes.c_float)
    raw = {}
    H, W = FUSION_HW
    opt = fusion_options()
    # dr_fusion: integrate + render
    lib = _fusion_ref()
    poses, frames, render_poses = fusion_render_case()
    h = ctypes.c_void_p(lib.ref_fusion_create(ctypes.byref(opt)))
    for k, (pose, (bgr, depth), rp) in enumerate(zip(poses, frames, render_poses)):
        b, dd = np.ascontiguousarray(bgr), np.ascontiguousarray(depth)
        lib.ref_fusion_integrate(h, ctypes.c_void_p(b.ctypes.data), dd.ctypes.data_as(fp), pose.ctypes.data_as(fp))
        rb = np.zeros((H, W, 3), np.uint8)
        rd = np.zeros((H, W), np.float32)
        lib.ref_fusion_render(h, rp.ctypes.data_as(fp), ctypes.c_void_p(rb.ctypes.data), rd.ctypes.data_as(fp), H * W)
        raw[f"render/{k}/depth"], raw[f"render/{k}/bgr"] = rd, rb
    lib.ref_fusion_destroy(h)
    # dr_fusion: mesh
    poses, frames, lo, up = fusion_mesh_case()
    h = ctypes.c_void_p(lib.ref_fusion_create(ctypes.byref(opt)))
    for pose, (bgr, depth) in zip(poses, frames):
        b, dd = np.ascontiguousarray(bgr), np.ascontiguousarray(depth)
        lib.ref_fusion_integrate(h, ctypes.c_void_p(b.ctypes.data), dd.ctypes.data_as(fp), pose.ctypes.data_as(fp))
        rb = np.zeros((H, W, 3), np.uint8)
        rd = np.zeros((H, W), np.float32)
        lib.ref_fusion_render(h, pose.ctypes.data_as(fp), ctypes.c_void_p(rb.ctypes.data), rd.ctypes.data_as(fp), H * W)
    cap = 3 * 2000000
    rv, rc = np.zeros((cap, 3), np.float32), np.zeros((cap, 3), np.float32)
    n = lib.ref_fusion_get_mesh(h, lo.ctypes.data_as(fp), up.ctypes.data_as(fp), rv.ctypes.data_as(fp), rc.ctypes.data_as(fp),
                                ctypes.c_longlong(cap))
    lib.ref_fusion_destroy(h)
    assert 0 < n <= cap
    rv, rc = rv[:n], rc[:n]
    raw["mesh/vert"], raw["mesh/color"] = rv, rc
    # tracker kernels
    tl = _ref_lib("libtracker_ref.so")
    f = ctypes.c_float
    for size, step in TRACKER_CASES:
        c = tracker_ref_case(size, step)
        n = c["n"]
        aff = tracker_oracle(c)._aff(c["new_exposure"], c["new_aff"])
        T = np.ascontiguousarray(c["refToNew"], np.float32)
        Ki = np.array([1.0 / c["fx"], 0, -c["cx"] / c["fx"], 0, 1.0 / c["fy"], -c["cy"] / c["fy"], 0, 0, 1], np.float32)
        o7, o45 = np.zeros(7, np.float32), np.zeros(45, np.float32)
        warped = np.zeros((7, n), np.float32)
        rc_ = tl.ref_tracker_eval(c["w"], c["h"], f(c["fx"]), f(c["fy"]), f(c["cx"]), f(c["cy"]), T.ctypes.data_as(fp),
                                  Ki.ctypes.data_as(fp), f(aff[0]), f(aff[1]), f(c["ref_aff"][1]), f(9.0), f(c["cutoffTH"]), n,
                                  c["pc_u"].ctypes.data_as(fp), c["pc_v"].ctypes.data_as(fp), c["pc_idepth"].ctypes.data_as(fp),
                                  c["pc_color"].ctypes.data_as(fp), np.ascontiguousarray(c["dInew"]).ctypes.data_as(fp),
                                  o7.ctypes.data_as(fp), o45.ctypes.data_as(fp), warped.ctypes.data_as(fp))
        assert rc_ == 0
        key = f"tracker/{size[0]}x{size[1]}/{step}"
        raw[key + "/o7"], raw[key + "/o45"], raw[key + "/warped"] = o7, o45, warped
    if full:
        os.makedirs(full, exist_ok=True)
        np.savez_compressed(os.path.join(full, "ref_gpu_full.npz"), **raw)
    return raw


def compact_gpu(raw):
    """What the tests need of the GPU-side reference outputs, in a small file."""
    d = {}
    for k in range(sum(key.startswith("render/") and key.endswith("/depth") for key in raw)):
        rd, rb = raw[f"render/{k}/depth"], raw[f"render/{k}/bgr"]
        d[f"render/{k}/depth_q"] = encode_depth(rd)
        idx = sample_index(rd.size, RENDER_SAMPLE, seed=k)
        d[f"render/{k}/idx"], d[f"render/{k}/bgr"] = idx, rb.reshape(-1, 3)[idx]
    d.update(compact_mesh(raw["mesh/vert"], raw["mesh/color"]))
    for size, step in TRACKER_CASES:
        key = f"tracker/{size[0]}x{size[1]}/{step}"
        warped = raw[key + "/warped"]
        idx = sample_index(warped.shape[1], TRACKER_SAMPLE)
        d[key + "/o7"], d[key + "/o45"] = raw[key + "/o7"], raw[key + "/o45"]
        d[key + "/valid"] = np.packbits(warped[6] != 0)
        d[key + "/idx"], d[key + "/residual"] = idx, warped[5][idx]
    return d


DEPTH_STEP = 2.0 ** -14     # m; rounding to it moves a depth by at most 3.1e-5 m, 1/10 of the render pin's mean tolerance


def encode_depth(rd):
    """A rendered depth map as row-wise differences of its values in DEPTH_STEP units (compresses ~2x better than float32)."""
    q = np.round(rd.astype(np.float64) / DEPTH_STEP).astype(np.int32)
    return np.diff(q, axis=1, prepend=0).astype(np.int32)


def decode_depth(dq):
    return (np.cumsum(dq, axis=1, dtype=np.int64) * DEPTH_STEP).astype(np.float32)


def compact_mesh(rv, rc):
    d = {"mesh/n": np.int64(len(rv))}
    idx = sample_index(len(rv), MESH_SAMPLE)
    d["mesh/sample_vert"] = rv[idx]
    clo, cup = mesh_crop_box(rv)
    inside = np.all((rv >= clo) & (rv <= cup), axis=1)
    d["mesh/crop_lo"], d["mesh/crop_up"] = clo, cup
    d["mesh/crop_vert"], d["mesh/crop_color"] = rv[inside], rc[inside].astype(np.float16)
    return d


def save(name, d):
    p = golden_path(name)
    np.savez_compressed(p, **d)
    print(f"wrote {p} ({os.path.getsize(p) / 1e3:.1f} kB)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("what", choices=["cpu", "gpu"])
    ap.add_argument("--reference", default=os.environ.get("TANDEM_REFERENCE", ""),
                    help="root of the reference checkout (for its Python model; cpu only)")
    ap.add_argument("--full", default=None, help="gpu: also write the reference's full outputs into this directory")
    ap.add_argument("--from-full", default=None, help="gpu: re-derive the stored file from such a full-output file")
    a = ap.parse_args()
    if a.what == "cpu":
        if not os.path.isdir(os.path.join(a.reference, "cva_mvsnet")):
            sys.exit("--reference must point at the reference checkout (containing cva_mvsnet/)")
        save("ref_mvsnet_fresh.npz", gen_mvsnet(a.reference))
        save("ref_front.npz", gen_front())
        save("ref_lm.npz", gen_lm())
    else:
        raw = dict(np.load(a.from_full)) if a.from_full else gen_gpu(a.full)
        save("ref_gpu.npz", compact_gpu(raw))


if __name__ == "__main__":
    main()
