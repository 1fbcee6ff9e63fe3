#!/usr/bin/env python
"""bench.py - keyframe depth maps/s of the CVA-MVSNet hot path (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision mixed16|fp32] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is one DrMvsnet window (7 views, 640x480, 3 stages, depth_num (48,32,8), view aggregation:
BASELINE.json configs[1]) through the hot path.  `value` times K steps with the window already resident in HBM
(CUDA events on the engine's stream, max over ranks); `e2e` times the same K steps through the public
DrMvsnet.CallAsync -> GetResult call with host buffers (pinned H2D of the u8 images and D2H of the four output maps
inside the timed region).  --dump-outputs DIR writes the four maps the end-to-end leg returned for its last step
(rank 0; the inputs are the same on every run) as DIR/<name>.npy, so that two builds can be compared output for output.
Multi-GPU: one process per GPU, independent windows per rank (weak scaling, no data-path
collective - SURVEY.md §8e); torch.distributed is only used for the barrier and the max-over-ranks reduction.
`--impl reference` times the reference's own CPU path: its PyTorch model cannot travel to the GPU box, so the
pinned CPU restatement (oracle/mvsnet_oracle.py, verified against the reference model and its shipped goldens) is
run on all host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it

WORKLOAD = "CVA-MVSNet 640x480, 7 views, 3-stage cascade (48/32/8), view aggregation (abl03), 1 window/step/GPU"
WEIGHTS = "abl03_view_aggregation"
# identical in both arms (the driver compares the two lines' `config`); per-arm run parameters live under "run"
CONFIG = {"workload": WORKLOAD,
          "l2": "no flush needed: each step streams > 1 GB of activations through a 126 MB L2 (GPU arm; the CPU arm has no device cache to flush)"}


def tune_host_malloc():
    """Keep freed result buffers inside the process.  DrMvsnet::GetResult hands every keyframe's four maps (4.9 MB) to the caller
    in freshly allocated memory (dr_mvsnet.h:12-34: four malloc'd arrays per output, ownership transferred).  With glibc's
    defaults such blocks are mmap'd and unmapped every time, and the kernel's page faults + zeroing for them (~0.9 ms per
    keyframe, measured) cost about as much as the whole forward (1.2 ms).  Raising the mmap / trim thresholds - an
    application-level allocator setting, equivalent to MALLOC_MMAP_THRESHOLD_ / MALLOC_TRIM_THRESHOLD_ in the environment -
    lets malloc recycle them.  Applied to both arms."""
    import ctypes
    try:
        libc = ctypes.CDLL("libc.so.6")
        M_TRIM_THRESHOLD, M_MMAP_THRESHOLD = -1, -3
        ok = libc.mallopt(M_MMAP_THRESHOLD, 1 << 30) and libc.mallopt(M_TRIM_THRESHOLD, 1 << 30)
        return "mallopt(M_MMAP_THRESHOLD, M_TRIM_THRESHOLD) raised: freed result buffers are recycled" if ok else "mallopt refused"
    except OSError:
        return "libc not found: allocator defaults"


def load_window(rank=0):
    g = np.load(os.path.join(ROOT, "tests", "golden", "sample_640x480.npz"))
    bgr = g["bgr"].copy()
    if rank > 0:  # independent windows per rank: seeded photometric jitter of the golden window
        rng = np.random.default_rng(rank)
        gain = 1.0 + 0.05 * rng.standard_normal()
        bgr = np.clip(bgr.astype(np.float32) * gain + rng.normal(0, 1.0, bgr.shape), 0, 255).astype(np.uint8)
    V, H, W = bgr.shape[:3]
    return dict(V=V, H=H, W=W, bgrs=[np.ascontiguousarray(bgr[v]) for v in range(V)],
                c2ws=[np.ascontiguousarray(g["c2w"][v]) for v in range(V)], K=g["K3"].astype(np.float32),
                Ks=[g["K1"], g["K2"], g["K3"]], ref_index=int(g["ref_index"]), dmin=float(g["depth_min"]),
                dmax=float(g["depth_max"]), discard=float(g["discard"]), bgr_all=bgr, c2w_all=g["c2w"])


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p)).get("bf16_tflops_sustained", 1374.6))
    return 1400.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def pick_cpu_threads(run=None):
    """Thread count of the reference arm: the fastest of {16, 32, 64, all} on ONE FULL forward of the workload each (after a
    short warm-up conv so that the thread pool exists).  Round 1 probed a toy convolution and the choice - hence the
    headline ratio - moved 2x between driver runs; a full forward per candidate costs ~10 s in total and is stable."""
    import torch
    ncpu = os.cpu_count() or 1
    # (all hardware threads is only a candidate up to 64: on the 128-thread host of the B200 boxes torch's CPU convolutions take
    #  53 s per forward with 128 threads against 1.7 s with 16 - measured in round 2, profiles/r02_bench_reference.json)
    cands = sorted({c for c in (16, 32, 64, ncpu if ncpu <= 64 else 64) if c <= ncpu}) or [ncpu]
    if run is None or len(cands) == 1:
        torch.set_num_threads(cands[-1])
        return cands[-1], {}
    timings = {}
    torch.set_num_threads(cands[0])
    run()                                   # cold start (allocator, oneDNN primitive caches) paid before any candidate is timed
    for c in cands:
        torch.set_num_threads(c)
        x = torch.rand(1, 8, 8, 60, 80)
        torch.nn.functional.conv3d(x, torch.rand(8, 8, 3, 3, 3), padding=1)
        t0 = time.perf_counter()
        run()
        timings[c] = time.perf_counter() - t0
    best = min(timings, key=timings.get)
    torch.set_num_threads(best)
    return best, {str(k): round(v, 3) for k, v in timings.items()}


def oracle_forward_fn(win, device=None):
    """The reference graph (cva_mvsnet.py:98-184) as restated by oracle/mvsnet_oracle.py (pinned against the reference model
    and its shipped goldens).  device=None: torch CPU fp32 = the reference's CPU path; device='cuda:0': the same torch ops on
    cuDNN fp32 (TF32 off) = the compute path of the reference's libdr `module.forward` (dr_mvsnet.cpp:292-294)."""
    import torch
    from oracle import mvsnet_oracle as O
    from tandem_b200 import default_weights
    from tandem_b200.weights_io import load_tdmw
    w, dn, va = load_tdmw(default_weights(WEIGHTS))
    img, order = O.preprocess_bgr(win["bgr_all"], win["ref_index"])
    Ks = [torch.from_numpy(np.asarray(k, np.float32)) for k in win["Ks"]]
    c2w = torch.from_numpy(win["c2w_all"][order])
    if device is not None:
        dev = torch.device(device)
        w = {k: torch.from_numpy(np.asarray(v)).to(dev) for k, v in w.items()}
        img, c2w, Ks = img.to(dev), c2w.to(dev), [k.to(dev) for k in Ks]

        def run():
            with torch.no_grad(), torch.device(dev):
                return O.forward(w, dn, img, Ks, c2w, win["dmin"], win["dmax"], win["discard"], va)
        return run

    def run():
        with torch.no_grad():
            return O.forward(w, dn, img, Ks, c2w, win["dmin"], win["dmax"], win["discard"], va)
    win["cpu_threads"], win["cpu_thread_probe_s"] = pick_cpu_threads(run)
    return run


def time_gpu_reference(win, local, steps=10, warmup=3):
    """GPU comparator (VERDICT r01 item 3 / SURVEY 8d iii): the reference graph in eager PyTorch on cuDNN on the same B200,
    timed with CUDA events outside our arm's timed regions: fp32 with TF32 off (bit-comparable arithmetic) and with TF32 on
    (what torch 1.9, the reference's libtorch, allows cuDNN by default).  Returns a dict for the JSON line."""
    import torch
    try:
        torch.backends.cudnn.benchmark = True
        run = oracle_forward_fn(win, device=f"cuda:{local}")
        res = {}
        for tf32 in (False, True):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            for _ in range(warmup):
                out = run()
            torch.cuda.synchronize(local)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                out = run()
            e1.record()
            torch.cuda.synchronize(local)
            res[tf32] = (e0.elapsed_time(e1) / steps, out[2]["depth_dense"].float().cpu().numpy(), out[2]["mask"].cpu().numpy())
        ms = res[False][0]
        return {"value": 1e3 / ms, "unit": "keyframes/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
                "tf32_value": 1e3 / res[True][0], "tf32_ms_per_step": res[True][0],
                "depth_dense_gpu": res[False][1], "mask_gpu": res[False][2], "mask_gpu_tf32": res[True][2], "depth_dense_gpu_tf32": res[True][1],
                "what": "oracle/mvsnet_oracle.py (the reference graph, pinned) in eager PyTorch on cuda: cuDNN fp32 (value: TF32 off; "
                        "tf32_value: TF32 allowed), cudnn.benchmark on, inputs resident - the compute path of the reference's libdr "
                        "module.forward (dr_mvsnet.cpp:292-294)"}
    except Exception as e:   # the comparator must never take the bench line down
        return {"unavailable": f"{type(e).__name__}: {e}"[:200]}


def time_cpu(win, steps, warmup):
    run = oracle_forward_fn(win)
    for _ in range(warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    dt = time.perf_counter() - t0
    return steps / dt, dt / steps * 1e3


def bind_to_gpu_numa(local, n_local):
    """Pin this rank (and every thread it creates afterwards: engine workers, the copy pool; page-locked allocations are then
    node-local too) to its GPU's NUMA node, sharing the node's CPUs evenly with the other ranks whose GPUs hang off the same
    node.  Returns a short description for the JSON line."""
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=index,pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=20).stdout
        bus = {}
        for line in q.strip().splitlines():
            idx, b = [x.strip() for x in line.split(",")]
            bus[int(idx)] = b.lower()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = [int(x) for x in vis.split(",")] if vis and all(t.strip().isdigit() for t in vis.split(",")) else sorted(bus)

        def node_of(i):
            b = bus[phys[i]]
            b = b[-12:] if len(b) > 12 else b            # nvidia-smi prints an 8-digit domain, sysfs a 4-digit one
            with open(f"/sys/bus/pci/devices/{b}/numa_node") as f:
                return int(f.read().strip())
        nodes = [node_of(i) for i in range(n_local)]
        node = nodes[local]
        if node < 0:
            return "numa node unknown (-1): not bound"
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        cpus = sorted(set(cpus) & os.sched_getaffinity(0))
        peers = [i for i in range(n_local) if nodes[i] == node]
        k, m = peers.index(local), len(peers)
        # physical cores first, hyper-thread siblings second, in Linux's usual numbering: give each rank a slice of both halves
        half = len(cpus) // 2
        lo, hi = cpus[:half], cpus[half:]
        mine = lo[k * len(lo) // m:(k + 1) * len(lo) // m] + hi[k * len(hi) // m:(k + 1) * len(hi) // m]
        if not mine:
            return "no cpus left for this rank: not bound"
        os.sched_setaffinity(0, mine)
        return f"GPU {local} -> NUMA node {node}, {len(mine)} of its {len(cpus)} cpus ({m} ranks on the node)"
    except Exception as e:
        return f"not bound ({type(e).__name__}: {e})"[:160]


def dist_setup(n):
    if n <= 1 or "RANK" not in os.environ:
        return 0, 1, 0, None
    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    # NCCL announces its version on stdout when the communicator is created (NCCL_DEBUG=VERSION in this image); stdout is
    # reserved for the ONE JSON line, so fd 1 points at stderr until the communicator exists.
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
        torch.cuda.synchronize(local)
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    return rank, world, local, dist


def ncu_traffic(record_name):
    """DRAM bytes (read + write) per launch of the roofline kernel, from the committed `ncu --set full` capture of the
    same kernel (profiles/rNN_ncu_traffic.json, written by tools/summarise_profiles.py). None when no capture matches."""
    import glob
    files = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r*_ncu_traffic.json")))
    if not files or not record_name.endswith("cost_volume"):
        return None, None
    pat = {"s1": ", 16, 2, ", "s2": ", 16, 1, ", "s3": ", 8, 1, "}.get(record_name[:2])   # <TV, C, CSPLIT, ND, ACC16> of the stage's kernel
    try:
        for k, v in json.load(open(files[-1])).items():
            if pat and "k_cost_volume_va16<" in k and pat in k:
                return float(v), os.path.basename(files[-1])
    except (OSError, ValueError):
        pass
    return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="mixed16", choices=["mixed16", "fp32", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip the eager-PyTorch/cuDNN comparator record")
    ap.add_argument("--no-bind", action="store_true", help="do not bind ranks to their GPU's NUMA node (multi-GPU runs)")
    ap.add_argument("--workload", default="mvsnet", choices=["mvsnet", "slab_tsdf"],
                    help="mvsnet: the BASELINE.json metric (default).  slab_tsdf: BASELINE configs[4], TSDF half - ONE 1024^3 volume "
                         "partitioned into Z-slabs over the ranks, integrate + slab-clipped ray-cast + nearest-hit all-reduce per frame "
                         "(strong scaling; a step = one 640x480 depth map)")
    ap.add_argument("--inflight", type=int, default=8, choices=[1, 2, 3, 4, 5, 6, 7, 8],
                    help="independent windows in flight per GPU (n DrMvsnet handles, one stream each, used round-robin) in both legs")
    ap.add_argument("--e2e-inflight", type=int, default=4, choices=[1, 2, 3, 4, 5, 6, 7, 8],
                    help="handles used by the end-to-end leg (the first k of the --inflight handles); measured best at 4: with more, "
                         "the extra host threads and staging buffers cost more than the added overlap gives")
    ap.add_argument("--tc", type=int, default=-1, help="1/0: force the tcgen05 conv path on/off (default: engine default)")
    ap.add_argument("--opt", action="append", default=[], help="engine option key=int for A/B runs, e.g. --opt fork_fpn=0")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result maps of the last timed end-to-end step as DIR/<name>.npy (float32)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.workload != "mvsnet"):
        ap.error("--dump-outputs applies to the mvsnet workload of --impl ours")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    host_malloc = tune_host_malloc()
    if a.workload == "slab_tsdf":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_slab_tsdf
        r = bench_slab_tsdf.main(["--frames", str(a.steps), "--warmup", str(a.warmup)])
        if r is not None:
            print(json.dumps({"metric": "TSDF depth maps integrated + ray-cast per second (1024^3 voxels @ 1 cm, Z-slab partition)",
                              "value": r["frames_per_s"], "unit": "frames/s", "n_gpus": r["n_gpus"], "steps": r["frames"],
                              "warmup": a.warmup, "ms_per_step": r["ms_per_frame(max over ranks, wall incl. H2D/D2H)"],
                              "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 sdf / u8 colour + weight",
                              "data": "synthetic 10 m room + 3 spheres, 640x480 depth maps (seeded noise, 2 % drop-outs)",
                              "config": {"workload": "BASELINE configs[4] TSDF half: one 10.24 m volume in Z-slabs over the ranks"},
                              "detail": r}))
        return 0

    if a.impl == "reference":
        rank = int(os.environ.get("RANK", 0))
        if rank != 0:
            return 0
        win = load_window(0)
        steps = a.steps
        kfs, ms = time_cpu(win, steps, min(a.warmup, 1))
        cores = win["cpu_threads"]
        print(json.dumps({
            "impl": "reference", "metric": "keyframe depth maps/sec", "value": kfs, "unit": "keyframes/s", "n_gpus": a.gpus,
            "steps": steps, "warmup": min(a.warmup, 1), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "golden sample window (tests/golden/sample_640x480.npz)",
            "config": CONFIG,
            "cpu_baseline": {"value": kfs, "unit": "keyframes/s", "cores": cores, "kind": "port",
                             "sample": f"{steps} full forwards of the workload window (oracle/mvsnet_oracle.py, torch CPU fp32, {cores} of {os.cpu_count()} host threads: fastest of one full forward per candidate {win.get('cpu_thread_probe_s')})"},
            "e2e": {"value": kfs, "unit": "keyframes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return 0

    rank, world, local, dist = dist_setup(a.gpus)
    affinity = bind_to_gpu_numa(local, int(os.environ.get("LOCAL_WORLD_SIZE", world))) if world > 1 and not a.no_bind else "single rank: not bound"
    import torch  # device plumbing + torch.distributed only
    from tandem_b200 import DrMvsnet, DrMvsnetOutput, default_weights
    from tandem_b200._lib import pinned_empty
    win = load_window(rank)
    m = DrMvsnet(default_weights(WEIGHTS), precision=a.precision, device=local)
    # second handle for the end-to-end leg: two windows in flight per GPU (window k+1's staging copy + H2D and window
    # k's D2H + copy-out overlap the other window's forward) - plain use of the public DrMvsnet call surface
    extra = [DrMvsnet(default_weights(WEIGHTS), precision=a.precision, device=local) for _ in range(a.inflight - 1)]
    if a.tc >= 0:
        for h in [m] + extra:
            h.set_option("use_tc", a.tc)
    for kv in a.opt:
        k, v = kv.split("=")
        for h in [m] + extra:
            h.set_option(k, int(v))

    def call():
        m.CallAsync(win["H"], win["W"], win["V"], win["ref_index"], win["bgrs"], win["K"], win["c2ws"], win["dmin"],
                    win["dmax"], win["discard"])
        return m.GetResult()

    out = call()  # builds the plan, uploads the window
    assert np.isfinite(out.depth_dense).all()
    hs = [m] + extra

    def submit(h):
        h.CallAsync(win["H"], win["W"], win["V"], win["ref_index"], win["bgrs"], win["K"], win["c2ws"], win["dmin"],
                    win["dmax"], win["discard"])

    for h in extra:                         # builds each handle's plan and makes its window resident
        submit(h); h.GetResult()
    for _ in range(a.warmup):               # W untimed steps (a step = one window's forward)
        DrMvsnet.run_resident_multi(hs, len(hs))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(local)

    sampler = ClockSampler(local) if rank == 0 else None
    # ---- device-resident: EXACTLY K steps, CUDA events on the engine stream ----
    barrier()
    if sampler:
        sampler.start()
    ms_dev, launches = DrMvsnet.run_resident_multi(hs, a.steps)   # K windows, one CUDA-event clock over all streams
    barrier()
    ms_single, _ = m.run_resident(max(a.steps // 2, 1))            # one window at a time: the latency of a keyframe
    ms_single /= max(a.steps // 2, 1)
    barrier()
    # ---- end to end through the public call with host buffers ----
    # Headline leg: the caller keeps its images and its (recycled) result maps in PAGE-LOCKED host memory - the library then
    # DMA's straight from / into them (H2D of the 7 u8 images + D2H of the 4 maps inside the timed region, every step).
    # Secondary leg ("pageable_*"): ordinary numpy arrays and a freshly allocated DrMvsnetOutput per call, i.e. the
    # reference's ownership contract verbatim, staged through the library's pinned buffers by its copy pool.
    pin_bgrs = []
    for b in win["bgrs"]:
        pb = pinned_empty(b.shape, np.uint8)
        pb[...] = b
        pin_bgrs.append(pb)

    def submit_pinned(h):
        h.CallAsync(win["H"], win["W"], win["V"], win["ref_index"], pin_bgrs, win["K"], win["c2ws"], win["dmin"],
                    win["dmax"], win["discard"])

    def e2e_leg(handles, sub, outs):
        n = len(handles)
        barrier()
        t0 = time.perf_counter()
        for j in range(min(n - 1, a.steps)):
            sub(handles[j])
        r = None
        for i in range(a.steps):            # EXACTLY K windows submitted and K results fetched
            if i + n - 1 < a.steps:
                sub(handles[(i + n - 1) % n])
            r = handles[i % n].GetResult(out=outs[i % n] if outs else None)
        torch.cuda.synchronize(local)
        ms = (time.perf_counter() - t0) * 1e3
        assert np.isfinite(r.depth_dense).all()
        last[0] = r
        return ms

    last = [None]                           # the result of the last step of the latest e2e leg
    hs_e2e = hs[:max(1, min(a.e2e_inflight, len(hs)))]
    pin_outs = [DrMvsnetOutput(win["H"], win["W"], pinned=True) for _ in hs_e2e]
    for _ in range(2):
        call()
    ms_pg_serial = e2e_leg(hs_e2e[:1], submit, None)
    ms_pg = e2e_leg(hs_e2e, submit, None) if len(hs_e2e) > 1 else ms_pg_serial
    for h in hs_e2e:
        h.set_option("eager_d2h", 0)        # GetResult DMA's into the caller's page-locked maps itself
    for h, o in zip(hs_e2e, pin_outs):
        submit_pinned(h); h.GetResult(out=o)
    ms_e2e_serial = e2e_leg(hs_e2e[:1], submit_pinned, pin_outs[:1])
    ms_e2e = e2e_leg(hs_e2e, submit_pinned, pin_outs) if len(hs_e2e) > 1 else ms_e2e_serial
    if a.dump_outputs and rank == 0:        # the headline e2e leg's last step, copied before the buffers are reused
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name in ("depth", "confidence", "depth_dense", "confidence_dense"):
            np.save(os.path.join(a.dump_outputs, name + ".npy"), np.array(getattr(last[0], name), np.float32))
    for h in hs_e2e:
        h.set_option("eager_d2h", 1)
    assert np.array_equal(pin_outs[0].depth_dense, out.depth_dense), "page-locked and pageable paths must return the same map"
    barrier()
    clocks = sampler.stop() if sampler else None

    from tandem_b200.parallel import reduce_max
    ms_dev, ms_e2e, ms_e2e_serial, ms_pg, ms_pg_serial = reduce_max(dist, [ms_dev, ms_e2e, ms_e2e_serial, ms_pg, ms_pg_serial],
                                                                    device=f"cuda:{local}")   # slowest rank

    if rank == 0:
        value = world * a.steps / (ms_dev / 1e3)
        e2e = world * a.steps / (ms_e2e / 1e3)
        # roofline, measured live: per-kernel CUDA-event durations of one forward (m.profile()) with each record's
        # algorithmic bytes / flops.  Reported per FAMILY (tcgen05 convs / cost volume / tail) and for the whole step; the
        # "dominant kernel" entry the contract asks for is the largest single record.
        rows = m.profile()
        tot = sum(r[1] for r in rows)
        top = max(rows, key=lambda r: r[1])
        peak, how = measured_peaks()
        tpeak = measured_tensor_peak()
        ach = top[2] / (top[1] * 1e-3) / 1e9
        alg_total = sum(r[2] for r in rows)
        traffic, traffic_src = ncu_traffic(top[0])

        def family(name):
            if "cost_volume" in name:
                return "cost_volume"
            if "[tc" in name or name.startswith("f.") and name != "f.img":
                return "convs"
            if "preprocess" in name:
                return "preprocess"
            return "tail"
        fam = {}
        for name, ms_k, by, fl in rows:
            f = fam.setdefault(family(name), {"ms": 0.0, "bytes": 0.0, "flops": 0.0, "launches": 0})
            f["ms"] += ms_k; f["bytes"] += by; f["flops"] += fl; f["launches"] += 1
        families = {k: {"ms": round(v["ms"], 4), "share_of_kernel_time": round(v["ms"] / tot, 4), "launches": v["launches"],
                        "algorithmic_GB": round(v["bytes"] / 1e9, 4),
                        "achieved_GBps": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1),
                        "frac_of_hbm_peak": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9 / peak, 4),
                        "achieved_TFLOPs": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2),
                        "frac_of_tensor_peak": round(v["flops"] / (v["ms"] * 1e-3) / 1e12 / tpeak, 4) if k == "convs" else None}
                    for k, v in fam.items()}
        roof = {"bound": "hbm", "kernel": top[0], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes": top[2],
                "note": "largest single kernel record; see `families` for the per-family fractions and step_* for the whole step",
                "peak_source": how, "kernel_ms": top[1], "kernel_share_of_step": top[1] / tot,
                "families": families, "tensor_peak_TFLOPs": tpeak,
                "step_algorithmic_GB": alg_total / 1e9, "step_achieved_GBps": alg_total / (ms_dev / a.steps * 1e-3) / 1e9,
                "step_frac_of_peak": alg_total / (ms_dev / a.steps * 1e-3) / 1e9 / peak,
                "single_window_frac_of_peak": alg_total / (ms_single * 1e-3) / 1e9 / peak}
        cpu = None
        if world == 1 and not a.no_cpu_baseline:
            kfs, ms = time_cpu(win, 2, 1)
            cpu = {"value": kfs, "unit": "keyframes/s", "cores": win["cpu_threads"], "kind": "port",
                   "sample": f"2 full forwards of the workload window after 1 warm-up (oracle/mvsnet_oracle.py, torch CPU fp32; threads: fastest of one full forward per candidate {win.get('cpu_thread_probe_s')})"}
        gpu_ref = None
        if world == 1 and not a.no_gpu_reference:
            gpu_ref = time_gpu_reference(win, local)
            dd = gpu_ref.pop("depth_dense_gpu", None)
            if dd is not None:   # our output vs the comparator's on the same window (sanity of both arms)
                # accuracy is compared on IDENTICAL inputs: the per-stage intrinsics the golden / comparator use (the timed legs go
                # through CallAsync, whose stage intrinsics follow the C++ wrapper's derivation, dr_mvsnet.cpp:220-247)
                m.CallAsyncStageK(win["H"], win["W"], win["V"], win["ref_index"], win["bgrs"], np.stack(win["Ks"]).astype(np.float32),
                                  win["c2ws"], win["dmin"], win["dmax"], win["discard"])
                out = m.GetResult()
                msk = dd > 0
                gpu_ref["abs_rel_ours_vs_gpu_reference"] = float(np.mean(np.abs(dd[msk] - out.depth_dense[msk]) / dd[msk]))
                # how well do the reference's OWN two arithmetic paths agree?  (golden = its CPU fp32 model output)
                gg = np.load(os.path.join(ROOT, "tests", "golden", "sample_640x480.npz"))
                gold, gmask = gg["abl03_stage3_depth_dense"], gg["abl03_stage3_depth"] == 0
                iou = lambda a_, b_: float(np.logical_and(a_, b_).sum() / max(np.logical_or(a_, b_).sum(), 1))
                gm = gold > 0
                gpu_ref["abs_rel_vs_cpu_reference"] = float(np.mean(np.abs(gold[gm] - dd[gm]) / gold[gm]))
                gpu_ref["mask_iou_vs_cpu_reference"] = iou(gpu_ref.pop("mask_gpu"), gmask)
                dt = gpu_ref.pop("depth_dense_gpu_tf32")
                gpu_ref["tf32_abs_rel_vs_cpu_reference"] = float(np.mean(np.abs(gold[gm] - dt[gm]) / gold[gm]))
                gpu_ref["tf32_mask_iou_vs_cpu_reference"] = iou(gpu_ref.pop("mask_gpu_tf32"), gmask)
                gpu_ref["ours_abs_rel_vs_cpu_reference"] = float(np.mean(np.abs(gold[gm] - out.depth_dense[gm]) / gold[gm]))
                gpu_ref["ours_mask_iou_vs_cpu_reference"] = iou(out.depth == 0, gmask)
                gpu_ref["speedup_device"] = value / gpu_ref["value"]
                gpu_ref["speedup_single_window"] = (1e3 / ms_single) / gpu_ref["value"]
                gpu_ref["speedup_device_vs_tf32"] = value / gpu_ref["tf32_value"]
        h2d = win["V"] * win["H"] * win["W"] * 3
        d2h = 4 * win["H"] * win["W"] * 4
        line = {
            "metric": "keyframe depth maps/sec", "value": value, "unit": "keyframes/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms_dev / a.steps, "single_window_ms": ms_single, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": {"mixed16": "f16 activations + bf16 cost volume, f32 accumulate", "fp32": "f32", "bf16": "bf16"}[a.precision],
            "data": "golden sample window (tests/golden/sample_640x480.npz: 7x640x480 u8 + poses), seeded jitter per rank; weights abl03 checkpoint",
            "config": CONFIG,
            "run": {"windows_per_step": world, "windows_in_flight_per_gpu": a.inflight, "parallelism": f"dp{world} (independent windows)"},
            "e2e": {"value": e2e, "unit": "keyframes/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / a.steps, "windows_in_flight_per_gpu": len(hs_e2e),
                    "serial_value": world * a.steps / (ms_e2e_serial / 1e3), "serial_ms_per_step": ms_e2e_serial / a.steps,
                    "note": "CallAsync -> GetResult(out=recycled) with PAGE-LOCKED host buffers (images and result maps): DMA straight from / into caller memory; serial_* = one window at a time (latency bound)",
                    "pageable_value": world * a.steps / (ms_pg / 1e3), "pageable_serial_value": world * a.steps / (ms_pg_serial / 1e3),
                    "pageable_note": "ordinary numpy inputs + a freshly allocated DrMvsnetOutput per call (the reference's ownership contract), staged through the library's pinned buffers by the process-wide copy pool",
                    "host_malloc": host_malloc, "affinity": affinity},
            "gpu_launches": launches * a.steps, "launches_per_step": launches,
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "gpu_reference": gpu_ref,
        }
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
