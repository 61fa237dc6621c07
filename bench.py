#!/usr/bin/env python
"""bench.py -- surround-BEV frame-sets/s on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the fused BEV path over one batch of synthetic frame-sets:
BASELINE configs[3] shape -- 32 frame-sets of 4 x 1920x1080 BGR -> 1000x1000 canvas,
blend=True -- per GPU (weak scaling: every rank renders its own batch; the path shards
by frame-set with no data-path collective).  One JSON line on stdout (rank 0).

  value     device-resident throughput (frames already in HBM), CUDA events, max over ranks
  e2e       same metric through the public API with pinned HOST frames: H2D of every
            frame and D2H of every canvas inside the timed region
  roofline  k_bev<false> (the dominant kernel): algorithmic bytes / measured kernel time
            against MEASURED_PEAKS.json's HBM copy bandwidth
  cpu_baseline / --impl reference: the reference's own cv2 call sequence
            (oracle/cv2_path.py; the reference is pure Python over OpenCV) on the host cores
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(FW=1920, FH=1080, BW=1000, BH=1000, n_cam=4, batch=32, blend=True, balance=False)
ALT_WORKLOADS = {   # BASELINE.json configs[1..3] shapes (all 4 cameras, batch frame-sets per GPU)
    "cfg4": {},
    "cfg2": dict(FW=1280, FH=960, BW=1000, BH=1000, blend=False, balance=False),
    "cfg3": dict(FW=1920, FH=1080, BW=1200, BH=1200, blend=True, balance=True),
    # BASELINE configs[4]: 8 cameras 3840x2160 -> 2000x2000, one camera per GPU on 8 GPUs (SURVEY 8d.5: cameras 4-7 are
    # the four fixtures with H rotated by 45 degrees about the canvas centre, 8 angular wedge masks)
    "cfg5": dict(FW=3840, FH=2160, BW=2000, BH=2000, n_cam=8, batch=8, blend=False, balance=False),
}
NAMES = ("front", "back", "left", "right")


# ----------------------------------------------------------------------------- inputs
def synthetic_calibration(FW, FH, BW, BH):
    """Fixture K/D/H rescaled to the workload geometry (tests/golden/fixtures.npz); falls
    back to a generic 190-degree fisheye rig if the fixtures are absent."""
    p = os.path.join(ROOT, "tests", "golden", "fixtures.npz")
    z = np.load(p)
    sx, sy, bx, by = FW / 1280, FH / 1024, BW / 1000, BH / 1000
    S, B = np.diag([sx, sy, 1.0]), np.diag([bx, by, 1.0])
    return {n: (S @ z[f"K_{n}"], z[f"D_{n}"], B @ z[f"H_{n}"] @ np.linalg.inv(S)) for n in NAMES}


def synthetic_frames(FW, FH, n_cam, batch, seed, out=None):
    """uint8 frame-sets: smooth gradients + seeded noise (data = synthetic)."""
    rng = np.random.default_rng(seed)
    if out is None:
        out = np.empty((batch, n_cam, FH, FW, 3), np.uint8)
    yy, xx = np.mgrid[0:FH, 0:FW]
    base = ((xx * 255 // FW) ^ (yy * 255 // FH)).astype(np.uint8)
    for b in range(batch):
        for c in range(n_cam):
            noise = rng.integers(0, 64, (FH, FW, 3), dtype=np.uint8)
            out[b, c] = np.roll(base, 37 * (b * n_cam + c), axis=1)[..., None] // 2 + noise + 16 * c
    return out


def dst_matrix(K, FW, FH, FS=1.0, SS=2.0):
    P = np.array(K, np.float64)
    P[0, 0] *= FS
    P[1, 1] *= FS
    P[0, 2] = FW / 2 * SS
    P[1, 2] = FH / 2 * SS
    return P


def rig(w):
    """(cameras [(K, D, H)], masks) of the workload: the four fixture cameras with the reference's masks, or the
    8-camera rig of BASELINE configs[4]."""
    import cv2
    from cameracalibration_b200.SurroundBirdEyeView import surroundBEV as S
    calib = synthetic_calibration(w["FW"], w["FH"], w["BW"], w["BH"])
    g = S._Geo()
    g.FW, g.FH, g.BW, g.BH = w["FW"], w["FH"], w["BW"], w["BH"]
    g.CW, g.CH = int(250 * w["BW"] / 1000), int(400 * w["BH"] / 1000)
    cams = [calib[n] for n in NAMES]
    if w["n_cam"] == 8:
        c, s_ = np.cos(np.pi / 4), np.sin(np.pi / 4)
        cx, cy = g.BW / 2, g.BH / 2
        rot = np.array([[c, -s_, cx - c * cx + s_ * cy], [s_, c, cy - s_ * cx - c * cy], [0, 0, 1.0]])
        cams = cams + [(K, D, rot @ H) for K, D, H in cams]
        ang = np.linspace(0, 2 * np.pi, 9)
        masks = []
        for i in range(8):
            tri = np.array([[cx, cy], [cx + g.BW * np.cos(ang[i]), cy + g.BW * np.sin(ang[i])],
                            [cx + g.BW * np.cos(ang[i + 1]), cy + g.BW * np.sin(ang[i + 1])]]).astype(np.int32)
            masks.append(cv2.fillPoly(np.zeros((g.BH, g.BW), np.uint8), [tri], 255))
        return cams, masks, g, calib
    return cams, None, g, calib


def build_engine(w, device):
    from cameracalibration_b200 import _lib as L
    from cameracalibration_b200 import ops
    from cameracalibration_b200.SurroundBirdEyeView import surroundBEV as S
    cams, masks, g, calib = rig(w)
    ctx = L.Context(device)
    eng = ops.BevEngine(w["n_cam"], (g.FW, g.FH), (g.BW, g.BH), ctx=ctx)
    if masks is None:
        if w["blend"]:
            polys = np.stack([S._fill(S._blend_points(n, g), g) for n in NAMES])
            masks = list(eng.blend_masks(polys, S._seam_lines(g)))
        else:
            masks = [S._fill(S._plain_points(n, g), g) for n in NAMES]
    for i, (K, D, H) in enumerate(cams):
        eng.set_camera(i, K, D, dst_matrix(K, g.FW, g.FH), g.und_size, H)
        eng.set_mask(i, masks[i])
    eng.finalize()
    return eng, calib, masks, g


def algorithmic_bytes(eng, masks, w):
    """SURVEY 8(d): per frame-set, unique 32-B sectors of source gathered under the masks
    + one canvas write.  Computed from the engine's own LUT."""
    pitch = w["FW"] * 3
    src = 0
    for c in range(w["n_cam"]):
        m1, _ = eng.get_maps(c)
        act = masks[c] != 0
        sx = m1[..., 0][act].astype(np.int64)
        sy = m1[..., 1][act].astype(np.int64)
        ok = (sx >= 0) & (sx + 1 < w["FW"]) & (sy >= 0) & (sy + 1 < w["FH"])
        sx, sy = sx[ok], sy[ok]
        sect = []
        for dy in (0, 1):
            off = (sy + dy) * pitch + sx * 3
            sect.append(off // 32)
            sect.append((off + 5) // 32)
        src += np.unique(np.concatenate(sect)).size * 32
    canvas = w["BW"] * w["BH"] * 3
    return int(src), int(canvas)


DUMP_BYTES = 64 << 20


def dump_outputs(path, canvases, seed=0):
    """Write the canvases of the last timed step (uint8 [n][BH][BW][3]) under `path` for output-by-output comparison of
    two builds: all of them as canvases.npy (float32) when that fits in DUMP_BYTES, otherwise a fixed, seeded sample
    of whole canvas rows as canvas_rows.npy (float32 [k][BW][3]) with their (canvas, row) numbers in
    canvas_row_index.npy (float64 [k][2])."""
    os.makedirs(path, exist_ok=True)
    canvases = np.asarray(canvases)
    n, h, w = canvases.shape[:3]
    if canvases.size * 4 <= DUMP_BYTES:
        np.save(os.path.join(path, "canvases.npy"), canvases.astype(np.float32))
        return
    k = (DUMP_BYTES - (1 << 20)) // (w * 3 * 4)                     # 1 MB left for the index and the .npy headers
    rows = np.sort(np.random.default_rng(seed).choice(n * h, k, replace=False))
    np.save(os.path.join(path, "canvas_rows.npy"), canvases.reshape(n * h, w, 3)[rows].astype(np.float32))
    np.save(os.path.join(path, "canvas_row_index.npy"), np.stack([rows // h, rows % h], 1).astype(np.float64))


# ----------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.max_mhz, self.mask = index, [], False, None, 0
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            pass

    def run(self):
        while self.ok and not self.stop_flag:
            try:
                mhz = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                util = self.nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                try:
                    r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((mhz, util))
                self.mask |= int(r)
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        mhz = sorted(m for m, _ in self.samples)
        return {"sm_mhz": float(mhz[len(mhz) // 2]), "sm_max_mhz": float(self.max_mhz or 0),
                "reasons": [n for bit, n in self.REASONS.items() if self.mask & bit], "samples": len(mhz)}


# ----------------------------------------------------------------------------- CPU reference arm
cpu_parallel = None   # set by cpu_reference: the same call sequence, one frame-set per host thread


def cpu_reference(w, calib, masks, n_sets, repeats, seconds_cap):
    """The reference's CPU path (its cv2 call sequence, oracle/cv2_path.py) on the same
    workload shape; returns (frame-sets/s, threads, description)."""
    global cpu_parallel
    import cv2
    from oracle import cv2_path as C
    g = C.Geometry(FW=w["FW"], FH=w["FH"], BW=w["BW"], BH=w["BH"],
                   CW=int(250 * w["BW"] / 1000), CH=int(400 * w["BH"] / 1000))
    ref = C.RefBev(calib, g, w["blend"], w["balance"], masks=[m.copy() for m in masks])
    sets = synthetic_frames(w["FW"], w["FH"], w["n_cam"], n_sets, seed=7)
    best = None
    default_threads = cv2.getNumThreads()
    for threads in sorted({default_threads, os.cpu_count() or default_threads}):   # cv2's default pool and every core
        cv2.setNumThreads(threads)
        for s in sets[:2]:
            ref(*s)
        t0, n = time.perf_counter(), 0
        for _ in range(repeats):
            for s in sets:
                ref(*s)
                n += 1
            if time.perf_counter() - t0 > seconds_cap / 2:
                break
        dt = time.perf_counter() - t0
        if best is None or n / dt > best[0]:
            best = (n / dt, threads, f"{n} frame-sets ({n_sets} distinct) of the workload in {dt:.1f} s, cv2 {cv2.__version__}, "
                                     f"best of cv2 thread counts {{default {default_threads}, all {os.cpu_count()}}}")
    cv2.setNumThreads(default_threads)
    cpu_parallel = cpu_frame_set_parallel(ref, list(sets), seconds_cap=min(5.0, seconds_cap / 3))
    return best


def cpu_frame_set_parallel(ref, sets, seconds_cap=5.0):
    """Secondary CPU figure: the same cv2 call sequence, but one frame-set per host thread (cv2's own pool
    off, cv2 releases the GIL) -- what a batch of independent frame-sets allows on a many-core host.  This is
    a different driver than the reference's serial loop, so it is reported next to the baseline, not as it."""
    import cv2
    from concurrent.futures import ThreadPoolExecutor
    workers = max(1, min(os.cpu_count() or 1, 64))
    before = cv2.getNumThreads()
    cv2.setNumThreads(1)
    try:
        with ThreadPoolExecutor(workers) as pool:
            list(pool.map(lambda s: ref(*s), [sets[i % len(sets)] for i in range(workers)]))      # warm-up
            t0, n = time.perf_counter(), 0
            while time.perf_counter() - t0 < seconds_cap:
                list(pool.map(lambda s: ref(*s), [sets[i % len(sets)] for i in range(2 * workers)]))
                n += 2 * workers
            dt = time.perf_counter() - t0
    finally:
        cv2.setNumThreads(before)
    return {"value": n / dt, "unit": "frame-sets/s", "threads": workers,
            "note": "one frame-set per host thread, cv2 internal threads off; not the reference's serial driver"}


# ----------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="frame-sets per GPU per step (default: the workload's own)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed end-to-end steps (default: min(steps, 20))")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--shard", default="frames", choices=["frames", "cameras", "cameras-p2p"],
                    help="multi-GPU policy: frame-sets per GPU (weak scaling, no collective; default) or cameras per GPU "
                         "(strong scaling over one batch: 'cameras' = slabs + ONE NCCL all-gather, every rank gets all canvases; "
                         "'cameras-p2p' = the fused kernel stores slabs into the owning rank over NVLink, canvases stay sharded)")
    ap.add_argument("--workload", default="cfg4", choices=sorted(ALT_WORKLOADS),
                    help="cfg4 (default) is the headline; the others are secondary measurements of BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the canvases of the last timed step (rank 0) to DIR/*.npy as float32")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    w = dict(WORKLOAD, **ALT_WORKLOADS[a.workload])
    if a.batch:
        w["batch"] = a.batch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    metric, unit = "surround_bev_frame_sets_per_sec", "frame-sets/s"
    config = {"workload": f"{w['batch']} frame-sets/GPU x {w['n_cam']} cams {w['FW']}x{w['FH']} BGR -> {w['BW']}x{w['BH']} BEV, "
                          f"blend={w['blend']} balance={w['balance']} (BASELINE {a.workload} shape)",
              "sharding": ("frame-sets per GPU, no data-path collective" if a.shard == "frames" else
                           "cameras per GPU, fused: the render kernel stores each slab into the rank that owns the frame-set (b % world) over "
                           "NVLink peer memory, a 4-byte all-gather is the step barrier, owners compose; canvases stay sharded" if a.shard == "cameras-p2p" else
                           "cameras per GPU: each rank renders its cameras' slabs (tile-aligned mask bounding boxes), ONE "
                           "ncclAllGather of the slabs per step over NVLink, local saturating compose; every rank ends with all canvases"),
              "launch": "one step captured as a CUDA graph, the K timed steps replayed by one bevk_graph_launch call",
              "l2": f"inputs ({w['batch'] * w['n_cam'] * w['FW'] * w['FH'] * 3 / 1e6:.0f} MB/step) larger than L2; "
                    "the frame-invariant LUT stays L2-resident by design"}

    if a.impl == "reference":
        if rank != 0:
            return 0
        if w["n_cam"] != 4:
            print(json.dumps({"impl": "reference", "unavailable": "the reference (surroundBEV.py:285-294) is hard-wired to 4 cameras; "
                                                                 "cfg5 has no reference arm, its oracle is per-camera raw2bev + N-way compose (tests/)"}))
            return 0
        calib = synthetic_calibration(w["FW"], w["FH"], w["BW"], w["BH"])
        from oracle import cv2_path as C
        from oracle import restate as R
        g = C.Geometry(FW=w["FW"], FH=w["FH"], BW=w["BW"], BH=w["BH"], CW=250 * w["BW"] // 1000, CH=400 * w["BH"] // 1000)
        masks = [R.blend_mask(n, g.BW, g.BH, g.CW, g.CH) if w["blend"] else C.plain_mask(n, g) for n in NAMES]
        import cv2
        if os.environ.get("BEVK_REF_THREADS"):
            cv2.setNumThreads(int(os.environ["BEVK_REF_THREADS"]))
        ref = C.RefBev(calib, g, w["blend"], w["balance"], masks=masks)
        per_step = 4   # bounded sample: 4 of the 32 frame-sets per step
        sets = synthetic_frames(w["FW"], w["FH"], w["n_cam"], per_step, seed=7)
        if not os.environ.get("BEVK_REF_THREADS"):
            # give the reference every host thread it can use: probe cv2's default pool and all cores, keep the faster
            probes = {}
            for th in sorted({cv2.getNumThreads(), os.cpu_count() or 1}):
                cv2.setNumThreads(th)
                ref(*sets[0])
                t0 = time.perf_counter()
                for s_ in sets[:2]:
                    ref(*s_)
                probes[th] = time.perf_counter() - t0
            cv2.setNumThreads(min(probes, key=probes.get))
        for _ in range(max(1, a.warmup)):
            ref(*sets[0])
        t0 = time.perf_counter()
        for _ in range(a.steps):
            last = [ref(*s) for s in sets]
        dt = time.perf_counter() - t0
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, np.stack(last))
        v = a.steps * per_step / dt
        line = {"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": a.gpus, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": v, "unit": unit, "cores": cv2.getNumThreads(), "kind": "port",
                                 "sample": f"{per_step} frame-sets per step x {a.steps} steps; the reference's cv2 call "
                                           f"sequence (oracle/cv2_path.py), cv2 {cv2.__version__}, os.cpu_count()={os.cpu_count()}"},
                "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        line["cpu_frame_set_parallel"] = cpu_frame_set_parallel(ref, sets)
        line["cpu_baseline"]["frame_set_parallel"] = line["cpu_frame_set_parallel"]
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    # bind this rank to the CPUs (and, by first touch, the memory) of its GPU's NUMA node before anything is allocated
    from cameracalibration_b200 import hostpin
    try:
        cpus = hostpin.pin_to_gpu(local)
    except Exception as e:   # placement is an optimisation, never a reason to fail
        cpus = sorted(os.sched_getaffinity(0))
        print(f"[bench] NUMA pinning skipped: {e}", file=sys.stderr)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    eng, calib, masks, g = build_engine(w, local)
    stream = torch.cuda.Stream(device=dev)          # the stream the kernels are launched on (and timed on)
    eng.ctx.set_stream(stream.cuda_stream)
    nb, nc = w["batch"], w["n_cam"]
    # frames policy: every rank has its own batch; cameras policy: all ranks work on the same batch
    host = synthetic_frames(w["FW"], w["FH"], nc, nb, seed=1000 + (rank if a.shard == "frames" else 0))
    d_frames = torch.from_numpy(host).to(dev)                       # [batch][cam][FH][FW][3], resident in HBM
    fbytes = w["FW"] * w["FH"] * 3
    ptrs = torch.tensor([d_frames.data_ptr() + i * fbytes for i in range(nb * nc)], dtype=torch.int64, device=dev)
    d_out = torch.empty((nb, w["BH"], w["BW"], 3), dtype=torch.uint8, device=dev)

    from cameracalibration_b200.sharding import ShardedBev
    sharded = ShardedBev(eng, "cameras" if (a.shard != "frames" and world > 1) else "frames")
    cams = a.shard != "frames" and world > 1
    p2p = cams and a.shard == "cameras-p2p"
    d_own = torch.empty(((nb + world - 1) // world, w["BH"], w["BW"], 3), dtype=torch.uint8, device=dev) if p2p else None

    use_table = bool(os.environ.get("BEVK_BENCH_TABLE"))   # A/B switch: frames through a device pointer table (round-1 gather kernel)

    def step():
        if p2p:
            # one camera block per rank; the fused kernel stores its slabs into the owners over NVLink (bevk_bev_run_scattered)
            sharded.render_scattered(d_frames, d_own, None, stream=stream.cuda_stream)
        elif cams:
            # one camera block per rank: slabs -> ONE ncclAllGather -> compose, all on `stream` (bevk_bev_run_sharded)
            sharded.render(d_frames, d_out, None, w["balance"], stream=stream.cuda_stream)
        elif use_table:
            eng.run_device(ptrs.data_ptr(), nb, d_out.data_ptr(), 0, w["balance"])
        else:
            # the batch is one uint8[batch][cam][FH][FW][3] tensor = a frame stack: TMA-staged kernel
            eng.run_stack(d_frames.data_ptr(), fbytes, nb, d_out.data_ptr(), 0, w["balance"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(max(3, a.warmup)):
        step()
    barrier()
    # One step is captured into a CUDA graph and the K timed steps are K replays enqueued by ONE C call
    # (bevk_graph_launch): the device never waits for Python, whatever else the host is doing (8 ranks + samplers).
    graph = None
    if not cams and not use_table and not os.environ.get("BEVK_BENCH_NO_GRAPH"):
        with eng.ctx.graph_capture() as graph:
            step()
        graph.launch(3)
        barrier()
    l0 = eng.ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    if graph is not None:
        graph.launch(a.steps)
    else:
        for _ in range(a.steps):
            step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    last = (d_own if p2p else d_out).cpu().numpy() if a.dump_outputs and rank == 0 else None   # before any untimed step
    launches = eng.ctx.launches - l0
    # keep the GPU under the same load a little longer so the clock sampler sees it (untimed)
    t_end = time.time() + 1.0
    while time.time() < t_end:
        for _ in range(20):
            step()
        torch.cuda.synchronize()
    sampler.stop_flag = True
    tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_all = float(tmax.item())
    value = (nb if cams else world * nb) * a.steps / (ms_all / 1e3)

    # ---- kernel-only time of k_bev via the ctx's own events (single launch, averaged) ----
    kt = []
    for _ in range(20):
        if cams:   # render + all-gather + compose are one step: time it as a whole on the stream
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record(stream)
            step()
            eb.record(stream)
            eb.synchronize()
            kt.append(ea.elapsed_time(eb))
        else:
            step()
            kt.append(eng.last_kernel_ms())
    k_ms = float(np.median(kt))
    path_used = eng.last_path()

    # ---- end to end through the public API, pinned host frames ----
    from cameracalibration_b200 import pinned_empty
    n_e2e = a.e2e_steps or min(a.steps, 20)
    # two distinct page-locked input batches, alternated step by step (2 x 796 MB >> L2: no step can be
    # served from a cache of the previous one); the last step uses batch 0 so the result can be checked
    pin_in = pinned_empty((2, nb, nc, w["FH"], w["FW"], 3))
    pin_in[0] = host
    pin_in[1] = host[::-1]
    pin_out = pinned_empty((nb, w["BH"], w["BW"], 3))
    eng.ctx.set_stream(None)
    sets = [[[pin_in[v, b, c] for c in range(nc)] for b in range(nb)] for v in range(2)]
    for i in range(2):
        eng.run(sets[i & 1], None, w["balance"], out=pin_out)
    barrier()
    t0 = time.perf_counter()
    for i in range(n_e2e):
        eng.run(sets[(n_e2e - 1 - i) & 1], None, w["balance"], out=pin_out)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    te = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * nb * n_e2e / float(te.item())   # e2e always runs the frames policy (each rank its own batch)
    if p2p:   # the device path left this rank only the canvases it owns
        own = list(range(rank, nb, world))
        same = bool((torch.from_numpy(np.asarray(pin_out)[own]).to(dev) == d_own[:len(own)]).all().item())
    else:
        same = bool((torch.from_numpy(np.asarray(pin_out)).to(dev) == d_out).all().item())

    # ---- the reference's own call: BevGenerator.__call__(front, back, left, right), one frame-set, NumPy in / NumPy out
    e2e_api = None
    if rank == 0 and not os.environ.get("BEVK_BENCH_NO_API") and nc == 4:
        from cameracalibration_b200.SurroundBirdEyeView import surroundBEV as S
        ar = S.BevGenerator.get_args()
        saved = {k: getattr(ar, k) for k in ("FRAME_WIDTH", "FRAME_HEIGHT", "BEV_WIDTH", "BEV_HEIGHT", "CAR_WIDTH", "CAR_HEIGHT")}
        ar.FRAME_WIDTH, ar.FRAME_HEIGHT, ar.BEV_WIDTH, ar.BEV_HEIGHT = w["FW"], w["FH"], w["BW"], w["BH"]
        ar.CAR_WIDTH, ar.CAR_HEIGHT = g.CW, g.CH
        try:
            gen = S.BevGenerator(blend=w["blend"], balance=w["balance"], calib=calib)
        finally:
            for k, v in saved.items():
                setattr(ar, k, v)
        e2e_api = {"api": "BevGenerator.__call__(front, back, left, right) -> ndarray, ONE frame-set per call, as "
                          "surroundBEV.py:312-325 is used; result freshly allocated (pageable)", "unit": unit}
        for kind in ("pageable", "pinned"):
            if kind == "pageable":
                fsets = [[np.array(host[b % nb, c_]) for c_ in range(nc)] for b in range(4)]      # what cv2.imread returns
            else:
                fsets = [[pin_in[0, b % nb, c_] for c_ in range(nc)] for b in range(4)]
            for i in range(6):
                res = gen(*fsets[i & 3])
            n_api = 60
            t0 = time.perf_counter()
            for i in range(n_api):
                res = gen(*fsets[i & 3])
            dt_api = time.perf_counter() - t0
            ok = bool((res == np.asarray(pin_out[(n_api - 1) & 3 if nb > 3 else 0])).all()) if not w["balance"] else None
            e2e_api[kind] = {"value": n_api / dt_api, "ms_per_call": dt_api / n_api * 1e3, "matches_batched_path": ok}
        e2e_api["value"] = e2e_api["pageable"]["value"]
    _, d2h_set = eng.host_copy_bytes(w["balance"])
    h2d_set = eng.last_h2d_bytes() // nb                    # bytes the last bevk_bev_run call actually moved, per frame-set

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)") if "hbm_gbs" in peaks else (6650.0, "fallback")
        src_b, canvas_b = algorithmic_bytes(eng, masks, w)
        alg = (src_b + canvas_b) * nb
        # one step == one k_bev launch: its average duration over the timed region is ms/step (events on the launch stream)
        launch_ms = ms / a.steps
        achieved = alg / (launch_ms / 1e3) / 1e9
        traffic = None
        try:   # per-launch DRAM bytes of the same kernel/workload from the committed ncu --set full capture
            tj = json.load(open(os.path.join(ROOT, "profiles", "k_bev_traffic.json")))
            if tj.get("workload_batch") == nb and not cams:
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
        except Exception:
            pass
        line = {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": a.steps, "warmup": max(3, a.warmup),
                "ms_per_step": ms_all / a.steps, "higher_is_better": True, "scaling": "strong" if cams else "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": config,
                "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": nb * h2d_set,
                        "d2h_bytes_per_step": nb * d2h_set, "steps": n_e2e, "frame_bytes_per_step": nb * nc * fbytes,
                        "api": "BevEngine.run (ctypes -> bevk_bev_run), pinned host frames; without balance only the "
                               "row spans of each frame its camera's LUT can sample cross PCIe (k_fetch_spans)", "matches_device_path": same},
                "e2e_api": e2e_api,
                "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "kernel": "k_bev_tma<false,4>" if eng.last_path() == "tma" else "k_bev<false,4>",
                             "kernel_ms": launch_ms,
                             "kernel_ms_isolated": k_ms, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg,
                             "algorithmic_bytes_per_frame_set": {"source_unique_32B_sectors": src_b, "canvas_write": canvas_b}},
                "link_bytes_per_step": sharded.link_bytes() if cams else 0,
                "clocks": sampler.summary(), "plan": dict(eng.plan_info(), tma=eng.tma_plan_info(), path=path_used)}
        if not a.no_cpu_baseline and world == 1 and nc == 4:
            v, cores, sample = cpu_reference(w, calib, masks, n_sets=4, repeats=100000, seconds_cap=20.0)
            line["cpu_baseline"] = {"value": v, "unit": unit, "cores": cores, "kind": "port",
                                    "sample": sample + f"; os.cpu_count()={os.cpu_count()}",
                                    "frame_set_parallel": cpu_parallel}
        if last is not None:
            dump_outputs(a.dump_outputs, last)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
