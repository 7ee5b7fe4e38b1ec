#!/usr/bin/env python3
"""bench.py — integrateCloud frames/s @ 640x480 into 2048^3 (BASELINE.json metric).

A "step" is one pass of the hot path over one batch of FRAMES_PER_STEP synthetic 640x480 depth
frames (ICL-NUIM-shaped interior stream S2, colour on, 2048^3 / 10 m grid: BASELINE.json
configs[2]).  The JSON line carries
  value        frames/s with the clouds already resident in HBM (b200tsdf_integrate_batch_device: one
               CUDA-graph launch per step of 32 frames),
  e2e          frames/s through the public API (b200tsdf_integrate_batch_rows) from pinned HOST buffers: host packing
               to 16-byte pixels (one rank) or raw row slices + NVLink all-gather (more ranks), H2D and a D2H read of
               the per-step result inside the timed region,
  host_load_leg the device-resident leg again with every host core busy (median of three repeats),
  roofline     achieved algorithmic GB/s of the dominant kernel against the measured HBM peak,
  cpu_baseline the reference's CPU path timed on this box's host cores (bounded sample).
`--impl reference` times the CPU arm alone (oracle/_ref = the reference's own sources when they
compiled here, else the oracle port).  Under torchrun (N > 1) the volume is sharded by coarse
cell across ranks (strong scaling: every rank sees every frame and fuses its own cells).
`--dump-outputs DIR` writes the volume the timed steps left behind (see dump_outputs) so that two
builds can be compared output for output: the inputs are seeded, identical from run to run.
"""
from __future__ import annotations

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

from cpu_tsdf_b200 import synth  # noqa: E402

FRAMES_PER_STEP = 32
N_DISTINCT = 64            # distinct frames/poses cycled through (inputs 64 x 9.8 MB = 629 MB > 126 MB L2)
RES, SIZE = 2048, 10.0
CAM = synth.Camera()
SCENE = synth.S2
W, H = CAM.width, CAM.height


def make_inputs(n=N_DISTINCT, color=True):
    """The first n frames of THE bench stream (both arms cycle through the same N_DISTINCT poses / clouds)."""
    poses, clouds = [], []
    for f in range(n):
        pose = synth.orbit_pose(SCENE, f * (100 // N_DISTINCT), 100)
        poses.append(pose)
        clouds.append(synth.make_frame(SCENE, pose, CAM, color=color, noise_seed=12345, frame=f))
    return poses, clouds


class HostLoad:
    """Busy-loops on every host core (stand-in for `stress-ng --cpu $(nproc)`, which this image lacks)."""

    def __init__(self, n):
        self.n, self.procs = n, []

    def __enter__(self):
        for _ in range(self.n):
            self.procs.append(subprocess.Popen([sys.executable, "-c", "while True: pass"]))
        time.sleep(2.0)                      # 128 interpreters booting at once are a fork storm, not the steady load that is meant
        return self

    def __exit__(self, *a):
        for p in self.procs:
            p.kill()
        for p in self.procs:
            p.wait()


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu=0):
        self.rows, self.proc, self.gpu = [], None, gpu

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa(gpu):
    """Run this process (and first-touch its pinned buffers) on the CPU cores local to the GPU: on a two-socket host a
    pinned buffer on the far socket costs a large part of the PCIe bandwidth the end-to-end leg is bound by."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1]
        avail = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in avail]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} GPU-local cores ({cpus[0]}..{cpus[-1]})"
    except Exception as e:            # no NVML, a container without the call, ...: keep the default placement
        return f"default ({type(e).__name__})"
    return "default"


DUMP_NODES = 1 << 20       # sampled nodes: 12 float32 values each = 48 MiB of .npy files


def dump_outputs(out_dir, nodes, n_updates):
    """What a caller of the timed path reads back after its last step, as float32 .npy files: every node array of the
    volume's node dump (keys = level, x, y, z; {sdf, weight}; split flag; rgb; variance state) at a fixed, seeded sample of
    DUMP_NODES node indices (every node when there are fewer; the dump is in octree order), and summary.npy = [number of
    nodes, voxel updates of the last frame].  Every integer written is below 2^24, so float32 holds it exactly."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(nodes["keys"])
    idx = np.arange(n) if n <= DUMP_NODES else np.sort(np.random.default_rng(0).choice(n, DUMP_NODES, replace=False))
    for name in ("keys", "dw", "split", "rgb", "M", "ns"):
        np.save(os.path.join(out_dir, name + ".npy"), nodes[name][idx].astype(np.float32))
    np.save(os.path.join(out_dir, "summary.npy"), np.array([n, n_updates], np.float64))


def oracle_volume(kind):
    from oracle.oracle_py import OracleVolume
    return OracleVolume(kind=kind, xres=RES, yres=RES, zres=RES, xsize=SIZE, ysize=SIZE, zsize=SIZE,
                        cx=CAM.cx, cy=CAM.cy, integrate_color=1)


def cpu_arm(poses, clouds, nframes, threads_list, kind=None):
    """Time the reference's CPU integrateCloud on the host cores: warm the volume with a few frames,
    then time `nframes` frames (integrateCloud only).  Best thread count wins (BASELINE.md §3)."""
    from oracle import oracle_py
    if kind is None:
        kind = "reference" if os.path.exists(oracle_py.REF_LIB) else "port"
    best = None
    for nt in threads_list:
        os.environ["OMP_NUM_THREADS"] = str(nt)
        v = oracle_volume(kind)
        v.cfg.num_threads = nt
        v.lib.orc_destroy(v.h)
        import ctypes
        v.h = v.lib.orc_create(ctypes.byref(v.cfg))
        v.reset()
        for i in range(2):
            v.integrate(clouds[i % len(clouds)], poses[i % len(poses)])
        t0 = time.perf_counter()
        for i in range(2, 2 + nframes):
            v.integrate(clouds[i % len(clouds)], poses[i % len(poses)])
        dt = time.perf_counter() - t0
        fps = nframes / dt
        if best is None or fps > best["value"]:
            best = {"value": fps, "cores": nt}
    best.update({"unit": "frames/s", "kind": "reference" if kind == "reference" else "port",
                 "sample": f"{nframes} frames of the same 640x480 S2 stream into 2048^3/10 m, colour on, after 2 warm-up frames; best of threads {threads_list}"})
    return best


def run_reference(args, rank, world):
    if rank != 0:
        return
    frames_per_step = 4
    n_need = min(N_DISTINCT, 3 + (args.warmup + args.steps) * frames_per_step)
    poses, clouds = make_inputs(n_need)
    ND = len(clouds)
    nproc = os.cpu_count() or 1
    from oracle import oracle_py
    kind = "reference" if os.path.exists(oracle_py.REF_LIB) else "port"
    import ctypes

    def make(nt):
        os.environ["OMP_NUM_THREADS"] = str(nt)
        v = oracle_volume(kind)
        v.cfg.num_threads = nt
        v.lib.orc_destroy(v.h); v.h = v.lib.orc_create(ctypes.byref(v.cfg))
        v.reset()
        return v

    # the reference's OpenMP update loop scales poorly (BASELINE.md §2): give it the thread count it runs best with
    nt = int(os.environ.get("B200TSDF_REF_THREADS", "0"))
    if not nt:
        best = None
        for cand in sorted({1, 2, 4, 8, 16, nproc}):
            if cand > nproc:
                continue
            pv = make(cand)
            pv.integrate(clouds[0], poses[0])
            t0 = time.perf_counter()
            for i in (1, 2):
                pv.integrate(clouds[i], poses[i])
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, cand)
            del pv
        nt = best[1]
    v = make(nt)
    k = 0
    for _ in range(args.warmup):
        for _ in range(frames_per_step):
            v.integrate(clouds[k % ND], poses[k % ND]); k += 1
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for _ in range(frames_per_step):
            v.integrate(clouds[k % ND], poses[k % ND]); k += 1
    dt = time.perf_counter() - t0
    fps = args.steps * frames_per_step / dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, v.dump_nodes(), v.stats().n_add_observation)
    line = {
        "impl": "reference", "metric": "integrateCloud frames/s @ 640x480 into 2048^3", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(frames_per_step, args.gpus),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": nt, "kind": kind,
                         "sample": f"{frames_per_step} frames per step of the 640x480 S2 stream into 2048^3/10 m, colour on"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(frames_per_step, n_gpus):
    return {"workload": "ICL-NUIM-shaped synthetic 640x480 stream (scene S2: 4 m room seen from inside, sigma(z) depth noise), "
                        "2048^3 voxels over 10 m, colour on (BASELINE.json configs[2] integrate leg)",
            "frames_per_step": frames_per_step, "image": [W, H], "grid": RES, "grid_size_m": SIZE,
            "point_bytes": 32, "distinct_frames": N_DISTINCT,
            "l2": "inputs larger than L2 (64 distinct frames = 629 MB device-resident, orbit covers a >126 MB brick working set)",
            "parallelism": "1 GPU" if n_gpus == 1 else f"volume sharded by coarse cell over {n_gpus} GPUs, every rank integrates every frame "
                           f"(end to end: each rank uploads 1/{n_gpus} of every frame, NVLink all-gather)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-host-load", action="store_true", help="skip the leg that repeats the device-resident measurement with all host cores busy")
    ap.add_argument("--pool-log2", type=int, default=18, help="brick pool capacity = 2^N slots (the bench scene allocates ~37k bricks)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the volume they left as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs a single rank: each rank of a sharded run holds only its own cells")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import cpu_tsdf_b200 as pkg
    from cpu_tsdf_b200.build import build_library
    build_library()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    all_cpus = os.sched_getaffinity(0)
    affinity = bind_to_gpu_numa(local_rank) if os.environ.get("B200TSDF_BIND_NUMA") == "1" else "default (unbound)"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    poses, clouds = make_inputs()
    vol = pkg.TSDFVolumeOctree(device=local_rank, pool_log2=args.pool_log2, shard_rank=rank, shard_count=world)
    vol.setGridSize(SIZE, SIZE, SIZE)
    vol.setResolution(RES, RES, RES)
    vol.setCameraIntrinsics(CAM.fx, CAM.fy, CAM.cx, CAM.cy)
    vol.setIntegrateColor(True)
    vol.reset()

    # device-resident inputs (torch owns the memory; the engine reads it through the C ABI)
    d_clouds = [torch.from_numpy(c).cuda() for c in clouds]
    # pinned host inputs for the end-to-end leg: a rank's host memory holds only ITS row slice of every frame (at N = 1 the
    # whole frame); the library uploads the slice over this GPU's PCIe link and all-gathers the frame over NVLink
    if world > 1:
        ids = [pkg.TSDFVolumeOctree.commUniqueId() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        vol.commInit(ids[0], rank, world)
    row0, row1 = vol.rowSlice(H)
    h_rows = [torch.from_numpy(np.ascontiguousarray(c[row0:row1])).pin_memory() for c in clouds]
    h_ptrs = [t.data_ptr() for t in h_rows]
    torch.cuda.synchronize()
    stride = 32

    d_ptrs = [t.data_ptr() for t in d_clouds]

    def step_device(k0):
        # one step = FRAMES_PER_STEP consecutive integrateCloud calls submitted as ONE batch: one record upload + one CUDA-graph launch
        idx = [(k0 + j) % N_DISTINCT for j in range(FRAMES_PER_STEP)]
        vol.integrateBatchDevice([d_ptrs[i] for i in idx], H, W, stride, [poses[i] for i in idx], rgba_off=16)

    def step_device_frames(k0):
        # the same frames one integrateCloud call (4 kernel launches) at a time: the path whose dominant kernel CUDA events can bracket
        for j in range(FRAMES_PER_STEP):
            i = (k0 + j) % N_DISTINCT
            vol.integrateCloudDevice(d_ptrs[i], H, W, stride, poses[i], rgba_off=16)

    def step_host(k0):
        # public API with HOST buffers: slice upload (H2D) + NVLink all-gather + one graph launch for the step's 32 frames
        idx = [(k0 + j) % N_DISTINCT for j in range(FRAMES_PER_STEP)]
        vol.integrateBatchRows([h_ptrs[i] for i in idx], H, W, stride, [poses[i] for i in idx], rgba_off=16)
        return vol.stats().n_updates         # D2H read of the step's result (synchronizes)

    def timed(step_fn, steps):
        nonlocal k
        barrier()
        vol.profile_begin()
        for _ in range(steps):
            step_fn(k); k += FRAMES_PER_STEP
        prof = vol.profile_end()
        barrier()
        ms = torch.tensor([prof.ms_elapsed], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return prof, float(ms.item())

    # ---- device-resident leg (headline `value`): batched graph launches ------------------------
    # (nvidia-smi needs ~0.2 s to start: sample from before the warm-up to after the end-to-end leg)
    sampler = ClockSampler(local_rank); sampler.start()
    time.sleep(0.4)
    k = 0
    for _ in range(args.warmup):
        step_device(k); k += FRAMES_PER_STEP
    vol.sync()
    prof, ms_total = timed(step_device, args.steps)
    nframes = args.steps * FRAMES_PER_STEP
    value = nframes / (ms_total / 1e3)
    if args.dump_outputs:                                      # before the legs below integrate more frames into the volume
        dump_outputs(args.dump_outputs, vol.download_nodes(), vol.stats().n_updates)

    # ---- the same work one frame per call, the dominant kernel bracketed by CUDA events (roofline leg) ----
    for _ in range(2):
        step_device_frames(k); k += FRAMES_PER_STEP
    prof_f, ms_frames = timed(step_device_frames, args.steps)

    # ---- end-to-end leg (host buffers, public API) ---------------------------------------------
    host_pack = os.environ.get("B200TSDF_HOST_PACK", "1" if world <= 1 else "0") != "0"     # the library's own default (multigpu.cuh)
    pack_threads = int(os.environ.get("B200TSDF_PACK_THREADS", "0")) or max(1, min(16, (os.cpu_count() or 1) // (2 * world)))
    for _ in range(max(1, args.warmup // 2)):
        step_host(k); k += FRAMES_PER_STEP
    barrier()
    vol.profile_begin()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host(k); k += FRAMES_PER_STEP
    prof_e = vol.profile_end()
    wall = time.perf_counter() - t0
    barrier()
    clocks = sampler.stop()
    e2e_ms = torch.tensor([max(prof_e.ms_elapsed, wall * 1e3)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = nframes / (float(e2e_ms.item()) / 1e3)

    # ---- the batched leg again with every host core busy (a library must not depend on an idle host); last, so that
    #      the 128 busy loops do not colour the end-to-end leg ----
    host_load = None
    if not args.no_host_load:
        import contextlib
        with (HostLoad(os.cpu_count() or 1) if rank == 0 else contextlib.nullcontext()):
            step_device(k); k += FRAMES_PER_STEP
            vol.sync()
            n_loaded = args.steps
            loaded = []
            for _ in range(3):                                 # three repeats: a descheduled submitting thread shows as an outlier, not as the figure
                _, ms_loaded = timed(step_device, n_loaded)
                loaded.append(n_loaded * FRAMES_PER_STEP / (ms_loaded / 1e3))
        host_load = {"value": sorted(loaded)[1], "unit": "frames/s", "steps": n_loaded, "repeats": loaded, "statistic": "median of 3 repeats",
                     "load": f"{os.cpu_count()} busy-loop processes (one per host core) during the batched device-resident leg"}

    # ---- roofline of the dominant kernel -----------------------------------------------------------
    upd = torch.tensor([prof.n_updates], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(upd, op=dist.ReduceOp.SUM)
    peak, peak_src = measured_peaks()

    def alg_bytes(pr):
        # algorithmic bytes (SURVEY.md §8d): 4 W H (depth) + N_upd * (8 read + 8 write) [+ (4+4) with colour]
        return 4.0 * W * H * pr.n_frames + pr.n_updates * (16.0 + 8.0)

    # single-frame figure: CUDA-event pairs around k_bricks on the engine's stream, one frame per call
    achieved = alg_bytes(prof_f) / (prof_f.ms_kernel / 1e3) / 1e9 if prof_f.ms_kernel > 0 else 0.0
    # batched figure (BASELINE.md §3.4): the same kernel inside the 32-frame graph launches of the headline leg, timed on the device
    # (%globaltimer, first block start -> last block end; no event can be placed inside a replayed graph)
    batched = None
    if prof.kernel_launches_device > 0 and prof.ms_kernel_device > 0:
        a_b = alg_bytes(prof) * (prof.kernel_launches_device / max(1, prof.n_frames)) / (prof.ms_kernel_device / 1e3) / 1e9
        batched = {"frames_per_graph_launch": FRAMES_PER_STEP, "achieved": a_b, "frac": a_b / peak,
                   "us_per_launch": 1e3 * prof.ms_kernel_device / prof.kernel_launches_device,
                   "launches_timed": int(prof.kernel_launches_device), "timer": "%globaltimer inside k_bricks"}
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if world == 1 and os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    st_last = vol.stats()
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic,
                "traffic_source": "ncu --set full capture of this kernel on this workload at N=1 (profiles/traffic.json); not measured at N>1",
                "peak_source": peak_src, "kernel": "k_bricks (one warp per interior 8^3 block, brick updated in place)",
                "bytes_per_launch": alg_bytes(prof_f) / max(1, prof_f.kernel_launches),
                "us_per_launch": 1e3 * prof_f.ms_kernel / max(1, prof_f.kernel_launches),
                "us_per_launch_device_timer": 1e3 * prof_f.ms_kernel_device / max(1, prof_f.kernel_launches_device),
                "updates_per_frame": prof_f.n_updates / max(1, prof_f.n_frames),
                "frames_per_s_one_call_per_frame": nframes / (ms_frames / 1e3),
                "batched": batched,
                "blocks_last_frame": int(st_last.n_block_visits), "bricks_allocated": int(st_last.n_bricks),
                "general_path_last_frame": {"upper_slow_folds": int(st_last.reserved), "upper_slow_visits": int(st_last.n_slow_visits)}}

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            os.sched_setaffinity(0, all_cpus)                 # the CPU arm gets every host core again
            nproc = os.cpu_count() or 1
            tl = sorted({1, min(4, nproc), nproc})
            cpu = cpu_arm(poses, clouds, 12, tl)
        line = {
            "metric": "integrateCloud frames/s @ 640x480 into 2048^3", "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(FRAMES_PER_STEP, world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "frames/s",
                    "h2d_bytes_per_step": int(prof_e.h2d_bytes // args.steps), "d2h_bytes_per_step": int(prof_e.d2h_bytes // args.steps),
                    "nvlink_bytes_per_step": int(prof_e.nvlink_bytes // args.steps),
                    "path": ("b200tsdf_integrate_batch_rows: host threads pack each rank's rows [%d, %d) of every 32 B/point frame to 16 B pixels into pinned "
                             "staging (bit-preserving), only those cross PCIe; NCCL all-gather over NVLink at N>1; one graph launch per pipeline stage of 1-2 frames"
                             if host_pack else
                             "b200tsdf_integrate_batch_rows: each rank uploads rows [%d, %d) of every frame from pinned host memory, packs to 16 B pixels on the device, "
                             "NCCL all-gather over NVLink, one graph launch per chunk of 8 frames") % (row0, row1),
                    "host_pack": {"enabled": host_pack, "threads": pack_threads if host_pack else 0,
                                  "input_bytes_per_step": int(FRAMES_PER_STEP * (row1 - row0) * W * stride)},
                    "timing": "max(CUDA events on the engine stream, host wall clock) over ranks", "host_affinity": affinity},
            "gpu_launches": int(prof.total_launches),
            "graph_launches": int(prof.graph_launches),
            "host_load_leg": host_load,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "updates_total": float(upd.item()),
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
