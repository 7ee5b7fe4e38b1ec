#!/usr/bin/env python3
"""End-to-end time of getOccupiedVoxelIndices and getVoxelCenters(-1) on the 2048^3 / 10 m colour stream of tests/golden
(tools/make_golden.py LONG_CASES["L2_2048_color100"], 100 frames): the CUDA engine against the reference's own methods
(oracle/_ref/libcpu_tsdf_ref_leaves.so, compiled verbatim by oracle/leaves.mk) on the same host.

Each call is timed with a host clock around the synchronous call, so the time includes the enumeration, the sort, the
decode and the copy of the result to the host.  Every implementation is warmed up first; the median and the spread of the
repeats are reported.  The engine's arrays are checked against the restatement's and the reference's before anything is
timed.

    python tools/bench_leaves.py [--out profiles/leaves.json] [--repeat 20] [--cpu-repeat 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cpu_tsdf_b200 import synth  # noqa: E402
from oracle import leaves_py  # noqa: E402
from oracle.oracle_py import OracleVolume  # noqa: E402
from tests.common import CAM, CFG_2048, frames  # noqa: E402


def timed(fn, warmup, repeat):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(repeat):
        t0 = time.perf_counter()
        fn()
        ts.append(1e3 * (time.perf_counter() - t0))
    return {"median_ms": float(np.median(ts)), "min_ms": float(np.min(ts)), "max_ms": float(np.max(ts)), "repeat": repeat}


def gpu_conditions():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "leaves.json"))
    ap.add_argument("--repeat", type=int, default=20)
    ap.add_argument("--cpu-repeat", type=int, default=5)
    a = ap.parse_args()
    import cpu_tsdf_b200 as pkg

    eng = pkg.TSDFVolumeOctree(device=0, pool_log2=20)
    eng.setResolution(2048, 2048, 2048)
    eng.setGridSize(10.0, 10.0, 10.0)
    eng.setCameraIntrinsics(CAM.fx, CAM.fy, CAM.cx, CAM.cy)
    eng.setIntegrateColor(True)
    eng.reset()
    leaves_py.load_reference()
    orc = OracleVolume(kind="port", **CFG_2048, integrate_color=1)
    ref = OracleVolume(kind=leaves_py.KIND, **CFG_2048, integrate_color=1)
    orc.reset()
    ref.reset()
    for pose, cloud in frames(synth.S2, 100, color=True, noise_seed=12345):
        eng.integrateCloud(cloud, None, pose)
        orc.integrate(cloud, pose)
        ref.integrate(cloud, pose)
    eng.sync()

    occ, ctr = eng.getOccupiedVoxelIndices(), eng.getVoxelCenters(-1)
    for name, a_occ, a_ctr in (("restatement", leaves_py.restatement_occupied_indices(orc), leaves_py.restatement_voxel_centers(orc, -1)),
                               ("reference", leaves_py.reference_occupied_indices(ref), leaves_py.reference_voxel_centers(ref, -1))):
        assert np.array_equal(occ, a_occ), f"getOccupiedVoxelIndices differs from the {name}"
        assert np.array_equal(ctr.view(np.uint32), a_ctr.view(np.uint32)), f"getVoxelCenters(-1) differs from the {name}"
    st = eng.stats()
    out = {
        "workload": "2048^3 / 10 m colour stream, 100 frames (tests/golden L2_2048_color100)",
        "timing": "host clock around each synchronous call (includes the device-to-host copy); median / min / max of the repeats after warm-up",
        **gpu_conditions(),
        "n_occupied": int(len(occ)), "n_leaves": int(len(ctr)), "n_bricks": int(st.n_bricks),
        "result_bytes": {"occupied": int(occ.nbytes), "leaves": int(ctr.nbytes)},
        "engine": {"getOccupiedVoxelIndices": timed(eng.getOccupiedVoxelIndices, 3, a.repeat),
                   "getVoxelCenters(-1)": timed(lambda: eng.getVoxelCenters(-1), 3, a.repeat)},
        "cpu_threads": os.cpu_count(),
    }
    # one call of each method per repeat (with a NULL output the orc_* entry points run the method once and copy nothing)
    out["reference"] = {"getOccupiedVoxelIndices": timed(lambda: ref.lib.orc_occupied_indices(ref.h, None), 1, a.cpu_repeat),
                        "getVoxelCenters(-1)": timed(lambda: ref.lib.orc_voxel_centers(ref.h, -1, None), 1, a.cpu_repeat)}
    out["speedup_vs_reference"] = {k: out["reference"][k]["median_ms"] / out["engine"][k]["median_ms"] for k in out["engine"]}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
