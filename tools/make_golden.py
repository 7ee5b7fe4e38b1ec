#!/usr/bin/env python3
"""Generate tests/golden/ref_digests.json from THE REFERENCE'S OWN SOURCES (oracle/_ref, built by
`make -C oracle ref` where /root/reference exists).  Each case runs a seeded synthetic sequence
through the reference and records SHA-256 digests of its node dump, query results, render and
mesh, plus a few scalar facts.  tests/test_golden.py replays the cases through the restatement
(CPU) and the CUDA engine (GPU) and requires identical digests."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cpu_tsdf_b200 import synth  # noqa: E402
from tests.common import CAM, frames, query_points, canon_soup, sha  # noqa: E402

CASES = {
    "c1_256_single": dict(cfg=dict(xres=256, yres=256, zres=256, cx=CAM.cx, cy=CAM.cy), scene="S1", n=1, stride=1, color=False, noise=None),
    "c2_512_orbit": dict(cfg=dict(xres=512, yres=512, zres=512, cx=CAM.cx, cy=CAM.cy), scene="S1", n=6, stride=15, color=False, noise=2),
    "c3_2048_color": dict(cfg=dict(xres=2048, yres=2048, zres=2048, xsize=10.0, ysize=10.0, zsize=10.0, cx=CAM.cx, cy=CAM.cy), scene="S2", n=3, stride=2, color=True, noise=4),
    "c4_256_color_noise": dict(cfg=dict(xres=256, yres=256, zres=256, cx=CAM.cx, cy=CAM.cy), scene="S1", n=5, stride=7, color=True, noise=5),
}


# BASELINE.json lengths (VERDICT r1: the long histories — prune-then-resplit, weight saturation — were only self-checked):
# configs[1] = 100-frame orbit into 512^3 with renderView at frames 0/25/50/75; configs[2] = >= 100 frames of the 2048^3 colour
# stream with marching cubes at w_min 2 (README.md:47) and 0 (integrate.cpp:336).  Node digests are also taken mid-stream.
LONG_CASES = {
    "L1_512_orbit100": dict(cfg=dict(xres=512, yres=512, zres=512, cx=CAM.cx, cy=CAM.cy), scene="S1", n=100, stride=1, color=False, noise=2,
                            checkpoints=(25, 50, 75, 100), render_frames=(0, 25, 50, 75), render_ds=2, mesh_wmin=(2.0,)),
    "L2_2048_color100": dict(cfg=dict(xres=2048, yres=2048, zres=2048, xsize=10.0, ysize=10.0, zsize=10.0, cx=CAM.cx, cy=CAM.cy), scene="S2", n=100,
                             stride=1, color=True, noise=12345, checkpoints=(50, 100), render_frames=(99,), render_ds=4, mesh_wmin=(2.0, 0.0)),
    # a camera that does not move: every voxel in view saturates at max_weight (octree.cpp:156-159) and keeps averaging
    "L3_256_static120": dict(cfg=dict(xres=256, yres=256, zres=256, cx=CAM.cx, cy=CAM.cy), scene="S1", n=120, stride=0, color=True, noise=9,
                             checkpoints=(60, 120), render_frames=(0,), render_ds=2, mesh_wmin=(2.0,)),
}


def run_case(vol_factory, case):
    """vol_factory(cfg, color) -> object with integrate/dump_nodes/query/render/mesh (oracle-style API)."""
    scene = getattr(synth, case["scene"])
    v = vol_factory(case["cfg"], case["color"])
    for pose, cloud in frames(scene, case["n"], stride=case["stride"], color=case["color"], noise_seed=case["noise"]):
        v.integrate(cloud, pose)
    d = v.dump_nodes()
    out = {"n_nodes": int(len(d["keys"])), "nodes": sha(d["keys"], d["dw"], d["split"], d["rgb"] if case["color"] else np.zeros(0))}
    pts = query_points(n=2000, extent=0.45 * case["cfg"].get("xsize", 3.0), radius=0.35 if case["scene"] == "S1" else 1.9)
    for mode in (0, 1):
        val, grad, hess, ok = v.query(pts, 7, mode)
        out[f"query{mode}"] = sha(ok, val[ok], grad[ok], hess[ok])
        out[f"query{mode}_ok"] = int(ok.sum())
    pose = synth.orbit_pose(scene, 10, 100)
    r = v.render(pose, 4)
    out["render"] = sha(np.nan_to_num(r[..., :3], nan=-7.0), np.nan_to_num(r[..., 4:7], nan=-7.0))
    out["render_hits"] = int(np.isfinite(r[..., 2]).sum())
    verts, cols = v.mesh(2.0, 1 if case["color"] else 0)
    out["mesh"] = sha(canon_soup(verts, cols))
    out["mesh_verts"] = int(len(verts))
    return out


def run_long_case(vol_factory, case):
    scene = getattr(synth, case["scene"])
    v = vol_factory(case["cfg"], case["color"])
    out = {}
    for f, (pose, cloud) in enumerate(frames(scene, case["n"], stride=case["stride"], color=case["color"], noise_seed=case["noise"])):
        v.integrate(cloud, pose)
        if f + 1 in case["checkpoints"]:
            d = v.dump_nodes()
            out[f"nodes@{f + 1}"] = sha(d["keys"], d["dw"], d["split"], d["rgb"] if case["color"] else np.zeros(0))
            out[f"n_nodes@{f + 1}"] = int(len(d["keys"]))
            out[f"max_weight@{f + 1}"] = float(d["dw"][:, 1].max())
    for f in case["render_frames"]:
        r = v.render(synth.orbit_pose(scene, f * case["stride"], 100), case["render_ds"])
        out[f"render@{f}"] = sha(np.nan_to_num(r[..., :3], nan=-7.0), np.nan_to_num(r[..., 4:7], nan=-7.0))
        out[f"render_hits@{f}"] = int(np.isfinite(r[..., 2]).sum())
    for wmin in case["mesh_wmin"]:
        verts, cols = v.mesh(wmin, 1 if case["color"] else 0)
        out[f"mesh@{wmin}"] = sha(np.asarray(verts, np.float32), cols if cols is not None else np.zeros(0))     # the reference's own triangle order
        out[f"mesh_verts@{wmin}"] = int(len(verts))
    return out


def main():
    from oracle import oracle_py
    from oracle.oracle_py import OracleVolume
    if not os.path.exists(oracle_py.REF_LIB):
        raise SystemExit("oracle/_ref is not built: run `make -C oracle ref` where /root/reference exists")

    def factory(cfg, color):
        v = OracleVolume(kind="reference", integrate_color=int(color), **cfg)
        v.reset()
        return v

    out = {"generator": "tools/make_golden.py", "source": "oracle/_ref = /root/reference/src/lib/*.cpp compiled verbatim (sdmiller/cpu_tsdf @ 9b973cb)",
           "cases": {name: run_case(factory, c) for name, c in CASES.items()},
           "long_cases": {name: run_long_case(factory, c) for name, c in LONG_CASES.items()}}
    path = os.path.join(ROOT, "tests", "golden", "ref_digests.json")
    json.dump(out, open(path, "w"), indent=1, sort_keys=True)
    print("wrote", path)
    for k, v in out["cases"].items():
        print(k, v["n_nodes"], v["render_hits"], v["mesh_verts"])
    for k, v in out["long_cases"].items():
        print(k, {a: b for a, b in v.items() if not isinstance(b, str)})


if __name__ == "__main__":
    main()
