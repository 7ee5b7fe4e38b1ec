"""Pins the CPU restatement (oracle/tsdf_oracle.cpp) against THE REFERENCE'S OWN SOURCES: octree structure, split/prune
history, per-node state, ray-march, query arithmetic, mesher traversal and .vol layout, bit for bit.

Each test runs its scenario through the restatement and compares what it observes with what the same scenario gave when run
through the reference's sources compiled verbatim against the Eigen/PCL compatibility layer in oracle/compat (oracle/Makefile
`ref`).  Those observations (SHA-256 digests of every compared array, and the counts and configuration values) are stored in
tests/golden/ref_pins.json; tools/make_ref_pins.py regenerates them where the reference sources are available."""
import json
import os
import tempfile

import numpy as np
import pytest

from cpu_tsdf_b200 import synth
from oracle import oracle_py
from oracle.oracle_py import OracleVolume
from tests.common import CFG_256, CFG_512, CFG_2048, frames, query_points, sha, sha_values

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pins.json")


def golden(key):
    return json.load(open(GOLDEN))[key]


def volume(kind, cfg, **kw):
    v = OracleVolume(kind=kind, **cfg, **kw)
    v.reset()
    return v


def node_digests(d, *, rgb=False, var=False):
    """What tests.common.assert_same_nodes compares: structure, split flags, {sdf, weight} bits [, rgb] [, variance state]."""
    out = {"n_nodes": int(len(d["keys"])), "keys": sha(d["keys"]), "split": sha(d["split"]), "dw": sha(d["dw"].view(np.uint32))}
    if rgb:
        out["rgb"] = sha(d["rgb"])
    if var:
        out["M"], out["ns"] = sha(d["M"].view(np.uint32)), sha(d["ns"])
    return out


def observe_defaults(kind):
    c = oracle_py.OrcConfig()
    oracle_py.load(kind).orc_default_config(c)
    out = {}
    for name, _ in oracle_py.OrcConfig._fields_:
        if name in ("num_threads",):
            continue
        v = getattr(c, name)
        out[name] = list(v) if hasattr(v, "__len__") else v
    return out


def test_defaults_match_reference_constructor():
    assert observe_defaults("port") == golden("defaults")


INTEGRATE_CASES = [
    (CFG_256, synth.S1, 5, 9, True),
    (CFG_512, synth.S1, 4, 13, False),
    (CFG_2048, synth.S2, 2, 3, True),
]


def integrate_key(cfg, scene, n, stride, color):
    return f"integrate[{cfg['xres']}-{'S1' if scene is synth.S1 else 'S2'}-{n}-{stride}-{color}]"


def observe_integrate(kind, cfg, scene, n, stride, color):
    v = volume(kind, cfg, integrate_color=int(color))
    for pose, cloud in frames(scene, n, stride=stride, color=color, noise_seed=7, dropout=0.01):
        v.integrate(cloud, pose)
    return {"levels": list(v.levels()), **node_digests(v.dump_nodes(), rgb=color, var=True)}


@pytest.mark.parametrize("cfg,scene,n,stride,color", INTEGRATE_CASES)
def test_integrate_structure_and_state(cfg, scene, n, stride, color):
    assert observe_integrate("port", cfg, scene, n, stride, color) == golden(integrate_key(cfg, scene, n, stride, color))


def file_digest(v, tmp_dir):
    p = os.path.join(tmp_dir, "v.vol")
    assert v.save(p) == 0
    b = open(p, "rb").read()
    return b, {"vol": sha(np.frombuffer(b, np.uint8)), "vol_bytes": len(b)}


def observe_cull_queries_render_mesh_vol(kind, tmp_dir):
    v = volume(kind, CFG_256, integrate_color=1)
    for pose, cloud in frames(synth.S1, 5, stride=7, color=True, noise_seed=5):
        v.integrate(cloud, pose)
    out = {}
    for f in (0, 19, 44):
        mask, kept = v.frustum_cull(synth.orbit_pose(synth.S1, f, 100))
        out[f"cull@{f}"], out[f"cull_kept@{f}"] = sha(mask), int(kept)
    pts = query_points()
    for mode in (0, 1):
        q = v.query(pts, 7, mode)
        out[f"query{mode}_ok"] = sha(q[3])
        for k in range(3):
            out[f"query{mode}_{k}"] = sha(q[k][q[3]].view(np.uint32))
    pose = synth.orbit_pose(synth.S1, 10, 100)
    r, c = v.render(pose, 2, colored=True)
    assert np.isfinite(r[..., 2]).sum() > 20000
    out["render2_xyz"], out["render2_normal"], out["render2_rgb"] = sha_values(r[..., :3]), sha_values(r[..., 4:7]), sha(c)
    out["render4"] = sha_values(v.render(pose, 4)[..., :7])
    for cm, wmin in ((0, 2.0), (1, 0.0), (2, 2.5)):
        verts, col = v.mesh(wmin, cm)
        assert len(verts) > 3000
        out[f"mesh{cm}@{wmin}"] = sha_values(verts)           # in order: the octree is walked depth-first
        out[f"mesh{cm}@{wmin}_rgb"] = None if col is None else sha(col)
    out.update(file_digest(v, tmp_dir)[1])
    return out


def test_cull_queries_render_mesh_vol(tmp_path):
    assert observe_cull_queries_render_mesh_vol("port", str(tmp_path)) == golden("cull_queries_render_mesh_vol")


def observe_rgb_normalized(kind, tmp_dir):
    v = volume(kind, CFG_256, integrate_color=1, color_mode=1)
    for pose, cloud in frames(synth.S1, 5, stride=7, color=True, noise_seed=5):
        v.integrate(cloud, pose)
    d = v.dump_nodes()
    out = node_digests(d, rgb=True, var=True)
    out["rgbn"] = sha(d["rgbn"].view(np.uint32))
    seen = d["dw"][:, 1] > 0
    assert seen.sum() > 50000 and np.nanmax(d["rgbn"][seen][:, 3]) > 100        # intensities are accumulated
    # unit colour direction wherever the pixel colour was not black (black gives 0/0 = NaN, as in the reference)
    rgb_dir = d["rgbn"][seen][:, :3]; ok = np.isfinite(rgb_dir).all(1)
    assert ok.sum() > 0.9 * seen.sum() and np.abs(np.linalg.norm(rgb_dir[ok], axis=1) - 1).max() < 0.2
    r, c = v.render(synth.orbit_pose(synth.S1, 10, 100), 4, colored=True)
    assert c.any()
    out["render4_xyz"], out["render4_rgb"] = sha_values(r[..., :3]), sha(c)
    verts, col = v.mesh(0.0, 1)
    assert len(verts) > 3000
    out["mesh"], out["mesh_rgb"] = sha(verts.view(np.uint32)), sha(col)
    b, fd = file_digest(v, tmp_dir)
    assert b"RGBNormalized\n#OCTREEBINARY\n" in b
    out.update(fd)
    # and the plain "RGB" mode is untouched by the new field
    w = volume(kind, CFG_256, integrate_color=1, color_mode=0)
    pose, cloud = next(frames(synth.S1, 1, color=True))
    w.integrate(cloud, pose)
    d = w.dump_nodes()
    assert "rgbn" not in d
    out["rgb_mode_rgb"] = sha(d["rgb"])
    return out


def test_rgb_normalized_voxels_match_the_reference(tmp_path):
    """setColorMode("RGBNormalized") (tsdf_volume_octree.h:290, octree.cpp:378-433): normalised colour + intensity averages
    per node, getRGB's float -> uint8 conversions, and the serializer that writes the first byte of each float.
    (Restatement only so far: the CUDA engine implements colour mode "RGB".)"""
    assert observe_rgb_normalized("port", str(tmp_path)) == golden("rgb_normalized")


def observe_get_tsdf_value(kind):
    v = volume(kind, CFG_256)
    for pose, cloud in frames(synth.S1, 3, stride=9, noise_seed=5):
        v.integrate(cloud, pose)
    pts = _interp_points()
    out = {}
    for vin in (True, False):
        val, ok = v.interpolate(pts, vin)
        out[f"valid_in={vin}"], out[f"values_in={vin}"] = sha(ok), sha(val.view(np.uint32))
    assert ok.sum() == 0 and v.interpolate(pts, True)[1].sum() > 500 and np.isnan(val).sum() > 100
    return out


def test_get_tsdf_value_matches_the_reference():
    """getTSDFValue / interpolateTrilinearly (cpp:454-541; protected in the reference, reached through a derived accessor in the
    verbatim build): values bit-equal, NaN pattern and the in/out `valid` flag equal — inside, on the border layer, outside."""
    assert observe_get_tsdf_value("port") == golden("get_tsdf_value")


def _interp_points():
    rng = np.random.default_rng(3)
    vs = 3.0 / 256
    near = rng.normal(size=(3000, 3)); near *= 0.35 / np.linalg.norm(near, axis=1, keepdims=True); near += rng.normal(scale=0.01, size=near.shape)
    border = rng.uniform(-1.5, 1.5, (600, 3)); border[:, 0] = np.where(rng.random(600) < 0.5, -1.5 + vs * rng.uniform(0, 2, 600), 1.5 - vs * rng.uniform(0, 2, 600))
    outside = rng.uniform(-2.0, 2.0, (400, 3))
    nan = np.array([[np.nan, 0, 0], [0, 0, np.nan]])
    return np.concatenate([near, border, outside, nan]).astype(np.float32)


def observe_all(kind):
    """Every observation above, keyed as in tests/golden/ref_pins.json."""
    with tempfile.TemporaryDirectory() as tmp:
        out = {"defaults": observe_defaults(kind)}
        for case in INTEGRATE_CASES:
            out[integrate_key(*case)] = observe_integrate(kind, *case)
        out["cull_queries_render_mesh_vol"] = observe_cull_queries_render_mesh_vol(kind, tmp)
        out["rgb_normalized"] = observe_rgb_normalized(kind, tmp)
        out["get_tsdf_value"] = observe_get_tsdf_value(kind)
    return out
