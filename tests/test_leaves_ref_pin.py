"""Pins the restatement's getVoxelCenters / getOccupiedVoxelIndices / isEmpty (oracle/leaves_py.py over the tree of
oracle/tsdf_oracle.cpp) against the reference's own methods (tsdf_volume_octree.cpp:576-609, h:283-287) compiled verbatim
in oracle/_ref (oracle/leaves.mk).

Each scenario runs through the restatement and is compared with what the same scenario gave through the reference:
SHA-256 digests of the centres (bit patterns, in order) for every nlevels of the sweep, of the occupied voxel indices, and
the counts.  Those observations are stored in tests/golden/ref_pins_leaves.json; `tools/make_ref_pins.py --leaves`
regenerates them where the reference sources are available."""
import json
import os

import numpy as np
import pytest

from cpu_tsdf_b200 import synth
from oracle import leaves_py
from oracle.oracle_py import OracleVolume
from tests.common import CFG_256, frames, sha
from tests.test_ref_pin import INTEGRATE_CASES, integrate_key

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pins_leaves.json")

# max_dist_pos < max_dist_neg: the return code of updateVoxel lets coarse cells take observations whose stored d is below 1
# (hpp:209-214), so getOccupiedVoxelIndices also returns the index of the centre of unsplit coarse leaves
ASYMMETRIC_CASE = (dict(CFG_256, max_dist_pos=0.01, max_dist_neg=0.05), synth.S1, 5, 9, False)


def sweep(coarse, finest):
    """nlevels values exercised: the root, the virtual levels above the coarse depth, the coarse depth and the stored levels
    below it, the finest level, beyond it, and no limit"""
    return sorted({-1, 0, 1, 4, coarse - 1, coarse, coarse + 1, finest, finest + 3})


def methods(kind):
    """(getVoxelCenters, getOccupiedVoxelIndices, isEmpty) of the restatement ("port") or of the reference"""
    if kind == "port":
        return leaves_py.restatement_voxel_centers, leaves_py.restatement_occupied_indices, leaves_py.restatement_is_empty
    return leaves_py.reference_voxel_centers, leaves_py.reference_occupied_indices, leaves_py.reference_is_empty


def oracle_volume(kind, **kw):
    if kind != "port":
        leaves_py.load_reference()
    v = OracleVolume(kind="port" if kind == "port" else leaves_py.KIND, **kw)
    v.reset()
    return v


def observe(kind, v):
    centers, occupied, is_empty = methods(kind)
    coarse, finest = v.levels()
    out = {"levels": [coarse, finest], "is_empty": is_empty(v)}
    for n in sweep(coarse, finest):
        c = centers(v, n)
        out[f"centers[{n}]"] = {"n": int(len(c)), "sha": sha(c.view(np.uint32))}
    occ = occupied(v)
    out["occupied"] = {"n": int(len(occ)), "sha": sha(occ)}
    return out


def coarse_leaves_occupied(v):
    d = v.dump_nodes()
    coarse, _ = v.levels()
    dd, w = d["dw"][:, 0], d["dw"][:, 1]
    return int(((d["keys"][:, 0] == coarse) & (d["split"] == 0) & (w > 0) & (np.abs(dd.astype(np.float64)) < 1)).sum())


def scenario_volume(kind, cfg, scene, n, stride, color):
    v = oracle_volume(kind, **cfg, integrate_color=int(color))
    for pose, cloud in frames(scene, n, stride=stride, color=color, noise_seed=7, dropout=0.01):
        v.integrate(cloud, pose)
    return v


def observe_case(kind, key):
    if key == "fresh":
        out = observe(kind, oracle_volume(kind, **CFG_256))
        assert out["is_empty"] and out["occupied"]["n"] == 0
        return out
    case = ASYMMETRIC_CASE if key == "asymmetric" else dict(zip(KEYS, INTEGRATE_CASES))[key]
    v = scenario_volume(kind, *case)
    out = observe(kind, v)
    if key == "asymmetric":
        out["coarse_leaves_occupied"] = coarse_leaves_occupied(v)
        assert out["coarse_leaves_occupied"] > 0
    return out


KEYS = [integrate_key(*c) for c in INTEGRATE_CASES]
CASES = KEYS + ["asymmetric", "fresh"]


@pytest.mark.parametrize("key", CASES)
def test_restatement_leaves_match_the_reference(key):
    assert observe_case("port", key) == json.load(open(GOLDEN))[key]


def observe_all(kind):
    return {key: observe_case(kind, key) for key in CASES}
