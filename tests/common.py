"""Shared helpers for the parity tests."""
from __future__ import annotations

import hashlib

import numpy as np

from cpu_tsdf_b200 import synth

CAM = synth.Camera()

# BASELINE.json configs, scaled to what the oracle finishes in seconds
CFG_256 = dict(xres=256, yres=256, zres=256, xsize=3.0, ysize=3.0, zsize=3.0, cx=CAM.cx, cy=CAM.cy)
CFG_512 = dict(xres=512, yres=512, zres=512, xsize=3.0, ysize=3.0, zsize=3.0, cx=CAM.cx, cy=CAM.cy)
CFG_2048 = dict(xres=2048, yres=2048, zres=2048, xsize=10.0, ysize=10.0, zsize=10.0, cx=CAM.cx, cy=CAM.cy)


def frames(scene, n, *, stride=1, color=False, noise_seed=None, total=100, dropout=0.0, max_depth=None):
    for f in range(n):
        pose = synth.orbit_pose(scene, f * stride, total)
        yield pose, synth.make_frame(scene, pose, CAM, color=color, noise_seed=noise_seed, frame=f,
                                     dropout=dropout, max_depth=max_depth)


def assert_same_nodes(a, b, *, rgb=False, var=False):
    assert len(a["keys"]) == len(b["keys"]), (len(a["keys"]), len(b["keys"]))
    assert np.array_equal(a["keys"], b["keys"]), "octree structure (level,x,y,z) differs"
    assert np.array_equal(a["split"], b["split"]), "split flags differ"
    # bit-exact {sdf, weight} at every node of every level
    assert np.array_equal(a["dw"].view(np.uint32), b["dw"].view(np.uint32)), "per-node {sdf,weight} differ"
    if rgb:
        assert np.array_equal(a["rgb"], b["rgb"]), "per-node rgb differs"
    if var:
        assert np.array_equal(a["M"].view(np.uint32), b["M"].view(np.uint32)) and np.array_equal(a["ns"], b["ns"])


def sha(*arrays):
    """SHA-256 of the arrays' bytes: equal digests = bit-identical arrays."""
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def sha_values(a):
    """Digest under np.array_equal(..., equal_nan=True): every NaN is the same value, and -0.0 equals 0.0."""
    a = np.asarray(a)
    nan = np.isnan(a)
    return sha(nan, np.where(nan, 0, a) + 0)


def canon_soup(verts, cols=None):
    """Order-independent form of a triangle soup (oracle order = octree DFS)."""
    t = np.asarray(verts, np.float32).reshape(-1, 9)
    if cols is not None:
        t = np.concatenate([t, np.asarray(cols).reshape(-1, 9).astype(np.float32)], axis=1)
    if len(t) == 0:
        return t
    return t[np.lexsort(t.T[::-1])]


def query_points(seed=1, n=4000, radius=0.35, extent=1.6):
    rng = np.random.default_rng(seed)
    far = rng.uniform(-extent, extent, (n // 2, 3))
    near = rng.normal(size=(n - n // 2, 3))
    near *= radius / np.linalg.norm(near, axis=1, keepdims=True)
    near += rng.normal(scale=0.01, size=near.shape)
    return np.concatenate([far, near]).astype(np.float32)
