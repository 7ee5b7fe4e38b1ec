"""getVoxelCenters / getOccupiedVoxelIndices / isEmpty for the two CPU oracles.  TEST INFRASTRUCTURE ONLY.

* The restatement: Octree::getLeaves (octree.cpp:99-109, 608-617) walked over the restatement's own tree, as
  orc_dump_nodes reports it (every node at depth >= the coarse level, with its split flag and {d, w}), and the levels
  above the coarse depth that Octree::init splits everywhere.  Centres are the octree's float ctr +/- size/4
  accumulation; indices are getVoxelIndex's double expression (tsdf_volume_octree.cpp:562-574); isEmpty is the flag
  that save() writes (cpp:239).
* The reference: its own methods, compiled verbatim into oracle/_ref/libcpu_tsdf_ref_leaves.so (oracle/leaves.mk).
"""
from __future__ import annotations

import ctypes as C
import os
import tempfile

import numpy as np

from oracle import oracle_py

REF_LEAVES_LIB = os.path.join(oracle_py.HERE, "_ref", "libcpu_tsdf_ref_leaves.so")
KIND = "reference-leaves"


def _interleave(x, y, z, bits):
    """bit-interleaved coordinates, x high then y then z: the child order of octree.cpp:257-264"""
    k = np.zeros(len(x), np.uint64)
    for b in range(bits - 1, -1, -1):
        k = (k << np.uint64(3)) | (((x >> b) & 1) << 2 | ((y >> b) & 1) << 1 | ((z >> b) & 1)).astype(np.uint64)
    return k


def _centers(size, level, x, y, z):
    return np.stack([_center(size, level, a) for a in (x, y, z)], axis=1).astype(np.float32)


def _center(size, level, x):
    """OctreeNode::split's float32 accumulation from the root (octree.cpp:244-266): c = 0, then for i = level-1 .. 0
    c += off if bit i of x is set else c -= off, off = size/4 halving each level"""
    out = np.zeros(len(x), np.float32)
    for lv in np.unique(level):
        m = level == lv
        xs = x[m]
        c = np.zeros(len(xs), np.float32)
        off = np.float32(np.float32(size) * np.float32(0.25))
        for i in range(int(lv) - 1, -1, -1):
            c = np.where(((xs >> i) & 1) == 1, c + off, c - off).astype(np.float32)
            off = np.float32(off * np.float32(0.5))
        out[m] = c
    return out


def _leaves(v, nlevels):
    """(level, x, y, z, dw) of Octree::getLeaves (leaves, nlevels) over an OracleVolume, in the walk's order"""
    coarse, finest = v.levels()
    if 0 <= nlevels <= coarse:                            # every node at that level: all exist, those above C are split
        i = np.arange(8 ** nlevels, dtype=np.int64)
        x = np.zeros_like(i); y = np.zeros_like(i); z = np.zeros_like(i)
        for b in range(nlevels):
            x |= ((i >> (3 * b + 2)) & 1) << b; y |= ((i >> (3 * b + 1)) & 1) << b; z |= ((i >> (3 * b)) & 1) << b
        return np.full(len(i), nlevels, np.int64), x, y, z, None
    d = v.dump_nodes()
    level = d["keys"][:, 0].astype(np.int64)
    split = d["split"] != 0
    keep = ~split if nlevels < 0 else (level <= nlevels) & (~split | (level == nlevels))
    level, dw = level[keep], d["dw"][keep]
    x, y, z = (d["keys"][keep, k].astype(np.int64) for k in (1, 2, 3))
    sh = finest - level
    order = np.argsort(_interleave(x << sh, y << sh, z << sh, finest), kind="stable")
    return level[order], x[order], y[order], z[order], dw[order]


def restatement_voxel_centers(v, nlevels: int = 4) -> np.ndarray:
    """getVoxelCenters (cpp:576-588) of the restatement: [n, 3] float32"""
    level, x, y, z, _ = _leaves(v, nlevels)
    return _centers(v.cfg.xsize, level, x, y, z)


def restatement_occupied_indices(v) -> np.ndarray:
    """getOccupiedVoxelIndices (cpp:590-609) of the restatement: [n, 3] int32"""
    level, x, y, z, dw = _leaves(v, -1)
    occ = (dw[:, 1] > 0) & (np.abs(dw[:, 0].astype(np.float64)) < 1)
    c = _centers(v.cfg.xsize, level[occ], x[occ], y[occ], z[occ]).astype(np.float64)
    size, res = float(np.float32(v.cfg.xsize)), float(v.cfg.xres)
    return np.floor((c + size / 2.0) / size * res).astype(np.int32)


def restatement_is_empty(v) -> bool:
    """isEmpty (h:283-287): the is_empty_ line of the .vol header save () writes (cpp:239)"""
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "v.vol")
        assert v.save(path) == 0
        with open(path, "rb") as f:
            lines = [f.readline() for _ in range(12)]
    # meta lines: title, resolution, size, truncation (3), sensor bounds (2), cell size, intrinsics, image size, is_empty_
    assert lines[0].startswith(b"# TSDFVolumeOctree")
    return lines[11].strip() == b"1"


def load_reference():
    """oracle/_ref/libcpu_tsdf_ref_leaves.so with the oracle API's signatures, registered under KIND so that
    OracleVolume(kind=KIND, ...) uses it"""
    if KIND in oracle_py._libs:
        return oracle_py._libs[KIND]
    if not os.path.exists(REF_LEAVES_LIB):
        raise FileNotFoundError(REF_LEAVES_LIB)
    lib = C.CDLL(REF_LEAVES_LIB)
    vp = C.c_void_p
    lib.orc_default_config.argtypes = [C.POINTER(oracle_py.OrcConfig)]
    lib.orc_create.argtypes = [C.POINTER(oracle_py.OrcConfig)]; lib.orc_create.restype = vp
    lib.orc_destroy.argtypes = [vp]
    lib.orc_reset.argtypes = [vp]
    lib.orc_integrate.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.orc_dump_nodes.argtypes = [vp, vp, vp, vp, vp, vp, vp]; lib.orc_dump_nodes.restype = C.c_int64
    lib.orc_levels.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.orc_save.argtypes = [vp, C.c_char_p]
    lib.orc_voxel_centers.argtypes = [vp, C.c_int, vp]; lib.orc_voxel_centers.restype = C.c_int64
    lib.orc_occupied_indices.argtypes = [vp, vp]; lib.orc_occupied_indices.restype = C.c_int64
    lib.orc_is_empty.argtypes = [vp]
    oracle_py._libs[KIND] = lib
    return lib


def reference_voxel_centers(v, nlevels: int = 4) -> np.ndarray:
    n = v.lib.orc_voxel_centers(v.h, nlevels, None)
    out = np.empty((n, 3), np.float32)
    v.lib.orc_voxel_centers(v.h, nlevels, out.ctypes.data_as(C.c_void_p))
    return out


def reference_occupied_indices(v) -> np.ndarray:
    n = v.lib.orc_occupied_indices(v.h, None)
    out = np.empty((n, 3), np.int32)
    v.lib.orc_occupied_indices(v.h, out.ctypes.data_as(C.c_void_p))
    return out


def reference_is_empty(v) -> bool:
    return bool(v.lib.orc_is_empty(v.h))
