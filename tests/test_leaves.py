"""getVoxelCenters / getOccupiedVoxelIndices / isEmpty on the CUDA engine (b200tsdf_voxel_centers,
b200tsdf_occupied_voxel_indices, b200tsdf_is_empty) against the restatement, array for array and in order.

The restatement's results (oracle/leaves_py.py) are pinned to the reference's own methods by tests/test_leaves_ref_pin.py."""
import ctypes as C
import os

import numpy as np
import pytest

from cpu_tsdf_b200 import synth
from oracle.leaves_py import restatement_is_empty, restatement_occupied_indices, restatement_voxel_centers
from oracle.oracle_py import OracleVolume
from tests.common import CAM, CFG_256, CFG_2048, frames
from tests.test_leaves_ref_pin import ASYMMETRIC_CASE, sweep
from tests.test_ref_pin import INTEGRATE_CASES

pytestmark = pytest.mark.gpu


def engine_volume(cfg, color=False, color_mode=0, track_variance=False, pool_log2=20, shard_count=1):
    import cpu_tsdf_b200 as pkg
    v = pkg.TSDFVolumeOctree(device=0, pool_log2=pool_log2, track_variance=track_variance, shard_count=shard_count)
    v.setResolution(cfg["xres"], cfg["yres"], cfg["zres"])
    v.setGridSize(cfg.get("xsize", 3.0), cfg.get("ysize", 3.0), cfg.get("zsize", 3.0))
    v.setCameraIntrinsics(CAM.fx, CAM.fy, cfg["cx"], cfg["cy"])
    if "max_dist_pos" in cfg:
        v.setDepthTruncationLimits(cfg["max_dist_pos"], cfg["max_dist_neg"])
    v.setIntegrateColor(bool(color))
    if color_mode:
        v.setColorMode("RGBNormalized")
    v.reset()
    return v


def fuse_both(cfg, scene, n, *, stride=1, color=False, noise_seed=7, dropout=0.0, color_mode=0, track_variance=False):
    eng = engine_volume(cfg, color, color_mode, track_variance)
    orc = OracleVolume(kind="port", **cfg, integrate_color=int(color), color_mode=color_mode)
    orc.reset()
    for pose, cloud in frames(scene, n, stride=stride, color=color, noise_seed=noise_seed, dropout=dropout):
        eng.integrateCloud(cloud, None, pose)
        orc.integrate(cloud, pose)
    return eng, orc


def assert_same_leaves(eng, orc, nlevels=None):
    coarse, finest = orc.levels()
    assert eng.isEmpty() == restatement_is_empty(orc)
    for n in (sweep(coarse, finest) if nlevels is None else nlevels):
        a, b = eng.getVoxelCenters(n), restatement_voxel_centers(orc, n)
        assert a.dtype == np.float32 and a.shape == b.shape, (n, a.shape, b.shape)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), f"getVoxelCenters({n}) differs"
    a, b = eng.getOccupiedVoxelIndices(), restatement_occupied_indices(orc)
    assert a.dtype == np.int32 and a.shape == b.shape, (a.shape, b.shape)
    assert np.array_equal(a, b), "getOccupiedVoxelIndices differs"
    return len(b)


@pytest.mark.parametrize("case", INTEGRATE_CASES + [ASYMMETRIC_CASE], ids=["256", "512", "2048", "asymmetric"])
def test_pinned_scenarios(case):
    cfg, scene, n, stride, color = case
    eng, orc = fuse_both(cfg, scene, n, stride=stride, color=color, dropout=0.01)
    assert assert_same_leaves(eng, orc) > 0


def test_fresh_volume():
    eng = engine_volume(CFG_256)
    orc = OracleVolume(kind="port", **CFG_256)
    orc.reset()
    assert eng.isEmpty() and len(eng.getOccupiedVoxelIndices()) == 0
    assert_same_leaves(eng, orc)


@pytest.mark.parametrize("name", ["L1_512_orbit100", "L2_2048_color100"])
def test_baseline_length_streams(name):
    """the 100-frame 512^3 orbit and the 100-frame 2048^3 colour stream of tests/golden (tools/make_golden.py LONG_CASES)"""
    if name == "L1_512_orbit100":
        cfg, scene, color, noise = dict(xres=512, yres=512, zres=512, cx=CAM.cx, cy=CAM.cy), synth.S1, False, 2
    else:
        cfg, scene, color, noise = CFG_2048, synth.S2, True, 12345
    eng, orc = fuse_both(cfg, scene, 100, color=color, noise_seed=noise)
    coarse, finest = orc.levels()
    assert assert_same_leaves(eng, orc, nlevels=(-1, 0, 4, coarse, coarse + 1, finest)) > 100000


def test_4096_volume_uses_the_40_bit_key():
    """4096^3 / 10 m: 12 levels, coarse cells below the root arrays (Rtop = 3 < C = 5), keys of 3 * 12 + 5 bits"""
    cfg = dict(xres=4096, yres=4096, zres=4096, xsize=10.0, ysize=10.0, zsize=10.0, cx=CAM.cx, cy=CAM.cy)
    eng, orc = fuse_both(cfg, synth.S2, 3, stride=7, noise_seed=5)
    assert orc.levels() == (5, 12)
    assert assert_same_leaves(eng, orc) > 100000


@pytest.mark.parametrize("variant", ["rgb_normalized", "track_variance"])
def test_storage_variants(variant):
    kw = dict(color=True, color_mode=1) if variant == "rgb_normalized" else dict(track_variance=True)
    eng, orc = fuse_both(CFG_256, synth.S1, 4, stride=9, **kw)
    assert assert_same_leaves(eng, orc) > 0


def test_is_empty_transitions_and_load(tmp_path):
    eng = engine_volume(CFG_256)
    assert eng.isEmpty()
    fresh = str(tmp_path / "fresh.vol")
    eng.save(fresh)
    for pose, cloud in frames(synth.S1, 3, stride=9, noise_seed=5):
        eng.integrateCloud(cloud, None, pose)
    assert not eng.isEmpty()
    eng.reset()
    assert eng.isEmpty()
    eng.load(fresh)
    assert eng.isEmpty()
    # a volume rebuilt by load () from a .vol the restatement wrote
    orc = OracleVolume(kind="port", **CFG_256, integrate_color=1)
    orc.reset()
    for pose, cloud in frames(synth.S1, 4, stride=9, color=True, noise_seed=5):
        orc.integrate(cloud, pose)
    path = str(tmp_path / "orc.vol")
    assert orc.save(path) == 0
    other = engine_volume(dict(CFG_2048))                  # load () adopts the file's configuration
    other.load(path)
    assert not other.isEmpty()
    assert assert_same_leaves(other, orc) > 0


def error_code(fn):
    import cpu_tsdf_b200 as pkg
    with pytest.raises(pkg.B200Error) as e:
        fn()
    return str(e.value)


def test_state_and_shard_errors():
    import cpu_tsdf_b200 as pkg
    v = pkg.TSDFVolumeOctree(device=0, pool_log2=14)
    for fn in (lambda: v.getVoxelCenters(4), v.getOccupiedVoxelIndices, v.isEmpty):
        assert error_code(fn).endswith("(code -5)")                    # B200TSDF_ESTATE before reset ()
    s = engine_volume(CFG_256, pool_log2=16, shard_count=2)
    for fn in (lambda: s.getVoxelCenters(-1), s.getOccupiedVoxelIndices):
        msg = error_code(fn)
        assert msg.endswith("(code -1)") and "gather" in msg               # B200TSDF_EINVAL: gather the shards first
    assert s.isEmpty()


def test_second_call_replaces_the_first_buffer():
    import cpu_tsdf_b200 as pkg
    eng, orc = fuse_both(CFG_256, synth.S1, 2, stride=9)
    lib = pkg.load_library()

    def raw(fn, *args):
        p, n = C.c_void_p(), C.c_size_t()
        assert fn(eng._h, *args, C.byref(p), C.byref(n)) == 0
        return p.value, n.value

    def view(p, n, ctype):
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(ctype)), (n * 3,)).reshape(n, 3).copy()

    p4, n4 = raw(lib.b200tsdf_voxel_centers, 4)
    assert np.array_equal(view(p4, n4, C.c_float), restatement_voxel_centers(orc, 4))
    pi, ni = raw(lib.b200tsdf_occupied_voxel_indices)
    pa, na = raw(lib.b200tsdf_voxel_centers, -1)
    assert na != n4
    assert np.array_equal(view(pa, na, C.c_float), restatement_voxel_centers(orc, -1))
    assert np.array_equal(view(pi, ni, C.c_int32), restatement_occupied_indices(orc))   # each entry point owns its own buffer
    p0, n0 = raw(lib.b200tsdf_voxel_centers, 0)
    assert n0 == 1 and np.array_equal(view(p0, n0, C.c_float), np.zeros((1, 3), np.float32))
