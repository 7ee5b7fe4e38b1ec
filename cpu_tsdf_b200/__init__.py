"""cpu_tsdf_b200 — B200-native TSDF volumetric fusion, a drop-in for the volumetric path of
sdmiller/cpu_tsdf.

This package is the Python mirror of the reference's C++ class surface
(cpu_tsdf::TSDFVolumeOctree, include/cpu_tsdf/tsdf_volume_octree.h:51-377, and
cpu_tsdf::MarchingCubesTSDFOctree, include/cpu_tsdf/marching_cubes_tsdf_octree.h:50-100) over
the C ABI of libb200tsdf.so (include/b200tsdf.h).  Method names, argument meaning and return
conventions follow the reference; numpy arrays stand in for pcl::PointCloud / Eigen types.

There is no CPU fallback: importing works anywhere, but creating a volume requires the CUDA
library built by `__graft_entry__.build()` and a CUDA device, and fails loudly otherwise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200tsdf.so")


class B200Error(RuntimeError):
    pass


class Config(C.Structure):
    """b200tsdf_config (include/b200tsdf.h)."""
    _fields_ = [
        ("xres", C.c_int32), ("yres", C.c_int32), ("zres", C.c_int32),
        ("xsize", C.c_float), ("ysize", C.c_float), ("zsize", C.c_float),
        ("max_dist_pos", C.c_float), ("max_dist_neg", C.c_float), ("max_weight", C.c_float),
        ("min_sensor_dist", C.c_float), ("max_sensor_dist", C.c_float),
        ("max_cell_x", C.c_float), ("max_cell_y", C.c_float), ("max_cell_z", C.c_float),
        ("fx", C.c_double), ("fy", C.c_double), ("cx", C.c_double), ("cy", C.c_double),
        ("image_width", C.c_int32), ("image_height", C.c_int32),
        ("integrate_color", C.c_int32), ("track_variance", C.c_int32),
        ("device", C.c_int32), ("pool_log2", C.c_int32),
        ("shard_rank", C.c_int32), ("shard_count", C.c_int32),
        ("debug_flags", C.c_int32), ("color_mode", C.c_int32), ("reserved", C.c_int32 * 2),
        ("global_transform", C.c_double * 16),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("n_updates", C.c_int64), ("n_node_visits", C.c_int64), ("n_culled_cells", C.c_int64),
        ("n_bricks", C.c_int64), ("n_block_visits", C.c_int64), ("pool_capacity", C.c_int64),
        ("coarse_level", C.c_int32), ("finest_level", C.c_int32), ("tiers", C.c_int32), ("reserved", C.c_int32),
        ("ms_last_integrate", C.c_double), ("ms_last_kernel", C.c_double),
        ("n_bail", C.c_int64), ("n_slow_visits", C.c_int64),
    ]


class Profile(C.Structure):
    _fields_ = [
        ("ms_elapsed", C.c_double), ("ms_kernel", C.c_double),
        ("kernel_launches", C.c_int64), ("total_launches", C.c_int64), ("n_frames", C.c_int64),
        ("n_updates", C.c_int64), ("n_node_visits", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
        ("ms_kernel_device", C.c_double), ("kernel_launches_device", C.c_int64), ("graph_launches", C.c_int64),
        ("nvlink_bytes", C.c_int64),
    ]


class OrganizeOpts(C.Structure):
    """b200tsdf_organize_opts"""
    _fields_ = [("cloud_units", C.c_float), ("zero_nans", C.c_int32), ("world_to_camera", C.c_void_p)]


EXPORTS = [
    "b200tsdf_default_config", "b200tsdf_create", "b200tsdf_destroy", "b200tsdf_last_error",
    "b200tsdf_set_config", "b200tsdf_get_config", "b200tsdf_reset", "b200tsdf_integrate",
    "b200tsdf_integrate_device", "b200tsdf_integrate_batch_device", "b200tsdf_integrate_async",
    "b200tsdf_comm_unique_id", "b200tsdf_comm_init", "b200tsdf_row_slice", "b200tsdf_integrate_batch_rows", "b200tsdf_gather_volume", "b200tsdf_sync", "b200tsdf_organize", "b200tsdf_integrate_unorganized", "b200tsdf_query", "b200tsdf_interpolate", "b200tsdf_render", "b200tsdf_mesh",
    "b200tsdf_free", "b200tsdf_save", "b200tsdf_load", "b200tsdf_export_shard", "b200tsdf_import_shard", "b200tsdf_voxel_center", "b200tsdf_voxel_index",
    "b200tsdf_get_stats", "b200tsdf_download_nodes", "b200tsdf_download_color_payload", "b200tsdf_frustum_cull",
    "b200tsdf_profile_begin", "b200tsdf_profile_end",
    "b200tsdf_mesh_flatten", "b200tsdf_mesh_cleanup", "b200tsdf_mesh_free", "b200tsdf_meshpost_last_error", "b200tsdf_debug_timing",
    "b200tsdf_voxel_centers", "b200tsdf_occupied_voxel_indices", "b200tsdf_is_empty",
]

_lib = None


def load_library() -> C.CDLL:
    """Load libb200tsdf.so (built in-tree by __graft_entry__.build()).  Raises if it is missing:
    there is deliberately no other implementation to fall back to."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200Error(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(the engine has no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.b200tsdf_default_config.argtypes = [C.POINTER(Config)]
    lib.b200tsdf_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    lib.b200tsdf_destroy.argtypes = [vp]
    lib.b200tsdf_last_error.argtypes = [vp]; lib.b200tsdf_last_error.restype = C.c_char_p
    lib.b200tsdf_set_config.argtypes = [vp, C.POINTER(Config)]
    lib.b200tsdf_get_config.argtypes = [vp, C.POINTER(Config)]
    lib.b200tsdf_reset.argtypes = [vp]
    lib.b200tsdf_integrate.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.b200tsdf_integrate_device.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.b200tsdf_integrate_async.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.b200tsdf_integrate_batch_device.argtypes = [vp, C.c_int, vp, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.b200tsdf_comm_unique_id.argtypes = [vp]
    lib.b200tsdf_comm_init.argtypes = [vp, vp, C.c_int, C.c_int]
    lib.b200tsdf_row_slice.argtypes = [vp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.b200tsdf_integrate_batch_rows.argtypes = [vp, C.c_int, vp, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.b200tsdf_gather_volume.argtypes = [vp, vp, C.c_int]
    lib.b200tsdf_sync.argtypes = [vp]
    szp = C.POINTER(C.c_size_t)
    lib.b200tsdf_mesh_flatten.argtypes = [C.c_int, vp, C.c_size_t, vp, C.c_size_t, C.c_float, C.POINTER(vp), szp, C.POINTER(vp), szp]
    lib.b200tsdf_mesh_cleanup.argtypes = [C.c_int, vp, C.c_size_t, vp, C.c_size_t, C.c_float, C.c_int, C.POINTER(vp), szp, C.POINTER(vp), szp]
    lib.b200tsdf_mesh_free.argtypes = [vp]
    lib.b200tsdf_meshpost_last_error.restype = C.c_char_p
    lib.b200tsdf_organize.argtypes = [vp, vp, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.POINTER(OrganizeOpts), vp, C.c_size_t, C.c_int, C.POINTER(C.c_int64)]
    lib.b200tsdf_integrate_unorganized.argtypes = [vp, vp, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.POINTER(OrganizeOpts), vp]
    lib.b200tsdf_query.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]
    lib.b200tsdf_interpolate.argtypes = [vp, vp, C.c_int, vp, vp]
    lib.b200tsdf_render.argtypes = [vp, vp, C.c_int, vp, C.c_size_t, C.c_int, C.c_int, vp]
    lib.b200tsdf_mesh.argtypes = [vp, C.c_float, C.c_int, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_size_t)]
    lib.b200tsdf_save.argtypes = [vp, C.c_char_p]
    lib.b200tsdf_load.argtypes = [vp, C.c_char_p]
    lib.b200tsdf_export_shard.argtypes = [vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    lib.b200tsdf_import_shard.argtypes = [vp, vp, C.c_size_t]
    lib.b200tsdf_voxel_center.argtypes = [vp, C.c_int64, C.c_int64, C.c_int64, vp]
    lib.b200tsdf_voxel_index.argtypes = [vp, C.c_float, C.c_float, C.c_float, vp, vp]
    lib.b200tsdf_get_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.b200tsdf_voxel_centers.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(C.c_size_t)]
    lib.b200tsdf_occupied_voxel_indices.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t)]
    lib.b200tsdf_is_empty.argtypes = [vp, C.POINTER(C.c_int32)]
    lib.b200tsdf_download_nodes.argtypes = [vp, vp, vp, vp, vp, vp, vp]; lib.b200tsdf_download_nodes.restype = C.c_int64
    lib.b200tsdf_download_color_payload.argtypes = [vp, vp]; lib.b200tsdf_download_color_payload.restype = C.c_int64
    lib.b200tsdf_frustum_cull.argtypes = [vp, vp, vp, vp]
    lib.b200tsdf_profile_begin.argtypes = [vp]
    lib.b200tsdf_profile_end.argtypes = [vp, C.POINTER(Profile)]
    _lib = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _pose(trans) -> np.ndarray:
    m = np.ascontiguousarray(np.asarray(trans, dtype=np.float64))
    if m.shape == (3, 4):
        m = np.vstack([m, [0, 0, 0, 1.0]])
    if m.shape != (4, 4):
        raise ValueError("pose must be a 4x4 (or 3x4) camera->world matrix")
    return np.ascontiguousarray(m)


class TSDFVolumeOctree:
    """cpu_tsdf::TSDFVolumeOctree (include/cpu_tsdf/tsdf_volume_octree.h:51-377).

    Setters only record values; they take effect at the next reset(), as in the reference
    (src/lib/tsdf_volume_octree.cpp:201-211).  Clouds are numpy float32 arrays [H, W, 4]
    (pcl::PointXYZ, 16 B/pt) or [H, W, 8] (pcl::PointXYZRGBA, 32 B/pt, colour bytes b,g,r,a in
    float slot 4); poses are camera->world 4x4 float64 (Eigen::Affine3d)."""

    def __init__(self, device: int = 0, pool_log2: int | None = None, track_variance: bool = False,
                 shard_rank: int = 0, shard_count: int = 1):
        self._lib = load_library()
        self._cfg = Config()
        self._lib.b200tsdf_default_config(C.byref(self._cfg))
        self._cfg.device = device
        if pool_log2 is not None:
            self._cfg.pool_log2 = pool_log2
        self._cfg.track_variance = int(track_variance)
        self._cfg.shard_rank, self._cfg.shard_count = shard_rank, shard_count
        self._h = C.c_void_p()
        rc = self._lib.b200tsdf_create(C.byref(self._cfg), C.byref(self._h))
        if rc != 0:
            raise B200Error({-2: "no CUDA device: the B200 engine has no CPU fallback"}.get(rc, f"b200tsdf_create failed ({rc})"))

    def __del__(self):
        try:
            if getattr(self, "_h", None) and self._h.value:
                self._lib.b200tsdf_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    # -- plumbing ------------------------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            raise B200Error(f"{self._lib.b200tsdf_last_error(self._h).decode()} (code {rc})")

    def _push(self):
        self._check(self._lib.b200tsdf_set_config(self._h, C.byref(self._cfg)))

    # -- setters / getters (tsdf_volume_octree.cpp:93-198, tsdf_volume_octree.h:119-198) ----
    def setResolution(self, xres, yres, zres):
        self._cfg.xres, self._cfg.yres, self._cfg.zres = int(xres), int(yres), int(zres); self._push()

    def getResolution(self):
        return self._cfg.xres, self._cfg.yres, self._cfg.zres

    def setGridSize(self, xsize, ysize, zsize):
        self._cfg.xsize, self._cfg.ysize, self._cfg.zsize = xsize, ysize, zsize; self._push()

    def getGridSize(self):
        return self._cfg.xsize, self._cfg.ysize, self._cfg.zsize

    def setImageSize(self, width, height):
        self._cfg.image_width, self._cfg.image_height = int(width), int(height); self._push()

    def getImageSize(self):
        return self._cfg.image_width, self._cfg.image_height

    def setDepthTruncationLimits(self, max_dist_pos, max_dist_neg):
        self._cfg.max_dist_pos, self._cfg.max_dist_neg = max_dist_pos, max_dist_neg; self._push()

    def getDepthTruncationLimits(self):
        return self._cfg.max_dist_pos, self._cfg.max_dist_neg

    def setWeightTruncationLimit(self, max_weight):
        self._cfg.max_weight = max_weight; self._push()

    def getWeightTruncationLimit(self):
        return self._cfg.max_weight

    def setGlobalTransform(self, trans):
        self._cfg.global_transform = (C.c_double * 16)(*_pose(trans).reshape(16)); self._push()

    def getGlobalTransform(self):
        return np.array(list(self._cfg.global_transform), dtype=np.float64).reshape(4, 4)

    def setCameraIntrinsics(self, fx, fy, cx, cy):
        self._cfg.fx, self._cfg.fy, self._cfg.cx, self._cfg.cy = fx, fy, cx, cy; self._push()

    def getCameraIntrinsics(self):
        return self._cfg.fx, self._cfg.fy, self._cfg.cx, self._cfg.cy

    def setMaxVoxelSize(self, x, y, z):
        self._cfg.max_cell_x, self._cfg.max_cell_y, self._cfg.max_cell_z = x, y, z; self._push()

    def setIntegrateColor(self, integrate_color: bool):
        self._cfg.integrate_color = int(bool(integrate_color)); self._push()

    def setColorMode(self, color_mode: str):
        """tsdf_volume_octree.h:290 — "RGB" (default) or "RGBNormalized" (octree.cpp:379-434; fused by the general kernel).
        "LAB" is refused at reset() (RGB2LAB needs libm pow, octree.cpp:436-470)."""
        modes = {"RGB": 0, "RGBNormalized": 1, "LAB": 2}
        if color_mode not in modes:
            raise ValueError(f"unknown colour mode {color_mode!r}")
        self._cfg.color_mode = modes[color_mode]; self._push()

    def setSensorDistanceBounds(self, min_sensor_dist, max_sensor_dist):
        self._cfg.min_sensor_dist, self._cfg.max_sensor_dist = min_sensor_dist, max_sensor_dist; self._push()

    def getSensorDistanceBounds(self):
        return self._cfg.min_sensor_dist, self._cfg.max_sensor_dist

    def setNumRandomSplts(self, n: int):
        if n != 1:                # hpp:69-88: rand()-driven, non-deterministic; default 1 (SURVEY.md §2)
            raise B200Error("num_random_splits != 1 is not supported")

    # -- the volumetric path ---------------------------------------------------------------
    def reset(self):
        """tsdf_volume_octree.cpp:201-219"""
        self._check(self._lib.b200tsdf_reset(self._h))

    def integrateCloud(self, cloud: np.ndarray, normals=None, trans=np.eye(4)) -> bool:
        """impl/tsdf_volume_octree.hpp:48-103 (normals are unused there as well)."""
        cloud = np.ascontiguousarray(cloud, dtype=np.float32)
        if cloud.ndim != 3 or cloud.shape[2] < 3:
            raise ValueError("cloud must be an organized [H, W, >=3] float32 array")
        H, W, nf = cloud.shape
        pose = _pose(trans)
        self._check(self._lib.b200tsdf_integrate(self._h, _ptr(cloud), nf * 4, 0, 16 if nf >= 5 else -1, W, H, _ptr(pose)))
        return True

    def integrateCloudAsync(self, host_ptr: int, height: int, width: int, stride: int, trans, rgba_off: int = -1) -> bool:
        """Streaming integrateCloud from a (pinned) host buffer that the caller keeps alive until
        sync(): returns once the copy and the kernels are enqueued (b200tsdf_integrate_async)."""
        pose = _pose(trans)
        self._check(self._lib.b200tsdf_integrate_async(self._h, C.c_void_p(host_ptr), stride, 0, rgba_off, width, height, _ptr(pose)))
        return True

    def integrateCloudDevice(self, d_ptr: int, height: int, width: int, stride: int, trans, rgba_off: int = -1) -> bool:
        """Same, for a cloud already resident in this handle's device memory (asynchronous)."""
        pose = _pose(trans)
        self._check(self._lib.b200tsdf_integrate_device(self._h, C.c_void_p(d_ptr), stride, 0, rgba_off, width, height, _ptr(pose)))
        return True

    def integrateBatchDevice(self, d_ptrs, height: int, width: int, stride: int, poses, rgba_off: int = -1) -> bool:
        """len(d_ptrs) consecutive integrateCloud calls on device-resident clouds: one record upload + one graph launch."""
        n = len(d_ptrs)
        arr = (C.c_void_p * n)(*[C.c_void_p(int(x)) for x in d_ptrs])
        ps = np.ascontiguousarray(np.stack([np.asarray(_pose(t)).reshape(4, 4) for t in poses]), dtype=np.float64)
        self._check(self._lib.b200tsdf_integrate_batch_device(self._h, n, arr, stride, 0, rgba_off, width, height, _ptr(ps)))
        return True

    # ---- multi-GPU data paths (one process per GPU; NCCL over NVLink inside the library) ----
    @staticmethod
    def commUniqueId() -> bytes:
        buf = C.create_string_buffer(128)
        rc = load_library().b200tsdf_comm_unique_id(buf)
        if rc:
            raise B200Error(f"b200tsdf_comm_unique_id failed ({rc}): NCCL not loadable")
        return buf.raw

    def commInit(self, unique_id: bytes, rank: int, nranks: int):
        self._check(self._lib.b200tsdf_comm_init(self._h, C.create_string_buffer(unique_id, 128), rank, nranks))

    def rowSlice(self, height: int):
        r0, r1 = C.c_int(0), C.c_int(0)
        self._check(self._lib.b200tsdf_row_slice(self._h, height, C.byref(r0), C.byref(r1)))
        return r0.value, r1.value

    def integrateBatchRows(self, row_ptrs, height: int, width: int, stride: int, poses, rgba_off: int = -1) -> bool:
        """len(row_ptrs) <= 32 frames of which this rank's HOST memory holds only its row slice (rowSlice): upload over this GPU's
        PCIe link, all-gather over NVLink, fuse (collective: every rank calls it with the same frames)."""
        n = len(row_ptrs)
        arr = (C.c_void_p * n)(*[C.c_void_p(int(x)) for x in row_ptrs])
        ps = np.ascontiguousarray(np.stack([np.asarray(_pose(t)).reshape(4, 4) for t in poses]), dtype=np.float64)
        self._check(self._lib.b200tsdf_integrate_batch_rows(self._h, n, arr, stride, 0, rgba_off, width, height, _ptr(ps)))
        return True

    def gatherVolume(self, full, root: int = 0):
        """Collective: all shards -> `full` (a reset, unsharded volume on the root's device; None on the other ranks), device to device."""
        self._check(self._lib.b200tsdf_gather_volume(self._h, None if full is None else full._h, root))

    def sync(self):
        self._check(self._lib.b200tsdf_sync(self._h))

    @staticmethod
    def _org_opts(cloud_units, zero_nans, world_to_camera):
        tf = None if world_to_camera is None else np.ascontiguousarray(world_to_camera, dtype=np.float64).reshape(4, 4)
        opts = OrganizeOpts(float(cloud_units), int(bool(zero_nans)), None if tf is None else tf.ctypes.data)
        return opts, tf                                    # tf is returned to keep it alive across the call

    def organizeCloud(self, points: np.ndarray, *, cloud_units=1.0, zero_nans=False, world_to_camera=None):
        """The z-buffer re-organisation of the reference's `integrate` program (integrate.cpp:548-607) for an
        unorganised cloud [n, 3] (or [n, 8] rows in pcl::PointXYZRGBA layout).  Returns ([H, W, 8] float32 rows in
        PointXYZRGBA layout, number of filled pixels)."""
        pts = np.ascontiguousarray(points, dtype=np.float32)
        if pts.ndim != 2 or pts.shape[1] < 3:
            raise ValueError("points must be [n, >=3] float32")
        W, H = self._cfg.image_width, self._cfg.image_height
        out = np.empty((H, W, 8), np.float32)
        opts, _keep = self._org_opts(cloud_units, zero_nans, world_to_camera)
        filled = C.c_int64(0)
        self._check(self._lib.b200tsdf_organize(self._h, _ptr(pts), pts.shape[0], pts.shape[1] * 4, 0, 16 if pts.shape[1] >= 5 else -1,
                                                C.byref(opts), _ptr(out), 32, 16, C.byref(filled)))
        return out, int(filled.value)

    def integrateUnorganizedCloud(self, points: np.ndarray, trans=np.eye(4), *, cloud_units=1.0, zero_nans=False,
                                  world_to_camera=None) -> bool:
        """integrate.cpp:582-635 + :673 in one call: z-buffer on the GPU, then integrateCloud, without the organized
        cloud leaving device memory."""
        pts = np.ascontiguousarray(points, dtype=np.float32)
        if pts.ndim != 2 or pts.shape[1] < 3:
            raise ValueError("points must be [n, >=3] float32")
        opts, _keep = self._org_opts(cloud_units, zero_nans, world_to_camera)
        pose = _pose(trans)
        self._check(self._lib.b200tsdf_integrate_unorganized(self._h, _ptr(pts), pts.shape[0], pts.shape[1] * 4, 0,
                                                             16 if pts.shape[1] >= 5 else -1, C.byref(opts), _ptr(pose)))
        return True

    def _query(self, pts, what, mode):
        xyz = np.ascontiguousarray(pts, dtype=np.float32).reshape(-1, 3)
        n = len(xyz)
        val = np.full(n, np.nan, np.float32); grad = np.full((n, 3), np.nan, np.float32)
        hess = np.full((n, 3, 3), np.nan, np.float32); ok = np.zeros(n, np.uint8)
        self._check(self._lib.b200tsdf_query(self._h, _ptr(xyz), n, what, mode, _ptr(val), _ptr(grad), _ptr(hess), _ptr(ok)))
        return val, grad, hess, ok.astype(bool)

    def getTSDFValue(self, pts, valid_in=True):
        """getTSDFValue / interpolateTrilinearly (cpp:454-541), batched: returns (values, valid); `valid` starts as valid_in and is
        only ever cleared, like the reference's `bool* valid`."""
        xyz = np.ascontiguousarray(pts, dtype=np.float32).reshape(-1, 3)
        n = len(xyz)
        val = np.zeros(n, np.float32); ok = np.full(n, 1 if valid_in else 0, np.uint8)
        self._check(self._lib.b200tsdf_interpolate(self._h, _ptr(xyz), n, _ptr(val), _ptr(ok)))
        return val, ok.astype(bool)

    interpolateTrilinearly = getTSDFValue

    def getFxn(self, pt):
        """cpp:655-672 — returns (ok, val); batched when pt is [N,3]."""
        val, _, _, ok = self._query(pt, 1, 0)
        return (ok, val) if np.ndim(pt) > 1 else (bool(ok[0]), float(val[0]))

    def getGradient(self, pt):
        """cpp:681-700"""
        _, g, _, ok = self._query(pt, 2, 0)
        return (ok, g) if np.ndim(pt) > 1 else (bool(ok[0]), g[0])

    def getHessian(self, pt):
        """cpp:703-725"""
        _, _, hs, ok = self._query(pt, 4, 0)
        return (ok, hs) if np.ndim(pt) > 1 else (bool(ok[0]), hs[0])

    def getFxnAndGradient(self, pt):
        """cpp:728-753"""
        v, g, _, ok = self._query(pt, 3, 1)
        return (ok, v, g) if np.ndim(pt) > 1 else (bool(ok[0]), float(v[0]), g[0])

    def getFxnGradientAndHessian(self, pt):
        """cpp:756-794"""
        v, g, hs, ok = self._query(pt, 7, 1)
        return (ok, v, g, hs) if np.ndim(pt) > 1 else (bool(ok[0]), float(v[0]), g[0], hs[0])

    def renderView(self, trans=np.eye(4), downsampleBy: int = 1) -> np.ndarray:
        """cpp:278-424 — organized cloud [H/ds, W/ds, 12] float32 in pcl::PointNormal layout
        (x,y,z,_, nx,ny,nz,_, curvature,...), camera frame, NaN xyz = miss."""
        W, H = self._cfg.image_width // downsampleBy, self._cfg.image_height // downsampleBy
        out = np.zeros((H, W, 12), np.float32)
        out[..., 3] = 1.0
        pose = _pose(trans)
        self._check(self._lib.b200tsdf_render(self._h, _ptr(pose), downsampleBy, _ptr(out), 48, 0, 16, None))
        return out

    def renderColoredView(self, trans=np.eye(4), downsampleBy: int = 1):
        """cpp:427-450 — (cloud [H,W,12] float32, rgb [H,W,3] uint8)."""
        W, H = self._cfg.image_width // downsampleBy, self._cfg.image_height // downsampleBy
        out = np.zeros((H, W, 12), np.float32)
        rgb = np.zeros((H, W, 3), np.uint8)
        pose = _pose(trans)
        self._check(self._lib.b200tsdf_render(self._h, _ptr(pose), downsampleBy, _ptr(out), 48, 0, 16, _ptr(rgb)))
        return out, rgb

    def save(self, filename: str):
        """cpp:222-245"""
        self._check(self._lib.b200tsdf_save(self._h, filename.encode()))

    def load(self, filename: str):
        """cpp:248-275 — adopts the file's configuration and rebuilds the volume on the device."""
        self._check(self._lib.b200tsdf_load(self._h, filename.encode()))
        self._check(self._lib.b200tsdf_get_config(self._h, C.byref(self._cfg)))

    def export_shard(self) -> np.ndarray:
        """Everything this (sharded) handle owns, as a byte buffer that any transport can ship (DESIGN.md §5)."""
        n = C.c_size_t()
        self._check(self._lib.b200tsdf_export_shard(self._h, None, 0, C.byref(n)))
        buf = np.empty(n.value, np.uint8)
        self._check(self._lib.b200tsdf_export_shard(self._h, _ptr(buf), buf.size, C.byref(n)))
        return buf

    def import_shard(self, buf: np.ndarray):
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        self._check(self._lib.b200tsdf_import_shard(self._h, _ptr(buf), buf.size))

    def getVoxelCenter(self, x, y, z):
        o = np.empty(3, np.float32)
        self._check(self._lib.b200tsdf_voxel_center(self._h, x, y, z, _ptr(o)))
        return o

    def getVoxelIndex(self, x, y, z):
        o = np.empty(3, np.int32); ins = np.zeros(1, np.int32)
        self._check(self._lib.b200tsdf_voxel_index(self._h, x, y, z, _ptr(o), _ptr(ins)))
        return bool(ins[0]), o

    def _leaves(self, fn, dtype, *args) -> np.ndarray:
        p, n = C.c_void_p(), C.c_size_t()
        self._check(fn(self._h, *args, C.byref(p), C.byref(n)))
        out = np.empty((n.value, 3), dtype)
        if n.value:
            C.memmove(out.ctypes.data, p.value, out.nbytes)
        return out

    def getVoxelCenters(self, nlevels: int = 4) -> np.ndarray:
        """cpp:576-588 — centres of Octree::getLeaves (leaves, nlevels) as [n, 3] float32, in the reference's depth-first
        order (nlevels = 0: the root; negative: every leaf)."""
        return self._leaves(self._lib.b200tsdf_voxel_centers, np.float32, int(nlevels))

    def getOccupiedVoxelIndices(self) -> np.ndarray:
        """cpp:590-609 — getVoxelIndex of the centre of every leaf with w > 0 and |d| < 1, as [n, 3] int32 in the reference's
        order (the reference appends them to a vector: concatenate to do the same)."""
        return self._leaves(self._lib.b200tsdf_occupied_voxel_indices, np.int32)

    def isEmpty(self) -> bool:
        """h:283-287 — True from reset() until the first integrateCloud; load() takes the file's flag."""
        out = C.c_int32()
        self._check(self._lib.b200tsdf_is_empty(self._h, C.byref(out)))
        return bool(out.value)

    def getFrustumCulledVoxels(self, trans):
        """cpp:619-652 — returns the boolean mask over the 8^coarse cells."""
        st = self.stats()
        n = 1 << st.coarse_level
        mask = np.zeros((n, n, n), np.uint8); kept = np.zeros(1, np.int32)
        pose = _pose(trans)
        self._check(self._lib.b200tsdf_frustum_cull(self._h, _ptr(pose), _ptr(mask), _ptr(kept)))
        return mask.astype(bool)

    # -- introspection ---------------------------------------------------------------------
    def stats(self) -> Stats:
        s = Stats()
        self._check(self._lib.b200tsdf_get_stats(self._h, C.byref(s)))
        return s

    def profile_begin(self):
        self._check(self._lib.b200tsdf_profile_begin(self._h))

    def profile_end(self) -> Profile:
        pr = Profile()
        self._check(self._lib.b200tsdf_profile_end(self._h, C.byref(pr)))
        return pr

    def download_nodes(self):
        n = self._lib.b200tsdf_download_nodes(self._h, None, None, None, None, None, None)
        if n < 0:
            self._check(int(n))
        keys = np.empty((n, 4), np.int32); dw = np.empty((n, 2), np.float32); flags = np.empty(n, np.uint8)
        rgb = np.empty((n, 3), np.uint8); M = np.empty(n, np.float32); ns = np.empty(n, np.int32)
        n2 = self._lib.b200tsdf_download_nodes(self._h, _ptr(keys), _ptr(dw), _ptr(flags), _ptr(rgb), _ptr(M), _ptr(ns))
        assert n2 == n
        out = {"keys": keys, "dw": dw, "split": flags, "rgb": rgb, "M": M, "ns": ns}
        if self._cfg.integrate_color and self._cfg.color_mode == 1:
            q = np.empty((n, 4), np.float32)
            assert self._lib.b200tsdf_download_color_payload(self._h, _ptr(q)) == n
            out["rgbn"] = q                                        # {r_n_, g_n_, b_n_, i_} per node
        return out


class MarchingCubesTSDFOctree:
    """cpu_tsdf::MarchingCubesTSDFOctree (include/cpu_tsdf/marching_cubes_tsdf_octree.h:50-100)."""

    def __init__(self):
        self.color_by_confidence_ = False
        self.color_by_rgb_ = False
        self.w_min_ = 2.5            # marching_cubes_tsdf_octree.h:58
        self.tsdf_volume_ = None

    def setInputTSDF(self, tsdf_volume: TSDFVolumeOctree):
        self.tsdf_volume_ = tsdf_volume

    def setColorByConfidence(self, v: bool):
        self.color_by_confidence_ = bool(v)

    def setColorByRGB(self, v: bool):
        self.color_by_rgb_ = bool(v)

    def setMinWeight(self, w_min: float):
        self.w_min_ = float(w_min)

    def reconstruct(self):
        """pcl::SurfaceReconstruction::reconstruct -> performReconstruction
        (src/lib/marching_cubes_tsdf_octree.cpp:108-143).  Returns (vertices [3T,3] float32,
        rgb [3T,3] uint8 or None, polygons [T,3] int32 = {3i, 3i+1, 3i+2})."""
        v = self.tsdf_volume_
        if v is None:
            raise B200Error("setInputTSDF first")
        mode = 2 if self.color_by_confidence_ else (1 if self.color_by_rgb_ else 0)
        pv, pc, n = C.c_void_p(), C.c_void_p(), C.c_size_t()
        v._check(v._lib.b200tsdf_mesh(v._h, self.w_min_, mode, C.byref(pv), C.byref(pc), C.byref(n)))
        nv = n.value
        verts = np.empty((nv, 3), np.float32)
        rgb = None
        if nv:
            C.memmove(verts.ctypes.data, pv.value, nv * 12)
            if pc.value:
                rgb = np.empty((nv, 3), np.uint8)
                C.memmove(rgb.ctypes.data, pc.value, nv * 3)
        polys = np.arange(nv, dtype=np.int32).reshape(-1, 3)
        return verts, rgb, polys


# ---- mesh post-processing of the reference's `integrate` program (src/prog/integrate.cpp:103-214) ----------
def _meshpost(fn_name, verts, tris, *args, device=0):
    lib = load_library()
    verts = np.ascontiguousarray(verts, np.float32).reshape(-1, 3)
    tris = np.ascontiguousarray(tris, np.int32).reshape(-1, 3)
    ov, ot = C.c_void_p(), C.c_void_p()
    nv, nt = C.c_size_t(0), C.c_size_t(0)
    rc = getattr(lib, fn_name)(device, _ptr(verts), len(verts), _ptr(tris), len(tris), *args,
                               C.byref(ov), C.byref(nv), C.byref(ot), C.byref(nt))
    if rc != 0:
        raise B200Error(f"{fn_name}: error {rc}: {lib.b200tsdf_meshpost_last_error().decode()}")
    try:
        v = np.ctypeslib.as_array(C.cast(ov, C.POINTER(C.c_float)), (max(nv.value, 1) * 3,))[:nv.value * 3].reshape(-1, 3).copy()
        t = np.ctypeslib.as_array(C.cast(ot, C.POINTER(C.c_int32)), (max(nt.value, 1) * 3,))[:nt.value * 3].reshape(-1, 3).copy()
    finally:
        lib.b200tsdf_mesh_free(ov); lib.b200tsdf_mesh_free(ot)
    return v, t


def flattenVertices(verts, tris, min_dist: float = 0.0001, device: int = 0):
    """integrate.cpp:103-150: weld vertices closer than min_dist, drop degenerate faces.  -> (verts [n,3], tris [m,3])"""
    return _meshpost("b200tsdf_mesh_flatten", verts, tris, C.c_float(min_dist), device=device)


def cleanupMesh(verts, tris, face_dist: float = 0.02, min_neighbors: int = 5, device: int = 0):
    """integrate.cpp:152-214: remove face clusters of at most min_neighbors faces and the vertices left unused."""
    return _meshpost("b200tsdf_mesh_cleanup", verts, tris, C.c_float(face_dist), int(min_neighbors), device=device)
