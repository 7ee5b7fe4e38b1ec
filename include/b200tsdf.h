/* b200tsdf.h — C ABI of the B200-native TSDF fusion engine (libb200tsdf.so).
 *
 * Drop-in boundary for the volumetric path of sdmiller/cpu_tsdf.  The reference has no FFI
 * layer: its boundary is the C++ class surface cpu_tsdf::TSDFVolumeOctree /
 * cpu_tsdf::MarchingCubesTSDFOctree.  Each entry point below names the reference method it
 * replaces (paths relative to the reference tree); the C++ shim in
 * include/cpu_tsdf_b200/tsdf_volume_octree.h and the Python mirror in cpu_tsdf_b200/ marshal
 * PCL/Eigen-shaped arguments into these calls.  See INTEGRATION.md.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a
 * negative B200TSDF_E* code (the library never throws across the ABI);
 * b200tsdf_last_error() gives a message.  A handle owns one CUDA device + one stream and is
 * not thread-safe for concurrent mutation (same contract as the reference, SURVEY.md §8b).
 * There is NO CPU fallback: without a CUDA device b200tsdf_create fails with
 * B200TSDF_ENODEVICE.
 */
#ifndef B200TSDF_H
#define B200TSDF_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define B200TSDF_OK          0
#define B200TSDF_EINVAL     -1   /* bad argument / unsupported configuration          */
#define B200TSDF_ENODEVICE  -2   /* no CUDA device (there is no CPU path)             */
#define B200TSDF_ECUDA      -3   /* CUDA runtime error                                */
#define B200TSDF_ENOMEM     -4   /* brick pool / device memory exhausted              */
#define B200TSDF_ESTATE     -5   /* call order (e.g. integrate before reset)          */
#define B200TSDF_EIO        -6   /* file I/O                                          */

#define B200TSDF_COLOR_RGB             0
#define B200TSDF_COLOR_RGB_NORMALIZED  1
#define B200TSDF_COLOR_LAB             2   /* not supported: b200tsdf_reset returns B200TSDF_EINVAL */

typedef struct b200tsdf b200tsdf_t;

/* Mirrors the TSDFVolumeOctree setters; defaults = its constructor
 * (src/lib/tsdf_volume_octree.cpp:54-85).  As in the reference, changes take effect at the
 * next b200tsdf_reset() (cpp:201-211). */
typedef struct b200tsdf_config
{
  int32_t xres, yres, zres;                 /* setResolution            cpp:93   */
  float   xsize, ysize, zsize;              /* setGridSize              cpp:111  */
  float   max_dist_pos, max_dist_neg;       /* setDepthTruncationLimits cpp:145  */
  float   max_weight;                       /* setWeightTruncationLimit cpp:162  */
  float   min_sensor_dist, max_sensor_dist; /* setSensorDistanceBounds  tsdf_volume_octree.h:174 */
  float   max_cell_x, max_cell_y, max_cell_z; /* setMaxVoxelSize        tsdf_volume_octree.h:154 */
  double  fx, fy, cx, cy;                   /* setCameraIntrinsics      cpp:176  */
  int32_t image_width, image_height;        /* setImageSize             cpp:129  */
  int32_t integrate_color;                  /* setIntegrateColor        tsdf_volume_octree.h:162 (colour mode "RGB") */
  int32_t track_variance;                   /* keep OctreeNode::M_/nsample_ (octree.cpp:160-161) for .vol fidelity */
  int32_t device;                           /* CUDA device ordinal                                */
  int32_t pool_log2;                        /* brick pool capacity = 2^pool_log2 (0 = default 20) */
  int32_t shard_rank, shard_count;          /* this handle owns coarse cells with hash(cell) % shard_count == shard_rank */
  int32_t debug_flags;                      /* bit0: general depth-first update kernel only; bit1: per-level upper sweeps instead of the fused per-cell ones; bit2: generic per-cell sweeps instead of the speculative tier-1 ones */
  int32_t color_mode;                       /* setColorMode (tsdf_volume_octree.h:290) — B200TSDF_COLOR_RGB (default) or B200TSDF_COLOR_RGB_NORMALIZED
                                               (octree.cpp:379-434; fused by the general kernel).  "LAB" (octree.cpp:436-581) is refused: RGB2LAB needs libm pow */
  int32_t reserved[2];
  double  global_transform[16];             /* setGlobalTransform tsdf_volume_octree.h:119; row-major 4x4 */
} b200tsdf_config;

void b200tsdf_default_config (b200tsdf_config* cfg);

/* TSDFVolumeOctree ctor / dtor (cpp:54, :86) */
int  b200tsdf_create (const b200tsdf_config* cfg, b200tsdf_t** out);
void b200tsdf_destroy (b200tsdf_t* h);
const char* b200tsdf_last_error (const b200tsdf_t* h);

/* the setters: stores the configuration used by the next reset() */
int  b200tsdf_set_config (b200tsdf_t* h, const b200tsdf_config* cfg);
int  b200tsdf_get_config (const b200tsdf_t* h, b200tsdf_config* cfg);

/* TSDFVolumeOctree::reset (cpp:201-219) */
int  b200tsdf_reset (b200tsdf_t* h);

/* TSDFVolumeOctree::integrateCloud<PointT,NormalT> (include/cpu_tsdf/impl/
 * tsdf_volume_octree.hpp:48-103).  points: organized W x H cloud in the sensor frame,
 * row-major (cloud(u,v) = points[v*W+u]), `stride` bytes per point, xyz as 3 floats at
 * xyz_off, PCL colour bytes (b,g,r,a) at rgba_off or -1.  NaN z = invalid.  pose_c2w =
 * camera->world Affine3d as a row-major 4x4.  The normals argument of the reference is unused
 * there (hpp:51) and has no counterpart.  The host buffer is not retained after return.
 * Points wider than 16 bytes are packed to 16-byte pixels {x, y, z, bgra} on the host (a small pool of worker threads,
 * csrc/host_pack.h; bit-preserving) so that only the bytes the fusion reads cross PCIe — pageable clouds included; environment
 * switches in INTEGRATION.md §5. */
int  b200tsdf_integrate (b200tsdf_t* h, const void* points, size_t stride, int xyz_off, int rgba_off,
                         int width, int height, const double* pose_c2w);
/* same, with the cloud already resident in device memory of h's device (no copy, async on the
 * handle's stream; call b200tsdf_sync before reading results on the host) */
int  b200tsdf_integrate_device (b200tsdf_t* h, const void* d_points, size_t stride, int xyz_off, int rgba_off,
                                int width, int height, const double* pose_c2w);
/* n consecutive integrateCloud calls (hpp:48-103) on clouds resident in device memory, fused in order: the frame
 * parameters go to the device in one copy and the launches of the whole batch are one CUDA-graph launch (captured once
 * per batch size, replayed afterwards), so the host issues ~3 driver calls per batch instead of ~6 per frame.
 * d_points: n device pointers (same layout for all); poses_c2w: n row-major 4x4 matrices back to back.  Asynchronous
 * like b200tsdf_integrate_device.  Configurations fused by the general depth-first kernel (track_variance, RGBNormalized payload)
 * are fused frame by frame inside the same call. */
int  b200tsdf_integrate_batch_device (b200tsdf_t* h, int n, const void* const* d_points, size_t stride, int xyz_off, int rgba_off,
                                      int width, int height, const double* poses_c2w);
/* streaming variant of b200tsdf_integrate for producers that keep their (pinned) frame buffers alive:
 * returns as soon as the copy and the kernels are enqueued.  `points` must stay valid and unmodified
 * until b200tsdf_sync() or until two further frames have been submitted on this handle (the call that submits
 * frame i+2 waits for the upload of frame i before it returns); when the upload is packed on the host (see
 * b200tsdf_integrate) the buffer is already free on return.
 * Error reporting of the asynchronous entry points (integrate_device / _batch_device / _async, and integrate itself, which
 * waits for its upload only): a device-side failure of frame i (brick pool exhausted, work queue overflow) is reported by
 * the next call on the handle (integrate*, query, render) and at the latest by sync / get_stats / mesh / save. */
int  b200tsdf_integrate_async (b200tsdf_t* h, const void* points, size_t stride, int xyz_off, int rgba_off,
                               int width, int height, const double* pose_c2w);
int  b200tsdf_sync (b200tsdf_t* h);

/* ---- unorganised clouds: the z-buffer re-organisation of the reference's `integrate` program ----
 * (src/prog/integrate.cpp:548-635).  Per input point, in this order: scale by cloud_units (:550-559),
 * turn (0,0,0) into NaN when zero_nans (:561-568), map world -> camera with world_to_camera when it is
 * not NULL (pcl::transformPointCloud with poses[i].inverse(), :570-571; row-major 4x4, rows 0..2 used),
 * project with the handle's intrinsics in float (reprojectPoint, :216-222), keep per pixel the point
 * with the smallest z, the earliest such point on ties (:603-606).  Unfilled pixels are x=y=0, z=NaN,
 * rgba=(0,0,0,255) (a default pcl::PointXYZRGBA with z overwritten, :597-598).  */
typedef struct b200tsdf_organize_opts
{
  float   cloud_units;          /* 1 = metres                                   */
  int32_t zero_nans;            /* --zero-nans                                  */
  const double* world_to_camera;/* NULL unless --world (clouds in world frame)  */
} b200tsdf_organize_opts;
/* z-buffer `n` host points (stride / xyz_off / rgba_off as for b200tsdf_integrate) into an organized
 * image_width x image_height cloud written to `out` (host; out_stride >= 16 bytes per pixel: xyz at 0,
 * 1.0f at 12 when out_stride >= 32, colour bytes b,g,r,a at out_rgba_off or not written when -1).
 * n_filled (may be NULL) receives the number of pixels that got a point. */
int  b200tsdf_organize (b200tsdf_t* h, const void* points, size_t n, size_t stride, int xyz_off, int rgba_off,
                        const b200tsdf_organize_opts* opts, void* out, size_t out_stride, int out_rgba_off,
                        int64_t* n_filled);
/* organise + integrateCloud without the organized cloud ever leaving HBM (integrate.cpp:582-635 + :673) */
int  b200tsdf_integrate_unorganized (b200tsdf_t* h, const void* points, size_t n, size_t stride, int xyz_off,
                                     int rgba_off, const b200tsdf_organize_opts* opts, const double* pose_c2w);

/* getFxn / getGradient / getHessian (cpp:655-725) with mode 0, or the combined
 * getFxnAndGradient / getFxnGradientAndHessian (cpp:728-794) with mode 1.  what: bit0 value,
 * bit1 gradient (3 floats), bit2 hessian (9 floats, row-major).  ok[i] = the reference's bool.
 * xyz/val/grad/hess/ok are host pointers. */
int  b200tsdf_query (b200tsdf_t* h, const float* xyz, int n, int what, int mode,
                     float* val, float* grad, float* hess, uint8_t* ok);

/* getTSDFValue (cpp:454-478) = interpolateTrilinearly (cpp:486-541; use_trilinear_interpolation_ is always true, cpp:80):
 * the trilinear blend of the eight voxels around each point.  val[i] is NaN when the point's voxel is outside the volume or on
 * its border layer; valid_in_out[i] is the caller's `*valid` on entry and is only ever cleared (border, or a neighbour with
 * weight 0), exactly like the reference's pointer argument.  Host pointers. */
int  b200tsdf_interpolate (b200tsdf_t* h, const float* xyz, int n, float* val, uint8_t* valid_in_out);

/* renderView (cpp:278-424) and, with rgb_out != NULL, renderColoredView (cpp:427-450).
 * out: (W/ds)*(H/ds) points of `stride` bytes; xyz at xyz_off, normal at normal_off
 * (pcl::PointNormal: 0 / 16 / 48).  Camera frame, NaN xyz = miss. */
int  b200tsdf_render (b200tsdf_t* h, const double* pose_c2w, int downsample, void* out, size_t stride,
                      int xyz_off, int normal_off, uint8_t* rgb_out);

/* MarchingCubesTSDFOctree::performReconstruction (src/lib/marching_cubes_tsdf_octree.cpp:
 * 108-143): triangle soup, 3 vertices per triangle, global transform applied.
 * color_mode 0 none / 1 setColorByRGB / 2 setColorByConfidence.  *verts (3 floats per vertex)
 * and *rgb (3 bytes per vertex, or NULL) are library-owned until the next mesh call or
 * b200tsdf_free. */
int  b200tsdf_mesh (b200tsdf_t* h, float w_min, int color_mode, float** verts, uint8_t** rgb, size_t* nverts);
void b200tsdf_free (void* p);

/* ---- mesh post-processing of the reference's `integrate` program (no volume handle needed) ----------
 * Meshes are indexed: nverts xyz triples + ntris index triples (a marching-cubes soup is tris = 0,1,2,...).
 * Outputs are malloc'ed by the library; release each with b200tsdf_mesh_free.  Vertex colours are not
 * carried: the reference converts the mesh cloud to pcl::PointXYZ in both functions (integrate.cpp:106, 186).
 * flattenVertices (src/prog/integrate.cpp:103-150): vertices closer than min_dist are welded (in index
 * order, as the reference's sweep does), faces that become degenerate are dropped. */
int  b200tsdf_mesh_flatten (int device, const float* verts, size_t nverts, const int32_t* tris, size_t ntris, float min_dist,
                            float** out_verts, size_t* out_nverts, int32_t** out_tris, size_t* out_ntris);
/* cleanupMesh (src/prog/integrate.cpp:152-214): faces whose centroids form clusters (cluster tolerance
 * face_dist) of at most min_neighbors faces are removed, then the vertices no face uses. */
int  b200tsdf_mesh_cleanup (int device, const float* verts, size_t nverts, const int32_t* tris, size_t ntris,
                            float face_dist, int min_neighbors,
                            float** out_verts, size_t* out_nverts, int32_t** out_tris, size_t* out_ntris);
void b200tsdf_mesh_free (void* p);
const char* b200tsdf_meshpost_last_error (void);   /* thread-local message of the last failed call above */

/* Diagnostics: per-phase timing of the bottom-up per-cell kernel (k_celltop_up).  The first call arms the counters,
 * every call returns and clears them: out16[0..5] = max SM cycles << 32 | tag (total, level-3, level-2, level-1, cell,
 * wait before the first cell), out16[6..10] = slow level-2 nodes, slow level-1 nodes, cell leaf visits, cell
 * fall-throughs, cells folded.  Used by tools/dbg_celltop.py; not needed for normal operation. */
int  b200tsdf_debug_timing (b200tsdf_t* h, unsigned long long* out16);

/* TSDFVolumeOctree::save (cpp:222-245): reference-compatible .vol */
int  b200tsdf_save (b200tsdf_t* h, const char* path);

/* TSDFVolumeOctree::load (cpp:248-275) / TSDFInterface::instantiateFromFile (src/lib/tsdf_interface.cpp:44-51):
 * reads a reference-format .vol (written by the reference or by b200tsdf_save), adopts its configuration
 * (resolution, size, truncation, intrinsics, ..., colour node type) and rebuilds the volume on the device.
 * OctreeNode::M_/nsample_ are kept only if track_variance was set on the handle. */
int  b200tsdf_load (b200tsdf_t* h, const char* path);

/* Shard gather (multi-GPU, DESIGN.md §5): a handle created with shard_count > 1 owns the coarse cells with
 * hash(cell) % shard_count == shard_rank.  b200tsdf_export_shard serialises everything this handle owns (the
 * coarse-cell entries and every brick below them) into a host buffer (*nbytes needed; pass buf == NULL to query);
 * b200tsdf_import_shard merges such a buffer into a handle with the same grid configuration.  Importing all
 * shards into one volume reproduces the unsharded volume bit for bit; rendering, queries and meshing then run on
 * that volume.  Only grids whose coarse cells are the top-tier roots are supported (e.g. 2048^3/10 m, 512^3/3 m). */
int  b200tsdf_export_shard (b200tsdf_t* h, void* buf, size_t capacity, size_t* nbytes);
int  b200tsdf_import_shard (b200tsdf_t* h, const void* buf, size_t nbytes);

/* ---- multi-GPU data paths (one process per GPU; DESIGN.md §5).  NCCL is loaded at run time; without it these return
 * B200TSDF_ESTATE.  b200tsdf_comm_unique_id: 128 bytes, created on one rank and handed to the others by any means;
 * b200tsdf_comm_init: collective, binds the handle to a communicator of `nranks` ranks (normally shard_rank / shard_count). */
int  b200tsdf_comm_unique_id (void* id128);
int  b200tsdf_comm_init (b200tsdf_t* h, const void* id128, int rank, int nranks);
/* rows [*row0, *row1) of a `height`-row frame are this rank's slice (ceil(height / nranks) rows per rank) */
int  b200tsdf_row_slice (const b200tsdf_t* h, int height, int* row0, int* row1);
/* n <= 32 consecutive integrateCloud calls where this rank's HOST memory holds only its row slice of every frame
 * (rows[i] -> points (v * width + u), v in the slice; layout as for b200tsdf_integrate).  The slice is uploaded over this
 * GPU's PCIe link, packed to 16-byte pixels and all-gathered over NVLink into the full frame on every rank (collective: all
 * ranks call with the same n), then the batch is fused like b200tsdf_integrate_batch_device.  Without a communicator the
 * slice is the whole frame and nothing is exchanged.  With a single rank the slice is packed on the host first (see
 * b200tsdf_integrate) and rows[i] are free on return; otherwise they must stay valid until b200tsdf_sync or two further calls. */
int  b200tsdf_integrate_batch_rows (b200tsdf_t* h, int n, const void* const* rows, size_t stride, int xyz_off, int rgba_off,
                                    int width, int height, const double* poses_c2w);
/* Collective: every rank's shard goes device to device (NCCL send/recv over NVLink, no host staging) to rank `root`, which
 * merges them into `full` — a handle on the root's device with shard_count 1 and the same grid, already reset (NULL on the
 * other ranks).  renderView / queries / marching cubes then run on `full` (reads across shards are replicas only). */
int  b200tsdf_gather_volume (b200tsdf_t* h, b200tsdf_t* full, int root);

/* getVoxelCenter / getVoxelIndex (cpp:553-574) */
int  b200tsdf_voxel_center (const b200tsdf_t* h, int64_t x, int64_t y, int64_t z, float* out3);
int  b200tsdf_voxel_index (const b200tsdf_t* h, float x, float y, float z, int32_t* out3, int32_t* inside);

/* ---- leaf enumeration: Octree::getLeaves (octree.cpp:99-109, 608-617) on the device ----------------------------
 * Results come in the order of the reference's depth-first walk and are owned by the handle until the next call of the
 * same entry point or b200tsdf_destroy.  Before the first reset () all three return B200TSDF_ESTATE.  On a handle created
 * with shard_count > 1 the two enumerations return B200TSDF_EINVAL: the coarse cells it does not own are unsplit leaves
 * there, so gather the shards into one volume first (b200tsdf_gather_volume / b200tsdf_import_shard). */
/* TSDFVolumeOctree::getVoxelCenters (nlevels) (cpp:576-588): the centres of getLeaves (leaves, nlevels), 3 floats each.
 * nlevels = 0 gives the root, a negative nlevels every leaf. */
int  b200tsdf_voxel_centers (b200tsdf_t* h, int nlevels, float** xyz, size_t* n);
/* TSDFVolumeOctree::getOccupiedVoxelIndices (cpp:590-609): getVoxelIndex of the centre of every leaf with w > 0 and
 * |d| < 1, 3 int32 each.  The reference appends to the caller's vector; so does the C++ shim. */
int  b200tsdf_occupied_voxel_indices (b200tsdf_t* h, int32_t** ijk, size_t* n);
/* TSDFVolumeOctree::isEmpty (h:283-287): *out = 1 after reset () until the first integrateCloud, and whatever a loaded
 * .vol says (cpp:239, 264) */
int  b200tsdf_is_empty (const b200tsdf_t* h, int32_t* out);

/* ---- introspection (tests, bench accounting) ------------------------------------------- */
typedef struct b200tsdf_stats
{
  int64_t n_updates;        /* voxels whose stored {sdf,weight} changed in the last frame (= addObservation calls) */
  int64_t n_node_visits;    /* updateVoxel visits in the last frame */
  int64_t n_culled_cells;   /* coarse cells kept by the frustum cull in the last frame */
  int64_t n_bricks;         /* allocated bricks */
  int64_t n_block_visits;   /* finest-tier bricks processed in the last frame */
  int64_t pool_capacity;
  int32_t coarse_level, finest_level, tiers, reserved;   /* reserved: upper-level slow folds in the last frame */
  double  ms_last_integrate;   /* device time of the last integrate (CUDA events on the handle's stream) */
  double  ms_last_kernel;      /* device time of the dominant (brick update) kernel in the last integrate */
  int64_t n_bail;              /* block roots handed to the general path in the last frame (prune-then-resplit) */
  int64_t n_slow_visits;       /* node visits made by the general path inside the upper sweeps in the last frame */
} b200tsdf_stats;
int  b200tsdf_get_stats (b200tsdf_t* h, b200tsdf_stats* s);

/* Measurement hooks for bench.py: CUDA events on the handle's own stream (torch.cuda.Event only
 * sees torch's stream).  profile_begin records the start event and clears the accumulators;
 * profile_end records the end event, synchronizes and reports. */
typedef struct b200tsdf_profile
{
  double  ms_elapsed;        /* start event -> end event on the handle's stream                     */
  double  ms_kernel;         /* sum of the dominant (brick update) kernel's launch durations          */
  int64_t kernel_launches;   /* launches of the dominant kernel                                       */
  int64_t total_launches;    /* all kernel launches of this library in the region                     */
  int64_t n_frames;          /* integrate calls in the region                                         */
  int64_t n_updates;         /* sum over frames of voxels whose {sdf,weight} changed                  */
  int64_t n_node_visits;
  int64_t h2d_bytes, d2h_bytes; /* bytes this library copied across PCIe in the region                */
  double  ms_kernel_device;  /* the same kernel timed on the device (%globaltimer, first block start -> last block end):  */
  int64_t kernel_launches_device; /* also available for frames replayed from a CUDA graph, where no event can be placed   */
  int64_t graph_launches;    /* cudaGraphLaunch calls in the region (b200tsdf_integrate_batch_device)                      */
  int64_t nvlink_bytes;      /* bytes this rank received / sent over NCCL in the region (row all-gather, shard gather)     */
} b200tsdf_profile;
int  b200tsdf_profile_begin (b200tsdf_t* h);
int  b200tsdf_profile_end (b200tsdf_t* h, b200tsdf_profile* out);

/* Every existing octree node at depth >= coarse level, sorted by (level,x,y,z) — the same
 * record the oracle dumps.  Pass all-NULL to get the count.  keys: 4 int32; dw: 2 floats;
 * flags bit0 = has children; rgb 3 bytes; M float; ns int32. */
int64_t b200tsdf_download_nodes (b200tsdf_t* h, int32_t* keys, float* dw, uint8_t* flags,
                                 uint8_t* rgb, float* M, int32_t* ns);
/* RGBNormalized volumes: the four floats {r_n_, g_n_, b_n_, i_} of every node, in the order of b200tsdf_download_nodes
 * (returns the node count, or 0 when the volume does not carry that payload) */
int64_t b200tsdf_download_color_payload (b200tsdf_t* h, float* out4);
/* frustum-culled coarse-cell mask of getFrustumCulledVoxels (cpp:619-652): 8^coarse bytes */
int  b200tsdf_frustum_cull (b200tsdf_t* h, const double* pose_c2w, uint8_t* mask, int32_t* kept);

#ifdef __cplusplus
}
#endif
#endif
