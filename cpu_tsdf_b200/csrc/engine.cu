// engine.cu — libb200tsdf.so: handle, device memory, kernels and the C ABI (include/b200tsdf.h).
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -fmad=false (see
// __graft_entry__.build).  There is no CPU path: b200tsdf_create fails without a CUDA device.
#include "../../include/b200tsdf.h"
#include "tsdf_core.cuh"
#include "mc_tables.cuh"
#include "host_math.h"
#include "params_setup.h"
#include "brick_kernels.cuh"
#include "brick_direct.cuh"
#include "organize.cuh"
#include "mesh_sort.h"
#include "host_pack.h"

#include <cuda_runtime.h>
#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

using namespace b2;

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) return h->fail (B200TSDF_ECUDA, std::string (#call) + ": " + cudaGetErrorString (e_)); \
  } while (0)

namespace {

struct Planes { float pl[6][4]; };

// d_stats[0..ST_N) are cumulative since reset(); [ST_N..2*ST_N) is the snapshot taken at the start of
// the current frame (so last-frame = cum - prev without a host round trip); the last slot is scratch
enum StatSlot { ST_UPDATES = 0, ST_VISITS = 1, ST_BLOCKS = 2, ST_N = 8, ST_TOTAL = 2 * ST_N + 1, ST_SCRATCH = 2 * ST_N };
constexpr int KRING = 64;     // ring of event pairs around the dominant kernel
constexpr int FRAME_RING = 64;  // per-frame records in flight (device ring + its pinned host image)
constexpr int BATCH_SEGS = 16;  // host staging segments of the batch path

// ---------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------
__global__ void k_fill_fresh (float2* __restrict__ nodes, size_t n)
{
  size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t) gridDim.x * blockDim.x;
  for (; i < n; i += stride) nodes[i] = make_float2 (-1.f, 0.f);
}

// top-tier bricks that contain the coarse cells themselves (Rtop < C) are permanent
__global__ void k_insert_top_bricks (Params p)
{
  int n = 1 << p.Rtop;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * n * n) return;
  int z = i % n, y = (i / n) % n, x = i / (n * n);
  find_or_insert_brick (p, p.T - 1, x, y, z);
}

// the static supercell list of grids whose coarse cells lie inside the tier-1 bricks: every root-array node (level Rtop = L - 6)
__global__ void k_build_superq (Params p, QNode* __restrict__ q, int n)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int nn = 1 << p.Rtop;
  QNode e; e.x = i / (nn * nn); e.y = (i / nn) % nn; e.z = i % nn; e.slot = -1; e.idx = i; e.kind = KIND_DONE; e.child_base = -1; e.rc = 0;
  q[i] = e;
}

// frustum cull of the coarse cells (tsdf_volume_octree.cpp:619-652); planes come from the host
__global__ void k_cull (Params p, Planes P, int* __restrict__ list, int* __restrict__ count, unsigned char* __restrict__ mask, QNode* __restrict__ q0)
{
  int n = 1 << p.C;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * n * n) return;
  int z = i % n, y = (i / n) % n, x = i / (n * n);
  float cx = center1d (p, p.C, x), cy = center1d (p, p.C, y), cz = center1d (p, p.C, z);
  bool in = frustum_contains (P.pl, cx, cy, cz);
  if (mask) mask[i] = in ? 1 : 0;
  if (in && list && owns_cell (p, x, y, z))
  {
    int k = atomicAdd (count, 1);
    list[k] = i;
    if (q0)
    {
      NodePos n;
      if (!locate_node (p, p.C, x, y, z, n)) { raise_err (p, ERR_MISSING_BRICK); n.slot = -1; n.idx = 0; }
      QNode e; e.x = x; e.y = y; e.z = z; e.slot = n.slot; e.idx = n.idx; e.kind = KIND_DONE; e.child_base = -1; e.rc = 0;
      q0[k] = e;
    }
  }
}

// frame front end in ONE launch: blocks [0, cull_blocks) run the frustum cull of the coarse cells, the
// rest the per-pixel pre-split.  The two are independent (the cull reads only geometry).  The work-list
// counters and the statistics snapshot are reset by the frame-begin bookkeeping of the previous k_front launch.
// The frame's parameters come from a record in device memory (FrameRec), so a captured launch can be replayed.
#define B2_STAGE_FRAME(fr)                                                      \
  __shared__ FrameRec s_fr_;                                                    \
  {                                                                             \
    const int* src_ = reinterpret_cast<const int*> (fr);                        \
    int* dst_ = reinterpret_cast<int*> (&s_fr_);                                \
    for (int w_ = threadIdx.x; w_ < (int) (sizeof (FrameRec) / sizeof (int)); w_ += blockDim.x) dst_[w_] = src_[w_]; \
  }                                                                             \
  __syncthreads ();                                                             \
  const Frame& f = s_fr_.f;

__global__ void k_front (Params p, const FrameRec* __restrict__ fr, int cull_blocks, int* __restrict__ list, int* __restrict__ d_count, QNode* __restrict__ q0,
                         unsigned long long* __restrict__ stats)
{
  pdl_launch_dependents ();
  B2_STAGE_FRAME (fr)
  pdl_wait ();                                          // the previous frame's bottom-up sweep has finished
  int* count = d_count + 16 * s_fr_.cset;
  int* next_counts = d_count + 16 * (s_fr_.cset ^ 1);
  // frame-begin bookkeeping (was a launch of its own): snapshot the cumulative counters, and clear the counter
  // set the NEXT frame will use (the sets alternate, so nothing in this frame touches it)
  if (blockIdx.x == 0 && threadIdx.x < 16)
  {
    if (threadIdx.x < ST_N) stats[ST_N + threadIdx.x] = stats[threadIdx.x];
    next_counts[threadIdx.x] = 0;
  }
  if ((int) blockIdx.x < cull_blocks)
  {
    int n = 1 << p.C;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * n * n) return;
    int z = i % n, y = (i / n) % n, x = i / (n * n);
    float cx = center1d (p, p.C, x), cy = center1d (p, p.C, y), cz = center1d (p, p.C, z);
    if (!frustum_contains (s_fr_.pl, cx, cy, cz) || !owns_cell (p, x, y, z)) return;
    int k = atomicAdd (count, 1);
    list[k] = i;
    if (q0)
    {
      NodePos nd;
      if (!locate_node (p, p.C, x, y, z, nd)) { raise_err (p, ERR_MISSING_BRICK); nd.slot = -1; nd.idx = 0; }
      QNode e; e.x = x; e.y = y; e.z = z; e.slot = nd.slot; e.idx = nd.idx; e.kind = KIND_DONE; e.child_base = -1; e.rc = 0;
      q0[k] = e;
    }
    return;
  }
  int i = (blockIdx.x - cull_blocks) * blockDim.x + threadIdx.x;
  if (i >= f.width * f.height) return;
  int u = i % f.width, v = i / f.width;
  const float* pt = frame_xyz (f, u, v);
  float z = pt[2];
  if (is_nan (z)) return;                                        // hpp:64
  float pw[3];
  affine_mul_f (f.tfwd, pt[0], pt[1], z, pw);                    // hpp:76
  int fx_, fy_, fz_;
  if (!world_to_finest (p, pw[0], pw[1], pw[2], fx_, fy_, fz_)) return;
  if (p.shard_count > 1)
  {
    int sh = p.L - p.C;
    if (!owns_cell (p, fx_ >> sh, fy_ >> sh, fz_ >> sh)) return;
  }
  presplit_point (p, fx_, fy_, fz_);
}

// general path: one thread per culled coarse cell runs updateVoxel depth-first
__global__ void k_update_dfs (Params p, Frame f, const int* __restrict__ list, const int* __restrict__ count, unsigned long long* __restrict__ stats)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *count) return;
  int n = 1 << p.C;
  int id = list[i];
  int z = id % n, y = (id / n) % n, x = id / (n * n);
  NodePos node;
  if (!locate_node (p, p.C, x, y, z, node)) { raise_err (p, ERR_MISSING_BRICK); return; }
  Counters cnt; cnt.n_updates = 0; cnt.n_visits = 0;
  update_voxel_dfs (p, f, node, cnt);
  atomicAdd (&stats[ST_UPDATES], (unsigned long long) cnt.n_updates);
  atomicAdd (&stats[ST_VISITS], (unsigned long long) cnt.n_visits);
}

// read-side kernels keep Params in shared memory (see find_leaf in tsdf_core.cuh)
#define B2_STAGE_PARAMS(gp)                                                     \
  __shared__ Params sp_;                                                        \
  {                                                                             \
    const int* src_ = reinterpret_cast<const int*> (&gp);                       \
    int* dst_ = reinterpret_cast<int*> (&sp_);                                  \
    for (int w_ = threadIdx.x; w_ < (int) (sizeof (Params) / sizeof (int)); w_ += blockDim.x) dst_[w_] = src_[w_]; \
  }                                                                             \
  __syncthreads ();                                                             \
  const Params& p = sp_;

__global__ void k_query (Params gp, const float* __restrict__ xyz, int n, int what, int mode,
                         float* val, float* grad, float* hess, unsigned char* ok)
{
  B2_STAGE_PARAMS (gp)
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float v, g[3], hs[9];
  bool good = query_point (p, xyz + 3 * i, mode, &v, g, hs);
  ok[i] = good ? 1 : 0;
  if (!good) return;
  if (what & 1) val[i] = v;
  if (what & 2) { grad[3 * i] = g[0]; grad[3 * i + 1] = g[1]; grad[3 * i + 2] = g[2]; }
  if (what & 4) for (int k = 0; k < 9; ++k) hess[9 * i + k] = hs[k];
}

// getTSDFValue = interpolateTrilinearly (tsdf_volume_octree.cpp:454-541), one thread per point
__global__ void k_interpolate (Params gp, const float* __restrict__ xyz, int n, float* __restrict__ val, unsigned char* __restrict__ valid)
{
  B2_STAGE_PARAMS (gp)
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  bool v = valid[i] != 0;
  val[i] = interpolate_trilinearly (p, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], &v);
  valid[i] = v ? 1 : 0;
}

__global__ void k_render (Params gp, RenderParams r, float* __restrict__ out /* 6 floats per pixel */, unsigned char* __restrict__ rgb)
{
  B2_STAGE_PARAMS (gp)
  // 8x8 pixel tiles keep neighbouring rays in one warp-pair
  int tx = threadIdx.x % 8, ty = threadIdx.x / 8;
  int x = blockIdx.x * 8 + tx, y = blockIdx.y * 8 + ty;
  if (x >= r.width || y >= r.height) return;
  size_t i = (size_t) y * r.width + x;
  float P[3], N[3];
  render_pixel (p, r, x, y, P, N, rgb ? rgb + 3 * i : nullptr);
  float* o = out + 6 * i;
  o[0] = P[0]; o[1] = P[1]; o[2] = P[2]; o[3] = N[0]; o[4] = N[1]; o[5] = N[2];
}

__global__ void k_list_bricks (Params p, int* __restrict__ list, int* __restrict__ count)
{
  size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i > p.pool_mask) return;
  if (p.keys[i] != KEY_EMPTY) list[atomicAdd (count, 1)] = (int) i;
}

// number of claimed directory slots (statistics): one atomic per warp
__global__ void k_count_bricks (Params p, int* __restrict__ count)
{
  size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
  const bool used = i <= p.pool_mask && p.keys[i] != KEY_EMPTY;
  const unsigned m = __ballot_sync (0xffffffffu, used);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd (count, __popc (m));
}

__global__ void k_gather_bricks (Params p, const int* __restrict__ list, int n,
                                 float2* nodes, uint32_t* split, uchar4* rgb, float* M, int* ns)
{
  int b = blockIdx.x;
  if (b >= n) return;
  size_t s = (size_t) list[b];
  for (int i = threadIdx.x; i < BRICK_NODES; i += blockDim.x)
  {
    nodes[(size_t) b * BRICK_NODES + i] = p.nodes[s * BRICK_NODES + i];
    if (rgb) rgb[(size_t) b * BRICK_NODES + i] = p.rgb[s * BRICK_NODES + i];
    if (M) { M[(size_t) b * BRICK_NODES + i] = p.M[s * BRICK_NODES + i]; ns[(size_t) b * BRICK_NODES + i] = p.ns[s * BRICK_NODES + i]; }
  }
  for (int i = threadIdx.x; i < BRICK_SPLIT_WORDS; i += blockDim.x)
    split[(size_t) b * BRICK_SPLIT_WORDS + i] = p.split[s * BRICK_SPLIT_WORDS + i];
}

__global__ void k_gather_rgbn (Params p, const int* __restrict__ list, int n, float4* __restrict__ out)
{
  int b = blockIdx.x;
  if (b >= n) return;
  size_t s = (size_t) list[b];
  for (int i = threadIdx.x; i < BRICK_NODES; i += blockDim.x) out[(size_t) b * BRICK_NODES + i] = p.rgbn[s * BRICK_NODES + i];
}

// .vol import: claim each brick's slot and copy its payload in
__global__ void k_load_bricks (Params p, const uint64_t* __restrict__ keys, int n, const float2* __restrict__ nodes, const uint32_t* __restrict__ split,
                               const uchar4* __restrict__ rgb, const float* __restrict__ M, const int* __restrict__ ns)
{
  __shared__ int slot_s;
  int b = blockIdx.x;
  if (b >= n) return;
  if (threadIdx.x == 0)
  {
    uint64_t key = keys[b];
    slot_s = find_or_insert_brick (p, (int) (key >> 60) - 1, (int) ((key >> 40) & 0xFFFFF), (int) ((key >> 20) & 0xFFFFF), (int) (key & 0xFFFFF));
  }
  __syncthreads ();
  if (slot_s < 0) return;
  size_t s = (size_t) slot_s;
  for (int i = threadIdx.x; i < BRICK_NODES; i += blockDim.x)
  {
    p.nodes[s * BRICK_NODES + i] = nodes[(size_t) b * BRICK_NODES + i];
    if (p.rgb && rgb) p.rgb[s * BRICK_NODES + i] = rgb[(size_t) b * BRICK_NODES + i];
    if (p.M && M) { p.M[s * BRICK_NODES + i] = M[(size_t) b * BRICK_NODES + i]; p.ns[s * BRICK_NODES + i] = ns[(size_t) b * BRICK_NODES + i]; }
  }
  for (int i = threadIdx.x; i < BRICK_SPLIT_WORDS; i += blockDim.x) p.split[s * BRICK_SPLIT_WORDS + i] = split[(size_t) b * BRICK_SPLIT_WORDS + i];
}

// shard import: scatter coarse-cell (root array) entries
__global__ void k_import_roots (Params p, int n, const int* __restrict__ idx, const float2* __restrict__ dw, const unsigned char* __restrict__ split,
                                const uchar4* __restrict__ rgb, const float* __restrict__ M, const int* __restrict__ ns)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int r = idx[i];
  p.root_dw[r] = dw[i];
  if (split[i]) atomicOr (&p.root_split[r >> 5], 1u << (r & 31)); else atomicAnd (&p.root_split[r >> 5], ~(1u << (r & 31)));
  if (p.root_rgb) p.root_rgb[r] = rgb[i];
  if (p.root_M) { p.root_M[r] = M[i]; p.root_ns[r] = ns[i]; }
}

// ---- marching cubes: one warp per allocated brick, warp-scan compaction of the triangle soup ----
__device__ __forceinline__ bool brick_root_is_split (const Params& p, int t, int bx, int by, int bz)
{
  int R = tier_root_level (p, t);
  if (R < p.C) return true;
  NodePos r;
  if (!locate_node (p, R, bx, by, bz, r)) return false;
  return is_split (p, r);
}

template <bool EMIT>
__global__ void k_mesh_bricks (Params gp, McParams mc, const int* __restrict__ list, int nbricks,
                               unsigned long long* __restrict__ total, float* __restrict__ verts, unsigned char* __restrict__ cols,
                               unsigned long long* __restrict__ okeys)
{
  B2_STAGE_PARAMS (gp)
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (warp >= nbricks) return;
  int slot = list[warp];
  uint64_t key = p.keys[slot];
  int t = (int) (key >> 60) - 1;
  int bx = (int) ((key >> 40) & 0xFFFFF), by = (int) ((key >> 20) & 0xFFFFF), bz = (int) (key & 0xFFFFF);
  int R = tier_root_level (p, t);
  bool root_split = brick_root_is_split (p, t, bx, by, bz);
  if (!root_split) return;                                     // nothing below an unsplit root exists
  const uint32_t* sw = p.split + (size_t) slot * BRICK_SPLIT_WORDS;
  for (int base = 0; base < BRICK_NODES; base += 32)
  {
    int i = base + lane;
    int ntri = 0;
    NodePos n; float2 dw = make_float2 (-1.f, 0.f);
    if (i < BRICK_NODES)
    {
      int k = i < 8 ? 1 : (i < 72 ? 2 : 3);
      int j = i - node_offset (k);
      int level = R + k;
      bool exists = true;
      if (k > 1) { int pj = j >> 3; exists = (sw[split_word_base (k - 1) + (pj >> 5)] >> (pj & 31)) & 1; }
      bool leaf = (level >= p.L) || !((sw[split_word_base (k) + (j >> 5)] >> (j & 31)) & 1);
      if (exists && leaf && level >= p.C)
      {
        int lx = 0, ly = 0, lz = 0;
        for (int q = k - 1; q >= 0; --q) { int c = (j >> (3 * q)) & 7; lx = (lx << 1) | (c >> 2); ly = (ly << 1) | ((c >> 1) & 1); lz = (lz << 1) | (c & 1); }
        n.level = level; n.x = (bx << k) | lx; n.y = (by << k) | ly; n.z = (bz << k) | lz;
        n.cx = center1d (p, level, n.x); n.cy = center1d (p, level, n.y); n.cz = center1d (p, level, n.z);
        n.size = level_size (p, level); n.slot = slot; n.idx = i;
        dw = p.nodes[(size_t) slot * BRICK_NODES + i];
        ntri = mc_leaf (p, mc, n, dw.x, dw.y, b200tsdf_mc::edge_table, b200tsdf_mc::tri_table, nullptr, nullptr);
      }
    }
    // warp-scan compaction: exclusive prefix of triangle counts, one atomic per warp
    int incl = ntri;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync (0xffffffffu, incl, o); if (lane >= o) incl += v; }
    int wtotal = __shfl_sync (0xffffffffu, incl, 31);
    if (wtotal == 0) continue;
    unsigned long long wbase = 0;
    if (lane == 0) wbase = atomicAdd (total, (unsigned long long) wtotal);
    wbase = __shfl_sync (0xffffffffu, wbase, 0);
    if (EMIT && ntri > 0)
    {
      size_t tri0 = (size_t) wbase + (incl - ntri);
      mc_leaf (p, mc, n, dw.x, dw.y, b200tsdf_mc::edge_table, b200tsdf_mc::tri_table,
               verts + tri0 * 9, cols ? cols + tri0 * 9 : nullptr);
      const unsigned long long k = mc_order_key (p, n) << 3;
      for (int t = 0; t < ntri; ++t) okeys[tri0 + t] = k | (unsigned long long) t;
    }
  }
}

// leaves held in the root arrays (unsplit coarse cells when Rtop == C)
template <bool EMIT>
__global__ void k_mesh_roots (Params gp, McParams mc, unsigned long long* __restrict__ total, float* __restrict__ verts, unsigned char* __restrict__ cols,
                              unsigned long long* __restrict__ okeys)
{
  B2_STAGE_PARAMS (gp)
  int n = 1 << p.Rtop;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * n * n || p.Rtop < p.C) return;
  int z = i % n, y = (i / n) % n, x = i / (n * n);
  NodePos nd = make_root (p, x, y, z);
  if (is_split (p, nd)) return;
  float2 dw = p.root_dw[nd.idx];
  int ntri = mc_leaf (p, mc, nd, dw.x, dw.y, b200tsdf_mc::edge_table, b200tsdf_mc::tri_table, nullptr, nullptr);
  if (!ntri) return;
  unsigned long long base = atomicAdd (total, (unsigned long long) ntri);
  if (EMIT)
  {
    mc_leaf (p, mc, nd, dw.x, dw.y, b200tsdf_mc::edge_table, b200tsdf_mc::tri_table, verts + base * 9, cols ? cols + base * 9 : nullptr);
    const unsigned long long k = mc_order_key (p, nd) << 3;
    for (int t = 0; t < ntri; ++t) okeys[base + t] = k | (unsigned long long) t;
  }
}

// ---- Octree::getLeaves: count pass (EMIT = false) and key pass over the stored levels >= C --------------------
// warp-level compaction: one atomic per warp, keys land in emission order (hash layout), sorted afterwards
template <bool EMIT>
__device__ __forceinline__ void leaf_emit_warp (bool emit, unsigned long long key, unsigned long long* total, unsigned long long* keys)
{
  const unsigned m = __ballot_sync (0xffffffffu, emit);
  if (!m) return;
  const int lane = threadIdx.x & 31;
  unsigned long long base = 0;
  if (lane == 0) base = atomicAdd (total, (unsigned long long) __popc (m));
  base = __shfl_sync (0xffffffffu, base, 0);
  if (EMIT && emit) keys[base + __popc (m & ((1u << lane) - 1u))] = key;
}

// one warp per allocated brick; occupied: getOccupiedVoxelIndices' filter on top of getLeaves (leaves, -1)
template <bool EMIT>
__global__ void k_leaf_bricks (Params gp, int nlevels, int occupied, const int* __restrict__ list, int nbricks,
                               unsigned long long* __restrict__ total, unsigned long long* __restrict__ keys)
{
  B2_STAGE_PARAMS (gp)
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (warp >= nbricks) return;
  int slot = list[warp];
  uint64_t key = p.keys[slot];
  int t = (int) (key >> 60) - 1;
  int bx = (int) ((key >> 40) & 0xFFFFF), by = (int) ((key >> 20) & 0xFFFFF), bz = (int) (key & 0xFFFFF);
  int R = tier_root_level (p, t);
  if (!brick_root_is_split (p, t, bx, by, bz)) return;         // nothing below an unsplit root exists
  const uint32_t* sw = p.split + (size_t) slot * BRICK_SPLIT_WORDS;
  for (int base = 0; base < BRICK_NODES; base += 32)
  {
    int i = base + lane;
    bool emit = false; unsigned long long k = 0;
    if (i < BRICK_NODES)
    {
      int kk = i < 8 ? 1 : (i < 72 ? 2 : 3);
      int j = i - node_offset (kk);
      int level = R + kk;
      if (level >= p.C)                                          // levels above C are split by Octree::init: never stored leaves
      {
        // level C exists everywhere, the first level of a brick wherever its root is split (checked above); below, the parent's bit
        bool exists = true;
        if (kk > 1 && level > p.C) { int pj = j >> 3; exists = (sw[split_word_base (kk - 1) + (pj >> 5)] >> (pj & 31)) & 1; }
        bool split = level < p.L && ((sw[split_word_base (kk) + (j >> 5)] >> (j & 31)) & 1);
        emit = exists && leaf_emitted (level, split, nlevels);
        if (emit && occupied) { float2 dw = p.nodes[(size_t) slot * BRICK_NODES + i]; emit = leaf_occupied (dw.x, dw.y); }
        if (EMIT && emit)
        {
          int lx = 0, ly = 0, lz = 0;
          for (int q = kk - 1; q >= 0; --q) { int c = (j >> (3 * q)) & 7; lx = (lx << 1) | (c >> 2); ly = (ly << 1) | ((c >> 1) & 1); lz = (lz << 1) | (c & 1); }
          k = leaf_key (p, level, (bx << kk) | lx, (by << kk) | ly, (bz << kk) | lz);
        }
      }
    }
    leaf_emit_warp<EMIT> (emit, k, total, keys);
  }
}

// the root arrays when they hold the coarse cells (Rtop == C)
template <bool EMIT>
__global__ void k_leaf_roots (Params gp, int nlevels, int occupied, unsigned long long* __restrict__ total, unsigned long long* __restrict__ keys)
{
  B2_STAGE_PARAMS (gp)
  const int n = 1 << p.Rtop;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  bool emit = false; unsigned long long k = 0;
  if (i < n * n * n && p.Rtop == p.C)
  {
    int z = i % n, y = (i / n) % n, x = i / (n * n);
    emit = leaf_emitted (p.C, (p.root_split[i >> 5] >> (i & 31)) & 1, nlevels);
    if (emit && occupied) { float2 dw = p.root_dw[i]; emit = leaf_occupied (dw.x, dw.y); }
    if (EMIT && emit) k = leaf_key (p, p.C, x, y, z);
  }
  leaf_emit_warp<EMIT> (emit, k, total, keys);
}

// getLeaves (leaves, nlevels) for 0 <= nlevels <= C returns every node at level nlevels (all of them exist and the ones above C
// are split), already in key order: the key of the i-th is i's bits moved up to the finest level
__global__ void k_leaf_level (int L, int level, size_t count, unsigned long long* __restrict__ keys)
{
  size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) keys[i] = ((unsigned long long) i << (3 * (L - level) + LEAF_LEVEL_BITS)) | (unsigned long long) level;
}

// key -> OctreeNode::getCenter (the float split accumulation) or, for occupied voxels, getVoxelIndex of that centre
__global__ void k_leaf_decode (Params gp, const unsigned long long* __restrict__ keys, size_t count, float* __restrict__ xyz, int* __restrict__ ijk)
{
  B2_STAGE_PARAMS (gp)
  size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  int level, x, y, z;
  leaf_decode (p, keys[i], level, x, y, z);
  const float cx = center1d (p, level, x), cy = center1d (p, level, y), cz = center1d (p, level, z);
  if (ijk)
  {
    int a, b, c;
    (void) voxel_index (p, cx, cy, cz, a, b, c);                // the reference pushes the index whatever the bool says
    ijk[3 * i] = a; ijk[3 * i + 1] = b; ijk[3 * i + 2] = c;
  }
  else { xyz[3 * i] = cx; xyz[3 * i + 1] = cy; xyz[3 * i + 2] = cz; }
}

} // namespace

// ---------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------
// ---- pinned staging for the host-packed uploads ---------------------------------------------------------------
// The packing threads read the caller's points and write the staging while the copy engine reads the staging: when all of it
// sits behind ONE socket's memory controllers that socket is the bottleneck (measured, tools/microbench/pack_numa.cu: 32 frames
// packed + uploaded in 3.6 ms with input and staging on the same node, 3.1 ms = the PCIe time with the staging elsewhere or
// interleaved).  The staging is therefore interleaved over the NUMA nodes (mbind; best effort — a refusal leaves default
// placement) and then pinned with cudaHostRegister.
struct Staging
{
  unsigned char* p = nullptr; size_t bytes = 0;
  int alloc (size_t n)
  {
    release ();
    const size_t pg = 1ul << 21;                                     // (rounded to 2 MB: friendlier to transparent huge pages)
    n = (n + pg - 1) / pg * pg;
    void* m = mmap (nullptr, n, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (m == MAP_FAILED) return -1;
    unsigned long mask = 0;
    if (FILE* f = std::fopen ("/sys/devices/system/node/has_memory", "r"))
    {
      char line[256] = {};
      if (std::fgets (line, sizeof (line), f))
        for (const char* c = line; *c;)
        {
          char* e = nullptr; const long lo = std::strtol (c, &e, 10); if (e == c) break;
          long hi = lo; if (*e == '-') { const char* b = e + 1; hi = std::strtol (b, &e, 10); if (e == b) break; }
          for (long k = lo; k <= hi && k < 64; ++k) if (k >= 0) mask |= 1ul << k;
          c = e; if (*c == ',') ++c; else break;
        }
      std::fclose (f);
    }
    if (mask & (mask - 1)) (void) syscall (SYS_mbind, m, n, 3 /* MPOL_INTERLEAVE */, &mask, (unsigned long) (8 * sizeof (mask)), 0u);
    std::memset (m, 0, n);                                           // fault the pages in under that policy, before pinning
    if (cudaHostRegister (m, n, cudaHostRegisterDefault) != cudaSuccess) { cudaGetLastError (); munmap (m, n); return -1; }
    p = static_cast<unsigned char*> (m); bytes = n;
    return 0;
  }
  void release ()
  {
    if (!p) return;
    cudaHostUnregister (p); munmap (p, bytes);
    p = nullptr; bytes = 0;
  }
};

struct b200tsdf
{
  b200tsdf_config cfg_pending{}, cfg{};
  bool has_volume = false;
  Params p{};
  int device = 0, sm_count = 148;
  cudaStream_t stream = nullptr, copy_stream = nullptr, gather_stream = nullptr;   // compute | H2D uploads | pack + NVLink all-gather
  size_t pool = 0;
  bool alloc_color = false, alloc_var = false, alloc_norm = false;
  size_t root_n = 0;
  int* d_err = nullptr;
  unsigned char* d_frame[2] = { nullptr, nullptr };
  size_t frame_cap = 0;
  cudaEvent_t ev_copied[2] = { nullptr, nullptr }, ev_consumed[2] = { nullptr, nullptr };
  cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr, ev_k0 = nullptr, ev_k1 = nullptr;
  uint64_t frame_no = 0;
  int count_set = 0;             // which of the two per-frame counter sets the last frame used
  int* d_culled = nullptr; int* d_count = nullptr; unsigned long long* d_stats = nullptr;
  size_t culled_cap = 0;
  bool timed = false;
  bool time_frames = false;      // set between profile_begin / profile_end: per-frame event records (ev_t0/ev_t1 and the ring around the dominant kernel)
  bool is_empty = true;          // TSDFVolumeOctree::is_empty_ (cpp:205, hpp:101)
  // fast-path work queues (levels C .. L-3)
  Queues Q{}; int q_levels = 0; QNode* q_mem = nullptr; size_t q_mem_cap = 0;
  int* d_blist = nullptr; int* d_bail = nullptr; size_t blist_cap = 0;
  // fused per-cell upper sweeps (coarse cells are the top-tier roots and the block roots are <= 3 levels below)
  // supercell path: sl = level of the tier-1 roots, nup = coarse levels above them (swept by k_upper_*), super_static = number of
  // supercells when every tier-1 root is one (coarse cells inside the brick), replayable = the frame's launches read only the record
  int cell_cap = 0; QNode* d_cellq = nullptr; size_t cellq_cap = 0; CellTop* d_celltop = nullptr; QNode* d_superq = nullptr;
  bool top_path = false, replayable = false; int sl = 0, nup = 0, super_static = 0;
  bool fast_path = false; int force_general = 0;
  bool use_pdl = true;           // programmatic dependent launch between the hot kernels (B200TSDF_PDL=0 turns it off)
  int bd_minb = 6;               // resident CTAs per SM the brick kernel is compiled for (80 registers; tuning knob: B200TSDF_BD_MINB=6|8)
  // device copy of Params (the rare out-of-line paths read it through a pointer) and the ring of per-frame records
  Params* d_params = nullptr;
  unsigned long long* d_dbg = nullptr;     // phase-timing counters of k_celltop_up once b200tsdf_debug_timing armed them
  int* h_err = nullptr;                    // pinned image of the device error bits, refreshed behind every frame (see note_device_err)
  FrameRec* d_ring = nullptr; FrameRec* h_ring = nullptr; uint64_t ring_seq = 0;
  cudaEvent_t ev_ring[2] = { nullptr, nullptr };
  // batches (b200tsdf_integrate_batch_device): their own record ring, used half by half, and one captured graph per
  // (half, batch size); a graph is valid until the next reset()
  // device slots: two halves of FRAME_RING / 2 records, reused in stream order; host staging: BATCH_SEGS segments written round
  // robin — the host only waits when it is BATCH_SEGS batches ahead of the device
  FrameRec* d_bring = nullptr; FrameRec* h_bring = nullptr; int bring_half = 0; int bring_seg = 0; bool bring_used[BATCH_SEGS] = {};
  cudaEvent_t ev_bring[BATCH_SEGS] = {};
  cudaEvent_t ev_half_done[2] = { nullptr, nullptr }; bool half_used[2] = { false, false }; FrameRec* batch_recs = nullptr;
  cudaGraphExec_t batch_exec[2][FRAME_RING / 2 + 1] = {};
  // multi-GPU (multigpu.cuh): NCCL communicator (opaque here), row-sliced uploads
  void* comm = nullptr; int comm_rank = 0, comm_size = 1;
  unsigned char* d_rows_raw[2] = { nullptr, nullptr }; unsigned char* d_rows_full[2] = { nullptr, nullptr };
  size_t rows_raw_cap = 0, rows_full_cap = 0; int rows_set = 0; bool rows_used[2] = { false, false }; int rows_last_up[2] = { 0, 0 };
  int rows_chunk = 0;            // frames per upload/fuse pipeline stage of b200tsdf_integrate_batch_rows (B200TSDF_ROWS_CHUNK=1..32; 0: 1 or 2 with host packing, else 8)
  cudaEvent_t ev_rows_up[2][32] = {}, ev_rows_ready[2][32] = {}, ev_rows_done[2] = { nullptr, nullptr };
  // host packing of the uploaded rows (host_pack.h): pinned staging per buffer set, the pool is created on first use
  int host_pack = -1;            // B200TSDF_HOST_PACK: 1 pack on the host, 0 upload the caller's points as they are (packed on the device when gathered); -1 by rank count
  int pack_threads = 0;          // B200TSDF_PACK_THREADS (0 = min (16, hardware threads / (2 ranks)))
  b2host::PackPool* pack_pool = nullptr;
  Staging h_pack[2]; size_t pack_cap = 0;
  Staging h_fpack[2];            // the same for the frame-at-a-time upload (d_frame[]), frame_cap bytes each
  long long nvlink_bytes = 0, prof_nvlink0 = 0;
  int launches_per_frame = 0; long long graph_launches = 0, prof_graph0 = 0;
  // measurement
  cudaEvent_t ev_p0 = nullptr, ev_p1 = nullptr;
  cudaEvent_t kring[KRING][2] = {};
  int kring_head = 0, kring_pending = 0;
  double prof_ms_kernel = 0; long long prof_kernel_launches = 0, prof_frames = 0;
  long long launches = 0, prof_launch0 = 0, h2d_bytes = 0, d2h_bytes = 0, prof_h2d0 = 0, prof_d2h0 = 0;
  unsigned long long prof_stats0[ST_N] = {};
  void drain_kring (int keep)
  {
    while (kring_pending > keep)
    {
      int i = (kring_head - kring_pending + 4 * KRING) % KRING;
      float ms = 0.f;
      cudaEventSynchronize (kring[i][1]);
      if (cudaEventElapsedTime (&ms, kring[i][0], kring[i][1]) == cudaSuccess) { prof_ms_kernel += ms; prof_kernel_launches++; }
      kring_pending--;
    }
  }
  std::string err;
  float* mesh_v = nullptr; unsigned char* mesh_c = nullptr;
  float* leaf_xyz = nullptr; int32_t* leaf_ijk = nullptr;   // last getVoxelCenters / getOccupiedVoxelIndices result (host)
  // grow-only device scratch for the read-side calls (queries, render): no allocation per call
  unsigned char* d_scratch = nullptr; size_t scratch_cap = 0;
  int scratch (size_t bytes)
  {
    if (bytes <= scratch_cap) return 0;
    cudaFree (d_scratch); d_scratch = nullptr; scratch_cap = 0;
    size_t want = bytes + bytes / 2 + 4096;
    if (cudaMalloc (&d_scratch, want) != cudaSuccess) return fail (B200TSDF_ENOMEM, "device scratch allocation failed");
    scratch_cap = want;
    return 0;
  }

  int fail (int code, const std::string& m) { err = m; return code; }
};

namespace {

void free_volume (b200tsdf* h)
{
  cudaFree (h->p.work); h->p.work = nullptr;
  cudaFree (h->p.keys); cudaFree (h->p.nodes); cudaFree (h->p.split); cudaFree (h->p.rgb); cudaFree (h->p.M); cudaFree (h->p.ns);
  cudaFree (h->p.root_dw); cudaFree (h->p.root_split); cudaFree (h->p.root_rgb); cudaFree (h->p.root_M); cudaFree (h->p.root_ns);
  cudaFree (h->p.rgbn); cudaFree (h->p.root_rgbn); h->p.rgbn = nullptr; h->p.root_rgbn = nullptr;
  h->p.keys = nullptr; h->p.nodes = nullptr; h->p.split = nullptr; h->p.rgb = nullptr; h->p.M = nullptr; h->p.ns = nullptr;
  h->p.root_dw = nullptr; h->p.root_split = nullptr; h->p.root_rgb = nullptr; h->p.root_M = nullptr; h->p.root_ns = nullptr;
  h->pool = 0; h->root_n = 0;
}

// launch with programmatic stream serialization (see pdl_wait in brick_kernels.cuh); also valid inside a stream capture
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl (void (*kernel) (KArgs...), dim3 grid, dim3 block, cudaStream_t s, Args... args)
{
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx (&cfg, kernel, KArgs (args)...);
}

void comm_release (b200tsdf* h);          // multigpu.cuh

void drop_batch_graphs (b200tsdf* h)
{
  for (int a = 0; a < 2; ++a)
    for (int n = 0; n <= FRAME_RING / 2; ++n)
      if (h->batch_exec[a][n]) { cudaGraphExecDestroy (h->batch_exec[a][n]); h->batch_exec[a][n] = nullptr; }
}

int check_device_err (b200tsdf* h)
{
  int e = 0;
  if (cudaMemcpyAsync (&e, h->d_err, sizeof (int), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) return h->fail (B200TSDF_ECUDA, "error flag readback failed");
  if (cudaStreamSynchronize (h->stream) != cudaSuccess) return h->fail (B200TSDF_ECUDA, std::string ("stream: ") + cudaGetErrorString (cudaGetLastError ()));
  if (e & ERR_POOL_FULL) return h->fail (B200TSDF_ENOMEM, "brick pool exhausted (raise pool_log2)");
  if (e & ERR_MISSING_BRICK) return h->fail (B200TSDF_ESTATE, "internal: split node without brick");
  if (e & ERR_QUEUE_FULL) return h->fail (B200TSDF_ENOMEM, "internal: work queue overflow");
  return 0;
}

// Deferred error reporting for the calls that do not wait for their kernels: a 4-byte copy of the (sticky) device error bits
// into pinned memory is queued behind the work, and every entry point looks at the pinned word first.  An overflow
// (pool, queue) or an inconsistency is therefore reported by the call that follows the frame which hit it, at the latest
// by b200tsdf_sync / get_stats / mesh / save, instead of being served silently (ADVICE r1).
int pending_device_err (b200tsdf* h)
{
  const int e = *(volatile int*) h->h_err;
  if (!e) return 0;
  if (e & ERR_POOL_FULL) return h->fail (B200TSDF_ENOMEM, "brick pool exhausted in an earlier frame (raise pool_log2); the volume is incomplete");
  if (e & ERR_MISSING_BRICK) return h->fail (B200TSDF_ESTATE, "internal: split node without brick (earlier frame)");
  return h->fail (B200TSDF_ENOMEM, "internal: work queue overflow in an earlier frame; the volume is incomplete");
}
void note_device_err (b200tsdf* h, cudaStream_t s) { cudaMemcpyAsync (h->h_err, h->d_err, sizeof (int), cudaMemcpyDeviceToHost, s); }

void fill_frame (const b200tsdf* h, Frame& f, const unsigned char* d_pts, size_t stride, int xyz_off, int rgba_off, int W, int H, const double* pose)
{
  f.pts = d_pts; f.stride = (int) stride; f.xyz_off = xyz_off; f.rgba_off = h->p.color ? rgba_off : -1; f.width = W; f.height = H;
  double inv[12];
  b2host::affine_inverse (pose, inv);                                 // hpp:54: trans.inverse ().cast<float> ()
  for (int i = 0; i < 12; ++i) { f.tinv[i] = (float) inv[i]; f.tfwd[i] = (float) pose[i]; }
}

} // namespace

extern "C" {

void b200tsdf_default_config (b200tsdf_config* c) { if (c) default_config (c); }

int b200tsdf_create (const b200tsdf_config* cfg, b200tsdf_t** out)
{
  if (!out) return B200TSDF_EINVAL;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount (&ndev) != cudaSuccess || ndev == 0) return B200TSDF_ENODEVICE;
  b200tsdf* h = new b200tsdf;
  if (cfg) h->cfg_pending = *cfg; else b200tsdf_default_config (&h->cfg_pending);
  h->device = h->cfg_pending.device;
  if (const char* e = std::getenv ("B200TSDF_PDL")) h->use_pdl = std::atoi (e) != 0;
  if (const char* e = std::getenv ("B200TSDF_ROWS_CHUNK")) { const int v = std::atoi (e); if (v >= 1 && v <= 32) h->rows_chunk = v; }
  if (const char* e = std::getenv ("B200TSDF_HOST_PACK")) h->host_pack = std::atoi (e) != 0 ? 1 : 0;
  if (const char* e = std::getenv ("B200TSDF_PACK_THREADS")) { const int v = std::atoi (e); if (v >= 1 && v <= 256) h->pack_threads = v; }
  if (const char* e = std::getenv ("B200TSDF_BD_MINB")) { const int v = std::atoi (e); if (v == 6 || v == 8) h->bd_minb = v; }
  if (h->device < 0 || h->device >= ndev) { delete h; return B200TSDF_EINVAL; }
  bool ok = cudaSetDevice (h->device) == cudaSuccess
         && cudaDeviceGetAttribute (&h->sm_count, cudaDevAttrMultiProcessorCount, h->device) == cudaSuccess
         && cudaStreamCreateWithFlags (&h->stream, cudaStreamNonBlocking) == cudaSuccess
         && cudaStreamCreateWithFlags (&h->copy_stream, cudaStreamNonBlocking) == cudaSuccess
         && cudaStreamCreateWithFlags (&h->gather_stream, cudaStreamNonBlocking) == cudaSuccess
         && cudaMalloc (&h->d_err, sizeof (int)) == cudaSuccess
         && cudaMalloc (&h->d_count, 64 * sizeof (int)) == cudaSuccess
         && cudaMalloc (&h->d_stats, ST_TOTAL * sizeof (unsigned long long)) == cudaSuccess
         && cudaMalloc (&h->d_params, sizeof (Params)) == cudaSuccess
         && cudaHostAlloc (&h->h_err, sizeof (int), cudaHostAllocDefault) == cudaSuccess
         && cudaMalloc (&h->d_ring, FRAME_RING * sizeof (FrameRec)) == cudaSuccess
         && cudaHostAlloc (&h->h_ring, FRAME_RING * sizeof (FrameRec), cudaHostAllocDefault) == cudaSuccess
         && cudaEventCreateWithFlags (&h->ev_ring[0], cudaEventDisableTiming) == cudaSuccess
         && cudaEventCreateWithFlags (&h->ev_ring[1], cudaEventDisableTiming) == cudaSuccess
         && cudaMalloc (&h->d_bring, FRAME_RING * sizeof (FrameRec)) == cudaSuccess
         && cudaHostAlloc (&h->h_bring, (size_t) BATCH_SEGS * (FRAME_RING / 2) * sizeof (FrameRec), cudaHostAllocDefault) == cudaSuccess
         && cudaEventCreateWithFlags (&h->ev_rows_done[0], cudaEventDisableTiming) == cudaSuccess
         && cudaEventCreateWithFlags (&h->ev_rows_done[1], cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; ok && i < BATCH_SEGS; ++i) ok = cudaEventCreateWithFlags (&h->ev_bring[i], cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; ok && i < 2; ++i) ok = cudaEventCreateWithFlags (&h->ev_half_done[i], cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; ok && i < 2; ++i)
    ok = cudaEventCreateWithFlags (&h->ev_copied[i], cudaEventDisableTiming) == cudaSuccess
      && cudaEventCreateWithFlags (&h->ev_consumed[i], cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaEventCreate (&h->ev_t0) == cudaSuccess && cudaEventCreate (&h->ev_t1) == cudaSuccess
          && cudaEventCreate (&h->ev_k0) == cudaSuccess && cudaEventCreate (&h->ev_k1) == cudaSuccess
          && cudaEventCreate (&h->ev_p0) == cudaSuccess && cudaEventCreate (&h->ev_p1) == cudaSuccess;
  for (int i = 0; ok && i < 64; ++i) ok = cudaEventCreateWithFlags (&h->ev_rows_ready[i / 32][i % 32], cudaEventDisableTiming) == cudaSuccess
                                          && cudaEventCreateWithFlags (&h->ev_rows_up[i / 32][i % 32], cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; ok && i < KRING; ++i)
    ok = cudaEventCreate (&h->kring[i][0]) == cudaSuccess && cudaEventCreate (&h->kring[i][1]) == cudaSuccess;
  if (ok) *h->h_err = 0;
  if (ok) { cudaMemset (h->d_err, 0, sizeof (int)); cudaMemset (h->d_stats, 0, ST_TOTAL * sizeof (unsigned long long)); }
  // the depth-first general path recurses up to (L - C + 1) levels
  if (ok) cudaDeviceSetLimit (cudaLimitStackSize, 16384);
  if (!ok) { b200tsdf_destroy (h); return B200TSDF_ECUDA; }
  *out = h;
  return B200TSDF_OK;
}

void b200tsdf_destroy (b200tsdf_t* h)
{
  if (!h) return;
  cudaSetDevice (h->device);
  if (h->stream) cudaStreamSynchronize (h->stream);
  if (h->copy_stream) cudaStreamSynchronize (h->copy_stream);
  if (h->gather_stream) cudaStreamSynchronize (h->gather_stream);
  free_volume (h);
  cudaFree (h->d_err); cudaFree (h->d_count); cudaFree (h->d_stats); cudaFree (h->d_culled); cudaFree (h->d_scratch);
  cudaFree (h->d_dbg); if (h->h_err) cudaFreeHost (h->h_err);
  cudaFree (h->d_params); cudaFree (h->d_ring); if (h->h_ring) cudaFreeHost (h->h_ring);
  for (int i = 0; i < 2; ++i) if (h->ev_ring[i]) cudaEventDestroy (h->ev_ring[i]);
  drop_batch_graphs (h);
  comm_release (h);
  delete h->pack_pool; h->pack_pool = nullptr;
  for (int i = 0; i < 2; ++i)
  {
    cudaFree (h->d_rows_raw[i]); cudaFree (h->d_rows_full[i]);
    h->h_pack[i].release (); h->h_fpack[i].release ();
    for (int k = 0; k < 32; ++k) { if (h->ev_rows_ready[i][k]) cudaEventDestroy (h->ev_rows_ready[i][k]); if (h->ev_rows_up[i][k]) cudaEventDestroy (h->ev_rows_up[i][k]); }
    if (h->ev_rows_done[i]) cudaEventDestroy (h->ev_rows_done[i]);
  }
  cudaFree (h->d_bring); if (h->h_bring) cudaFreeHost (h->h_bring);
  for (int i = 0; i < BATCH_SEGS; ++i) if (h->ev_bring[i]) cudaEventDestroy (h->ev_bring[i]);
  for (int i = 0; i < 2; ++i) if (h->ev_half_done[i]) cudaEventDestroy (h->ev_half_done[i]);
  cudaFree (h->d_frame[0]); cudaFree (h->d_frame[1]); cudaFree (h->q_mem); cudaFree (h->d_blist); cudaFree (h->d_bail); cudaFree (h->d_cellq); cudaFree (h->d_superq); cudaFree (h->d_celltop);
  for (int i = 0; i < 2; ++i) { if (h->ev_copied[i]) cudaEventDestroy (h->ev_copied[i]); if (h->ev_consumed[i]) cudaEventDestroy (h->ev_consumed[i]); }
  if (h->ev_t0) cudaEventDestroy (h->ev_t0); if (h->ev_t1) cudaEventDestroy (h->ev_t1);
  if (h->ev_k0) cudaEventDestroy (h->ev_k0); if (h->ev_k1) cudaEventDestroy (h->ev_k1);
  if (h->ev_p0) cudaEventDestroy (h->ev_p0); if (h->ev_p1) cudaEventDestroy (h->ev_p1);
  for (int i = 0; i < KRING; ++i) { if (h->kring[i][0]) cudaEventDestroy (h->kring[i][0]); if (h->kring[i][1]) cudaEventDestroy (h->kring[i][1]); }
  if (h->stream) cudaStreamDestroy (h->stream);
  if (h->copy_stream) cudaStreamDestroy (h->copy_stream);
  if (h->gather_stream) cudaStreamDestroy (h->gather_stream);
  std::free (h->mesh_v); std::free (h->mesh_c);
  std::free (h->leaf_xyz); std::free (h->leaf_ijk);
  delete h;
}

const char* b200tsdf_last_error (const b200tsdf_t* h) { return h ? h->err.c_str () : "null handle"; }

int b200tsdf_set_config (b200tsdf_t* h, const b200tsdf_config* cfg)
{
  if (!h || !cfg) return B200TSDF_EINVAL;
  int dev = h->cfg_pending.device;
  h->cfg_pending = *cfg;
  h->cfg_pending.device = dev;               // a handle is bound to its device at creation
  // setGlobalTransform is the one setter that does not wait for reset () in the reference: global_transform_ is only read by
  // save () and the mesher (tsdf_volume_octree.h:131-133, cpp:242, marching_cubes_tsdf_octree.cpp:122-128)
  std::memcpy (h->cfg.global_transform, cfg->global_transform, sizeof (h->cfg.global_transform));
  return B200TSDF_OK;
}

int b200tsdf_get_config (const b200tsdf_t* h, b200tsdf_config* cfg)
{
  if (!h || !cfg) return B200TSDF_EINVAL;
  *cfg = h->cfg_pending;
  return B200TSDF_OK;
}

// ---- reset (tsdf_volume_octree.cpp:201-219, Octree::init octree.cpp:584-599) --------------------
int b200tsdf_reset (b200tsdf_t* h)
{
  if (!h) return B200TSDF_EINVAL;
  cudaSetDevice (h->device);
  const b200tsdf_config& c = h->cfg_pending;
  Params np = h->p;
  size_t pool = 0, root_n = 0;
  if (const char* msg = derive_params (c, np, pool, root_n)) return h->fail (B200TSDF_EINVAL, msg);
  bool color = np.color != 0, var = np.track_var != 0, norm = np.color_norm != 0;
  int C = np.C, Rtop = np.Rtop;

  CK (cudaStreamSynchronize (h->stream));
  CK (cudaStreamSynchronize (h->copy_stream));
  drop_batch_graphs (h);                                   // captured launches carry the old configuration
  for (int i = 0; i < BATCH_SEGS; ++i) h->bring_used[i] = false;
  h->half_used[0] = h->half_used[1] = false;
  if (pool != h->pool || root_n != h->root_n || color != h->alloc_color || var != h->alloc_var || norm != h->alloc_norm)
  {
    h->has_volume = false;                                 // a failed allocation below must not leave a half-built volume usable
    free_volume (h);
    CK (cudaMalloc (&h->p.keys, pool * sizeof (uint64_t)));
    CK (cudaMalloc (&h->p.nodes, pool * BRICK_NODES * sizeof (float2)));
    CK (cudaMalloc (&h->p.split, pool * BRICK_SPLIT_WORDS * sizeof (uint32_t)));
    CK (cudaMalloc (&h->p.work, pool));
    if (color) CK (cudaMalloc (&h->p.rgb, pool * BRICK_NODES * sizeof (uchar4)));
    if (var) { CK (cudaMalloc (&h->p.M, pool * BRICK_NODES * sizeof (float))); CK (cudaMalloc (&h->p.ns, pool * BRICK_NODES * sizeof (int))); }
    CK (cudaMalloc (&h->p.root_dw, root_n * sizeof (float2)));
    CK (cudaMalloc (&h->p.root_split, ((root_n + 31) / 32) * sizeof (uint32_t)));
    if (color) CK (cudaMalloc (&h->p.root_rgb, root_n * sizeof (uchar4)));
    if (norm) { CK (cudaMalloc (&h->p.rgbn, pool * BRICK_NODES * sizeof (float4))); CK (cudaMalloc (&h->p.root_rgbn, root_n * sizeof (float4))); }
    if (var) { CK (cudaMalloc (&h->p.root_M, root_n * sizeof (float))); CK (cudaMalloc (&h->p.root_ns, root_n * sizeof (int))); }
    h->pool = pool; h->root_n = root_n; h->alloc_color = color; h->alloc_var = var; h->alloc_norm = norm;
  }
  size_t ncells = (size_t) 1 << (3 * C);
  if (ncells > h->culled_cap)
  {
    cudaFree (h->d_culled); h->d_culled = nullptr;
    CK (cudaMalloc (&h->d_culled, ncells * sizeof (int)));
    h->culled_cap = ncells;
  }
  {
    // work queues for levels C .. B = L-3 (fast path needs the block-root level at or below the coarse depth)
    int Bl = np.L - 3;
    h->force_general = c.debug_flags & 1;
    h->fast_path = (Bl >= np.C) && !var && !np.color_norm && !h->force_general && (Bl - np.C + 1 <= MAX_QLEVELS);
    h->q_levels = h->fast_path ? (Bl - np.C + 1) : 0;
    size_t total = 0; size_t caps[MAX_QLEVELS] = {};
    for (int i = 0; i < h->q_levels; ++i)
    {
      int lv = np.C + i;
      size_t full = lv >= 7 ? ((size_t) 1 << 21) : ((size_t) 1 << (3 * lv));
      caps[i] = std::min (full, (size_t) 1 << 21);
      total += caps[i];
    }
    if (total > h->q_mem_cap)
    {
      cudaFree (h->q_mem); h->q_mem = nullptr; h->q_mem_cap = 0;
      CK (cudaMalloc (&h->q_mem, total * sizeof (QNode)));
      h->q_mem_cap = total;
    }
    size_t off = 0;
    for (int i = 0; i < MAX_QLEVELS; ++i) { h->Q.q[i] = nullptr; h->Q.cap[i] = 0; }
    for (int i = 0; i < h->q_levels; ++i) { h->Q.q[i] = h->q_mem + off; h->Q.cap[i] = (int) caps[i]; off += caps[i]; }
    h->Q.n = h->d_count;
    // supercell path (k_celltop_down / k_bricks / k_celltop_up, brick_kernels.cuh): needs tier-1 bricks (T >= 2), whose roots sit
    // at level SL = L - 6.  Coarse levels above SL are swept by k_upper_*; coarse cells below SL are handled inside the brick.
    h->sl = np.L - 6;
    h->nup = std::max (0, h->sl - np.C);
    h->super_static = 0;
    h->top_path = h->fast_path && np.T >= 2 && h->sl >= 0 && !(c.debug_flags & 6);
    if (h->top_path && np.C > h->sl)
    {
      // every tier-1 root is a supercell; they must be the root-array nodes (T == 2) and fit the per-cell scratch
      if (np.Rtop != h->sl || h->sl > 4) h->top_path = false;
      else h->super_static = 1 << (3 * h->sl);
    }
    if (h->top_path)
    {
      h->cell_cap = 16384;
      size_t need = (size_t) h->cell_cap * 585;
      if (need > h->cellq_cap)
      {
        cudaFree (h->d_cellq); cudaFree (h->d_celltop); h->d_cellq = nullptr; h->d_celltop = nullptr; h->cellq_cap = 0;
        CK (cudaMalloc (&h->d_cellq, need * sizeof (QNode)));
        CK (cudaMalloc (&h->d_celltop, (size_t) h->cell_cap * sizeof (CellTop)));
        h->cellq_cap = need;
      }
      if (h->super_static && !h->d_superq) CK (cudaMalloc (&h->d_superq, 4096 * sizeof (QNode)));
    }
    h->replayable = h->fast_path;                         // every kernel of the brick paths reads the frame from its record (the general depth-first kernel takes it by value)
    size_t bl = h->q_levels ? caps[h->q_levels - 1] : 0;
    if (h->top_path) bl = std::max (bl, (size_t) h->cell_cap * 512);
    if (bl > h->blist_cap)
    {
      cudaFree (h->d_blist); cudaFree (h->d_bail); h->d_blist = h->d_bail = nullptr; h->blist_cap = 0;
      CK (cudaMalloc (&h->d_blist, bl * BL_CLASSES * sizeof (int)));          // one list per work class
      CK (cudaMalloc (&h->d_bail, bl * sizeof (int)));
      h->blist_cap = bl;
    }
  }
  Params& p = h->p;
  {
    // keep the storage pointers, take every scalar from the derived set
    Params st = p;
    p = np;
    p.work = st.work;
    p.keys = st.keys; p.nodes = st.nodes; p.split = st.split; p.rgb = st.rgb; p.M = st.M; p.ns = st.ns;
    p.root_dw = st.root_dw; p.root_split = st.root_split; p.root_rgb = st.root_rgb; p.root_M = st.root_M; p.root_ns = st.root_ns;
    p.rgbn = st.rgbn; p.root_rgbn = st.root_rgbn;
  }
  p.err = h->d_err;
  p.diag = h->d_stats + 3;
  p.dbg = h->d_dbg;
  CK (cudaMemcpyAsync (h->d_params, &p, sizeof (Params), cudaMemcpyHostToDevice, h->stream));
  CK (cudaStreamSynchronize (h->stream));                            // (&p is host memory that may change after reset)
  // fresh state everywhere (OctreeNode ctor: d=-1, w=0; octree.h:71-74)
  cudaStream_t s = h->stream;
  CK (cudaMemsetAsync (p.keys, 0, pool * sizeof (uint64_t), s));
  CK (cudaMemsetAsync (p.split, 0, pool * BRICK_SPLIT_WORDS * sizeof (uint32_t), s));
  CK (cudaMemsetAsync (p.work, 0, pool, s));
  k_fill_fresh<<<148 * 8, 256, 0, s>>> (p.nodes, pool * BRICK_NODES);
  if (color) CK (cudaMemsetAsync (p.rgb, 0, pool * BRICK_NODES * sizeof (uchar4), s));
  if (var) { CK (cudaMemsetAsync (p.M, 0, pool * BRICK_NODES * sizeof (float), s)); CK (cudaMemsetAsync (p.ns, 0, pool * BRICK_NODES * sizeof (int), s)); }
  k_fill_fresh<<<64, 256, 0, s>>> (p.root_dw, root_n);
  CK (cudaMemsetAsync (p.root_split, 0, ((root_n + 31) / 32) * sizeof (uint32_t), s));
  if (color) CK (cudaMemsetAsync (p.root_rgb, 0, root_n * sizeof (uchar4), s));
  if (norm) { CK (cudaMemsetAsync (p.rgbn, 0, pool * BRICK_NODES * sizeof (float4), s)); CK (cudaMemsetAsync (p.root_rgbn, 0, root_n * sizeof (float4), s)); }
  if (var) { CK (cudaMemsetAsync (p.root_M, 0, root_n * sizeof (float), s)); CK (cudaMemsetAsync (p.root_ns, 0, root_n * sizeof (int), s)); }
  CK (cudaMemsetAsync (h->d_err, 0, sizeof (int), s));
  *h->h_err = 0;
  CK (cudaMemsetAsync (h->d_count, 0, 64 * sizeof (int), s));
  h->count_set = 0;
  CK (cudaMemsetAsync (h->d_stats, 0, ST_TOTAL * sizeof (unsigned long long), s));
  h->kring_pending = 0; h->kring_head = 0;
  if (Rtop < C) k_insert_top_bricks<<<(unsigned) ((root_n + 127) / 128), 128, 0, s>>> (p);
  if (h->top_path && h->super_static) k_build_superq<<<(h->super_static + 127) / 128, 128, 0, s>>> (p, h->d_superq, h->super_static);
  CK (cudaGetLastError ());
  h->cfg = c;
  h->has_volume = true;
  h->frame_no = 0;
  h->timed = false;
  h->is_empty = true;
  return check_device_err (h);
}

// ---- integrateCloud (hpp:48-103) ------------------------------------------------------------------
// The frame's parameters (pose, planes, cloud pointer, counter set) are written into a FrameRec; the hot kernels
// read it from the device ring, so the very same launches can be captured once into a CUDA graph and replayed.
static void fill_rec (b200tsdf* h, FrameRec& r, const unsigned char* d_pts, size_t stride, int xyz_off, int rgba_off, int W, int H, const double* pose)
{
  const Params& p = h->p;
  fill_frame (h, r.f, d_pts, stride, xyz_off, rgba_off, W, H, pose);
  b2host::frustum_planes (pose, p.width, p.height, p.fx, p.fy, p.min_sensor, p.max_sensor, r.pl);
  h->count_set ^= 1;                                                  // counter sets alternate between frames
  r.cset = h->count_set;
  r.timing = h->time_frames ? 1 : 0;
  r.pad_[0] = r.pad_[1] = 0; r.kt[0] = r.kt[1] = 0;
}

// the launches of one frame.  `rec` is the host image of *d_rec (only the paths that are not replayable read it).
// with_events: bracket the dominant kernel with an event pair of the ring (never inside a capture)
static int launch_frame (b200tsdf* h, cudaStream_t s, const FrameRec& rec, const FrameRec* d_rec, bool with_events)
{
  const Params& p = h->p;
  const Frame& f = rec.f;
  int* cnt = h->d_count + 16 * rec.cset;
  const int npix = f.width * f.height;
  const int ncells = 1 << (3 * p.C);
  {
    const int cull_blocks = (ncells + 255) / 256;
    const bool pdl = h->replayable && h->use_pdl;
    if (pdl) CK (launch_pdl (k_front, dim3 (cull_blocks + (npix + 255) / 256), dim3 (256), s, p, d_rec, cull_blocks, h->d_culled, h->d_count, h->Q.q[0], h->d_stats));
    else k_front<<<cull_blocks + (npix + 255) / 256, 256, 0, s>>> (p, d_rec, cull_blocks, h->d_culled, h->d_count, h->fast_path ? h->Q.q[0] : nullptr, h->d_stats);
  }
  h->launches += 1;
  int kr = -1;
  if (with_events)
  {
    if (h->kring_pending >= KRING) h->drain_kring (KRING / 2);
    kr = h->kring_head;
  }
  if (h->fast_path)
  {
    const int nl = h->q_levels;
    QNode* bq = nullptr;                                   // the queue the block-root entries of k_bricks live in
    if (h->top_path)
    {
      // coarse levels above the supercells, top-down (none for 2048^3 / 10 m and 512^3 / 3 m)
      for (int li = 0; li < h->nup; ++li) { k_upper_down<<<148 * 2, 128, 0, s>>> (p, d_rec, h->Q, li, 0, h->d_blist, h->d_stats); h->launches++; }
      QNode* cells = h->super_static ? h->d_superq : h->Q.q[h->nup];
      const int qslot = h->super_static ? -1 : h->nup;
      auto kd = p.color ? k_celltop_down<true> : k_celltop_down<false>;
      if (h->use_pdl) CK (launch_pdl (kd, dim3 (h->sm_count * 4), dim3 (TOP_THREADS), s, p, d_rec, cells, h->d_count, h->d_cellq, h->d_celltop, h->cell_cap, h->d_blist, (int) h->blist_cap, h->d_stats, h->sl, qslot, h->super_static));
      else kd<<<h->sm_count * 4, TOP_THREADS, 0, s>>> (p, d_rec, cells, h->d_count, h->d_cellq, h->d_celltop, h->cell_cap, h->d_blist, (int) h->blist_cap, h->d_stats, h->sl, qslot, h->super_static);
      h->launches++;
      bq = h->d_cellq;
    }
    else
    {
      for (int li = 0; li < nl; ++li) { k_upper_down<<<148 * 2, 128, 0, s>>> (p, d_rec, h->Q, li, li == nl - 1, h->d_blist, h->d_stats); h->launches++; }
      bq = h->Q.q[nl - 1];
    }
    if (kr >= 0) CK (cudaEventRecord (h->kring[kr][0], s));
    // the dominant kernel: one warp per interior block root, the brick updated in place
    {
      auto kb = h->bd_minb == 6 ? (p.color ? k_bricks<true, 6> : k_bricks<false, 6>) : (p.color ? k_bricks<true, 8> : k_bricks<false, 8>);
      const dim3 g (h->sm_count * h->bd_minb), b (BD_WARPS * 32);
      if (h->top_path && h->use_pdl) CK (launch_pdl (kb, g, b, s, p, (const Params*) h->d_params, d_rec, bq, (const int*) h->d_blist, (int) h->blist_cap, h->d_count, h->d_stats, p.L - 3));
      else kb<<<g, b, 0, s>>> (p, h->d_params, d_rec, bq, h->d_blist, (int) h->blist_cap, h->d_count, h->d_stats, p.L - 3);
    }
    if (kr >= 0) CK (cudaEventRecord (h->kring[kr][1], s));
    h->launches++;
    if (h->top_path)
    {
      QNode* cells = h->super_static ? h->d_superq : h->Q.q[h->nup];
      const int qslot = h->super_static ? -1 : h->nup;
      auto ku = p.color ? k_celltop_up<true> : k_celltop_up<false>;
      if (h->use_pdl) CK (launch_pdl (ku, dim3 (h->sm_count), dim3 (128), s, p, d_rec, cells, (const int*) h->d_count, (const QNode*) h->d_cellq, (const CellTop*) h->d_celltop, h->cell_cap, h->d_stats, h->sl, qslot, h->super_static));
      else ku<<<h->sm_count, 128, 0, s>>> (p, d_rec, cells, h->d_count, h->d_cellq, h->d_celltop, h->cell_cap, h->d_stats, h->sl, qslot, h->super_static);
      h->launches++;
      for (int li = h->nup - 1; li >= 0; --li) { k_upper_up<<<148 * 2, 128, 0, s>>> (p, d_rec, h->Q, li, h->d_stats); h->launches++; }
    }
    else
      for (int li = nl - 2; li >= 0; --li) { k_upper_up<<<148 * 2, 128, 0, s>>> (p, d_rec, h->Q, li, h->d_stats); h->launches++; }
  }
  else
  {
    if (kr >= 0) CK (cudaEventRecord (h->kring[kr][0], s));
    // general path: every culled cell depth-first (grid covers the worst case; threads past *count exit)
    k_update_dfs<<<(ncells + 31) / 32, 32, 0, s>>> (p, f, h->d_culled, cnt, h->d_stats);
    if (kr >= 0) CK (cudaEventRecord (h->kring[kr][1], s));
    h->launches++;
  }
  if (kr >= 0) { h->kring_head = (kr + 1) % KRING; h->kring_pending++; }
  h->prof_frames++;
  return B200TSDF_OK;
}

// a slot of the record ring for the next frame: the host image is only rewritten once the copy that read it FRAME_RING
// frames ago has certainly executed
static int ring_slot (b200tsdf* h, int& slot)
{
  slot = (int) (h->ring_seq % FRAME_RING);
  const int half = FRAME_RING / 2;
  if (h->ring_seq >= (uint64_t) FRAME_RING && slot % half == 0) CK (cudaEventSynchronize (h->ev_ring[slot / half]));
  return B200TSDF_OK;
}
static int ring_advance (b200tsdf* h, int slot, cudaStream_t s)
{
  const int half = FRAME_RING / 2;
  if (slot % half == half - 1) CK (cudaEventRecord (h->ev_ring[slot / half], s));   // covers the copies of this half
  h->ring_seq++;
  return B200TSDF_OK;
}

static int integrate_on_device (b200tsdf* h, const unsigned char* d_pts, size_t stride, int xyz_off, int rgba_off, int W, int H, const double* pose)
{
  cudaStream_t s = h->stream;
  if (int rc = pending_device_err (h)) return rc;
  int slot = 0;
  { int rc = ring_slot (h, slot); if (rc) return rc; }
  FrameRec& rec = h->h_ring[slot];
  fill_rec (h, rec, d_pts, stride, xyz_off, rgba_off, W, H, pose);
  if (h->time_frames) CK (cudaEventRecord (h->ev_t0, s));
  CK (cudaMemcpyAsync (h->d_ring + slot, &rec, sizeof (FrameRec), cudaMemcpyHostToDevice, s));
  { int rc = launch_frame (h, s, rec, h->d_ring + slot, h->time_frames); if (rc) return rc; }
  if (h->time_frames) CK (cudaEventRecord (h->ev_t1, s));
  note_device_err (h, s);
  { int rc = ring_advance (h, slot, s); if (rc) return rc; }
  CK (cudaGetLastError ());
  h->timed = h->time_frames;
  h->is_empty = false;                                             // hpp:101
  return B200TSDF_OK;
}

// layout of an organized cloud as the integrate entry points accept it (ADVICE r1: the same checks everywhere)
static int check_cloud_layout (b200tsdf* h, size_t stride, int xyz_off, int rgba_off, int width, int height)
{
  if (width <= 0 || height <= 0) return h->fail (B200TSDF_EINVAL, "bad cloud shape");
  if (stride < 12 || (stride & 3) || xyz_off < 0 || (xyz_off & 3) || (size_t) xyz_off + 12 > stride
      || (rgba_off >= 0 && ((size_t) rgba_off + 4 > stride || (rgba_off & 3))))
    return h->fail (B200TSDF_EINVAL, "bad point layout (need 4-byte aligned xyz_off + 12 <= stride and rgba_off + 4 <= stride)");
  if ((double) width * (double) height * (double) stride >= 2147483648.0) return h->fail (B200TSDF_EINVAL, "organized cloud of 2 GiB or more");
  if (width != h->cfg.image_width || height != h->cfg.image_height)
    return h->fail (B200TSDF_EINVAL, "organized cloud size differs from setImageSize() (the reference indexes cloud(u,v) with the image size, cpp:611-617)");
  return B200TSDF_OK;
}

int b200tsdf_integrate_device (b200tsdf_t* h, const void* d_points, size_t stride, int xyz_off, int rgba_off,
                               int width, int height, const double* pose)
{
  if (!h || !d_points || !pose) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "integrateCloud before reset()");
  if (int rc = check_cloud_layout (h, stride, xyz_off, rgba_off, width, height)) return rc;
  cudaSetDevice (h->device);
  return integrate_on_device (h, (const unsigned char*) d_points, stride, xyz_off, rgba_off, width, height, pose);
}

// a batch of frames resident in device memory: one upload of the frame records, one graph launch
// The two halves of a batch: (1) the frame records are written into a host staging segment and uploaded on `rec_stream`
// into one half of the device slots; (2) the captured launches of that half are replayed on the compute stream.  The row
// path (multigpu.cuh) uploads the records on its copy stream AHEAD of the frames themselves — a record upload issued on
// the compute stream would queue behind every frame copy already submitted to the one host-to-device copy engine.
static int batch_records (b200tsdf* h, int m, const void* const* d_points, size_t stride, int xyz_off, int rgba_off, int width, int height,
                          const double* poses_c2w, cudaStream_t rec_stream)
{
  constexpr int HALF = FRAME_RING / 2;
  const int a = h->bring_half, sg = h->bring_seg;
  if (h->bring_used[sg]) CK (cudaEventSynchronize (h->ev_bring[sg]));    // the copy that last read this staging segment has run
  FrameRec* recs = h->h_bring + (size_t) sg * HALF;
  for (int i = 0; i < m; ++i)
  {
    if (!d_points[i]) return h->fail (B200TSDF_EINVAL, "null cloud in batch");
    fill_rec (h, recs[i], (const unsigned char*) d_points[i], stride, xyz_off, rgba_off, width, height, poses_c2w + 16 * (size_t) i);
  }
  // the device half is rewritten only after the launches that last read it (other stream: wait for their event)
  if (rec_stream != h->stream && h->half_used[a]) CK (cudaStreamWaitEvent (rec_stream, h->ev_half_done[a], 0));
  CK (cudaMemcpyAsync (h->d_bring + a * HALF, recs, (size_t) m * sizeof (FrameRec), cudaMemcpyHostToDevice, rec_stream));
  CK (cudaEventRecord (h->ev_bring[sg], rec_stream));      // the staging segment is free again once this copy has run
  h->bring_used[sg] = true; h->bring_seg = (sg + 1) % BATCH_SEGS;
  h->batch_recs = recs;
  return B200TSDF_OK;
}
static int batch_launch (b200tsdf* h, int m)
{
  constexpr int HALF = FRAME_RING / 2;
  cudaStream_t s = h->stream;
  const int a = h->bring_half;
  cudaGraphExec_t& exec = h->batch_exec[a][m];          // (nothing of a frame is baked into the launches: they read the record)
  if (!exec)
  {
    const long long l0 = h->launches, f0 = h->prof_frames;
    cudaGraph_t g = nullptr;
    CK (cudaStreamBeginCapture (s, cudaStreamCaptureModeThreadLocal));
    int rc = B200TSDF_OK;
    for (int i = 0; i < m && rc == B200TSDF_OK; ++i) rc = launch_frame (h, s, h->batch_recs[i], h->d_bring + a * HALF + i, false);
    cudaError_t ce = cudaStreamEndCapture (s, &g);
    h->launches_per_frame = (int) ((h->launches - l0) / std::max (1, m));
    h->launches = l0; h->prof_frames = f0;
    if (rc) { if (g) cudaGraphDestroy (g); return rc; }
    if (ce != cudaSuccess) return h->fail (B200TSDF_ECUDA, std::string ("graph capture: ") + cudaGetErrorString (ce));
    ce = cudaGraphInstantiate (&exec, g, 0);
    cudaGraphDestroy (g);
    if (ce != cudaSuccess) { exec = nullptr; return h->fail (B200TSDF_ECUDA, std::string ("graph instantiate: ") + cudaGetErrorString (ce)); }
  }
  CK (cudaGraphLaunch (exec, s));
  CK (cudaEventRecord (h->ev_half_done[a], s));
  h->half_used[a] = true;
  note_device_err (h, s);
  h->bring_half ^= 1;
  h->launches += (long long) m * h->launches_per_frame; h->graph_launches++;
  h->prof_frames += m;
  h->timed = false;
  h->is_empty = false;
  return B200TSDF_OK;
}

int b200tsdf_integrate_batch_device (b200tsdf_t* h, int n, const void* const* d_points, size_t stride, int xyz_off, int rgba_off,
                                     int width, int height, const double* poses_c2w)
{
  if (!h || n < 0 || (n && (!d_points || !poses_c2w))) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "integrateCloud before reset()");
  if (int rc = check_cloud_layout (h, stride, xyz_off, rgba_off, width, height)) return rc;
  cudaSetDevice (h->device);
  if (int rc = pending_device_err (h)) return rc;
  constexpr int HALF = FRAME_RING / 2;
  for (int done = 0; done < n;)
  {
    const int m = std::min (HALF, n - done);
    if (!h->replayable)
    {
      // the general depth-first kernel takes the frame by value: frame by frame
      for (int i = 0; i < m; ++i)
        if (int rc = integrate_on_device (h, (const unsigned char*) d_points[done + i], stride, xyz_off, rgba_off, width, height, poses_c2w + 16 * (size_t) (done + i))) return rc;
      done += m;
      continue;
    }
    if (int rc = batch_records (h, m, d_points + done, stride, xyz_off, rgba_off, width, height, poses_c2w + 16 * (size_t) done, h->stream)) return rc;
    if (int rc = batch_launch (h, m)) return rc;
    done += m;
  }
  CK (cudaGetLastError ());
  return B200TSDF_OK;
}

// the host threads that pack uploaded points to 16-byte pixels (host_pack.h), created on first use
static void ensure_pack_pool (b200tsdf* h, int nr)
{
  if (h->pack_pool) return;
  int t = h->pack_threads;
  if (t <= 0) { const int hw = (int) std::thread::hardware_concurrency (); t = std::max (1, std::min (16, hw / (2 * nr))); }
  // B200TSDF_PACK_CPUS: "local" = the cores next to this GPU's PCIe root (sysfs local_cpulist), or an explicit cpulist
  std::string cpus;
  if (const char* e = std::getenv ("B200TSDF_PACK_CPUS"))
  {
    cpus = e;
    if (cpus == "local")
    {
      cpus.clear ();
      char bus[32] = {};
      if (cudaDeviceGetPCIBusId (bus, sizeof (bus), h->device) == cudaSuccess)
      {
        for (char* c = bus; *c; ++c) *c = (char) std::tolower ((unsigned char) *c);
        if (FILE* f = std::fopen ((std::string ("/sys/bus/pci/devices/") + bus + "/local_cpulist").c_str (), "r"))
        {
          char line[512] = {};
          if (std::fgets (line, sizeof (line), f)) { cpus = line; while (!cpus.empty () && (cpus.back () == '\n' || cpus.back () == ' ')) cpus.pop_back (); }
          std::fclose (f);
        }
      }
    }
  }
  // (no exception may cross the C ABI: if the threads cannot be created the caller's thread packs alone)
  try { h->pack_pool = new b2host::PackPool (t, cpus); }
  catch (...) { h->pack_pool = new b2host::PackPool (1); }
}

// is the upload of `stride`-byte points packed on the host?  (-1: by rank count, see b200tsdf_integrate_batch_rows)
static bool host_pack_wanted (const b200tsdf* h, size_t stride, int nr) { return (h->host_pack < 0 ? nr <= 1 : h->host_pack != 0) && stride > 16; }

static int integrate_host (b200tsdf* h, const void* points, size_t stride, int xyz_off, int rgba_off,
                           int width, int height, const double* pose, bool wait_copy)
{
  if (!h || !points || !pose) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "integrateCloud before reset()");
  if (int rc = check_cloud_layout (h, stride, xyz_off, rgba_off, width, height)) return rc;
  cudaSetDevice (h->device);
  // points wider than 16 bytes are packed to {x, y, z, bgra} by the host threads into pinned staging (also the way out of a
  // pageable pcl cloud at full PCIe speed); the caller's buffer is free again when this call returns
  const bool hpack = host_pack_wanted (h, stride, h->comm ? h->comm_size : 1);
  const size_t npts = (size_t) width * height;
  const size_t bytes = hpack ? npts * 16 : npts * stride;
  if (bytes > h->frame_cap || (hpack && !h->h_fpack[0].p))
  {
    CK (cudaStreamSynchronize (h->stream)); CK (cudaStreamSynchronize (h->copy_stream));
    const size_t cap = std::max (bytes, h->frame_cap);
    for (int i = 0; i < 2; ++i)
    {
      cudaFree (h->d_frame[i]); h->d_frame[i] = nullptr; CK (cudaMalloc (&h->d_frame[i], cap));
      h->h_fpack[i].release ();
      if (hpack && h->h_fpack[i].alloc (cap))
      {
        // no pinned staging to be had on this system: upload the points as they are from now on
        h->host_pack = 0;
        for (int k = 0; k < 2; ++k) h->h_fpack[k].release ();
        h->frame_cap = 0;                                  // (d_frame[] is re-sized by the unpacked path)
        return integrate_host (h, points, stride, xyz_off, rgba_off, width, height, pose, wait_copy);
      }
    }
    h->frame_cap = cap;
    h->frame_no = 0;
  }
  // double-buffered upload on the copy stream: frame i+1 crosses PCIe while frame i is fused
  int b = (int) (h->frame_no & 1);
  if (h->frame_no >= 2)
  {
    CK (cudaEventSynchronize (h->ev_copied[b]));           // the upload of frame i-2 has left the caller's buffer / the staging (the documented contract)
    CK (cudaStreamWaitEvent (h->copy_stream, h->ev_consumed[b], 0));
  }
  const void* src = points;
  size_t f_stride = stride; int f_xyz = xyz_off, f_rgba = rgba_off;
  if (hpack)
  {
    ensure_pack_pool (h, h->comm ? h->comm_size : 1);
    const int nb = (int) std::max<size_t> (1, std::min<size_t> (4 * (size_t) h->pack_pool->threads (), npts / 4096));
    const int pack_rgba = h->p.color ? rgba_off : -1;
    unsigned char* stage = h->h_fpack[b].p;
    std::function<void (int)> job = [&] (int j)
    {
      const size_t p0 = npts * (size_t) j / nb, p1 = npts * (size_t) (j + 1) / nb;
      b2host::pack_points16 (static_cast<const unsigned char*> (points) + p0 * stride, stride, xyz_off, pack_rgba, p1 - p0, stage + p0 * 16);
    };
    h->pack_pool->run (nb, job);
    src = stage; f_stride = 16; f_xyz = 0; f_rgba = (h->p.color && rgba_off >= 0) ? 12 : -1;
  }
  CK (cudaMemcpyAsync (h->d_frame[b], src, bytes, cudaMemcpyHostToDevice, h->copy_stream));
  h->h2d_bytes += (long long) bytes;
  CK (cudaEventRecord (h->ev_copied[b], h->copy_stream));
  CK (cudaStreamWaitEvent (h->stream, h->ev_copied[b], 0));
  int rc = integrate_on_device (h, h->d_frame[b], f_stride, f_xyz, f_rgba, width, height, pose);
  if (rc) return rc;
  CK (cudaEventRecord (h->ev_consumed[b], h->stream));
  h->frame_no++;
  if (wait_copy && !hpack) CK (cudaEventSynchronize (h->ev_copied[b]));       // the caller may reuse its buffer now
  return B200TSDF_OK;
}

int b200tsdf_integrate (b200tsdf_t* h, const void* points, size_t stride, int xyz_off, int rgba_off,
                        int width, int height, const double* pose)
{ return integrate_host (h, points, stride, xyz_off, rgba_off, width, height, pose, true); }

int b200tsdf_integrate_async (b200tsdf_t* h, const void* points, size_t stride, int xyz_off, int rgba_off,
                              int width, int height, const double* pose)
{ return integrate_host (h, points, stride, xyz_off, rgba_off, width, height, pose, false); }

// ---- unorganised clouds (integrate.cpp:548-635) ------------------------------------------------
namespace {

// uploads the points, z-buffers them and writes the organized cloud to d_out (device).  Scratch layout:
// [points n*stride | zkey npix*8 | filled counter 8 | organized npix*out_stride (when d_out == nullptr)]
int organize_on_device (b200tsdf* h, const void* points, size_t n, size_t stride, int xyz_off, int rgba_off,
                        const b200tsdf_organize_opts* opts, size_t out_stride, int out_rgba_off,
                        unsigned char** d_out, unsigned long long** d_filled)
{
  if (!h || (!points && n) || !opts) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "organize before reset() (the image size and intrinsics are read at reset)");
  if (stride < 12 || xyz_off < 0 || (size_t) xyz_off + 12 > stride || (rgba_off >= 0 && (size_t) rgba_off + 4 > stride))
    return h->fail (B200TSDF_EINVAL, "bad point layout");
  if (out_stride < 16 || (out_stride & 3) || (out_rgba_off >= 0 && ((size_t) out_rgba_off + 4 > out_stride || out_rgba_off < 12)))
    return h->fail (B200TSDF_EINVAL, "bad organized layout");
  if (n >= (1ull << 32)) return h->fail (B200TSDF_EINVAL, "more than 2^32-1 points in one cloud");
  cudaSetDevice (h->device);
  OrgParams o{};
  // the program keeps its intrinsics as float globals (integrate.cpp:63-68, 349-361)
  o.fx = (float) h->cfg.fx; o.fy = (float) h->cfg.fy; o.cx = (float) h->cfg.cx; o.cy = (float) h->cfg.cy;
  o.width = h->cfg.image_width; o.height = h->cfg.image_height;
  o.cloud_units = opts->cloud_units; o.zero_nans = opts->zero_nans; o.has_tf = opts->world_to_camera != nullptr;
  if (o.has_tf) for (int i = 0; i < 12; ++i) o.tf[i] = opts->world_to_camera[i];
  size_t npix = (size_t) o.width * o.height;
  size_t off_key = (n * stride + 255) & ~(size_t) 255, off_cnt = off_key + npix * 8, off_out = off_cnt + 256;
  { int rc = h->scratch (off_out + npix * out_stride + 64); if (rc) return rc; }
  unsigned char* d_pts = h->d_scratch;
  unsigned long long* zkey = (unsigned long long*) (h->d_scratch + off_key);
  *d_filled = (unsigned long long*) (h->d_scratch + off_cnt);
  *d_out = h->d_scratch + off_out;
  cudaStream_t s = h->stream;
  if (n) { CK (cudaMemcpyAsync (d_pts, points, n * stride, cudaMemcpyHostToDevice, s)); h->h2d_bytes += (long long) (n * stride); }
  k_org_clear<<<(unsigned) ((npix + 255) / 256), 256, 0, s>>> (zkey, (int) npix, *d_filled);
  if (n)
  {
    size_t blocks = std::min<size_t> ((n + 255) / 256, (size_t) h->sm_count * 16);
    k_org_zmin<<<(unsigned) blocks, 256, 0, s>>> (o, d_pts, n, stride, xyz_off, zkey);
  }
  k_org_gather<<<(unsigned) ((npix + 255) / 256), 256, 0, s>>> (o, d_pts, stride, xyz_off, rgba_off, zkey, *d_out, out_stride, out_rgba_off, *d_filled);
  h->launches += n ? 3 : 2;
  CK (cudaGetLastError ());
  return B200TSDF_OK;
}

} // namespace

int b200tsdf_organize (b200tsdf_t* h, const void* points, size_t n, size_t stride, int xyz_off, int rgba_off,
                       const b200tsdf_organize_opts* opts, void* out, size_t out_stride, int out_rgba_off, int64_t* n_filled)
{
  if (!h || !out) return B200TSDF_EINVAL;
  unsigned char* d_out = nullptr; unsigned long long* d_filled = nullptr;
  int rc = organize_on_device (h, points, n, stride, xyz_off, rgba_off, opts, out_stride, out_rgba_off, &d_out, &d_filled);
  if (rc) return rc;
  size_t bytes = (size_t) h->cfg.image_width * h->cfg.image_height * out_stride;
  unsigned long long filled = 0;
  // bytes of a pixel that the layout does not name (padding) are zero in the result
  CK (cudaMemcpyAsync (out, d_out, bytes, cudaMemcpyDeviceToHost, h->stream));
  CK (cudaMemcpyAsync (&filled, d_filled, 8, cudaMemcpyDeviceToHost, h->stream));
  CK (cudaStreamSynchronize (h->stream));
  h->d2h_bytes += (long long) bytes + 8;
  if (n_filled) *n_filled = (int64_t) filled;
  return B200TSDF_OK;
}

int b200tsdf_integrate_unorganized (b200tsdf_t* h, const void* points, size_t n, size_t stride, int xyz_off, int rgba_off,
                                    const b200tsdf_organize_opts* opts, const double* pose)
{
  if (!h || !pose) return B200TSDF_EINVAL;
  unsigned char* d_out = nullptr; unsigned long long* d_filled = nullptr;
  // organized pixels are 16 bytes in HBM: x, y, z, then the colour bytes b,g,r,a
  int rc = organize_on_device (h, points, n, stride, xyz_off, rgba_off, opts, 16, 12, &d_out, &d_filled);
  if (rc) return rc;
  return integrate_on_device (h, d_out, 16, 0, 12, h->cfg.image_width, h->cfg.image_height, pose);
}

int b200tsdf_sync (b200tsdf_t* h)
{
  if (!h) return B200TSDF_EINVAL;
  cudaSetDevice (h->device);
  CK (cudaStreamSynchronize (h->copy_stream));
  CK (cudaStreamSynchronize (h->gather_stream));
  return check_device_err (h);
}

int b200tsdf_get_stats (b200tsdf_t* h, b200tsdf_stats* s)
{
  if (!h || !s) return B200TSDF_EINVAL;
  std::memset (s, 0, sizeof (*s));
  if (!h->has_volume) return B200TSDF_OK;
  cudaSetDevice (h->device);
  int rc = b200tsdf_sync (h);
  if (rc) return rc;
  unsigned long long st[2 * ST_N]; int cnt[16];
  CK (cudaMemcpy (st, h->d_stats, sizeof (st), cudaMemcpyDeviceToHost));
  CK (cudaMemcpy (cnt, h->d_count + 16 * h->count_set, sizeof (cnt), cudaMemcpyDeviceToHost));
  h->d2h_bytes += (long long) (sizeof (st) + sizeof (cnt));
  s->n_updates = (int64_t) (st[ST_UPDATES] - st[ST_N + ST_UPDATES]);
  s->n_node_visits = (int64_t) (st[ST_VISITS] - st[ST_N + ST_VISITS]);
  s->n_block_visits = (int64_t) (st[ST_BLOCKS] - st[ST_N + ST_BLOCKS]);
  s->reserved = (int32_t) (st[3] - st[ST_N + 3]);          // diagnostics: slow folds in the last frame
  s->n_bail = cnt[10]; s->n_slow_visits = (int64_t) (st[4] - st[ST_N + 4]);
  s->n_culled_cells = cnt[0];
  s->pool_capacity = (int64_t) h->pool;
  s->coarse_level = h->p.C; s->finest_level = h->p.L; s->tiers = h->p.T;
  // allocated bricks (no allocation, no list: this call sits in measured loops)
  int* d_n = h->d_count + 40;
  CK (cudaMemsetAsync (d_n, 0, sizeof (int), h->stream));
  k_count_bricks<<<(unsigned) ((h->pool + 255) / 256), 256, 0, h->stream>>> (h->p, d_n);
  int nb = 0;
  CK (cudaMemcpyAsync (&nb, d_n, sizeof (int), cudaMemcpyDeviceToHost, h->stream));
  CK (cudaStreamSynchronize (h->stream));
  s->n_bricks = nb;
  if (h->timed)
  {
    float ms = 0.f;
    if (cudaEventElapsedTime (&ms, h->ev_t0, h->ev_t1) == cudaSuccess) s->ms_last_integrate = ms;
    int last = (h->kring_head + KRING - 1) % KRING;
    if (h->kring_pending > 0 && cudaEventElapsedTime (&ms, h->kring[last][0], h->kring[last][1]) == cudaSuccess) s->ms_last_kernel = ms;
  }
  return B200TSDF_OK;
}

// ---- point queries (tsdf_volume_octree.cpp:655-794) -------------------------------------------------
int b200tsdf_query (b200tsdf_t* h, const float* xyz, int n, int what, int mode,
                    float* val, float* grad, float* hess, uint8_t* ok)
{
  if (!h || !xyz || !ok || n < 0) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "query before reset()");
  if (((what & 1) && !val) || ((what & 2) && !grad) || ((what & 4) && !hess)) return h->fail (B200TSDF_EINVAL, "missing output buffer");
  if (n == 0) return B200TSDF_OK;
  cudaSetDevice (h->device);
  // one scratch block: xyz (12n) | val (4n) | grad (12n) | hess (36n) | ok (n)
  { int rc = h->scratch ((size_t) n * 65 + 64); if (rc) return rc; }
  float* d_xyz = (float*) h->d_scratch;
  float* d_val = d_xyz + (size_t) 3 * n;
  float* d_grad = d_val + n;
  float* d_hess = d_grad + (size_t) 3 * n;
  unsigned char* d_ok = (unsigned char*) (d_hess + (size_t) 9 * n);
  cudaStream_t s = h->stream;
  CK (cudaMemcpyAsync (d_xyz, xyz, (size_t) n * 12, cudaMemcpyHostToDevice, s));
  k_query<<<(n + 127) / 128, 128, 0, s>>> (h->p, d_xyz, n, what, mode, d_val, d_grad, d_hess, d_ok);
  CK (cudaMemcpyAsync (ok, d_ok, (size_t) n, cudaMemcpyDeviceToHost, s));
  if (what & 1) CK (cudaMemcpyAsync (val, d_val, (size_t) n * 4, cudaMemcpyDeviceToHost, s));
  if (what & 2) CK (cudaMemcpyAsync (grad, d_grad, (size_t) n * 12, cudaMemcpyDeviceToHost, s));
  if (what & 4) CK (cudaMemcpyAsync (hess, d_hess, (size_t) n * 36, cudaMemcpyDeviceToHost, s));
  note_device_err (h, s);
  CK (cudaStreamSynchronize (s));
  return pending_device_err (h);
}

// ---- getTSDFValue / interpolateTrilinearly (tsdf_volume_octree.cpp:454-541) ---------------------------------
int b200tsdf_interpolate (b200tsdf_t* h, const float* xyz, int n, float* val, uint8_t* valid_in_out)
{
  if (!h || !xyz || !val || !valid_in_out || n < 0) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "getTSDFValue before reset()");
  if (n == 0) return B200TSDF_OK;
  cudaSetDevice (h->device);
  { int rc = h->scratch ((size_t) n * 17 + 64); if (rc) return rc; }
  float* d_xyz = (float*) h->d_scratch;
  float* d_val = d_xyz + (size_t) 3 * n;
  unsigned char* d_ok = (unsigned char*) (d_val + n);
  cudaStream_t s = h->stream;
  CK (cudaMemcpyAsync (d_xyz, xyz, (size_t) n * 12, cudaMemcpyHostToDevice, s));
  CK (cudaMemcpyAsync (d_ok, valid_in_out, (size_t) n, cudaMemcpyHostToDevice, s));
  k_interpolate<<<(n + 127) / 128, 128, 0, s>>> (h->p, d_xyz, n, d_val, d_ok);
  CK (cudaMemcpyAsync (val, d_val, (size_t) n * 4, cudaMemcpyDeviceToHost, s));
  CK (cudaMemcpyAsync (valid_in_out, d_ok, (size_t) n, cudaMemcpyDeviceToHost, s));
  note_device_err (h, s);
  CK (cudaStreamSynchronize (s));
  return pending_device_err (h);
}

// ---- renderView / renderColoredView (tsdf_volume_octree.cpp:278-450) ----------------------------------
int b200tsdf_render (b200tsdf_t* h, const double* pose, int downsample, void* out, size_t stride,
                     int xyz_off, int normal_off, uint8_t* rgb_out)
{
  if (!h || !pose || !out || downsample < 1) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "renderView before reset()");
  if (stride < 12 || xyz_off < 0 || normal_off < 0 || (size_t) xyz_off + 12 > stride || (size_t) normal_off + 12 > stride)
    return h->fail (B200TSDF_EINVAL, "bad output point layout (need xyz_off + 12 <= stride and normal_off + 12 <= stride)");
  cudaSetDevice (h->device);
  const Params& p = h->p;
  RenderParams r;
  if (p.width / downsample <= 0 || p.height / downsample <= 0) return h->fail (B200TSDF_EINVAL, "downsample too large");
  make_render_params (h->cfg, p, pose, downsample, r);
  size_t npix = (size_t) r.width * r.height;
  { int rc = h->scratch (npix * 6 * sizeof (float) + npix * 3 + 64); if (rc) return rc; }
  float* d_out = (float*) h->d_scratch;
  unsigned char* d_rgb = rgb_out ? h->d_scratch + npix * 6 * sizeof (float) : nullptr;
  cudaStream_t s = h->stream;
  dim3 grid ((r.width + 7) / 8, (r.height + 7) / 8);
  k_render<<<grid, 64, 0, s>>> (p, r, d_out, d_rgb);
  std::vector<float> tmp (npix * 6);
  CK (cudaMemcpyAsync (tmp.data (), d_out, npix * 6 * sizeof (float), cudaMemcpyDeviceToHost, s));
  if (rgb_out) CK (cudaMemcpyAsync (rgb_out, d_rgb, npix * 3, cudaMemcpyDeviceToHost, s));
  note_device_err (h, s);
  CK (cudaStreamSynchronize (s));
  if (int rc = pending_device_err (h)) return rc;
  unsigned char* base = (unsigned char*) out;
  for (size_t i = 0; i < npix; ++i)
  {
    std::memcpy (base + i * stride + xyz_off, &tmp[6 * i], 12);
    std::memcpy (base + i * stride + normal_off, &tmp[6 * i + 3], 12);
  }
  return B200TSDF_OK;
}

// ---- marching cubes (marching_cubes_tsdf_octree.cpp:108-236) --------------------------------------------
int b200tsdf_mesh (b200tsdf_t* h, float w_min, int color_mode, float** verts, uint8_t** rgb, size_t* nverts)
{
  if (!h || !verts || !nverts) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "reconstruct before reset()");
  cudaSetDevice (h->device);
  const Params& p = h->p;
  McParams mc;
  make_mc_params (h->cfg, p, w_min, color_mode, mc);
  cudaStream_t s = h->stream;
  int* d_list = nullptr; int* d_n = h->d_count + 40;
  unsigned long long* d_total = h->d_stats + ST_SCRATCH;
  CK (cudaMalloc (&d_list, h->pool * sizeof (int)));
  CK (cudaMemsetAsync (d_n, 0, sizeof (int), s));
  CK (cudaMemsetAsync (d_total, 0, sizeof (unsigned long long), s));
  k_list_bricks<<<(unsigned) ((h->pool + 255) / 256), 256, 0, s>>> (p, d_list, d_n);
  int nb = 0;
  CK (cudaMemcpyAsync (&nb, d_n, sizeof (int), cudaMemcpyDeviceToHost, s));
  CK (cudaStreamSynchronize (s));
  int root_n = (int) h->root_n;
  if (nb) k_mesh_bricks<false><<<(nb * 32 + 127) / 128, 128, 0, s>>> (p, mc, d_list, nb, d_total, nullptr, nullptr, nullptr);
  k_mesh_roots<false><<<(root_n + 127) / 128, 128, 0, s>>> (p, mc, d_total, nullptr, nullptr, nullptr);
  unsigned long long ntri = 0;
  CK (cudaMemcpyAsync (&ntri, d_total, sizeof (ntri), cudaMemcpyDeviceToHost, s));
  CK (cudaStreamSynchronize (s));
  std::free (h->mesh_v); std::free (h->mesh_c); h->mesh_v = nullptr; h->mesh_c = nullptr;
  *verts = nullptr; if (rgb) *rgb = nullptr; *nverts = (size_t) ntri * 3;
  if (ntri)
  {
    // emission order depends on the hash layout and on atomics; the triangles are then sorted into the reference's
    // own order (depth first over the octree, mc_order_key) so that the soup is reproducible and comparable as is
    float *d_v = nullptr, *d_v2 = nullptr; unsigned char *d_c = nullptr, *d_c2 = nullptr; unsigned long long* d_k = nullptr;
    CK (cudaMalloc (&d_v, ntri * 9 * sizeof (float))); CK (cudaMalloc (&d_v2, ntri * 9 * sizeof (float)));
    CK (cudaMalloc (&d_k, ntri * sizeof (unsigned long long)));
    if (color_mode) { CK (cudaMalloc (&d_c, ntri * 9)); CK (cudaMalloc (&d_c2, ntri * 9)); }
    CK (cudaMemsetAsync (d_total, 0, sizeof (unsigned long long), s));
    if (nb) k_mesh_bricks<true><<<(nb * 32 + 127) / 128, 128, 0, s>>> (p, mc, d_list, nb, d_total, d_v, d_c, d_k);
    k_mesh_roots<true><<<(root_n + 127) / 128, 128, 0, s>>> (p, mc, d_total, d_v, d_c, d_k);
    if (b2_sort_triangles (s, (size_t) ntri, 3 * p.L + 3, d_k, d_v, d_c, d_v2, d_c2) != 0)
    { cudaFree (d_v); cudaFree (d_v2); cudaFree (d_c); cudaFree (d_c2); cudaFree (d_k); cudaFree (d_list); return h->fail (B200TSDF_ECUDA, "triangle sort failed"); }
    h->mesh_v = (float*) std::malloc (ntri * 9 * sizeof (float));
    CK (cudaMemcpyAsync (h->mesh_v, d_v2, ntri * 9 * sizeof (float), cudaMemcpyDeviceToHost, s));
    if (color_mode) { h->mesh_c = (unsigned char*) std::malloc (ntri * 9); CK (cudaMemcpyAsync (h->mesh_c, d_c2, ntri * 9, cudaMemcpyDeviceToHost, s)); }
    CK (cudaStreamSynchronize (s));
    cudaFree (d_v); cudaFree (d_v2); cudaFree (d_c); cudaFree (d_c2); cudaFree (d_k);
    *verts = h->mesh_v; if (rgb) *rgb = h->mesh_c;
  }
  cudaFree (d_list);
  return check_device_err (h);
}

void b200tsdf_free (void* p) { (void) p; /* mesh buffers are owned by the handle */ }

} // extern "C"

// ---- getVoxelCenters / getOccupiedVoxelIndices (tsdf_volume_octree.cpp:576-609) ---------------------------------
// Octree::getLeaves on the device: a count pass and a key pass over the stored levels (one warp per brick, one thread per
// root-array node), a radix sort of the keys into the order of the reference's depth-first walk, a decode pass into
// centres or voxel indices, one copy to the host.  The node payload never leaves HBM: 12 bytes per returned node cross PCIe.
namespace {
struct DevMem
{
  void* p = nullptr;
  ~DevMem () { cudaFree (p); }
  template <typename T> T* as () const { return static_cast<T*> (p); }
};

// *out: host buffer of 3 values per node (float centres, or int32 indices when occupied), malloc'ed; *n: node count
int leaves_on_device (b200tsdf* h, int nlevels, bool occupied, void** out, size_t* n)
{
  const char* what = occupied ? "getOccupiedVoxelIndices" : "getVoxelCenters";
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, std::string (what) + " before reset()");
  if (h->p.shard_count > 1)
    return h->fail (B200TSDF_EINVAL, std::string (what) + " on a shard: the coarse cells it does not own are unsplit leaves here; "
                    "gather the shards into one volume first (b200tsdf_gather_volume or b200tsdf_import_shard)");
  cudaSetDevice (h->device);
  if (int rc = pending_device_err (h)) return rc;
  const Params& p = h->p;
  cudaStream_t s = h->stream;
  const int key_bits = 3 * p.L + LEAF_LEVEL_BITS;
  size_t count = 0;
  DevMem keys, sorted;
  if (!occupied && nlevels >= 0 && nlevels <= p.C)
  {
    if (3 * nlevels >= 31) return h->fail (B200TSDF_ENOMEM, std::string (what) + ": more than 2^31 nodes requested");
    count = (size_t) 1 << (3 * nlevels);
    CK (cudaMalloc (&sorted.p, count * sizeof (unsigned long long)));
    k_leaf_level<<<(unsigned) ((count + 255) / 256), 256, 0, s>>> (p.L, nlevels, count, sorted.as<unsigned long long> ());
  }
  else
  {
    if (occupied) nlevels = -1;                              // octree_->getLeaves (leaves): no level limit
    DevMem list;
    int* d_n = h->d_count + 40;
    unsigned long long* d_total = h->d_stats + ST_SCRATCH;
    CK (cudaMalloc (&list.p, h->pool * sizeof (int)));
    CK (cudaMemsetAsync (d_n, 0, sizeof (int), s));
    CK (cudaMemsetAsync (d_total, 0, sizeof (unsigned long long), s));
    k_list_bricks<<<(unsigned) ((h->pool + 255) / 256), 256, 0, s>>> (p, list.as<int> (), d_n);
    int nb = 0;
    CK (cudaMemcpyAsync (&nb, d_n, sizeof (int), cudaMemcpyDeviceToHost, s));
    CK (cudaStreamSynchronize (s));
    const unsigned brick_blocks = (unsigned) (((size_t) nb * 32 + 127) / 128), root_blocks = (unsigned) ((h->root_n + 127) / 128);
    if (nb) k_leaf_bricks<false><<<brick_blocks, 128, 0, s>>> (p, nlevels, occupied, list.as<int> (), nb, d_total, nullptr);
    k_leaf_roots<false><<<root_blocks, 128, 0, s>>> (p, nlevels, occupied, d_total, nullptr);
    unsigned long long total = 0;
    CK (cudaMemcpyAsync (&total, d_total, sizeof (total), cudaMemcpyDeviceToHost, s));
    CK (cudaStreamSynchronize (s));
    if (total >= ((unsigned long long) 1 << 31)) return h->fail (B200TSDF_ENOMEM, std::string (what) + ": more than 2^31 nodes");
    count = (size_t) total;
    if (count)
    {
      CK (cudaMalloc (&keys.p, count * sizeof (unsigned long long)));
      CK (cudaMalloc (&sorted.p, count * sizeof (unsigned long long)));
      CK (cudaMemsetAsync (d_total, 0, sizeof (unsigned long long), s));
      if (nb) k_leaf_bricks<true><<<brick_blocks, 128, 0, s>>> (p, nlevels, occupied, list.as<int> (), nb, d_total, keys.as<unsigned long long> ());
      k_leaf_roots<true><<<root_blocks, 128, 0, s>>> (p, nlevels, occupied, d_total, keys.as<unsigned long long> ());
      CK (cudaGetLastError ());
      if (int e = b2_sort_keys (s, count, key_bits, keys.as<unsigned long long> (), sorted.as<unsigned long long> ()))
        return h->fail (B200TSDF_ECUDA, std::string (what) + ": key sort failed: " + cudaGetErrorString ((cudaError_t) e));
    }
  }
  CK (cudaGetLastError ());
  *out = nullptr; *n = count;
  if (!count) return check_device_err (h);
  DevMem vals;
  CK (cudaMalloc (&vals.p, count * 12));
  k_leaf_decode<<<(unsigned) ((count + 255) / 256), 256, 0, s>>> (p, sorted.as<unsigned long long> (), count,
                                                                  occupied ? nullptr : vals.as<float> (), occupied ? vals.as<int> () : nullptr);
  CK (cudaGetLastError ());
  void* host = std::malloc (count * 12);
  if (!host) return h->fail (B200TSDF_ENOMEM, std::string (what) + ": host allocation failed");
  cudaError_t e = cudaMemcpyAsync (host, vals.p, count * 12, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize (s);
  if (e != cudaSuccess) { std::free (host); return h->fail (B200TSDF_ECUDA, std::string (what) + ": " + cudaGetErrorString (e)); }
  h->d2h_bytes += (long long) (count * 12);
  *out = host;
  return check_device_err (h);
}
} // namespace

extern "C" {

int b200tsdf_voxel_centers (b200tsdf_t* h, int nlevels, float** xyz, size_t* n)
{
  if (!h || !xyz || !n) return B200TSDF_EINVAL;
  void* out = nullptr; size_t cnt = 0;
  int rc = leaves_on_device (h, nlevels, false, &out, &cnt);
  if (rc) { std::free (out); return rc; }
  std::free (h->leaf_xyz);
  h->leaf_xyz = static_cast<float*> (out);
  *xyz = h->leaf_xyz; *n = cnt;
  return B200TSDF_OK;
}

int b200tsdf_occupied_voxel_indices (b200tsdf_t* h, int32_t** ijk, size_t* n)
{
  if (!h || !ijk || !n) return B200TSDF_EINVAL;
  void* out = nullptr; size_t cnt = 0;
  int rc = leaves_on_device (h, -1, true, &out, &cnt);
  if (rc) { std::free (out); return rc; }
  std::free (h->leaf_ijk);
  h->leaf_ijk = static_cast<int32_t*> (out);
  *ijk = h->leaf_ijk; *n = cnt;
  return B200TSDF_OK;
}

int b200tsdf_is_empty (const b200tsdf_t* h, int32_t* out)
{
  if (!h || !out) return B200TSDF_EINVAL;
  if (!h->has_volume) return B200TSDF_ESTATE;
  *out = h->is_empty ? 1 : 0;
  return B200TSDF_OK;
}

int b200tsdf_voxel_center (const b200tsdf_t* h, int64_t x, int64_t y, int64_t z, float* o)
{
  if (!h || !o || !h->has_volume) return B200TSDF_EINVAL;
  o[0] = voxel_center1 (h->p, x); o[1] = voxel_center1 (h->p, y); o[2] = voxel_center1 (h->p, z);
  return B200TSDF_OK;
}

int b200tsdf_voxel_index (const b200tsdf_t* h, float x, float y, float z, int32_t* o, int32_t* inside)
{
  if (!h || !o || !h->has_volume) return B200TSDF_EINVAL;
  int xi, yi, zi;
  bool in = voxel_index (h->p, x, y, z, xi, yi, zi);
  o[0] = xi; o[1] = yi; o[2] = zi;
  if (inside) *inside = in;
  return B200TSDF_OK;
}

int b200tsdf_frustum_cull (b200tsdf_t* h, const double* pose, uint8_t* mask, int32_t* kept)
{
  if (!h || !pose || !mask) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "cull before reset()");
  cudaSetDevice (h->device);
  const Params& p = h->p;
  Planes P;
  b2host::frustum_planes (pose, p.width, p.height, p.fx, p.fy, p.min_sensor, p.max_sensor, P.pl);
  int ncells = 1 << (3 * p.C);
  unsigned char* d_mask = nullptr;
  CK (cudaMalloc (&d_mask, ncells));
  k_cull<<<(ncells + 127) / 128, 128, 0, h->stream>>> (p, P, nullptr, nullptr, d_mask, nullptr);
  CK (cudaMemcpyAsync (mask, d_mask, ncells, cudaMemcpyDeviceToHost, h->stream));
  CK (cudaStreamSynchronize (h->stream));
  cudaFree (d_mask);
  if (kept) { int k = 0; for (int i = 0; i < ncells; ++i) k += mask[i]; *kept = k; }
  return B200TSDF_OK;
}

} // extern "C"

extern "C" {

// Diagnostics (not part of include/b200tsdf.h): phase timing of k_celltop_up.  First call arms it; every call returns and
// clears the 16 counters ([0..5] max SM cycles << 32 | tag of total / level-3 / level-2 / level-1 / cell / wait-before-first-cell,
// [6..10] slow level-2 nodes, slow level-1 nodes, cell leaf visits, cell fall-throughs, cells folded).
int b200tsdf_debug_timing (b200tsdf_t* h, unsigned long long* out16)
{
  if (!h || !out16) return B200TSDF_EINVAL;
  cudaSetDevice (h->device);
  CK (cudaStreamSynchronize (h->stream));
  if (!h->d_dbg)
  {
    CK (cudaMalloc (&h->d_dbg, 16 * 8)); CK (cudaMemset (h->d_dbg, 0, 16 * 8));
    h->p.dbg = h->d_dbg;                                   // armed from the next frame on (this handle only)
    drop_batch_graphs (h);
  }
  CK (cudaMemcpy (out16, h->d_dbg, 16 * 8, cudaMemcpyDeviceToHost));
  CK (cudaMemset (h->d_dbg, 0, 16 * 8));
  return B200TSDF_OK;
}

int b200tsdf_profile_begin (b200tsdf_t* h)
{
  if (!h) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "profile before reset()");
  cudaSetDevice (h->device);
  CK (cudaStreamSynchronize (h->copy_stream));
  CK (cudaStreamSynchronize (h->stream));
  h->drain_kring (0);
  h->prof_ms_kernel = 0; h->prof_kernel_launches = 0; h->prof_frames = 0;
  h->time_frames = true; h->prof_graph0 = h->graph_launches; h->prof_nvlink0 = h->nvlink_bytes;
  h->prof_launch0 = h->launches; h->prof_h2d0 = h->h2d_bytes; h->prof_d2h0 = h->d2h_bytes;
  CK (cudaMemcpy (h->prof_stats0, h->d_stats, sizeof (h->prof_stats0), cudaMemcpyDeviceToHost));
  CK (cudaEventRecord (h->ev_p0, h->stream));
  return B200TSDF_OK;
}

int b200tsdf_profile_end (b200tsdf_t* h, b200tsdf_profile* out)
{
  if (!h || !out) return B200TSDF_EINVAL;
  cudaSetDevice (h->device);
  CK (cudaEventRecord (h->ev_p1, h->stream));
  CK (cudaStreamSynchronize (h->copy_stream));
  CK (cudaEventSynchronize (h->ev_p1));
  h->drain_kring (0);
  std::memset (out, 0, sizeof (*out));
  float ms = 0.f;
  CK (cudaEventElapsedTime (&ms, h->ev_p0, h->ev_p1));
  unsigned long long st[ST_N];
  CK (cudaMemcpy (st, h->d_stats, sizeof (st), cudaMemcpyDeviceToHost));
  out->ms_elapsed = ms;
  out->ms_kernel = h->prof_ms_kernel; out->kernel_launches = h->prof_kernel_launches;
  out->total_launches = h->launches - h->prof_launch0;
  out->n_frames = h->prof_frames;
  out->n_updates = (int64_t) (st[ST_UPDATES] - h->prof_stats0[ST_UPDATES]);
  out->n_node_visits = (int64_t) (st[ST_VISITS] - h->prof_stats0[ST_VISITS]);
  out->ms_kernel_device = 1e-6 * (double) (st[5] - h->prof_stats0[5]);
  out->kernel_launches_device = (int64_t) (st[6] - h->prof_stats0[6]);
  out->graph_launches = h->graph_launches - h->prof_graph0;
  out->nvlink_bytes = h->nvlink_bytes - h->prof_nvlink0;
  h->time_frames = false;
  out->h2d_bytes = h->h2d_bytes - h->prof_h2d0; out->d2h_bytes = h->d2h_bytes - h->prof_d2h0;
  return check_device_err (h);
}

} // extern "C"

// ---------------------------------------------------------------------------------------------
// host snapshot: a compact host copy of the volume with its own (re-hashed) directory, walked with
// the same tsdf_core.cuh routines.  Used for the node dump (tests) and the recursive .vol writer
// (I/O); it is not a compute path.
// ---------------------------------------------------------------------------------------------
namespace {

struct Snapshot
{
  Params p{};
  std::vector<uint64_t> keys; std::vector<float2> nodes; std::vector<uint32_t> split;
  std::vector<uchar4> rgb; std::vector<float> M; std::vector<int> ns;
  std::vector<float2> root_dw; std::vector<uint32_t> root_split; std::vector<uchar4> root_rgb;
  std::vector<float> root_M; std::vector<int> root_ns;
  std::vector<float4> rgbn, root_rgbn;
  int err = 0;
};

int take_snapshot (b200tsdf* h, Snapshot& S)
{
  cudaSetDevice (h->device);
  int rc = b200tsdf_sync (h);
  if (rc) return rc;
  const Params& dp = h->p;
  cudaStream_t s = h->stream;
  int* d_list = nullptr; int* d_n = h->d_count + 40;
  CK (cudaMalloc (&d_list, h->pool * sizeof (int)));
  CK (cudaMemsetAsync (d_n, 0, sizeof (int), s));
  k_list_bricks<<<(unsigned) ((h->pool + 255) / 256), 256, 0, s>>> (dp, d_list, d_n);
  int nb = 0;
  CK (cudaMemcpyAsync (&nb, d_n, sizeof (int), cudaMemcpyDeviceToHost, s));
  CK (cudaStreamSynchronize (s));
  std::vector<int> list (nb);
  std::vector<uint64_t> dkeys (h->pool);
  CK (cudaMemcpy (dkeys.data (), dp.keys, h->pool * sizeof (uint64_t), cudaMemcpyDeviceToHost));
  if (nb) CK (cudaMemcpy (list.data (), d_list, (size_t) nb * sizeof (int), cudaMemcpyDeviceToHost));
  float2* g_nodes = nullptr; uint32_t* g_split = nullptr; uchar4* g_rgb = nullptr; float* g_M = nullptr; int* g_ns = nullptr;
  size_t nbz = std::max (nb, 1);
  CK (cudaMalloc (&g_nodes, nbz * BRICK_NODES * sizeof (float2)));
  CK (cudaMalloc (&g_split, nbz * BRICK_SPLIT_WORDS * sizeof (uint32_t)));
  if (dp.rgb) CK (cudaMalloc (&g_rgb, nbz * BRICK_NODES * sizeof (uchar4)));
  if (dp.M) { CK (cudaMalloc (&g_M, nbz * BRICK_NODES * sizeof (float))); CK (cudaMalloc (&g_ns, nbz * BRICK_NODES * sizeof (int))); }
  if (nb) k_gather_bricks<<<nb, 128, 0, s>>> (dp, d_list, nb, g_nodes, g_split, g_rgb, g_M, g_ns);
  CK (cudaStreamSynchronize (s));
  std::vector<float2> c_nodes ((size_t) nb * BRICK_NODES); std::vector<uint32_t> c_split ((size_t) nb * BRICK_SPLIT_WORDS);
  std::vector<uchar4> c_rgb; std::vector<float> c_M; std::vector<int> c_ns;
  if (nb)
  {
    CK (cudaMemcpy (c_nodes.data (), g_nodes, c_nodes.size () * sizeof (float2), cudaMemcpyDeviceToHost));
    CK (cudaMemcpy (c_split.data (), g_split, c_split.size () * sizeof (uint32_t), cudaMemcpyDeviceToHost));
    if (dp.rgb) { c_rgb.resize ((size_t) nb * BRICK_NODES); CK (cudaMemcpy (c_rgb.data (), g_rgb, c_rgb.size () * sizeof (uchar4), cudaMemcpyDeviceToHost)); }
    if (dp.M)
    {
      c_M.resize ((size_t) nb * BRICK_NODES); c_ns.resize ((size_t) nb * BRICK_NODES);
      CK (cudaMemcpy (c_M.data (), g_M, c_M.size () * sizeof (float), cudaMemcpyDeviceToHost));
      CK (cudaMemcpy (c_ns.data (), g_ns, c_ns.size () * sizeof (int), cudaMemcpyDeviceToHost));
    }
  }
  std::vector<float4> c_rgbn;
  if (dp.rgbn)
  {
    float4* g_q = nullptr;
    CK (cudaMalloc (&g_q, nbz * BRICK_NODES * sizeof (float4)));
    if (nb) k_gather_rgbn<<<nb, 128, 0, s>>> (dp, d_list, nb, g_q);
    c_rgbn.resize ((size_t) nb * BRICK_NODES);
    if (nb) CK (cudaMemcpy (c_rgbn.data (), g_q, c_rgbn.size () * sizeof (float4), cudaMemcpyDeviceToHost));
    cudaFree (g_q);
  }
  cudaFree (d_list); cudaFree (g_nodes); cudaFree (g_split); cudaFree (g_rgb); cudaFree (g_M); cudaFree (g_ns);
  // compact directory
  size_t hp = 16;
  while (hp < (size_t) nb * 2) hp <<= 1;
  S.p = dp;
  S.keys.assign (hp, KEY_EMPTY);
  S.nodes.assign (hp * BRICK_NODES, make_float2 (-1.f, 0.f));
  S.split.assign (hp * BRICK_SPLIT_WORDS, 0u);
  if (dp.rgb) S.rgb.assign (hp * BRICK_NODES, make_uchar4 (0, 0, 0, 0));
  if (dp.M) { S.M.assign (hp * BRICK_NODES, 0.f); S.ns.assign (hp * BRICK_NODES, 0); }
  if (dp.rgbn) S.rgbn.assign (hp * BRICK_NODES, make_float4 (0.f, 0.f, 0.f, 0.f));
  S.p.rgbn = dp.rgbn ? S.rgbn.data () : nullptr;
  S.p.keys = S.keys.data (); S.p.pool_mask = (uint32_t) (hp - 1);
  S.p.nodes = S.nodes.data (); S.p.split = S.split.data ();
  S.p.rgb = dp.rgb ? S.rgb.data () : nullptr; S.p.M = dp.M ? S.M.data () : nullptr; S.p.ns = dp.M ? S.ns.data () : nullptr;
  S.p.err = &S.err;
  for (int i = 0; i < nb; ++i)
  {
    uint64_t key = dkeys[list[i]];
    int t = (int) (key >> 60) - 1;
    int slot = find_or_insert_brick (S.p, t, (int) ((key >> 40) & 0xFFFFF), (int) ((key >> 20) & 0xFFFFF), (int) (key & 0xFFFFF));
    std::memcpy (&S.nodes[(size_t) slot * BRICK_NODES], &c_nodes[(size_t) i * BRICK_NODES], BRICK_NODES * sizeof (float2));
    std::memcpy (&S.split[(size_t) slot * BRICK_SPLIT_WORDS], &c_split[(size_t) i * BRICK_SPLIT_WORDS], BRICK_SPLIT_WORDS * sizeof (uint32_t));
    if (dp.rgb) std::memcpy (&S.rgb[(size_t) slot * BRICK_NODES], &c_rgb[(size_t) i * BRICK_NODES], BRICK_NODES * sizeof (uchar4));
    if (dp.rgbn) std::memcpy (&S.rgbn[(size_t) slot * BRICK_NODES], &c_rgbn[(size_t) i * BRICK_NODES], BRICK_NODES * sizeof (float4));
    if (dp.M)
    {
      std::memcpy (&S.M[(size_t) slot * BRICK_NODES], &c_M[(size_t) i * BRICK_NODES], BRICK_NODES * sizeof (float));
      std::memcpy (&S.ns[(size_t) slot * BRICK_NODES], &c_ns[(size_t) i * BRICK_NODES], BRICK_NODES * sizeof (int));
    }
  }
  size_t rn = h->root_n;
  S.root_dw.resize (rn); S.root_split.resize ((rn + 31) / 32);
  CK (cudaMemcpy (S.root_dw.data (), dp.root_dw, rn * sizeof (float2), cudaMemcpyDeviceToHost));
  CK (cudaMemcpy (S.root_split.data (), dp.root_split, S.root_split.size () * sizeof (uint32_t), cudaMemcpyDeviceToHost));
  S.p.root_dw = S.root_dw.data (); S.p.root_split = S.root_split.data ();
  S.p.root_rgb = nullptr; S.p.root_M = nullptr; S.p.root_ns = nullptr; S.p.root_rgbn = nullptr;
  if (dp.root_rgbn) { S.root_rgbn.resize (rn); CK (cudaMemcpy (S.root_rgbn.data (), dp.root_rgbn, rn * sizeof (float4), cudaMemcpyDeviceToHost)); S.p.root_rgbn = S.root_rgbn.data (); }
  if (dp.root_rgb) { S.root_rgb.resize (rn); CK (cudaMemcpy (S.root_rgb.data (), dp.root_rgb, rn * sizeof (uchar4), cudaMemcpyDeviceToHost)); S.p.root_rgb = S.root_rgb.data (); }
  if (dp.root_M)
  {
    S.root_M.resize (rn); S.root_ns.resize (rn);
    CK (cudaMemcpy (S.root_M.data (), dp.root_M, rn * sizeof (float), cudaMemcpyDeviceToHost));
    CK (cudaMemcpy (S.root_ns.data (), dp.root_ns, rn * sizeof (int), cudaMemcpyDeviceToHost));
    S.p.root_M = S.root_M.data (); S.p.root_ns = S.root_ns.data ();
  }
  return B200TSDF_OK;
}

struct NodeRec { int32_t k[4]; float d, w; uint8_t split, r, g, b; float M; int32_t ns; float q[4]; };

void node_payload (const Params& p, const NodePos& n, NodeRec& r)
{
  float2 dw = *node_dw (p, n);
  r.d = dw.x; r.w = dw.y; r.r = r.g = r.b = 0; r.M = 0.f; r.ns = 0; r.q[0] = r.q[1] = r.q[2] = r.q[3] = 0.f;
  if (p.color_norm)
  {
    const float4 q = *node_rgbn (p, n); r.q[0] = q.x; r.q[1] = q.y; r.q[2] = q.z; r.q[3] = q.w;
    const uchar4 c = node_get_rgb (p, n); r.r = c.x; r.g = c.y; r.b = c.z;                 // getRGB, octree.cpp:396-402
  }
  if (n.slot < 0)
  {
    if (p.root_rgb && !p.color_norm) { uchar4 c = p.root_rgb[n.idx]; r.r = c.x; r.g = c.y; r.b = c.z; }
    if (p.root_M) { r.M = p.root_M[n.idx]; r.ns = p.root_ns[n.idx]; }
  }
  else
  {
    size_t i = (size_t) n.slot * BRICK_NODES + n.idx;
    if (p.rgb && !p.color_norm) { uchar4 c = p.rgb[i]; r.r = c.x; r.g = c.y; r.b = c.z; }
    if (p.M) { r.M = p.M[i]; r.ns = p.ns[i]; }
  }
}

void collect_nodes (const Params& p, const NodePos& n, std::vector<NodeRec>& out)
{
  NodeRec r; r.k[0] = n.level; r.k[1] = n.x; r.k[2] = n.y; r.k[3] = n.z;
  node_payload (p, n, r);
  bool sp = is_split (p, n);
  r.split = sp;
  out.push_back (r);
  if (!sp) return;
  int cs = children_slot (p, n, false);
  if (cs < 0) return;
  for (int c = 0; c < 8; ++c) collect_nodes (p, make_child (p, n, c, cs), out);
}

// OctreeNode::serialize (octree.cpp:289-304) / RGBNode::serialize (:360-367), recursive
void write_vol_node (const Params& p, std::FILE* f, const NodePos& n, bool have_state)
{
  NodeRec r; r.d = -1.f; r.w = 0.f; r.r = r.g = r.b = 0; r.M = 0.f; r.ns = 0; r.q[0] = r.q[1] = r.q[2] = r.q[3] = 0.f;
  if (have_state) node_payload (p, n, r);
  // RGBNormalized::serialize writes sizeof (uint8_t) of each of its four FLOATS, i.e. their first bytes (octree.cpp:417-424)
  if (p.color_norm) for (int k = 0; k < 4; ++k) std::fwrite (&r.q[k], 1, 1, f);
  else if (p.color) { std::fwrite (&r.r, 1, 1, f); std::fwrite (&r.g, 1, 1, f); std::fwrite (&r.b, 1, 1, f); }
  std::fwrite (&r.d, 4, 1, f); std::fwrite (&r.w, 4, 1, f);
  std::fwrite (&n.cx, 4, 1, f); std::fwrite (&n.cy, 4, 1, f); std::fwrite (&n.cz, 4, 1, f);
  std::fwrite (&n.size, 4, 1, f); std::fwrite (&r.M, 4, 1, f); std::fwrite (&r.ns, 4, 1, f);
  bool sp = have_state ? is_split (p, n) : true;
  int cs = -1;
  if (sp && have_state) { cs = children_slot (p, n, false); if (cs < 0) sp = false; }
  size_t nchild = sp ? 8 : 0;
  std::fwrite (&nchild, sizeof (size_t), 1, f);
  if (!sp) return;
  for (int c = 0; c < 8; ++c)
  {
    if (have_state) write_vol_node (p, f, make_child (p, n, c, cs), true);
    else
    {
      // levels above the root arrays carry no state: geometry only
      NodePos ch = n;
      int bx = (c >> 2) & 1, by = (c >> 1) & 1, bz = c & 1;
      float off = n.size * 0.25f;
      ch.level = n.level + 1; ch.x = 2 * n.x + bx; ch.y = 2 * n.y + by; ch.z = 2 * n.z + bz;
      ch.cx = bx ? n.cx + off : n.cx - off; ch.cy = by ? n.cy + off : n.cy - off; ch.cz = bz ? n.cz + off : n.cz - off;
      ch.size = n.size * 0.5f;
      if (ch.level == p.Rtop) { ch.slot = -1; ch.idx = root_index (p, ch.x, ch.y, ch.z); write_vol_node (p, f, ch, true); }
      else write_vol_node (p, f, ch, false);
    }
  }
}

std::string fmt16 (double x) { char b[64]; std::snprintf (b, sizeof (b), "%.16g", x); return b; }

} // namespace

extern "C" {

int64_t b200tsdf_download_nodes (b200tsdf_t* h, int32_t* keys, float* dw, uint8_t* flags,
                                 uint8_t* rgb, float* M, int32_t* ns)
{
  if (!h || !h->has_volume) return B200TSDF_EINVAL;
  Snapshot S;
  int rc = take_snapshot (h, S);
  if (rc) return rc;
  const Params& p = S.p;
  std::vector<NodeRec> recs;
  int n = 1 << p.C;
  for (int x = 0; x < n; ++x) for (int y = 0; y < n; ++y) for (int z = 0; z < n; ++z)
  {
    NodePos nd;
    if (!locate_node (p, p.C, x, y, z, nd)) return h->fail (B200TSDF_ESTATE, "coarse cell without storage");
    collect_nodes (p, nd, recs);
  }
  if (!keys && !dw && !flags && !rgb && !M && !ns) return (int64_t) recs.size ();
  std::sort (recs.begin (), recs.end (), [] (const NodeRec& a, const NodeRec& b) {
    return std::lexicographical_compare (a.k, a.k + 4, b.k, b.k + 4); });
  for (size_t i = 0; i < recs.size (); ++i)
  {
    const NodeRec& r = recs[i];
    if (keys) std::memcpy (keys + 4 * i, r.k, 16);
    if (dw) { dw[2 * i] = r.d; dw[2 * i + 1] = r.w; }
    if (flags) flags[i] = r.split;
    if (rgb) { rgb[3 * i] = r.r; rgb[3 * i + 1] = r.g; rgb[3 * i + 2] = r.b; }
    if (M) M[i] = r.M;
    if (ns) ns[i] = r.ns;
  }
  return (int64_t) recs.size ();
}

int64_t b200tsdf_download_color_payload (b200tsdf_t* h, float* out4)
{
  if (!h || !h->has_volume || !out4) return B200TSDF_EINVAL;
  if (!h->p.color_norm) return 0;
  Snapshot S;
  int rc = take_snapshot (h, S);
  if (rc) return rc;
  const Params& p = S.p;
  std::vector<NodeRec> recs;
  int n = 1 << p.C;
  for (int x = 0; x < n; ++x) for (int y = 0; y < n; ++y) for (int z = 0; z < n; ++z)
  {
    NodePos nd;
    if (!locate_node (p, p.C, x, y, z, nd)) return h->fail (B200TSDF_ESTATE, "coarse cell without storage");
    collect_nodes (p, nd, recs);
  }
  std::sort (recs.begin (), recs.end (), [] (const NodeRec& a, const NodeRec& b) {
    return std::lexicographical_compare (a.k, a.k + 4, b.k, b.k + 4); });
  for (size_t i = 0; i < recs.size (); ++i) std::memcpy (out4 + 4 * i, recs[i].q, 16);
  return (int64_t) recs.size ();
}

// save (tsdf_volume_octree.cpp:222-245; Octree::serialize octree.cpp:645-657; serializeASCII
// eigen_extensions.h:249-257)
int b200tsdf_save (b200tsdf_t* h, const char* path)
{
  if (!h || !path) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "save before reset()");
  Snapshot S;
  int rc = take_snapshot (h, S);
  if (rc) return rc;
  const b200tsdf_config& c = h->cfg;
  std::FILE* f = std::fopen (path, "wb");
  if (!f) return h->fail (B200TSDF_EIO, std::string ("cannot open ") + path);
  std::string hd = "# TSDFVolumeOctree Meta Information\n";
  hd += std::to_string (c.xres) + " " + std::to_string (c.yres) + " " + std::to_string (c.zres) + "\n";
  hd += fmt16 (c.xsize) + " " + fmt16 (c.ysize) + " " + fmt16 (c.zsize) + "\n";
  hd += fmt16 (c.max_dist_pos) + "\n" + fmt16 (c.max_dist_neg) + "\n" + fmt16 (c.max_weight) + "\n";
  hd += fmt16 (c.min_sensor_dist) + "\n" + fmt16 (c.max_sensor_dist) + "\n";
  hd += fmt16 (c.max_cell_x) + " " + fmt16 (c.max_cell_y) + " " + fmt16 (c.max_cell_z) + "\n";
  hd += fmt16 (c.fx) + " " + fmt16 (c.fy) + " " + fmt16 (c.cx) + " " + fmt16 (c.cy) + "\n";
  hd += std::to_string (c.image_width) + " " + std::to_string (c.image_height) + "\n";
  hd += std::string (h->is_empty ? "1" : "0") + "\n0\n0\n";     // is_empty_, weight_by_depth_, weight_by_variance_
  hd += "% 4 4\n";
  std::string cell[16]; size_t width = 0;
  for (int i = 0; i < 16; ++i) { cell[i] = fmt16 (c.global_transform[i]); width = std::max (width, cell[i].size ()); }
  for (int r = 0; r < 4; ++r)
  {
    for (int k = 0; k < 4; ++k) { if (k) hd += " "; hd += std::string (width - cell[r * 4 + k].size (), ' ') + cell[r * 4 + k]; }
    hd += "\n";
  }
  hd += std::string (S.p.color_norm ? "RGBNormalized" : (S.p.color ? "RGB" : "NOCOLOR")) + "\n#OCTREEBINARY\n";
  std::fwrite (hd.data (), 1, hd.size (), f);
  size_t res[3] = { (size_t) c.xres, (size_t) c.yres, (size_t) c.zres };
  std::fwrite (res, sizeof (size_t), 3, f);
  std::fwrite (&c.xsize, 4, 1, f); std::fwrite (&c.ysize, 4, 1, f); std::fwrite (&c.zsize, 4, 1, f);
  NodePos root;
  root.level = 0; root.x = root.y = root.z = 0; root.cx = root.cy = root.cz = 0.f; root.size = S.p.size; root.slot = -1; root.idx = 0;
  write_vol_node (S.p, f, root, S.p.Rtop == 0);
  bool bad = std::ferror (f);
  std::fclose (f);
  return bad ? h->fail (B200TSDF_EIO, "write failed") : B200TSDF_OK;
}


// ---- load (tsdf_volume_octree.cpp:248-275; Octree::deserialize octree.cpp:659-678; OctreeNode::deserialize :306-325) ----
namespace {
struct VolLoader
{
  std::FILE* f; bool rgb; const Params* p; bool bad = false; std::string why;
  // host image of the volume being rebuilt
  std::vector<float2> root_dw; std::vector<uint32_t> root_split; std::vector<uchar4> root_rgb; std::vector<float> root_M; std::vector<int> root_ns;
  std::vector<uint64_t> keys; std::vector<float2> nodes; std::vector<uint32_t> split; std::vector<uchar4> rgbv; std::vector<float> Mv; std::vector<int> nsv;
  std::unordered_map<uint64_t, int> index;
  int brick_of (int t, int x, int y, int z)
  {
    uint64_t key = brick_key (t, x, y, z);
    auto it = index.find (key);
    if (it != index.end ()) return it->second;
    index[key] = (int) keys.size ();
    keys.push_back (key);
    nodes.resize (keys.size () * BRICK_NODES, make_float2 (-1.f, 0.f));
    split.resize (keys.size () * BRICK_SPLIT_WORDS, 0u);
    rgbv.resize (keys.size () * BRICK_NODES, make_uchar4 (0, 0, 0, 0));
    Mv.resize (keys.size () * BRICK_NODES, 0.f); nsv.resize (keys.size () * BRICK_NODES, 0);
    return (int) keys.size () - 1;
  }
  void node (int level, int x, int y, int z)
  {
    if (bad) return;
    unsigned char c3[3] = { 0, 0, 0 };
    float v[7]; int nsamp; size_t nchild;
    bool ok = true;
    if (rgb) ok = ok && std::fread (c3, 1, 3, f) == 3;
    ok = ok && std::fread (v, 4, 7, f) == 7 && std::fread (&nsamp, 4, 1, f) == 1 && std::fread (&nchild, sizeof (size_t), 1, f) == 1;
    if (!ok || (nchild != 0 && nchild != 8)) { bad = true; why = "truncated or malformed node record"; return; }
    const Params& P = *p;
    if (level < P.C && nchild != 8) { bad = true; why = "tree is shallower than the coarse depth implied by max_cell_size"; return; }
    if (level > P.L || (level == P.L && nchild)) { bad = true; why = "tree is deeper than the resolution"; return; }
    if (level >= P.Rtop)
    {
      if (level == P.Rtop)
      {
        int ri = root_index (P, x, y, z);
        root_dw[ri] = make_float2 (v[0], v[1]); root_rgb[ri] = make_uchar4 (c3[0], c3[1], c3[2], 0); root_M[ri] = v[6]; root_ns[ri] = nsamp;
        if (nchild && level >= P.C) root_split[ri >> 5] |= 1u << (ri & 31);
      }
      else
      {
        int t = tier_of_level (P, level), k = level - tier_root_level (P, t);
        int b = brick_of (t, x >> k, y >> k, z >> k);
        int j = path_index (k, x, y, z), idx = node_offset (k) + j;
        size_t o = (size_t) b * BRICK_NODES + idx;
        nodes[o] = make_float2 (v[0], v[1]); rgbv[o] = make_uchar4 (c3[0], c3[1], c3[2], 0); Mv[o] = v[6]; nsv[o] = nsamp;
        if (nchild && level >= P.C && level < P.L) split[(size_t) b * BRICK_SPLIT_WORDS + split_word_base (k) + (j >> 5)] |= 1u << (j & 31);
      }
    }
    for (size_t c = 0; c < nchild; ++c) node (level + 1, 2 * x + (int) ((c >> 2) & 1), 2 * y + (int) ((c >> 1) & 1), 2 * z + (int) (c & 1));
  }
};
}

int b200tsdf_load (b200tsdf_t* h, const char* path)
{
  if (!h || !path) return B200TSDF_EINVAL;
  std::FILE* f = std::fopen (path, "rb");
  if (!f) return h->fail (B200TSDF_EIO, std::string ("cannot open ") + path);
  b200tsdf_config c = h->cfg_pending;
  char line[1024];
  auto fail = [&] (const std::string& m) { std::fclose (f); return h->fail (B200TSDF_EIO, std::string (path) + ": " + m); };
  if (!std::fgets (line, sizeof (line), f)) return fail ("empty file");
  int is_empty = 0, wd = 0, wv = 0;
  double gt[16];
  int nread = std::fscanf (f, "%d %d %d %f %f %f %f %f %f %f %f %f %f %f %lf %lf %lf %lf %d %d %d %d %d",
                           &c.xres, &c.yres, &c.zres, &c.xsize, &c.ysize, &c.zsize, &c.max_dist_pos, &c.max_dist_neg, &c.max_weight,
                           &c.min_sensor_dist, &c.max_sensor_dist, &c.max_cell_x, &c.max_cell_y, &c.max_cell_z,
                           &c.fx, &c.fy, &c.cx, &c.cy, &c.image_width, &c.image_height, &is_empty, &wd, &wv);
  if (nread != 23) return fail ("bad header");
  // the reference has no setter for these two: only a .vol written with them set turns the alternative weightings on (hpp:200-204)
  if (wd || wv) return fail ("weight_by_depth_ / weight_by_variance_ volumes are not supported (the fusion here uses w_new = 1)");
  char pct[8]; int rr = 0, cc = 0;
  if (std::fscanf (f, " %1s %d %d", pct, &rr, &cc) != 3 || pct[0] != '%' || rr != 4 || cc != 4) return fail ("bad transform header");
  for (int i = 0; i < 16; ++i) if (std::fscanf (f, "%lf", &gt[i]) != 1) return fail ("bad transform");
  char type[64];
  if (std::fscanf (f, "%63s", type) != 1) return fail ("missing node type");
  bool rgb = std::string (type) == "RGB";
  if (!rgb && std::string (type) != "NOCOLOR") return fail (std::string ("unsupported node type ") + type);
  do { if (!std::fgets (line, sizeof (line), f)) return fail ("missing #OCTREEBINARY"); } while (!(line[0] == '#' && line[1] == 'O'));
  size_t res3[3]; float size3[3];
  if (std::fread (res3, sizeof (size_t), 3, f) != 3 || std::fread (size3, 4, 3, f) != 3) return fail ("truncated octree header");
  c.integrate_color = rgb ? 1 : 0;
  for (int i = 0; i < 16; ++i) c.global_transform[i] = gt[i];
  h->cfg_pending = c;
  int rc = b200tsdf_reset (h);
  if (rc) { std::fclose (f); return rc; }
  const Params& p = h->p;
  VolLoader L; L.f = f; L.rgb = rgb; L.p = &p;
  size_t rn = h->root_n;
  L.root_dw.assign (rn, make_float2 (-1.f, 0.f)); L.root_split.assign ((rn + 31) / 32, 0u);
  L.root_rgb.assign (rn, make_uchar4 (0, 0, 0, 0)); L.root_M.assign (rn, 0.f); L.root_ns.assign (rn, 0);
  L.node (0, 0, 0, 0);
  std::fclose (f);
  if (L.bad) return h->fail (B200TSDF_EIO, std::string (path) + ": " + L.why);
  cudaSetDevice (h->device);
  CK (cudaMemcpy (p.root_dw, L.root_dw.data (), rn * sizeof (float2), cudaMemcpyHostToDevice));
  CK (cudaMemcpy (p.root_split, L.root_split.data (), L.root_split.size () * sizeof (uint32_t), cudaMemcpyHostToDevice));
  if (p.root_rgb) CK (cudaMemcpy (p.root_rgb, L.root_rgb.data (), rn * sizeof (uchar4), cudaMemcpyHostToDevice));
  if (p.root_M) { CK (cudaMemcpy (p.root_M, L.root_M.data (), rn * sizeof (float), cudaMemcpyHostToDevice)); CK (cudaMemcpy (p.root_ns, L.root_ns.data (), rn * sizeof (int), cudaMemcpyHostToDevice)); }
  int nb = (int) L.keys.size ();
  if (nb)
  {
    uint64_t* dk = nullptr; float2* dn = nullptr; uint32_t* ds = nullptr; uchar4* dc = nullptr; float* dM = nullptr; int* dns = nullptr;
    CK (cudaMalloc (&dk, (size_t) nb * 8)); CK (cudaMalloc (&dn, (size_t) nb * BRICK_NODES * sizeof (float2))); CK (cudaMalloc (&ds, (size_t) nb * BRICK_SPLIT_WORDS * 4));
    CK (cudaMemcpy (dk, L.keys.data (), (size_t) nb * 8, cudaMemcpyHostToDevice));
    CK (cudaMemcpy (dn, L.nodes.data (), (size_t) nb * BRICK_NODES * sizeof (float2), cudaMemcpyHostToDevice));
    CK (cudaMemcpy (ds, L.split.data (), (size_t) nb * BRICK_SPLIT_WORDS * 4, cudaMemcpyHostToDevice));
    if (p.rgb) { CK (cudaMalloc (&dc, (size_t) nb * BRICK_NODES * 4)); CK (cudaMemcpy (dc, L.rgbv.data (), (size_t) nb * BRICK_NODES * 4, cudaMemcpyHostToDevice)); }
    if (p.M)
    {
      CK (cudaMalloc (&dM, (size_t) nb * BRICK_NODES * 4)); CK (cudaMalloc (&dns, (size_t) nb * BRICK_NODES * 4));
      CK (cudaMemcpy (dM, L.Mv.data (), (size_t) nb * BRICK_NODES * 4, cudaMemcpyHostToDevice));
      CK (cudaMemcpy (dns, L.nsv.data (), (size_t) nb * BRICK_NODES * 4, cudaMemcpyHostToDevice));
    }
    k_load_bricks<<<nb, 128, 0, h->stream>>> (p, dk, nb, dn, ds, dc, dM, dns);
    CK (cudaStreamSynchronize (h->stream));
    cudaFree (dk); cudaFree (dn); cudaFree (ds); cudaFree (dc); cudaFree (dM); cudaFree (dns);
  }
  h->is_empty = is_empty != 0;
  return check_device_err (h);
}


// ---- shard export / import ------------------------------------------------------------------------------------
namespace {
struct ShardHeader { uint32_t magic, version; int32_t L, C, T, Rtop, color, var; uint32_t n_roots, n_bricks; float size; uint32_t pad; };
constexpr uint32_t SHARD_MAGIC = 0x42325348;   // "B2SH"
}

int b200tsdf_export_shard (b200tsdf_t* h, void* buf, size_t capacity, size_t* nbytes)
{
  if (!h || !nbytes) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "export before reset()");
  if (h->p.Rtop != h->p.C) return h->fail (B200TSDF_EINVAL, "shard export needs a grid whose coarse cells are the top-tier roots");
  if (h->p.color_norm) return h->fail (B200TSDF_EINVAL, "shard export does not carry the RGBNormalized payload");
  Snapshot S;
  int rc = take_snapshot (h, S);
  if (rc) return rc;
  const Params& p = S.p;
  const bool color = p.rgb != nullptr, var = p.M != nullptr;
  // owned coarse cells and the bricks below them
  std::vector<int> roots;
  int n = 1 << p.C;
  for (int x = 0; x < n; ++x) for (int y = 0; y < n; ++y) for (int z = 0; z < n; ++z) if (owns_cell (p, x, y, z)) roots.push_back (root_index (p, x, y, z));
  std::vector<uint32_t> bricks;
  for (uint32_t s = 0; s <= p.pool_mask; ++s)
  {
    uint64_t key = p.keys[s];
    if (key == KEY_EMPTY) continue;
    int t = (int) (key >> 60) - 1;
    int sh = tier_root_level (p, t) - p.C;
    int bx = (int) ((key >> 40) & 0xFFFFF), by = (int) ((key >> 20) & 0xFFFFF), bz = (int) (key & 0xFFFFF);
    if (owns_cell (p, bx >> sh, by >> sh, bz >> sh)) bricks.push_back (s);
  }
  const size_t root_rec = 4 + 8 + 1 + 4 + 4 + 4, brick_rec = 8 + BRICK_NODES * 8 + BRICK_SPLIT_WORDS * 4 + (color ? BRICK_NODES * 4 : 0) + (var ? BRICK_NODES * 8 : 0);
  size_t need = sizeof (ShardHeader) + roots.size () * root_rec + bricks.size () * brick_rec;
  *nbytes = need;
  if (!buf) return B200TSDF_OK;
  if (capacity < need) return h->fail (B200TSDF_EINVAL, "export buffer too small");
  unsigned char* o = (unsigned char*) buf;
  ShardHeader hd{}; hd.magic = SHARD_MAGIC; hd.version = 1; hd.L = p.L; hd.C = p.C; hd.T = p.T; hd.Rtop = p.Rtop; hd.color = color; hd.var = var;
  hd.n_roots = (uint32_t) roots.size (); hd.n_bricks = (uint32_t) bricks.size (); hd.size = p.size;
  std::memcpy (o, &hd, sizeof (hd)); o += sizeof (hd);
  for (int r : roots)
  {
    std::memcpy (o, &r, 4); o += 4;
    std::memcpy (o, &p.root_dw[r], 8); o += 8;
    *o++ = (unsigned char) ((p.root_split[r >> 5] >> (r & 31)) & 1);
    uchar4 c = p.root_rgb ? p.root_rgb[r] : make_uchar4 (0, 0, 0, 0); std::memcpy (o, &c, 4); o += 4;
    float M = p.root_M ? p.root_M[r] : 0.f; int nsv = p.root_ns ? p.root_ns[r] : 0;
    std::memcpy (o, &M, 4); o += 4; std::memcpy (o, &nsv, 4); o += 4;
  }
  for (uint32_t s : bricks)
  {
    std::memcpy (o, &p.keys[s], 8); o += 8;
    std::memcpy (o, &p.nodes[(size_t) s * BRICK_NODES], BRICK_NODES * 8); o += BRICK_NODES * 8;
    std::memcpy (o, &p.split[(size_t) s * BRICK_SPLIT_WORDS], BRICK_SPLIT_WORDS * 4); o += BRICK_SPLIT_WORDS * 4;
    if (color) { std::memcpy (o, &p.rgb[(size_t) s * BRICK_NODES], BRICK_NODES * 4); o += BRICK_NODES * 4; }
    if (var) { std::memcpy (o, &p.M[(size_t) s * BRICK_NODES], BRICK_NODES * 4); o += BRICK_NODES * 4; std::memcpy (o, &p.ns[(size_t) s * BRICK_NODES], BRICK_NODES * 4); o += BRICK_NODES * 4; }
  }
  return B200TSDF_OK;
}

int b200tsdf_import_shard (b200tsdf_t* h, const void* buf, size_t nbytes)
{
  if (!h || !buf || nbytes < sizeof (ShardHeader)) return B200TSDF_EINVAL;
  if (!h->has_volume) return h->fail (B200TSDF_ESTATE, "import before reset()");
  const Params& p = h->p;
  ShardHeader hd; std::memcpy (&hd, buf, sizeof (hd));
  const bool color = p.rgb != nullptr, var = p.M != nullptr;
  if (hd.magic != SHARD_MAGIC || hd.version != 1) return h->fail (B200TSDF_EINVAL, "not a shard buffer");
  if (hd.L != p.L || hd.C != p.C || hd.T != p.T || hd.Rtop != p.Rtop || hd.size != p.size || (hd.color != 0) != color || (hd.var != 0) != var)
    return h->fail (B200TSDF_EINVAL, "shard was exported from a different grid configuration");
  const size_t root_rec = 4 + 8 + 1 + 4 + 4 + 4, brick_rec = 8 + BRICK_NODES * 8 + BRICK_SPLIT_WORDS * 4 + (color ? BRICK_NODES * 4 : 0) + (var ? BRICK_NODES * 8 : 0);
  if (nbytes != sizeof (ShardHeader) + (size_t) hd.n_roots * root_rec + (size_t) hd.n_bricks * brick_rec) return h->fail (B200TSDF_EINVAL, "truncated shard buffer");
  cudaSetDevice (h->device);
  int rc = b200tsdf_sync (h);
  if (rc) return rc;
  const unsigned char* o = (const unsigned char*) buf + sizeof (ShardHeader);
  size_t nr = hd.n_roots, nb = hd.n_bricks;
  std::vector<int> ridx (nr); std::vector<float2> rdw (nr); std::vector<unsigned char> rsp (nr); std::vector<uchar4> rrgb (nr); std::vector<float> rM (nr); std::vector<int> rns (nr);
  for (size_t i = 0; i < nr; ++i)
  {
    std::memcpy (&ridx[i], o, 4); o += 4; std::memcpy (&rdw[i], o, 8); o += 8; rsp[i] = *o++;
    std::memcpy (&rrgb[i], o, 4); o += 4; std::memcpy (&rM[i], o, 4); o += 4; std::memcpy (&rns[i], o, 4); o += 4;
    if (ridx[i] < 0 || (size_t) ridx[i] >= h->root_n) return h->fail (B200TSDF_EINVAL, "corrupt shard buffer");
  }
  std::vector<uint64_t> keys (nb); std::vector<float2> nodes (nb * BRICK_NODES); std::vector<uint32_t> split (nb * BRICK_SPLIT_WORDS);
  std::vector<uchar4> rgb (color ? nb * BRICK_NODES : 0); std::vector<float> Mv (var ? nb * BRICK_NODES : 0); std::vector<int> nsv (var ? nb * BRICK_NODES : 0);
  for (size_t i = 0; i < nb; ++i)
  {
    std::memcpy (&keys[i], o, 8); o += 8;
    std::memcpy (&nodes[i * BRICK_NODES], o, BRICK_NODES * 8); o += BRICK_NODES * 8;
    std::memcpy (&split[i * BRICK_SPLIT_WORDS], o, BRICK_SPLIT_WORDS * 4); o += BRICK_SPLIT_WORDS * 4;
    if (color) { std::memcpy (&rgb[i * BRICK_NODES], o, BRICK_NODES * 4); o += BRICK_NODES * 4; }
    if (var) { std::memcpy (&Mv[i * BRICK_NODES], o, BRICK_NODES * 4); o += BRICK_NODES * 4; std::memcpy (&nsv[i * BRICK_NODES], o, BRICK_NODES * 4); o += BRICK_NODES * 4; }
  }
  cudaStream_t s = h->stream;
  auto up = [&] (const void* src, size_t bytes, void** dst) -> cudaError_t { if (!bytes) { *dst = nullptr; return cudaSuccess; } cudaError_t e = cudaMalloc (dst, bytes); if (e != cudaSuccess) return e; return cudaMemcpy (*dst, src, bytes, cudaMemcpyHostToDevice); };
  void *d_idx = nullptr, *d_dw = nullptr, *d_sp = nullptr, *d_rgb = nullptr, *d_M = nullptr, *d_ns = nullptr;
  if (nr)
  {
    CK (up (ridx.data (), nr * 4, &d_idx)); CK (up (rdw.data (), nr * 8, &d_dw)); CK (up (rsp.data (), nr, &d_sp));
    CK (up (rrgb.data (), nr * 4, &d_rgb)); CK (up (rM.data (), nr * 4, &d_M)); CK (up (rns.data (), nr * 4, &d_ns));
    k_import_roots<<<(unsigned) ((nr + 127) / 128), 128, 0, s>>> (p, (int) nr, (const int*) d_idx, (const float2*) d_dw, (const unsigned char*) d_sp, (const uchar4*) d_rgb, (const float*) d_M, (const int*) d_ns);
    CK (cudaStreamSynchronize (s));
    cudaFree (d_idx); cudaFree (d_dw); cudaFree (d_sp); cudaFree (d_rgb); cudaFree (d_M); cudaFree (d_ns);
  }
  if (nb)
  {
    void *dk = nullptr, *dn = nullptr, *ds = nullptr, *dc = nullptr, *dM = nullptr, *dns = nullptr;
    CK (up (keys.data (), nb * 8, &dk)); CK (up (nodes.data (), nb * BRICK_NODES * 8, &dn)); CK (up (split.data (), nb * BRICK_SPLIT_WORDS * 4, &ds));
    if (color) CK (up (rgb.data (), nb * BRICK_NODES * 4, &dc));
    if (var) { CK (up (Mv.data (), nb * BRICK_NODES * 4, &dM)); CK (up (nsv.data (), nb * BRICK_NODES * 4, &dns)); }
    k_load_bricks<<<(unsigned) nb, 128, 0, s>>> (p, (const uint64_t*) dk, (int) nb, (const float2*) dn, (const uint32_t*) ds, (const uchar4*) dc, (const float*) dM, (const int*) dns);
    CK (cudaStreamSynchronize (s));
    cudaFree (dk); cudaFree (dn); cudaFree (ds); cudaFree (dc); cudaFree (dM); cudaFree (dns);
  }
  h->is_empty = false;
  return check_device_err (h);
}

} // extern "C"


#include "multigpu.cuh"
