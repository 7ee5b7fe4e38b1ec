// tsdf_core.cuh — data layout and per-node arithmetic of the B200 TSDF engine.
//
// The reference keeps the volume as a pointer-based octree of heap nodes
// (include/cpu_tsdf/octree.h:55-172).  Here the same information — every node's {d,w}, a
// "has children" bit, optional rgb / variance state — lives in flat arrays:
//
//   * root arrays: one entry per node at level Rtop = L - 3T (dense, 8^Rtop entries);
//   * bricks: a brick of tier t is the three levels below a node at level R_t = L - 3(t+1):
//     8 + 64 + 512 nodes in hierarchical (octree) order, children of node j at 8j..8j+7.
//     Tier 0 bricks are the 8^3 finest-voxel blocks.  Bricks live in an open-addressing hash
//     keyed by (tier, root coords); the payload slot IS the hash slot, so there is no
//     allocator and no pointer to chase: nodes[slot*584 + i], split[slot*20 + w].
//
// A node "exists" iff every ancestor at level >= C has its split bit set.  Invariant: storage
// of non-existent nodes is always fresh (d=-1, w=0, split=0, rgb=0, M=0, ns=0), so splitting
// is one atomicOr and pruning resets eight nodes.
//
// Everything here is __host__ __device__: kernels in engine.cu call it on the GPU, and
// tests/emu compiles the very same code for the host to check the logic without a GPU
// (a test harness — the shipped library has no CPU path).
//
// Arithmetic follows the reference expression by expression with contraction disabled
// (__f*_rn intrinsics on the device): see DESIGN.md "Arithmetic conventions".
#pragma once
#include <stdint.h>
#include <math.h>
#include <limits.h>

#if defined(__CUDACC__)
#define B2_HD __host__ __device__ __forceinline__
#define B2_HDN __host__ __device__
#else
#define B2_HD inline
#define B2_HDN
#endif

#if !defined(__CUDACC__)
struct float2 { float x, y; };
struct uchar4 { unsigned char x, y, z, w; };
struct float4 { float x, y, z, w; };
static inline float4 make_float4 (float a, float b, float c, float d) { float4 r; r.x = a; r.y = b; r.z = c; r.w = d; return r; }
static inline float2 make_float2 (float a, float b) { float2 r; r.x = a; r.y = b; return r; }
static inline uchar4 make_uchar4 (unsigned char a, unsigned char b, unsigned char c, unsigned char d)
{ uchar4 r; r.x = a; r.y = b; r.z = c; r.w = d; return r; }
#endif

namespace b2 {

constexpr int BRICK_NODES = 584;        // 8 + 64 + 512
constexpr int BRICK_SPLIT_WORDS = 20;   // word 0: 8 bits, words 1-2: 64 bits, word 3: spare, words 4-19: 512 bits
constexpr uint64_t KEY_EMPTY = 0ull;
constexpr int MAX_PROBE = 4096;

enum ErrBits { ERR_POOL_FULL = 1, ERR_MISSING_BRICK = 2, ERR_QUEUE_FULL = 4 };

// ---- rounding-exact scalar ops ------------------------------------------------------------
B2_HD float fadd (float a, float b)
{
#ifdef __CUDA_ARCH__
  return __fadd_rn (a, b);
#else
  return a + b;
#endif
}
B2_HD float fsub (float a, float b)
{
#ifdef __CUDA_ARCH__
  return __fsub_rn (a, b);
#else
  return a - b;
#endif
}
B2_HD float fmul (float a, float b)
{
#ifdef __CUDA_ARCH__
  return __fmul_rn (a, b);
#else
  return a * b;
#endif
}
B2_HD float fdiv (float a, float b)
{
#ifdef __CUDA_ARCH__
  return __fdiv_rn (a, b);
#else
  return a / b;
#endif
}
B2_HD double dadd (double a, double b)
{
#ifdef __CUDA_ARCH__
  return __dadd_rn (a, b);
#else
  return a + b;
#endif
}
B2_HD double dmul (double a, double b)
{
#ifdef __CUDA_ARCH__
  return __dmul_rn (a, b);
#else
  return a * b;
#endif
}
B2_HD double ddiv (double a, double b)
{
#ifdef __CUDA_ARCH__
  return __ddiv_rn (a, b);
#else
  return a / b;
#endif
}
// double -> int the way x86-64 cvttsd2si does it (the reference's platform): out of range or
// NaN gives INT_MIN (tsdf_volume_octree.cpp:614-615 relies on the conversion)
B2_HD int to_int_x86 (double v)
{
  if (!(v > -2147483649.0 && v < 2147483648.0)) return INT_MIN;
  return (int) v;
}
B2_HD bool is_nan (float v) { return v != v; }

// ---- parameters ---------------------------------------------------------------------------
struct Params
{
  // grid
  int L, C, T, Rtop;          // finest level, coarse level, tiers, level of the root arrays
  int res;                    // 2^L
  float size;                 // xsize_ (cubic grids only, SURVEY.md §A.3-4)
  float half;                 // size/2 (Octree::getContainingVoxel bounds, octree.cpp:631)
  float finest_size;          // xsize_/xres_ (hpp:80, :165)
  double dsize, dres;         // (double)xsize_, (double)xres_ for getVoxelIndex/Center
  float voff;                 // float(xsize_/2.0)   getVoxelCenter cpp:556
  // fusion
  float max_dist_pos, max_dist_neg, max_weight, min_sensor, max_sensor;
  double rc_thresh;           // 0.99 * max_dist_pos_ / max_dist_neg_ (hpp:211)
  double fx, fy, cx, cy;
  float fx_f, fy_f, cx_f, cy_f;   // float-rounded intrinsics for the guarded fast projection (see project_pixel)
  int fast_proj;                  // 1 when the guard's error bound holds (image < 8192 px)
  // float forms of the double comparisons, used by the brick kernel (brick_direct.cuh): for a float d,
  // (double) d < t  <=>  d < (smallest float >= t)
  float rc_lo_f, rc_hi_f;         // thresholds -0.99 and rc_thresh of the return code (hpp:209-214)
  float proj_guard;               // half-width of the band around an integer inside which the float pixel estimate is not trusted
  int exact_div_ok;               // 1 when every divisor of the update lies where __fdiv_rn takes its fast path (see div_with)
  int width, height;
  int color, track_var;
  int color_norm;                 // colour payload is RGBNormalized (setColorMode ("RGBNormalized"), octree.cpp:379-434) instead of RGB
  // sharding: this device owns coarse cells with cell_hash % shard_count == shard_rank
  int shard_rank, shard_count;
  // storage
  uint64_t* keys;             // [pool]
  uint32_t pool_mask;
  float2* nodes;              // [pool][584]
  uint32_t* split;            // [pool][20]
  uchar4* rgb;                // [pool][584] or null
  float* M;                   // [pool][584] or null
  int* ns;                    // [pool][584] or null
  float2* root_dw;            // [8^Rtop]
  uint32_t* root_split;       // bitset over 8^Rtop
  uchar4* root_rgb;
  float4* rgbn;               // [pool][584] {r_n_, g_n_, b_n_, i_} when color_norm, else null
  float4* root_rgbn;
  float* root_M;
  int* root_ns;
  unsigned char* work;        // [pool] finest-tier bricks: interior level-2 nodes seen by the last update (scheduling hint only)
  int* err;                   // device error bits
  unsigned long long* diag;   // [0] slow folds in the upper sweeps, [1] visits inside them (this handle's counters; may be null)
  unsigned long long* dbg;    // optional phase timing of k_celltop_up (b200tsdf_debug_timing), normally null
};

struct Frame
{
  const unsigned char* pts;   // organized cloud, device memory
  int stride, xyz_off, rgba_off, width, height;
  float tinv[12];             // float(trans.inverse()) rows 0..2   (hpp:54)
  float tfwd[12];             // trans.cast<float>()     rows 0..2   (hpp:76)
};

B2_HD const float* frame_xyz (const Frame& f, int u, int v)
{ return (const float*) (f.pts + ((size_t) v * f.width + u) * f.stride + f.xyz_off); }
B2_HD const unsigned char* frame_bgr (const Frame& f, int u, int v)
{ return f.pts + ((size_t) v * f.width + u) * f.stride + f.rgba_off; }

// ---- third-party arithmetic conventions (see oracle/ref_arith.h for the citations) ---------
// Eigen Affine3f * Vector3f: t + (l0*x + (l1*y + l2*z))
B2_HD void affine_mul_f (const float* m, float x, float y, float z, float* o)
{
  o[0] = fadd (m[3],  fadd (fmul (m[0], x), fadd (fmul (m[1], y), fmul (m[2],  z))));
  o[1] = fadd (m[7],  fadd (fmul (m[4], x), fadd (fmul (m[5], y), fmul (m[6],  z))));
  o[2] = fadd (m[11], fadd (fmul (m[8], x), fadd (fmul (m[9], y), fmul (m[10], z))));
}
// Eigen Matrix3f * Vector3f: l0*x + (l1*y + l2*z)
B2_HD void linear_mul_f (const float* m, float x, float y, float z, float* o)
{
  o[0] = fadd (fmul (m[0], x), fadd (fmul (m[1], y), fmul (m[2],  z)));
  o[1] = fadd (fmul (m[4], x), fadd (fmul (m[5], y), fmul (m[6],  z)));
  o[2] = fadd (fmul (m[8], x), fadd (fmul (m[9], y), fmul (m[10], z)));
}
// pcl::transformPoint (SSE2 Transformer<float>::se3): c0*x + (c1*y + (c2*z + c3))
B2_HD void pcl_transform_point_f (const float* m, float x, float y, float z, float* o)
{
  o[0] = fadd (fmul (m[0], x), fadd (fmul (m[1], y), fadd (fmul (m[2],  z), m[3])));
  o[1] = fadd (fmul (m[4], x), fadd (fmul (m[5], y), fadd (fmul (m[6],  z), m[7])));
  o[2] = fadd (fmul (m[8], x), fadd (fmul (m[9], y), fadd (fmul (m[10], z), m[11])));
}
// Vector3f::normalize(): z = x^2 + (y^2 + z^2); if (z > 0) v /= sqrt(z)
B2_HD void normalize3 (float* v)
{
  float z = fadd (fmul (v[0], v[0]), fadd (fmul (v[1], v[1]), fmul (v[2], v[2])));
  if (z > 0.f)
  {
    float n = sqrtf (z);     // correctly rounded on both host and device
    v[0] = fdiv (v[0], n); v[1] = fdiv (v[1], n); v[2] = fdiv (v[2], n);
  }
}

// ---- geometry ------------------------------------------------------------------------------
// centre of the node with integer coordinate x at `level`, accumulated exactly as
// OctreeNode::split does from the root (octree.cpp:244-266): ctr +/- size/4, size halves
B2_HD float center1d (const Params& p, int level, int x)
{
  float c = 0.f;
  float off = p.size * 0.25f;
  for (int i = level - 1; i >= 0; --i)
  {
    c = ((x >> i) & 1) ? fadd (c, off) : fsub (c, off);
    off *= 0.5f;
  }
  return c;
}
// node size at a level: size_/2 repeated (exact)
B2_HD float level_size (const Params& p, int level)
{
  float s = p.size;
  for (int i = 0; i < level; ++i) s *= 0.5f;
  return s;
}

// ---- brick addressing ----------------------------------------------------------------------
B2_HD int tier_of_level (const Params& p, int level) { return (p.L - level) / 3; }          // level in (Rtop, L]
B2_HD int tier_root_level (const Params& p, int t) { return p.L - 3 * (t + 1); }
// hierarchical index of the node with brick-relative coords (low k bits) at relative level k
B2_HD int path_index (int k, int x, int y, int z)
{
  int j = 0;
  for (int i = k - 1; i >= 0; --i)
    j = (j << 3) | (((x >> i) & 1) << 2) | (((y >> i) & 1) << 1) | ((z >> i) & 1);
  return j;
}
B2_HD int node_offset (int k) { return k == 1 ? 0 : (k == 2 ? 8 : 72); }
B2_HD int split_word_base (int k) { return k == 1 ? 0 : (k == 2 ? 1 : 4); }

B2_HD uint64_t brick_key (int t, int bx, int by, int bz)
{ return ((uint64_t) (t + 1) << 60) | ((uint64_t) bx << 40) | ((uint64_t) by << 20) | (uint64_t) bz; }
B2_HD uint32_t hash_key (uint64_t k)
{
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return (uint32_t) k;
}

B2_HD uint64_t atomic_cas64 (uint64_t* a, uint64_t cmp, uint64_t val)
{
#ifdef __CUDA_ARCH__
  return atomicCAS ((unsigned long long*) a, (unsigned long long) cmp, (unsigned long long) val);
#else
  uint64_t old = *a; if (old == cmp) *a = val; return old;
#endif
}
B2_HD uint32_t atomic_or32 (uint32_t* a, uint32_t v)
{
#ifdef __CUDA_ARCH__
  return atomicOr (a, v);
#else
  uint32_t old = *a; *a = old | v; return old;
#endif
}
B2_HD uint32_t atomic_and32 (uint32_t* a, uint32_t v)
{
#ifdef __CUDA_ARCH__
  return atomicAnd (a, v);
#else
  uint32_t old = *a; *a = old & v; return old;
#endif
}
B2_HD void raise_err (const Params& p, int bit)
{
#ifdef __CUDA_ARCH__
  atomicOr (p.err, bit);
#else
  *p.err |= bit;
#endif
}

// lookup only; -1 if absent
B2_HD int find_brick (const Params& p, int t, int bx, int by, int bz)
{
  uint64_t key = brick_key (t, bx, by, bz);
  uint32_t s = hash_key (key) & p.pool_mask;
  for (int i = 0; i < MAX_PROBE; ++i)
  {
    uint64_t k = p.keys[s];
    if (k == key) return (int) s;
    if (k == KEY_EMPTY) return -1;
    s = (s + 1) & p.pool_mask;
  }
  return -1;
}
// find or claim; the payload of an unclaimed slot is fresh by invariant, so claiming is one CAS
B2_HD int find_or_insert_brick (const Params& p, int t, int bx, int by, int bz)
{
  uint64_t key = brick_key (t, bx, by, bz);
  uint32_t s = hash_key (key) & p.pool_mask;
  for (int i = 0; i < MAX_PROBE; ++i)
  {
    uint64_t k = p.keys[s];
    if (k == key) return (int) s;
    if (k == KEY_EMPTY)
    {
      uint64_t prev = atomic_cas64 (&p.keys[s], KEY_EMPTY, key);
      if (prev == KEY_EMPTY || prev == key) return (int) s;
    }
    s = (s + 1) & p.pool_mask;
  }
  raise_err (p, ERR_POOL_FULL);
  return -1;
}

// ---- a node position during traversal ------------------------------------------------------
struct NodePos
{
  int level, x, y, z;     // integer coordinates at the node's own level
  float cx, cy, cz, size; // OctreeNode::ctr_*_, size_
  int slot;               // brick holding this node's state, -1 = root arrays
  int idx;                // node index inside the brick (0..583) or linear root index
};

B2_HD int root_index (const Params& p, int x, int y, int z)
{ int n = 1 << p.Rtop; return (x * n + y) * n + z; }

B2_HD float2* node_dw (const Params& p, const NodePos& n)
{ return n.slot < 0 ? &p.root_dw[n.idx] : &p.nodes[(size_t) n.slot * BRICK_NODES + n.idx]; }

// split-bit location of a node (finest-level nodes have none)
B2_HD uint32_t* split_word (const Params& p, const NodePos& n, uint32_t& mask)
{
  if (n.slot < 0) { mask = 1u << (n.idx & 31); return &p.root_split[n.idx >> 5]; }
  int k = n.level - tier_root_level (p, tier_of_level (p, n.level));
  int j = n.idx - node_offset (k);
  mask = 1u << (j & 31);
  return &p.split[(size_t) n.slot * BRICK_SPLIT_WORDS + split_word_base (k) + (j >> 5)];
}
B2_HD bool is_split (const Params& p, const NodePos& n)
{
  if (n.level < p.C) return true;        // levels above the coarse depth are split by init (octree.cpp:584-599)
  if (n.level >= p.L) return false;
  uint32_t m; const uint32_t* w = split_word (p, n, m);
  return (*w & m) != 0;
}

// child c (= (x>cx)*4 + (y>cy)*2 + (z>cz), octree.cpp:119, :257-264) of a node whose children
// exist.  `child_slot` is the brick that holds the children: the node's own brick unless the
// node is the last level of its brick (or a root-array node), in which case it is the brick
// rooted at the node.  Returns false if that brick is missing.
B2_HD int children_slot (const Params& p, const NodePos& n, bool insert)
{
  bool own = n.slot >= 0 && (n.level - tier_root_level (p, tier_of_level (p, n.level))) < 3;
  if (own) return n.slot;
  int t = tier_of_level (p, n.level + 1);
  return insert ? find_or_insert_brick (p, t, n.x, n.y, n.z) : find_brick (p, t, n.x, n.y, n.z);
}
B2_HD NodePos make_child (const Params& p, const NodePos& n, int c, int child_slot)
{
  NodePos ch;
  int bx = (c >> 2) & 1, by = (c >> 1) & 1, bz = c & 1;
  float off = n.size * 0.25f;
  ch.level = n.level + 1;
  ch.x = 2 * n.x + bx; ch.y = 2 * n.y + by; ch.z = 2 * n.z + bz;
  ch.cx = bx ? fadd (n.cx, off) : fsub (n.cx, off);
  ch.cy = by ? fadd (n.cy, off) : fsub (n.cy, off);
  ch.cz = bz ? fadd (n.cz, off) : fsub (n.cz, off);
  ch.size = n.size * 0.5f;
  ch.slot = child_slot;
  if (child_slot == n.slot && n.slot >= 0)
  {
    int k = n.level - tier_root_level (p, tier_of_level (p, n.level));
    int j = n.idx - node_offset (k);
    ch.idx = node_offset (k + 1) + (j << 3) + c;
  }
  else ch.idx = c;           // first level of the brick rooted at n
  return ch;
}
// node at (level, x, y, z) for level == Rtop (root arrays)
B2_HD NodePos make_root (const Params& p, int x, int y, int z)
{
  NodePos n;
  n.level = p.Rtop; n.x = x; n.y = y; n.z = z;
  n.cx = center1d (p, p.Rtop, x); n.cy = center1d (p, p.Rtop, y); n.cz = center1d (p, p.Rtop, z);
  n.size = level_size (p, p.Rtop);
  n.slot = -1; n.idx = root_index (p, x, y, z);
  return n;
}

// any node at level >= Rtop by coordinates; false if its brick does not exist
B2_HD bool locate_node (const Params& p, int level, int x, int y, int z, NodePos& n)
{
  n.level = level; n.x = x; n.y = y; n.z = z;
  n.cx = center1d (p, level, x); n.cy = center1d (p, level, y); n.cz = center1d (p, level, z);
  n.size = level_size (p, level);
  if (level == p.Rtop) { n.slot = -1; n.idx = root_index (p, x, y, z); return true; }
  int t = tier_of_level (p, level);
  int k = level - tier_root_level (p, t);
  n.slot = find_brick (p, t, x >> k, y >> k, z >> k);
  n.idx = node_offset (k) + path_index (k, x, y, z);
  return n.slot >= 0;
}

// reset one node's storage to the fresh state (OctreeNode ctor, octree.h:67-74; RGBNode :177)
B2_HD void reset_node (const Params& p, const NodePos& n)
{
  *node_dw (p, n) = make_float2 (-1.f, 0.f);
  if (n.slot < 0)
  {
    if (p.root_rgb) p.root_rgb[n.idx] = make_uchar4 (0, 0, 0, 0);
    if (p.root_rgbn) p.root_rgbn[n.idx] = make_float4 (0.f, 0.f, 0.f, 0.f);
    if (p.root_M) { p.root_M[n.idx] = 0.f; p.root_ns[n.idx] = 0; }
  }
  else
  {
    size_t i = (size_t) n.slot * BRICK_NODES + n.idx;
    if (p.rgb) p.rgb[i] = make_uchar4 (0, 0, 0, 0);
    if (p.rgbn) p.rgbn[i] = make_float4 (0.f, 0.f, 0.f, 0.f);
    if (p.M) { p.M[i] = 0.f; p.ns[i] = 0; }
  }
}

// ---- RGBNormalized payload (octree.cpp:379-402) ----------------------------------------------------------------
B2_HD float4* node_rgbn (const Params& p, const NodePos& n)
{ return n.slot < 0 ? &p.root_rgbn[n.idx] : &p.rgbn[(size_t) n.slot * BRICK_NODES + n.idx]; }
// RGBNormalized::addObservation's colour part (:383-392) with w_ = the node's weight BEFORE this observation, w_new = 1.
// A black pixel gives i = 0 and r / i = NaN, which the running averages then keep: reproduced, not repaired.
B2_HD void rgbn_observe (float4& q, float w_old, uint32_t bgra)
{
  const float r = (float) ((bgra >> 16) & 0xFFu), g = (float) ((bgra >> 8) & 0xFFu), b = (float) (bgra & 0xFFu);
  const float wsum = fadd (w_old, 1.f);
  const float i = sqrtf (fadd (fadd (fmul (r, r), fmul (g, g)), fmul (b, b)));      // (exact integer below 2^24 under the root)
  const float rf = fdiv (r, i), gf = fdiv (g, i), bf = fdiv (b, i);
  q.x = fdiv (fadd (fmul (w_old, q.x), fmul (1.f, rf)), wsum);
  q.y = fdiv (fadd (fmul (w_old, q.y), fmul (1.f, gf)), wsum);
  q.z = fdiv (fadd (fmul (w_old, q.z), fmul (1.f, bf)), wsum);
  q.w = fdiv (fadd (fmul (w_old, q.w), fmul (1.f, i)), wsum);
}
// float -> uint8_t the way x86-64 compiles it (cvttss2si then a byte truncation): RGBNormalized::getRGB, octree.cpp:396-402
B2_HD unsigned char f2u8_x86 (float v)
{
  const int t = (v >= -2147483648.f && v < 2147483648.f) ? (int) v : INT_MIN;
  return (unsigned char) t;
}
// getRGB of a node of a colour volume
B2_HD uchar4 node_get_rgb (const Params& p, const NodePos& n)
{
  if (p.color_norm)
  {
    const float4 q = *node_rgbn (p, n);
    return make_uchar4 (f2u8_x86 (fmul (q.x, q.w)), f2u8_x86 (fmul (q.y, q.w)), f2u8_x86 (fmul (q.z, q.w)), 0);
  }
  return n.slot < 0 ? p.root_rgb[n.idx] : p.rgb[(size_t) n.slot * BRICK_NODES + n.idx];
}

// ---- the projective observation of a node (hpp:143-161) --------------------------------------
struct Obs
{
  bool valid;       // false -> updateVoxel returns 0 before touching the node
  bool near_;       // |d_new| < 3*getMaxSize()/4 (hpp:161)
  int u, v;
  float d_new;      // pt.z - v_g.z, unclamped
};

// reprojectPoint (tsdf_volume_octree.cpp:611-617): u = (int)(x*fx/z + cx) in DOUBLE, truncation toward
// zero.  The double divide is ~10x the cost of everything else in a node visit, so a float estimate
// is tried first and accepted only where it provably truncates to the same integer: its error is
// below 2^-24 * (3.01|x fx/z| + |cx| + |a|) < 4e-3 for |a| < 3e4, and the estimate must sit at least
// 1e-2 away from an integer (and above 0).  Otherwise the reference's double expression is evaluated.
B2_HD int project1 (const Params& p, float x, float z, double fd, double cd, float ff, float cf)
{
  if (p.fast_proj)
  {
    float a = fadd (fdiv (fmul (x, ff), z), cf);
    float fr = a - floorf (a);
    if (a > 0.01f && a < 30000.f && fr > 0.01f && fr < 0.99f) return (int) a;
  }
  return to_int_x86 (dadd (ddiv (dmul ((double) x, fd), (double) z), cd));
}

// |d_new| < 3*getMaxSize()/4. (hpp:161): the right-hand side depends on the node size only
B2_HD double near_threshold (float size)
{
  float max_size = (float) dmul (1.7320508075688772, (double) size);          // getMaxSize(), octree.cpp:68-72
  return ddiv ((double) fmul (3.f, max_size), 4.0);
}

B2_HD Obs observe_thr (const Params& p, const Frame& f, float cx, float cy, float cz, double near_thr)
{
  Obs o; o.valid = false; o.near_ = false; o.u = o.v = 0; o.d_new = 0.f;
  float vg[3];
  pcl_transform_point_f (f.tinv, cx, cy, cz, vg);                              // hpp:145
  if (vg[2] < p.min_sensor || vg[2] > p.max_sensor) return o;                  // hpp:146
  if (!(vg[2] > 0)) return o;                                                  // cpp:616
  int u = project1 (p, vg[0], vg[2], p.fx, p.cx, p.fx_f, p.cx_f);
  int v = project1 (p, vg[1], vg[2], p.fy, p.cy, p.fy_f, p.cy_f);
  if (!(u >= 0 && u < p.width && v >= 0 && v < p.height)) return o;
  float z = frame_xyz (f, u, v)[2];
  if (is_nan (z)) return o;                                                    // hpp:152
  o.valid = true; o.u = u; o.v = v;
  o.d_new = fsub (z, vg[2]);                                                   // hpp:159
  o.near_ = (double) fabsf (o.d_new) < near_thr;
  return o;
}

B2_HD Obs observe (const Params& p, const Frame& f, float cx, float cy, float cz, float size)
{ return observe_thr (p, f, cx, cy, cz, near_threshold (size)); }

// truncation + addObservation + return code (hpp:189-214, octree.cpp:152-163, :328-337) on VALUES:
// dw / c / M / ns are the node's state (in registers, shared memory or wherever the caller staged
// it).  Returns 1 / 0 / -1 like updateVoxel; `updated` says whether the state changed.
// (bgra = the PCL colour word of the observed pixel, bytes b,g,r,a; used when have_bgra)
B2_HD int leaf_update_core (const Params& p, float d_new, bool have_bgra, uint32_t bgra, float2& dw, uchar4& c, float& M, int& ns, bool& updated)
{
  updated = false;
  if (d_new > p.max_dist_pos) d_new = p.max_dist_pos;
  else if (d_new < -p.max_dist_neg) return 0;
  d_new = fdiv (d_new, p.max_dist_neg);
  const float w_new = 1.f;
  if (p.color && have_bgra)
  {
    const float cb = (float) (bgra & 0xFFu), cg = (float) ((bgra >> 8) & 0xFFu), cr = (float) ((bgra >> 16) & 0xFFu);
    float wsum = fadd (dw.y, w_new);
    c.x = (unsigned char) fdiv (fadd (fmul (dw.y, (float) c.x), fmul (w_new, cr)), wsum);   // r
    c.y = (unsigned char) fdiv (fadd (fmul (dw.y, (float) c.y), fmul (w_new, cg)), wsum);   // g
    c.z = (unsigned char) fdiv (fadd (fmul (dw.y, (float) c.z), fmul (w_new, cb)), wsum);   // b
  }
  float d_old = dw.x;
  float d = fdiv (fadd (fmul (dw.x, dw.y), fmul (d_new, w_new)), fadd (dw.y, w_new));
  float w = fadd (dw.y, w_new);
  if (w > p.max_weight) w = p.max_weight;
  dw = make_float2 (d, w);
  if (p.track_var)
  {
    M = fadd (M, fmul (fmul (w_new, fsub (d_new, d)), fsub (d_new, d_old)));
    ns = ns + 1;
  }
  updated = true;
  if ((double) d < -0.99) return 0;
  else if ((double) d < p.rc_thresh) return 1;
  else return -1;
}

B2_HD int leaf_update_values (const Params& p, const Frame& f, const Obs& o, float2& dw, uchar4& c, float& M, int& ns, bool& updated)
{
  bool have = p.color && !p.color_norm && f.rgba_off >= 0;
  uint32_t bgra = 0;
  if (have) { const unsigned char* b = frame_bgr (f, o.u, o.v); bgra = (uint32_t) b[0] | ((uint32_t) b[1] << 8) | ((uint32_t) b[2] << 16) | ((uint32_t) b[3] << 24); }
  return leaf_update_core (p, o.d_new, have, bgra, dw, c, M, ns, updated);
}

// the same on a node in global storage
B2_HD int leaf_update (const Params& p, const Frame& f, const NodePos& n, const Obs& o, bool& updated)
{
  float2* dwp = node_dw (p, n);
  float2 dw = *dwp;
  uchar4 c = make_uchar4 (0, 0, 0, 0);
  uchar4* cp = nullptr;
  if (p.color && !p.color_norm) { cp = n.slot < 0 ? &p.root_rgb[n.idx] : &p.rgb[(size_t) n.slot * BRICK_NODES + n.idx]; c = *cp; }
  float M = 0.f; int ns = 0;
  float* Mp = nullptr; int* np = nullptr;
  if (p.track_var)
  {
    Mp = n.slot < 0 ? &p.root_M[n.idx] : &p.M[(size_t) n.slot * BRICK_NODES + n.idx];
    np = n.slot < 0 ? &p.root_ns[n.idx] : &p.ns[(size_t) n.slot * BRICK_NODES + n.idx];
    M = *Mp; ns = *np;
  }
  const float w_old = dw.y;
  int rc = leaf_update_values (p, f, o, dw, c, M, ns, updated);
  if (updated)
  {
    *dwp = dw;
    if (cp) *cp = c;
    if (Mp) { *Mp = M; *np = ns; }
    if (p.color_norm && f.rgba_off >= 0)
    {
      float4* qp = node_rgbn (p, n); float4 q = *qp;
      rgbn_observe (q, w_old, *reinterpret_cast<const uint32_t*> (frame_bgr (f, o.u, o.v)));
      *qp = q;
    }
  }
  return rc;
}

struct Counters { long long n_updates, n_visits; };

// ---- updateVoxel as a depth-first recursion over the flat layout (hpp:113-218) -----------------
// This is the general path: it handles every case including prune-then-resplit (SURVEY.md §A.14).
// The brick-parallel kernels in engine.cu are the fast path for the common cases and fall back
// to this routine per subtree.
//
// split_and_expand is hpp:161-188 for a leaf that splits now: its eight children are FRESH by the
// storage invariant, so their state is known without loading it, and their observations do not
// depend on each other — all eight depth lookups are issued before any child is processed, which
// keeps the (latency-bound) general path short.
B2_HDN inline bool split_and_expand (const Params& p, const Frame& f, const NodePos& n, uint32_t* sw, uint32_t smask, Counters& cnt);

// leaf update (hpp:189-214) of a node known to be in the constructor state (octree.h:71-74): nothing is loaded
B2_HD int fresh_leaf_store (const Params& p, const Frame& f, const NodePos& n, const Obs& o, Counters& cnt)
{
  float2 dw = make_float2 (-1.f, 0.f); uchar4 c = make_uchar4 (0, 0, 0, 0); float M = 0.f; int ns = 0;
  bool updated;
  int rc = leaf_update_values (p, f, o, dw, c, M, ns, updated);
  if (updated)
  {
    cnt.n_updates++;
    *node_dw (p, n) = dw;
    if (p.color && !p.color_norm) { if (n.slot < 0) p.root_rgb[n.idx] = c; else p.rgb[(size_t) n.slot * BRICK_NODES + n.idx] = c; }
    if (p.color_norm && f.rgba_off >= 0)
    {
      float4 q = make_float4 (0.f, 0.f, 0.f, 0.f);                  // constructor state, octree.h:217-223
      rgbn_observe (q, 0.f, *reinterpret_cast<const uint32_t*> (frame_bgr (f, o.u, o.v)));
      *node_rgbn (p, n) = q;
    }
    if (p.track_var)
    {
      if (n.slot < 0) { p.root_M[n.idx] = M; p.root_ns[n.idx] = ns; }
      else { p.M[(size_t) n.slot * BRICK_NODES + n.idx] = M; p.ns[(size_t) n.slot * BRICK_NODES + n.idx] = ns; }
    }
  }
  return rc;
}

B2_HDN inline int visit_fresh_leaf (const Params& p, const Frame& f, const NodePos& n, const Obs& o, Counters& cnt)
{
  cnt.n_visits++;
  if (!o.valid) return 0;
  if (o.near_ && n.size > p.finest_size)
  {
    uint32_t smask = 0; uint32_t* sw = split_word (p, n, smask);
    if (split_and_expand (p, f, n, sw, smask, cnt)) return 1;
  }
  return fresh_leaf_store (p, f, n, o, cnt);
}

// returns true if the node stays split (some child is non-empty), false if the children were pruned again
B2_HDN inline bool split_and_expand (const Params& p, const Frame& f, const NodePos& n, uint32_t* sw, uint32_t smask, Counters& cnt)
{
  int cs = children_slot (p, n, true);
  if (cs < 0) return false;
  atomic_or32 (sw, smask);                                       // split (): children are fresh by invariant
  NodePos ch[8]; Obs oc[8];
  for (int c = 0; c < 8; ++c)
  {
    ch[c] = make_child (p, n, c, cs);
    oc[c] = observe (p, f, ch[c].cx, ch[c].cy, ch[c].cz, ch[c].size);
  }
  bool all_empty = true;
  for (int c = 0; c < 8; ++c) all_empty &= (visit_fresh_leaf (p, f, ch[c], oc[c], cnt) < 0);
  if (!all_empty) return true;
  atomic_and32 (sw, ~smask);                                     // children.clear ()
  for (int c = 0; c < 8; ++c) reset_node (p, ch[c]);
  return false;
}

// ---- the same visit of a FRESH subtree, breadth first and cooperative --------------------------------------------
// A node whose pre-existing children were pruned is visited as a leaf and may split again (SURVEY.md A.14); everything
// below it is then in the constructor state and the visit is a pure function of the frame.  The depth-first routine
// above makes one lane walk the whole subtree; this one keeps the subtree as an array of records (creation order =
// breadth first, a node's eight children adjacent) so that `nlanes` lanes visit a whole level together, then folds
// the return codes level by level from the bottom.  Nodes that do not fit in the record array are walked depth
// first by the lane that reached them.  The result (tree, values, counters) is identical to the recursion's.
struct FreshRec { NodePos n; float dnew; int uv; short first; signed char rc; unsigned char state; };
enum { FR_LEAF = 0, FR_INTERNAL = 1 };
struct CoopSingle { B2_HD int lane () const { return 0; } B2_HD int nlanes () const { return 1; } B2_HD void sync () const {} };

B2_HD int atomic_add_int (int* a, int v)
{
#ifdef __CUDA_ARCH__
  return atomicAdd (a, v);
#else
  int o = *a; *a = o + v; return o;
#endif
}

// n has just been split (split bit set, children storage cs, all fresh).  rec: cap records (cap a multiple of 8, >= 8),
// counter: one int, both shared by the cooperating lanes.  Returns true if some child is non-empty (n stays split);
// otherwise the caller clears n's children (rec[0..7].n) and updates n as a leaf.
template <typename Coop>
B2_HDN inline bool fresh_children_bfs (const Params& p, const Frame& f, const NodePos& n, int cs, FreshRec* rec, int cap, int* counter,
                                       const Coop& co, Counters& cnt)
{
  const int lane = co.lane (), nl = co.nlanes ();
  for (int c = lane; c < 8; c += nl) rec[c].n = make_child (p, n, c, cs);
  int lev_lo[24]; int nlev = 0;
  int lo = 0, hi = 8;
  co.sync ();
  while (lo < hi)
  {
    lev_lo[nlev++] = lo;
    if (lane == 0) *counter = hi;
    co.sync ();
    for (int i = lo + lane; i < hi; i += nl)
    {
      const NodePos q = rec[i].n;
      cnt.n_visits++;
      const Obs o = observe (p, f, q.cx, q.cy, q.cz, q.size);
      int rc = 0; unsigned char st = FR_LEAF;
      if (o.valid)
      {
        bool handled = false;
        if (o.near_ && q.size > p.finest_size)
        {
          const int cs2 = children_slot (p, q, true);
          if (cs2 >= 0)
          {
            const int base = atomic_add_int (counter, 8);
            if (base + 8 <= cap)
            {
              uint32_t m = 0; uint32_t* sw = split_word (p, q, m);
              atomic_or32 (sw, m);                                     // split (): the children are fresh by invariant
              for (int c = 0; c < 8; ++c) rec[base + c].n = make_child (p, q, c, cs2);
              st = FR_INTERNAL; rec[i].first = (short) base; rec[i].dnew = o.d_new; rec[i].uv = o.u | (o.v << 16);
            }
            else
            {
              cnt.n_visits--;                                          // visit_fresh_leaf counts the node itself
              rc = visit_fresh_leaf (p, f, q, o, cnt);                 // no room for its children: depth first from here
            }
            handled = true;
          }
        }
        if (!handled) rc = fresh_leaf_store (p, f, q, o, cnt);
      }
      rec[i].rc = (signed char) rc; rec[i].state = st;
    }
    co.sync ();
    const int total = *counter;
    const int room = hi + ((cap - hi) / 8) * 8;                        // allocations beyond the array were refused
    lo = hi;
    hi = total < room ? total : room;
    co.sync ();
  }
  const int end = lo;
  for (int L = nlev - 1; L >= 0; --L)                                  // hpp:176-188 + fall-through, deepest level first
  {
    const int a = lev_lo[L], b = (L + 1 < nlev) ? lev_lo[L + 1] : end;
    for (int i = a + lane; i < b; i += nl)
    {
      if (rec[i].state != FR_INTERNAL) continue;
      const int first = rec[i].first;
      bool any = false;
      for (int c = 0; c < 8; ++c) any |= rec[first + c].rc >= 0;
      if (any) { rec[i].rc = 1; continue; }
      const NodePos q = rec[i].n;
      uint32_t m = 0; uint32_t* sw = split_word (p, q, m);
      atomic_and32 (sw, ~m);                                           // children.clear ()
      for (int c = 0; c < 8; ++c) reset_node (p, rec[first + c].n);
      Obs o; o.valid = true; o.near_ = true; o.d_new = rec[i].dnew; o.u = rec[i].uv & 0xFFFF; o.v = rec[i].uv >> 16;
      rec[i].rc = (signed char) fresh_leaf_store (p, f, q, o, cnt);
    }
    co.sync ();
  }
  bool any = false;
  for (int c = 0; c < 8; ++c) any |= rec[c].rc >= 0;
  return any;
}

#if defined(B2_EMU_BFS) && !defined(__CUDACC__)
extern int b2_emu_bfs_cap;               // tests/emu/emu.cpp: record capacity for the host emulation (0 = recursion only)
#endif

B2_HDN inline int update_voxel_dfs (const Params& p, const Frame& f, const NodePos& n, Counters& cnt)
{
  cnt.n_visits++;
  uint32_t smask = 0; uint32_t* sw = nullptr;
  if (n.level < p.L) sw = split_word (p, n, smask);
  if (sw && (*sw & smask))                                       // hpp:122-142
  {
    int cs = children_slot (p, n, false);
    if (cs < 0) { raise_err (p, ERR_MISSING_BRICK); return 0; }
    bool all_empty = true;
    for (int c = 0; c < 8; ++c)
      all_empty &= (update_voxel_dfs (p, f, make_child (p, n, c, cs), cnt) < 0);
    if (!all_empty) return 1;
    atomic_and32 (sw, ~smask);                                   // children.clear ()
    for (int c = 0; c < 8; ++c) reset_node (p, make_child (p, n, c, cs));
  }
  Obs o = observe (p, f, n.cx, n.cy, n.cz, n.size);
  if (!o.valid) return 0;
  if (o.near_ && n.size > p.finest_size)                         // hpp:161-188
  {
#if defined(B2_EMU_BFS) && !defined(__CUDACC__)
    if (b2_emu_bfs_cap >= 8)
    {
      // host emulation of the cooperative routine (one "lane"): every split in the emulated frame goes through it
      static thread_local FreshRec recs[1024];
      int cs = children_slot (p, n, true), counter = 0;
      if (cs >= 0)
      {
        atomic_or32 (sw, smask);
        if (fresh_children_bfs (p, f, n, cs, recs, b2_emu_bfs_cap, &counter, CoopSingle (), cnt)) return 1;
        atomic_and32 (sw, ~smask);
        for (int c = 0; c < 8; ++c) reset_node (p, recs[c].n);
      }
    }
    else
#endif
    if (split_and_expand (p, f, n, sw, smask, cnt)) return 1;
  }
  bool updated;
  int rc = leaf_update (p, f, n, o, updated);
  if (updated) cnt.n_updates++;
  return rc;
}

// ---- pre-split (hpp:56-90): make the finest voxel containing a surface sample exist -------------
// Sets the split bit of every ancestor (levels C..L-1) of the finest voxel containing the world
// point.  Returns false if the point is outside the volume (octree.cpp:631).
B2_HD bool world_to_finest (const Params& p, float x, float y, float z, int& fx_, int& fy_, int& fz_)
{
  if (is_nan (z) || fabsf (x) > p.half || fabsf (y) > p.half || fabsf (z) > p.half) return false;
  float cx = 0.f, cy = 0.f, cz = 0.f, off = p.size * 0.25f;
  int ix = 0, iy = 0, iz = 0;
  for (int l = 0; l < p.L; ++l)                                  // OctreeNode::getContainingVoxel, octree.cpp:119
  {
    int bx = fsub (x, cx) > 0, by = fsub (y, cy) > 0, bz = fsub (z, cz) > 0;
    ix = 2 * ix + bx; iy = 2 * iy + by; iz = 2 * iz + bz;
    cx = bx ? fadd (cx, off) : fsub (cx, off);
    cy = by ? fadd (cy, off) : fsub (cy, off);
    cz = bz ? fadd (cz, off) : fsub (cz, off);
    off *= 0.5f;
  }
  fx_ = ix; fy_ = iy; fz_ = iz;
  return true;
}

// coarse-cell ownership for multi-GPU sharding (SURVEY.md §8e): whole refinement pyramids stay on one device
B2_HD bool owns_cell (const Params& p, int cx, int cy, int cz)
{
  if (p.shard_count <= 1) return true;
  uint32_t h = hash_key (((uint64_t) cx << 40) | ((uint64_t) cy << 20) | (uint64_t) cz);
  return (int) (h % (uint32_t) p.shard_count) == p.shard_rank;
}

B2_HD void presplit_point (const Params& p, int fx_, int fy_, int fz_)
{
  // root array node (level Rtop) if it is a coarse-or-deeper level
  if (p.Rtop >= p.C)
  {
    int sh = p.L - p.Rtop;
    int ri = root_index (p, fx_ >> sh, fy_ >> sh, fz_ >> sh);
    uint32_t m = 1u << (ri & 31);
    if (!(p.root_split[ri >> 5] & m)) atomic_or32 (&p.root_split[ri >> 5], m);
  }
  for (int t = p.T - 1; t >= 0; --t)
  {
    int R = tier_root_level (p, t);
    int sh = p.L - R;
    int slot = find_or_insert_brick (p, t, fx_ >> sh, fy_ >> sh, fz_ >> sh);
    if (slot < 0) return;
    uint32_t* sw = &p.split[(size_t) slot * BRICK_SPLIT_WORDS];
    for (int k = 1; k <= 3; ++k)
    {
      int level = R + k;
      if (level < p.C || level >= p.L) continue;
      int s2 = p.L - level;
      int j = path_index (k, fx_ >> s2, fy_ >> s2, fz_ >> s2);
      uint32_t m = 1u << (j & 31);
      uint32_t* w = sw + split_word_base (k) + (j >> 5);
      if (!(*w & m)) atomic_or32 (w, m);
    }
  }
}

// ---- getContainingVoxel over the flat layout (octree.cpp:112-121, :628-634) --------------------
struct Leaf { bool found; NodePos n; float d, w; };

B2_HD Leaf find_leaf_impl (const Params& p, float x, float y, float z)
{
  Leaf lf; lf.found = false;
  if (is_nan (z) || fabsf (x) > p.half || fabsf (y) > p.half || fabsf (z) > p.half) return lf;
  NodePos n;
  n.level = 0; n.x = n.y = n.z = 0; n.cx = n.cy = n.cz = 0.f; n.size = p.size; n.slot = -1; n.idx = 0;
  // levels above Rtop have no storage; descend arithmetically
  while (n.level < p.Rtop)
  {
    int bx = fsub (x, n.cx) > 0, by = fsub (y, n.cy) > 0, bz = fsub (z, n.cz) > 0;
    float off = n.size * 0.25f;
    n.x = 2 * n.x + bx; n.y = 2 * n.y + by; n.z = 2 * n.z + bz;
    n.cx = bx ? fadd (n.cx, off) : fsub (n.cx, off);
    n.cy = by ? fadd (n.cy, off) : fsub (n.cy, off);
    n.cz = bz ? fadd (n.cz, off) : fsub (n.cz, off);
    n.size *= 0.5f; n.level++;
  }
  n.slot = -1; n.idx = root_index (p, n.x, n.y, n.z);
  for (;;)
  {
    if (!is_split (p, n)) break;
    int cs = children_slot (p, n, false);
    if (cs < 0) break;            // cannot happen when the invariant holds
    int c = ((fsub (x, n.cx) > 0) << 2) | ((fsub (y, n.cy) > 0) << 1) | (int) (fsub (z, n.cz) > 0);
    n = make_child (p, n, c, cs);
  }
  float2 dw = *node_dw (p, n);
  lf.found = true; lf.n = n; lf.d = dw.x; lf.w = dw.y;
  return lf;
}

// On the device the descent is ONE out-of-line routine: renderView / queries / marching cubes call it ~70
// times per item, and inlining every call made those kernels ~40k instructions (instruction-cache bound).
// Callers stage Params in shared memory so the reference they pass does not force a local copy.
#ifdef __CUDA_ARCH__
__device__ __noinline__ void find_leaf_out (const Params& p, float x, float y, float z, Leaf* out) { *out = find_leaf_impl (p, x, y, z); }
B2_HD Leaf find_leaf (const Params& p, float x, float y, float z) { Leaf l; find_leaf_out (p, x, y, z, &l); return l; }
#else
B2_HD Leaf find_leaf (const Params& p, float x, float y, float z) { return find_leaf_impl (p, x, y, z); }
#endif

// ---- getVoxelCenter / getVoxelIndex (tsdf_volume_octree.cpp:553-574) ----------------------------
B2_HD float voxel_center1 (const Params& p, long long i)
{ return (float) (dadd (ddiv (dmul ((double) i + 0.5, p.dsize), p.dres), -(double) p.voff)); }
B2_HD int voxel_index1 (const Params& p, float x)
{ return to_int_x86 (floor (dmul (ddiv (dadd ((double) x, ddiv (p.dsize, 2.0)), p.dsize), p.dres))); }
B2_HD bool voxel_index (const Params& p, float x, float y, float z, int& xi, int& yi, int& zi)
{
  xi = voxel_index1 (p, x); yi = voxel_index1 (p, y); zi = voxel_index1 (p, z);
  return xi >= 0 && yi >= 0 && zi >= 0 && xi < p.res && yi < p.res && zi < p.res;
}

// ---- interpolateTrilinearly (tsdf_volume_octree.cpp:486-541) -------------------------------------
B2_HD float interpolate_trilinearly (const Params& p, float x, float y, float z, bool* valid)
{
  int xi, yi, zi;
  bool exists = voxel_index (p, x, y, z, xi, yi, zi);
  if (!exists || xi <= 0 || xi >= p.res - 1 || yi <= 0 || yi >= p.res - 1 || zi <= 0 || zi >= p.res - 1)
  {
    if (valid) *valid = false;
    return nanf ("");
  }
  if (x < voxel_center1 (p, xi)) xi -= 1;
  if (y < voxel_center1 (p, yi)) yi -= 1;
  if (z < voxel_center1 (p, zi)) zi -= 1;
  float vx = voxel_center1 (p, xi), vy = voxel_center1 (p, yi), vz = voxel_center1 (p, zi);
  float vx1 = voxel_center1 (p, xi + 1), vy1 = voxel_center1 (p, yi + 1), vz1 = voxel_center1 (p, zi + 1);
  float a = fdiv (fmul (fsub (x, vx), (float) p.res), p.size);
  float b = fdiv (fmul (fsub (y, vy), (float) p.res), p.size);
  float c = fdiv (fmul (fsub (z, vz), (float) p.res), p.size);
  Leaf o   = find_leaf (p, vx,  vy,  vz),  ox  = find_leaf (p, vx1, vy,  vz);
  Leaf oy  = find_leaf (p, vx,  vy1, vz),  oz  = find_leaf (p, vx,  vy,  vz1);
  Leaf oxy = find_leaf (p, vx1, vy1, vz),  oxz = find_leaf (p, vx1, vy,  vz1);
  Leaf oyz = find_leaf (p, vx,  vy1, vz1), oxyz = find_leaf (p, vx1, vy1, vz1);
  if (valid)
    *valid = *valid && (o.w > 0) && (ox.w > 0) && (oy.w > 0) && (oz.w > 0) && (oxy.w > 0) && (oxz.w > 0) && (oyz.w > 0) && (oxyz.w > 0);
  float ia = fsub (1.f, a), ib = fsub (1.f, b), ic = fsub (1.f, c);
  float s = fmul (fmul (fmul (o.d, ia), ib), ic);
  s = fadd (s, fmul (fmul (fmul (oz.d, ia), ib), c));
  s = fadd (s, fmul (fmul (fmul (oy.d, ia), b), ic));
  s = fadd (s, fmul (fmul (fmul (oyz.d, ia), b), c));
  s = fadd (s, fmul (fmul (fmul (ox.d, a), ib), ic));
  s = fadd (s, fmul (fmul (fmul (oxz.d, a), ib), c));
  s = fadd (s, fmul (fmul (fmul (oxy.d, a), b), ic));
  s = fadd (s, fmul (fmul (fmul (oxyz.d, a), b), c));
  return s;
}

// ---- getNeighbors + getFxn/getGradient/getHessian (tsdf_volume_octree.cpp:655-828) ----------------
B2_HD int sgn (float x) { return x > 0 ? 1 : -1; }

B2_HD bool query_point (const Params& p, const float* pt, int mode, float* val, float* grad, float* hess)
{
  int xi, yi, zi;
  if (!voxel_index (p, pt[0], pt[1], pt[2], xi, yi, zi)) return false;
  if (pt[0] < voxel_center1 (p, xi)) xi -= 1;
  if (pt[1] < voxel_center1 (p, yi)) yi -= 1;
  if (pt[2] < voxel_center1 (p, zi)) zi -= 1;
  if (xi < 0 || xi >= p.res - 1 || yi < 0 || yi >= p.res - 1 || zi < 0 || zi >= p.res - 1) return false;
  float c = p.finest_size;                 // xsize_ / xres_
  float fv = 0.f, g0 = 0.f, g1 = 0.f, g2 = 0.f, h01 = 0.f, h02 = 0.f, h12 = 0.f;
  for (int dx = 0; dx <= 1; dx++)
    for (int dy = 0; dy <= 1; dy++)
      for (int dz = 0; dz <= 1; dz++)
      {
        float fx_ = voxel_center1 (p, xi + dx), fy_ = voxel_center1 (p, yi + dy), fz_ = voxel_center1 (p, zi + dz);
        Leaf lf = find_leaf (p, fx_, fy_, fz_);
        if (!lf.found) return false;
        float vx = mode ? fx_ : lf.n.cx, vy = mode ? fy_ : lf.n.cy, vz = mode ? fz_ : lf.n.cz;
        // unqualified fabs() in the reference is the C double version: the factors and products are
        // DOUBLE, only the `+=` rounds to float (cpp:668, 694-696, 716-718; DESIGN.md "Arithmetic conventions")
        const double dc = (double) c, dd = (double) lf.d;
        double ax = dadd (dc, -fabs ((double) fsub (pt[0], vx))), ay = dadd (dc, -fabs ((double) fsub (pt[1], vy))), az = dadd (dc, -fabs ((double) fsub (pt[2], vz)));
        double sx = (double) -sgn (fsub (pt[0], vx)), sy = (double) -sgn (fsub (pt[1], vy)), sz = (double) -sgn (fsub (pt[2], vz));
        fv = (float) dadd ((double) fv, dmul (dmul (dmul (ax, ay), az), dd));
        g0 = (float) dadd ((double) g0, dmul (dmul (dmul (sx, ay), az), dd));
        g1 = (float) dadd ((double) g1, dmul (dmul (dmul (ax, sy), az), dd));
        g2 = (float) dadd ((double) g2, dmul (dmul (dmul (ax, ay), sz), dd));
        double bx = dadd (dc, -fabs ((double) fsub (pt[0], fx_))), by = dadd (dc, -fabs ((double) fsub (pt[1], fy_))), bz = dadd (dc, -fabs ((double) fsub (pt[2], fz_)));
        int tx = sgn (fsub (pt[0], fx_)), ty = sgn (fsub (pt[1], fy_)), tz = sgn (fsub (pt[2], fz_));
        h01 = (float) dadd ((double) h01, dmul (dmul ((double) (tx * ty), bz), dd));
        h02 = (float) dadd ((double) h02, dmul (dmul (dmul ((double) tx, by), (double) tz), dd));
        h12 = (float) dadd ((double) h12, dmul (dmul (dmul (bx, (double) ty), (double) tz), dd));
      }
  float c3 = fmul (fmul (c, c), c);
  if (val) *val = fdiv (fv, c3);
  if (grad) { grad[0] = fdiv (g0, c3); grad[1] = fdiv (g1, c3); grad[2] = fdiv (g2, c3); }
  if (hess)
  {
    for (int k = 0; k < 9; ++k) hess[k] = 0.f;
    hess[1] = fdiv (h01, c3); hess[2] = fdiv (h02, c3); hess[5] = fdiv (h12, c3);
    hess[3] = hess[1]; hess[6] = hess[2]; hess[7] = hess[5];
  }
  return true;
}

// ---- renderView, one pixel (tsdf_volume_octree.cpp:278-424) ---------------------------------------
struct RenderParams
{
  int width, height;            // image_width_/ds, image_height_/ds
  double fx, fy, cx, cy;        // intrinsics / ds
  float rot[12];                // trans.rotation().cast<float>() in [0..2],[4..6],[8..10]; translation in [3],[7],[11]
  double inv[12];               // trans.inverse() rows 0..2 (double), for transformPointCloudWithNormals
  float tfwd[12];               // trans.cast<float>() (renderColoredView, cpp:443)
  float min_step;               // max_dist_neg_ * 3/4.
  float half_voxel;             // (zsize_/zres_)/2.
};

// out_p / out_n: camera-frame point and normal (PointNormal xyz / normal_xyz); rgb optional
B2_HD void render_pixel (const Params& p, const RenderParams& r, int x, int y, float* out_p, float* out_n, unsigned char* rgb)
{
  const float qnan = nanf ("");
  float P[3] = { 0.f, 0.f, 0.f }, N[3] = { 0.f, 0.f, 0.f };
  bool have_point = false;
  float du[3] = { (float) ddiv (dadd ((double) x, -r.cx), r.fx), (float) ddiv (dadd ((double) y, -r.cy), r.fy), 1.f };
  normalize3 (du);
  { float t[3]; linear_mul_f (r.rot, du[0], du[1], du[2], t); du[0] = t[0]; du[1] = t[1]; du[2] = t[2]; }
  const float org[3] = { r.rot[3], r.rot[7], r.rot[11] };
  float pos[3] = { org[0], org[1], org[2] };
  float d = 0.f, w = 0.f, last_w = 0.f, last_d = 0.f;
  float t = p.min_sensor;
  for (int k = 0; k < 3; ++k) pos[k] = fadd (pos[k], fmul (t, du[k]));
  float step = r.min_step;
  bool hit_voxel = false, found_crossing = false;
  while (t < p.max_sensor)
  {
    Leaf lf = find_leaf (p, pos[0], pos[1], pos[2]);
    if (lf.found)
    {
      hit_voxel = true;
      d = lf.d; w = lf.w;
      if (((d < 0 && last_d > 0) || (d > 0 && last_d < 0)) && last_w != 0.f && w != 0.f)
      {
        found_crossing = true;
        float old_t = fsub (t, step);
        step = r.half_voxel;
        float new_d, new_w;
        float last_new_d = d, last_new_w = w;
        while (t >= old_t)
        {
          t = fsub (t, step);
          for (int k = 0; k < 3; ++k) pos[k] = fsub (pos[k], fmul (step, du[k]));
          Leaf l2 = find_leaf (p, pos[0], pos[1], pos[2]);
          if (!l2.found) break;
          new_d = l2.d; new_w = l2.w;
          if ((last_d > 0 && new_d > 0) || (last_d < 0 && new_d < 0))
          {
            last_d = new_d; last_w = new_w;
            d = last_new_d; w = last_new_w;
            t = fadd (t, step);
            for (int k = 0; k < 3; ++k) pos[k] = fadd (pos[k], fmul (step, du[k]));
            break;
          }
          last_new_d = d; last_new_w = w;
        }
        break;
      }
      last_d = d; last_w = w;
      float s1 = lf.n.size * 0.25f;                       // (float)voxel->getMinSize () / 4.f
      float s2 = fmul (fabsf (d), p.max_dist_neg);
      step = s1 < s2 ? s2 : s1;                           // std::max (a, b) = (a < b) ? b : a
    }
    else if (hit_voxel) break;
    t = fadd (t, step);
    for (int k = 0; k < 3; ++k) pos[k] = fadd (pos[k], fmul (step, du[k]));
  }
  if (!found_crossing) { P[0] = P[1] = P[2] = qnan; }
  else
  {
    bool has_data = true;
    float tcurr = t, tprev = fsub (t, step);
    last_d = interpolate_trilinearly (p, fadd (org[0], fmul (tprev, du[0])), fadd (org[1], fmul (tprev, du[1])), fadd (org[2], fmul (tprev, du[2])), &has_data);
    d = interpolate_trilinearly (p, fadd (org[0], fmul (tcurr, du[0])), fadd (org[1], fmul (tcurr, du[1])), fadd (org[2], fmul (tcurr, du[2])), &has_data);
    // cpp:389 — fabs() is the C double version: the right-hand side is evaluated in double, rounded once
    float t_star = (float) dadd ((double) t, dmul ((double) step, dadd (-1.0, fabs ((double) fdiv (last_d, fsub (last_d, d))))));
    P[0] = fadd (org[0], fmul (t_star, du[0])); P[1] = fadd (org[1], fmul (t_star, du[1])); P[2] = fadd (org[2], fmul (t_star, du[2]));
    have_point = true;
    Leaf lf = find_leaf (p, P[0], P[1], P[2]);
    if (!lf.found) { N[0] = N[1] = N[2] = qnan; }
    else
    {
      float size = lf.n.size;
      bool valid = true;
      float d_xm = interpolate_trilinearly (p, fsub (P[0], size), P[1], P[2], &valid);
      float d_xp = interpolate_trilinearly (p, fadd (P[0], size), P[1], P[2], &valid);
      float d_ym = interpolate_trilinearly (p, P[0], fsub (P[1], size), P[2], &valid);
      float d_yp = interpolate_trilinearly (p, P[0], fadd (P[1], size), P[2], &valid);
      float d_zm = interpolate_trilinearly (p, P[0], P[1], fsub (P[2], size), &valid);
      float d_zp = interpolate_trilinearly (p, P[0], P[1], fadd (P[2], size), &valid);
      if (!valid) { N[0] = N[1] = N[2] = qnan; }
      else
      {
        float two = fmul (2.f, size);
        N[0] = fdiv (fmul (fsub (d_xp, d_xm), p.max_dist_neg), two);
        N[1] = fdiv (fmul (fsub (d_yp, d_ym), p.max_dist_neg), two);
        N[2] = fdiv (fmul (fsub (d_zp, d_zm), p.max_dist_neg), two);
        normalize3 (N);
      }
    }
  }
  (void) have_point;
  if (rgb) { rgb[0] = rgb[1] = rgb[2] = 0; }
  // pcl::transformPointCloudWithNormals (cloud, cloud, trans.inverse ()) for a non-dense cloud (cpp:422)
  bool finite = isfinite (P[0]) && isfinite (P[1]) && isfinite (P[2]);
  if (finite)
  {
    const double* m = r.inv;
    double p0 = P[0], p1 = P[1], p2 = P[2], n0 = N[0], n1 = N[1], n2 = N[2];
    float q[3], nn[3];
    q[0] = (float) dadd (dadd (dadd (dmul (m[0], p0), dmul (m[1], p1)), dmul (m[2],  p2)), m[3]);
    q[1] = (float) dadd (dadd (dadd (dmul (m[4], p0), dmul (m[5], p1)), dmul (m[6],  p2)), m[7]);
    q[2] = (float) dadd (dadd (dadd (dmul (m[8], p0), dmul (m[9], p1)), dmul (m[10], p2)), m[11]);
    nn[0] = (float) dadd (dadd (dmul (m[0], n0), dmul (m[1], n1)), dmul (m[2],  n2));
    nn[1] = (float) dadd (dadd (dmul (m[4], n0), dmul (m[5], n1)), dmul (m[6],  n2));
    nn[2] = (float) dadd (dadd (dmul (m[8], n0), dmul (m[9], n1)), dmul (m[10], n2));
    P[0] = q[0]; P[1] = q[1]; P[2] = q[2]; N[0] = nn[0]; N[1] = nn[1]; N[2] = nn[2];
    if (rgb)                                               // renderColoredView, cpp:436-448
    {
      float vt[3];
      affine_mul_f (r.tfwd, P[0], P[1], P[2], vt);
      Leaf lf = find_leaf (p, vt[0], vt[1], vt[2]);
      if (lf.found)
      {
        if (p.color)
        {
          uchar4 c = node_get_rgb (p, lf.n);
          rgb[0] = c.x; rgb[1] = c.y; rgb[2] = c.z;
        }
        else rgb[0] = rgb[1] = rgb[2] = 127;               // OctreeNode::getRGB, octree.cpp:173-178
      }
    }
  }
  out_p[0] = P[0]; out_p[1] = P[1]; out_p[2] = P[2];
  out_n[0] = N[0]; out_n[1] = N[1]; out_n[2] = N[2];
}

// ---- marching cubes for one leaf (marching_cubes_tsdf_octree.cpp:91-106, :145-236 + pcl createSurface) ----
struct McParams
{
  float w_min;
  int color_mode;               // 0 none, 1 rgb, 2 confidence
  float lower[3], size_voxel[3];// pcl::MarchingCubes lower_boundary_, size_voxel_ (set by setInputTSDF, cpp:43-83)
  double gt[12];                // global transform rows 0..2
};

// Position of a leaf in the reference's mesh order.  performReconstruction walks the octree depth first with the
// children in index order (octree.cpp:257-264: x is the high bit, then y, then z), one cube per leaf, so leaves come
// out sorted by the bit-interleaved finest-level coordinates of their first voxel; a cube's triangles follow in
// table order (key << 3 | triangle).
B2_HD unsigned long long mc_order_key (const Params& p, const NodePos& n)
{
  const int sh = p.L - n.level;
  const unsigned X = (unsigned) n.x << sh, Y = (unsigned) n.y << sh, Z = (unsigned) n.z << sh;
  unsigned long long k = 0;
  for (int l = p.L - 1; l >= 0; --l) k = (k << 3) | (((X >> l) & 1u) << 2) | (((Y >> l) & 1u) << 1) | ((Z >> l) & 1u);
  return k;
}

// ---- Octree::getLeaves (octree.cpp:99-109, 608-617) -----------------------------------------------
// The nodes getLeaves returns never contain one another, so the order of its depth-first walk is the order of
// mc_order_key.  The level sits in the low LEAF_LEVEL_BITS bits so that a key alone gives the node back (levels 0..19
// need 5 bits): 3L + 5 significant bits.
constexpr int LEAF_LEVEL_BITS = 5;
B2_HD unsigned long long leaf_key (const Params& p, int level, int x, int y, int z)
{
  NodePos n; n.level = level; n.x = x; n.y = y; n.z = z;
  return (mc_order_key (p, n) << LEAF_LEVEL_BITS) | (unsigned long long) level;
}
B2_HD void leaf_decode (const Params& p, unsigned long long key, int& level, int& x, int& y, int& z)
{
  level = (int) (key & ((1u << LEAF_LEVEL_BITS) - 1));
  const unsigned long long m = key >> LEAF_LEVEL_BITS;
  unsigned X = 0, Y = 0, Z = 0;
  for (int l = 0; l < p.L; ++l)
  {
    X |= (unsigned) ((m >> (3 * l + 2)) & 1u) << l; Y |= (unsigned) ((m >> (3 * l + 1)) & 1u) << l; Z |= (unsigned) ((m >> (3 * l)) & 1u) << l;
  }
  x = (int) (X >> (p.L - level)); y = (int) (Y >> (p.L - level)); z = (int) (Z >> (p.L - level));
}
// Whether the walk of getLeaves (leaves, nlevels) returns an existing node at level >= 1: a child is pushed when it has no
// children or when the level budget (nlevels - level) has reached 0; a negative budget never does.
B2_HD bool leaf_emitted (int level, bool split, int nlevels)
{
  return nlevels < 0 ? !split : (level <= nlevels && (!split || level == nlevels));
}
// getOccupiedVoxelIndices (tsdf_volume_octree.cpp:598-601): w > 0 && fabs (d) < 1, fabs being the double one
B2_HD bool leaf_occupied (float d, float w) { return w > 0 && fabs ((double) d) < 1; }

// getGridValue (cpp:91-106)
B2_HD float mc_grid_value (const Params& p, const McParams& mc, int x, int y, int z)
{
  Leaf lf = find_leaf (p, voxel_center1 (p, x), voxel_center1 (p, y), voxel_center1 (p, z));
  if (!lf.found || lf.w < mc.w_min || fabsf (lf.d) >= 1.f) return nanf ("");
  return fmul (lf.d, p.max_dist_neg);
}

// Evaluates the cube anchored at leaf `n` (state d,w).  Returns the number of triangles and, if
// verts != nullptr, writes 9 floats per triangle (global transform applied) and 3 colour bytes
// per vertex.  edge/tri tables are passed in so host and device can each use their own copy.
B2_HD int mc_leaf (const Params& p, const McParams& mc, const NodePos& n, float d, float w,
                   const unsigned short* edge_table, const signed char (*tri_table)[16],
                   float* verts, unsigned char* cols)
{
  if (!(w >= mc.w_min && fabsf (d) < 1.f)) return 0;                           // cpp:190
  int idx[3];
  voxel_index (p, n.cx, n.cy, n.cz, idx[0], idx[1], idx[2]);                   // cpp:195
  if (idx[0] <= 0 || idx[0] >= p.res - 1 || idx[1] <= 0 || idx[1] >= p.res - 1 || idx[2] <= 0 || idx[2] >= p.res - 1) return 0;
  const int o[8][3] = { {0,0,0}, {1,0,0}, {1,0,1}, {0,0,1}, {0,1,0}, {1,1,0}, {1,1,1}, {0,1,1} };
  float leaf[8];
  int cubeindex = 0;
  for (int k = 0; k < 8; ++k)                                                  // getValidNeighborList1D, cpp:145-177
  {
    leaf[k] = mc_grid_value (p, mc, idx[0] + o[k][0], idx[1] + o[k][1], idx[2] + o[k][2]);
    if (is_nan (leaf[k])) return 0;
    if (leaf[k] < 0.f) cubeindex |= (1 << k);
  }
  unsigned short em = edge_table[cubeindex];
  if (em == 0) return 0;
  int ntri = 0;
  while (ntri < 5 && tri_table[cubeindex][3 * ntri] != -1) ++ntri;
  if (!verts) return ntri;
  float center[3], pc[8][3];
  for (int k = 0; k < 3; ++k) center[k] = fadd (mc.lower[k], fmul (mc.size_voxel[k], (float) idx[k]));
  for (int i = 0; i < 8; ++i)
  {
    pc[i][0] = center[0]; pc[i][1] = center[1]; pc[i][2] = center[2];
    if (i & 0x4) pc[i][1] = fadd (center[1], mc.size_voxel[1]);
    if (i & 0x2) pc[i][2] = fadd (center[2], mc.size_voxel[2]);
    if ((i & 0x1) ^ ((i >> 1) & 0x1)) pc[i][0] = fadd (center[0], mc.size_voxel[0]);
  }
  const int ec[12][2] = { {0,1}, {1,2}, {2,3}, {3,0}, {4,5}, {5,6}, {6,7}, {7,4}, {0,4}, {1,5}, {2,6}, {3,7} };
  unsigned char cr = 0, cg = 0, cb = 0;
  if (mc.color_mode == 2)
  {
    double sd = (100. - (double) w) / 100.;
    double rr = (1 - sd) * 255., bb = sd * 255.;
    rr = rr < 255. ? rr : 255.; rr = rr > 0. ? rr : 0.;
    bb = bb < 255. ? bb : 255.; bb = bb > 0. ? bb : 0.;
    cr = (unsigned char) rr; cb = (unsigned char) bb;
  }
  else if (mc.color_mode == 1 && p.color)
  {
    uchar4 c = node_get_rgb (p, n);
    cr = c.x; cg = c.y; cb = c.z;
  }
  for (int i = 0; i < 3 * ntri; ++i)
  {
    int e = tri_table[cubeindex][i];
    int a = ec[e][0], b = ec[e][1];
    float mu = fdiv (fsub (0.f, leaf[a]), fsub (leaf[b], leaf[a]));          // interpolateEdge, iso level 0
    float q[3];
    for (int k = 0; k < 3; ++k) q[k] = fadd (pc[a][k], fmul (mu, fsub (pc[b][k], pc[a][k])));
    const double* m = mc.gt;                                                   // transformPointCloud (dense, double)
    double p0 = q[0], p1 = q[1], p2 = q[2];
    verts[3 * i + 0] = (float) dadd (dadd (dadd (dmul (m[0], p0), dmul (m[1], p1)), dmul (m[2],  p2)), m[3]);
    verts[3 * i + 1] = (float) dadd (dadd (dadd (dmul (m[4], p0), dmul (m[5], p1)), dmul (m[6],  p2)), m[7]);
    verts[3 * i + 2] = (float) dadd (dadd (dadd (dmul (m[8], p0), dmul (m[9], p1)), dmul (m[10], p2)), m[11]);
    if (cols) { cols[3 * i] = cr; cols[3 * i + 1] = cg; cols[3 * i + 2] = cb; }
  }
  return ntri;
}

} // namespace b2
