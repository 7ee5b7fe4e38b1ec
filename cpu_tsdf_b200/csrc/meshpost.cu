// meshpost.cu — flattenVertices / cleanupMesh of the reference's `integrate` program on the GPU
// (src/prog/integrate.cpp:103-214; SURVEY.md §8(f) row 3).  Part of libb200tsdf.so; see
// meshpost_core.cuh for the formulation.  Ordered compaction uses cub::DeviceScan (CUDA toolkit).
#include "../../include/b200tsdf.h"
#include "meshpost_core.cuh"

#include "mesh_sort.h"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda_runtime.h>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace b2;

namespace {

thread_local std::string g_meshpost_err;

struct DevBuf
{
  std::vector<void*> all;
  cudaStream_t s = nullptr;
  template <typename T> T* get (size_t n)
  {
    void* p = nullptr;
    if (cudaMalloc (&p, std::max<size_t> (n, 1) * sizeof (T)) != cudaSuccess) return nullptr;
    all.push_back (p);
    return (T*) p;
  }
  ~DevBuf () { for (void* p : all) cudaFree (p); if (s) cudaStreamDestroy (s); }
};

int mp_fail (int code, const std::string& m) { g_meshpost_err = m; return code; }

#define MCK(call)                                                                                   \
  do {                                                                                              \
    cudaError_t e_ = (call);                                                                        \
    if (e_ != cudaSuccess) return mp_fail (B200TSDF_ECUDA, std::string (#call) + ": " + cudaGetErrorString (e_)); \
  } while (0)
#define MNN(ptr) do { if (!(ptr)) return mp_fail (B200TSDF_ENOMEM, "device allocation failed (mesh post-processing)"); } while (0)

constexpr int TPB = 256;
inline unsigned nblk (size_t n) { return (unsigned) ((n + TPB - 1) / TPB); }

// ---- shared kernels --------------------------------------------------------------------------------
__global__ void k_grid_clear (uint64_t* keys, int* head, size_t slots)
{
  size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i < slots) { keys[i] = GRID_EMPTY; head[i] = -1; }
}
__global__ void k_grid_insert (PointGrid g, int n)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) grid_insert (g, i);
}
__global__ void k_iota (int* a, int n)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = i;
}

int build_grid (DevBuf& B, PointGrid& g, const float* d_pts, int n, double cell)
{
  size_t slots = 1024;
  while (slots < 2 * (size_t) n) slots <<= 1;
  g.keys = B.get<uint64_t> (slots); g.head = B.get<int> (slots); g.next = B.get<int> (n);
  MNN (g.keys); MNN (g.head); MNN (g.next);
  g.mask = (uint32_t) (slots - 1); g.inv_cell = 1.0 / cell; g.pts = d_pts;
  k_grid_clear<<<nblk (slots), TPB, 0, B.s>>> (g.keys, g.head, slots);
  if (n) k_grid_insert<<<nblk (n), TPB, 0, B.s>>> (g, n);
  MCK (cudaGetLastError ());
  return 0;
}

int exclusive_scan (DevBuf& B, const int* in, int* out, size_t n)
{
  size_t bytes = 0;
  MCK (cub::DeviceScan::ExclusiveSum (nullptr, bytes, in, out, (int) n, B.s));
  void* tmp = B.get<unsigned char> (bytes);
  MNN (tmp);
  MCK (cub::DeviceScan::ExclusiveSum (tmp, bytes, in, out, (int) n, B.s));
  return 0;
}

int check_mesh_args (const float* verts, size_t nverts, const int32_t* tris, size_t ntris,
                     float** out_verts, size_t* out_nverts, int32_t** out_tris, size_t* out_ntris)
{
  if ((!verts && nverts) || (!tris && ntris) || !out_verts || !out_nverts || !out_tris || !out_ntris)
    return mp_fail (B200TSDF_EINVAL, "null argument");
  if (nverts >= (size_t) 1 << 31 || ntris >= ((size_t) 1 << 31) / 3) return mp_fail (B200TSDF_EINVAL, "mesh too large for 32-bit indices");
  for (size_t i = 0; i < 3 * ntris; ++i)
    if (tris[i] < 0 || (size_t) tris[i] >= nverts) return mp_fail (B200TSDF_EINVAL, "triangle index out of range");
  *out_verts = nullptr; *out_tris = nullptr; *out_nverts = 0; *out_ntris = 0;
  return 0;
}

int open_device (DevBuf& B, int device)
{
  int ndev = 0;
  if (cudaGetDeviceCount (&ndev) != cudaSuccess || device < 0 || device >= ndev)
    return mp_fail (B200TSDF_ENODEVICE, "no such CUDA device (mesh post-processing has no CPU path)");
  MCK (cudaSetDevice (device));
  MCK (cudaStreamCreateWithFlags (&B.s, cudaStreamNonBlocking));
  return 0;
}

// copies the compacted mesh back into malloc'ed host arrays (released with b200tsdf_free)
int download_mesh (DevBuf& B, const float* d_verts, size_t nv, const int* d_tris, size_t nt,
                   float** out_verts, size_t* out_nverts, int32_t** out_tris, size_t* out_ntris)
{
  float* hv = (float*) std::malloc (std::max<size_t> (nv, 1) * 12);
  int32_t* ht = (int32_t*) std::malloc (std::max<size_t> (nt, 1) * 12);
  if (!hv || !ht) { std::free (hv); std::free (ht); return mp_fail (B200TSDF_ENOMEM, "host allocation failed"); }
  cudaError_t e = cudaSuccess;
  if (nv) e = cudaMemcpyAsync (hv, d_verts, nv * 12, cudaMemcpyDeviceToHost, B.s);
  if (e == cudaSuccess && nt) e = cudaMemcpyAsync (ht, d_tris, nt * 12, cudaMemcpyDeviceToHost, B.s);
  if (e == cudaSuccess) e = cudaStreamSynchronize (B.s);
  if (e != cudaSuccess) { std::free (hv); std::free (ht); return mp_fail (B200TSDF_ECUDA, cudaGetErrorString (e)); }
  *out_verts = hv; *out_nverts = nv; *out_tris = ht; *out_ntris = nt;
  return 0;
}

// ---- flattenVertices -------------------------------------------------------------------------------
__global__ void k_fv_round (PointGrid g, float r2, unsigned char* state, int n, int* remaining)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  bool und = i < n && fv_round (g, r2, state, i);
  unsigned m = __ballot_sync (0xffffffffu, und);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd (remaining, __popc (m));
}
// fall-back for pathological chains (each round only resolves the head of a chain): index order, one thread
__global__ void k_fv_serial (PointGrid g, float r2, unsigned char* state, int n)
{
  for (int i = 0; i < n; ++i) fv_round (g, r2, state, i);
}
__global__ void k_fv_target (PointGrid g, float r2, const unsigned char* state, int n, int* rep, int* kept)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  rep[i] = fv_target (g, r2, state, i);
  kept[i] = state[i] == FV_KEPT;
}
__global__ void k_fv_vertices (const float* verts, const int* kept, const int* rank, int n, float* out)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !kept[i]) return;
  size_t o = 3 * (size_t) rank[i];
  out[o] = verts[3 * (size_t) i]; out[o + 1] = verts[3 * (size_t) i + 1]; out[o + 2] = verts[3 * (size_t) i + 2];
}
// integrate.cpp:129-146: remap the corners, flag the faces that stay
__global__ void k_fv_faces (int* tris, const int* rep, const int* rank, int nt, int* keep)
{
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  int a = rank[rep[tris[3 * (size_t) t]]], b = rank[rep[tris[3 * (size_t) t + 1]]], c = rank[rep[tris[3 * (size_t) t + 2]]];
  tris[3 * (size_t) t] = a; tris[3 * (size_t) t + 1] = b; tris[3 * (size_t) t + 2] = c;
  keep[t] = !(a == b || b == c || c == a);
}
__global__ void k_compact_tris (const int* tris, const int* keep, const int* pos, int nt, int* out)
{
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || !keep[t]) return;
  size_t o = 3 * (size_t) pos[t];
  out[o] = tris[3 * (size_t) t]; out[o + 1] = tris[3 * (size_t) t + 1]; out[o + 2] = tris[3 * (size_t) t + 2];
}

// ---- cleanupMesh -----------------------------------------------------------------------------------
__global__ void k_cm_centroids (const float* verts, const int* tris, int nt, float* cent)
{
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < nt) face_centroid (verts, tris + 3 * (size_t) t, cent + 3 * (size_t) t);
}
__global__ void k_cm_count (PointGrid g, float r2, int K, int nt, int* cnt, int* nb)
{
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < nt) cnt[t] = cm_count (g, r2, K, t, nb);
}
__global__ void k_cm_union (int K, int nt, const int* cnt, const int* nb, int* parent, int* touches_big)
{
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || cnt[t] >= K) return;
  int big = 0;
  for (int k = 0; k < cnt[t]; ++k)
  {
    int j = nb[(size_t) t * (CM_MAX_K - 1) + k];
    if (cnt[j] >= K) big = 1; else uf_union (parent, t, j);
  }
  touches_big[t] = big;
}
__global__ void k_cm_sizes (int K, int nt, const int* cnt, int* parent, const int* touches_big, int* size, int* has_big)
{
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || cnt[t] >= K) return;
  int r = uf_find (parent, t);
  atomicAdd (&size[r], 1);
  if (touches_big[t]) has_big[r] = 1;
}
// EuclideanClusterExtraction returns the clusters with 1..K points; their faces are erased (integrate.cpp:168-183)
__global__ void k_cm_keep (int K, int nt, const int* cnt, int* parent, const int* size, const int* has_big, int* keep)
{
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  bool remove = false;
  if (cnt[t] < K) { int r = uf_find (parent, t); remove = !has_big[r] && size[r] <= K; }
  keep[t] = !remove;
}
__global__ void k_cm_mark_vertices (const int* tris, const int* keep, int nt, int* used)
{
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || !keep[t]) return;
  used[tris[3 * (size_t) t]] = 1; used[tris[3 * (size_t) t + 1]] = 1; used[tris[3 * (size_t) t + 2]] = 1;
}
__global__ void k_cm_faces (const int* tris, const int* keep, const int* pos, const int* vrank, int nt, int* out)
{
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt || !keep[t]) return;
  size_t o = 3 * (size_t) pos[t];
  out[o] = vrank[tris[3 * (size_t) t]]; out[o + 1] = vrank[tris[3 * (size_t) t + 1]]; out[o + 2] = vrank[tris[3 * (size_t) t + 2]];
}

int last_plus (DevBuf& B, const int* flag, const int* scan, size_t n, size_t* total)
{
  *total = 0;
  if (!n) return 0;
  int a = 0, b = 0;
  MCK (cudaMemcpyAsync (&a, flag + n - 1, 4, cudaMemcpyDeviceToHost, B.s));
  MCK (cudaMemcpyAsync (&b, scan + n - 1, 4, cudaMemcpyDeviceToHost, B.s));
  MCK (cudaStreamSynchronize (B.s));
  *total = (size_t) a + (size_t) b;
  return 0;
}

} // namespace

extern "C" const char* b200tsdf_meshpost_last_error (void) { return g_meshpost_err.c_str (); }
extern "C" void b200tsdf_mesh_free (void* p) { std::free (p); }

extern "C" int b200tsdf_mesh_flatten (int device, const float* verts, size_t nverts, const int32_t* tris, size_t ntris, float min_dist,
                                      float** out_verts, size_t* out_nverts, int32_t** out_tris, size_t* out_ntris)
{
  int rc = check_mesh_args (verts, nverts, tris, ntris, out_verts, out_nverts, out_tris, out_ntris);
  if (rc) return rc;
  DevBuf B;
  if ((rc = open_device (B, device))) return rc;
  const int nv = (int) nverts, nt = (int) ntris;
  float* d_verts = B.get<float> (3 * nverts); int* d_tris = B.get<int> (3 * ntris);
  unsigned char* state = B.get<unsigned char> (nverts);
  int *rep = B.get<int> (nverts), *kept = B.get<int> (nverts), *rank = B.get<int> (nverts), *remaining = B.get<int> (1);
  int *keep = B.get<int> (ntris), *pos = B.get<int> (ntris), *d_tris_out = B.get<int> (3 * ntris);
  MNN (d_verts); MNN (d_tris); MNN (state); MNN (rep); MNN (kept); MNN (rank); MNN (remaining); MNN (keep); MNN (pos); MNN (d_tris_out);
  if (nv) MCK (cudaMemcpyAsync (d_verts, verts, nverts * 12, cudaMemcpyHostToDevice, B.s));
  if (nt) MCK (cudaMemcpyAsync (d_tris, tris, ntris * 12, cudaMemcpyHostToDevice, B.s));
  MCK (cudaMemsetAsync (state, FV_UNDECIDED, std::max<size_t> (nverts, 1), B.s));
  // pcl::search::KdTree::radiusSearch (i, min_dist): FLANN compares squared float distances with float (radius*radius)
  const float r2 = min_dist > 0.f ? (float) ((double) min_dist * (double) min_dist) : 0.f;      // radius <= 0 (or NaN): nothing is in range
  PointGrid g{};
  if ((rc = build_grid (B, g, d_verts, nv, std::max ((double) min_dist * 1.001, 1e-7)))) return rc;
  int left = nv;
  for (int round = 0; left > 0 && round < 48; ++round)
  {
    MCK (cudaMemsetAsync (remaining, 0, 4, B.s));
    k_fv_round<<<nblk (nv), TPB, 0, B.s>>> (g, r2, state, nv, remaining);
    MCK (cudaMemcpyAsync (&left, remaining, 4, cudaMemcpyDeviceToHost, B.s));
    MCK (cudaStreamSynchronize (B.s));
  }
  if (left > 0) k_fv_serial<<<1, 1, 0, B.s>>> (g, r2, state, nv);
  size_t nv_new = 0, nt_new = 0;
  float* d_verts_out = B.get<float> (3 * nverts);
  MNN (d_verts_out);
  if (nv)
  {
    k_fv_target<<<nblk (nv), TPB, 0, B.s>>> (g, r2, state, nv, rep, kept);
    if ((rc = exclusive_scan (B, kept, rank, nverts))) return rc;
    k_fv_vertices<<<nblk (nv), TPB, 0, B.s>>> (d_verts, kept, rank, nv, d_verts_out);
    if ((rc = last_plus (B, kept, rank, nverts, &nv_new))) return rc;
  }
  if (nt)
  {
    k_fv_faces<<<nblk (nt), TPB, 0, B.s>>> (d_tris, rep, rank, nt, keep);
    if ((rc = exclusive_scan (B, keep, pos, ntris))) return rc;
    k_compact_tris<<<nblk (nt), TPB, 0, B.s>>> (d_tris, keep, pos, nt, d_tris_out);
    if ((rc = last_plus (B, keep, pos, ntris, &nt_new))) return rc;
  }
  MCK (cudaGetLastError ());
  return download_mesh (B, d_verts_out, nv_new, d_tris_out, nt_new, out_verts, out_nverts, out_tris, out_ntris);
}

extern "C" int b200tsdf_mesh_cleanup (int device, const float* verts, size_t nverts, const int32_t* tris, size_t ntris,
                                      float face_dist, int min_neighbors,
                                      float** out_verts, size_t* out_nverts, int32_t** out_tris, size_t* out_ntris)
{
  int rc = check_mesh_args (verts, nverts, tris, ntris, out_verts, out_nverts, out_tris, out_ntris);
  if (rc) return rc;
  if (min_neighbors < 1 || min_neighbors > CM_MAX_K) return mp_fail (B200TSDF_EINVAL, "min_neighbors must be in 1..16");
  DevBuf B;
  if ((rc = open_device (B, device))) return rc;
  const int nv = (int) nverts, nt = (int) ntris, K = min_neighbors;
  float* d_verts = B.get<float> (3 * nverts); int* d_tris = B.get<int> (3 * ntris); float* cent = B.get<float> (3 * ntris);
  int *cnt = B.get<int> (ntris), *nb = B.get<int> (ntris * (CM_MAX_K - 1)), *parent = B.get<int> (ntris), *touches = B.get<int> (ntris);
  int *size = B.get<int> (ntris), *has_big = B.get<int> (ntris), *keep = B.get<int> (ntris), *pos = B.get<int> (ntris);
  int *used = B.get<int> (nverts), *vrank = B.get<int> (nverts), *d_tris_out = B.get<int> (3 * ntris);
  float* d_verts_out = B.get<float> (3 * nverts);
  MNN (d_verts); MNN (d_tris); MNN (cent); MNN (cnt); MNN (nb); MNN (parent); MNN (touches); MNN (size); MNN (has_big); MNN (keep); MNN (pos);
  MNN (used); MNN (vrank); MNN (d_tris_out); MNN (d_verts_out);
  if (nv) MCK (cudaMemcpyAsync (d_verts, verts, nverts * 12, cudaMemcpyHostToDevice, B.s));
  if (nt) MCK (cudaMemcpyAsync (d_tris, tris, ntris * 12, cudaMemcpyHostToDevice, B.s));
  size_t nv_new = 0, nt_new = 0;
  if (nt)
  {
    // EuclideanClusterExtraction::setClusterTolerance (face_dist): radiusSearch with float (tolerance * tolerance)
    const float r2 = face_dist > 0.f ? (float) ((double) face_dist * (double) face_dist) : 0.f;
    k_cm_centroids<<<nblk (nt), TPB, 0, B.s>>> (d_verts, d_tris, nt, cent);
    PointGrid g{};
    if ((rc = build_grid (B, g, cent, nt, std::max ((double) face_dist * 1.001, 1e-7)))) return rc;
    k_cm_count<<<nblk (nt), TPB, 0, B.s>>> (g, r2, K, nt, cnt, nb);
    k_iota<<<nblk (nt), TPB, 0, B.s>>> (parent, nt);
    MCK (cudaMemsetAsync (size, 0, ntris * 4, B.s)); MCK (cudaMemsetAsync (has_big, 0, ntris * 4, B.s));
    MCK (cudaMemsetAsync (touches, 0, ntris * 4, B.s));
    k_cm_union<<<nblk (nt), TPB, 0, B.s>>> (K, nt, cnt, nb, parent, touches);
    k_cm_sizes<<<nblk (nt), TPB, 0, B.s>>> (K, nt, cnt, parent, touches, size, has_big);
    k_cm_keep<<<nblk (nt), TPB, 0, B.s>>> (K, nt, cnt, parent, size, has_big, keep);
    if ((rc = exclusive_scan (B, keep, pos, ntris))) return rc;
    if ((rc = last_plus (B, keep, pos, ntris, &nt_new))) return rc;
  }
  // integrate.cpp:184-213: drop the vertices no remaining face uses, keep the order of the rest
  if (nv)
  {
    MCK (cudaMemsetAsync (used, 0, nverts * 4, B.s));
    if (nt) k_cm_mark_vertices<<<nblk (nt), TPB, 0, B.s>>> (d_tris, keep, nt, used);
    if ((rc = exclusive_scan (B, used, vrank, nverts))) return rc;
    k_fv_vertices<<<nblk (nv), TPB, 0, B.s>>> (d_verts, used, vrank, nv, d_verts_out);
    if ((rc = last_plus (B, used, vrank, nverts, &nv_new))) return rc;
    if (nt) k_cm_faces<<<nblk (nt), TPB, 0, B.s>>> (d_tris, keep, pos, vrank, nt, d_tris_out);
  }
  MCK (cudaGetLastError ());
  return download_mesh (B, d_verts_out, nv_new, d_tris_out, nt_new, out_verts, out_nverts, out_tris, out_ntris);
}

// ---- triangle ordering for b200tsdf_mesh (engine.cu) -----------------------------------------------------------------
namespace {
__global__ void k_gather_triangles (const unsigned int* __restrict__ order, size_t ntri, const float* __restrict__ v, const unsigned char* __restrict__ c,
                                    float* __restrict__ vo, unsigned char* __restrict__ co)
{
  // nine threads per triangle: thread q copies float q (and colour byte q) of the triangle
  size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ntri * 9) return;
  size_t t = i / 9, q = i - t * 9, src = (size_t) order[t] * 9 + q;
  vo[i] = v[src];
  if (c) co[i] = c[src];
}
}

int b2_sort_triangles (cudaStream_t s, size_t ntri, int key_bits, unsigned long long* d_keys, const float* d_v, const unsigned char* d_c,
                       float* d_v_out, unsigned char* d_c_out)
{
  if (!ntri) return 0;
  if (ntri >= ((size_t) 1 << 31)) return (int) cudaErrorInvalidValue;
  unsigned long long* keys2 = nullptr; unsigned int *idx = nullptr, *idx2 = nullptr; void* tmp = nullptr;
  size_t bytes = 0;
  cudaError_t e = cudaMalloc (&keys2, ntri * 8);
  if (e == cudaSuccess) e = cudaMalloc (&idx, ntri * 4);
  if (e == cudaSuccess) e = cudaMalloc (&idx2, ntri * 4);
  if (e == cudaSuccess) { k_iota<<<nblk (ntri), TPB, 0, s>>> ((int*) idx, (int) ntri); e = cudaGetLastError (); }
  if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs (nullptr, bytes, d_keys, keys2, idx, idx2, (int) ntri, 0, key_bits, s);
  if (e == cudaSuccess) e = cudaMalloc (&tmp, bytes);
  if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs (tmp, bytes, d_keys, keys2, idx, idx2, (int) ntri, 0, key_bits, s);
  if (e == cudaSuccess) { k_gather_triangles<<<nblk (ntri * 9), TPB, 0, s>>> (idx2, ntri, d_v, d_c, d_v_out, d_c_out); e = cudaGetLastError (); }
  if (e == cudaSuccess) e = cudaStreamSynchronize (s);
  cudaFree (keys2); cudaFree (idx); cudaFree (idx2); cudaFree (tmp);
  return (int) e;
}

int b2_sort_keys (cudaStream_t s, size_t n, int key_bits, const unsigned long long* d_keys, unsigned long long* d_keys_out)
{
  if (!n) return 0;
  if (n >= ((size_t) 1 << 31)) return (int) cudaErrorInvalidValue;
  void* tmp = nullptr;
  size_t bytes = 0;
  cudaError_t e = cub::DeviceRadixSort::SortKeys (nullptr, bytes, d_keys, d_keys_out, (int) n, 0, key_bits, s);
  if (e == cudaSuccess) e = cudaMalloc (&tmp, bytes);
  if (e == cudaSuccess) e = cub::DeviceRadixSort::SortKeys (tmp, bytes, d_keys, d_keys_out, (int) n, 0, key_bits, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize (s);
  cudaFree (tmp);
  return (int) e;
}
