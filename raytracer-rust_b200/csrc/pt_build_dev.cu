// pt_build_dev.cu — see pt_build_dev.h.  CUDA for sm_100a; CUB (header-only, part of the toolkit) provides the radix sort.
//
// Replaces, for large meshes, the host recursion of pt_build.cpp — itself the restatement of the reference's host-side
// recursive sort, BVHNode::new (/root/reference/src/acceleration/bvh.rs:15-76, sort at :45-53).
#include <cuda_runtime.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "pt_build_dev.h"

namespace pt {
namespace {

#define CKB(call)                                                                                                        \
  do {                                                                                                                   \
    cudaError_t e_ = (call);                                                                                             \
    if (e_ != cudaSuccess)                                                                                               \
      throw std::runtime_error(std::string(#call) + ": " + cudaGetErrorString(e_) + " (pt_build_dev.cu:" + std::to_string(__LINE__) + ")"); \
  } while (0)

template <typename T>
struct Buf {
  T *p = nullptr;
  size_t n = 0;
  explicit Buf(size_t count = 0) {
    if (count) alloc(count);
  }
  void alloc(size_t count) {
    release();
    CKB(cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T)));
    n = count;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
  }
  T *take() {
    T *r = p;
    p = nullptr;
    return r;
  }
  ~Buf() { release(); }
  Buf(const Buf &) = delete;
  Buf &operator=(const Buf &) = delete;
};

// Temporaries come out of ONE allocation per build step: cudaMalloc / cudaFree synchronise the device and their cost
// varies by an order of magnitude from call to call (measured: 137 to 495 ms for the same 2 M-triangle commit with ~25
// separate buffers), which is the same order as the whole build.
struct Arena {
  char *base = nullptr;
  size_t size = 0, used = 0;
  explicit Arena(size_t bytes) : size(bytes) { CKB(cudaMalloc(&base, std::max<size_t>(bytes, 256))); }
  ~Arena() {
    if (base) cudaFree(base);
  }
  Arena(const Arena &) = delete;
  Arena &operator=(const Arena &) = delete;
  static size_t need(size_t count, size_t elem) { return (count * elem + 255) & ~(size_t)255; }
  template <typename T>
  T *get(size_t count) {
    const size_t b = need(std::max<size_t>(count, 1), sizeof(T));
    if (used + b > size) throw std::runtime_error("pt_build_dev: arena too small");
    T *p = reinterpret_cast<T *>(base + used);
    used += b;
    return p;
  }
};

constexpr int kThreads = 256;
inline unsigned blocks_for(size_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

// order-preserving integer image of a float; -0.0 keyed as +0.0 when `canon` (the sort's comparator calls them equal)
__device__ __forceinline__ uint32_t fkey(float f, bool canon) {
  if (canon && f == 0.0f) f = 0.0f;
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float fkey_inv(uint32_t k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

// The node of depth L that holds position p.  The shape of the reference tree is a function of the triangle count alone:
// a node of size s > 4 (and depth < 25) splits at s / 2 (bvh.rs:19-27,55-56).  `real` is false when an ancestor was
// already a leaf: the descent then continues through VIRTUAL nodes, which only serve to give every position a sort key
// that keeps it where it is.
struct Seg {
  uint32_t lo, hi, idx;
  bool real;
};
__device__ __forceinline__ Seg descend(uint32_t p, uint32_t n, int L) {
  Seg s{0u, n, 0u, true};
  for (int d = 0; d < L; d++) {
    const uint32_t size = s.hi - s.lo;
    if (size <= 4u || d >= 25) s.real = false;
    const uint32_t mid = s.lo + size / 2u;
    if (p < mid) s.hi = mid, s.idx = s.idx * 2u;
    else s.lo = mid, s.idx = s.idx * 2u + 1u;
  }
  return s;
}

// per triangle: centroid ((v0 + v1) + v2) * (1/3) (bvh.rs:46; this TU is compiled with --fmad=false) and vertex bounds
__global__ void k_tri_prepare(const float *tris, uint32_t n, float *cen, float *tbox, uint32_t *idx, uint8_t *dead) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float *t = tris + (size_t)i * 12;
  for (int a = 0; a < 3; a++) {
    cen[(size_t)i * 3 + a] = ((t[a] + t[3 + a]) + t[6 + a]) * (1.0f / 3.0f);
    tbox[(size_t)i * 6 + a] = fminf(fminf(t[a], t[3 + a]), t[6 + a]);
    tbox[(size_t)i * 6 + 3 + a] = fmaxf(fmaxf(t[a], t[3 + a]), t[6 + a]);
  }
  idx[i] = i;
  dead[i] = 0;
}

__global__ void k_fill_u32(uint32_t *p, size_t n, uint32_t lo_value, uint32_t hi_value) {  // segment bounds: [lo x3, hi x3] per node
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = (i % 6) < 3 ? lo_value : hi_value;
}

// vertex bounds of every real node of depth L (bvh.rs:17): warp-aggregated atomic min / max on ordered integer keys
__global__ void k_level_bounds(const uint32_t *idx, const float *tbox, uint32_t n, int L, uint32_t *segb) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  Seg s{0u, 0u, 0u, false};
  if (p < n) s = descend(p, n, L);
  const bool part = p < n && s.real;
  const uint32_t mask = __ballot_sync(0xffffffffu, part);
  if (!part) return;
  const float *b = tbox + (size_t)idx[p] * 6;
  uint32_t k[6];
  for (int a = 0; a < 6; a++) k[a] = fkey(b[a], false);
  const int leader = __ffs((int)mask) - 1;
  const uint32_t lead_idx = __shfl_sync(mask, s.idx, leader);
  uint32_t *dst = segb + (size_t)s.idx * 6;
  if (__all_sync(mask, s.idx == lead_idx)) {
    for (int a = 0; a < 3; a++) k[a] = __reduce_min_sync(mask, k[a]);
    for (int a = 3; a < 6; a++) k[a] = __reduce_max_sync(mask, k[a]);
    if ((int)(threadIdx.x & 31u) == leader) {
      for (int a = 0; a < 3; a++) atomicMin(dst + a, k[a]);
      for (int a = 3; a < 6; a++) atomicMax(dst + a, k[a]);
    }
  } else {
    for (int a = 0; a < 3; a++) atomicMin(dst + a, k[a]);
    for (int a = 3; a < 6; a++) atomicMax(dst + a, k[a]);
  }
}

// flat test (aabb.rs:40: a zero-extent node is never entered), split axis (bvh.rs:36-43) and the level's sort key
__global__ void k_level_keys(const uint32_t *idx, const float *cen, const uint32_t *segb, uint32_t n, int L, uint8_t *dead,
                             unsigned long long *keys) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const Seg s = descend(p, n, L);
  const uint32_t tri = idx[p];
  uint32_t key = p - s.lo;  // leaves and virtual nodes: stay in place
  if (s.real) {
    const uint32_t *b = segb + (size_t)s.idx * 6;
    const float lx = fkey_inv(b[0]), ly = fkey_inv(b[1]), lz = fkey_inv(b[2]), hx = fkey_inv(b[3]), hy = fkey_inv(b[4]), hz = fkey_inv(b[5]);
    if (lx == hx || ly == hy || lz == hz) dead[tri] = 1;
    const uint32_t size = s.hi - s.lo;
    if (size > 4u && L < 25 && keys != nullptr) {
      const float ex = hx - lx, ey = hy - ly, ez = hz - lz;
      const int axis = (ex > ey && ex > ez) ? 0 : (ey > ez ? 1 : 2);
      key = fkey(cen[(size_t)tri * 3 + axis], true);
    }
  }
  if (keys) keys[p] = ((unsigned long long)s.idx << 32) | (unsigned long long)key;
}

__global__ void k_finish_order(const uint32_t *idx, const uint8_t *dead, uint32_t n, int32_t *order, uint8_t *dead_by_pos) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const uint32_t tri = idx[p];
  order[tri] = (int32_t)p;
  dead_by_pos[p] = dead[tri];
}

// normals by DFS position, original index in .w (pt_build.h)
__global__ void k_normals(const float *tris, const int32_t *order, uint32_t n, float4 *normals) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float *t = tris + (size_t)i * 12;
  normals[order[i]] = make_float4(t[9], t[10], t[11], __uint_as_float(i));
}

// ---- step 2: the wide tree ------------------------------------------------------------------------------------
// Structure of one wide node, computed on the host from the live counts alone (gen_structure below).
struct WNode {
  uint32_t child_lo[8];   // first live rank of the child's range (its triangles are live_tri[child_lo .. child_lo + cnt))
  uint32_t child_cnt[8];  // live triangles: 0 = no child, 1..3 = leaf, > 3 = inner node
  uint32_t child_base;    // index of the first inner child (inner children are consecutive, in child order)
  uint32_t tri_base;      // first Tri48 record of this node's leaf children
};

struct Box {
  float lo[3], hi[3];
};

__device__ __forceinline__ void box_grow(Box &b, const float *p) {
  for (int a = 0; a < 3; a++) b.lo[a] = fminf(b.lo[a], p[a]), b.hi[a] = fmaxf(b.hi[a], p[a]);
}

// A reference leaf with four live triangles becomes two leaves of two (a wide-node leaf holds at most three).  WHICH two go
// together is free — the records carry their own ids — so each quad is re-paired to the split with the smallest summed box
// area: on a regular mesh the reference's centroid order pairs triangles of neighbouring cells as often as the two halves
// of one cell, and a mismatched pair doubles the leaf's box.
__device__ __forceinline__ float pair_area(const float *a, const float *b) {
  float lo[3], hi[3];
  for (int k = 0; k < 3; k++) {
    lo[k] = fminf(fminf(fminf(a[k], a[3 + k]), a[6 + k]), fminf(fminf(b[k], b[3 + k]), b[6 + k]));
    hi[k] = fmaxf(fmaxf(fmaxf(a[k], a[3 + k]), a[6 + k]), fmaxf(fmaxf(b[k], b[3 + k]), b[6 + k]));
  }
  const float x = hi[0] - lo[0], y = hi[1] - lo[1], z = hi[2] - lo[2];
  return x * y + y * z + z * x;
}
__global__ void k_pair_quads(const uint32_t *quads, uint32_t nq, uint32_t *live_tri, const float *tris) {
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  uint32_t *t = live_tri + quads[q];
  const uint32_t i0 = t[0], i1 = t[1], i2 = t[2], i3 = t[3];
  const float *p0 = tris + (size_t)i0 * 12, *p1 = tris + (size_t)i1 * 12, *p2 = tris + (size_t)i2 * 12, *p3 = tris + (size_t)i3 * 12;
  const float a01 = pair_area(p0, p1) + pair_area(p2, p3), a02 = pair_area(p0, p2) + pair_area(p1, p3), a03 = pair_area(p0, p3) + pair_area(p1, p2);
  if (a02 < a01 && a02 <= a03) t[1] = i2, t[2] = i1;       // (0,2) (1,3)
  else if (a03 < a01 && a03 < a02) t[1] = i3, t[3] = i1;   // (0,3) (2,1)
}

// Bottom-up, one thread per wide node of a level (deepest level first), indexed by STRUCTURAL id (the breadth-first
// numbering of gen_structure): the node's box = union of its children's boxes (from triangles or from the level below).
__global__ void k_boxes_level(const WNode *wn, uint32_t first, uint32_t count, const uint32_t *live_tri, const float *tris, Box *nodebox) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const uint32_t node = first + t;
  const WNode w = wn[node];
  Box nb;
  for (int a = 0; a < 3; a++) nb.lo[a] = INFINITY, nb.hi[a] = -INFINITY;
  uint32_t inner_rank = 0;
  for (int c = 0; c < 8; c++) {
    const uint32_t cnt = w.child_cnt[c];
    if (cnt == 0u) break;  // children are packed at the front
    if (cnt > 3u) {
      const Box b = nodebox[w.child_base + inner_rank++];
      for (int a = 0; a < 3; a++) nb.lo[a] = fminf(nb.lo[a], b.lo[a]), nb.hi[a] = fmaxf(nb.hi[a], b.hi[a]);
    } else {
      for (uint32_t k = 0; k < cnt; k++) {
        const float *tp = tris + (size_t)live_tri[w.child_lo[c] + k] * 12;
        box_grow(nb, tp), box_grow(nb, tp + 3), box_grow(nb, tp + 6);
      }
    }
  }
  nodebox[node] = nb;
}

// inner children of the structural node that sits at final position f of its level
__global__ void k_inner_count(const WNode *wn, const uint32_t *sid, uint32_t count, uint32_t *out) {
  const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= count) return;
  const WNode &w = wn[sid[f]];
  uint32_t k = 0;
  for (int c = 0; c < 8; c++) k += w.child_cnt[c] > 3u ? 1u : 0u;
  out[f] = k;
}

// Top-down, one thread per wide node of a level.  The traversal finds the inner child in slot s at
// child_base + popc(inner slots below s) (pt_bvh8.h), so a node's inner children must be numbered in SLOT order, and the
// slots come from the geometry (octant of the child's centre).  `sid[f]` = structural id of the node whose FINAL index is
// level_first + f; this kernel assigns the slots, writes the Node8 at the final index and hands its inner children, in
// slot order, the final positions cbase[f] + k of the next level (`sid_next`).  Also writes the Tri48 records of the leaf
// children (their place, tri_base, is structural: any place is as good as another).
__global__ void k_emit_level(const WNode *wn, const uint32_t *sid, uint32_t level_first, uint32_t count, const uint32_t *cbase,
                             uint32_t next_first, uint32_t *sid_next, const uint32_t *live_tri, const float *tris, const int32_t *order,
                             const Box *nodebox, float4 *nodes, float4 *tri48, float *root_frame, int *error) {
  const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= count) return;
  const uint32_t u = sid[f];
  const WNode w = wn[u];
  const Box nb = nodebox[u];
  Box cb[8];
  uint32_t child_sid[8];
  bool inner[8];
  int nch = 0;
  uint32_t inner_rank = 0;
  for (int c = 0; c < 8; c++) {
    const uint32_t cnt = w.child_cnt[c];
    if (cnt == 0u) break;
    nch = c + 1;
    inner[c] = cnt > 3u;
    child_sid[c] = 0u;
    if (inner[c]) {
      child_sid[c] = w.child_base + inner_rank++;
      cb[c] = nodebox[child_sid[c]];
    } else {
      for (int a = 0; a < 3; a++) cb[c].lo[a] = INFINITY, cb[c].hi[a] = -INFINITY;
      for (uint32_t k = 0; k < cnt; k++) {
        const float *tp = tris + (size_t)live_tri[w.child_lo[c] + k] * 12;
        box_grow(cb[c], tp), box_grow(cb[c], tp + 3), box_grow(cb[c], tp + 6);
      }
    }
  }

  // octant-ordered slots: slot s lives at corner (s&1 ? +x : -x, s&2 ? +y : -y, s&4 ? +z : -z); greedy on the projection
  // of (child centre - node centre) on the corner direction (same rule as pt_build.cpp: collapse)
  int slot_child[8];
  for (int s = 0; s < 8; s++) slot_child[s] = -1;
  {
    double ccx[8], ccy[8], ccz[8];
    const double ncx = 0.5f * (nb.lo[0] + nb.hi[0]), ncy = 0.5f * (nb.lo[1] + nb.hi[1]), ncz = 0.5f * (nb.lo[2] + nb.hi[2]);
    for (int i = 0; i < nch; i++) {
      ccx[i] = 0.5 * ((double)cb[i].lo[0] + cb[i].hi[0]) - ncx;
      ccy[i] = 0.5 * ((double)cb[i].lo[1] + cb[i].hi[1]) - ncy;
      ccz[i] = 0.5 * ((double)cb[i].lo[2] + cb[i].hi[2]) - ncz;
    }
    uint32_t child_done = 0u;
    for (int round = 0; round < nch; round++) {
      int bi = -1, bs = -1;
      double bc = -1.7976931348623157e308;
      for (int i = 0; i < nch; i++) {
        if (child_done & (1u << i)) continue;
        for (int s = 0; s < 8; s++) {
          if (slot_child[s] >= 0) continue;
          const double d = ((s & 1) ? ccx[i] : -ccx[i]) + ((s & 2) ? ccy[i] : -ccy[i]) + ((s & 4) ? ccz[i] : -ccz[i]);
          if (d > bc) bc = d, bi = i, bs = s;
        }
      }
      child_done |= 1u << bi;
      slot_child[bs] = bi;
    }
  }

  // frame = node box padded on every side (pt_build.cpp: make_frame)
  float origin[3];
  int biased[3];
  double scale[3];
  for (int a = 0; a < 3; a++) {
    const float lo = nb.lo[a], hi = nb.hi[a];
    const float ext = hi - lo;
    const float maxabs = fmaxf(fabsf(lo), fabsf(hi));
    const float pad = ext * (1.0f / 512.0f) + maxabs * 0x1p-20f + 1e-30f;
    float flo = lo - pad, fhi = hi + pad;
    if (!(flo < lo)) flo = nextafterf(lo, -INFINITY);
    if (!(fhi > hi)) fhi = nextafterf(hi, INFINITY);
    const double need = ((double)fhi - (double)flo) / 255.0;
    int ex;
    frexp(need, &ex);
    int b = ex + 127;
    if (b < 1) b = 1;
    if (b > 254 - 15) {
      *error = 1;  // mesh extent too large for the quantised frame (trav_node adds 15 to the exponent)
      b = 254 - 15;
    }
    origin[a] = flo;
    biased[a] = b;
    scale[a] = ldexp(1.0, b - 127);
  }
  if (level_first == 0u && f == 0u) {
    for (int a = 0; a < 3; a++) {
      root_frame[a] = origin[a];
      const double top = (double)origin[a] + 255.0 * scale[a];
      float h = (float)top;
      if ((double)h < top) h = nextafterf(h, INFINITY);
      root_frame[3 + a] = h;
    }
  }

  uint32_t meta[8] = {0, 0, 0, 0, 0, 0, 0, 0}, qlo[3][8], qhi[3][8];
  for (int a = 0; a < 3; a++)
    for (int s = 0; s < 8; s++) qlo[a][s] = 255u, qhi[a][s] = 0u;
  uint32_t imask = 0u, tri_off = 0u, inner_seen = 0u;
  const uint32_t my_cbase = cbase[f];
  for (int s = 0; s < 8; s++) {
    const int c = slot_child[s];
    if (c < 0) continue;
    if (inner[c]) {
      imask |= 1u << s;
      meta[s] = 0x20u | (24u + (uint32_t)s);
      sid_next[my_cbase + inner_seen++] = child_sid[c];
    } else {
      const uint32_t cnt = w.child_cnt[c];
      const uint32_t unary = cnt == 1u ? 1u : (cnt == 2u ? 3u : 7u);
      meta[s] = (unary << 5) | tri_off;
      for (uint32_t k = 0; k < cnt; k++) {
        const uint32_t orig = live_tri[w.child_lo[c] + k];
        const float *tp = tris + (size_t)orig * 12;
        float4 *r = tri48 + (size_t)(w.tri_base + tri_off + k) * 3;
        // edge vectors with the reference's own subtraction (bvh.rs:94-95), so precomputing them changes no bit
        r[0] = make_float4(tp[0], tp[1], tp[2], __uint_as_float(orig));
        r[1] = make_float4(tp[3] - tp[0], tp[4] - tp[1], tp[5] - tp[2], __uint_as_float((uint32_t)order[orig]));
        r[2] = make_float4(tp[6] - tp[0], tp[7] - tp[1], tp[8] - tp[2], 0.0f);
      }
      tri_off += cnt;
    }
    for (int a = 0; a < 3; a++) {
      const float clo = cb[c].lo[a], chi = cb[c].hi[a];
      const double padc = (double)fmaxf(fabsf(clo), fabsf(chi)) * 0x1p-21 + 1e-30;
      double ql = floor(((double)clo - padc - (double)origin[a]) / scale[a]);
      double qh = ceil(((double)chi + padc - (double)origin[a]) / scale[a]);
      ql = fmin(fmax(ql, 0.0), 255.0);
      qh = fmin(fmax(qh, 0.0), 255.0);
      qlo[a][s] = (uint32_t)ql;
      qhi[a][s] = (uint32_t)qh;
    }
  }

  auto pack4 = [](const uint32_t *b) { return __uint_as_float(b[0] | (b[1] << 8) | (b[2] << 16) | (b[3] << 24)); };
  const uint32_t ebits = (uint32_t)biased[0] | ((uint32_t)biased[1] << 8) | ((uint32_t)biased[2] << 16) | (imask << 24);
  float4 *out = nodes + (size_t)(level_first + f) * 5;
  out[0] = make_float4(origin[0], origin[1], origin[2], __uint_as_float(ebits));
  out[1] = make_float4(__uint_as_float(next_first + my_cbase), __uint_as_float(w.tri_base), pack4(meta), pack4(meta + 4));
  out[2] = make_float4(pack4(qlo[0]), pack4(qlo[0] + 4), pack4(qlo[1]), pack4(qlo[1] + 4));
  out[3] = make_float4(pack4(qlo[2]), pack4(qlo[2] + 4), pack4(qhi[0]), pack4(qhi[0] + 4));
  out[4] = make_float4(pack4(qhi[1]), pack4(qhi[1] + 4), pack4(qhi[2]), pack4(qhi[2] + 4));
}

// ---- step 2, DevBuildMode::Sah: pt_build.cpp's binned SAH tree and collapse plan, decision for decision ------------
// A split decision depends on the SET of triangles in a node only (bins hold min / max / counts; the sweep runs over the
// non-empty bins in double, axes x -> y -> z, strict <), so kernels that see the same sets make the same decisions.
// Triangles are addressed by ORIGINAL index; `prim` is the permutation of the live ones, initially ascending (the host's
// live_ids), and every node owns a contiguous range of it.  Node ids depend on ranges alone, not on scheduling: a range
// [f, f + c) owns ids [2f, 2f + 2c - 1); a leaf takes 2f, an inner node split at `mid` takes 2 mid - 1, its children the
// ranges below and above.
constexpr int kBins = 16, kLeafMax = 3;
constexpr uint32_t kWarpMax = 32;  // nodes of at most this many triangles: one warp builds the whole subtree (k_small)
constexpr int kBinWords = 13;      // per bin: box lo / hi keys, centroid lo / hi keys (fkey), count
constexpr int kNodeBinWords = 3 * kBins * kBinWords;

struct OpenNode {  // a node of > kWarpMax triangles waiting for its level
  uint32_t first, count;
  int32_t parent, side;  // side 1: right child
  float cb[6];           // centroid bounds lo xyz, hi xyz
};
struct SmallNode {
  uint32_t first, count;
  int32_t parent, side;
};
struct SplitDev {  // decision for one open node: axis < 0 = all centroids coincide, split at mid
  int32_t axis, split;
  uint32_t mid;
  float lo, k;
};
struct B2Dev {  // binary tree by node id; count == 0: no node has this id
  Box *box;
  uint32_t *first, *count;
  int32_t *left, *right, *parent;
};

__device__ __forceinline__ bool bin_word_is_min(int w) { return w < 3 || (w >= 6 && w < 9); }

__device__ __forceinline__ double box_area(const Box &b) {  // pt_build.cpp: Box3::area
  const double x = (double)b.hi[0] - b.lo[0], y = (double)b.hi[1] - b.lo[1], z = (double)b.hi[2] - b.lo[2];
  if (x < 0) return 0.0;
  return 2.0 * (x * y + y * z + z * x);
}

__device__ __forceinline__ void link_node(const B2Dev &b2, int32_t id, int32_t parent, int32_t side, int32_t *root_id) {
  b2.parent[id] = parent;
  if (parent < 0) *root_id = id;
  else (side ? b2.right : b2.left)[parent] = id;
}

// live triangles in ascending original index, centroids 0.5 (lo + hi) of every triangle's box (pt_build.cpp:872-884)
__global__ void k_live_flags(const uint8_t *dead, uint32_t n, uint32_t *flag) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flag[i] = dead[i] ? 0u : 1u;
}
__global__ void k_live_scatter(const uint32_t *flag, const uint32_t *rank, const float *tbox, uint32_t n, uint32_t *prim, float *pcen) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (flag[i]) prim[rank[i]] = i;
  for (int a = 0; a < 3; a++) pcen[(size_t)i * 3 + a] = 0.5f * (tbox[(size_t)i * 6 + a] + tbox[(size_t)i * 6 + 3 + a]);
}

// centroid bounds of the root (only when it is an open node)
__global__ void k_root_cb(const uint32_t *prim, const float *pcen, uint32_t nl, uint32_t *keys) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t k[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
  if (i < nl) {
    const float *c = pcen + (size_t)prim[i] * 3;
    for (int a = 0; a < 3; a++) k[a] = k[3 + a] = fkey(c[a], false);
  }
  for (int a = 0; a < 3; a++) k[a] = __reduce_min_sync(0xffffffffu, k[a]), k[3 + a] = __reduce_max_sync(0xffffffffu, k[3 + a]);
  if ((threadIdx.x & 31u) == 0u)
    for (int a = 0; a < 3; a++) atomicMin(keys + a, k[a]), atomicMax(keys + 3 + a, k[3 + a]);
}
__global__ void k_root_open(const uint32_t *keys, uint32_t nl, OpenNode *open, uint32_t *off) {
  OpenNode o;
  o.first = 0u, o.count = nl, o.parent = -1, o.side = 0;
  for (int a = 0; a < 6; a++) o.cb[a] = fkey_inv(keys[a]);
  open[0] = o;
  off[0] = 0u;
}

// the open node that holds active element t: the last j with off[j] <= t
__device__ __forceinline__ uint32_t find_open(const uint32_t *off, uint32_t n_open, uint32_t t) {
  uint32_t lo = 0u, hi = n_open;
  while (hi - lo > 1u) {
    const uint32_t m = (lo + hi) >> 1;
    if (off[m] <= t) lo = m;
    else hi = m;
  }
  return lo;
}

__device__ __forceinline__ void axis_scale(const float *cb, bool ok[3], float kk[3]) {  // pt_build.cpp:276-280
  for (int a = 0; a < 3; a++) {
    const float cext = cb[3 + a] - cb[a];
    ok[a] = cext > 0.0f;
    kk[a] = ok[a] ? (float)kBins / cext : 0.0f;
  }
}
__device__ __forceinline__ int bin_of(float c, float lo, float k) {
  const int bi = (int)((c - lo) * k);
  return min(max(bi, 0), kBins - 1);
}

__global__ void k_bins_init(uint32_t *bins, size_t words) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < words) bins[i] = bin_word_is_min((int)(i % kBinWords)) ? 0xffffffffu : 0u;
}

// One thread per triangle of an open node: its box, centroid and count into the node's 3 x 16 bins.  A block whose
// triangles all belong to one node aggregates in shared memory first.  Min, max and integer sums do not depend on the
// order of the updates.  A node whose centroids coincide on every axis is binned into bin 0 of axis 0 (box and count only).
__global__ void k_bin(const OpenNode *open, const uint32_t *off, uint32_t n_open, uint32_t total, const uint32_t *prim, const float *tbox,
                      const float *pcen, uint32_t *bins) {
  __shared__ uint32_t sb[kNodeBinWords];
  const uint32_t t0 = blockIdx.x * blockDim.x, t = t0 + threadIdx.x;
  const uint32_t j0 = find_open(off, n_open, t0), j1 = find_open(off, n_open, min(total, t0 + blockDim.x) - 1u);
  const bool shared = j0 == j1;
  if (shared) {
    for (int w = threadIdx.x; w < kNodeBinWords; w += blockDim.x) sb[w] = bin_word_is_min(w % kBinWords) ? 0xffffffffu : 0u;
    __syncthreads();
  }
  if (t < total) {
    const uint32_t j = shared ? j0 : find_open(off, n_open, t);
    const OpenNode &o = open[j];
    const uint32_t p = prim[o.first + (t - off[j])];
    uint32_t key[12];
    for (int a = 0; a < 6; a++) key[a] = fkey(tbox[(size_t)p * 6 + a], false);
    for (int a = 0; a < 3; a++) key[6 + a] = key[9 + a] = fkey(pcen[(size_t)p * 3 + a], false);
    bool ok[3];
    float kk[3];
    axis_scale(o.cb, ok, kk);
    const bool none = !ok[0] && !ok[1] && !ok[2];
    uint32_t *base = shared ? sb : bins + (size_t)j * kNodeBinWords;
    for (int a = 0; a < 3; a++) {
      if (!ok[a] && !(none && a == 0)) continue;
      const int bi = ok[a] ? bin_of(pcen[(size_t)p * 3 + a], o.cb[a], kk[a]) : 0;
      uint32_t *d = base + (a * kBins + bi) * kBinWords;
      for (int w = 0; w < 12; w++) {
        if (bin_word_is_min(w)) atomicMin(d + w, key[w]);
        else atomicMax(d + w, key[w]);
      }
      atomicAdd(d + 12, 1u);
    }
  }
  if (shared) {
    __syncthreads();
    uint32_t *d = bins + (size_t)j0 * kNodeBinWords;
    for (int w = threadIdx.x; w < kNodeBinWords; w += blockDim.x) {
      const int k = w % kBinWords;
      if (sb[w - k + 12] == 0u) continue;  // empty bin
      if (k == 12) atomicAdd(d + w, sb[w]);
      else if (bin_word_is_min(k)) atomicMin(d + w, sb[w]);
      else atomicMax(d + w, sb[w]);
    }
  }
}

__device__ __forceinline__ Box bin_box(const uint32_t *b, int first_word) {
  Box r;
  for (int a = 0; a < 3; a++) r.lo[a] = fkey_inv(b[first_word + a]), r.hi[a] = fkey_inv(b[first_word + 3 + a]);
  return r;
}
__device__ __forceinline__ void box_union(Box &acc, const Box &b) {
  for (int a = 0; a < 3; a++) acc.lo[a] = fminf(acc.lo[a], b.lo[a]), acc.hi[a] = fmaxf(acc.hi[a], b.hi[a]);
}
__device__ __forceinline__ Box box_empty() {
  Box r;
  for (int a = 0; a < 3; a++) r.lo[a] = INFINITY, r.hi[a] = -INFINITY;
  return r;
}

// One thread per open node: the sweep of pt_build.cpp:321-370 over its bins, the node's record, its children.  Children
// of more than kWarpMax triangles become candidates of the next level (slots 2j, 2j + 1, compacted in order by the
// caller: the next level's nodes stay sorted by range); the others go to the list k_small works on.
__global__ void k_sweep(const OpenNode *open, uint32_t n_open, const uint32_t *bins, SplitDev *splits, B2Dev b2, int32_t *root_id,
                        OpenNode *cand, uint8_t *cand_flag, SmallNode *small, uint32_t *counters) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_open) return;
  const OpenNode o = open[j];
  const uint32_t *B = bins + (size_t)j * kNodeBinWords;
  bool ok[3];
  float kk[3];
  axis_scale(o.cb, ok, kk);
  const int a0 = ok[0] ? 0 : (ok[1] ? 1 : (ok[2] ? 2 : 0));  // every triangle sits in one bin of this axis
  Box nb = box_empty();
  for (int bi = 0; bi < kBins; bi++)
    if (B[(a0 * kBins + bi) * kBinWords + 12]) box_union(nb, bin_box(B + (a0 * kBins + bi) * kBinWords, 0));
  int best_axis = -1, best_split = -1;
  double best_cost = 1.7976931348623157e308;
  for (int a = 0; a < 3; a++) {
    if (!ok[a]) continue;
    const uint32_t *ba = B + a * kBins * kBinWords;
    int idx[kBins], m = 0;
    for (int bi = 0; bi < kBins; bi++)
      if (ba[bi * kBinWords + 12]) idx[m++] = bi;
    if (m < 2) continue;
    double right_area[kBins];
    uint32_t right_n[kBins];
    Box acc = box_empty();
    uint32_t cnt = 0u;
    for (int q = m - 1; q > 0; q--) {
      box_union(acc, bin_box(ba + idx[q] * kBinWords, 0));
      cnt += ba[idx[q] * kBinWords + 12];
      right_area[q] = box_area(acc);
      right_n[q] = cnt;
    }
    acc = box_empty();
    cnt = 0u;
    for (int q = 0; q < m - 1; q++) {
      box_union(acc, bin_box(ba + idx[q] * kBinWords, 0));
      cnt += ba[idx[q] * kBinWords + 12];
      const double cost = box_area(acc) * (double)(int32_t)cnt + right_area[q + 1] * (double)(int32_t)right_n[q + 1];
      if (cost < best_cost) best_cost = cost, best_axis = a, best_split = idx[q] + 1;
    }
  }
  SplitDev sp;
  sp.axis = best_axis, sp.split = best_split, sp.lo = 0.0f, sp.k = 0.0f;
  float cbl[6], cbr[6];
  uint32_t nleft;
  if (best_axis < 0) {  // all centroids coincide: both halves keep the node's (point) centroid bounds
    nleft = o.count / 2u;
    for (int a = 0; a < 6; a++) cbl[a] = cbr[a] = o.cb[a];
  } else {
    sp.lo = o.cb[best_axis], sp.k = kk[best_axis];
    for (int a = 0; a < 3; a++) cbl[a] = cbr[a] = INFINITY, cbl[3 + a] = cbr[3 + a] = -INFINITY;
    nleft = 0u;
    const uint32_t *ba = B + best_axis * kBins * kBinWords;
    for (int bi = 0; bi < kBins; bi++) {
      const uint32_t c = ba[bi * kBinWords + 12];
      if (!c) continue;
      const Box cbox = bin_box(ba + bi * kBinWords, 6);
      float *dst = bi < best_split ? cbl : cbr;
      if (bi < best_split) nleft += c;
      for (int a = 0; a < 3; a++) dst[a] = fminf(dst[a], cbox.lo[a]), dst[3 + a] = fmaxf(dst[3 + a], cbox.hi[a]);
    }
  }
  const uint32_t mid = o.first + nleft;
  sp.mid = mid;
  splits[j] = sp;
  const int32_t id = (int32_t)(2u * mid - 1u);
  b2.box[id] = nb, b2.first[id] = o.first, b2.count[id] = o.count;
  link_node(b2, id, o.parent, o.side, root_id);
  atomicAdd(counters + 3, 1u);  // inner nodes
  for (int s = 0; s < 2; s++) {
    const uint32_t cf = s ? mid : o.first, cc = s ? o.first + o.count - mid : nleft;
    if (cc > kWarpMax) {
      OpenNode c;
      c.first = cf, c.count = cc, c.parent = id, c.side = s;
      for (int a = 0; a < 6; a++) c.cb[a] = s ? cbr[a] : cbl[a];
      cand[2 * j + s] = c;
      cand_flag[2 * j + s] = 1;
      atomicAdd(counters + 1, cc);  // elements of the next level
    } else {
      cand_flag[2 * j + s] = 0;
      small[atomicAdd(counters + 2, 1u)] = SmallNode{cf, cc, id, s};
    }
  }
}

// Partition of every open node's range as pt_build.cpp's std::partition does it — from the left the first element that
// goes right, from the right the first that goes left, swap, repeat (the bidirectional algorithm of libstdc++ and libc++) —
// so that every leaf ends up with the host's triangles in the host's order (the traversal's triangle order, hence its
// node and triangle test counts, depends on it).  In closed form: the k-th element (ascending) left of `mid` that goes
// right trades places with the k-th element (descending) right of `mid` that goes left.  Flag, one exclusive scan
// (caller), ranks of the right-hand movers, swaps.  All centroids coincide: the host keeps the order and splits at mid.
__global__ void k_part_flag(const OpenNode *open, const uint32_t *off, uint32_t n_open, uint32_t total, const uint32_t *prim, const float *pcen,
                            const SplitDev *splits, uint32_t *flag) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint32_t j = find_open(off, n_open, t);
  const uint32_t pos = open[j].first + (t - off[j]);
  const SplitDev sp = splits[j];
  if (sp.axis < 0) flag[t] = pos < sp.mid ? 1u : 0u;
  else flag[t] = bin_of(pcen[(size_t)prim[pos] * 3 + sp.axis], sp.lo, sp.k) < sp.split ? 1u : 0u;
}
__global__ void k_part_rank(const OpenNode *open, const uint32_t *off, uint32_t n_open, uint32_t total, const SplitDev *splits, const uint32_t *flag,
                            const uint32_t *scan, uint32_t *partner) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint32_t j = find_open(off, n_open, t), oj = off[j];
  const uint32_t first = open[j].first, pos = first + (t - oj), mid = splits[j].mid;
  if (pos >= mid && flag[t]) partner[first + (mid - first - 1u - (scan[t] - scan[oj]))] = pos;
}
__global__ void k_part_swap(const OpenNode *open, const uint32_t *off, uint32_t n_open, uint32_t total, const SplitDev *splits, const uint32_t *flag,
                            const uint32_t *scan, const uint32_t *partner, uint32_t *prim) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint32_t j = find_open(off, n_open, t), oj = off[j];
  const uint32_t first = open[j].first, pos = first + (t - oj);
  if (pos >= splits[j].mid || flag[t]) return;
  const uint32_t q = partner[first + (pos - first) - (scan[t] - scan[oj])];
  const uint32_t x = prim[pos];
  prim[pos] = prim[q];
  prim[q] = x;
}
__global__ void k_open_counts(const OpenNode *open, uint32_t n_open, uint32_t *cnt) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n_open) cnt[j] = open[j].count;
}

// One warp per node of <= kWarpMax triangles builds its whole subtree: lane i holds the i-th triangle of the range.  The
// bins of the host's sweep are not needed here — a split position after a non-empty bin is the same as "every triangle
// whose bin is <= this lane's bin goes left", so each lane evaluates the candidate of its own bin, per axis, over the
// exact left and right boxes (min / max over the lanes), and the warp takes the host's first minimum: lowest cost, then
// lowest axis, then lowest bin.
constexpr int kSmallWarps = 4;
__global__ void __launch_bounds__(32 * kSmallWarps) k_small(const SmallNode *small, uint32_t n_small, uint32_t *prim, const float *tbox,
                                                            const float *pcen, B2Dev b2, int32_t *root_id, uint32_t *counters) {
  __shared__ uint32_t s_prim[kSmallWarps][32], s_slot[kSmallWarps][32];
  __shared__ float s_val[kSmallWarps][32][9];
  const int wib = threadIdx.x >> 5;
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t w = blockIdx.x * kSmallWarps + wib;
  if (w >= n_small) return;  // whole warps
  const SmallNode sn = small[w];
  uint32_t p = 0u;
  float v[9];  // box lo xyz, hi xyz, centroid xyz
  for (int a = 0; a < 3; a++) v[a] = INFINITY, v[3 + a] = -INFINITY, v[6 + a] = 0.0f;
  if (lane < sn.count) {
    p = prim[sn.first + lane];
    for (int a = 0; a < 6; a++) v[a] = tbox[(size_t)p * 6 + a];
    for (int a = 0; a < 3; a++) v[6 + a] = pcen[(size_t)p * 3 + a];
  }
  struct Item {
    int32_t f, c, parent, side;
  } stack[32];
  int sp = 0;
  stack[sp++] = Item{0, (int32_t)sn.count, sn.parent, sn.side};
  uint32_t inner = 0u;
  while (sp > 0) {
    const Item it = stack[--sp];
    const bool in = (int)lane >= it.f && (int)lane < it.f + it.c;
    Box nb;
    float cb[6];
    for (int a = 0; a < 3; a++) {
      nb.lo[a] = in ? v[a] : INFINITY, nb.hi[a] = in ? v[3 + a] : -INFINITY;
      cb[a] = in ? v[6 + a] : INFINITY, cb[3 + a] = in ? v[6 + a] : -INFINITY;
    }
    for (int o = 16; o > 0; o >>= 1)
      for (int a = 0; a < 3; a++) {
        nb.lo[a] = fminf(nb.lo[a], __shfl_xor_sync(0xffffffffu, nb.lo[a], o));
        nb.hi[a] = fmaxf(nb.hi[a], __shfl_xor_sync(0xffffffffu, nb.hi[a], o));
        cb[a] = fminf(cb[a], __shfl_xor_sync(0xffffffffu, cb[a], o));
        cb[3 + a] = fmaxf(cb[3 + a], __shfl_xor_sync(0xffffffffu, cb[3 + a], o));
      }
    const uint32_t gfirst = sn.first + (uint32_t)it.f;
    if (it.c <= kLeafMax) {
      if (lane == 0u) {
        const int32_t id = (int32_t)(2u * gfirst);
        b2.box[id] = nb, b2.first[id] = gfirst, b2.count[id] = (uint32_t)it.c, b2.left[id] = -1, b2.right[id] = -1;
        link_node(b2, id, it.parent, it.side, root_id);
      }
      continue;
    }
    bool ok[3];
    float kk[3];
    axis_scale(cb, ok, kk);
    int bin[3];
    for (int a = 0; a < 3; a++) bin[a] = (in && ok[a]) ? bin_of(v[6 + a], cb[a], kk[a]) : -1;
    Box L[3], R[3];
    int nl[3] = {0, 0, 0}, nr[3] = {0, 0, 0};
    for (int a = 0; a < 3; a++) L[a] = box_empty(), R[a] = box_empty();
    for (int q = it.f; q < it.f + it.c; q++) {
      float u[6];
      int bq[3];
      for (int a = 0; a < 6; a++) u[a] = __shfl_sync(0xffffffffu, v[a], q);
      for (int a = 0; a < 3; a++) bq[a] = __shfl_sync(0xffffffffu, bin[a], q);
      for (int a = 0; a < 3; a++) {
        const bool left = bq[a] <= bin[a];
        Box &d = left ? L[a] : R[a];
        for (int e = 0; e < 3; e++) d.lo[e] = fminf(d.lo[e], u[e]), d.hi[e] = fmaxf(d.hi[e], u[3 + e]);
        (left ? nl[a] : nr[a])++;
      }
    }
    bool valid = false;
    double best = 0.0;
    int ba = 3, bb = kBins;
    for (int a = 0; a < 3; a++) {
      if (bin[a] < 0 || nr[a] == 0) continue;
      const double cost = box_area(L[a]) * (double)nl[a] + box_area(R[a]) * (double)nr[a];
      if (!valid || cost < best) valid = true, best = cost, ba = a, bb = bin[a];
    }
    for (int o = 16; o > 0; o >>= 1) {
      const bool ov = __shfl_xor_sync(0xffffffffu, (int)valid, o) != 0;
      const double oc = __shfl_xor_sync(0xffffffffu, best, o);
      const int oa = __shfl_xor_sync(0xffffffffu, ba, o), ob = __shfl_xor_sync(0xffffffffu, bb, o);
      if (ov && (!valid || oc < best || (oc == best && (oa < ba || (oa == ba && ob < bb))))) valid = true, best = oc, ba = oa, bb = ob;
    }
    int32_t mid_l;
    if (!valid) {
      mid_l = it.f + it.c / 2;  // all centroids coincide
    } else {
      // the host's std::partition (see k_part_rank): the k-th right-goer left of mid <-> the k-th left-goer from the right
      const bool go_left = in && bin[ba] <= bb;
      const int32_t nleft = __popc(__ballot_sync(0xffffffffu, go_left));
      const bool mis_l = in && (int)lane < it.f + nleft && !go_left, mis_r = (int)lane >= it.f + nleft && go_left;
      const uint32_t ml = __ballot_sync(0xffffffffu, mis_l), mr = __ballot_sync(0xffffffffu, mis_r), below = (1u << lane) - 1u;
      const int k = mis_l ? __popc(ml & below) : __popc(mr & ~below & ~(1u << lane));
      if (mis_l) s_slot[wib][16 + k] = lane;
      if (mis_r) s_slot[wib][k] = lane;
      __syncwarp();
      const uint32_t dest = mis_l ? s_slot[wib][k] : (mis_r ? s_slot[wib][16 + k] : lane);
      __syncwarp();
      s_prim[wib][dest] = p;
      for (int a = 0; a < 9; a++) s_val[wib][dest][a] = v[a];
      __syncwarp();
      p = s_prim[wib][lane];
      for (int a = 0; a < 9; a++) v[a] = s_val[wib][lane][a];
      __syncwarp();
      mid_l = it.f + nleft;
    }
    const int32_t id = (int32_t)(2u * (sn.first + (uint32_t)mid_l) - 1u);
    if (lane == 0u) {
      b2.box[id] = nb, b2.first[id] = gfirst, b2.count[id] = (uint32_t)it.c;
      link_node(b2, id, it.parent, it.side, root_id);
    }
    inner++;
    stack[sp++] = Item{mid_l, it.f + it.c - mid_l, id, 1};
    stack[sp++] = Item{it.f, mid_l - it.f, id, 0};
  }
  if (lane < sn.count) prim[sn.first + lane] = p;
  if (lane == 0u && inner) atomicAdd(counters + 3, inner);
}

// The collapse plan of pt_build.cpp:449-526, bottom-up: a thread starts at a leaf and climbs while it is the second of
// two children to arrive at the parent.  Costs are stored as float, temporaries are double, like the host's.
__device__ void plan_inner(const B2Dev &b2, int32_t n, double c_n, float *cost, uint8_t *split) {
  const double area = box_area(b2.box[n]);
  const float *L = cost + (size_t)b2.left[n] * 8, *R = cost + (size_t)b2.right[n] * 8;
  float l[7], r[7];
  for (int i = 0; i < 7; i++) l[i] = __ldcg(L + i), r[i] = __ldcg(R + i);
  double D[9];
  uint8_t K[9];
  for (int j = 2; j <= 8; j++) {
    D[j] = 1.7976931348623157e308, K[j] = 1;
    for (int k = 1; k < j; k++) {
      const double v = (double)l[k - 1] + (double)r[j - k - 1];
      if (v < D[j]) D[j] = v, K[j] = (uint8_t)k;
    }
  }
  const uint32_t count = b2.count[n];
  const double c_leaf = count <= (uint32_t)kLeafMax ? area * (double)count * 1.0 : 1.7976931348623157e308;
  const double c_inner = area * c_n + D[8];
  float *C = cost + (size_t)n * 8;
  uint8_t *S = split + (size_t)n * 8;
  C[0] = (float)(c_inner < c_leaf ? c_inner : c_leaf);
  S[7] = K[8];
  for (int i = 2; i <= 7; i++) {
    if (D[i] < (double)C[i - 2]) C[i - 1] = (float)D[i], S[i - 1] = K[i];
    else C[i - 1] = C[i - 2], S[i - 1] = 0;
  }
}
__global__ void k_plan(B2Dev b2, uint32_t n_ids, double c_n, float *cost, uint8_t *split, uint32_t *arrive) {
  const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n_ids || b2.count[id] == 0u || b2.left[id] >= 0) return;
  const float leaf_cost = (float)(box_area(b2.box[id]) * (double)b2.count[id] * 1.0);
  for (int i = 0; i < 8; i++) cost[(size_t)id * 8 + i] = leaf_cost;
  int32_t n = (int32_t)id;
  for (;;) {
    const int32_t p = b2.parent[n];
    if (p < 0) return;
    __threadfence();
    if (atomicAdd(arrive + p, 1u) == 0u) return;  // the sibling's subtree is still being planned
    __threadfence();
    plan_inner(b2, p, c_n, cost, split);
    n = p;
  }
}

// Wide structure, one level per launch pair: the children of every node of the level (pt_build.cpp: plan_children, left
// before right), then — after two exclusive scans give each node its first inner child and first triangle record — the
// WNode records in breadth-first order (gen_structure's layout: inner children consecutive in child order) and the next
// level's node list.  A binary node is a leaf of the wide tree exactly when it has <= 3 triangles (a binary leaf; an inner
// binary node has >= 4 and its c_leaf is infinite), so WNode's count rule holds for these trees too.
__global__ void k_wide_children(const int32_t *lvl, uint32_t count, B2Dev b2, const uint8_t *split, int32_t *ch, uint32_t *n_inner, uint32_t *n_tris) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int32_t n = lvl[i];
  int32_t c[8];
  int nch = 0;
  if (b2.left[n] < 0) {
    c[nch++] = n;  // a mesh of <= 3 live triangles: a root with one leaf
  } else {
    int32_t st_node[16], st_slots[16];
    int sp = 0;
    const int k = split[(size_t)n * 8 + 7];
    st_node[sp] = b2.right[n], st_slots[sp++] = 8 - k;
    st_node[sp] = b2.left[n], st_slots[sp++] = k;
    while (sp > 0) {
      const int32_t x = st_node[--sp];
      const int s = st_slots[sp];
      if (b2.left[x] < 0 || s == 1) {
        c[nch++] = x;
        continue;
      }
      const int kk = split[(size_t)x * 8 + s - 1];
      if (kk == 0) {
        st_node[sp] = x, st_slots[sp++] = s - 1;
      } else {
        st_node[sp] = b2.right[x], st_slots[sp++] = s - kk;
        st_node[sp] = b2.left[x], st_slots[sp++] = kk;
      }
    }
  }
  uint32_t ni = 0u, nt = 0u;
  for (int q = 0; q < 8; q++) {
    ch[(size_t)i * 8 + q] = q < nch ? c[q] : -1;
    if (q < nch) {
      const uint32_t cnt = b2.count[c[q]];
      if (cnt > (uint32_t)kLeafMax) ni++;
      else nt += cnt;
    }
  }
  n_inner[i] = ni, n_tris[i] = nt;
}
__global__ void k_wide_write(const int32_t *lvl, uint32_t count, const int32_t *ch, B2Dev b2, const uint32_t *n_inner, const uint32_t *n_tris,
                             const uint32_t *cbase, const uint32_t *tbase, uint32_t level_first, uint32_t next_first, uint32_t tri_first, WNode *wn,
                             int32_t *lvl_next, uint32_t *totals) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  WNode w;
  w.child_base = next_first + cbase[i];
  w.tri_base = tri_first + tbase[i];
  uint32_t r = 0u;
  for (int q = 0; q < 8; q++) {
    const int32_t x = ch[(size_t)i * 8 + q];
    w.child_lo[q] = x < 0 ? 0u : b2.first[x];
    w.child_cnt[q] = x < 0 ? 0u : b2.count[x];
    if (x >= 0 && w.child_cnt[q] > (uint32_t)kLeafMax) lvl_next[cbase[i] + r++] = x;
  }
  wn[level_first + i] = w;
  if (i == count - 1u) totals[0] = cbase[i] + n_inner[i], totals[1] = tbase[i] + n_tris[i];
}

// ---- host side ----------------------------------------------------------------------------------------------------
// The wide tree's structure from the live counts alone.  Binary tree = the reference's own (split at size / 2 while
// size > 4, bvh.rs:19-27,55-56) with every range measured in LIVE triangles (R = live rank of a DFS position); ranges
// with <= 3 live triangles are leaves, a reference leaf that still holds 4 live ones is halved once more.  A wide node
// takes up to three binary levels; a split with an empty side costs no level.  Breadth-first numbering: a node's inner
// children get consecutive ids, every level is a contiguous id range.
struct Item {
  uint32_t ref_lo, ref_hi, live_lo, live_hi;
  int32_t depth;  // reference depth; -1 = below a reference leaf (split by live count)
};
struct Structure {
  std::vector<uint32_t> quads;  // first live rank of every reference leaf that holds 4 live triangles (see k_pair_quads)
  std::vector<WNode> nodes;
  std::vector<uint32_t> level_first;  // level l = ids [level_first[l], level_first[l + 1])
  uint32_t n_tri_records = 0;
};

void expand(const Item &it, int levels, const std::vector<uint32_t> &R, std::vector<Item> &out, std::vector<uint32_t> &quads) {
  const uint32_t live = it.live_hi - it.live_lo;
  if (live == 0u) return;
  if (live <= 3u || levels == 0) {
    out.push_back(it);
    return;
  }
  Item l = it, r = it;
  const uint32_t rsize = it.ref_hi - it.ref_lo;
  if (it.depth >= 0 && rsize > 4u && it.depth < 25) {
    const uint32_t mid = it.ref_lo + rsize / 2u;
    l.ref_hi = mid, r.ref_lo = mid;
    l.depth = r.depth = it.depth + 1;
    l.live_hi = r.live_lo = R[mid];
  } else {
    if (it.depth >= 0 && live == 4u) quads.push_back(it.live_lo);
    const uint32_t lm = it.live_lo + live / 2u;
    l.depth = r.depth = -1;
    l.live_hi = r.live_lo = lm;
  }
  if (l.live_hi == l.live_lo) expand(r, levels, R, out, quads);
  else if (r.live_hi == r.live_lo) expand(l, levels, R, out, quads);
  else expand(l, levels - 1, R, out, quads), expand(r, levels - 1, R, out, quads);
}

Structure gen_structure(uint32_t n, const std::vector<uint32_t> &R) {
  Structure st;
  std::vector<Item> queue{Item{0u, n, 0u, R[n], 0}};
  st.level_first.push_back(0u);
  size_t level_end = 1;
  std::vector<Item> ch;
  for (size_t qi = 0; qi < queue.size(); qi++) {
    if (qi == level_end) {
      st.level_first.push_back((uint32_t)qi);
      level_end = queue.size();
    }
    const Item it = queue[qi];
    ch.clear();
    if (it.live_hi - it.live_lo <= 3u) ch.push_back(it);  // a mesh of <= 3 live triangles: a root with one leaf
    else expand(it, 3, R, ch, st.quads);
    WNode w;
    memset(&w, 0, sizeof(w));
    w.child_base = (uint32_t)queue.size();
    w.tri_base = st.n_tri_records;
    for (size_t c = 0; c < ch.size(); c++) {
      const uint32_t live = ch[c].live_hi - ch[c].live_lo;
      w.child_lo[c] = ch[c].live_lo;
      w.child_cnt[c] = live;
      if (live > 3u) queue.push_back(ch[c]);
      else st.n_tri_records += live;
    }
    st.nodes.push_back(w);
  }
  st.level_first.push_back((uint32_t)queue.size());
  return st;
}

// nodes / leaves / depth of the reference tree (they depend on n only)
void ref_counts(uint64_t n, int depth, int64_t &nodes, int64_t &leaves, int32_t &max_depth, std::unordered_map<uint64_t, std::pair<int64_t, int64_t>> &memo) {
  max_depth = std::max(max_depth, depth);
  if (n <= 4 || depth >= 25) {
    nodes += 1, leaves += 1;
    return;
  }
  if (depth < 20) {  // memoised by size where the depth cap cannot interfere (n < 2^27)
    auto f = memo.find(n);
    if (f != memo.end()) {
      nodes += f->second.first, leaves += f->second.second;
      int32_t d = depth;
      for (uint64_t s = n; s > 4; s = s - s / 2) d++;
      max_depth = std::max(max_depth, d);
      return;
    }
  }
  int64_t a = 1, b = 0;
  ref_counts(n / 2, depth + 1, a, b, max_depth, memo);
  ref_counts(n - n / 2, depth + 1, a, b, max_depth, memo);
  if (depth < 20) memo[n] = {a, b};
  nodes += a, leaves += b;
}

double ms_between(std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
  return std::chrono::duration<double, std::milli>(b - a).count();
}

uint32_t widest_level(const std::vector<uint32_t> &level_first) {
  uint32_t widest = 0;
  for (size_t l = 0; l + 1 < level_first.size(); l++) widest = std::max(widest, level_first[l + 1] - level_first[l]);
  return widest;
}
size_t scan_temp_bytes(uint32_t items) {
  size_t bytes = 0;
  CKB(cub::DeviceScan::ExclusiveSum(nullptr, bytes, (uint32_t *)nullptr, (uint32_t *)nullptr, (int)items, nullptr));
  return bytes;
}
// arena bytes emit_wide takes for a wide tree of this shape (level l = ids [level_first[l], level_first[l + 1]))
size_t emit_need(const std::vector<uint32_t> &level_first) {
  const uint32_t widest = widest_level(level_first);
  return Arena::need(level_first.back(), sizeof(Box)) + Arena::need(6, 4) + Arena::need(1, sizeof(int)) + 4 * Arena::need(widest, 4) +
         Arena::need(scan_temp_bytes(widest), 1);
}

// Boxes, frames, slots, quantised nodes and triangle records of the wide tree described by `wn` (breadth-first
// structural ids, level l = [level_first[l], level_first[l + 1])) — shared by both device step-2 builders.
void emit_wide(Arena &a, cudaStream_t stream, const WNode *wn, const uint32_t *live, const std::vector<uint32_t> &level_first, uint32_t n_tri_records,
               const float *tris, const int32_t *order, Buf<float4> &d_nodes, Buf<float4> &d_tri48, MeshBuild &m) {
  const uint32_t n_nodes = level_first.back(), n_levels = (uint32_t)level_first.size() - 1, widest = widest_level(level_first);
  const size_t scan_bytes = scan_temp_bytes(widest);
  Box *d_box = a.get<Box>(n_nodes);
  d_nodes.alloc((size_t)n_nodes * 5), d_tri48.alloc((size_t)std::max(n_tri_records, 1u) * 3);
  float *d_root = a.get<float>(6);
  int *d_err = a.get<int>(1);
  CKB(cudaMemsetAsync(d_err, 0, sizeof(int), stream));
  for (uint32_t l = n_levels; l-- > 0;) {
    const uint32_t first = level_first[l], count = level_first[l + 1] - first;
    k_boxes_level<<<blocks_for(count), kThreads, 0, stream>>>(wn, first, count, live, tris, d_box);
  }
  CKB(cudaGetLastError());
  uint32_t *d_sid[2] = {a.get<uint32_t>(widest), a.get<uint32_t>(widest)}, *d_cnt = a.get<uint32_t>(widest), *d_cbase = a.get<uint32_t>(widest);
  uint8_t *d_scan = a.get<uint8_t>(scan_bytes);
  CKB(cudaMemsetAsync(d_sid[0], 0, 4, stream));  // level 0: final position 0 holds structural node 0
  for (uint32_t l = 0; l < n_levels; l++) {
    const uint32_t first = level_first[l], count = level_first[l + 1] - first;
    k_inner_count<<<blocks_for(count), kThreads, 0, stream>>>(wn, d_sid[l & 1], count, d_cnt);
    size_t sb = scan_bytes;
    CKB(cub::DeviceScan::ExclusiveSum(d_scan, sb, d_cnt, d_cbase, (int)count, stream));
    k_emit_level<<<blocks_for(count), kThreads, 0, stream>>>(wn, d_sid[l & 1], first, count, d_cbase, level_first[l + 1], d_sid[(l + 1) & 1], live, tris,
                                                        order, d_box, d_nodes.p, d_tri48.p, d_root, d_err);
    CKB(cudaGetLastError());
  }
  int err = 0;
  float root[6];
  CKB(cudaMemcpyAsync(&err, d_err, sizeof(int), cudaMemcpyDeviceToHost, stream));
  CKB(cudaMemcpyAsync(root, d_root, sizeof(root), cudaMemcpyDeviceToHost, stream));
  CKB(cudaStreamSynchronize(stream));
  if (err) throw std::runtime_error("mesh extent too large for the quantised BVH frame");
  for (int a3 = 0; a3 < 3; a3++) m.root_lo[a3] = root[a3], m.root_hi[a3] = root[3 + a3];
  m.wide_depth = (int32_t)n_levels - 1;
}

// DevBuildMode::Sah, step 2 up to the WNode records: binary SAH tree (large nodes level by level, then one warp per small
// subtree), collapse plan, wide structure.
struct SahTree {
  std::unique_ptr<Arena> work, wide;  // binary tree + plan; wide structure + room for emit_wide
  const WNode *wn = nullptr;
  const uint32_t *live = nullptr;  // triangle (original index) at every position of the final permutation
  std::vector<uint32_t> level_first;
  int sah_levels = 0;
  double sah_ms = 0, plan_ms = 0, structure_ms = 0;
};

SahTree build_sah(uint32_t n, uint32_t nl, const uint8_t *d_dead, const float *d_tbox, cudaStream_t stream) {
  auto now = [] { return std::chrono::steady_clock::now(); };
  const auto t0 = now();
  SahTree r;
  const uint32_t max_open = nl / (kWarpMax + 1u) + 1u;  // an open node holds > kWarpMax triangles
  const size_t n_ids = 2 * (size_t)nl;
  size_t sel_bytes = 0;
  CKB(cub::DeviceSelect::Flagged(nullptr, sel_bytes, (OpenNode *)nullptr, (uint8_t *)nullptr, (OpenNode *)nullptr, (uint32_t *)nullptr,
                                 (int)(2 * max_open), stream));
  const size_t temp_bytes = std::max(scan_temp_bytes(n), sel_bytes);
  r.work.reset(new Arena(2 * Arena::need(n, 4) + 2 * Arena::need(nl, 4) + Arena::need((size_t)n * 3, 4) + Arena::need(n_ids, sizeof(Box)) +
                         5 * Arena::need(n_ids, 4) + Arena::need(n_ids * 8, 4) + Arena::need(n_ids * 8, 1) + Arena::need(n_ids, 4) +
                         4 * Arena::need(max_open, sizeof(OpenNode)) + Arena::need(2 * max_open, 1) + 2 * Arena::need(max_open, 4) +
                         Arena::need(max_open, sizeof(SplitDev)) + Arena::need((size_t)max_open * kNodeBinWords, 4) + Arena::need(nl, sizeof(SmallNode)) +
                         Arena::need(10, 4) + Arena::need(1, 4) + Arena::need(temp_bytes, 1) + 8192));
  Arena &a = *r.work;
  uint32_t *d_flag = a.get<uint32_t>(n), *d_scan = a.get<uint32_t>(n), *d_prim = a.get<uint32_t>(nl), *d_tmp = a.get<uint32_t>(nl);
  float *d_pcen = a.get<float>((size_t)n * 3);
  B2Dev b2;
  b2.box = a.get<Box>(n_ids), b2.first = a.get<uint32_t>(n_ids), b2.count = a.get<uint32_t>(n_ids);
  b2.left = a.get<int32_t>(n_ids), b2.right = a.get<int32_t>(n_ids), b2.parent = a.get<int32_t>(n_ids);
  float *d_cost = a.get<float>(n_ids * 8);
  uint8_t *d_split = a.get<uint8_t>(n_ids * 8);
  uint32_t *d_arrive = a.get<uint32_t>(n_ids);
  OpenNode *d_open[2] = {a.get<OpenNode>(max_open), a.get<OpenNode>(max_open)}, *d_cand = a.get<OpenNode>(2 * max_open);
  uint8_t *d_cand_flag = a.get<uint8_t>(2 * max_open);
  uint32_t *d_off = a.get<uint32_t>(max_open), *d_cnt = a.get<uint32_t>(max_open);
  SplitDev *d_splits = a.get<SplitDev>(max_open);
  uint32_t *d_bins = a.get<uint32_t>((size_t)max_open * kNodeBinWords);
  SmallNode *d_small = a.get<SmallNode>(nl);
  uint32_t *d_counters = a.get<uint32_t>(10);  // next level's nodes, next level's triangles, small nodes, inner nodes, root centroid keys
  int32_t *d_root = a.get<int32_t>(1);
  uint8_t *d_temp = a.get<uint8_t>(temp_bytes);

  CKB(cudaMemsetAsync(b2.count, 0, n_ids * 4, stream));
  CKB(cudaMemsetAsync(d_arrive, 0, n_ids * 4, stream));
  uint32_t counters[10] = {0u, 0u, nl <= kWarpMax ? 1u : 0u, 0u, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
  CKB(cudaMemcpy(d_counters, counters, sizeof(counters), cudaMemcpyHostToDevice));
  if (nl <= kWarpMax) {
    const SmallNode root{0u, nl, -1, 0};
    CKB(cudaMemcpy(d_small, &root, sizeof(root), cudaMemcpyHostToDevice));
  }
  size_t tb = temp_bytes;
  k_live_flags<<<blocks_for(n), kThreads, 0, stream>>>(d_dead, n, d_flag);
  CKB(cub::DeviceScan::ExclusiveSum(d_temp, tb, d_flag, d_scan, (int)n, stream));
  k_live_scatter<<<blocks_for(n), kThreads, 0, stream>>>(d_flag, d_scan, d_tbox, n, d_prim, d_pcen);
  CKB(cudaGetLastError());

  // large nodes, one level per pass
  uint32_t n_open = 0, total = 0, n_small = counters[2];
  if (nl > kWarpMax) {
    k_root_cb<<<blocks_for(nl), kThreads, 0, stream>>>(d_prim, d_pcen, nl, d_counters + 4);
    k_root_open<<<1, 1, 0, stream>>>(d_counters + 4, nl, d_open[0], d_off);
    CKB(cudaGetLastError());
    n_open = 1, total = nl;
  }
  int cur = 0;
  while (n_open > 0) {
    r.sah_levels++;
    const size_t words = (size_t)n_open * kNodeBinWords;
    k_bins_init<<<blocks_for(words), kThreads, 0, stream>>>(d_bins, words);
    k_bin<<<blocks_for(total), kThreads, 0, stream>>>(d_open[cur], d_off, n_open, total, d_prim, d_tbox, d_pcen, d_bins);
    CKB(cudaMemsetAsync(d_counters, 0, 8, stream));
    k_sweep<<<blocks_for(n_open), kThreads, 0, stream>>>(d_open[cur], n_open, d_bins, d_splits, b2, d_root, d_cand, d_cand_flag, d_small, d_counters);
    k_part_flag<<<blocks_for(total), kThreads, 0, stream>>>(d_open[cur], d_off, n_open, total, d_prim, d_pcen, d_splits, d_flag);
    CKB(cudaGetLastError());
    tb = temp_bytes;
    CKB(cub::DeviceScan::ExclusiveSum(d_temp, tb, d_flag, d_scan, (int)total, stream));
    k_part_rank<<<blocks_for(total), kThreads, 0, stream>>>(d_open[cur], d_off, n_open, total, d_splits, d_flag, d_scan, d_tmp);
    k_part_swap<<<blocks_for(total), kThreads, 0, stream>>>(d_open[cur], d_off, n_open, total, d_splits, d_flag, d_scan, d_tmp, d_prim);
    CKB(cudaGetLastError());
    tb = temp_bytes;
    CKB(cub::DeviceSelect::Flagged(d_temp, tb, d_cand, d_cand_flag, d_open[cur ^ 1], d_counters, (int)(2 * n_open), stream));
    CKB(cudaMemcpyAsync(counters, d_counters, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CKB(cudaStreamSynchronize(stream));
    cur ^= 1;
    n_open = counters[0], total = counters[1], n_small = counters[2];
    if (n_open > 0) {
      k_open_counts<<<blocks_for(n_open), kThreads, 0, stream>>>(d_open[cur], n_open, d_cnt);
      CKB(cudaGetLastError());
      tb = temp_bytes;
      CKB(cub::DeviceScan::ExclusiveSum(d_temp, tb, d_cnt, d_off, (int)n_open, stream));
    }
  }
  // small nodes: one warp each, whole subtrees
  k_small<<<(n_small + kSmallWarps - 1) / kSmallWarps, 32 * kSmallWarps, 0, stream>>>(d_small, n_small, d_prim, d_tbox, d_pcen, b2, d_root, d_counters);
  CKB(cudaGetLastError());
  int32_t root = -1;
  CKB(cudaMemcpyAsync(counters, d_counters, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
  CKB(cudaMemcpyAsync(&root, d_root, sizeof(root), cudaMemcpyDeviceToHost, stream));
  CKB(cudaStreamSynchronize(stream));
  const uint32_t n_inner = counters[3];
  if (root < 0 || (nl <= (uint32_t)kLeafMax) != (n_inner == 0u)) throw std::runtime_error("pt_build_dev: inconsistent SAH tree");
  const auto t1 = now();

  // collapse plan (PTC_SAH_CN: node cost, as pt_build.cpp)
  const double c_n = getenv("PTC_SAH_CN") ? atof(getenv("PTC_SAH_CN")) : 1.8;
  k_plan<<<blocks_for(n_ids), kThreads, 0, stream>>>(b2, (uint32_t)n_ids, c_n, d_cost, d_split, d_arrive);
  CKB(cudaGetLastError());
  CKB(cudaStreamSynchronize(stream));
  const auto t2 = now();

  // wide structure: at most one wide node per inner binary node (one when the root is a leaf)
  const uint32_t cap = std::max(n_inner, 1u);
  const std::vector<uint32_t> cap_shape{0u, cap};
  r.wide.reset(new Arena(Arena::need(cap, sizeof(WNode)) + 2 * Arena::need(cap, 4) + Arena::need((size_t)cap * 8, 4) + 4 * Arena::need(cap, 4) +
                         Arena::need(scan_temp_bytes(cap), 1) + Arena::need(2, 4) + emit_need(cap_shape) + 8192));
  Arena &w = *r.wide;
  WNode *d_wn = w.get<WNode>(cap);
  int32_t *d_lvl[2] = {w.get<int32_t>(cap), w.get<int32_t>(cap)}, *d_ch = w.get<int32_t>((size_t)cap * 8);
  uint32_t *d_ni = w.get<uint32_t>(cap), *d_nt = w.get<uint32_t>(cap), *d_cb = w.get<uint32_t>(cap), *d_tb = w.get<uint32_t>(cap);
  const size_t scan2 = scan_temp_bytes(cap);
  uint8_t *d_scan2 = w.get<uint8_t>(scan2);
  uint32_t *d_tot = w.get<uint32_t>(2);
  CKB(cudaMemcpyAsync(d_lvl[0], d_root, 4, cudaMemcpyDeviceToDevice, stream));
  r.level_first.assign(1, 0u);
  uint32_t count = 1, tri_first = 0;
  for (int c = 0; count > 0; c ^= 1) {
    const uint32_t first = r.level_first.back(), next_first = first + count;
    if (next_first > cap) throw std::runtime_error("pt_build_dev: wide tree larger than its bound");
    k_wide_children<<<blocks_for(count), kThreads, 0, stream>>>(d_lvl[c], count, b2, d_split, d_ch, d_ni, d_nt);
    CKB(cudaGetLastError());
    size_t sb = scan2;
    CKB(cub::DeviceScan::ExclusiveSum(d_scan2, sb, d_ni, d_cb, (int)count, stream));
    sb = scan2;
    CKB(cub::DeviceScan::ExclusiveSum(d_scan2, sb, d_nt, d_tb, (int)count, stream));
    k_wide_write<<<blocks_for(count), kThreads, 0, stream>>>(d_lvl[c], count, d_ch, b2, d_ni, d_nt, d_cb, d_tb, first, next_first, tri_first, d_wn,
                                                         d_lvl[c ^ 1], d_tot);
    CKB(cudaGetLastError());
    uint32_t tot[2];
    CKB(cudaMemcpyAsync(tot, d_tot, sizeof(tot), cudaMemcpyDeviceToHost, stream));
    CKB(cudaStreamSynchronize(stream));
    r.level_first.push_back(next_first);
    count = tot[0], tri_first += tot[1];
  }
  if (tri_first != nl) throw std::runtime_error("pt_build_dev: wide tree does not hold every live triangle once");
  r.wn = d_wn, r.live = d_prim;
  r.sah_ms = ms_between(t0, t1), r.plan_ms = ms_between(t1, t2), r.structure_ms = ms_between(t2, now());
  return r;
}

}  // namespace

void build_mesh_device(MeshBuild &m, DevMeshBuffers &out, DevBuildTiming *timing, DevBuildMode mode) {
  const int64_t n64 = m.n;
  if (n64 <= 0) throw std::runtime_error("mesh without triangles");
  if (n64 >= ((int64_t)1 << 27)) throw std::runtime_error("mesh too large for the device builder");
  const uint32_t n = (uint32_t)n64;
  auto now = [] { return std::chrono::steady_clock::now(); };
  const auto t0 = now();
  int device = 0;
  CKB(cudaGetDevice(&device));
  cudaStream_t stream = nullptr;  // legacy default stream: the build is a synchronous host call

  // ---- upload
  int sort_levels = 0;  // levels of the reference tree that still have a node to split
  while (sort_levels < 25 && (((uint64_t)n + ((1ull << sort_levels) - 1)) >> sort_levels) > 4ull) sort_levels++;
  size_t temp_bytes = 0;
  {
    cub::DoubleBuffer<unsigned long long> kb(nullptr, nullptr);
    cub::DoubleBuffer<uint32_t> vb(nullptr, nullptr);
    CKB(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, kb, vb, (int)n, 0, 64, stream));
  }
  const size_t segb_count = ((size_t)1 << sort_levels) * 6;
  Arena a1(Arena::need((size_t)n * 12, 4) + Arena::need((size_t)n * 3, 4) + Arena::need((size_t)n * 6, 4) + 2 * Arena::need(n, 4) +
           2 * Arena::need(n, 8) + 2 * Arena::need(n, 1) + Arena::need(n, 4) + Arena::need(segb_count, 4) + Arena::need(temp_bytes, 1) + 4096);
  struct P {
    float *p;
  } d_tris{a1.get<float>((size_t)n * 12)}, d_cen{a1.get<float>((size_t)n * 3)}, d_tbox{a1.get<float>((size_t)n * 6)};
  struct PU {
    uint32_t *p;
  } d_idx[2] = {{a1.get<uint32_t>(n)}, {a1.get<uint32_t>(n)}}, d_segb{a1.get<uint32_t>(segb_count)};
  struct PK {
    unsigned long long *p;
  } d_keys[2] = {{a1.get<unsigned long long>(n)}, {a1.get<unsigned long long>(n)}};
  struct PB {
    uint8_t *p;
  } d_dead{a1.get<uint8_t>(n)}, d_dead_pos{a1.get<uint8_t>(n)}, d_temp{a1.get<uint8_t>(temp_bytes)};
  struct PI {
    int32_t *p;
  } d_order{a1.get<int32_t>(n)};
  CKB(cudaMemcpyAsync(d_tris.p, m.tris.data(), (size_t)n * 48, cudaMemcpyHostToDevice, stream));
  k_tri_prepare<<<blocks_for(n), kThreads, 0, stream>>>(d_tris.p, n, d_cen.p, d_tbox.p, d_idx[0].p, d_dead.p);
  CKB(cudaGetLastError());
  CKB(cudaStreamSynchronize(stream));
  const auto t1 = now();

  // ---- step 1: the reference tree, one level per pass
  int cur = 0;
  for (int L = 0; L <= sort_levels; L++) {
    const size_t segs = (size_t)1 << L;
    k_fill_u32<<<blocks_for(segs * 6), kThreads, 0, stream>>>(d_segb.p, segs * 6, 0xffffffffu, 0u);
    k_level_bounds<<<blocks_for(n), kThreads, 0, stream>>>(d_idx[cur].p, d_tbox.p, n, L, d_segb.p);
    const bool sort = L < sort_levels;
    k_level_keys<<<blocks_for(n), kThreads, 0, stream>>>(d_idx[cur].p, d_cen.p, d_segb.p, n, L, d_dead.p, sort ? d_keys[cur].p : nullptr);
    CKB(cudaGetLastError());
    if (sort) {
      cub::DoubleBuffer<unsigned long long> kb(d_keys[cur].p, d_keys[cur ^ 1].p);
      cub::DoubleBuffer<uint32_t> vb(d_idx[cur].p, d_idx[cur ^ 1].p);
      size_t tb = temp_bytes;
      CKB(cub::DeviceRadixSort::SortPairs(d_temp.p, tb, kb, vb, (int)n, 0, 32 + L, stream));  // stable, like the host's sort
      if (vb.Current() != d_idx[cur].p) cur ^= 1;  // (keys follow the same selector)
    }
  }
  k_finish_order<<<blocks_for(n), kThreads, 0, stream>>>(d_idx[cur].p, d_dead.p, n, d_order.p, d_dead_pos.p);
  CKB(cudaGetLastError());
  m.dead.resize(n);
  m.order.resize(n);
  std::vector<uint8_t> dead_pos;
  std::vector<uint32_t> idx_host;
  CKB(cudaMemcpyAsync(m.dead.data(), d_dead.p, n, cudaMemcpyDeviceToHost, stream));
  CKB(cudaMemcpyAsync(m.order.data(), d_order.p, (size_t)n * 4, cudaMemcpyDeviceToHost, stream));
  if (mode == DevBuildMode::Median) {  // the host derives the median tree's structure from them
    dead_pos.resize(n), idx_host.resize(n);
    CKB(cudaMemcpyAsync(dead_pos.data(), d_dead_pos.p, n, cudaMemcpyDeviceToHost, stream));
    CKB(cudaMemcpyAsync(idx_host.data(), d_idx[cur].p, (size_t)n * 4, cudaMemcpyDeviceToHost, stream));
  }
  CKB(cudaStreamSynchronize(stream));
  {
    int64_t nodes = 0, leaves = 0;
    int32_t depth = 0;
    std::unordered_map<uint64_t, std::pair<int64_t, int64_t>> memo;
    ref_counts(n, 0, nodes, leaves, depth, memo);
    m.ref_nodes = nodes, m.ref_leaves = leaves, m.ref_depth = depth;
  }
  const auto t2 = now();
  if (mode == DevBuildMode::RefOnly) {  // the caller builds the traversal tree itself (host SAH + collapse) from this dead mask and order
    m.ref_done = true;
    if (timing) {
      timing->upload_ms = ms_between(t0, t1), timing->ref_ms = ms_between(t1, t2), timing->total_ms = ms_between(t0, t2);
      timing->ref_levels = sort_levels + 1;
    }
    return;
  }

  // ---- step 2
  std::vector<uint32_t> R, live_tri;
  if (mode == DevBuildMode::Median) {  // structure on the host (live ranks only), boxes + nodes + triangle records on the device
    R.resize((size_t)n + 1);
    live_tri.reserve(n);
    R[0] = 0;
    for (uint32_t p = 0; p < n; p++) {
      R[p + 1] = R[p] + (dead_pos[p] ? 0u : 1u);
      if (!dead_pos[p]) live_tri.push_back(idx_host[p]);
    }
    m.live = (int64_t)R[n];
  } else {
    m.live = (int64_t)std::count(m.dead.begin(), m.dead.end(), (uint8_t)0);
  }
  Buf<float4> d_normals(n);
  k_normals<<<blocks_for(n), kThreads, 0, stream>>>(d_tris.p, d_order.p, n, d_normals.p);
  CKB(cudaGetLastError());
  if (m.live == 0) {
    // every triangle is unreachable in the reference: an empty root (no child bits) never reports a hit (as pt_build.cpp)
    m.nodes.assign(1, Node8());
    const uint32_t e = 127u | (127u << 8) | (127u << 16), one = 1u, inv = 0xffffffffu;
    float fe, fone, finv;
    memcpy(&fe, &e, 4), memcpy(&fone, &one, 4), memcpy(&finv, &inv, 4);
    m.nodes[0].q[0] = make_float4(0, 0, 0, fe);
    m.nodes[0].q[1] = make_float4(fone, 0.0f, 0.0f, 0.0f);
    m.nodes[0].q[2] = make_float4(finv, finv, finv, finv);
    m.nodes[0].q[3] = make_float4(finv, finv, 0.0f, 0.0f);
    m.nodes[0].q[4] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    Tri48 z;
    z.t[0] = z.t[1] = z.t[2] = make_float4(0, 0, 0, 0);
    m.tri48.assign(1, z);
    for (int a = 0; a < 3; a++) m.root_lo[a] = 1.0f, m.root_hi[a] = -1.0f;
    m.wide_depth = 0;
    m.normals.resize(n);
    CKB(cudaMemcpy(m.normals.data(), d_normals.p, (size_t)n * 16, cudaMemcpyDeviceToHost));
    Buf<float4> d_nodes(5), d_tri48(3);
    CKB(cudaMemcpy(d_nodes.p, m.nodes.data(), 80, cudaMemcpyHostToDevice));
    CKB(cudaMemcpy(d_tri48.p, m.tri48.data(), 48, cudaMemcpyHostToDevice));
    out.nodes = d_nodes.take(), out.tris = d_tri48.take(), out.normals = d_normals.take(), out.device = device;
    m.built = true;
    return;
  }
  uint32_t n_nodes = 0, n_tri_records = 0;
  Buf<float4> d_nodes, d_tri48;
  auto t3 = now();
  if (mode == DevBuildMode::Median) {
    const Structure st = gen_structure(n, R);
    n_nodes = (uint32_t)st.nodes.size(), n_tri_records = st.n_tri_records;
    t3 = now();
    Arena a2(Arena::need(n_nodes, sizeof(WNode)) + Arena::need(live_tri.size(), 4) + Arena::need(st.quads.size(), 4) + emit_need(st.level_first) + 8192);
    struct PW {
      WNode *p;
    } d_wn{a2.get<WNode>(n_nodes)};
    PU d_live{a2.get<uint32_t>(live_tri.size())};
    CKB(cudaMemcpyAsync(d_wn.p, st.nodes.data(), (size_t)n_nodes * sizeof(WNode), cudaMemcpyHostToDevice, stream));
    CKB(cudaMemcpyAsync(d_live.p, live_tri.data(), live_tri.size() * 4, cudaMemcpyHostToDevice, stream));
    if (!st.quads.empty()) {
      PU d_quads{a2.get<uint32_t>(st.quads.size())};
      CKB(cudaMemcpyAsync(d_quads.p, st.quads.data(), st.quads.size() * 4, cudaMemcpyHostToDevice, stream));
      k_pair_quads<<<blocks_for(st.quads.size()), kThreads, 0, stream>>>(d_quads.p, (uint32_t)st.quads.size(), d_live.p, d_tris.p);
      CKB(cudaGetLastError());
    }
    emit_wide(a2, stream, d_wn.p, d_live.p, st.level_first, n_tri_records, d_tris.p, d_order.p, d_nodes, d_tri48, m);
  } else {
    SahTree sah = build_sah(n, (uint32_t)m.live, d_dead.p, d_tbox.p, stream);
    n_nodes = sah.level_first.back(), n_tri_records = (uint32_t)m.live;
    t3 = now();
    emit_wide(*sah.wide, stream, sah.wn, sah.live, sah.level_first, n_tri_records, d_tris.p, d_order.p, d_nodes, d_tri48, m);
    if (timing) {
      timing->sah_ms = sah.sah_ms, timing->plan_ms = sah.plan_ms, timing->sah_levels = sah.sah_levels;
      timing->structure_ms = sah.structure_ms;
    }
  }
  const auto t4 = now();

  // ---- host copies (ptc_scene_mesh_info, replicas of ptc_multi_create)
  m.nodes.resize(n_nodes);
  m.tri48.resize(std::max(n_tri_records, 1u));
  m.normals.resize(n);
  CKB(cudaMemcpyAsync(m.nodes.data(), d_nodes.p, (size_t)n_nodes * 80, cudaMemcpyDeviceToHost, stream));
  CKB(cudaMemcpyAsync(m.tri48.data(), d_tri48.p, m.tri48.size() * 48, cudaMemcpyDeviceToHost, stream));
  CKB(cudaMemcpyAsync(m.normals.data(), d_normals.p, (size_t)n * 16, cudaMemcpyDeviceToHost, stream));
  CKB(cudaStreamSynchronize(stream));
  out.nodes = d_nodes.take(), out.tris = d_tri48.take(), out.normals = d_normals.take(), out.device = device;
  m.built = true;
  const auto t5 = now();
  if (timing) {
    timing->upload_ms = ms_between(t0, t1), timing->ref_ms = ms_between(t1, t2), timing->emit_ms = ms_between(t3, t4);
    if (mode == DevBuildMode::Median) timing->structure_ms = ms_between(t2, t3);
    timing->download_ms = ms_between(t4, t5), timing->total_ms = ms_between(t0, t5);
    timing->ref_levels = sort_levels + 1;
  }
}

}  // namespace pt
