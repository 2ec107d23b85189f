// lt_bvh.cu -- device-side BVH construction (SURVEY.md 8(f)-1): an LBVH (Morton order + Karras 2012
// hierarchy) or a PLOC tree (Meister & Bittner 2018, bottom-up clustering over the same Morton order), emitted in
// the REFERENCE's flattened layout -- 32-byte LinearBVHNode in DFS order with the first child adjacent, ordered
// 76-byte Primitive array, LightContainer -- so every kernel, the CPU oracle and even the reference's own renderer
// can traverse it unchanged.
//
// These are opt-in alternatives to the host builder (lens_trace_b200/host/acceleration_structure_explicit.cpp,
// which restates the reference's median split).  The trees differ from the median-split tree, so hit ids on
// exact ties can differ; every parity test therefore compares results ON THE SAME BUFFERS.
//
//   1. centroid of each triangle's bounding box (as src/model.cpp:49-53), scene bounds (atomics on
//      order-preserving integer images of the floats)
//   2. 63-bit Morton code (21 bits per axis); key = (code, primitive index) made unique by sorting pairs with
//      a stable radix sort (cub) -- ties keep input order
//   3. the hierarchy over the sorted leaves: inner node ids [0, n-1), root 0; children, parents, leaf counts,
//      boxes and split axes
//      LBVH: internal node i covers a key range found by binary search on common-prefix lengths (Karras);
//            boxes bottom-up, the second arrival at a node proceeds (atomic flag per internal node)
//      PLOC: clusters merge with their mutual nearest neighbour within PLOC_RADIUS positions, one iteration per
//            launch group, until one cluster is left (DESIGN.md section 4)
//   4. DFS index and leaf rank of every node from the leaf counts of the first siblings on its parent chain; the
//      same walk yields the depth (stack bound)
//   5. emit LinearBVHNode[], ordered Primitive[], LightContainer; then the usual re-flatten
#include "lt_device.cuh"
#include "lt_internal.h"

#include <cub/device/device_radix_sort.cuh>
#include <string.h>

#include <algorithm>
#include <vector>

namespace {

__device__ __forceinline__ unsigned orderedBits(float f) {  // monotonic float -> uint
  unsigned u = (unsigned)__float_as_int(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float fromOrderedBits(unsigned u) {
  return __int_as_float((int)((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u));
}

// PLOC search radius: a cluster looks for its nearest neighbour among the PLOC_RADIUS clusters on each side of it
// in the current cluster array.  Chosen from 8, 16 and 32 on the synthetic meshes (profiles/ploc_radius_sweep.txt;
// B200 at its 1000 W power limit; build = H2D + build + re-flatten, best of 3; box tests per GI ray, 1080p):
//   radius   1 M triangles: build ms, box tests/ray, SAH cost    5 M triangles: build ms, box tests/ray, SAH cost
//     8        13.0   32.64   25.84                                44.6   34.73   28.47
//    16        12.3   33.23   26.33                                44.6   35.38   29.02
//    32        14.1   33.38   26.52                                45.3   35.29   28.98
// The build time does not depend on it measurably; the smallest radius gives the best trees here.
constexpr int PLOC_RADIUS = 8;
constexpr int PLOC_BLOCK = 256;

struct LtBox {
  float lo[3], hi[3];
};

struct BuildScratch {
  unsigned* bounds;             // [6] ordered-int min xyz, max xyz of the centroids
  unsigned long long* keys[2];  // Morton keys (double buffer for the sort)
  int* order[2];                // primitive indices (double buffer)
  int2* children;               // internal node -> (first, second child); >= 0 internal, < 0 -> ~leaf position
  int* parent;                  // [0, n-1): parent of internal i; [n-1, 2n-1): parent of leaf position j at n-1+j
  int* leaves;                  // internal node -> number of leaves below it
  float* boxes;                 // 6 floats per internal node
  int* axis;                    // split axis of internal nodes
  int* dfsIndex;                // DFS index of internal nodes [0,n-1) and leaves [n-1, 2n-1)
  int* leafRank;                // leaf position j -> its place in the ordered primitives
  int* maxDepth;
  int* emissiveCount;           // large scenes: emissive primitives found, and the first 4096 of them
  int* emissive;
  int* flags;                   // LBVH: arrival counters
  // PLOC: the cluster array (node reference as in `children`, box) double-buffered, and per-iteration flags
  int* clusterNode[2];
  LtBox* clusterBox[2];
  int* nn;         // position of each cluster's nearest neighbour
  int* merge;      // 1: the cluster merges with its neighbour and the new node takes its position
  int* keep;       // 0: the cluster merges into the one at a lower position
  int* mergeRank;  // exclusive scans of merge and keep
  int* newPos;
  int* newCount;   // clusters after the iteration
  void* sortTemp;
  size_t sortBytes;
  void* scanTemp;
  size_t scanBytes;
};

// Carves the scratch buffers out of `base` (nullptr: only measures) and returns the bytes used.
size_t carve_scratch(BuildScratch& S, char* base, int n, LtBvhBuilder builder) {
  size_t used = 0;
  auto take = [&](size_t bytes) {
    char* r = base ? base + used : nullptr;
    used += (bytes + 255) & ~(size_t)255;
    return (void*)r;
  };
  const bool ploc = builder == LT_BVH_PLOC;
  memset(&S, 0, sizeof S);
  S.bounds = (unsigned*)take(6 * sizeof(unsigned));
  S.maxDepth = (int*)take(sizeof(int));
  S.emissiveCount = (int*)take(sizeof(int));
  S.emissive = (int*)take(4096 * sizeof(int));
  S.keys[0] = (unsigned long long*)take(sizeof(unsigned long long) * n);
  S.keys[1] = (unsigned long long*)take(sizeof(unsigned long long) * n);
  S.order[0] = (int*)take(sizeof(int) * n);
  S.order[1] = (int*)take(sizeof(int) * n);
  S.children = (int2*)take(sizeof(int2) * n);
  S.leaves = (int*)take(sizeof(int) * n);
  S.parent = (int*)take(sizeof(int) * 2 * n);
  S.boxes = (float*)take(sizeof(float) * 6 * n);
  S.axis = (int*)take(sizeof(int) * n);
  S.dfsIndex = (int*)take(sizeof(int) * 2 * n);
  S.leafRank = (int*)take(sizeof(int) * n);
  if (ploc) {
    for (int b = 0; b < 2; b++) {
      S.clusterNode[b] = (int*)take(sizeof(int) * n);
      S.clusterBox[b] = (LtBox*)take(sizeof(LtBox) * n);
    }
    S.nn = (int*)take(sizeof(int) * n);
    S.merge = (int*)take(sizeof(int) * n);
    S.keep = (int*)take(sizeof(int) * n);
    S.mergeRank = (int*)take(sizeof(int) * n);
    S.newPos = (int*)take(sizeof(int) * n);
    S.newCount = (int*)take(sizeof(int));
    S.scanBytes = lt_scan_temp_bytes(n);
    S.scanTemp = take(S.scanBytes);
  } else {
    S.flags = (int*)take(sizeof(int) * n);
  }
  cub::DoubleBuffer<unsigned long long> kb(S.keys[0], S.keys[1]);
  cub::DoubleBuffer<int> vb(S.order[0], S.order[1]);
  cub::DeviceRadixSort::SortPairs(nullptr, S.sortBytes, kb, vb, n, 0, 63);
  S.sortTemp = take(S.sortBytes);
  return used;
}

__global__ void k_centroid_bounds(const RefPrim* __restrict__ prims, int n, unsigned* bounds) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const RefPrim& p = prims[i];
  for (int k = 0; k < 3; k++) {
    float lo = fminf(fminf(p.a[k], p.b[k]), p.c[k]), hi = fmaxf(fmaxf(p.a[k], p.b[k]), p.c[k]);
    float c = FADD(FMUL(0.5f, lo), FMUL(0.5f, hi));
    atomicMin(&bounds[k], orderedBits(c));
    atomicMax(&bounds[3 + k], orderedBits(c));
  }
}

__device__ __forceinline__ unsigned long long spread21(unsigned v) {  // 21 bits -> every third bit
  unsigned long long x = v & 0x1fffffull;
  x = (x | x << 32) & 0x1f00000000ffffull;
  x = (x | x << 16) & 0x1f0000ff0000ffull;
  x = (x | x << 8) & 0x100f00f00f00f00full;
  x = (x | x << 4) & 0x10c30c30c30c30c3ull;
  x = (x | x << 2) & 0x1249249249249249ull;
  return x;
}

__global__ void k_morton(const RefPrim* __restrict__ prims, int n, const unsigned* __restrict__ bounds,
                         unsigned long long* keys, int* order) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const RefPrim& p = prims[i];
  unsigned q[3];
  for (int k = 0; k < 3; k++) {
    float lo = fminf(fminf(p.a[k], p.b[k]), p.c[k]), hi = fmaxf(fmaxf(p.a[k], p.b[k]), p.c[k]);
    float c = FADD(FMUL(0.5f, lo), FMUL(0.5f, hi));
    float mn = fromOrderedBits(bounds[k]), mx = fromOrderedBits(bounds[3 + k]);
    float ext = mx - mn;
    float u = ext > 0.0f ? (c - mn) / ext : 0.0f;
    q[k] = (unsigned)fminf(fmaxf(u * 2097152.0f, 0.0f), 2097151.0f);
  }
  keys[i] = spread21(q[0]) << 2 | spread21(q[1]) << 1 | spread21(q[2]);
  order[i] = i;
}

// common-prefix length of the keys at sorted positions i and j; equal codes are separated by position
__device__ __forceinline__ int delta(const unsigned long long* __restrict__ keys, int n, int i, int j) {
  if (j < 0 || j >= n) return -1;
  unsigned long long a = keys[i], b = keys[j];
  if (a == b) return 64 + __clz(i ^ j);
  return __clzll(a ^ b);
}

__global__ void k_karras(const unsigned long long* __restrict__ keys, int n, int2* children, int* parent,
                         int* leaves, int* axis) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1) return;
  int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
  int dmin = delta(keys, n, i, i - d);
  int lmax = 2;
  while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
  int l = 0;
  for (int t = lmax >> 1; t >= 1; t >>= 1)
    if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
  int j = i + l * d;
  int dnode = delta(keys, n, i, j);
  int s = 0;
  for (int t = (l + 1) >> 1;; t = (t + 1) >> 1) {
    if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    if (t == 1) break;
  }
  int gamma = i + s * d + min(d, 0);
  int first = min(i, j), last = max(i, j);
  int left = (first == gamma) ? ~gamma : gamma;
  int right = (last == gamma + 1) ? ~(gamma + 1) : gamma + 1;
  children[i] = make_int2(left, right);
  leaves[i] = last - first + 1;
  // the children differ first in Morton bit b; bits cycle x,y,z from the top, and the left child has the 0
  // bit, i.e. the lower coordinate on that axis -- exactly what near/far ordering by axis sign expects
  unsigned long long diff = keys[gamma] ^ keys[gamma + 1];
  int b = diff ? 63 - __clzll(diff) : 2;
  axis[i] = 2 - (b % 3);
  if (left >= 0) parent[left] = i; else parent[n - 1 + gamma] = i;
  if (right >= 0) parent[right] = i; else parent[n - 1 + gamma + 1] = i;
  if (i == 0) parent[0] = -1;
}

// The bottom-up climb of both box fits: a thread that has finished a node's box (a leaf's, or an inner node's) fences
// it and arrives at the parent, one arrival flag per inner node.  The first arrival stops, because the sibling subtree
// is not ready yet; the second one fits the parent from both children, first child then second, reading the sibling's
// box past L1 (another SM may have written it), fences it and climbs on.
template <class Fit>
__device__ __forceinline__ void climb_boxes(int node, const int* __restrict__ parent, int* flags, Fit fit) {
  while (node >= 0) {
    if (atomicAdd(&flags[node], 1) == 0) return;  // first arrival: the sibling subtree is not ready yet
    __threadfence();
    fit(node);
    __threadfence();
    node = parent[node];
  }
}

// LBVH boxes: one thread per leaf climbs; the second child to arrive at a node computes it
__global__ void k_fit_boxes(const RefPrim* __restrict__ prims, const int* __restrict__ order, int n,
                            const int2* __restrict__ children, const int* __restrict__ parent, float* boxes,
                            int* flags) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  climb_boxes(parent[n - 1 + j], parent, flags, [&](int node) {
    float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    int2 ch = children[node];
    int refs[2] = {ch.x, ch.y};
    for (int c = 0; c < 2; c++) {
      if (refs[c] < 0) {
        const RefPrim& p = prims[order[~refs[c]]];
        for (int k = 0; k < 3; k++) {
          mn[k] = fminf(mn[k], fminf(fminf(p.a[k], p.b[k]), p.c[k]));
          mx[k] = fmaxf(mx[k], fmaxf(fmaxf(p.a[k], p.b[k]), p.c[k]));
        }
      } else {
        const volatile float* b = boxes + 6 * refs[c];
        for (int k = 0; k < 3; k++) {
          mn[k] = fminf(mn[k], b[k]);
          mx[k] = fmaxf(mx[k], b[3 + k]);
        }
      }
    }
    for (int k = 0; k < 3; k++) {
      boxes[6 * node + k] = mn[k];
      boxes[6 * node + 3 + k] = mx[k];
    }
  });
}

// ---- refit of a tree in the reference layout (lt_scene_refit) ----

// std::min / std::max: the first operand on ties, so that of -0 and +0 the earlier one is kept, as the host builder
// (acceleration_structure_explicit.cpp) and Model's primitive bounds compute them.  fminf / fmaxf promise no sign.
__device__ __forceinline__ float first_min(float a, float b) { return b < a ? b : a; }
__device__ __forceinline__ float first_max(float a, float b) { return a < b ? b : a; }

// parent of every node of a DFS-layout tree: inner node i has children i + 1 and offset
__global__ void k_dfs_parents(const RefNode* __restrict__ nodes, int n, int* parent) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (i == 0) parent[0] = -1;
  if (nodes[i].primitiveCount == 0) {
    parent[i + 1] = i;
    parent[nodes[i].offset] = i;
  }
}

// One thread per leaf: the leaf's box covers all primitiveCount primitives from its offset, in order; then the climb
// fits every inner node from its first child (i + 1) and its second (offset), in that order.
__global__ void k_refit(RefNode* nodes, int n, const RefPrim* __restrict__ prims, const int* __restrict__ parent,
                        int* flags) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int count = nodes[i].primitiveCount, first = nodes[i].offset;
  if (count == 0) return;
  float mn[3], mx[3];
  for (int j = 0; j < count; j++) {
    const RefPrim& p = prims[first + j];
    for (int k = 0; k < 3; k++) {
      const float lo = first_min(first_min(p.a[k], p.b[k]), p.c[k]);
      const float hi = first_max(first_max(p.a[k], p.b[k]), p.c[k]);
      mn[k] = j ? first_min(mn[k], lo) : lo;
      mx[k] = j ? first_max(mx[k], hi) : hi;
    }
  }
  for (int k = 0; k < 3; k++) {
    nodes[i].boundsMin[k] = mn[k];
    nodes[i].boundsMax[k] = mx[k];
  }
  __threadfence();
  climb_boxes(parent[i], parent, flags, [&](int node) {
    const volatile RefNode* a = nodes + node + 1;
    const volatile RefNode* b = nodes + nodes[node].offset;
    for (int k = 0; k < 3; k++) {
      nodes[node].boundsMin[k] = first_min(a->boundsMin[k], b->boundsMin[k]);
      nodes[node].boundsMax[k] = first_max(a->boundsMax[k], b->boundsMax[k]);
    }
  });
}

// bad |= 1 for a materialIndex outside [0, matCount), |= 2 for a non-finite vertex coordinate
__global__ void k_check_prims(const RefPrim* __restrict__ prims, int n, int matCount, int* bad) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const RefPrim& p = prims[i];
  int why = p.materialIndex < 0 || p.materialIndex >= matCount ? 1 : 0;
  for (int k = 0; k < 3; k++)
    if (!isfinite(p.a[k]) || !isfinite(p.b[k]) || !isfinite(p.c[k])) why |= 2;
  if (why) atomicOr(bad, why);
}

// ---- PLOC iteration over the cluster array of length m ----

__global__ void k_ploc_init(const RefPrim* __restrict__ prims, const int* __restrict__ order, int n, int* node,
                            LtBox* box) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const RefPrim& p = prims[order[j]];
  LtBox b;
  for (int k = 0; k < 3; k++) {
    b.lo[k] = fminf(fminf(p.a[k], p.b[k]), p.c[k]);
    b.hi[k] = fmaxf(fmaxf(p.a[k], p.b[k]), p.c[k]);
  }
  node[j] = ~j;
  box[j] = b;
}

// murmur3 finalizer of a ^ (b * golden ratio): the tie key of the pair {a < b}
__device__ __forceinline__ unsigned pair_hash(int a, int b) {
  unsigned h = (unsigned)a ^ ((unsigned)b * 0x9E3779B9u);
  h ^= h >> 16;
  h *= 0x85EBCA6Bu;
  h ^= h >> 13;
  h *= 0xC2B2AE35u;
  h ^= h >> 16;
  return h;
}

// nn[i] = the j in [i-R, i+R] (j != i) whose pair {min, max} has the smallest key (half-area of the union box, pair
// hash, min, max).  The half-area is compared by its bit pattern: an order on every float, NaN included, which is
// the float order for the non-negative numbers it takes on finite input.  One block covers PLOC_BLOCK consecutive
// clusters and stages the boxes of its range +- R (structure of arrays: no bank conflicts).
__global__ void __launch_bounds__(PLOC_BLOCK) k_ploc_nn(int m, const LtBox* __restrict__ box, int* nn) {
  constexpr int R = PLOC_RADIUS, W = PLOC_BLOCK + 2 * PLOC_RADIUS;
  __shared__ float s[6][W];
  const int b0 = blockIdx.x * PLOC_BLOCK;
  for (int t = threadIdx.x; t < W; t += PLOC_BLOCK) {
    int g = b0 - R + t;
    if (g >= 0 && g < m) {
      const LtBox b = box[g];
      for (int k = 0; k < 3; k++) {
        s[k][t] = b.lo[k];
        s[3 + k][t] = b.hi[k];
      }
    }
  }
  __syncthreads();
  const int i = b0 + threadIdx.x;
  if (i >= m) return;
  const int c = threadIdx.x + R;
  const float lx = s[0][c], ly = s[1][c], lz = s[2][c], hx = s[3][c], hy = s[4][c], hz = s[5][c];
  unsigned bestD = 0xffffffffu;
  int best = -1;
#pragma unroll
  for (int o = -R; o <= R; o++) {
    const int j = i + o;
    if (o == 0 || j < 0 || j >= m) continue;
    const int t = c + o;
    const float dx = FSUB(fmaxf(hx, s[3][t]), fminf(lx, s[0][t]));
    const float dy = FSUB(fmaxf(hy, s[4][t]), fminf(ly, s[1][t]));
    const float dz = FSUB(fmaxf(hz, s[5][t]), fminf(lz, s[2][t]));
    const unsigned d = __float_as_uint(FADD(FADD(FMUL(dx, dy), FMUL(dy, dz)), FMUL(dz, dx)));
    bool better = d < bestD || best < 0;
    if (!better && d == bestD) {  // equal areas: the pair hash, then the pair itself
      const int a = min(i, j), b = max(i, j), ba = min(i, best), bb = max(i, best);
      const unsigned h = pair_hash(a, b), bh = pair_hash(ba, bb);
      better = h < bh || (h == bh && (a < ba || (a == ba && b < bb)));
    }
    if (better) {
      bestD = d;
      best = j;
    }
  }
  nn[i] = best;
}

__global__ void k_ploc_flags(int m, const int* __restrict__ nn, int* merge, int* keep) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const int j = nn[i];
  const bool mutual = nn[j] == i;
  merge[i] = mutual && i < j;
  keep[i] = !(mutual && j < i);
}

__device__ __forceinline__ float box_centre(const LtBox& b, int k) { return FADD(FMUL(0.5f, b.lo[k]), FMUL(0.5f, b.hi[k])); }

// Survivors move to newPos; a merging pair becomes inner node m-2-mergeRank at the lower position (ids are handed
// out downwards from n-2, so the last merge makes node 0, the root).  The split axis is the one on which the
// children's box centres lie farthest apart (lowest axis on ties); the child with the lower centre on it comes
// first (the lower cluster position on ties), which is what near/far ordering by the ray direction's sign expects.
__global__ void k_ploc_compact(int n, int m, const int* __restrict__ nodeIn, const LtBox* __restrict__ boxIn,
                               const int* __restrict__ nn, const int* __restrict__ merge, const int* __restrict__ keep,
                               const int* __restrict__ mergeRank, const int* __restrict__ newPos, int* nodeOut,
                               LtBox* boxOut, int2* children, int* parent, int* leaves, float* boxes, int* axis,
                               int* newCount) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  if (i == m - 1) *newCount = newPos[i] + keep[i];
  if (!keep[i]) return;
  const int p = newPos[i];
  if (!merge[i]) {
    nodeOut[p] = nodeIn[i];
    boxOut[p] = boxIn[i];
    return;
  }
  const int j = nn[i];
  const int id = m - 2 - mergeRank[i];
  const LtBox A = boxIn[i], B = boxIn[j];
  int ax = 0;
  float spread = -1.0f;
  for (int k = 0; k < 3; k++) {
    const float d = fabsf(FSUB(box_centre(A, k), box_centre(B, k)));
    if (d > spread) {
      spread = d;
      ax = k;
    }
  }
  const bool swap = box_centre(B, ax) < box_centre(A, ax);
  const int first = swap ? nodeIn[j] : nodeIn[i], second = swap ? nodeIn[i] : nodeIn[j];
  LtBox u;
  for (int k = 0; k < 3; k++) {
    u.lo[k] = fminf(A.lo[k], B.lo[k]);
    u.hi[k] = fmaxf(A.hi[k], B.hi[k]);
    boxes[6 * id + k] = u.lo[k];
    boxes[6 * id + 3 + k] = u.hi[k];
  }
  children[id] = make_int2(first, second);
  leaves[id] = (first < 0 ? 1 : leaves[first]) + (second < 0 ? 1 : leaves[second]);
  axis[id] = ax;
  parent[first < 0 ? n - 1 + ~first : first] = id;
  parent[second < 0 ? n - 1 + ~second : second] = id;
  if (id == 0) parent[0] = -1;
  nodeOut[p] = id;
  boxOut[p] = u;
}

// ---- emission (both builders) ----

// DFS (pre-order, first child adjacent) index and leaf rank from the parent chain: a step out of a first child adds 1
// to the DFS index; a step out of a second child adds 2 * leaves(first sibling) (the size of the sibling's subtree)
// to it and leaves(first sibling) to the leaf rank.
__global__ void k_dfs_index(int n, const int2* __restrict__ children, const int* __restrict__ parent,
                            const int* __restrict__ leaves, int* dfsIndex, int* leafRank, int* maxDepth) {
  int v = blockIdx.x * blockDim.x + threadIdx.x;  // [0, n-1) internal, [n-1, 2n-1) leaves
  if (v >= 2 * n - 1) return;
  bool leaf = v >= n - 1;
  int dfs = 0, rank = 0, depth = 0;
  int childRef = leaf ? ~(v - (n - 1)) : v;
  int node = parent[v];
  while (node >= 0) {
    const int2 ch = children[node];
    if (ch.x == childRef) {
      dfs++;
    } else {
      const int l = ch.x < 0 ? 1 : leaves[ch.x];
      dfs += 2 * l;
      rank += l;
    }
    depth++;
    childRef = node;
    node = parent[node];
  }
  dfsIndex[v] = dfs;
  if (leaf) {
    leafRank[v - (n - 1)] = rank;
    atomicMax(maxDepth, depth);  // inner nodes above a leaf = stack bound
  }
}

__global__ void k_emit_nodes(const RefPrim* __restrict__ prims, const int* __restrict__ order, int n,
                             const int2* __restrict__ children, const float* __restrict__ boxes,
                             const int* __restrict__ axisArr, const int* __restrict__ dfsIndex,
                             const int* __restrict__ leafRank, RefNode* nodes, RefPrim* orderedPrims) {
  int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= 2 * n - 1) return;
  RefNode out;
  if (v >= n - 1) {  // leaf at sorted position j
    int j = v - (n - 1);
    int r = leafRank[j];
    RefPrim p = prims[order[j]];
    orderedPrims[r] = p;
    for (int k = 0; k < 3; k++) {
      out.boundsMin[k] = fminf(fminf(p.a[k], p.b[k]), p.c[k]);
      out.boundsMax[k] = fmaxf(fmaxf(p.a[k], p.b[k]), p.c[k]);
    }
    out.offset = r;
    out.primitiveCount = 1;
    out.axis = 0;
  } else {
    for (int k = 0; k < 3; k++) {
      out.boundsMin[k] = boxes[6 * v + k];
      out.boundsMax[k] = boxes[6 * v + 3 + k];
    }
    int2 ch = children[v];
    int rightV = ch.y < 0 ? n - 1 + ~ch.y : ch.y;
    out.offset = dfsIndex[rightV];
    out.primitiveCount = 0;
    out.axis = (uint8_t)axisArr[v];
  }
  out.pad = 0;
  nodes[dfsIndex[v]] = out;
}

// lights in leaf order, first 64 (single thread: the list is tiny and must be ordered)
__global__ void k_collect_lights(const RefPrim* __restrict__ orderedPrims, int n, const RefMaterial* __restrict__ mats,
                                 int matCount, RefLights* lights) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  RefLights out;
  out.count = 0;
  for (int k = 0; k < 64; k++) out.primitives[k] = 0;
  for (int i = 0; i < n && out.count < 64; i++) {
    int m = orderedPrims[i].materialIndex;
    if (m >= 0 && m < matCount) {
      const RefMaterial& mat = mats[m];
      if (mat.emission[0] > 0 || mat.emission[1] > 0 || mat.emission[2] > 0) out.primitives[out.count++] = (unsigned)i;
    }
  }
  *lights = out;
}

// parallel variant for large scenes: flag emissive primitives, the host keeps the first 64 in order
__global__ void k_flag_emissive(const RefPrim* __restrict__ orderedPrims, int n, const RefMaterial* __restrict__ mats,
                                int matCount, int* counter, int* firstEmissive /* up to 4096 indices */) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int m = orderedPrims[i].materialIndex;
  if (m < 0 || m >= matCount) return;
  const RefMaterial& mat = mats[m];
  if (mat.emission[0] > 0 || mat.emission[1] > 0 || mat.emission[2] > 0) {
    int slot = atomicAdd(counter, 1);
    if (slot < 4096) firstEmissive[slot] = i;
  }
}

}  // namespace

int lt_launch_refit_parents(const RefNode* dNodes, int n, int* dParent, cudaStream_t stream) {
  k_dfs_parents<<<(n + 255) / 256, 256, 0, stream>>>(dNodes, n, dParent);
  return 1;
}

int lt_launch_refit(RefNode* dNodes, int n, const RefPrim* dPrims, const int* dParent, int* dFlags,
                    cudaStream_t stream) {
  cudaMemsetAsync(dFlags, 0, sizeof(int) * (size_t)n, stream);
  k_refit<<<(n + 255) / 256, 256, 0, stream>>>(dNodes, n, dPrims, dParent, dFlags);
  return 1;
}

int lt_launch_check_prims(const RefPrim* dPrims, int n, int matCount, int* dBad, cudaStream_t stream) {
  cudaMemsetAsync(dBad, 0, sizeof(int), stream);
  k_check_prims<<<(n + 255) / 256, 256, 0, stream>>>(dPrims, n, matCount, dBad);
  return 1;
}

size_t lt_bvh_scratch_bytes(int n, LtBvhBuilder builder) {
  BuildScratch S;
  return carve_scratch(S, nullptr, n, builder);
}

// PLOC: merges the n sorted leaves into one tree (children, parent, leaves, boxes, axis).  The host reads the cluster
// count back after every iteration; an iteration that merges nothing means a bug and ends the build with an error
// (the smallest pair under the strict key order is always mutual, so every iteration merges at least once).
// Returns the kernels launched, or -1.
static int ploc_hierarchy(const RefPrim* dPrims, const int* order, int n, BuildScratch& S, cudaStream_t stream) {
  const int T = 256;
  k_ploc_init<<<(n + T - 1) / T, T, 0, stream>>>(dPrims, order, n, S.clusterNode[0], S.clusterBox[0]);
  int launches = 1, cur = 0, m = n;
  while (m > 1) {
    const int blocks = (m + T - 1) / T;
    k_ploc_nn<<<(m + PLOC_BLOCK - 1) / PLOC_BLOCK, PLOC_BLOCK, 0, stream>>>(m, S.clusterBox[cur], S.nn);
    k_ploc_flags<<<blocks, T, 0, stream>>>(m, S.nn, S.merge, S.keep);
    lt_launch_exclusive_scan(S.scanTemp, S.scanBytes, S.merge, S.mergeRank, m, stream);
    lt_launch_exclusive_scan(S.scanTemp, S.scanBytes, S.keep, S.newPos, m, stream);
    k_ploc_compact<<<blocks, T, 0, stream>>>(n, m, S.clusterNode[cur], S.clusterBox[cur], S.nn, S.merge, S.keep,
                                             S.mergeRank, S.newPos, S.clusterNode[cur ^ 1], S.clusterBox[cur ^ 1],
                                             S.children, S.parent, S.leaves, S.boxes, S.axis, S.newCount);
    launches += 5;
    int next = m;
    if (cudaMemcpyAsync(&next, S.newCount, sizeof(int), cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
        cudaStreamSynchronize(stream) != cudaSuccess || next < 1 || next >= m)
      return -1;
    m = next;
    cur ^= 1;
  }
  return launches;
}

// Builds nodes / ordered primitives / lights (all device buffers in the reference layouts).  Returns the
// number of kernels launched, or -1 on a CUDA error.  *outMaxDepth receives the stack bound.
int lt_launch_bvh_build(LtBvhBuilder builder, const RefPrim* dPrims, int n, const RefMaterial* dMats, int matCount,
                        RefNode* dNodes, RefPrim* dOrderedPrims, RefLights* dLights, void* scratch, size_t scratchBytes,
                        int* outMaxDepth, cudaStream_t stream) {
  if (n < 2) return -1;  // a single triangle has no hierarchy: callers use lt_scene_upload for that
  BuildScratch S;
  if (carve_scratch(S, (char*)scratch, n, builder) > scratchBytes) return -1;
  cub::DoubleBuffer<unsigned long long> kb(S.keys[0], S.keys[1]);
  cub::DoubleBuffer<int> vb(S.order[0], S.order[1]);

  const int T = 256;
  const unsigned initBounds[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
  cudaMemcpyAsync(S.bounds, initBounds, sizeof initBounds, cudaMemcpyHostToDevice, stream);
  cudaMemsetAsync(S.maxDepth, 0, sizeof(int), stream);
  cudaMemsetAsync(S.emissiveCount, 0, sizeof(int), stream);
  k_centroid_bounds<<<(n + T - 1) / T, T, 0, stream>>>(dPrims, n, S.bounds);
  k_morton<<<(n + T - 1) / T, T, 0, stream>>>(dPrims, n, S.bounds, S.keys[0], S.order[0]);
  cub::DeviceRadixSort::SortPairs(S.sortTemp, S.sortBytes, kb, vb, n, 0, 63, stream);
  const unsigned long long* keys = kb.Current();
  const int* order = vb.Current();
  int launches = 3;
  if (builder == LT_BVH_PLOC) {
    const int h = ploc_hierarchy(dPrims, order, n, S, stream);
    if (h < 0) return -1;
    launches += h;
  } else {
    cudaMemsetAsync(S.flags, 0, sizeof(int) * n, stream);
    k_karras<<<(n - 1 + T - 1) / T, T, 0, stream>>>(keys, n, S.children, S.parent, S.leaves, S.axis);
    k_fit_boxes<<<(n + T - 1) / T, T, 0, stream>>>(dPrims, order, n, S.children, S.parent, S.boxes, S.flags);
    launches += 2;
  }
  k_dfs_index<<<(2 * n - 1 + T - 1) / T, T, 0, stream>>>(n, S.children, S.parent, S.leaves, S.dfsIndex, S.leafRank,
                                                         S.maxDepth);
  k_emit_nodes<<<(2 * n - 1 + T - 1) / T, T, 0, stream>>>(dPrims, order, n, S.children, S.boxes, S.axis, S.dfsIndex,
                                                          S.leafRank, dNodes, dOrderedPrims);
  k_collect_lights<<<1, 1, 0, stream>>>(dOrderedPrims, n < 65536 ? n : 0, dMats, matCount, dLights);
  launches += 3;
  if (n >= 65536) {  // large scenes: parallel flagging, ordered selection on the host
    k_flag_emissive<<<(n + T - 1) / T, T, 0, stream>>>(dOrderedPrims, n, dMats, matCount, S.emissiveCount, S.emissive);
    launches++;
    int count = 0;
    cudaMemcpyAsync(&count, S.emissiveCount, sizeof(int), cudaMemcpyDeviceToHost, stream);
    cudaStreamSynchronize(stream);
    if (count > 4096) count = 4096;
    std::vector<int> idx(count);
    if (count) cudaMemcpy(idx.data(), S.emissive, sizeof(int) * count, cudaMemcpyDeviceToHost);
    std::sort(idx.begin(), idx.end());
    RefLights L;
    memset(&L, 0, sizeof L);
    for (int k = 0; k < count && L.count < 64; k++) L.primitives[L.count++] = (unsigned)idx[k];
    cudaMemcpyAsync(dLights, &L, sizeof L, cudaMemcpyHostToDevice, stream);
  }
  if (outMaxDepth) {
    cudaMemcpyAsync(outMaxDepth, S.maxDepth, sizeof(int), cudaMemcpyDeviceToHost, stream);
    cudaStreamSynchronize(stream);
  }
  return cudaGetLastError() == cudaSuccess ? launches : -1;
}
