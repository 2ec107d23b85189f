// lt_kernels.cu -- hand-written sm_100a kernels for lens_trace's ray-scene hot path.
//
// Path (reference file:line):  camera ray basic.cu:350-358 -> intersect basic.cu:156-243 ->
// intersectBounds basic.cu:136-154 -> intersectTriangle basic.cu:93-134 -> shade (basic.cu:300-329,
// basic_lighting.cl:220-277, global_illumination.cl:242-376, custom_opencl.cl:226-244) -> blend /
// running mean (global_illumination.cl:408-419, accumulator.frag:10-19).
//
// Design (DESIGN.md has the long form):
//  * 64-byte child-pair nodes (LtWideNode) and 48-byte triangles (LtTri), 128-bit loads only.
//  * One traversal routine shared by primary, shadow and extension rays.  Each thread owns one
//    pixel and runs a per-thread state machine whose every iteration traces exactly one ray, so a
//    warp stays converged in the traversal loop while its lanes are at different path stages.
//  * Traversal stack in shared memory, laid out [level][thread] (bank-conflict free).
//  * All FP32 arithmetic is written with explicit round-to-nearest intrinsics in the operation
//    order the reference compiles to, so results do not depend on compiler contraction.
//  * Tensor cores are not used: nothing here is a dense contraction.
#include "lt_internal.h"
#include "lt_device.cuh"

#include <cub/device/device_scan.cuh>
#include <stdlib.h>

#define LT_LAUNCH_FLAG_NO_STREAM 64  // == LT_FLAG_NO_STREAM (include/lens_trace_b200.h)

template <bool STATS>
__global__ void __launch_bounds__(LT_BLOCK) k_flat(LtSceneDev sc, LtLaunch L, float* __restrict__ out,
                                                   LtCounters* gcnt) {
  LT_SMEM_POINTERS(sc)
  int px, py;
  if (!thread_pixel(L.width, L.height, px, py)) return;
  LtCounters cnt = {0, 0, 0};
  float fx, fy;
  Trav t;
  t.r = camera_ray(L.cam, px, lt_image_row(L, py), L.width, L.fullHeight, fx, fy);
  const float tInit = lt_tinit(L.kernel), epsThr = lt_eps(L.kernel);
  float color[3] = {0.0f, 0.0f, 0.0f};
  const bool cull = (L.flags & 2) != 0;  // LT_FLAG_CULL
  if (cull) trace_cull<STATS>(t, sc, -1, tInit, epsThr, stk, tstk, cnt);
  else trace<STATS>(t, sc, -1, tInit, epsThr, false, stk, list, cnt);
  if (t.h.hit == 1) {
    if (L.kernel == 2) {  // custom_opencl.cl:240
      color[0] = t.h.u;
      color[1] = t.h.v;
      color[2] = bary0(t.h.u, t.h.v);
    } else {  // basic.cu:312-326
      const RefMaterial* mat = sc.mats + sc.prims[t.h.prim].materialIndex;
      if (mat->dissolve < 1.0f) {
        lens_path<STATS>(sc, t, tInit, epsThr, stk, list, tstk, cull, cnt);
        if (t.h.hit == 1) mat = sc.mats + sc.prims[t.h.prim].materialIndex;
      }
      color[0] = mat->diffuse[0];
      color[1] = mat->diffuse[1];
      color[2] = mat->diffuse[2];
    }
  }
  long long id = ((long long)py * L.width + px) * L.depth;
  FrameSink sink;
  sink.begin(L, out, id);
  // the image is the same for every frame (no RNG): apply the frame combiner `frames` times
  for (int f = 0; f < L.frames; f++) sink.frame(L, L.cam.frameCount + (unsigned)f * L.frameStride, color);
  sink.end(out, id);
  if (STATS) {
    cnt.rays *= (unsigned)L.frames;
    cnt.nodeTests *= (unsigned)L.frames;
    cnt.triTests *= (unsigned)L.frames;
    flush_counters(gcnt, cnt);
  }
}

// Persistent form of k_flat for the exact, uncounted launches on large scenes.  Blocks stay resident (SMs x blocks
// per SM) and every WARP takes the next 8x4 pixel tile from a global counter when all its rays are done.  Measured
// on the 1 M-triangle mesh, 1080p primary rays (profiles/r2a_*, tools/ray_length_histogram.py): with a fixed
// 16x8 tile per block the SMs were active 45 % of the kernel's duration (0.99 ms; the rays of the height field make
// 733 dependent box-pair steps, those of the walls 22) -- warps that fetch tiles on their own: 0.73 ms.  Dealing
// single pixels to idle lanes (as k_wf_trace deals queue entries) was measured too and LOSES, 1.83 ms: the camera
// rays of a tile walk the tree together (lane utilisation 0.90) and share its cache lines.  Rays run through the
// same software-pipelined traversal as k_wf_trace; the lens path (basic.cu:245-298) is two more rays of the same
// lane.  Same tests in the same order per ray as k_flat, hence the same picture (LT_FLAG_NO_STREAM selects k_flat;
// tests compare the two).
__global__ void __launch_bounds__(LT_BLOCK) k_flat_stream(LtSceneDev sc, LtLaunch L, float* __restrict__ out,
                                                          int* __restrict__ work) {
  extern __shared__ int smemStack[];
  int* stk = smemStack + threadIdx.x;
  int* list = smemStack + lt_stack_levels(sc) * LT_BLOCK + threadIdx.x;
  const unsigned stkAddr = (unsigned)__cvta_generic_to_shared(stk);
  const unsigned fifoAddr = (unsigned)__cvta_generic_to_shared(list);
  const unsigned lane = threadIdx.x & 31u;
  const float tInit = lt_tinit(L.kernel), epsThr = lt_eps(L.kernel);
  const float camC = cosf(L.cam.yaw), camS = sinf(L.cam.yaw);
  const int tilesX = (L.width + 7) >> 3, tilesY = (L.height + 3) >> 2;
  const int nTiles = tilesX * tilesY;
  LtCounters cnt = {0, 0, 0};
  while (true) {
    int tile = 0;
    if (lane == 0u) tile = atomicAdd(work, 1);
    tile = __shfl_sync(0xffffffffu, tile, 0);
    if (tile >= nTiles) break;
    const int ty = tile / tilesX, tx = tile - ty * tilesX;
    const int px = (tx << 3) + (int)(lane & 7u), py = (ty << 2) + (int)(lane >> 3);
    if (px >= L.width || py >= L.height) continue;  // (the other lanes of the warp run their pixels; no barrier follows)
    float fx, fy;
    Trav t;
    t.r = camera_ray_cs(L.cam, camC, camS, px, lt_image_row(L, py), L.width, L.fullHeight, fx, fy);
    float color[3] = {0.0f, 0.0f, 0.0f};
    int baseMat = 0;  // material of the camera ray's hit (kept when the lens path ends in a miss)
    float r2w = 0.0f;
    int ignore = -1;
    for (int stage = 0; stage < 3; stage++) {  // 0 camera ray, 1 and 2 the rays through a lens (basic.cu:245-298)
      trav_begin<false>(t, sc, ignore, tInit, false, cnt);
      while (!trav_iter_lean<false>(t, sc, stkAddr, fifoAddr, epsThr, kLeanNodeSteps, kLeanTriTests, cnt)) {
      }
      const Hit h = t.h;
      if (stage == 0) {
        if (h.hit != 1) break;
        if (L.kernel == 2) {  // custom_opencl.cl:240
          color[0] = h.u;
          color[1] = h.v;
          color[2] = bary0(h.u, h.v);
          break;
        }
        baseMat = sc.prims[h.prim].materialIndex;  // basic.cu:312-326
        if (!(sc.mats[baseMat].dissolve < 1.0f)) break;
        ignore = lens_refract_in(sc, t.r, h, r2w);
      } else if (stage == 1) {
        ignore = lens_refract_out(sc, t.r, h, r2w);
      } else if (h.hit == 1) {
        baseMat = sc.prims[h.prim].materialIndex;
      }
    }
    if (L.kernel != 2 && (t.h.hit == 1 || ignore >= 0)) {
      const RefMaterial* mat = sc.mats + baseMat;
      color[0] = mat->diffuse[0];
      color[1] = mat->diffuse[1];
      color[2] = mat->diffuse[2];
    }
    const long long id = ((long long)py * L.width + px) * L.depth;
    FrameSink sink;
    sink.begin(L, out, id);
    for (int f = 0; f < L.frames; f++) sink.frame(L, L.cam.frameCount + (unsigned)f * L.frameStride, color);
    sink.end(out, id);
  }
}

// One thread = one pixel, persistent over all frames and samples of the launch.  The warp alternates
// between two phases:
//   S (shade/regenerate): lanes whose ray has finished consume the hit and produce their next ray
//     (primary, shadow or extension); the hash-RNG draws, the expensive part, are one shared code
//     site whatever the path stage;
//   T (traverse): all lanes with an unfinished ray run the traversal in its leaf-list form (whole
//     batches of box tests, then the recorded triangles; the stackless form on a threaded tree); the
//     loop is left as soon as fewer than kPathRefillLanes lanes are still traversing and some lane is
//     waiting for a new ray, so long rays never hold the other 31 lanes idle.  Traversal state is
//     resumable.
constexpr int kPathRefillLanes = 4;
template <bool STATS>
__global__ void __launch_bounds__(LT_BLOCK) k_path(LtSceneDev sc, LtLaunch L, float* __restrict__ out,
                                                   LtCounters* gcnt) {
  LT_SMEM_POINTERS(sc)
  (void)tstk;  // the persistent megakernel does not cull (LT_FLAG_CULL selects the wavefront pipeline)
  const unsigned fifoAddr = (unsigned)__cvta_generic_to_shared(list);
  int px, py;
  bool alive = thread_pixel(L.width, L.height, px, py);
  LtCounters cnt = {0, 0, 0};
  const PathConsts pc = path_consts(L);

  float fx = 0.0f, fy = 0.0f;
  Ray cameraRay = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 1.0f};
  long long id = 0;
  FrameSink sink;
  sink.acc[0] = sink.acc[1] = sink.acc[2] = 0.0f;
  if (alive) {
    cameraRay = camera_ray(L.cam, px, lt_image_row(L, py), L.width, L.fullHeight, fx, fy);
    id = ((long long)py * L.width + px) * L.depth;
    sink.begin(L, out, id);
  }

  int frame = 0, sample = 0;
  float frameColor[3] = {0.0f, 0.0f, 0.0f};
  unsigned sampleIndex = (pc.samplesPerFrame == 25) ? L.cam.frameCount * 32u : L.cam.frameCount;
  PathState ps;
  ps.nrm[0] = ps.nrm[1] = ps.nrm[2] = 0.0f;
  ps.diffuse[0] = ps.diffuse[1] = ps.diffuse[2] = 0.0f;
  ps.extW = 0.0f;
  ps.hitPrim = 0;
  ps.depth = 0;
  path_reset(ps);

  const bool threaded = !STATS && sc.tnodes != nullptr;  // small scene: stackless threaded tree, same tests
  Trav t;
  t.r = cameraRay;
  bool traversing = false;
  if (alive) {
    if (threaded) trav_begin_threaded(t, sc, -1, pc.tInit, false);
    else trav_begin<STATS>(t, sc, -1, pc.tInit, false, cnt);
    traversing = (t.cur != LT_DONE);
  }

  while (true) {
    // ---------------- phase S: consume finished rays, generate the next ones ----------------
    while (alive && !traversing) {
      float tStart;
      int ignore;
      bool anyHit;
      const Hit h = t.h;
      if (shade_step(sc, pc, ps, t.r, h, fx, fy, sampleIndex, tStart, ignore, anyHit)) {
        float c[3];
        sample_colour(pc, ps, c);
        blend_sample(pc, sample, c, frameColor);
        sample++;
        if (sample == pc.samplesPerFrame) {
          finish_frame_colour(pc, L.kernelMode, frameColor);
          sink.frame(L, L.cam.frameCount + (unsigned)frame * L.frameStride, frameColor);
          sample = 0;
          frame++;
          if (frame >= L.frames) {
            sink.end(out, id);
            alive = false;
            break;
          }
        }
        unsigned fcNext = L.cam.frameCount + (unsigned)frame * L.frameStride;
        sampleIndex = (pc.samplesPerFrame == 25) ? fcNext * 32u + (unsigned)sample : fcNext;
        path_reset(ps);
        t.r = cameraRay;
        ignore = -1;
        tStart = pc.tInit;
        anyHit = false;
      }
      if (threaded) trav_begin_threaded(t, sc, ignore, tStart, anyHit);
      else trav_begin<STATS>(t, sc, ignore, tStart, anyHit, cnt);
      traversing = (t.cur != LT_DONE);
    }
    if (!__any_sync(0xffffffffu, alive)) break;

    // ---------------- phase T: resumable traversal ----------------
    while (true) {
      unsigned active = __ballot_sync(0xffffffffu, traversing);
      if (active == 0u) break;
      bool waiting = __any_sync(0xffffffffu, alive && !traversing);
      if (waiting && __popc(active) < kPathRefillLanes) break;
      if (traversing) {
        if (threaded) {
          traversing = !trav_iter_threaded(t, sc.tnodes, sc.tris, fifoAddr, pc.epsThr, kThreadedNodeSteps, kThreadedTriTests);
        } else {
          int n = trav_collect<STATS>(t, sc, stk, list, LT_MAX_BATCH, cnt);
          trav_test<STATS>(t, sc, list, n, pc.epsThr, cnt);
          traversing = (t.cur != LT_DONE);
        }
      }
    }
  }
  if (STATS) flush_counters(gcnt, cnt);
}

// ------------------------------------------------------------------------------------------------
// primary hit records (parity/debug output)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(LT_BLOCK) k_primary_hits(LtSceneDev sc, RefCamera cam, int kernel, int flags,
                                                           int width, int height, int* __restrict__ ids,
                                                           int* __restrict__ hit, float* __restrict__ tuv) {
  LT_SMEM_POINTERS(sc)
  int px, py;
  if (!thread_pixel(width, height, px, py)) return;
  LtCounters cnt = {0, 0, 0};
  float fx, fy;
  Trav t;
  t.r = camera_ray(cam, px, py, width, height, fx, fy);
  if (flags & 2) trace_cull<false>(t, sc, -1, lt_tinit(kernel), lt_eps(kernel), stk, tstk, cnt);
  else trace<false>(t, sc, -1, lt_tinit(kernel), lt_eps(kernel), false, stk, list, cnt);
  const Hit h = t.h;
  long long i = (long long)py * width + px;
  if (ids) ids[i] = h.prim;
  if (hit) hit[i] = h.hit;
  if (tuv) {
    tuv[3 * i + 0] = h.t;
    tuv[3 * i + 1] = h.u;
    tuv[3 * i + 2] = h.v;
  }
}

// device evaluation of the hash RNG and hemisphere sampler on caller-supplied inputs (parity hook)
__global__ void k_debug_random(const float* __restrict__ fx, const float* __restrict__ fy, const float* __restrict__ seed,
                               int n, float* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = lt_random(fx[i], fy[i], seed[i]);
}

__global__ void k_debug_hemisphere(const float* __restrict__ u1, const float* __restrict__ u2,
                                   const float* __restrict__ up, int n, float* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float upv[3] = {up[3 * i], up[3 * i + 1], up[3 * i + 2]};
  float d[4];
  sample_hemisphere(u1[i], u2[i], upv, d);
  out[4 * i + 0] = d[0]; out[4 * i + 1] = d[1]; out[4 * i + 2] = d[2]; out[4 * i + 3] = d[3];
}

// ------------------------------------------------------------------------------------------------
// upload-time re-flatten: reference nodes/primitives -> LtWideNode / LtTri (once per scene)
// ------------------------------------------------------------------------------------------------
__global__ void k_inner_flags(const RefNode* __restrict__ nodes, int n, int* __restrict__ flags) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flags[i] = nodes[i].primitiveCount == 0 ? 1 : 0;
}

__global__ void k_build_wide(const RefNode* __restrict__ nodes, int n, const int* __restrict__ innerRank,
                             LtWideNode* __restrict__ wide) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  RefNode nd = nodes[i];
  if (nd.primitiveCount != 0) return;
  int li = i + 1, ri = nd.offset;
  RefNode l = nodes[li], r = nodes[ri];
  LtWideNode w;
  w.bx = make_float4(l.boundsMin[0], l.boundsMax[0], r.boundsMin[0], r.boundsMax[0]);
  w.by = make_float4(l.boundsMin[1], l.boundsMax[1], r.boundsMin[1], r.boundsMax[1]);
  w.bz = make_float4(l.boundsMin[2], l.boundsMax[2], r.boundsMin[2], r.boundsMax[2]);
  int lref = l.primitiveCount > 0 ? ~l.offset : innerRank[li];
  int rref = r.primitiveCount > 0 ? ~r.offset : innerRank[ri];
  w.meta = make_int4(lref, rref, (int)nd.axis, (int)((unsigned)l.primitiveCount | ((unsigned)r.primitiveCount << 16)));
  wide[innerRank[i]] = w;
}

// Threaded form of a LARGE tree (LtThreadNode, see lens_trace_b200_device.cuh; small trees are threaded on the host,
// lt_capi.cu: build_threaded): one thread per reference node walks from the root to its node through the
// depth-first index ranges (the left subtree of inner node i is [i+1, offset), the right one [offset, end)) and
// accumulates, for all eight sign octants at once, the node's position in that octant's visit order -- descending
// into the child the octant visits second skips the whole subtree of the one it visits first.
__global__ void k_build_threaded(const RefNode* __restrict__ nodes, int n, LtThreadNode* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  int pos[8];
#pragma unroll
  for (int o = 0; o < 8; o++) pos[o] = 0;
  int i = 0, end = n;
  while (i != t) {
    const int right = nodes[i].offset, axis = nodes[i].axis;
    const int sizeL = right - (i + 1), sizeR = end - right;
    const bool goRight = t >= right;
#pragma unroll
    for (int o = 0; o < 8; o++) {
      const bool neg = (o >> axis) & 1;       // this octant visits the second child first (basic.cu:180-186)
      const bool childIsFar = goRight != neg;
      pos[o] += 1 + (childIsFar ? (neg ? sizeR : sizeL) : 0);
    }
    if (goRight) {
      i = right;
    } else {
      end = right;
      i = i + 1;
    }
  }
  const RefNode r = nodes[t];
  const bool leaf = r.primitiveCount > 0;
  const int size = end - t;
#pragma unroll
  for (int o = 0; o < 8; o++) {
    const int e = pos[o] + size;
    const int skip = e >= n ? LT_DONE : o * n + e;
    const bool nx = o & 1, ny = o & 2, nz = o & 4;
    LtThreadNode rec;
    rec.a = make_float4(nx ? r.boundsMax[0] : r.boundsMin[0], ny ? r.boundsMax[1] : r.boundsMin[1],
                        nz ? r.boundsMax[2] : r.boundsMin[2], nx ? r.boundsMin[0] : r.boundsMax[0]);
    rec.b = make_float4(ny ? r.boundsMin[1] : r.boundsMax[1], nz ? r.boundsMin[2] : r.boundsMax[2],
                        __int_as_float(leaf ? ~r.offset : 0), __int_as_float(skip));
    out[(size_t)o * n + pos[o]] = rec;
  }
}

int lt_launch_build_threaded(const RefNode* dNodes, int nodeCount, LtThreadNode* dOut, cudaStream_t stream) {
  k_build_threaded<<<(nodeCount + 127) / 128, 128, 0, stream>>>(dNodes, nodeCount, dOut);
  return 1;
}

__global__ void k_build_tris(const RefPrim* __restrict__ prims, int n, LtTri* __restrict__ tris) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const RefPrim* p = prims + i;
  float ax = p->a[0], ay = p->a[1], az = p->a[2];
  LtTri t;
  t.q0 = make_float4(ax, ay, az, FSUB(p->b[0], ax));
  t.q1 = make_float4(FSUB(p->b[1], ay), FSUB(p->b[2], az), FSUB(p->c[0], ax), FSUB(p->c[1], ay));
  t.q2 = make_float4(FSUB(p->c[2], az), __int_as_float(p->materialIndex), 0.0f, 0.0f);
  tris[i] = t;
}

// ------------------------------------------------------------------------------------------------
// host-side launchers
// ------------------------------------------------------------------------------------------------
int lt_launch_debug_random(const float* fx, const float* fy, const float* seed, int n, float* out, cudaStream_t stream) {
  k_debug_random<<<(n + 255) / 256, 256, 0, stream>>>(fx, fy, seed, n, out);
  return 1;
}

int lt_launch_debug_hemisphere(const float* u1, const float* u2, const float* up, int n, float* out,
                               cudaStream_t stream) {
  k_debug_hemisphere<<<(n + 255) / 256, 256, 0, stream>>>(u1, u2, up, n, out);
  return 1;
}

int lt_launch_inner_flags(const RefNode* dNodes, int nodeCount, int* dFlags, cudaStream_t stream) {
  k_inner_flags<<<(nodeCount + 255) / 256, 256, 0, stream>>>(dNodes, nodeCount, dFlags);
  return 1;
}

size_t lt_scan_temp_bytes(int n) {
  size_t bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, bytes, (const int*)nullptr, (int*)nullptr, n);
  return bytes;
}

int lt_launch_exclusive_scan(void* dTemp, size_t tempBytes, const int* dIn, int* dOut, int n, cudaStream_t stream) {
  cub::DeviceScan::ExclusiveSum(dTemp, tempBytes, dIn, dOut, n, stream);
  return 1;
}

int lt_launch_reflatten(const RefNode* dNodes, int nodeCount, const RefPrim* dPrims, int primCount,
                        const int* dInnerRank, LtWideNode* dWide, LtTri* dTris, cudaStream_t stream) {
  k_build_wide<<<(nodeCount + 255) / 256, 256, 0, stream>>>(dNodes, nodeCount, dInnerRank, dWide);
  k_build_tris<<<(primCount + 255) / 256, 256, 0, stream>>>(dPrims, primCount, dTris);
  return 2;
}

static size_t stack_bytes(const LtSceneDev& sc, bool cull) { return lt_traversal_smem(sc, cull); }

// Dynamic shared memory beyond 48 KB needs an opt-in per kernel (and per device): the culled mode on a tree deeper
// than 40 levels asks for up to (2 * 64 + 16) * 512 = 73 728 bytes.
#define LT_MAX_TRAVERSAL_SMEM ((2 * 64 + LT_MAX_BATCH) * LT_BLOCK * (int)sizeof(int))
static void opt_in_smem(size_t smem) {
  if (smem <= 48 * 1024) return;
  static bool done[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || done[dev]) return;
  done[dev] = true;
  cudaFuncSetAttribute(k_flat<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, LT_MAX_TRAVERSAL_SMEM);
  cudaFuncSetAttribute(k_flat<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LT_MAX_TRAVERSAL_SMEM);
  cudaFuncSetAttribute(k_path<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, LT_MAX_TRAVERSAL_SMEM);
  cudaFuncSetAttribute(k_path<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LT_MAX_TRAVERSAL_SMEM);
  cudaFuncSetAttribute(k_primary_hits, cudaFuncAttributeMaxDynamicSharedMemorySize, LT_MAX_TRAVERSAL_SMEM);
  cudaFuncSetAttribute(k_flat_stream, cudaFuncAttributeMaxDynamicSharedMemorySize, LT_MAX_TRAVERSAL_SMEM);
}

static int tile_blocks(int width, int height) { return ((width + 15) / 16) * ((height + 7) / 8); }

// the threaded tree is used by the exact, uncounted kernels only (the stats kernels count in the stack traversal,
// whose tests are the same ones; LT_FLAG_NO_THREADED = 16 selects the stack traversal for comparison)
// coherent: the launch traces camera rays and shadow rays towards a light only (the two lighting kernels on the
// megakernel) -- a large scene's threaded copies (tnodesCoherent) then pay: 1 M triangles, 1080p, primary + shadow
// 0.96 instead of 1.10 ms.  For the incoherent rays of GI they lose (56.8 instead of 42.6 ms per 16-spp frame: eight
// copies of the tree no longer fit in L2), and the tile-fetching k_flat_stream is faster on the child-pair tree
// (0.66 against 0.72 ms: half the dependent steps per ray)
static LtSceneDev scene_for_flags(const LtSceneDev& sc, int flags, bool coherent = false) {
  LtSceneDev s = sc;
  if (coherent && s.tnodes == nullptr) s.tnodes = s.tnodesCoherent;
  if (flags & (1 | 2 | 16)) s.tnodes = nullptr;
  return s;
}

static int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

int lt_launch_render(const LtSceneDev& scIn, const LtLaunch& L, float* dOut, LtCounters* dCounters, int* dWork,
                     int smCount, cudaStream_t stream) {
  // camera rays and one shadow ray per hit: the two lighting kernels
  const bool coherentRays = L.kernel == 3 || L.kernel == 4;
  const LtSceneDev sc = scene_for_flags(scIn, L.flags, coherentRays);
  int blocks = tile_blocks(L.width, L.height);
  size_t smem = stack_bytes(sc, (L.flags & 2) != 0);
  opt_in_smem(smem);
  bool stats = (L.flags & 1) != 0;
  bool flat = (L.kernel <= 2);
  // exact, uncounted launches of the deterministic pipelines on large scenes: persistent warps fetching tiles
  if (flat && !(L.flags & (1 | 2 | LT_LAUNCH_FLAG_NO_STREAM)) && dWork != nullptr && sc.tnodes == nullptr &&
      sc.nodeCount >= env_int("LT_STREAM_MIN_NODES", 100000)) {
    int blocksPerSm = (int)((200 * 1024) / smem);
    if (blocksPerSm > 8) blocksPerSm = 8;  // measured 4 .. 10: no difference (the longest tile bounds the kernel)
    if (blocksPerSm < 1) blocksPerSm = 1;
    int grid = smCount * blocksPerSm;
    const int warpsNeeded = (((L.width + 7) >> 3) * ((L.height + 3) >> 2) + 3) / 4;  // blocks of 4 warps, one tile each
    if (grid > warpsNeeded) grid = warpsNeeded;
    cudaMemsetAsync(dWork, 0, sizeof(int), stream);
    k_flat_stream<<<grid, LT_BLOCK, smem, stream>>>(sc, L, dOut, dWork);
    return 1;
  }
  if (flat) {
    if (stats) k_flat<true><<<blocks, LT_BLOCK, smem, stream>>>(sc, L, dOut, dCounters);
    else k_flat<false><<<blocks, LT_BLOCK, smem, stream>>>(sc, L, dOut, nullptr);
  } else {
    if (stats) k_path<true><<<blocks, LT_BLOCK, smem, stream>>>(sc, L, dOut, dCounters);
    else k_path<false><<<blocks, LT_BLOCK, smem, stream>>>(sc, L, dOut, nullptr);
  }
  return 1;
}

int lt_launch_primary_hits(const LtSceneDev& scIn, const RefCamera& cam, int kernel, int flags, int width, int height,
                           int* dIds, int* dHit, float* dTuv, cudaStream_t stream) {
  const LtSceneDev sc = scene_for_flags(scIn, flags);
  opt_in_smem(stack_bytes(sc, (flags & 2) != 0));
  k_primary_hits<<<tile_blocks(width, height), LT_BLOCK, stack_bytes(sc, (flags & 2) != 0), stream>>>(
      sc, cam, kernel, flags, width, height, dIds, dHit, dTuv);
  return 1;
}
