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
#include <mutex>

// LIST: thread i renders pixel M.list[i] (a masked launch); M2: and keeps the Welford sums at M.m2 (running mean only)
template <bool STATS, bool LIST, bool M2>
__global__ void __launch_bounds__(LT_BLOCK) k_flat(LtSceneDev sc, LtLaunch L, float* __restrict__ out,
                                                   LtCounters* gcnt, LtList M) {
  LT_TRAV_SMEM(s, lt_stack_levels(sc))
  int px, py;
  if (LIST ? !thread_list_pixel(M.list, M.count, L.width, px, py) : !thread_pixel(L.width, L.height, px, py)) return;
  LtCounters cnt = {0, 0, 0};
  float fx, fy;
  Trav t;
  t.r = camera_ray(L.cam, px, lt_image_row(L, py), L.width, L.fullHeight, fx, fy);
  const float tInit = lt_tinit(L.kernel), epsThr = lt_eps(L.kernel);
  float color[3] = {0.0f, 0.0f, 0.0f};
  const bool cull = (L.flags & LT_DEV_FLAG_CULL) != 0;
  if (cull) trace_cull<STATS>(t, sc, -1, tInit, epsThr, s, cnt);
  else trace<STATS>(t, sc, -1, tInit, epsThr, false, s, cnt);
  if (t.h.hit == 1) {
    if (L.kernel == LT_DEV_KERNEL_CUSTOM_BARY) {  // custom_opencl.cl:240
      color[0] = t.h.u;
      color[1] = t.h.v;
      color[2] = bary0(t.h.u, t.h.v);
    } else {  // basic.cu:312-326
      const RefMaterial* mat = sc.mats + sc.prims[t.h.prim].materialIndex;
      if (mat->dissolve < 1.0f) {
        lens_path<STATS>(sc, t, tInit, epsThr, s, cull, cnt);
        if (t.h.hit == 1) mat = sc.mats + sc.prims[t.h.prim].materialIndex;
      }
      color[0] = mat->diffuse[0];
      color[1] = mat->diffuse[1];
      color[2] = mat->diffuse[2];
    }
  }
  const long long pixel = (long long)py * L.width + px;
  long long id = pixel * L.depth;
  FrameSink sink;
  sink.begin(L, out, id);
  M2Sink w;
  if (M2) w.begin(L.cam.frameCount > 0, M.m2, pixel);
  // the image is the same for every frame (no RNG): apply the frame combiner `frames` times
  for (int f = 0; f < L.frames; f++) sink_frame<M2>(sink, w, L, L.cam.frameCount + (unsigned)f * L.frameStride, color);
  sink.end(out, id);
  if (M2) w.end(M.m2, pixel);
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
  LT_TRAV_SMEM(s, lt_stack_levels(sc))
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
      while (!trav_iter_lean<false>(t, sc, s.stkAddr, s.fifoAddr, epsThr, kLeanNodeSteps, kLeanTriTests, cnt)) {
      }
      const Hit h = t.h;
      if (stage == 0) {
        if (h.hit != 1) break;
        if (L.kernel == LT_DEV_KERNEL_CUSTOM_BARY) {  // custom_opencl.cl:240
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
    if (L.kernel != LT_DEV_KERNEL_CUSTOM_BARY && (t.h.hit == 1 || ignore >= 0)) {
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
// LIST, M2: as k_flat
template <bool STATS, bool LIST, bool M2>
__global__ void __launch_bounds__(LT_BLOCK) k_path(LtSceneDev sc, LtLaunch L, float* __restrict__ out,
                                                   LtCounters* gcnt, LtList M) {
  // the persistent megakernel does not cull (LT_FLAG_CULL selects the wavefront pipeline)
  LT_TRAV_SMEM(s, lt_stack_levels(sc))
  int px, py;
  bool alive = LIST ? thread_list_pixel(M.list, M.count, L.width, px, py) : thread_pixel(L.width, L.height, px, py);
  LtCounters cnt = {0, 0, 0};
  const PathConsts pc = path_consts(L);

  float fx = 0.0f, fy = 0.0f;
  Ray cameraRay = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 1.0f};
  long long id = 0;
  FrameSink sink;
  sink.acc[0] = sink.acc[1] = sink.acc[2] = 0.0f;
  M2Sink w;
  if (M2) w.m2[0] = w.m2[1] = w.m2[2] = 0.0f;
  if (alive) {
    cameraRay = camera_ray(L.cam, px, lt_image_row(L, py), L.width, L.fullHeight, fx, fy);
    id = ((long long)py * L.width + px) * L.depth;
    sink.begin(L, out, id);
    if (M2) w.begin(L.cam.frameCount > 0, M.m2, (long long)py * L.width + px);
  }

  int frame = 0, sample = 0;
  float frameColor[3] = {0.0f, 0.0f, 0.0f};
  unsigned sampleIndex = (pc.samplesPerFrame == 25) ? L.cam.frameCount * 32u : L.cam.frameCount;
  PathState ps;
  ps.nrm[0] = ps.nrm[1] = ps.nrm[2] = 0.0f;
  ps.diffuse[0] = ps.diffuse[1] = ps.diffuse[2] = 0.0f;
  ps.dLight = 0.0f;
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
          sink_frame<M2>(sink, w, L, L.cam.frameCount + (unsigned)frame * L.frameStride, frameColor);
          sample = 0;
          frame++;
          if (frame >= L.frames) {
            sink.end(out, id);
            if (M2) w.end(M.m2, id / L.depth);
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
          traversing = !trav_iter_threaded(t, sc, s.fifoAddr, pc.epsThr, kThreadedNodeSteps, kThreadedTriTests);
        } else {
          int n = trav_collect<STATS>(t, sc, s.stk, s.list, LT_MAX_BATCH, cnt);
          trav_test<STATS>(t, sc, s.list, n, pc.epsThr, cnt);
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
  LT_TRAV_SMEM(s, lt_stack_levels(sc))
  int px, py;
  if (!thread_pixel(width, height, px, py)) return;
  LtCounters cnt = {0, 0, 0};
  float fx, fy;
  Trav t;
  t.r = camera_ray(cam, px, py, width, height, fx, fy);
  if (flags & LT_DEV_FLAG_CULL) trace_cull<false>(t, sc, -1, lt_tinit(kernel), lt_eps(kernel), s, cnt);
  else trace<false>(t, sc, -1, lt_tinit(kernel), lt_eps(kernel), false, s, cnt);
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
// lt_tree.cpp: lt_build_threaded): one thread per reference node walks from the root to its node through the
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

// One frame of a plug-in (lt_render_plugin_frames) folded into the accumulator: the arithmetic of the built-in
// pipelines' FrameSink for the frame with frameCount L.cam.frameCount, one pixel per thread.  Per pixel at depth 3 it
// reads 12 B of sample and 12 B of accumulator and writes 12 B.
__global__ void k_plugin_accumulate(LtLaunch L, const float* __restrict__ sample, float* __restrict__ acc,
                                    long long pixels) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < pixels; i += stride) {
    const long long id = i * L.depth;
    const float c[3] = {sample[id + 0], sample[id + 1], sample[id + 2]};
    FrameSink sink;
    sink.begin(L, acc, id);
    sink.frame(L, L.cam.frameCount, c);
    sink.end(acc, id);
  }
}

// The pixels of a mask (nonzero bytes, width x height row-major; nullptr: every pixel) as the pixel list of a masked
// launch: thread t of a full-image grid looks at the pixel thread_pixel gives it, and each warp appends its set pixels
// in lane order with one atomic, so a warp's 8x4 tile stays together in the list and the camera rays of the threads
// that render it stay coherent.  The order of the warps' runs varies from call to call; no pixel's value depends on it.
__global__ void __launch_bounds__(LT_BLOCK) k_mask_compact(const unsigned char* __restrict__ mask, int width,
                                                           int height, int* __restrict__ list, int* __restrict__ count) {
  int px, py;
  const bool valid = thread_pixel(width, height, px, py);
  const int pixel = valid ? py * width + px : 0;
  const bool set = valid && (mask == nullptr || mask[pixel] != 0);
  const unsigned lane = threadIdx.x & 31u, m = __ballot_sync(0xffffffffu, set);
  if (m == 0u) return;
  int base = 0;
  if (lane == 0u) base = atomicAdd(count, __popc(m));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (set) list[base + __popc(m & ((1u << lane) - 1u))] = pixel;
}

// lt_debug_ctx_list_order: the list of a masked launch in reverse order, so that tests can render one mask through two
// list orders
__global__ void k_list_reverse(int* __restrict__ list, int count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count / 2) return;
  const int a = list[i], b = list[count - 1 - i];
  list[i] = b;
  list[count - 1 - i] = a;
}

// Appends the pixel of every lane with `set` to list at *count, in lane order, with one atomic per warp (the whole warp
// calls it, as k_mask_compact appends); list == nullptr only counts.
__device__ __forceinline__ void warp_append(bool set, int pixel, int* __restrict__ list, int* __restrict__ count) {
  const unsigned lane = threadIdx.x & 31u, m = __ballot_sync(0xffffffffu, set);
  if (m == 0u) return;
  int base = 0;
  if (lane == 0u) base = atomicAdd(count, __popc(m));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (set && list) list[base + __popc(m & ((1u << lane) - 1u))] = pixel;
}

// The first list of an adaptive call on one part of a row partition (lt_render_adaptive on a multi-GPU context, and
// lt_debug_ctx_adaptive_part): the pixels of every parts-th block of LT_TILE_ROWS rows from block `part`, in the order
// k_mask_compact lists a full image.  The 16x8 tiles of thread_pixel lie inside one row block, so whole tiles are listed.
__global__ void __launch_bounds__(LT_BLOCK) k_rows_compact(int width, int height, int parts, int part,
                                                           int* __restrict__ list, int* __restrict__ count) {
  int px, py;
  const bool valid = thread_pixel(width, height, px, py);
  warp_append(valid && (py / LT_TILE_ROWS) % parts == part, py * width + px, list, count);
}

// lt_render_adaptive's stopping rule after a round of `count` listed pixels, each with n frames behind it: thread i
// looks at pixel list[i], records n in frames (when given), and the pixel goes on when no channel's relative standard
// error e_k = sqrt(m2_k / (n (n - 1))) / max(mean_k, floor) is NaN and one exceeds target (FP32, one rounding per
// operation; a NaN mean is kept by the comparison, as torch's clamp_min keeps it).  The pixels that go on are appended to
// `next` as k_mask_compact appends, so a warp's run of a tile stays together and the next round's camera rays stay
// coherent; next == nullptr (the round that reaches max_frames) only counts them.  Reads 28 B per listed pixel at depth 3.
__global__ void __launch_bounds__(LT_BLOCK) k_adaptive_select(const int* __restrict__ list, int count,
                                                              const float* __restrict__ mean, int depth,
                                                              const float* __restrict__ m2, unsigned* __restrict__ frames,
                                                              unsigned n, float target, float floor,
                                                              int* __restrict__ next, int* __restrict__ nextCount) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  int pixel = 0;
  bool more = false;
  if (i < count) {
    pixel = list[i];
    if (frames) frames[pixel] = n;
    const float d = __fmul_rn((float)n, (float)(n - 1u));
    bool nan = false, above = false;
    for (int k = 0; k < 3; k++) {
      const float mk = mean[(long long)pixel * depth + k];
      const float e = __fdiv_rn(__fsqrt_rn(__fdiv_rn(m2[3ll * pixel + k], d)), mk < floor ? floor : mk);
      nan |= e != e;
      above |= e > target;
    }
    more = !nan && above;
  }
  warp_append(more, pixel, next, nextCount);
}

// ------------------------------------------------------------------------------------------------
// host-side launchers
// ------------------------------------------------------------------------------------------------
int lt_launch_list_reverse(int* dList, int count, cudaStream_t stream) {
  if (count < 2) return 0;
  k_list_reverse<<<(count / 2 + 255) / 256, 256, 0, stream>>>(dList, count);
  return 1;
}

int lt_launch_mask_compact(const unsigned char* dMask, int width, int height, int* dList, int* dCount,
                           cudaStream_t stream) {
  cudaMemsetAsync(dCount, 0, sizeof(int), stream);
  k_mask_compact<<<((width + 15) / 16) * ((height + 7) / 8), LT_BLOCK, 0, stream>>>(dMask, width, height, dList, dCount);
  return 1;
}

int lt_launch_rows_compact(int width, int height, int parts, int part, int* dList, int* dCount, cudaStream_t stream) {
  cudaMemsetAsync(dCount, 0, sizeof(int), stream);
  k_rows_compact<<<((width + 15) / 16) * ((height + 7) / 8), LT_BLOCK, 0, stream>>>(width, height, parts, part, dList,
                                                                                     dCount);
  return 1;
}

int lt_launch_adaptive_select(const int* dList, int count, const float* dMean, int depth, const float* dM2,
                              unsigned* dFrames, unsigned n, float target, float floor, int* dNext, int* dNextCount,
                              cudaStream_t stream) {
  cudaMemsetAsync(dNextCount, 0, sizeof(int), stream);
  k_adaptive_select<<<(count + LT_BLOCK - 1) / LT_BLOCK, LT_BLOCK, 0, stream>>>(dList, count, dMean, depth, dM2, dFrames,
                                                                                n, target, floor, dNext, dNextCount);
  return 1;
}

int lt_launch_debug_random(const float* fx, const float* fy, const float* seed, int n, float* out, cudaStream_t stream) {
  k_debug_random<<<(n + 255) / 256, 256, 0, stream>>>(fx, fy, seed, n, out);
  return 1;
}

int lt_launch_debug_hemisphere(const float* u1, const float* u2, const float* up, int n, float* out,
                               cudaStream_t stream) {
  k_debug_hemisphere<<<(n + 255) / 256, 256, 0, stream>>>(u1, u2, up, n, out);
  return 1;
}

int lt_launch_plugin_accumulate(const LtLaunch& L, const float* sample, float* acc, int smCount, cudaStream_t stream) {
  const long long pixels = (long long)L.width * L.height;
  const long long need = (pixels + 255) / 256, cap = (long long)smCount * 8;
  k_plugin_accumulate<<<(unsigned)(need < cap ? need : cap), 256, 0, stream>>>(L, sample, acc, pixels);
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

// The culled mode on a tree deeper than 40 levels asks for up to (2 * 64 + 16) * 512 = 73 728 bytes.
static const int kMaxTraversalSmem = (int)lt_traversal_smem(64, LT_BLOCK, true);
// the traversal kernels' dynamic shared-memory limit raised to kMaxTraversalSmem on the current device
static void opt_in_traversal_kernels() {
  const void* const mine[] = {(const void*)k_flat<false, false, false>, (const void*)k_flat<true, false, false>,
                              (const void*)k_flat<false, true, false>,  (const void*)k_flat<true, true, false>,
                              (const void*)k_flat<false, true, true>,   (const void*)k_flat<true, true, true>,
                              (const void*)k_path<false, false, false>, (const void*)k_path<true, false, false>,
                              (const void*)k_path<false, true, false>,  (const void*)k_path<true, true, false>,
                              (const void*)k_path<false, true, true>,   (const void*)k_path<true, true, true>,
                              (const void*)k_primary_hits,              (const void*)k_flat_stream};
  for (const void* k : mine) cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxTraversalSmem);
  for (const void* k : lt_wf_traversal_kernels)
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxTraversalSmem);
}

// Once per device.  A thread that finds the device done may launch at once, so call_once returns to no thread before
// every attribute is set: several host threads render on one device when a caller drives two contexts there, and in
// the members of a shared group (lt_debug_ctx_create_shared).
void lt_opt_in_traversal_smem(size_t smem) {
  if (smem <= 48 * 1024) return;
  static std::once_flag done[64];
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return;
  std::call_once(done[dev], opt_in_traversal_kernels);
}

template <bool LIST, bool M2>
static void launch_megakernel(const LtSceneDev& sc, const LtPlan& plan, const LtLaunch& L, float* dOut,
                              LtCounters* dCounters, const LtList& M, cudaStream_t stream) {
  const size_t smem = plan.smemStack;
  if (plan.pipeline == LT_PIPE_FLAT) {
    if (plan.stats) k_flat<true, LIST, M2><<<plan.grid, LT_BLOCK, smem, stream>>>(sc, L, dOut, dCounters, M);
    else k_flat<false, LIST, M2><<<plan.grid, LT_BLOCK, smem, stream>>>(sc, L, dOut, nullptr, M);
  } else {
    if (plan.stats) k_path<true, LIST, M2><<<plan.grid, LT_BLOCK, smem, stream>>>(sc, L, dOut, dCounters, M);
    else k_path<false, LIST, M2><<<plan.grid, LT_BLOCK, smem, stream>>>(sc, L, dOut, nullptr, M);
  }
}

int lt_launch_render(const LtSceneDev& sc, const LtPlan& plan, const LtLaunch& L, float* dOut, LtCounters* dCounters,
                     int* dWork, cudaStream_t stream, const LtList* list) {
  lt_opt_in_traversal_smem(plan.smemStack);
  if (plan.pipeline == LT_PIPE_FLAT_STREAM) {
    cudaMemsetAsync(dWork, 0, sizeof(int), stream);
    k_flat_stream<<<plan.grid, LT_BLOCK, plan.smemStack, stream>>>(sc, L, dOut, dWork);
  } else if (!list) {
    launch_megakernel<false, false>(sc, plan, L, dOut, dCounters, LtList{}, stream);
  } else if (!list->m2) {
    launch_megakernel<true, false>(sc, plan, L, dOut, dCounters, *list, stream);
  } else {
    launch_megakernel<true, true>(sc, plan, L, dOut, dCounters, *list, stream);
  }
  return 1;
}

int lt_launch_primary_hits(const LtSceneDev& sc, const LtPlan& plan, const RefCamera& cam, int kernel, int flags,
                           int width, int height, int* dIds, int* dHit, float* dTuv, cudaStream_t stream) {
  lt_opt_in_traversal_smem(plan.smemStack);
  k_primary_hits<<<plan.grid, LT_BLOCK, plan.smemStack, stream>>>(sc, cam, kernel, flags, width, height, dIds, dHit,
                                                                   dTuv);
  return 1;
}
