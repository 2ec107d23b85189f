// lt_wavefront.cu -- wavefront form of the stochastic pipelines (basic_lighting / accumulator /
// global_illumination): the same per-path arithmetic as k_path (lt_kernels.cu), reorganised so that
// every kernel does one kind of work for every ray that needs it.
//
//   primary    round 0 fused: camera ray -> trace -> shade for every (pixel, frame) path of the batch
//   trace      persistent warps pull rays from the queue; a lane that finishes its ray pulls the
//              next one at once, so lanes never wait for the longest ray of their warp
//   shade      one thread per finished ray: consume the hit (shade_step), append the next ray of the
//              path to the other queue or deposit the finished sample
//   (trace, shade) x (2 + 2*maxRayDepth) rounds, no host synchronisation: queue sizes stay on the device
//   accumulate per pixel, frames of the batch in order: running mean / weighted sum / store
//
// In a round all rays are of one kind (all primary, all shadow, all extension), shading code runs on
// dense arrays, and the running mean is applied in frame order, so results are bit-identical to
// k_path's.  Path state lives in HBM (64 B/path) between rounds.
#include "lt_internal.h"
#include "lt_device.cuh"

#define WF_BLOCK LT_BLOCK
#define WF_CHUNK 128  // queue entries a warp claims per global atomic (measured 32..1024: 64-256 equal, 1024 -8 %)
// idle lanes a warp waits for before it fetches new rays: lanes that start together walk the top of the tree
// together and share its cache lines (measured: 8 is ~1 % faster than 1 on both the 83-node and the 2 M-node tree)
#define WF_REFILL_LANES 8
#define WF_THREADED_BLOCKS_PER_SM 8  // persistent trace blocks per SM on the threaded tree

struct LtWfBuffers {
  float4* st;         // 64-byte record per path, two 32-byte sectors that are read and written independently:
                      //   S0 = [0] nrm.xyz, -  [1] diffuse.rgb, -      (written when a surface hit is shaded)
                      //   S1 = [2] direct.rgb, extW  [3] indirect.rgb, -   (written when a shadow result is shaded)
                      // stage and depth travel in the queue entry's path word, hitPrim is the ray's ignore index
  float4* frameCol;   // running frame colour of the path (the 25-sample blend, or the single sample)
  float4* rayO[2];    // origin.xyz, tStart
  float4* rayD[2];    // direction.xyz, bits((ignore + 1) | anyHit << 31)
  int* rayPath[2];    // path id of the queue entry | stage << 25 | depth << 27  (WF_PATH_* below)
  float4* hits;       // t, u, v, bits(prim | hit << 31), indexed like the current queue
  int* counts;        // [2q], [2q+1] sizes of the front and the back region of queue q (one 64-bit word per queue, so
                      // that one atomic reserves both), [4] trace work counter.  Rays that need the select-chain
                      // slab test (a zero direction component) are appended from the END of the queue, so they
                      // share warps with each other and not with the ordinary rays
  int capacity;       // entries per queue
};

#define WF_PATH_BITS 25  // a batch holds at most 2^25 paths (lt_capi.cu caps it)
__device__ __forceinline__ int wf_pack_path(int path, int stage, int depth) {
  return path | (stage << WF_PATH_BITS) | (depth << (WF_PATH_BITS + 2));
}

__device__ __forceinline__ void pixel_of_path(long long path, int pixels, int width, int& px, int& py, int& frameLocal) {
  frameLocal = (int)(path / pixels);
  int pixel = (int)(path - (long long)frameLocal * pixels);
  py = pixel / width;
  px = pixel - py * width;
}

// frame index, pixel and film position of a path: table look-up + exact multiply-shift division when the launch
// has them (P.film), the reference's own operations otherwise
struct LtWfPrimary;
__device__ __forceinline__ void film_of_path(const LtWfPrimary& P, long long path, int pixels, const LtLaunch& L,
                                             int& frameLocal, float& fx, float& fy);

// queue entry v of [0, front + back): the front region grows from slot 0, the back region from the last slot
__device__ __forceinline__ int queue_slot(int v, int front, int capacity) {
  return v < front ? v : capacity - 1 - (v - front);
}

// does this ray need the select-chain slab test (trav_begin sets LT_EXACT_SLAB for exactly these)?
__device__ __forceinline__ bool ray_is_degenerate(const Ray& r) {
  return !(finite3(FRCP(r.dx), FRCP(r.dy), FRCP(r.dz)) && finite3(r.ox, r.oy, r.oz));
}

// Block-aggregated append of this thread's ray (if emit) to queue `dst`; every thread of the block calls it the
// same number of times.  One global atomic per block and call -- on a packed 64-bit counter (front count in the
// low word, back count in the high word) -- instead of up to two per warp: ncu attributed 31 % of the shade
// kernel's stall samples to the wait for those same-address atomics.
__device__ __forceinline__ void queue_append(const LtWfBuffers& B, int dst, bool emit, const Ray& r, float tStart,
                                             int ignore, bool anyHit, int path, unsigned lane) {
  __shared__ unsigned s_warpCount[WF_BLOCK / 32];  // front | back << 16 of each warp
  __shared__ unsigned long long s_base;
  const unsigned warp = threadIdx.x >> 5;
  bool back = emit && ray_is_degenerate(r);
  bool front = emit && !back;
  unsigned fm = __ballot_sync(0xffffffffu, front), bm = __ballot_sync(0xffffffffu, back);
  if (lane == 0u) s_warpCount[warp] = (unsigned)__popc(fm) | ((unsigned)__popc(bm) << 16);
  __syncthreads();
  unsigned before = 0u, total = 0u;
#pragma unroll
  for (unsigned w = 0; w < WF_BLOCK / 32; w++) {
    unsigned c = s_warpCount[w];
    total += c;
    if (w < warp) before += c;
  }
  if (threadIdx.x == 0 && total != 0u)
    s_base = atomicAdd(reinterpret_cast<unsigned long long*>(B.counts) + dst,
                       (unsigned long long)(total & 0xffffu) | ((unsigned long long)(total >> 16) << 32));
  __syncthreads();
  if (emit) {
    const unsigned long long base = s_base;
    int slot;
    if (front) slot = (int)(unsigned)base + (int)(before & 0xffffu) + __popc(fm & ((1u << lane) - 1u));
    else slot = B.capacity - 1 - ((int)(unsigned)(base >> 32) + (int)(before >> 16) + __popc(bm & ((1u << lane) - 1u)));
    B.rayO[dst][slot] = make_float4(r.ox, r.oy, r.oz, tStart);
    B.rayD[dst][slot] = make_float4(r.dx, r.dy, r.dz,
                                    __int_as_float((int)((unsigned)(ignore + 1) | (anyHit ? 0x80000000u : 0u))));
    B.rayPath[dst][slot] = path;
  }
}

// warp-aggregated form (no block barrier) for the primary round, where most warps of a sparse view emit nothing
__device__ __forceinline__ void queue_append_warp(const LtWfBuffers& B, int dst, bool emit, const Ray& r, float tStart,
                                                  int ignore, bool anyHit, int path, unsigned lane) {
  bool back = emit && ray_is_degenerate(r);
  bool front = emit && !back;
  unsigned fm = __ballot_sync(0xffffffffu, front), bm = __ballot_sync(0xffffffffu, back);
  if ((fm | bm) == 0u) return;
  unsigned long long base = 0ull;
  if (lane == 0u)
    base = atomicAdd(reinterpret_cast<unsigned long long*>(B.counts) + dst,
                     (unsigned long long)__popc(fm) | ((unsigned long long)__popc(bm) << 32));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (emit) {
    int slot;
    if (front) slot = (int)(unsigned)base + __popc(fm & ((1u << lane) - 1u));
    else slot = B.capacity - 1 - ((int)(unsigned)(base >> 32) + __popc(bm & ((1u << lane) - 1u)));
    B.rayO[dst][slot] = make_float4(r.ox, r.oy, r.oz, tStart);
    B.rayD[dst][slot] = make_float4(r.dx, r.dy, r.dz,
                                    __int_as_float((int)((unsigned)(ignore + 1) | (anyHit ? 0x80000000u : 0u))));
    B.rayPath[dst][slot] = path;
  }
}

__device__ __forceinline__ unsigned sample_index_of(const LtLaunch& L, const PathConsts& pc, int frame, int sample) {
  unsigned fc = L.cam.frameCount + (unsigned)frame * L.frameStride;
  return pc.samplesPerFrame == 25 ? fc * 32u + (unsigned)sample : fc;
}

// Round 0 fused: camera ray -> trace -> shade for every path of the batch.  Primary rays are coherent
// (neighbouring pixels), so one ray per thread is efficient here, and no ray/hit record of the primary
// round ever touches memory; paths that end at once (miss, light hit) only deposit their colour.
// The camera ray of a pixel is the same in every frame and sample of a launch (no sub-pixel jitter anywhere in the
// reference, basic.cu:350-358), so its hit is traced once per pixel per launch and every (pixel, frame) path of
// every batch starts from that record: exactly the hit each of them would have found.
// With `classify` (one-sample-per-frame kernels) it also sorts the pixels into three classes, because two of them
// need no path at all: a camera ray that misses is black in every frame, one that hits a light primitive is white
// in every frame (accumulator.cl:233-238, global_illumination.cl:257-266); only surface hits are "alive" and get
// (pixel, frame) paths.  The alive pixels are compacted into a list (order irrelevant: paths are independent).
struct LtWfPrimary {
  float4* hits;        // per pixel: t, u, v, bits(prim | hit << 31)
  float2* film;        // per pixel: the film position camera_ray computes (FP32 divisions, once per launch)
  unsigned long long divM;  // exact division of a path id (< 2^25) by `pixels`: (id * divM) >> divS
  int divS;                 // (Granlund & Montgomery: divS = 25 + ceil(log2 pixels), divM = ceil(2^divS / pixels))
  int* alive;          // compacted list of alive pixels
  unsigned char* cls;  // per pixel: 0 black, 1 white, 2 alive
  int* aliveCount;
};

__device__ __forceinline__ void film_of_path(const LtWfPrimary& P, long long path, int pixels, const LtLaunch& L,
                                             int& frameLocal, float& fx, float& fy) {
  if (P.film != nullptr) {
    frameLocal = (int)(((unsigned long long)path * P.divM) >> P.divS);
    float2 f = P.film[(int)(path - (long long)frameLocal * pixels)];
    fx = f.x;
    fy = f.y;
  } else {
    int px, py;
    pixel_of_path(path, pixels, L.width, px, py, frameLocal);
    fx = FADD(FDIV((float)px, (float)L.width), -0.5f);
    fy = FADD(FDIV((float)lt_image_row(L, py), (float)L.fullHeight), -0.5f);
  }
}

__global__ void __launch_bounds__(WF_BLOCK) k_wf_primary_trace(LtSceneDev sc, LtLaunch L, LtWfPrimary P, int pixels,
                                                               int classify) {
  LT_SMEM_POINTERS(sc)
  (void)tstk;
  const int pixel = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = pixel < pixels;
  bool alive = false;
  if (valid) {
    int py = pixel / L.width, px = pixel - py * L.width;
    float fx, fy;
    Trav t;
    t.r = camera_ray(L.cam, px, lt_image_row(L, py), L.width, L.fullHeight, fx, fy);
    LtCounters cnt = {0, 0, 0};
    trace<false>(t, sc, -1, lt_tinit(L.kernel), lt_eps(L.kernel), false, stk, list, cnt);
    P.hits[pixel] = make_float4(t.h.t, t.h.u, t.h.v,
                                __int_as_float((int)((unsigned)t.h.prim | (t.h.hit ? 0x80000000u : 0u))));
    P.film[pixel] = make_float2(fx, fy);
    if (classify) {
      const PathConsts pc = path_consts(L);
      const bool lightHit = (pc.isGI || pc.whiteOnLight) && is_light(sc, t.h.prim);  // shade_step, ST_PRIMARY
      alive = !lightHit && t.h.hit == 1;
      P.cls[pixel] = lightHit ? 1 : (alive ? 2 : 0);
    }
  }
  if (classify) {
    const unsigned lane = threadIdx.x & 31u;
    const unsigned m = __ballot_sync(0xffffffffu, alive);
    if (m != 0u) {
      int base = 0;
      if (lane == 0u) base = atomicAdd(P.aliveCount, __popc(m));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (alive) P.alive[base + __popc(m & ((1u << lane) - 1u))] = pixel;
    }
  }
}

// primaryHits != nullptr: the per-pixel records of k_wf_primary_trace replace the trace (exact, uncounted launches)
// P.alive != nullptr: only the alive pixels get paths (nf frames x aliveCount pixels, enumerated through the list);
// the path id stays frame * pixels + pixel, so nothing downstream changes.
template <bool STATS>
__global__ void __launch_bounds__(WF_BLOCK) k_wf_primary(LtSceneDev sc, LtLaunch L, LtWfBuffers B, int nf,
                                                         int pixels, int sample, LtCounters* gcnt, LtWfPrimary P) {
  LT_SMEM_POINTERS(sc)
  const float4* __restrict__ primaryHits = P.hits;
  const bool cull = (L.flags & 2) != 0;  // LT_FLAG_CULL: closest-hit rays skip subtrees behind the current hit
  const PathConsts pc = path_consts(L);
  const unsigned lane = threadIdx.x & 31u;
  LtCounters cnt = {0, 0, 0};
  const int perFrame = (!STATS && P.alive != nullptr) ? *P.aliveCount : pixels;
  const long long nPaths = (long long)nf * perFrame;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long rounds = (nPaths + stride - 1) / stride;
  for (long long it = 0; it < rounds; it++) {
    long long p = it * stride + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    bool emit = false;
    Trav t;
    float tStart = 0.0f;
    int ignore = -1, packed = 0;
    bool anyHit = false;
    if (p < nPaths) {
      if (!STATS && P.alive != nullptr) {  // p enumerates (frame, alive pixel): turn it into the path id
        int fl = (int)(p / perFrame);
        int pixel = P.alive[(int)(p - (long long)fl * perFrame)];
        p = (long long)fl * pixels + pixel;
      }
      int px = 0, py = 0, fl;
      float fx, fy;
      if (!STATS && primaryHits != nullptr) {
        film_of_path(P, p, pixels, L, fl, fx, fy);  // the film position camera_ray computes
        float4 hv = primaryHits[(int)(p - (long long)fl * pixels)];
        unsigned hb = (unsigned)__float_as_int(hv.w);
        t.h.t = hv.x; t.h.u = hv.y; t.h.v = hv.z;
        t.h.prim = (int)(hb & 0x7fffffffu);
        t.h.hit = (int)(hb >> 31);
        t.r.ox = t.r.oy = t.r.oz = 0.0f;  // a primary hit is shaded from its hit record alone (shade_step, ST_PRIMARY)
        t.r.dx = t.r.dy = 0.0f;
        t.r.dz = 1.0f;
      } else {
        pixel_of_path(p, pixels, L.width, px, py, fl);
        t.r = camera_ray(L.cam, px, lt_image_row(L, py), L.width, L.fullHeight, fx, fy);
        if (cull) trace_cull<STATS>(t, sc, -1, pc.tInit, pc.epsThr, stk, tstk, cnt);
        else trace<STATS>(t, sc, -1, pc.tInit, pc.epsThr, false, stk, list, cnt);
      }
      PathState ps;
      ps.nrm[0] = ps.nrm[1] = ps.nrm[2] = 0.0f;
      ps.diffuse[0] = ps.diffuse[1] = ps.diffuse[2] = 0.0f;
      ps.extW = 0.0f;
      ps.hitPrim = 0;
      ps.depth = 0;
      path_reset(ps);
      const Hit h = t.h;
      bool done = shade_step(sc, pc, ps, t.r, h, fx, fy, sample_index_of(L, pc, fl, sample), tStart, ignore, anyHit);
      if (done) {
        float col[3], fc[3] = {0.0f, 0.0f, 0.0f};
        sample_colour(pc, ps, col);
        if (sample > 0) {
          float4 prev = B.frameCol[p];
          fc[0] = prev.x; fc[1] = prev.y; fc[2] = prev.z;
        }
        blend_sample(pc, sample, col, fc);
        B.frameCol[p] = make_float4(fc[0], fc[1], fc[2], 0.0f);
      } else {
        emit = true;  // a surface hit: the shadow ray of the direct light sample (direct = indirect = 0 so far)
        float4* wr = B.st + 4ll * p;
        wr[0] = make_float4(ps.nrm[0], ps.nrm[1], ps.nrm[2], 0.0f);
        wr[1] = make_float4(ps.diffuse[0], ps.diffuse[1], ps.diffuse[2], 0.0f);
        packed = wf_pack_path((int)p, ps.stage, ps.depth);
      }
    }
    queue_append_warp(B, 0, emit, t.r, tStart, ignore, anyHit, packed, lane);
  }
  if (STATS) flush_counters(gcnt, cnt);
}

// zero the queue counters before a batch
__global__ void k_wf_reset(LtWfBuffers B) {
  for (int k = 0; k < 6; k++) B.counts[k] = 0;
}

// persistent trace: lanes pull queue entries through one warp-aggregated atomic per refill
// THREADED: stackless traversal of the per-octant threaded tree (sc.tnodes, small scenes); shared memory then
// holds only the leaf FIFO.  Same tests in the same order, hence the same hit records.
// Exact variants: at most 56 registers, so that one block of the other batch's shade kernel (64 registers) fits on an
// SM beside 8 trace blocks.  Left to itself ptxas gives the stack variant 64 registers (no spill instead of 4 bytes),
// and the 1M-triangle GI step then takes 42.7 instead of 42.0-42.4 ms (B200, 1000 W power limit).
template <bool STATS, bool THREADED>
__global__ void __launch_bounds__(WF_BLOCK) __maxnreg__(STATS ? 64 : 56)
    k_wf_trace(LtSceneDev sc, LtLaunch L, LtWfBuffers B, int q, LtCounters* gcnt, const float4* __restrict__ rayO,
               const float4* __restrict__ rayD) {
  extern __shared__ int smemStack[];
  int* stk = smemStack + threadIdx.x;
  int* list = smemStack + (THREADED ? 0 : lt_stack_levels(sc) * LT_BLOCK) + threadIdx.x;
  float* tstk = reinterpret_cast<float*>(smemStack + (lt_stack_levels(sc) + LT_MAX_BATCH) * LT_BLOCK) + threadIdx.x;
  const bool cull = !THREADED && (L.flags & 2) != 0;  // LT_FLAG_CULL: closest-hit rays skip subtrees behind the current hit
  const int nFront = B.counts[2 * q];
  const int n = nFront + B.counts[2 * q + 1];  // virtual entries: front region, then the back region
  const float epsThr = lt_eps(L.kernel);
  const unsigned lane = threadIdx.x & 31u;
  const unsigned stkAddr = (unsigned)__cvta_generic_to_shared(stk);
  const unsigned fifoAddr = (unsigned)__cvta_generic_to_shared(list);
  LtCounters cnt = {0, 0, 0};
  // rayO / rayD = B.rayO[q] / B.rayD[q], resolved by the host: indexing the by-value struct with a run-time q would
  // go through a local-memory copy and generic loads
  Trav t;
  t.cur = LT_DONE;
  int entry = -1;
  // the warp takes queue entries in chunks (one global atomic per WF_CHUNK rays) and deals them to
  // its lanes from warp-uniform registers
  int chunkNext = 0, chunkEnd = 0;
  bool exhausted = false;  // warp-uniform: the queue has no more entries
  while (true) {
    bool has = entry >= 0;
    unsigned need = __ballot_sync(0xffffffffu, !has);
    if (__popc(need) >= WF_REFILL_LANES && !exhausted) {
      if (chunkNext >= chunkEnd) {
        int base = 0;
        if (lane == 0u) base = atomicAdd(&B.counts[4], WF_CHUNK);
        base = __shfl_sync(0xffffffffu, base, 0);
        chunkNext = base;
        chunkEnd = min(base + WF_CHUNK, n);
        if (base >= n) exhausted = true;
      }
      if (!exhausted) {
        int idx = chunkNext + __popc(need & ((1u << lane) - 1u));
        chunkNext += __popc(need);
        if (!has && idx < chunkEnd) {
          idx = queue_slot(idx, nFront, B.capacity);
          float4 o = rayO[idx], d = rayD[idx];
          t.r.ox = o.x; t.r.oy = o.y; t.r.oz = o.z;
          t.r.dx = d.x; t.r.dy = d.y; t.r.dz = d.z;
          unsigned bits = (unsigned)__float_as_int(d.w);
          if (THREADED) trav_begin_threaded(t, sc, (int)(bits & 0x7fffffffu) - 1, o.w, (bits >> 31) != 0u);
          else trav_begin<STATS>(t, sc, (int)(bits & 0x7fffffffu) - 1, o.w, (bits >> 31) != 0u, cnt);
          entry = idx;
          if (t.cur == LT_DONE) {  // missed the root box: finished already
            B.hits[idx] = make_float4(t.h.t, 0.0f, 0.0f, __int_as_float(0));
            entry = -1;
          }
        }
      }
    }
    has = entry >= 0;
    if (!__any_sync(0xffffffffu, has)) {
      if (exhausted) break;
      continue;  // every ray just fetched missed the root box: fetch again
    }
    if (has) {
      bool finished;
      if (THREADED) {
        finished = trav_iter_threaded(t, sc.tnodes, sc.tris, fifoAddr, epsThr, kThreadedNodeSteps, kThreadedTriTests);
      } else if (cull && !t.anyHit) {  // a round holds one kind of ray, so this does not split warps
        for (int k = 0; k < 2 * kLeanNodeSteps && t.cur != LT_DONE; k++)
          trav_step_cull<STATS>(t, sc, stk, tstk, epsThr, cnt);
        finished = t.cur == LT_DONE;
      } else {
        finished = trav_iter_lean<STATS>(t, sc, stkAddr, fifoAddr, epsThr, kLeanNodeSteps, kLeanTriTests, cnt);
      }
      if (finished) {
        B.hits[entry] = make_float4(t.h.t, t.h.u, t.h.v,
                                    __int_as_float((int)((unsigned)t.h.prim | (t.h.hit ? 0x80000000u : 0u))));
        entry = -1;
      }
    }
  }
  if (STATS) flush_counters(gcnt, cnt);
}

// one thread per finished ray of queue q: shade, then append the path's next ray to queue 1-q
// Q (the queue consumed; 1 - Q is appended to) is a template parameter so that B.rayO[Q] etc. are static indexes:
// with a run-time index the compiler copies the pointer arrays of the by-value struct to local memory and every
// queue access starts with a dependent LDL.  Registers sized for 8 resident blocks (<= 64): measured against 10 and
// 12 -- the kernel waits on dependent loads, and registers buy it more loads in flight per thread than warps do.
template <int Q>
__global__ void __launch_bounds__(WF_BLOCK, 8) k_wf_shade(LtSceneDev sc, LtLaunch L, LtWfBuffers B, int pixels,
                                                          int frame0, int sample, LtWfPrimary P) {
  constexpr int q = Q;
  const PathConsts pc = path_consts(L);
  const int nFront = B.counts[2 * q];
  const int n = nFront + B.counts[2 * q + 1];
  const unsigned lane = threadIdx.x & 31u;
  const int rounds = (n + (int)(gridDim.x * blockDim.x) - 1) / (int)(gridDim.x * blockDim.x);
  for (int it = 0; it < rounds; it++) {
    int i = (it * (int)gridDim.x + (int)blockIdx.x) * (int)blockDim.x + (int)threadIdx.x;
    bool valid = i < n;
    if (valid) i = queue_slot(i, nFront, B.capacity);
    bool emit = false;
    Ray r = {0, 0, 0, 0, 0, 1};
    float tStart = 0.0f;
    int ignore = -1, path = 0;
    bool anyHit = false;
    if (valid) {
      const int word = B.rayPath[q][i];
      path = word & ((1 << WF_PATH_BITS) - 1);
      float4 o = B.rayO[q][i], d = B.rayD[q][i], hv = B.hits[i];
      r.ox = o.x; r.oy = o.y; r.oz = o.z;
      r.dx = d.x; r.dy = d.y; r.dz = d.z;
      Hit h;
      h.t = hv.x; h.u = hv.y; h.v = hv.z;
      unsigned hb = (unsigned)__float_as_int(hv.w);
      h.prim = (int)(hb & 0x7fffffffu);
      h.hit = (int)(hb >> 31);
      PathState ps;
      ps.stage = (word >> WF_PATH_BITS) & 3;
      ps.depth = (int)((unsigned)word >> (WF_PATH_BITS + 2));
      // every ray after the primary one ignores the primitive its path stands on (basic_lighting.cl:271,
      // global_illumination.cl:294,311,350)
      ps.hitPrim = (int)((unsigned)__float_as_int(d.w) & 0x7fffffffu) - 1;
      // Only the half of the record this step reads is loaded:
      //   shadow result   : nrm, diffuse (S0); the accumulators (S1) unless it is the direct sample, where they are 0
      //   extension result: nothing for a surface hit; S0 + S1 for a light hit; S1 for a miss (final colour)
      const bool shadowStage = ps.stage == ST_SHADOW_DIRECT || ps.stage == ST_SHADOW_EXT;
      const bool lightHit = ps.stage == ST_EXTENSION && is_light(sc, h.prim);
      const bool surfaceHit = ps.stage == ST_EXTENSION && !lightHit && h.hit == 1;
      const bool needS0 = shadowStage || lightHit;
      const bool needS1 = ps.stage == ST_SHADOW_EXT || (ps.stage == ST_EXTENSION && !surfaceHit);
      const float4* rec = B.st + 4ll * path;
      float4 a = make_float4(0.0f, 0.0f, 0.0f, 0.0f), b = a, c = a, dd = a;
      if (needS0) {
        a = rec[0];
        b = rec[1];
      }
      if (needS1) {
        c = rec[2];
        dd = rec[3];
      }
      ps.nrm[0] = a.x; ps.nrm[1] = a.y; ps.nrm[2] = a.z;
      ps.diffuse[0] = b.x; ps.diffuse[1] = b.y; ps.diffuse[2] = b.z;
      ps.direct[0] = c.x; ps.direct[1] = c.y; ps.direct[2] = c.z; ps.extW = c.w;
      ps.indirect[0] = dd.x; ps.indirect[1] = dd.y; ps.indirect[2] = dd.z;
      int fl;
      float fx, fy;
      film_of_path(P, path, pixels, L, fl, fx, fy);
      unsigned sampleIndex = sample_index_of(L, pc, frame0 + fl, sample);
      bool done = shade_step(sc, pc, ps, r, h, fx, fy, sampleIndex, tStart, ignore, anyHit, lightHit ? 1 : 0);
      if (done) {
        float col[3], fc[3];
        sample_colour(pc, ps, col);
        float4 prev = B.frameCol[path];
        fc[0] = prev.x; fc[1] = prev.y; fc[2] = prev.z;
        blend_sample(pc, sample, col, fc);
        B.frameCol[path] = make_float4(fc[0], fc[1], fc[2], 0.0f);
      } else {
        emit = true;
        float4* wr = B.st + 4ll * path;
        if (surfaceHit) {  // new shading point
          wr[0] = make_float4(ps.nrm[0], ps.nrm[1], ps.nrm[2], 0.0f);
          wr[1] = make_float4(ps.diffuse[0], ps.diffuse[1], ps.diffuse[2], 0.0f);
        } else {  // shadow result or light hit: accumulators, w of the new extension direction
          wr[2] = make_float4(ps.direct[0], ps.direct[1], ps.direct[2], ps.extW);
          wr[3] = make_float4(ps.indirect[0], ps.indirect[1], ps.indirect[2], 0.0f);
        }
        path = wf_pack_path(path, ps.stage, ps.depth);
      }
    }
    queue_append(B, 1 - q, emit, r, tStart, ignore, anyHit, path, lane);
  }
}

// between rounds: the consumed queue becomes the next output queue
__global__ void k_wf_swap(LtWfBuffers B, int q) {
  B.counts[2 * q] = 0;
  B.counts[2 * q + 1] = 0;
  B.counts[4] = 0;
}

// frames of the batch, in order, through the frame combiner (accumulator.frag:10-19)
__global__ void __launch_bounds__(WF_BLOCK) k_wf_accumulate(LtLaunch L, LtWfBuffers B, float* __restrict__ out,
                                                            int pixels, int frame0, int batchFrames,
                                                            const unsigned char* __restrict__ cls) {
  const PathConsts pc = path_consts(L);
  int pixel = blockIdx.x * blockDim.x + threadIdx.x;
  if (pixel >= pixels) return;
  long long id = (long long)pixel * L.depth;
  FrameSink sink;  // a batch that starts at frame0 > 0 continues from what earlier batches wrote to `out`
  if (frame0 == 0) sink.begin(L, out, id);
  else {
    sink.acc[0] = out[id + 0]; sink.acc[1] = out[id + 1]; sink.acc[2] = out[id + 2];
  }
  const int pixelClass = cls ? cls[pixel] : 2;  // black / white pixels have no paths: their sample is constant
  for (int f = 0; f < batchFrames; f++) {
    float4 v = make_float4((float)pixelClass, (float)pixelClass, (float)pixelClass, 0.0f);
    if (pixelClass == 2) v = B.frameCol[(long long)f * pixels + pixel];
    float c[3] = {v.x, v.y, v.z};
    finish_frame_colour(pc, L.kernelMode, c);
    sink.frame(L, L.cam.frameCount + (unsigned)(frame0 + f) * L.frameStride, c);
  }
  sink.end(out, id);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
#define LT_LAUNCH_FLAG_NO_THREADED 16  // == LT_FLAG_NO_THREADED (include/lens_trace_b200.h)

size_t lt_wf_bytes_per_path() {
  return sizeof(float4) * (4 + 1 + 2 * 2 + 1) + sizeof(int) * 2;  // state, frame colour, 2 queues, hits, path ids
}

size_t lt_wf_workspace_bytes(long long nPaths) { return lt_wf_bytes_per_path() * (size_t)nPaths + 256; }

static LtWfBuffers carve(void* workspace, long long nPaths) {
  LtWfBuffers B;
  char* p = (char*)workspace;
  auto take = [&](size_t bytes) {
    char* r = p;
    p += (bytes + 255) & ~(size_t)255;
    return r;
  };
  B.counts = (int*)take(256);
  size_t f4 = sizeof(float4) * (size_t)nPaths;
  B.st = (float4*)take(4 * f4);
  B.frameCol = (float4*)take(f4);
  for (int k = 0; k < 2; k++) {
    B.rayO[k] = (float4*)take(f4);
    B.rayD[k] = (float4*)take(f4);
    B.rayPath[k] = (int*)take(sizeof(int) * (size_t)nPaths);
  }
  B.hits = (float4*)take(f4);
  B.capacity = (int)nPaths;
  return B;
}

size_t lt_wf_workspace_bytes_padded(long long nPaths) {
  // carve() rounds every array up to 256 bytes; the total is a multiple of 256 as well, because batch workspace
  // k > 0 and the primary-record block start at multiples of it and hold float4 arrays (an odd path count would
  // otherwise leave them 8 bytes off a 16-byte boundary: misaligned float4 accesses)
  return ((lt_wf_workspace_bytes(nPaths) + 256 * 16) + 255) & ~(size_t)255;
}

// per-launch primary records: hit (16 B), alive list entry (4 B), class (1 B) per pixel + the alive count
size_t lt_wf_primary_hits_bytes(long long pixels) {
  return (sizeof(float4) + sizeof(float2) + sizeof(int) + 1) * (size_t)pixels + 1024 + 5 * 256;  // 5 arrays, 256-aligned
}

int lt_launch_render_wavefront(const LtSceneDev& scIn, const LtLaunch& L, float* dOut, LtCounters* dCounters,
                               void* workspace, int batchFrames, int smCount, cudaStream_t stream,
                               cudaEvent_t* traceEvents, int maxTraceLaunches, int* traceLaunches,
                               unsigned char* pairKinds, const LtWfAux* aux) {
  LtSceneDev sc = scIn;
  if (L.flags & (1 | 2 | LT_LAUNCH_FLAG_NO_THREADED)) sc.tnodes = nullptr;  // stats / culled / forced stack traversal
  int pairs = 0;
  // which: 0 = before, 1 = after a launch; kind (LT_TIMED_*): what the bracketed kernel does.  Traversal launches
  // are always bracketed when events are given, the other kinds only when the caller passes pairKinds.
  auto mark = [&](int which, cudaStream_t s, int kind = LT_TIMED_TRAVERSAL) {
    if (!traceEvents || pairs >= maxTraceLaunches) return;
    if (kind != LT_TIMED_TRAVERSAL && !pairKinds) return;
    cudaEventRecord(traceEvents[2 * pairs + which], s);
    if (which == 1) {
      if (pairKinds) pairKinds[pairs] = (unsigned char)kind;
      pairs++;
    }
  };
  const int pixels = L.width * L.height;
  const bool stats = (L.flags & 1) != 0;
  const bool isGI = (L.kernel == 5 || L.kernel == 6);
  const int samples = (L.kernel == 3 || L.kernel == 5) ? 25 : 1;
  const int maxDepth = L.maxRayDepth > 0 ? L.maxRayDepth : 16;
  const int rounds = isGI ? 2 + 2 * maxDepth : 2;
  const size_t smem = lt_traversal_smem(sc, (L.flags & 2) != 0);
  if (smem > 48 * 1024) {  // beyond 48 KB (culled mode on a tree deeper than 40) dynamic shared memory is an opt-in
    static bool done[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !done[dev]) {
      done[dev] = true;
      const int most = (2 * 64 + LT_MAX_BATCH) * LT_BLOCK * (int)sizeof(int);
      cudaFuncSetAttribute(k_wf_primary_trace, cudaFuncAttributeMaxDynamicSharedMemorySize, most);
      cudaFuncSetAttribute(k_wf_primary<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, most);
      cudaFuncSetAttribute(k_wf_primary<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, most);
      cudaFuncSetAttribute(k_wf_trace<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, most);
      cudaFuncSetAttribute(k_wf_trace<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, most);
    }
  }
  int blocksPerSm = (int)((200 * 1024) / smem);  // shared memory is what limits residency of the persistent kernel
  if (blocksPerSm > 8) blocksPerSm = 8;
  if (blocksPerSm < 1) blocksPerSm = 1;
  // small scenes: stackless traversal of the threaded tree (exact mode only; the stats variant counts in the
  // stack kernel, whose tests are the same ones)
  const bool threaded = sc.tnodes != nullptr;
  const size_t smemTrace = threaded ? (size_t)LT_MAX_BATCH * LT_BLOCK * sizeof(int) : smem;
  if (threaded) blocksPerSm = WF_THREADED_BLOCKS_PER_SM;
  // Two batches in flight on two streams: the trace kernel of one batch runs beside the shade kernel of the other
  // (different bottlenecks: L1 data pipe vs DRAM).  Measured: reserving room on the SMs for the other batch's blocks
  // (fewer persistent trace blocks) does not pay, nor do 3 or 4 batches in flight (profiles/r2u_overlap_sweep.txt).
  const bool overlap = aux != nullptr && L.frames > batchFrames;
  const int nStreams = overlap ? 2 : 1;
  const int persistentBlocks = smCount * blocksPerSm;
  const size_t wsBytes = lt_wf_workspace_bytes_padded((long long)batchFrames * pixels);
  int preLaunches = 0;
  // primary hits once per pixel per launch (exact, uncounted pipelines); kept behind the batch workspaces
  LtWfPrimary P = {};
  if (!stats && !(L.flags & 2)) {
    char* pb = (char*)workspace + (size_t)nStreams * wsBytes;  // 256-aligned: wsBytes is a multiple of 256
    auto take = [&](size_t bytes) {
      char* r = pb;
      pb += (bytes + 255) & ~(size_t)255;
      return r;
    };
    P.hits = (float4*)take(sizeof(float4) * (size_t)pixels);
    P.film = (float2*)take(sizeof(float2) * (size_t)pixels);
    int l = 0;
    while ((1ll << l) < pixels) l++;
    P.divS = 25 + l;
    P.divM = (unsigned long long)(((1ull << P.divS) + (unsigned long long)pixels - 1ull) / (unsigned long long)pixels);
    const bool classify = samples == 1;
    if (classify) {
      P.alive = (int*)take(sizeof(int) * (size_t)pixels);
      P.aliveCount = (int*)take(256);
      P.cls = (unsigned char*)take((size_t)pixels);
      cudaMemsetAsync(P.aliveCount, 0, sizeof(int), stream);
    }
    mark(0, stream);
    k_wf_primary_trace<<<(pixels + WF_BLOCK - 1) / WF_BLOCK, WF_BLOCK, smem, stream>>>(sc, L, P, pixels, classify ? 1 : 0);
    mark(1, stream);
    preLaunches = 1;
  }
  float4* primaryHits = P.hits;
  if (overlap) {
    cudaEventRecord(aux->fork, stream);
    cudaStreamWaitEvent(aux->extra, aux->fork, 0);
  }
  int launches = preLaunches, batch = 0, lastSide = 0;
  for (int frame0 = 0; frame0 < L.frames; frame0 += batchFrames, batch++) {
    const int side = overlap ? (batch & 1) : 0;
    cudaStream_t st = side ? aux->extra : stream;
    int nf = L.frames - frame0 < batchFrames ? L.frames - frame0 : batchFrames;
    long long nPaths = (long long)nf * pixels;
    LtWfBuffers B = carve((char*)workspace + (size_t)side * wsBytes, (long long)batchFrames * pixels);
    LtLaunch Lb = L;
    Lb.cam.frameCount = L.cam.frameCount + (unsigned)frame0 * L.frameStride;  // frame index 0 of the batch
    int grid = (int)((nPaths + WF_BLOCK - 1) / WF_BLOCK);
    if (grid > smCount * 32) grid = smCount * 32;
    for (int s = 0; s < samples; s++) {
      // round 0 (primary rays) fused into one kernel; its survivors are queue 0
      k_wf_reset<<<1, 1, 0, st>>>(B);
      // a traversal kernel only when it traces the camera rays itself
      mark(0, st, primaryHits ? LT_TIMED_PRIMARY_SHADE : LT_TIMED_TRAVERSAL);
      if (stats) k_wf_primary<true><<<grid, WF_BLOCK, smem, st>>>(sc, Lb, B, nf, pixels, s, dCounters, P);
      else k_wf_primary<false><<<grid, WF_BLOCK, smem, st>>>(sc, Lb, B, nf, pixels, s, nullptr, P);
      mark(1, st, primaryHits ? LT_TIMED_PRIMARY_SHADE : LT_TIMED_TRAVERSAL);
      launches += 2;
      int q = 0;
      for (int r = 1; r < rounds; r++) {
        mark(0, st);
        if (stats) k_wf_trace<true, false><<<persistentBlocks, WF_BLOCK, smem, st>>>(sc, Lb, B, q, dCounters, B.rayO[q], B.rayD[q]);
        else if (threaded) k_wf_trace<false, true><<<persistentBlocks, WF_BLOCK, smemTrace, st>>>(sc, Lb, B, q, nullptr, B.rayO[q], B.rayD[q]);
        else k_wf_trace<false, false><<<persistentBlocks, WF_BLOCK, smem, st>>>(sc, Lb, B, q, nullptr, B.rayO[q], B.rayD[q]);
        mark(1, st);
        mark(0, st, LT_TIMED_SHADE);
        if (q == 0) k_wf_shade<0><<<grid, WF_BLOCK, 0, st>>>(sc, Lb, B, pixels, 0, s, P);
        else k_wf_shade<1><<<grid, WF_BLOCK, 0, st>>>(sc, Lb, B, pixels, 0, s, P);
        mark(1, st, LT_TIMED_SHADE);
        k_wf_swap<<<1, 1, 0, st>>>(B, q);
        launches += 3;
        q = 1 - q;
      }
    }
    // the frame combiner is applied in frame order: this batch's accumulate follows the previous batch's
    if (overlap && batch > 0) cudaStreamWaitEvent(st, aux->order[1 - side], 0);
    mark(0, st, LT_TIMED_ACCUMULATE);
    k_wf_accumulate<<<(pixels + WF_BLOCK - 1) / WF_BLOCK, WF_BLOCK, 0, st>>>(L, B, dOut, pixels, frame0, nf, P.cls);
    mark(1, st, LT_TIMED_ACCUMULATE);
    if (overlap) cudaEventRecord(aux->order[side], st);
    lastSide = side;
    launches++;
  }
  // join: the last accumulate follows every earlier one (chain of order events), and every stream's last kernel is
  // its accumulate, so waiting for the last batch's event puts all of it before what follows on `stream`
  if (overlap && lastSide != 0) cudaStreamWaitEvent(stream, aux->order[lastSide], 0);
  if (traceLaunches) *traceLaunches = pairs;
  return launches;
}
