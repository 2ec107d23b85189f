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
// k_path's.  Between rounds a path's state travels in its queue entry, beside its ray, so every load
// of a queue entry is indexed by its slot and can be issued at once.
// Round 1 holds the first shadow rays of the paths, then extension and shadow rounds alternate (WfRound).  The
// shade kernel is compiled for each kind of round and loads only what that kind reads: a shadow entry its ray,
// shading normal and colours, an extension entry its hit, colours and one float (dLight).  Counting launches that
// retrace light hits mix extension rays into shadow rounds; they keep the full entries (WF_GENERIC).
#include "lt_internal.h"
#include "lt_device.cuh"

#define WF_BLOCK LT_BLOCK
#define WF_CHUNK 128  // queue entries a warp claims per global atomic (measured 32..1024: 64-256 equal, 1024 -8 %)
// idle lanes a warp waits for before it fetches new rays: lanes that start together walk the top of the tree
// together and share its cache lines (measured: 8 is ~1 % faster than 1 on both the 83-node and the 2 M-node tree)
#define WF_REFILL_LANES 8

struct LtWfBuffers {
  float4* frameCol;   // running frame colour of the path (the 25-sample blend, or the single sample)
  float4* rayO[2];    // origin.xyz, tStart
  float4* rayD[2];    // direction.xyz, bits((ignore + 1) | anyHit << 31)
  int* rayPath[2];    // path id of the queue entry | stage << 25 | depth << 27  (WF_PATH_* below)
  // Path state of the queue entry (WfPayload), indexed like the rays: the shade kernel loads it in queue order
  // together with the ray and the hit instead of by path id after them.  Stage and depth travel in the path word,
  // hitPrim is the ray's ignore index.
  float4* payA[2];    // nrm.xyz of the shading point, then bits(material index) for a shadow ray / dLight for an
                      // extension ray (WF_GENERIC); other launches keep only dLight of an extension ray: wf_dlight
  float4* payB[2];    // direct.rgb, indirect.r
  float2* payC[2];    // indirect.gb
  float4* hits;       // t, u, v, bits(prim | hit << 31), indexed like the current queue; other launches than
                      // WF_GENERIC keep only the last word of a shadow ray's hit: wf_hit_words
  int* counts;        // [2q], [2q+1] sizes of the front and the back region of queue q (one 64-bit word per queue, so
                      // that one atomic reserves both), [4] trace work counter.  Rays that need the select-chain
                      // slab test (a zero direction component) are appended from the END of the queue, so they
                      // share warps with each other and not with the ordinary rays
  int capacity;       // entries per queue
};

// The kind of a round, which decides what its queue entries hold and what the shade kernel loads of them.
// WF_GENERIC: every entry holds its full payload and its full hit record (rounds that may mix kinds).
// WF_FIRST_SHADOW: round 1, the shadow rays k_wf_primary emits; direct and indirect are still zero, so the entries
// hold no payB / payC.  WF_SHADOW: the shadow rays of later bounces.  WF_EXTENSION: extension rays; their entries
// hold no payA but dLight.  In the last three a shadow ray's hit is one word.
enum WfRound { WF_GENERIC, WF_FIRST_SHADOW, WF_SHADOW, WF_EXTENSION };

// A round holds either shadow or extension entries, never both, so dLight and the shadow hit words can be dense
// arrays over the start of the buffers whose float4 form the other kind uses: the workspace does not grow.
__device__ __forceinline__ float* wf_dlight(const LtWfBuffers& B, int q) { return reinterpret_cast<float*>(B.payA[q]); }
__device__ __forceinline__ int* wf_hit_words(const LtWfBuffers& B) { return reinterpret_cast<int*>(B.hits); }

#define WF_PATH_BITS 25  // a batch holds at most 2^25 paths (lt_plan.cpp caps it)
__device__ __forceinline__ int wf_pack_path(int path, int stage, int depth) {
  return path | (stage << WF_PATH_BITS) | (depth << (WF_PATH_BITS + 2));
}

// ray word of a queue entry (rayD.w): the primitive the ray ignores + 1 (0: none) | anyHit << 31
__device__ __forceinline__ int wf_ray_word(int ignore, bool anyHit) {
  return (int)((unsigned)(ignore + 1) | (anyHit ? 0x80000000u : 0u));
}
__device__ __forceinline__ int wf_ray_ignore(int word) { return (int)((unsigned)word & 0x7fffffffu) - 1; }
__device__ __forceinline__ bool wf_ray_any_hit(int word) { return ((unsigned)word >> 31) != 0u; }

// hit word of a traced ray (the last word of a hit record, all of a shadow ray's hit): prim | hit << 31
__device__ __forceinline__ int wf_hit_word(const Hit& h) { return (int)((unsigned)h.prim | (h.hit ? 0x80000000u : 0u)); }
__device__ __forceinline__ void wf_hit_unpack(int word, Hit& h) {
  h.prim = (int)((unsigned)word & 0x7fffffffu);
  h.hit = (int)((unsigned)word >> 31);
}

// In a masked launch (LIST) the pixel axis of the path ids is the list index: path id = frame * count + i, pixel list[i]
template <bool LIST = false>
__device__ __forceinline__ void pixel_of_path(long long path, int pixels, int width, int& px, int& py, int& frameLocal,
                                              const int* list = nullptr) {
  frameLocal = (int)(path / pixels);
  int pixel = (int)(path - (long long)frameLocal * pixels);
  if (LIST) pixel = list[pixel];
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

// What the next shading of a queue entry reads of its path, beside the ray (LtWfBuffers::payA/B/C).  A shadow ray's
// shading reads the normal and the diffuse colour of its shading point, an extension ray's only dLight: one word
// holds the material index (the diffuse colour is a load from the small materials table) or dLight.
struct WfPayload {
  float4 a, b;
  float2 c;
};

__device__ __forceinline__ WfPayload wf_payload(const PathState& ps, float sel) {
  WfPayload pl;
  pl.a = make_float4(ps.nrm[0], ps.nrm[1], ps.nrm[2], sel);
  pl.b = make_float4(ps.direct[0], ps.direct[1], ps.direct[2], ps.indirect[0]);
  pl.c = make_float2(ps.indirect[1], ps.indirect[2]);
  return pl;
}

// the stores of one queue entry, for a round of kind OUT
template <int OUT>
__device__ __forceinline__ void queue_store(const LtWfBuffers& B, int dst, int slot, const Ray& r, float tStart,
                                            int ignore, bool anyHit, int path, const WfPayload& pl) {
  B.rayO[dst][slot] = make_float4(r.ox, r.oy, r.oz, tStart);
  B.rayD[dst][slot] = make_float4(r.dx, r.dy, r.dz, __int_as_float(wf_ray_word(ignore, anyHit)));
  B.rayPath[dst][slot] = path;
  if (OUT == WF_EXTENSION) wf_dlight(B, dst)[slot] = pl.a.w;
  else B.payA[dst][slot] = pl.a;
  if (OUT != WF_FIRST_SHADOW) {
    B.payB[dst][slot] = pl.b;
    B.payC[dst][slot] = pl.c;
  }
}

// Block-aggregated append of this thread's ray (if emit) to queue `dst`; every thread of the block calls it the
// same number of times.  One global atomic per block and call -- on a packed 64-bit counter (front count in the
// low word, back count in the high word) -- instead of up to two per warp: ncu attributed 31 % of the shade
// kernel's stall samples to the wait for those same-address atomics.
template <int OUT>
__device__ __forceinline__ void queue_append(const LtWfBuffers& B, int dst, bool emit, const Ray& r, float tStart,
                                             int ignore, bool anyHit, int path, const WfPayload& pl, unsigned lane) {
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
    queue_store<OUT>(B, dst, slot, r, tStart, ignore, anyHit, path, pl);
  }
}

// warp-aggregated form (no block barrier) for the primary round, where most warps of a sparse view emit nothing;
// out: WF_FIRST_SHADOW or WF_GENERIC
__device__ __forceinline__ void queue_append_warp(const LtWfBuffers& B, int dst, bool emit, const Ray& r, float tStart,
                                                  int ignore, bool anyHit, int path, const WfPayload& pl,
                                                  unsigned lane, int out) {
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
    if (out == WF_FIRST_SHADOW) queue_store<WF_FIRST_SHADOW>(B, dst, slot, r, tStart, ignore, anyHit, path, pl);
    else queue_store<WF_GENERIC>(B, dst, slot, r, tStart, ignore, anyHit, path, pl);
  }
}

// sample index of a path whose frame has camera frameCount fc
__device__ __forceinline__ unsigned sample_index_fc(const PathConsts& pc, unsigned fc, int sample) {
  return pc.samplesPerFrame == 25 ? fc * 32u + (unsigned)sample : fc;
}
__device__ __forceinline__ unsigned sample_index_of(const LtLaunch& L, const PathConsts& pc, int frame, int sample) {
  return sample_index_fc(pc, L.cam.frameCount + (unsigned)frame * L.frameStride, sample);
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
  // a call of several views (lt_render_views): frameCount of each (view, frame) pair of the batch, in batch order;
  // nullptr otherwise (the frames of the one camera L.cam)
  const unsigned* frameCounts;
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

// LIST: a masked launch; `pixels` counts the listed pixels, and thread i traces pixel M.list[i] and writes its records
// at i, so that the alive list holds list indices
template <bool LIST>
__global__ void __launch_bounds__(WF_BLOCK) k_wf_primary_trace(LtSceneDev sc, LtLaunch L, LtWfPrimary P, int pixels,
                                                               int classify, LtList M) {
  LT_TRAV_SMEM(s, lt_stack_levels(sc))
  const int pixel = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = pixel < pixels;
  bool alive = false;
  if (valid) {
    const int image = LIST ? M.list[pixel] : pixel;
    int py = image / L.width, px = image - py * L.width;
    float fx, fy;
    Trav t;
    t.r = camera_ray(L.cam, px, lt_image_row(L, py), L.width, L.fullHeight, fx, fy);
    LtCounters cnt = {0, 0, 0};
    trace<false>(t, sc, -1, lt_tinit(L.kernel), lt_eps(L.kernel), false, s, cnt);
    P.hits[pixel] = make_float4(t.h.t, t.h.u, t.h.v, __int_as_float(wf_hit_word(t.h)));
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
// out: the kind of round 1 (WF_FIRST_SHADOW, or WF_GENERIC), which decides what its entries hold
// VIEWS: the nf frames are one view's frames inside a batch that holds several views (L.cam is that view's camera, P
// its records); their paths are numbered from pathBase in the batch
// LIST: a masked launch (`pixels` listed pixels); a launch that traces its camera rays here finds their pixels in M.list
template <bool STATS, bool VIEWS, bool LIST>
__global__ void __launch_bounds__(WF_BLOCK) k_wf_primary(LtSceneDev sc, LtLaunch L, LtWfBuffers B, int nf,
                                                         int pixels, int sample, LtCounters* gcnt, LtWfPrimary P,
                                                         int out, int pathBase, LtList M) {
  LT_TRAV_SMEM(s, lt_stack_levels(sc))
  const float4* __restrict__ primaryHits = P.hits;
  const bool cull = (L.flags & LT_DEV_FLAG_CULL) != 0;  // closest-hit rays skip subtrees behind the current hit
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
    WfPayload pl = {};
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
        t.h.t = hv.x; t.h.u = hv.y; t.h.v = hv.z;
        wf_hit_unpack(__float_as_int(hv.w), t.h);
        t.r.ox = t.r.oy = t.r.oz = 0.0f;  // a primary hit is shaded from its hit record alone (shade_step, ST_PRIMARY)
        t.r.dx = t.r.dy = 0.0f;
        t.r.dz = 1.0f;
      } else {
        pixel_of_path<LIST>(p, pixels, L.width, px, py, fl, M.list);
        t.r = camera_ray(L.cam, px, lt_image_row(L, py), L.width, L.fullHeight, fx, fy);
        if (cull) trace_cull<STATS>(t, sc, -1, pc.tInit, pc.epsThr, s, cnt);
        else trace<STATS>(t, sc, -1, pc.tInit, pc.epsThr, false, s, cnt);
      }
      PathState ps;
      ps.nrm[0] = ps.nrm[1] = ps.nrm[2] = 0.0f;
      ps.diffuse[0] = ps.diffuse[1] = ps.diffuse[2] = 0.0f;
      ps.dLight = 0.0f;
      ps.hitPrim = 0;
      ps.depth = 0;
      path_reset(ps);
      const Hit h = t.h;
      bool done = shade_step(sc, pc, ps, t.r, h, fx, fy, sample_index_of(L, pc, fl, sample), tStart, ignore, anyHit);
      if (VIEWS) p += pathBase;
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
        pl = wf_payload(ps, __int_as_float(sc.prims[h.prim].materialIndex));
        packed = wf_pack_path((int)p, ps.stage, ps.depth);
      }
    }
    queue_append_warp(B, 0, emit, t.r, tStart, ignore, anyHit, packed, pl, lane, out);
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
// hitWords: wf_hit_words(B) on a WF_FIRST_SHADOW or WF_SHADOW round, whose rays store only the last word of their hit;
// nullptr on the others, whose rays store the full record.  (A counting launch traces its shadow rays as closest-hit
// rays, so the round decides this, not the ray.)
template <bool STATS, bool THREADED>
__global__ void __launch_bounds__(WF_BLOCK) __maxnreg__(STATS ? 64 : 56)
    k_wf_trace(LtSceneDev sc, LtLaunch L, LtWfBuffers B, int q, LtCounters* gcnt, const float4* __restrict__ rayO,
               const float4* __restrict__ rayD, int* __restrict__ hitWords) {
  LT_TRAV_SMEM(s, THREADED ? 0 : lt_stack_levels(sc))
  const bool cull = !THREADED && (L.flags & LT_DEV_FLAG_CULL) != 0;  // closest-hit rays skip subtrees behind the current hit
  const int nFront = B.counts[2 * q];
  const int n = nFront + B.counts[2 * q + 1];  // virtual entries: front region, then the back region
  const float epsThr = lt_eps(L.kernel);
  const unsigned lane = threadIdx.x & 31u;
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
          const int rayWord = __float_as_int(d.w);
          if (THREADED) trav_begin_threaded(t, sc, wf_ray_ignore(rayWord), o.w, wf_ray_any_hit(rayWord));
          else trav_begin<STATS>(t, sc, wf_ray_ignore(rayWord), o.w, wf_ray_any_hit(rayWord), cnt);
          entry = idx;
          if (t.cur == LT_DONE) {  // missed the root box: finished already
            if (hitWords) hitWords[idx] = 0;
            else B.hits[idx] = make_float4(t.h.t, 0.0f, 0.0f, __int_as_float(0));
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
        finished = trav_iter_threaded(t, sc, s.fifoAddr, epsThr, kThreadedNodeSteps, kThreadedTriTests);
      } else if (cull && !t.anyHit) {  // a round holds one kind of ray, so this does not split warps
        for (int k = 0; k < 2 * kLeanNodeSteps && t.cur != LT_DONE; k++)
          trav_step_cull<STATS>(t, sc, s.stk, s.tstk, epsThr, cnt);
        finished = t.cur == LT_DONE;
      } else {
        finished = trav_iter_lean<STATS>(t, sc, s.stkAddr, s.fifoAddr, epsThr, kLeanNodeSteps, kLeanTriTests, cnt);
      }
      if (finished) {
        const int word = wf_hit_word(t.h);
        if (hitWords) hitWords[entry] = word;
        else B.hits[entry] = make_float4(t.h.t, t.h.u, t.h.v, __int_as_float(word));
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
// K (WfRound) is the kind of the round: it fixes the stage of every entry and which arrays are loaded.  A shadow
// result reads ray, hit word, payA and (after the first bounce) payB / payC; an extension result reads neither its ray
// nor the normal: a surface hit rebuilds the shading point from the hit, a light hit reads dLight, a miss only
// finishes the sample.  VIEWS: the batch holds (view, frame) pairs; P.frameCounts gives each pair's frameCount.
template <int Q, int K, bool VIEWS>
__global__ void __launch_bounds__(WF_BLOCK, 8) k_wf_shade(LtSceneDev sc, LtLaunch L, LtWfBuffers B, int pixels,
                                                          int frame0, int sample, LtWfPrimary P) {
  constexpr int q = Q;
  constexpr bool generic = K == WF_GENERIC, extension = K == WF_EXTENSION;
  // the kind of the round that consumes what this one appends
  constexpr int OUT = generic ? WF_GENERIC : (extension ? WF_SHADOW : WF_EXTENSION);
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
    WfPayload pl = {};
    if (valid) {
      const int word = B.rayPath[q][i];
      path = word & ((1 << WF_PATH_BITS) - 1);
      float4 o = make_float4(0.0f, 0.0f, 0.0f, 0.0f), d = make_float4(0.0f, 0.0f, 1.0f, 0.0f);
      float4 hv = make_float4(0.0f, 0.0f, 0.0f, 0.0f), pa = hv, pb = hv;
      float2 pc2 = make_float2(0.0f, 0.0f);  // direct and indirect are zero before the first shadow ray is shaded
      float dLight = 0.0f;
      if (!extension) {
        o = B.rayO[q][i];
        d = B.rayD[q][i];
        pa = B.payA[q][i];
      }
      if (generic || extension) hv = B.hits[i];
      else hv.w = __int_as_float(wf_hit_words(B)[i]);
      if (K != WF_FIRST_SHADOW) {
        pb = B.payB[q][i];
        pc2 = B.payC[q][i];
      }
      if (extension) dLight = wf_dlight(B, q)[i];
      r.ox = o.x; r.oy = o.y; r.oz = o.z;
      r.dx = d.x; r.dy = d.y; r.dz = d.z;
      Hit h;
      h.t = hv.x; h.u = hv.y; h.v = hv.z;
      wf_hit_unpack(__float_as_int(hv.w), h);
      PathState ps;
      ps.stage = generic ? (word >> WF_PATH_BITS) & 3
                         : (K == WF_FIRST_SHADOW ? ST_SHADOW_DIRECT : (K == WF_SHADOW ? ST_SHADOW_EXT : ST_EXTENSION));
      ps.depth = (int)((unsigned)word >> (WF_PATH_BITS + 2));
      // every ray after the primary one ignores the primitive its path stands on (basic_lighting.cl:271,
      // global_illumination.cl:294,311,350); an extension result sets it or does not read it
      ps.hitPrim = wf_ray_ignore(__float_as_int(d.w));
      const bool shadowStage = ps.stage == ST_SHADOW_DIRECT || ps.stage == ST_SHADOW_EXT;
      const bool lightHit = ps.stage == ST_EXTENSION && is_light(sc, h.prim);
      const bool surfaceHit = ps.stage == ST_EXTENSION && !lightHit && h.hit == 1;
      ps.nrm[0] = pa.x; ps.nrm[1] = pa.y; ps.nrm[2] = pa.z;
      ps.dLight = extension ? dLight : pa.w;  // read by the light hit of an extension ray only
      ps.diffuse[0] = ps.diffuse[1] = ps.diffuse[2] = 0.0f;  // an extension result sets it or does not read it
      if (shadowStage) {
        const RefMaterial* mat = sc.mats + __float_as_int(pa.w);
        ps.diffuse[0] = mat->diffuse[0]; ps.diffuse[1] = mat->diffuse[1]; ps.diffuse[2] = mat->diffuse[2];
      }
      ps.direct[0] = pb.x; ps.direct[1] = pb.y; ps.direct[2] = pb.z;
      ps.indirect[0] = pb.w; ps.indirect[1] = pc2.x; ps.indirect[2] = pc2.y;
      int fl;
      float fx, fy;
      film_of_path(P, path, pixels, L, fl, fx, fy);
      unsigned sampleIndex =
          VIEWS ? sample_index_fc(pc, P.frameCounts[fl], sample) : sample_index_of(L, pc, frame0 + fl, sample);
      bool done = shade_step(sc, pc, ps, r, h, fx, fy, sampleIndex, tStart, ignore, anyHit, lightHit ? 1 : 0);
      if (done) {
        float col[3], fc[3] = {0.0f, 0.0f, 0.0f};
        sample_colour(pc, ps, col);
        if (sample > 0) {  // blend_sample copies the first sample of a frame
          float4 prev = B.frameCol[path];
          fc[0] = prev.x; fc[1] = prev.y; fc[2] = prev.z;
        }
        blend_sample(pc, sample, col, fc);
        B.frameCol[path] = make_float4(fc[0], fc[1], fc[2], 0.0f);
      } else {
        emit = true;
        // a surface hit is the new shading point of a shadow ray; otherwise the next ray is an extension ray
        pl = wf_payload(ps, surfaceHit ? __int_as_float(sc.prims[h.prim].materialIndex) : ps.dLight);
        path = wf_pack_path(path, ps.stage, ps.depth);
      }
    }
    queue_append<OUT>(B, 1 - q, emit, r, tStart, ignore, anyHit, path, pl, lane);
  }
}

// between rounds: the consumed queue becomes the next output queue
__global__ void k_wf_swap(LtWfBuffers B, int q) {
  B.counts[2 * q] = 0;
  B.counts[2 * q + 1] = 0;
  B.counts[4] = 0;
}

// frames of the batch, in order, through the frame combiner (accumulator.frag:10-19)
// LIST: a masked launch, thread i folds the frames of list index i into pixel M.list[i]; M2: and its Welford sums
template <bool LIST, bool M2>
__global__ void __launch_bounds__(WF_BLOCK) k_wf_accumulate(LtLaunch L, LtWfBuffers B, float* __restrict__ out,
                                                            int pixels, int frame0, int batchFrames,
                                                            const unsigned char* __restrict__ cls, LtList M) {
  const PathConsts pc = path_consts(L);
  int pixel = blockIdx.x * blockDim.x + threadIdx.x;
  if (pixel >= pixels) return;
  const long long image = LIST ? M.list[pixel] : pixel;
  long long id = image * L.depth;
  FrameSink sink;  // a batch that starts at frame0 > 0 continues from what earlier batches wrote to `out`
  if (frame0 == 0) sink.begin(L, out, id);
  else {
    sink.acc[0] = out[id + 0]; sink.acc[1] = out[id + 1]; sink.acc[2] = out[id + 2];
  }
  M2Sink w;
  if (M2) w.begin(frame0 > 0 || L.cam.frameCount > 0, M.m2, image);
  const int pixelClass = cls ? cls[pixel] : 2;  // black / white pixels have no paths: their sample is constant
  for (int f = 0; f < batchFrames; f++) {
    float4 v = make_float4((float)pixelClass, (float)pixelClass, (float)pixelClass, 0.0f);
    if (pixelClass == 2) v = B.frameCol[(long long)f * pixels + pixel];
    float c[3] = {v.x, v.y, v.z};
    finish_frame_colour(pc, L.kernelMode, c);
    sink_frame<M2>(sink, w, L, L.cam.frameCount + (unsigned)(frame0 + f) * L.frameStride, c);
  }
  sink.end(out, id);
  if (M2) w.end(M.m2, image);
}

// The film table of a masked launch whose camera rays k_wf_primary traces itself (counting or culled launches): the
// film position camera_ray computes for list index i, so that the shade kernels read it as in the other launches
__global__ void __launch_bounds__(WF_BLOCK) k_wf_list_film(LtLaunch L, float2* __restrict__ film, LtList M) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M.count) return;
  const int pixel = M.list[i], py = pixel / L.width, px = pixel - py * L.width;
  film[i] = make_float2(FADD(FDIV((float)px, (float)L.width), -0.5f),
                        FADD(FDIV((float)lt_image_row(L, py), (float)L.fullHeight), -0.5f));
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
size_t lt_wf_bytes_per_path() {
  // frame colour, hits; per queue: ray (2 x 16 B), payload (40 B), path word.  The hit words and dLight live inside
  // the hits and payA arrays (wf_hit_words, wf_dlight).
  return sizeof(float4) * 2 + 2 * (sizeof(float4) * 4 + sizeof(float2) + sizeof(int));
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
  B.frameCol = (float4*)take(f4);
  for (int k = 0; k < 2; k++) {
    B.rayO[k] = (float4*)take(f4);
    B.rayD[k] = (float4*)take(f4);
    B.rayPath[k] = (int*)take(sizeof(int) * (size_t)nPaths);
    B.payA[k] = (float4*)take(f4);
    B.payB[k] = (float4*)take(f4);
    B.payC[k] = (float2*)take(sizeof(float2) * (size_t)nPaths);
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

// Views a batch of batchFrames (view, frame) pairs touches at most: a batch that starts at the last frame of a view
// reaches (frames + batchFrames - 2) / frames views beyond it.
int lt_wf_views_per_batch(int batchFrames, int frames, int views) {
  const long long n = ((long long)frames + batchFrames - 2) / frames + 1;
  return n < views ? (int)n : views;
}

// a call of several views keeps, per batch workspace, the primary records of every view its batch touches
size_t lt_wf_view_records_bytes(long long pixels, int viewsPerBatch) {
  return ((lt_wf_primary_hits_bytes(pixels) + 255) & ~(size_t)255) * (size_t)viewsPerBatch;
}

// the kernels whose shared memory grows with the stack depth (lt_opt_in_traversal_smem)
const void* const lt_wf_traversal_kernels[10] = {
    (const void*)k_wf_primary_trace<false>,        (const void*)k_wf_primary_trace<true>,
    (const void*)k_wf_primary<false, false, false>, (const void*)k_wf_primary<true, false, false>,
    (const void*)k_wf_primary<false, true, false>,  (const void*)k_wf_primary<true, true, false>,
    (const void*)k_wf_primary<false, false, true>,  (const void*)k_wf_primary<true, false, true>,
    (const void*)k_wf_trace<false, false>,          (const void*)k_wf_trace<true, false>};

// Round r >= 1 of a sample (WfRound).  The exact pipelines fold the retracing of a light hit into its shading, so round
// 1 holds the first shadow rays of the paths, and after it extension and shadow rounds alternate: an extension result
// emits only shadow rays, a shadow result only extension rays.  Counting launches that retrace light hits append
// extension rays to shadow rounds.
static int wf_round_kind(int flags, int r) {
  if (!lt_fold_light_hits(flags)) return WF_GENERIC;
  return r == 1 ? WF_FIRST_SHADOW : (r & 1) ? WF_SHADOW : WF_EXTENSION;
}

template <int Q, bool V>
static void launch_shade(int kind, int grid, cudaStream_t st, const LtSceneDev& sc, const LtLaunch& L,
                         const LtWfBuffers& B, int pixels, int sample, const LtWfPrimary& P) {
  switch (kind) {
    case WF_FIRST_SHADOW: k_wf_shade<Q, WF_FIRST_SHADOW, V><<<grid, WF_BLOCK, 0, st>>>(sc, L, B, pixels, 0, sample, P); break;
    case WF_SHADOW: k_wf_shade<Q, WF_SHADOW, V><<<grid, WF_BLOCK, 0, st>>>(sc, L, B, pixels, 0, sample, P); break;
    case WF_EXTENSION: k_wf_shade<Q, WF_EXTENSION, V><<<grid, WF_BLOCK, 0, st>>>(sc, L, B, pixels, 0, sample, P); break;
    default: k_wf_shade<Q, WF_GENERIC, V><<<grid, WF_BLOCK, 0, st>>>(sc, L, B, pixels, 0, sample, P); break;
  }
}

// The views of a batch: one segment per view it touches, (view, frames first .. first + count - 1 of that view) at pair
// offset `at` of the batch.  Pairs are view-major, so the segments of a batch are consecutive views.
struct WfSegment {
  int view, first, count, at;
};
static int batch_segments(long long pair0, int nf, int frames, WfSegment* seg) {
  int n = 0;
  for (int at = 0; at < nf;) {
    const long long pair = pair0 + at;
    WfSegment s;
    s.view = (int)(pair / frames);
    s.first = (int)(pair - (long long)s.view * frames);
    s.count = frames - s.first < nf - at ? frames - s.first : nf - at;
    s.at = at;
    seg[n++] = s;
    at += s.count;
  }
  return n;
}

int lt_launch_render_wavefront(const LtSceneDev& sc, const LtPlan& plan, const LtLaunch& L, float* dOut,
                               LtCounters* dCounters, void* workspace, int smCount, cudaStream_t stream,
                               cudaEvent_t* traceEvents, int maxTraceLaunches, int* traceLaunches,
                               unsigned char* pairKinds, const LtWfAux* aux, const LtViews* views,
                               const LtList* list) {
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
  lt_opt_in_traversal_smem(plan.smemStack);
  // a masked launch (list): the pixel axis is the list index, `pixels` the listed pixels (views are not masked)
  const int pixels = list ? list->count : L.width * L.height;
  const LtList M = list ? *list : LtList{};
  const bool stats = plan.stats, threaded = plan.tree != LT_TREE_CHILD_PAIR, overlap = plan.streams == 2;
  const int batchFrames = plan.batchFrames;
  const size_t smem = plan.smemStack;
  const size_t wsBytes = lt_wf_workspace_bytes_padded((long long)batchFrames * pixels);
  // A call of several views: the batches run over (view, frame) pairs, view-major, so every view's frames still reach
  // its image in frame order.  Each batch traces the camera rays of the views it touches into its own record slots
  // (one per view, behind the batch workspaces); a view whose frames two batches share is traced by both, to the same
  // records.
  const int V = views ? views->count : 1;
  const long long totalPairs = (long long)L.frames * V;
  const int viewsPerBatch = views ? lt_wf_views_per_batch(batchFrames, L.frames, V) : 1;
  const size_t slotBytes = (lt_wf_primary_hits_bytes(pixels) + 255) & ~(size_t)255;
  const size_t imageFloats = (size_t)pixels * L.depth;
  int preLaunches = 0;
  int l = 0;
  while ((1ll << l) < pixels) l++;
  // the primary records of slot k of side `side` (one launch: slot 0 of side 0)
  auto records = [&](int side, int k) {
    LtWfPrimary P = {};
    char* pb = (char*)workspace + (size_t)plan.streams * wsBytes + ((size_t)side * viewsPerBatch + k) * slotBytes;
    auto take = [&](size_t bytes) {
      char* r = pb;
      pb += (bytes + 255) & ~(size_t)255;
      return r;
    };
    P.hits = (float4*)take(sizeof(float4) * (size_t)pixels);
    P.film = (float2*)take(sizeof(float2) * (size_t)pixels);
    P.divS = 25 + l;
    P.divM = (unsigned long long)(((1ull << P.divS) + (unsigned long long)pixels - 1ull) / (unsigned long long)pixels);
    if (plan.classify) {
      P.alive = (int*)take(sizeof(int) * (size_t)pixels);
      P.aliveCount = (int*)take(256);
      P.cls = (unsigned char*)take((size_t)pixels);
    }
    return P;
  };
  auto trace_primary = [&](const LtLaunch& Lv, const LtWfPrimary& P, cudaStream_t st) {
    if (plan.classify) cudaMemsetAsync(P.aliveCount, 0, sizeof(int), st);
    mark(0, st);
    if (list)
      k_wf_primary_trace<true><<<(pixels + WF_BLOCK - 1) / WF_BLOCK, WF_BLOCK, smem, st>>>(sc, Lv, P, pixels,
                                                                                        plan.classify ? 1 : 0, M);
    else
      k_wf_primary_trace<false><<<(pixels + WF_BLOCK - 1) / WF_BLOCK, WF_BLOCK, smem, st>>>(sc, Lv, P, pixels,
                                                                                         plan.classify ? 1 : 0, M);
    mark(1, st);
  };
  // primary hits once per pixel per launch; kept behind the batch workspaces
  LtWfPrimary P = {};
  if (plan.sharedPrimary && !views) {
    P = records(0, 0);
    trace_primary(L, P, stream);
    preLaunches = 1;
  } else if (list) {  // camera rays traced by k_wf_primary: only the film table, for the shade kernels
    P = records(0, 0);
    P.hits = nullptr;
    k_wf_list_film<<<(pixels + WF_BLOCK - 1) / WF_BLOCK, WF_BLOCK, 0, stream>>>(L, P.film, M);
    preLaunches = 1;
  }
  if (overlap) {
    cudaEventRecord(aux->fork, stream);
    cudaStreamWaitEvent(aux->extra, aux->fork, 0);
  }
  std::vector<WfSegment> segs((size_t)viewsPerBatch);
  std::vector<LtWfPrimary> segP((size_t)viewsPerBatch);
  std::vector<LtLaunch> segL((size_t)viewsPerBatch);
  int launches = preLaunches, batch = 0, lastSide = 0;
  for (long long pair0 = 0; pair0 < totalPairs; pair0 += batchFrames, batch++) {
    const int side = overlap ? (batch & 1) : 0;
    cudaStream_t st = side ? aux->extra : stream;
    int nf = totalPairs - pair0 < batchFrames ? (int)(totalPairs - pair0) : batchFrames;
    long long nPaths = (long long)nf * pixels;
    LtWfBuffers B = carve((char*)workspace + (size_t)side * wsBytes, (long long)batchFrames * pixels);
    LtLaunch Lb = L;
    int nSeg = 0;
    if (views) {
      nSeg = batch_segments(pair0, nf, L.frames, segs.data());
      for (int k = 0; k < nSeg; k++) {
        segL[k] = L;
        segL[k].cam = views->cams[segs[k].view];
        segP[k] = plan.sharedPrimary ? records(side, k) : LtWfPrimary{};
        if (plan.sharedPrimary) {
          trace_primary(segL[k], segP[k], st);
          launches++;
        }
      }
      // the shade kernels take the film table of the first slot (it does not depend on the camera) and each pair's
      // frameCount
      P = segP[0];
      P.frameCounts = views->dFrameCounts + pair0;
    } else {
      Lb.cam.frameCount = L.cam.frameCount + (unsigned)pair0 * L.frameStride;  // frame index 0 of the batch
    }
    int grid = (int)((nPaths + WF_BLOCK - 1) / WF_BLOCK);
    if (grid > smCount * 32) grid = smCount * 32;
    for (int s = 0; s < plan.samplesPerFrame; s++) {
      // round 0 (primary rays) fused into one kernel; its survivors are queue 0
      k_wf_reset<<<1, 1, 0, st>>>(B);
      const int out = wf_round_kind(L.flags, 1);
      if (views) {  // one launch per view of the batch, its paths numbered from its pair offset
        for (int k = 0; k < nSeg; k++) {
          LtLaunch Ls = segL[k];
          Ls.cam.frameCount = segL[k].cam.frameCount + (unsigned)segs[k].first * L.frameStride;
          int g = (int)(((long long)segs[k].count * pixels + WF_BLOCK - 1) / WF_BLOCK);
          if (g > smCount * 32) g = smCount * 32;
          mark(0, st, plan.sharedPrimary ? LT_TIMED_PRIMARY_SHADE : LT_TIMED_TRAVERSAL);
          if (stats)
            k_wf_primary<true, true, false><<<g, WF_BLOCK, smem, st>>>(sc, Ls, B, segs[k].count, pixels, s, dCounters,
                                                                       segP[k], out, segs[k].at * pixels, M);
          else
            k_wf_primary<false, true, false><<<g, WF_BLOCK, smem, st>>>(sc, Ls, B, segs[k].count, pixels, s, nullptr,
                                                                        segP[k], out, segs[k].at * pixels, M);
          mark(1, st, plan.sharedPrimary ? LT_TIMED_PRIMARY_SHADE : LT_TIMED_TRAVERSAL);
        }
        launches += 1 + nSeg;
      } else {
        // a traversal kernel only when it traces the camera rays itself
        mark(0, st, plan.sharedPrimary ? LT_TIMED_PRIMARY_SHADE : LT_TIMED_TRAVERSAL);
        if (list) {
          if (stats) k_wf_primary<true, false, true><<<grid, WF_BLOCK, smem, st>>>(sc, Lb, B, nf, pixels, s, dCounters, P, out, 0, M);
          else k_wf_primary<false, false, true><<<grid, WF_BLOCK, smem, st>>>(sc, Lb, B, nf, pixels, s, nullptr, P, out, 0, M);
        } else {
          if (stats) k_wf_primary<true, false, false><<<grid, WF_BLOCK, smem, st>>>(sc, Lb, B, nf, pixels, s, dCounters, P, out, 0, M);
          else k_wf_primary<false, false, false><<<grid, WF_BLOCK, smem, st>>>(sc, Lb, B, nf, pixels, s, nullptr, P, out, 0, M);
        }
        mark(1, st, plan.sharedPrimary ? LT_TIMED_PRIMARY_SHADE : LT_TIMED_TRAVERSAL);
        launches += 2;
      }
      int q = 0;
      for (int r = 1; r < plan.rounds; r++) {
        const int kind = wf_round_kind(L.flags, r);
        int* hitWords = (kind == WF_FIRST_SHADOW || kind == WF_SHADOW) ? (int*)B.hits : nullptr;  // wf_hit_words
        mark(0, st);
        if (stats) k_wf_trace<true, false><<<plan.grid, WF_BLOCK, smem, st>>>(sc, Lb, B, q, dCounters, B.rayO[q], B.rayD[q], hitWords);
        else if (threaded) k_wf_trace<false, true><<<plan.grid, WF_BLOCK, plan.smemTrace, st>>>(sc, Lb, B, q, nullptr, B.rayO[q], B.rayD[q], hitWords);
        else k_wf_trace<false, false><<<plan.grid, WF_BLOCK, smem, st>>>(sc, Lb, B, q, nullptr, B.rayO[q], B.rayD[q], hitWords);
        mark(1, st);
        mark(0, st, LT_TIMED_SHADE);
        if (views) {
          if (q == 0) launch_shade<0, true>(kind, grid, st, sc, Lb, B, pixels, s, P);
          else launch_shade<1, true>(kind, grid, st, sc, Lb, B, pixels, s, P);
        } else {
          if (q == 0) launch_shade<0, false>(kind, grid, st, sc, Lb, B, pixels, s, P);
          else launch_shade<1, false>(kind, grid, st, sc, Lb, B, pixels, s, P);
        }
        mark(1, st, LT_TIMED_SHADE);
        k_wf_swap<<<1, 1, 0, st>>>(B, q);
        launches += 3;
        q = 1 - q;
      }
    }
    // the frame combiner is applied in frame order: this batch's accumulate follows the previous batch's
    if (overlap && batch > 0) cudaStreamWaitEvent(st, aux->order[1 - side], 0);
    mark(0, st, LT_TIMED_ACCUMULATE);
    if (views) {  // each view's frames of the batch into its own image
      for (int k = 0; k < nSeg; k++) {
        LtWfBuffers Bs = B;
        Bs.frameCol = B.frameCol + (size_t)segs[k].at * pixels;
        k_wf_accumulate<false, false><<<(pixels + WF_BLOCK - 1) / WF_BLOCK, WF_BLOCK, 0, st>>>(
            segL[k], Bs, dOut + (size_t)segs[k].view * imageFloats, pixels, segs[k].first, segs[k].count, segP[k].cls, M);
      }
      launches += nSeg;
    } else {
      const int g = (pixels + WF_BLOCK - 1) / WF_BLOCK;
      if (!list) k_wf_accumulate<false, false><<<g, WF_BLOCK, 0, st>>>(L, B, dOut, pixels, (int)pair0, nf, P.cls, M);
      else if (!M.m2) k_wf_accumulate<true, false><<<g, WF_BLOCK, 0, st>>>(L, B, dOut, pixels, (int)pair0, nf, P.cls, M);
      else k_wf_accumulate<true, true><<<g, WF_BLOCK, 0, st>>>(L, B, dOut, pixels, (int)pair0, nf, P.cls, M);
      launches++;
    }
    mark(1, st, LT_TIMED_ACCUMULATE);
    if (overlap) cudaEventRecord(aux->order[side], st);
    lastSide = side;
  }
  // join: the last accumulate follows every earlier one (chain of order events), and every stream's last kernel is
  // its accumulate, so waiting for the last batch's event puts all of it before what follows on `stream`
  if (overlap && lastSide != 0) cudaStreamWaitEvent(stream, aux->order[lastSide], 0);
  if (traceLaunches) *traceLaunches = pairs;
  return launches;
}
