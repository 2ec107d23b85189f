// lt_device.cuh -- device-side building blocks shared by the megakernels (lt_kernels.cu) and the
// wavefront pipeline (lt_wavefront.cu): exact-arithmetic helpers, the resumable traversal, camera ray,
// frame combiner, hash RNG, light / hemisphere sampling and the per-ray shading step.
#pragma once
#include "lt_device_types.h"

#ifndef __CUDACC_RTC__
#include <float.h>
#include <math.h>
#else  // NVRTC (plug-in kernels): no host headers
#ifndef FLT_MAX
#define FLT_MAX 3.402823466e+38F
#endif
#endif

#define LT_BLOCK 128
// Per-thread stacks and leaf FIFOs live in shared memory as [level][thread]: LT_THREAD_STRIDE ints between the levels
// of one thread.  The library's kernels run blocks of LT_BLOCK threads; a plug-in build (any block shape) defines
// the stride as its run-time block size before including this file.
#ifndef LT_THREAD_STRIDE
#define LT_THREAD_STRIDE LT_BLOCK
#endif
#define LT_LEVEL_BYTES ((unsigned)(LT_THREAD_STRIDE) * 4u)

// ------------------------------------------------------------------------------------------------
// exact-arithmetic helpers: never contracted, independent of -fmad
// ------------------------------------------------------------------------------------------------
#define FADD(a, b) __fadd_rn((a), (b))
#define FSUB(a, b) __fsub_rn((a), (b))
#define FMUL(a, b) __fmul_rn((a), (b))
#define FFMA(a, b, c) __fmaf_rn((a), (b), (c))
#define FRCP(a) __frcp_rn((a))
#define FDIV(a, b) __fdiv_rn((a), (b))
#define FSQRT(a) __fsqrt_rn((a))

struct Ray {
  float ox, oy, oz;
  float dx, dy, dz;
};

struct Hit {
  float t, u, v;
  int prim;  // primitiveIndex (0 when nothing was hit, as in the reference payload)
  int hit;   // hitType
};

// dot as basic.cu:71 compiles: fma(z,z', fma(x,x', y*y')) + 0.0f
__device__ __forceinline__ float dot3z(float ax, float ay, float az, float bx, float by, float bz) {
  return FADD(FFMA(az, bz, FFMA(ax, bx, FMUL(ay, by))), 0.0f);
}

// intersectBounds, basic.cu:136-154: lo/hi are the dirIsNeg-selected bounds per axis.
__device__ __forceinline__ bool slab(float lox, float hix, float loy, float hiy, float loz, float hiz,
                                     const Ray& r, float ix, float iy, float iz) {
  float tx0 = FMUL(FSUB(lox, r.ox), ix);
  float tx1 = FMUL(FSUB(hix, r.ox), ix);
  float ty0 = FMUL(FSUB(loy, r.oy), iy);
  float ty1 = FMUL(FSUB(hiy, r.oy), iy);
  float tz0 = FMUL(FSUB(loz, r.oz), iz);
  float tz1 = FMUL(FSUB(hiz, r.oz), iz);
  bool miss1 = (tx0 > ty1) || (ty0 > tx1);
  float a = (ty0 > tx0) ? ty0 : tx0;
  float b = (ty1 < tx1) ? ty1 : tx1;
  bool miss2 = (a > tz1) || (tz0 > b);
  float b2 = (tz1 < b) ? tz1 : b;
  return !miss1 && !miss2 && (b2 > 0.0f);
}

// intersectTriangle, basic.cu:93-134, on the pre-subtracted record.  Returns true when the hit
// record was replaced (strict t < best, no t > 0 test -- both as in the reference).
__device__ __forceinline__ bool tri_test(const LtTri* __restrict__ tris, int prim, const Ray& r, float epsThr,
                                         Hit& h) {
  const float4* tp = reinterpret_cast<const float4*>(tris + prim);
  float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
  float ax = q0.x, ay = q0.y, az = q0.z;
  float e1x = q0.w, e1y = q1.x, e1z = q1.y;
  float e2x = q1.z, e2y = q1.w, e2z = q2.x;
  float pvx = FFMA(r.dy, e2z, -FMUL(r.dz, e2y));
  float pvy = FFMA(r.dz, e2x, -FMUL(r.dx, e2z));
  float pvz = FFMA(r.dx, e2y, -FMUL(r.dy, e2x));
  float det = dot3z(e1x, e1y, e1z, pvx, pvy, pvz);
  if (fabsf(det) < epsThr) return false;
  float inv = FRCP(det);
  float tx = FSUB(r.ox, ax), ty = FSUB(r.oy, ay), tz = FSUB(r.oz, az);
  float u = FMUL(dot3z(tx, ty, tz, pvx, pvy, pvz), inv);
  if (u < 0.0f || u > 1.0f) return false;
  float qx = FFMA(ty, e1z, -FMUL(tz, e1y));
  float qy = FFMA(tz, e1x, -FMUL(tx, e1z));
  float qz = FFMA(tx, e1y, -FMUL(ty, e1x));
  float v = FMUL(dot3z(r.dx, r.dy, r.dz, qx, qy, qz), inv);
  if (v < 0.0f || FADD(u, v) > 1.0f) return false;
  float t = FMUL(dot3z(e2x, e2y, e2z, qx, qy, qz), inv);
  if (t < h.t) {
    h.t = t;
    h.u = u;
    h.v = v;
    return true;
  }
  return false;
}

// The same test for rays whose origin and direction reciprocals are all finite (every ray but the
// axis-parallel ones).  Without NaNs the select chain above is an interval test:
// hit <=> max(lo) <= min(hi) && min(hi) > 0, and (bound-o)*inv is monotonic in the bound, so the
// dirIsNeg-selected lo/hi are min/max of the two products.  Same FSUB/FMUL, so same decisions.
__device__ __forceinline__ bool slab_fast(float mnx, float mxx, float mny, float mxy, float mnz, float mxz,
                                          const Ray& r, float ix, float iy, float iz) {
  float ax = FMUL(FSUB(mnx, r.ox), ix), bx = FMUL(FSUB(mxx, r.ox), ix);
  float ay = FMUL(FSUB(mny, r.oy), iy), by = FMUL(FSUB(mxy, r.oy), iy);
  float az = FMUL(FSUB(mnz, r.oz), iz), bz = FMUL(FSUB(mxz, r.oz), iz);
  float lo = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fminf(az, bz));
  float hi = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fmaxf(az, bz));
  return lo <= hi && hi > 0.0f;
}

// intersect / intersectIgnorePrimitiveIndex (basic.cu:156-243) on the child-pair layout, as a
// resumable state machine.  Visits children near-first by the sign of the ray direction on the
// split axis and defers the far child, so triangles are tested in exactly the reference's order; a
// child whose box is missed is never pushed.  anyHit = stop at the first accepted triangle: exact
// for shadow rays because the callers read only hitType (basic_lighting.cl:272,
// global_illumination.cl:296,352).
#define LT_EXACT_SLAB 8u  // negMask bit: ray has a non-finite reciprocal/origin -> select-chain slab test

struct Trav {
  Ray r;
  float ix, iy, iz;
  unsigned negMask;  // bit k: direction reciprocal on axis k is negative; LT_EXACT_SLAB
  int cur;           // >= 0 wide node, < 0 leaf (~primitive), LT_DONE finished
  int sp;
  int ignore;        // intersectIgnorePrimitiveIndex's primitive, < 0 = none
  bool anyHit;
  int qHead, qTail;  // FIFO of reached-but-untested leaves (trav_iter_lean / trav_iter_threaded), shared-memory list
  Hit h;
};

__device__ __forceinline__ bool finite3(float a, float b, float c) {
  return fabsf(a) <= FLT_MAX && fabsf(b) <= FLT_MAX && fabsf(c) <= FLT_MAX;
}

__device__ __forceinline__ bool box_test(const Trav& t, float mnx, float mxx, float mny, float mxy, float mnz,
                                         float mxz) {
  if (t.negMask & LT_EXACT_SLAB) {
    bool nx = t.negMask & 1u, ny = t.negMask & 2u, nz = t.negMask & 4u;
    return slab(nx ? mxx : mnx, nx ? mnx : mxx, ny ? mxy : mny, ny ? mny : mxy, nz ? mxz : mnz, nz ? mnz : mxz, t.r,
                t.ix, t.iy, t.iz);
  }
  return slab_fast(mnx, mxx, mny, mxy, mnz, mxz, t.r, t.ix, t.iy, t.iz);
}

template <bool STATS>
__device__ __forceinline__ void trav_begin(Trav& t, const LtSceneDev& sc, int ignore, float tInit, bool anyHit,
                                           LtCounters& cnt) {
  t.ix = FRCP(t.r.dx);
  t.iy = FRCP(t.r.dy);
  t.iz = FRCP(t.r.dz);
  t.negMask = (t.ix < 0.0f ? 1u : 0u) | (t.iy < 0.0f ? 2u : 0u) | (t.iz < 0.0f ? 4u : 0u);
  if (!(finite3(t.ix, t.iy, t.iz) && finite3(t.r.ox, t.r.oy, t.r.oz))) t.negMask |= LT_EXACT_SLAB;
  t.h.t = tInit; t.h.u = 0.0f; t.h.v = 0.0f; t.h.prim = 0; t.h.hit = 0;
  t.ignore = ignore;
  t.anyHit = STATS ? false : anyHit;
  t.sp = 0;
  t.qHead = t.qTail = 0;
  if (STATS) {
    cnt.rays++;
    cnt.nodeTests++;
  }
  // root box (reference node 0)
  bool hit = box_test(t, sc.rootMin[0], sc.rootMax[0], sc.rootMin[1], sc.rootMax[1], sc.rootMin[2], sc.rootMax[2]);
  t.cur = hit ? sc.rootRef : LT_DONE;
  if (STATS && hit && t.cur < 0 && sc.rootCount > 1 && ~t.cur != ignore) cnt.triTests += (unsigned)(sc.rootCount - 1);
}

__device__ __forceinline__ int trav_pop(Trav& t, const int* __restrict__ stk) {
  // branch-free: an empty stack yields LT_DONE (slot 0 is read but not used)
  bool can = t.sp > 0;
  t.sp -= can ? 1 : 0;
  int v = stk[t.sp * LT_THREAD_STRIDE];
  return can ? v : LT_DONE;
}

// ---- shared-memory access through 32-bit shared addresses, 256-bit node loads ----
__device__ __forceinline__ void sts32(unsigned addr, int v) {
  asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ int lds32(unsigned addr) {
  int v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}

// One 256-bit read-only load (LDG.E.ENL2.256.CONSTANT, sm_100): a 32-byte record costs one L1 request -- and, for
// the divergent addresses of a traversal, one wavefront per distinct 128-byte line -- instead of two.
// 256-bit loads need CUDA 12.9 or newer.  Plug-ins are compiled by whichever NVRTC the process has loaded (a PyTorch
// built for CUDA 12.8 brings its own); with an older compiler the record is read as two 128-bit loads, same values.
__device__ __forceinline__ void ldg256(const void* p, float4& a, float4& b) {
#if __CUDACC_VER_MAJOR__ > 12 || (__CUDACC_VER_MAJOR__ == 12 && __CUDACC_VER_MINOR__ >= 9)
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
               : "l"(p));
#else
  asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "l"(p));
  asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4+16];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(p));
#endif
}

// one inner-node step; requires t.cur >= 0
template <bool STATS>
__device__ __forceinline__ void trav_node_step(Trav& t, const LtSceneDev& sc, int* __restrict__ stk, LtCounters& cnt) {
  const float4* np = reinterpret_cast<const float4*>(sc.wnodes + t.cur);
  float4 bx, by, bz, mf;
  ldg256(np, bx, by);
  ldg256(np + 2, bz, mf);
  int4 m = make_int4(__float_as_int(mf.x), __float_as_int(mf.y), __float_as_int(mf.z), __float_as_int(mf.w));
  bool hl, hr;
  // The select-chain test is valid for every ray, the interval test only for rays without
  // non-finite reciprocals; both give the same answer where both apply.  If any lane that is at this
  // instruction needs the select chain, all of them take it: one instruction stream per warp.
  if (__any_sync(__activemask(), (t.negMask & LT_EXACT_SLAB) != 0u)) {
    bool nx = t.negMask & 1u, ny = t.negMask & 2u, nz = t.negMask & 4u;
    hl = slab(nx ? bx.y : bx.x, nx ? bx.x : bx.y, ny ? by.y : by.x, ny ? by.x : by.y, nz ? bz.y : bz.x,
              nz ? bz.x : bz.y, t.r, t.ix, t.iy, t.iz);
    hr = slab(nx ? bx.w : bx.z, nx ? bx.z : bx.w, ny ? by.w : by.z, ny ? by.z : by.w, nz ? bz.w : bz.z,
              nz ? bz.z : bz.w, t.r, t.ix, t.iy, t.iz);
  } else {
    hl = slab_fast(bx.x, bx.y, by.x, by.y, bz.x, bz.y, t.r, t.ix, t.iy, t.iz);
    hr = slab_fast(bx.z, bx.w, by.z, by.w, bz.z, bz.w, t.r, t.ix, t.iy, t.iz);
  }
  if (STATS) {
    cnt.nodeTests += 2;
    // a leaf with primitiveCount n is tested n times by the reference (always the same triangle)
    unsigned lc = (unsigned)m.w & 0xffffu, rc = (unsigned)m.w >> 16;
    if (hl && m.x < 0 && lc > 1 && ~m.x != t.ignore) cnt.triTests += lc - 1;
    if (hr && m.y < 0 && rc > 1 && ~m.y != t.ignore) cnt.triTests += rc - 1;
  }
  // near child first by the sign of the direction on the split axis (basic.cu:180-186); written
  // with selects so the lanes of a warp do not split on the four hit/miss combinations
  bool axisNeg = (t.negMask >> m.z) & 1u;
  int nearRef = axisNeg ? m.y : m.x, farRef = axisNeg ? m.x : m.y;
  bool hn = axisNeg ? hr : hl, hf = axisNeg ? hl : hr;
  bool both = hn && hf, none = !hn && !hf;
  bool canPop = none && t.sp > 0;
  t.sp -= canPop ? 1 : 0;
  int slot = t.sp * LT_THREAD_STRIDE;
  int popped = stk[slot];
  if (both) stk[slot] = farRef;
  t.sp += both ? 1 : 0;
  t.cur = hn ? nearRef : (hf ? farRef : (canPop ? popped : LT_DONE));
}

// Traversal never depends on triangle results (the reference does not cull by t, basic.cu:136-154),
// so box tests and triangle tests are decoupled: the node phase walks the tree and only RECORDS the
// leaves it reaches, in order, in a small per-thread list in shared memory; the leaf phase then
// tests the recorded triangles in that order.  A warp therefore switches between "all lanes test
// boxes" and "all lanes test triangles" once per batch instead of at every leaf.
#define LT_MAX_BATCH 16  // list entries per thread (shared memory: [LT_MAX_BATCH][LT_BLOCK] ints)

// node phase: advance until the ray is exhausted (t.cur == LT_DONE) or `batch` leaves are recorded.
// Returns the number of recorded leaves.
template <bool STATS>
__device__ __forceinline__ int trav_collect(Trav& t, const LtSceneDev& sc, int* __restrict__ stk,
                                            int* __restrict__ list, int batch, LtCounters& cnt) {
  int n = 0;
  while (t.cur != LT_DONE && n < batch) {
    if (t.cur >= 0) {
      trav_node_step<STATS>(t, sc, stk, cnt);
    } else {
      int prim = ~t.cur;
      if (prim != t.ignore) {
        list[n * LT_THREAD_STRIDE] = prim;
        n++;
      }
      t.cur = trav_pop(t, stk);
    }
  }
  return n;
}

// leaf phase: test the recorded triangles in order.  Returns true if the ray is finished early
// (any-hit ray that found a hit).
template <bool STATS>
__device__ __forceinline__ bool trav_test(Trav& t, const LtSceneDev& sc, const int* __restrict__ list, int n,
                                          float epsThr, LtCounters& cnt) {
  for (int i = 0; i < n; i++) {
    int prim = list[i * LT_THREAD_STRIDE];
    if (STATS) cnt.triTests++;
    if (tri_test(sc.tris, prim, t.r, epsThr, t.h)) {
      t.h.prim = prim;
      t.h.hit = 1;
      if (t.anyHit) {
        t.cur = LT_DONE;
        return true;
      }
    }
  }
  return false;
}

// ---- software-pipelined traversal for the persistent loops (k_flat_stream, k_wf_trace) ----------
// Because traversal never waits for triangle results, one iteration advances the tree walk by up to
// `nodeSteps` box-pair tests (recording reached leaves in a FIFO, in order) AND tests up to `triTests`
// recorded triangles (oldest first).  Within a warp both halves of the iteration are populated by most
// lanes, whatever the phase of their rays.  Returns true when the ray is finished (tree exhausted and
// FIFO empty, or any-hit ray found a hit).  Written for instruction count: shared memory is addressed
// through 32-bit shared addresses (no generic-pointer conversion per access), the two children of a node
// are classified once and a hit leaf child is recorded in the FIFO inside the node step itself (no
// pop/drain round trip); only a leaf that had to wait on the stack behind an inner sibling is recorded
// after being popped.
constexpr int kLeanNodeSteps = 8;  // box-pair tests per iteration
constexpr int kLeanTriTests = 3;   // triangle tests per iteration
template <bool STATS>
__device__ __forceinline__ bool trav_iter_lean(Trav& t, const LtSceneDev& sc, unsigned stkAddr, unsigned fifoAddr,
                                               float epsThr, int nodeSteps, int triTests, LtCounters& cnt) {
  // one step records up to three leaves (near child, far child, and a leaf popped behind them)
  for (int steps = 0; steps < nodeSteps && t.cur != LT_DONE && t.qTail - t.qHead <= LT_MAX_BATCH - 3; steps++) {
    if (t.cur >= 0) {
      const float4* np = reinterpret_cast<const float4*>(sc.wnodes + t.cur);
      float4 bx, by, bz, mf;
      ldg256(np, bx, by);
      ldg256(np + 2, bz, mf);
      int4 m = make_int4(__float_as_int(mf.x), __float_as_int(mf.y), __float_as_int(mf.z), __float_as_int(mf.w));
      unsigned hits;  // bit 0: left child box hit, bit 1: right child box hit
      if (__any_sync(__activemask(), (t.negMask & LT_EXACT_SLAB) != 0u)) {
        bool nx = t.negMask & 1u, ny = t.negMask & 2u, nz = t.negMask & 4u;
        bool hl = slab(nx ? bx.y : bx.x, nx ? bx.x : bx.y, ny ? by.y : by.x, ny ? by.x : by.y, nz ? bz.y : bz.x,
                       nz ? bz.x : bz.y, t.r, t.ix, t.iy, t.iz);
        bool hr = slab(nx ? bx.w : bx.z, nx ? bx.z : bx.w, ny ? by.w : by.z, ny ? by.z : by.w, nz ? bz.w : bz.z,
                       nz ? bz.z : bz.w, t.r, t.ix, t.iy, t.iz);
        hits = (hl ? 1u : 0u) | (hr ? 2u : 0u);
      } else {
        bool hl = slab_fast(bx.x, bx.y, by.x, by.y, bz.x, bz.y, t.r, t.ix, t.iy, t.iz);
        bool hr = slab_fast(bx.z, bx.w, by.z, by.w, bz.z, bz.w, t.r, t.ix, t.iy, t.iz);
        hits = (hl ? 1u : 0u) | (hr ? 2u : 0u);
      }
      if (STATS) {
        cnt.nodeTests += 2;
        unsigned lc = (unsigned)m.w & 0xffffu, rc = (unsigned)m.w >> 16;
        if ((hits & 1u) && m.x < 0 && lc > 1 && ~m.x != t.ignore) cnt.triTests += lc - 1;
        if ((hits & 2u) && m.y < 0 && rc > 1 && ~m.y != t.ignore) cnt.triTests += rc - 1;
      }
      // near child first by the sign of the direction on the split axis (basic.cu:180-186)
      bool axisNeg = (t.negMask >> m.z) & 1u;
      int nearRef = axisNeg ? m.y : m.x, farRef = axisNeg ? m.x : m.y;
      bool hn = (hits & (axisNeg ? 2u : 1u)) != 0u, hf = (hits & (axisNeg ? 1u : 2u)) != 0u;
      bool nearInner = hn && nearRef >= 0;       // descend into near; far (if hit) must wait on the stack
      bool recNear = hn && nearRef < 0 && ~nearRef != t.ignore;
      bool farNow = hf && !nearInner;            // far is next in order right away
      bool recFar = farNow && farRef < 0 && ~farRef != t.ignore;
      if (recNear) {
        sts32(fifoAddr + ((unsigned)(t.qTail & (LT_MAX_BATCH - 1)) * LT_LEVEL_BYTES), ~nearRef);
        t.qTail++;
      }
      if (recFar) {
        sts32(fifoAddr + ((unsigned)(t.qTail & (LT_MAX_BATCH - 1)) * LT_LEVEL_BYTES), ~farRef);
        t.qTail++;
      }
      bool push = hf && nearInner;
      bool farInner = farNow && farRef >= 0;
      bool pop = !nearInner && !farInner;
      bool canPop = pop && t.sp > 0;
      t.sp -= canPop ? 1 : 0;
      unsigned slot = stkAddr + ((unsigned)t.sp * LT_LEVEL_BYTES);
      int popped = lds32(slot);
      if (push) sts32(slot, farRef);
      t.sp += push ? 1 : 0;
      t.cur = nearInner ? nearRef : (farInner ? farRef : (canPop ? popped : LT_DONE));
    }
    // a leaf that waited on the stack (or the root itself): record it and take the next entry
    if (t.cur < 0 && t.cur != LT_DONE) {
      int prim = ~t.cur;
      if (prim != t.ignore) {
        sts32(fifoAddr + ((unsigned)(t.qTail & (LT_MAX_BATCH - 1)) * LT_LEVEL_BYTES), prim);
        t.qTail++;
      }
      bool can = t.sp > 0;
      t.sp -= can ? 1 : 0;
      int v = lds32(stkAddr + ((unsigned)t.sp * LT_LEVEL_BYTES));
      t.cur = can ? v : LT_DONE;
    }
  }
  for (int k = 0; k < triTests && t.qHead != t.qTail; k++) {
    int prim = lds32(fifoAddr + ((unsigned)(t.qHead & (LT_MAX_BATCH - 1)) * LT_LEVEL_BYTES));
    t.qHead++;
    if (STATS) cnt.triTests++;
    if (tri_test(sc.tris, prim, t.r, epsThr, t.h)) {
      t.h.prim = prim;
      t.h.hit = 1;
      if (t.anyHit) {
        t.cur = LT_DONE;
        t.qHead = t.qTail;
      }
    }
  }
  return t.cur == LT_DONE && t.qHead == t.qTail;
}

// ---- stackless traversal of the threaded tree (LtThreadNode, small scenes) -----------------------
// Same triangle tests in the same order as the stack traversal above, hence the same hits, and the same box tests
// (full copies) or a subset of them that cannot change which leaves are reached (pruned copies, see LtThreadNode):
// the records of the ray's sign octant are laid out in visit order, so a step is one box test and
// `cur = hit && inner ? cur + 1 : skip`.  No stack, no near/far selection, no per-axis min/max: the
// record's bounds are already the dirIsNeg-selected ones, so for rays with finite reciprocals
// (lo - o) * inv <= (hi - o) * inv per axis and the select chain of basic.cu:136-154 reduces to
// max3(entries) <= min3(exits) && min3(exits) > 0 on the same FSUB/FMUL products.
__device__ __forceinline__ void trav_begin_threaded(Trav& t, const LtSceneDev& sc, int ignore, float tInit, bool anyHit) {
  t.ix = FRCP(t.r.dx);
  t.iy = FRCP(t.r.dy);
  t.iz = FRCP(t.r.dz);
  t.negMask = (t.ix < 0.0f ? 1u : 0u) | (t.iy < 0.0f ? 2u : 0u) | (t.iz < 0.0f ? 4u : 0u);
  const int oct = (int)(t.negMask & 7u);
  if (!(finite3(t.ix, t.iy, t.iz) && finite3(t.r.ox, t.r.oy, t.r.oz))) t.negMask |= LT_EXACT_SLAB;
  // the pruned copies rely on (b - o) * inv being monotonic in the bound b: not so for a non-finite reciprocal or
  // origin, nor for a zero reciprocal (inf * 0 = NaN when b - o overflows); those rays walk the full copies
  const bool full = (t.negMask & LT_EXACT_SLAB) || t.ix == 0.0f || t.iy == 0.0f || t.iz == 0.0f;
  const int rootRecord = full ? oct * sc.nodeCount : sc.prunedBase + oct * sc.prunedStride;
  // every ray starts at the root: its box comes from the kernel parameters (constant bank) instead of a gather,
  // and an inner root that is hit continues at its near child, the next record of the copy
  t.cur = rootRecord;
  if (sc.rootRef >= 0)
    t.cur = box_test(t, sc.rootMin[0], sc.rootMax[0], sc.rootMin[1], sc.rootMax[1], sc.rootMin[2], sc.rootMax[2])
                ? rootRecord + 1 : LT_DONE;
  t.h.t = tInit; t.h.u = 0.0f; t.h.v = 0.0f; t.h.prim = 0; t.h.hit = 0;
  t.ignore = ignore;
  t.anyHit = anyHit;
  t.sp = 0;
  t.qHead = t.qTail = 0;
}

// node phase, EXACT = select chain (valid for every ray) or interval form (rays with finite reciprocals).
// Each step records at most one leaf, so `maxSteps` <= free FIFO slots needs no per-step capacity check.
template <bool EXACT>
__device__ __forceinline__ void trav_threaded_nodes(Trav& t, const LtThreadNode* __restrict__ tn, unsigned fifoAddr,
                                                    int maxSteps, int notIgnore) {
  for (int steps = 0; steps < maxSteps && t.cur != LT_DONE; steps++) {
    float4 a, b;
    ldg256(tn + t.cur, a, b);
    float tx0 = FMUL(FSUB(a.x, t.r.ox), t.ix), tx1 = FMUL(FSUB(a.w, t.r.ox), t.ix);
    float ty0 = FMUL(FSUB(a.y, t.r.oy), t.iy), ty1 = FMUL(FSUB(b.x, t.r.oy), t.iy);
    float tz0 = FMUL(FSUB(a.z, t.r.oz), t.iz), tz1 = FMUL(FSUB(b.y, t.r.oz), t.iz);
    bool hit;
    if (EXACT) {
      bool miss1 = (tx0 > ty1) || (ty0 > tx1);
      float lo = (ty0 > tx0) ? ty0 : tx0;
      float hi = (ty1 < tx1) ? ty1 : tx1;
      bool miss2 = (lo > tz1) || (tz0 > hi);
      float hi2 = (tz1 < hi) ? tz1 : hi;
      hit = !miss1 && !miss2 && (hi2 > 0.0f);
    } else {
      float lo = fmaxf(fmaxf(tx0, ty0), tz0);
      float hi = fminf(fminf(tx1, ty1), tz1);
      hit = lo <= hi && hi > 0.0f;
    }
    int link = __float_as_int(b.z), skip = __float_as_int(b.w);
    if (hit && link < 0 && link != notIgnore) {
      sts32(fifoAddr + ((unsigned)(t.qTail & (LT_MAX_BATCH - 1)) * LT_LEVEL_BYTES), ~link);
      t.qTail++;
    }
    t.cur = (hit && link >= 0) ? t.cur + 1 : skip;
  }
}

// iteration shape of the persistent loops (k_path, k_wf_trace) on the threaded tree: single-box steps, so twice the
// steps of kLeanNodeSteps
constexpr int kThreadedNodeSteps = 2 * kLeanNodeSteps;
constexpr int kThreadedTriTests = kLeanTriTests;
__device__ __forceinline__ bool trav_iter_threaded(Trav& t, const LtThreadNode* __restrict__ tn,
                                                   const LtTri* __restrict__ tris, unsigned fifoAddr, float epsThr,
                                                   int nodeSteps, int triTests) {
  // rays change only between iterations, so which slab form the warp runs is decided once per iteration
  const bool exact = __any_sync(__activemask(), (t.negMask & LT_EXACT_SLAB) != 0u);
  const int maxSteps = min(nodeSteps, LT_MAX_BATCH - (t.qTail - t.qHead));
  const int notIgnore = ~t.ignore;  // a leaf's link is ~primitivesOffset
  if (exact) trav_threaded_nodes<true>(t, tn, fifoAddr, maxSteps, notIgnore);
  else trav_threaded_nodes<false>(t, tn, fifoAddr, maxSteps, notIgnore);
  for (int k = 0; k < triTests && t.qHead != t.qTail; k++) {
    int prim = lds32(fifoAddr + ((unsigned)(t.qHead & (LT_MAX_BATCH - 1)) * LT_LEVEL_BYTES));
    t.qHead++;
    if (tri_test(tris, prim, t.r, epsThr, t.h)) {
      t.h.prim = prim;
      t.h.hit = 1;
      if (t.anyHit) {
        t.cur = LT_DONE;
        t.qHead = t.qTail;
      }
    }
  }
  return t.cur == LT_DONE && t.qHead == t.qTail;
}

// ------------------------------------------------------------------------------------------------
// OPT-IN culled traversal (LT_FLAG_CULL): same tree, same order, same triangle arithmetic, but a
// subtree is skipped when its box is entered farther along the ray than the current hit (plus a
// margin of 1e-4 relative + 1e-5 absolute, ~100x the rounding error of t).  The reference never
// culls (basic.cu:136-154 ignores the payload), so this does LESS work than the reference; the
// output is identical unless a triangle's computed t undercuts its own box entry by more than the
// margin, which no test scene exhibits (tests/test_gpu_parity.py::test_culling_is_output_identical),
// but which is validated, not proven.  Closest-hit rays only; rays that need the select-chain slab
// (non-finite reciprocals) are never culled.  Triangles are tested as soon as their leaf is reached.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool slab_fast_entry(float mnx, float mxx, float mny, float mxy, float mnz, float mxz,
                                                const Ray& r, float ix, float iy, float iz, float& entry) {
  float ax = FMUL(FSUB(mnx, r.ox), ix), bx = FMUL(FSUB(mxx, r.ox), ix);
  float ay = FMUL(FSUB(mny, r.oy), iy), by = FMUL(FSUB(mxy, r.oy), iy);
  float az = FMUL(FSUB(mnz, r.oz), iz), bz = FMUL(FSUB(mxz, r.oz), iz);
  float lo = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fminf(az, bz));
  float hi = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fmaxf(az, bz));
  entry = lo;
  return lo <= hi && hi > 0.0f;
}

__device__ __forceinline__ float cull_limit(float t) { return t + (fabsf(t) * 1.0e-4f + 1.0e-5f); }

// one step of the culled traversal: a box-pair test with culling, or a triangle test followed by
// popping the next entry that survives the current limit.  tstk holds the entry distance of every
// stacked reference ([level][thread], like stk).
template <bool STATS>
__device__ __forceinline__ void trav_step_cull(Trav& t, const LtSceneDev& sc, int* __restrict__ stk,
                                               float* __restrict__ tstk, float epsThr, LtCounters& cnt) {
  if (t.cur >= 0) {
    const float4* np = reinterpret_cast<const float4*>(sc.wnodes + t.cur);
    float4 bx = __ldg(np), by = __ldg(np + 1), bz = __ldg(np + 2);
    int4 m = __ldg(reinterpret_cast<const int4*>(np) + 3);
    bool hl, hr;
    float el = -FLT_MAX, er = -FLT_MAX;
    if (t.negMask & LT_EXACT_SLAB) {
      bool nx = t.negMask & 1u, ny = t.negMask & 2u, nz = t.negMask & 4u;
      hl = slab(nx ? bx.y : bx.x, nx ? bx.x : bx.y, ny ? by.y : by.x, ny ? by.x : by.y, nz ? bz.y : bz.x,
                nz ? bz.x : bz.y, t.r, t.ix, t.iy, t.iz);
      hr = slab(nx ? bx.w : bx.z, nx ? bx.z : bx.w, ny ? by.w : by.z, ny ? by.z : by.w, nz ? bz.w : bz.z,
                nz ? bz.z : bz.w, t.r, t.ix, t.iy, t.iz);
    } else {
      hl = slab_fast_entry(bx.x, bx.y, by.x, by.y, bz.x, bz.y, t.r, t.ix, t.iy, t.iz, el);
      hr = slab_fast_entry(bx.z, bx.w, by.z, by.w, bz.z, bz.w, t.r, t.ix, t.iy, t.iz, er);
    }
    if (STATS) cnt.nodeTests += 2;
    float lim = cull_limit(t.h.t);
    hl = hl && !(el > lim);
    hr = hr && !(er > lim);
    bool axisNeg = (t.negMask >> m.z) & 1u;
    int nearRef = axisNeg ? m.y : m.x, farRef = axisNeg ? m.x : m.y;
    float farEntry = axisNeg ? el : er;
    bool hn = axisNeg ? hr : hl, hf = axisNeg ? hl : hr;
    if (hn) {
      t.cur = nearRef;
      if (hf) {
        stk[t.sp * LT_THREAD_STRIDE] = farRef;
        tstk[t.sp * LT_THREAD_STRIDE] = farEntry;
        t.sp++;
      }
      return;
    }
    if (hf) {
      t.cur = farRef;
      return;
    }
  } else {
    int prim = ~t.cur;
    if (prim != t.ignore) {
      if (STATS) cnt.triTests++;
      if (tri_test(sc.tris, prim, t.r, epsThr, t.h)) {
        t.h.prim = prim;
        t.h.hit = 1;
      }
    }
  }
  // pop the next stacked reference whose box entry is still within the limit
  float lim = cull_limit(t.h.t);
  t.cur = LT_DONE;
  while (t.sp > 0) {
    t.sp--;
    if (!(tstk[t.sp * LT_THREAD_STRIDE] > lim)) {
      t.cur = stk[t.sp * LT_THREAD_STRIDE];
      break;
    }
  }
}

template <bool STATS>
__device__ __forceinline__ void trace_cull(Trav& t, const LtSceneDev& sc, int ignore, float tInit, float epsThr,
                                           int* __restrict__ stk, float* __restrict__ tstk, LtCounters& cnt) {
  trav_begin<STATS>(t, sc, ignore, tInit, false, cnt);
  while (t.cur != LT_DONE) trav_step_cull<STATS>(t, sc, stk, tstk, epsThr, cnt);
}

// dynamic shared memory of every traversal kernel: [stackDepth][LT_BLOCK] stack, [LT_MAX_BATCH][LT_BLOCK] leaf
// list/FIFO, [stackDepth][LT_BLOCK] entry distances (culled mode only)
__host__ __device__ inline int lt_stack_levels(const LtSceneDev& sc) { return sc.stackDepth < 1 ? 1 : sc.stackDepth; }
#ifndef __CUDACC_RTC__
__host__ inline size_t lt_traversal_smem(const LtSceneDev& sc, bool cull) {
  return (size_t)(lt_stack_levels(sc) * (cull ? 2 : 1) + LT_MAX_BATCH) * LT_BLOCK * sizeof(int);
}
#endif
#define LT_SMEM_POINTERS(sc)                                                            \
  extern __shared__ int smemStack[];                                                    \
  int* stk = smemStack + threadIdx.x;                                                   \
  int* list = smemStack + lt_stack_levels(sc) * LT_BLOCK + threadIdx.x;                 \
  float* tstk = reinterpret_cast<float*>(smemStack + (lt_stack_levels(sc) + LT_MAX_BATCH) * LT_BLOCK) + threadIdx.x;

// run one ray to completion (deterministic kernels, hit-record kernel)
template <bool STATS>
__device__ __forceinline__ void trace(Trav& t, const LtSceneDev& sc, int ignore, float tInit, float epsThr,
                                      bool anyHit, int* __restrict__ stk, int* __restrict__ list, LtCounters& cnt) {
  if (!STATS && sc.tnodes != nullptr) {  // small scene: stackless traversal of the threaded tree, same tests
    trav_begin_threaded(t, sc, ignore, tInit, anyHit);
    const unsigned fifoAddr = (unsigned)__cvta_generic_to_shared(list);
    while (!trav_iter_threaded(t, sc.tnodes, sc.tris, fifoAddr, epsThr, LT_MAX_BATCH, LT_MAX_BATCH)) {
    }
    return;
  }
  trav_begin<STATS>(t, sc, ignore, tInit, anyHit, cnt);
  while (t.cur != LT_DONE) {
    int n = trav_collect<STATS>(t, sc, stk, list, LT_MAX_BATCH, cnt);
    trav_test<STATS>(t, sc, list, n, epsThr, cnt);
  }
}

// ------------------------------------------------------------------------------------------------
// per-kernel constants (see oracle/lt_oracle.c: flavour_for_kernel)
// ------------------------------------------------------------------------------------------------
__host__ __device__ inline float lt_tinit(int kernel) { return kernel == 0 ? 10000000.0f : FLT_MAX; }
__host__ __device__ inline float lt_eps(int kernel) {
  // fabs(det) < eps; the macro-defined epsilons are compared in fp64, i.e. against the next float up
  switch (kernel) {
    case 0: case 1: case 2: return 0x1.ad7f2ap-24f;  // (float)1e-7: basic.cu:95, basic.cl:78
    case 3: return 0x1.ad7f2ap-24f;                   // (float)1e-7 >= 1e-7 (double) already
    default: return 0x1.a36e30p-14f;                  // smallest float >= 1e-4 (double); (float)1e-4 is below
  }
}

// camera ray, basic.cu:350-358; fused forms as NVRTC+ptxas emit them (oracle/notes_fma_order.md)
// image row of local row j of this launch (identity unless the launch is one device's share of a tile split)
__device__ __forceinline__ int lt_image_row(const LtLaunch& L, int j) {
  if (L.rowStride <= 1) return j;
  const int b = j / L.rowBlock;
  return (b * L.rowStride + L.rowPhase) * L.rowBlock + (j - b * L.rowBlock);
}

// c, s = cosf(cam.yaw), sinf(cam.yaw): the same for every pixel, so persistent kernels evaluate them once
__device__ __forceinline__ Ray camera_ray_cs(const RefCamera& cam, float c, float s, int px, int py, int width,
                                             int height, float& fx, float& fy) {
  fx = FADD(FDIV((float)px, (float)width), -0.5f);
  fy = FADD(FDIV((float)py, (float)height), -0.5f);
  float dx0 = FSUB(0.0f, fx);
  Ray r;
  r.ox = FADD(fx, cam.position[0]);
  r.oy = FADD(fy, cam.position[1]);
  r.oz = FADD(cam.position[2], 0.0f);
  r.dx = FFMA(dx0, c, FMUL(s, 5.0f));
  r.dy = FSUB(0.0f, fy);
  r.dz = FFMA(c, 5.0f, -FMUL(dx0, s));
  return r;
}

__device__ __forceinline__ Ray camera_ray(const RefCamera& cam, int px, int py, int width, int height, float& fx,
                                          float& fy) {
  fx = FADD(FDIV((float)px, (float)width), -0.5f);
  fy = FADD(FDIV((float)py, (float)height), -0.5f);
  float c = cosf(cam.yaw), s = sinf(cam.yaw);
  float dx0 = FSUB(0.0f, fx);
  Ray r;
  r.ox = FADD(fx, cam.position[0]);
  r.oy = FADD(fy, cam.position[1]);
  r.oz = FADD(cam.position[2], 0.0f);
  r.dx = FFMA(dx0, c, FMUL(s, 5.0f));
  r.dy = FSUB(0.0f, fy);
  r.dz = FFMA(c, 5.0f, -FMUL(dx0, s));
  return r;
}

__device__ __forceinline__ float bary0(float u, float v) {
  return (float)__dsub_rn(__dsub_rn(1.0, (double)u), (double)v);
}

// thread -> pixel: a warp covers an 8x4 pixel tile, a block 16x8 (coherent primary rays).
__device__ __forceinline__ bool thread_pixel(int width, int height, int& px, int& py) {
  int tilesX = (width + 15) >> 4;
  int tile = blockIdx.x;
  int tyi = tile / tilesX, txi = tile - tyi * tilesX;
  int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  px = (txi << 4) + ((warp & 1) << 3) + (lane & 7);
  py = (tyi << 3) + ((warp >> 1) << 2) + (lane >> 3);
  return px < width && py < height;
}

// running mean / weighted sum / plain store of one finished frame
struct FrameSink {
  float acc[3];
  __device__ __forceinline__ void begin(const LtLaunch& L, const float* out, long long id) {
    acc[0] = acc[1] = acc[2] = 0.0f;
    bool needPrev = (L.accumMode == 2) || (L.accumMode == 1 && L.cam.frameCount > 0);
    if (needPrev) {
      acc[0] = out[id + 0];
      acc[1] = out[id + 1];
      acc[2] = out[id + 2];
    }
  }
  // accumulator.frag:10-19: color = (sample + prev*frameCount) / (frameCount + 1) when frameCount > 0
  __device__ __forceinline__ void frame(const LtLaunch& L, unsigned frameCount, const float c[3]) {
#pragma unroll
    for (int k = 0; k < 3; k++) {
      if (L.accumMode == 1) {
        float v = c[k];
        if (frameCount > 0) v = FDIV(FADD(v, FMUL(acc[k], (float)frameCount)), (float)(frameCount + 1u));
        acc[k] = v;
      } else if (L.accumMode == 2) {
        acc[k] = FADD(acc[k], FMUL(L.accumWeight, c[k]));
      } else {
        acc[k] = c[k];
      }
    }
  }
  __device__ __forceinline__ void end(float* out, long long id) const {
    out[id + 0] = acc[0];
    out[id + 1] = acc[1];
    out[id + 2] = acc[2];
  }
};

__device__ __forceinline__ void flush_counters(LtCounters* g, const LtCounters& c) {
  if (g) {
    atomicAdd(&g->rays, c.rays);
    atomicAdd(&g->nodeTests, c.nodeTests);
    atomicAdd(&g->triTests, c.triTests);
  }
}

// ------------------------------------------------------------------------------------------------
// kernel 1: deterministic pipelines -- basic (flat diffuse + lens refraction) and custom barycentric
// ------------------------------------------------------------------------------------------------
// barycentric interpolation as basic.cu:257-265 compiles: fma(v, C, fma(A, w0, u*B))
__device__ __forceinline__ void lerp_fused(const float* a, const float* b, const float* c, float w0, float u,
                                           float v, float out[3]) {
#pragma unroll
  for (int k = 0; k < 3; k++) out[k] = FFMA(v, c[k], FFMA(a[k], w0, FMUL(u, b[k])));
}

// The two refraction steps of traceRayThroughLens (basic.cu:245-298) on their own, for kernels that run the lens
// rays through a resumable traversal: each turns (ray, hit) into the next ray of the lens path and returns the
// primitive that ray ignores.  lens_refract_in keeps the w of the refracted direction for lens_refract_out.
__device__ __forceinline__ int lens_refract_in(const LtSceneDev& sc, Ray& r, const Hit& h, float& r2w) {
  const RefPrim* prim = sc.prims + h.prim;
  const RefMaterial* mat = sc.mats + prim->materialIndex;
  float w0 = bary0(h.u, h.v);
  float pos[3], nrm[3];
  lerp_fused(prim->a, prim->b, prim->c, w0, h.u, h.v, pos);
  lerp_fused(prim->na, prim->nb, prim->nc, w0, h.u, h.v, nrm);
  float n = FRCP(mat->ior);
  float c = dot3z(r.dx, r.dy, r.dz, nrm[0], nrm[1], nrm[2]);
  float sinT2 = (float)__dmul_rn(__dsub_rn(1.0, (double)FMUL(c, c)), (double)FMUL(n, n));
  float cosT = (float)__dsqrt_rn(__dsub_rn(1.0, (double)sinT2));
  float k = FFMA(c, -n, -cosT);
  float dx = FFMA(r.dx, n, FMUL(nrm[0], k));
  float dy = FFMA(r.dy, n, FMUL(nrm[1], k));
  float dz = FFMA(r.dz, n, FMUL(nrm[2], k));
  r2w = FFMA(n, 0.0f, FMUL(k, 0.0f));
  r.ox = pos[0]; r.oy = pos[1]; r.oz = pos[2];
  r.dx = dx; r.dy = dy; r.dz = dz;
  return h.prim;
}

__device__ __forceinline__ int lens_refract_out(const LtSceneDev& sc, Ray& r, const Hit& h, float r2w) {
  const RefPrim* prim = sc.prims + h.prim;
  const RefMaterial* mat = sc.mats + prim->materialIndex;
  float w0 = bary0(h.u, h.v);
  float pos[3], nrm[3];
  lerp_fused(prim->a, prim->b, prim->c, w0, h.u, h.v, pos);
  lerp_fused(prim->na, prim->nb, prim->nc, w0, h.u, h.v, nrm);
  float ior = mat->ior;
  float c2 = FFMA(0.0f, r2w, FFMA(-r.dz, nrm[2], FFMA(r.dx, -nrm[0], -FMUL(r.dy, nrm[1]))));
  float sinT2b = (float)__dmul_rn(__dsub_rn(1.0, (double)FMUL(c2, c2)), (double)FMUL(ior, ior));
  float cosTb = (float)__dsqrt_rn(__dsub_rn(1.0, (double)sinT2b));
  float k2 = FFMA(c2, -ior, -cosTb);
  float dx = FFMA(r.dx, ior, -FMUL(k2, nrm[0]));
  float dy = FFMA(r.dy, ior, -FMUL(k2, nrm[1]));
  float dz = FFMA(r.dz, ior, -FMUL(k2, nrm[2]));
  r.ox = pos[0]; r.oy = pos[1]; r.oz = pos[2];
  r.dx = dx; r.dy = dy; r.dz = dz;
  return h.prim;
}

// traceRayThroughLens + refract, basic.cu:79-86,245-298 (operation order: oracle/notes_fma_order.md)
// On entry t holds the primary ray and its hit; on exit the refracted ray and its hit.
template <bool STATS>
__device__ void lens_path(const LtSceneDev& sc, Trav& t, float tInit, float epsThr, int* stk, int* list,
                          float* tstk, bool cull, LtCounters& cnt) {
  float r2w;
  {
    const Hit h = t.h;
    const int firstPrim = lens_refract_in(sc, t.r, h, r2w);
    if (cull) trace_cull<STATS>(t, sc, firstPrim, tInit, epsThr, stk, tstk, cnt);
    else trace<STATS>(t, sc, firstPrim, tInit, epsThr, false, stk, list, cnt);
  }
  {
    const Hit h = t.h;
    const int secondPrim = lens_refract_out(sc, t.r, h, r2w);
    if (cull) trace_cull<STATS>(t, sc, secondPrim, tInit, epsThr, stk, tstk, cnt);
    else trace<STATS>(t, sc, secondPrim, tInit, epsThr, false, stk, list, cnt);
  }
}

// ------------------------------------------------------------------------------------------------
// kernel 2: stochastic pipelines -- direct lighting, accumulator, global illumination
// ------------------------------------------------------------------------------------------------
// fmod(x, M_PI) bit-exact: q is within one of the true quotient, fma gives the exact remainder
// (both x and q*pi are multiples of 2^-51 and the result is < 2*pi), then one exact correction.
__device__ __forceinline__ double fmod_pi(double x) {
  const double PI = 3.14159265358979323846;
  double ax = fabs(x);
  double r = ax;
  if (ax >= PI) {
    double q = floor(__dmul_rn(ax, 0.31830988618379067154));
    r = __fma_rn(-q, PI, ax);
    if (r < 0.0) r = __dadd_rn(r, PI);
    else if (r >= PI) r = __dsub_rn(r, PI);
  }
  return copysign(r, x);
}

// random(), basic_lighting.cl:64-67
__device__ __forceinline__ float lt_random(float fx, float fy, float seed) {
  float d = FADD(FMUL(fx, 12.9898f), FMUL(fy, 78.233f));
  double x = __dadd_rn((double)d, __dmul_rn(1113.1, (double)seed));
  float a = (float)__dmul_rn(sin(fmod_pi(x)), 43758.5453);
  return FSUB(a, floorf(a));
}

__device__ __forceinline__ float len3(float x, float y, float z) {
  return FSQRT(FADD(FADD(FMUL(x, x), FMUL(y, y)), FMUL(z, z)));
}
__device__ __forceinline__ float dot3plain(const float a[3], const float b[3]) {
  return FADD(FADD(FMUL(a[0], b[0]), FMUL(a[1], b[1])), FMUL(a[2], b[2]));
}
// basic_lighting.cl:236-244 / global_illumination.cl:235-240 (no contraction)
__device__ __forceinline__ void lerp_plain(const float* a, const float* b, const float* c, float w0, float u,
                                           float v, float out[3]) {
#pragma unroll
  for (int k = 0; k < 3; k++) out[k] = FADD(FADD(FMUL(a[k], w0), FMUL(b[k], u)), FMUL(c[k], v));
}

__device__ __forceinline__ bool is_light(const LtSceneDev& sc, int prim) {
  bool hit = false;
  unsigned n = min(sc.lights->count, 64u);
  for (unsigned x = 0; x < n; x++) hit = hit || ((unsigned)prim == sc.lights->primitives[x]);
  return hit;
}

// light sample: basic_lighting.cl:246-262 with the three random numbers already drawn
// (rIdx = random(seed), rU = random(seed+1), rV = random(seed+2)).  Overwrites r with the shadow
// ray (origin = pos, direction = normalize(L - P)) and returns its initial t.
__device__ __forceinline__ float make_shadow_ray(const LtSceneDev& sc, const float pos[3], float rIdx, float rU,
                                                 float rV, Ray& sr) {
  int idx = (int)FMUL(rIdx, (float)sc.lights->count);
  idx = max(0, min(idx, 63));
  const RefPrim* lp = sc.prims + sc.lights->primitives[idx];
  float ux = rU, uy = rV;
  if (FADD(ux, uy) > 1.0f) {
    ux = FSUB(1.0f, ux);
    uy = FSUB(1.0f, uy);
  }
  float w0 = bary0(ux, uy);
  float Lp[3];
  lerp_plain(lp->a, lp->b, lp->c, w0, ux, uy, Lp);
  float dx = FSUB(Lp[0], pos[0]), dy = FSUB(Lp[1], pos[1]), dz = FSUB(Lp[2], pos[2]);
  float len = len3(dx, dy, dz);
  sr.ox = pos[0]; sr.oy = pos[1]; sr.oz = pos[2];
  sr.dx = FDIV(dx, len);
  sr.dy = FDIV(dy, len);
  sr.dz = FDIV(dz, len);
  return (float)__dsub_rn((double)len, 0.01);
}

// uniformSampleHemisphere + alignHemisphereWithCoordinateSystem, global_illumination.cl:69-82
__device__ __forceinline__ void sample_hemisphere(float u1, float u2, const float up[3], float dir[4]) {
  float z = u1;
  float r = FSQRT(fmaxf(0.0f, FSUB(1.0f, FMUL(z, z))));
  // `float phi = 2.0 * M_PI * uv.y;` (:72): the product is fp64, phi and its cos/sin are FP32
  float phi = (float)__dmul_rn(6.28318530717958647692, (double)u2);
  float hx = FMUL(r, cosf(phi));
  float hy = z;
  float hz = FMUL(r, sinf(phi));
  const float cx = 0.0072f, cy = 1.0f, cz = 0.0034f;
  float rx = FSUB(FMUL(up[1], cz), FMUL(up[2], cy));
  float ry = FSUB(FMUL(up[2], cx), FMUL(up[0], cz));
  float rz = FSUB(FMUL(up[0], cy), FMUL(up[1], cx));
  float rl = len3(rx, ry, rz);
  rx = FDIV(rx, rl); ry = FDIV(ry, rl); rz = FDIV(rz, rl);
  float fwx = FSUB(FMUL(ry, up[2]), FMUL(rz, up[1]));
  float fwy = FSUB(FMUL(rz, up[0]), FMUL(rx, up[2]));
  float fwz = FSUB(FMUL(rx, up[1]), FMUL(ry, up[0]));
  dir[0] = FADD(FADD(FMUL(hx, rx), FMUL(hy, up[0])), FMUL(hz, fwx));
  dir[1] = FADD(FADD(FMUL(hx, ry), FMUL(hy, up[1])), FMUL(hz, fwy));
  dir[2] = FADD(FADD(FMUL(hx, rz), FMUL(hy, up[2])), FMUL(hz, fwz));
  dir[3] = hy;
}

enum PathStage { ST_PRIMARY = 0, ST_SHADOW_DIRECT = 1, ST_EXTENSION = 2, ST_SHADOW_EXT = 3 };

// ------------------------------------------------------------------------------------------------
// one shading step of the stochastic pipelines: consume a finished ray, produce the next one
// ------------------------------------------------------------------------------------------------
struct PathConsts {
  float tInit;
  float epsThr;
  bool isGI;          // global_illumination.cl (both variants)
  bool whiteOnLight;  // accumulator.cl:233-238
  int samplesPerFrame;
  int maxDepth;
  bool foldLightHits;  // see shade_step: a light hit's remaining depths are accumulated without retracing the ray
};

__device__ __forceinline__ PathConsts path_consts(const LtLaunch& L) {
  PathConsts pc;
  pc.tInit = lt_tinit(L.kernel);
  pc.epsThr = lt_eps(L.kernel);
  pc.isGI = (L.kernel == 5 || L.kernel == 6);
  pc.whiteOnLight = (L.kernel == 4);
  pc.samplesPerFrame = (L.kernel == 3 || L.kernel == 5) ? 25 : 1;
  pc.maxDepth = L.maxRayDepth > 0 ? L.maxRayDepth : 16;
  // counting launches (LT_FLAG_STATS = 1) trace what the reference traces, unless LT_FLAG_STATS_TRACED = 128 asks for
  // the counts of what the exact pipelines really trace
  pc.foldLightHits = !(L.flags & 1) || (L.flags & 128);
  return pc;
}

struct PathState {
  float nrm[3], diffuse[3];
  float direct[3], indirect[3];
  float extW;   // w of the extension direction (= hemisphere.y, global_illumination.cl:239)
  int hitPrim;  // primitive the current shading point lies on (= previousPrimitive of the reference)
  int depth;
  int stage;    // PathStage
};

__device__ __forceinline__ void path_reset(PathState& ps) {
  ps.direct[0] = ps.direct[1] = ps.direct[2] = 0.0f;
  ps.indirect[0] = ps.indirect[1] = ps.indirect[2] = 0.0f;
  ps.stage = ST_PRIMARY;
}

// r/h: the ray that just finished (in stage ps.stage) and its hit.  Returns true when the sample is
// complete; otherwise r, tStart, ignore, anyHit describe the next ray of the path.
// The shading position doubles as the origin of the shadow ray and of the next extension ray, the
// shadow ray's direction is positionToLight, and previousNormal/previousPrimitive of the reference
// coincide with nrm/hitPrim at every point they are read -- so none of them is stored separately.
// lightHitKnown: -1 = scan the light list here; 0 / 1 = the caller already did (is_light(sc, h.prim))
__device__ __forceinline__ bool shade_step(const LtSceneDev& sc, const PathConsts& pc, PathState& ps, Ray& r,
                                           const Hit& h, float fx, float fy, unsigned sampleIndex, float& tStart,
                                           int& ignore, bool& anyHit, int lightHitKnown = -1) {
  bool sampleDone = false, wantShadow = false, wantExt = false, retrace = false;
  unsigned seedBase = 0;

  if (ps.stage == ST_PRIMARY || ps.stage == ST_EXTENSION) {
    // basic_lighting.cl:230-246 / accumulator.cl:233-238 / global_illumination.cl:255-274, 310-331
    bool lightHit = (ps.stage == ST_EXTENSION || pc.isGI || pc.whiteOnLight) &&
                    (lightHitKnown >= 0 ? lightHitKnown != 0 : is_light(sc, h.prim));
    if (lightHit) {
      if (ps.stage == ST_PRIMARY) {
        ps.direct[0] = ps.direct[1] = ps.direct[2] = 1.0f;
        sampleDone = true;
      } else {
        // dot(previousNormal (w = 1), direction (w = hemisphere.y)), global_illumination.cl:321.
        // The reference does not advance the ray, so it traces the same ray again at the next depth, finds the same
        // hit (the hit is a function of the ray alone) and lands here again, until maxDepth.  Those traversals change
        // nothing but the depth: the remaining terms 1/(depth+1) * d are added here, in the same order, without
        // tracing (the counting launches still retrace, so that their counts are the reference's).
        const float d = FADD(FADD(FADD(FMUL(ps.nrm[0], r.dx), FMUL(ps.nrm[1], r.dy)), FMUL(ps.nrm[2], r.dz)),
                             FMUL(1.0f, ps.extW));
        do {
          float w = (float)__ddiv_rn(1.0, (double)(ps.depth + 1));
          float c = FMUL(FMUL(w, 1.0f), d);
          ps.indirect[0] = FADD(ps.indirect[0], c);
          ps.indirect[1] = FADD(ps.indirect[1], c);
          ps.indirect[2] = FADD(ps.indirect[2], c);
          ps.depth++;
        } while (pc.foldLightHits && ps.depth < pc.maxDepth);
        if (ps.depth >= pc.maxDepth) sampleDone = true;
        else retrace = true;
      }
    } else if (h.hit == 1) {
      const RefPrim* prim = sc.prims + h.prim;
      const RefMaterial* mat = sc.mats + prim->materialIndex;
      float w0 = bary0(h.u, h.v);
      float pos[3];
      lerp_plain(prim->a, prim->b, prim->c, w0, h.u, h.v, pos);
      lerp_plain(prim->na, prim->nb, prim->nc, w0, h.u, h.v, ps.nrm);
      ps.diffuse[0] = mat->diffuse[0]; ps.diffuse[1] = mat->diffuse[1]; ps.diffuse[2] = mat->diffuse[2];
      ps.hitPrim = h.prim;
      r.ox = pos[0]; r.oy = pos[1]; r.oz = pos[2];  // origin of the shadow ray and of the next extension
      wantShadow = true;
      seedBase = (ps.stage == ST_PRIMARY) ? sampleIndex : sampleIndex + (unsigned)ps.depth + 5u;
      ps.stage = (ps.stage == ST_PRIMARY) ? ST_SHADOW_DIRECT : ST_SHADOW_EXT;
    } else {
      sampleDone = true;
    }
  } else {
    // the shadow ray's direction is positionToLight, its origin the shaded position
    bool lit = (h.hit == 0);
    // float4 dot: the w term is 0 * normal.w = +0, which turns a -0 sum into +0
    float d = FADD(FADD(FADD(FMUL(r.dx, ps.nrm[0]), FMUL(r.dy, ps.nrm[1])), FMUL(r.dz, ps.nrm[2])), 0.0f);
    if (ps.stage == ST_SHADOW_DIRECT) {  // basic_lighting.cl:272-274, global_illumination.cl:296-309
      if (lit) {
        ps.direct[0] = FMUL(ps.diffuse[0], d); ps.direct[1] = FMUL(ps.diffuse[1], d); ps.direct[2] = FMUL(ps.diffuse[2], d);
      }
      if (pc.isGI && pc.maxDepth > 0) {
        wantExt = true;
        seedBase = sampleIndex + 3u;
        ps.depth = 0;
      } else {
        sampleDone = true;
      }
    } else {  // global_illumination.cl:352-365
      if (lit) {
        float w = (float)__ddiv_rn(1.0, (double)(ps.depth + 1));
        ps.indirect[0] = FADD(ps.indirect[0], FMUL(FMUL(w, ps.diffuse[0]), d));
        ps.indirect[1] = FADD(ps.indirect[1], FMUL(FMUL(w, ps.diffuse[1]), d));
        ps.indirect[2] = FADD(ps.indirect[2], FMUL(FMUL(w, ps.diffuse[2]), d));
        seedBase = sampleIndex + (unsigned)ps.depth + 8u;
        ps.depth++;
        // the reference still draws a direction at the last depth, but never traces it
        if (ps.depth >= pc.maxDepth) sampleDone = true;
        else wantExt = true;
      } else {
        sampleDone = true;
      }
    }
  }

  // the hash RNG (fp64 fmod + sin), one code site for every stage
  float rA = 0.0f, rB = 0.0f, rC = 0.0f;
  if (wantShadow || wantExt) {
    rA = lt_random(fx, fy, (float)seedBase);
    rB = lt_random(fx, fy, (float)(seedBase + 1u));
    if (wantShadow) rC = lt_random(fx, fy, (float)(seedBase + 2u));
  }

  ignore = -1;
  tStart = pc.tInit;
  anyHit = false;
  if (wantShadow) {
    float pos[3] = {r.ox, r.oy, r.oz};
    tStart = make_shadow_ray(sc, pos, rA, rB, rC, r);
    ignore = ps.hitPrim;
    anyHit = true;
  } else if (wantExt) {  // global_illumination.cl:300-305, 355-361
    float dir[4];
    sample_hemisphere(rA, rB, ps.nrm, dir);
    r.dx = dir[0]; r.dy = dir[1]; r.dz = dir[2];  // origin stays the shaded position
    ps.extW = dir[3];
    ignore = ps.hitPrim;
    ps.stage = ST_EXTENSION;
  } else if (retrace) {
    ignore = ps.hitPrim;
  }
  return sampleDone;
}

// colour of a finished sample: GI returns directColor + indirectColor (global_illumination.cl:375);
// the lighting kernels return outputColor as is (basic_lighting.cl:277) -- the add would turn -0 into +0
__device__ __forceinline__ void sample_colour(const PathConsts& pc, const PathState& ps, float c[3]) {
  c[0] = ps.direct[0]; c[1] = ps.direct[1]; c[2] = ps.direct[2];
  if (pc.isGI) {
    c[0] = FADD(ps.direct[0], ps.indirect[0]);
    c[1] = FADD(ps.direct[1], ps.indirect[1]);
    c[2] = FADD(ps.direct[2], ps.indirect[2]);
  }
}

// basic_lighting.cl:309-320 / global_illumination.cl:408-419: first sample copies, later samples
// blend with a = (25 - x)/25
__device__ __forceinline__ void blend_sample(const PathConsts& pc, int sample, const float c[3], float frameColor[3]) {
  if (pc.samplesPerFrame == 1 || sample == 0) {
    frameColor[0] = c[0]; frameColor[1] = c[1]; frameColor[2] = c[2];
  } else {
    float a = FDIV((float)(25 - sample), 25.0f);
    float ia = FSUB(1.0f, a);
#pragma unroll
    for (int k = 0; k < 3; k++) frameColor[k] = FADD(FMUL(ia, frameColor[k]), FMUL(a, c[k]));
  }
}
__device__ __forceinline__ void finish_frame_colour(const PathConsts& pc, int kernelMode, float frameColor[3]) {
  // every stochastic kernel file clamps in linearKernel and not in tileKernel (basic_lighting.cl:318-320
  // vs :365-367, accumulator.cl:316-318 vs :356-358, both global_illumination.cl)
  if (kernelMode == 0) {
#pragma unroll
    for (int k = 0; k < 3; k++) frameColor[k] = fminf(fmaxf(frameColor[k], 0.0f), 1.0f);
  }
}
