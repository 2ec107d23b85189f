// lens_trace_b200_device.cuh -- device-side view of an uploaded scene, for plug-in kernels.
//
// A user-written .cu kernel with the reference's kernel ABI (linearKernel / tileKernel, see
// include/lens_trace_b200.h: lt_plugin_load) may `#include "lens_trace_b200_device.cuh"` -- the library hands
// this header to NVRTC itself -- and call lt_trace() instead of walking the 32-byte node array on its own.
// lt_trace() has the reference's intersect()/intersectIgnorePrimitiveIndex() semantics (basic.cu:156-243: near
// child first, strict t < best, no t > 0 test, first primitive of a leaf only) and the same FP32 operation
// order as the built-in pipelines, on the re-flattened 64-byte child-pair nodes and 48-byte triangles.
// The library fills `lt_scene` (a __constant__ in the plug-in's module) before every launch.
//
// The same file defines the buffer layouts for the library itself (lens_trace_b200/csrc/lt_internal.h).
#pragma once
#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#include <stdint.h>
#else
typedef int int32_t;
typedef unsigned int uint32_t;
typedef unsigned short uint16_t;
typedef unsigned char uint8_t;
#endif

// ---- reference layouts (as uploaded by the caller) ----
struct RefNode {  // include/lens_trace/acceleration_structure_explicit.h:20-32 (32 B)
  float boundsMin[3];
  float boundsMax[3];
  int32_t offset;  // primitivesOffset | secondChildOffset
  uint16_t primitiveCount;
  uint8_t axis;
  uint8_t pad;
};
static_assert(sizeof(RefNode) == 32, "LinearBVHNode is 32 bytes");

struct RefPrim {  // include/lens_trace/acceleration_structure_explicit.h:34-42 (76 B)
  float a[3], b[3], c[3];
  float na[3], nb[3], nc[3];
  int32_t materialIndex;
};
static_assert(sizeof(RefPrim) == 76, "Primitive is 76 bytes");

struct RefMaterial {  // include/lens_trace/model.h:26-31 (32 B)
  float diffuse[3];
  float ior;
  float dissolve;
  float emission[3];
};
static_assert(sizeof(RefMaterial) == 32, "Material is 32 bytes");

struct RefLights {  // include/lens_trace/acceleration_structure_explicit.h:44-47 (260 B)
  uint32_t count;
  uint32_t primitives[64];
};

struct RefCamera {  // src/camera.cpp:14-19 (28 B)
  float position[3];
  float yaw, pitch, roll;
  uint32_t frameCount;
};
static_assert(sizeof(RefCamera) == 28, "camera buffer is 28 bytes");

// ---- re-flattened device layouts ----
// One 64-byte record per INNER reference node, holding the boxes of both children so that one
// dependent round trip tests two reference nodes.  Child reference: >= 0 -> index of the child's
// own LtWideNode; < 0 -> ~primitivesOffset of a leaf child.  Four 128-bit loads.
struct __align__(16) LtWideNode {
  float4 bx;   // Lmin.x Lmax.x Rmin.x Rmax.x   (L = reference node i+1, R = secondChildOffset)
  float4 by;   // Lmin.y Lmax.y Rmin.y Rmax.y
  float4 bz;   // Lmin.z Lmax.z Rmin.z Rmax.z
  int4 meta;   // Lref, Rref, axis, (Lcount | Rcount << 16)  (leaf primitiveCount, stats only)
};
static_assert(sizeof(LtWideNode) == 64, "wide node is 64 bytes");

// 48-byte triangle record for the intersection test: A, e1 = B - A, e2 = C - A (the same IEEE
// subtractions basic.cu:100-101 performs per test, done once at upload).  Three 128-bit loads.
struct __align__(16) LtTri {
  float4 q0;  // A.x A.y A.z e1.x
  float4 q1;  // e1.y e1.z e2.x e2.y
  float4 q2;  // e2.z bits(materialIndex) 0 0
};
static_assert(sizeof(LtTri) == 48, "triangle record is 48 bytes");

// Threaded ("skip pointer") form of the same tree, built for scenes small enough that eight copies stay
// cache resident.  The reference visits children near-first by the sign of the ray direction on the split
// axis and never culls by t, so for each of the 8 sign octants the visit order of the whole tree is one
// fixed depth-first sequence.  Copy o (records [o*nodeCount, (o+1)*nodeCount)) holds the reference nodes in
// that sequence: the next record is the first node to visit after a box hit, `skip` the first node after
// the subtree -- a traversal is `i = hit && inner ? i + 1 : skip` with no stack.  The bounds are stored
// already selected by the octant's dirIsNeg (basic.cu:88-91), so the slab test needs no selects either.
// Host-built copies are followed by eight PRUNED copies (copy o at records prunedBase + o * prunedStride): the
// same sequences without the inner nodes whose two child boxes lie inside their own box and which a ray that
// entered the nearest kept ancestor usually enters too.  For a ray with finite, nonzero direction reciprocals and a
// finite origin a contained child is hit only if its parent is, so the walk records the same leaves; every other ray
// starts in the full copies.  When every leaf box lies inside all its ancestors' boxes, that argument makes a leaf's
// reach depend on its own box alone, and the pruned copies are those of a TRAVERSAL TREE: a SAH tree over the
// reference's leaves (each copied as is: box, primitive, count) with exact min/max inner boxes.  It reaches the same
// leaves in another order; LtSceneDev::rank restores the reference's choice among hits of equal t.  Otherwise they
// are pruned copies of the reference tree itself, in the reference's order.  One 32-byte sector, two 128-bit loads.
struct __align__(16) LtThreadNode {
  float4 a;  // lo.x lo.y lo.z hi.x      lo = dirIsNeg ? boundsMax : boundsMin, hi the other one
  float4 b;  // hi.y hi.z bits(link) bits(skip)   link < 0: leaf, ~primitivesOffset; >= 0: inner node
             //                                   skip: absolute record index, LT_DONE at the end of the tree
};
static_assert(sizeof(LtThreadNode) == 32, "threaded node is 32 bytes");

#define LT_DONE ((int)0x80000000)  // traversal sentinel (== ~0x7fffffff, never a primitive)

struct LtSceneDev {
  const LtWideNode* wnodes;
  const LtTri* tris;
  const RefPrim* prims;       // original 76-byte records, read only when shading a hit
  const RefMaterial* mats;
  const RefLights* lights;
  float rootMin[3];
  float rootMax[3];
  int rootRef;                // child reference of the root (leaf root -> ~primitivesOffset)
  int rootCount;              // primitiveCount of a leaf root (stats only)
  int stackDepth;             // entries a traversal stack needs (tree depth), <= 64
  int nodeCount, primCount, matCount;
  int prunedBase, prunedStride;  // pruned copy o of tnodes: records [prunedBase + o * prunedStride, + prunedStride);
                                 // 0 and nodeCount: the full copies (device-built copies, or no pruned copies)
  const LtThreadNode* tnodes;  // 8 * nodeCount full threaded records, then the pruned ones, or NULL (scene too large)
  const int* rank;  // [8][primCount]: position, in octant o's reference visit order, of the leaf whose primitive is p;
                    // set when the pruned copies are a traversal tree (NULL otherwise).  The reference keeps the first
                    // of several triangles with equal t, i.e. the least (t, rank): tri_test breaks equal-t ties by it
};


// ------------------------------------------------------------------------------------------------
// plug-in API (compiled only for plug-ins: NVRTC, or nvcc with -DLT_PLUGIN_API)
//
// The functions below are thin names over the library's OWN device code (lt_device.cuh, handed to NVRTC from memory
// together with this header): lt_trace runs the same traversal the built-in pipelines run -- the stackless threaded
// tree with one 256-bit load per box for small scenes, the child-pair tree with the traversal stack in shared memory
// for large ones -- so a plug-in shader gets the tuned path and, where it follows the reference's kernels, the same
// bits.  Shared memory: the library launches a plug-in that references `lt_scene` with the dynamic shared memory
// lt_trace needs ((stack levels + 16) ints per thread); a plug-in must not declare dynamic shared memory of its own.
// ------------------------------------------------------------------------------------------------
#if defined(__CUDACC_RTC__) || defined(LT_PLUGIN_API)

__constant__ LtSceneDev lt_scene;  // set by the library before each launch of a plug-in that references it

#define LT_THREAD_STRIDE (blockDim.x * blockDim.y * blockDim.z)  // plug-ins run any block shape
#define LT_THREAD_INDEX ((threadIdx.z * blockDim.y + threadIdx.y) * blockDim.x + threadIdx.x)
#include "lt_device.cuh"

struct LtRay {
  float ox, oy, oz;  // origin
  float dx, dy, dz;  // direction (not necessarily normalised: t is in units of its length)
};

struct LtHit {
  float t, u, v;
  int primitiveIndex;  // 0 when nothing was hit, like the reference's payload
  int hitType;         // 1 = hit
};

// |det| thresholds of intersectTriangle as the reference's kernel files compile them (the macro-defined epsilons
// are compared in double precision): basic.cu / basic.cl / custom_opencl.cl / basic_lighting.cl, and the
// accumulator / global-illumination files
#define LT_EPSILON_BASIC 0x1.ad7f2ap-24f
#define LT_EPSILON_GI 0x1.a36e30p-14f

// The reference's intersect (ignorePrimitiveIndex < 0) / intersectIgnorePrimitiveIndex (basic.cu:156-243): near
// child first, strict t < best, no t > 0 test, first primitive of a leaf only.  tMax is the payload's initial t
// (basic.cu passes its FLT_MAX = 1e7, the OpenCL files the real FLT_MAX).  anyHit stops at the first accepted
// triangle (valid when only hitType is read, as the reference's shadow rays do).
__device__ __forceinline__ LtHit lt_trace(const LtRay& r, float tMax, int ignorePrimitiveIndex = -1, bool anyHit = false,
                                          float epsilon = LT_EPSILON_BASIC) {
  LT_TRAV_SMEM(s, lt_scene.tnodes ? 0 : lt_stack_levels(lt_scene))
  Trav t;
  t.r.ox = r.ox; t.r.oy = r.oy; t.r.oz = r.oz;
  t.r.dx = r.dx; t.r.dy = r.dy; t.r.dz = r.dz;
  LtCounters cnt = {0, 0, 0};
  trace<false>(t, lt_scene, ignorePrimitiveIndex, tMax, epsilon, anyHit, s, cnt);
  LtHit h;
  h.t = t.h.t; h.u = t.h.u; h.v = t.h.v;
  h.primitiveIndex = t.h.prim;
  h.hitType = t.h.hit;
  return h;
}

// shadow query (basic_lighting.cl:264-272): is anything but `ignorePrimitiveIndex` hit before tMax?
__device__ __forceinline__ bool lt_occluded(const LtRay& r, float tMax, int ignorePrimitiveIndex = -1,
                                            float epsilon = LT_EPSILON_BASIC) {
  return lt_trace(r, tMax, ignorePrimitiveIndex, true, epsilon).hitType == 1;
}

// camera ray of pixel (px, py) (basic.cu:350-358); fx, fy receive the film position the hash RNG is keyed on
__device__ __forceinline__ LtRay lt_camera_ray(const RefCamera& cam, int px, int py, int width, int height, float& fx,
                                               float& fy) {
  Ray c = camera_ray(cam, px, py, width, height, fx, fy);
  LtRay r;
  r.ox = c.ox; r.oy = c.oy; r.oz = c.oz;
  r.dx = c.dx; r.dy = c.dy; r.dz = c.dz;
  return r;
}

// random() of basic_lighting.cl:64-67 is lt_random(fx, fy, seed) (lt_device.cuh): fp64 fmod + sin, bit-exact.

// uniformSampleHemisphere + alignHemisphereWithCoordinateSystem (global_illumination.cl:69-82); dir[3] = hemisphere.y,
// the w the reference's float4 direction carries into its dot products
__device__ __forceinline__ void lt_sample_hemisphere(float u1, float u2, const float up[3], float dir[4]) {
  sample_hemisphere(u1, u2, up, dir);
}

// position and normal at barycentrics (u, v) of a primitive, unfused (basic_lighting.cl:236-244)
__device__ __forceinline__ void lt_interpolate(int primitiveIndex, float u, float v, float position[3], float normal[3]) {
  const RefPrim* p = lt_scene.prims + primitiveIndex;
  const float w0 = bary0(u, v);
  lerp_plain(p->a, p->b, p->c, w0, u, v, position);
  lerp_plain(p->na, p->nb, p->nc, w0, u, v, normal);
}

__device__ __forceinline__ const RefMaterial& lt_material_of(int primitiveIndex) {
  return lt_scene.mats[lt_scene.prims[primitiveIndex].materialIndex];
}

__device__ __forceinline__ bool lt_is_light(int primitiveIndex) { return is_light(lt_scene, primitiveIndex); }

// light sample (basic_lighting.cl:246-262) from three random numbers: the shadow ray from `position` towards the
// sampled point of the sampled light primitive; returns the ray's tMax (distance - 0.01)
__device__ __forceinline__ float lt_sample_light(const float position[3], float rIndex, float rU, float rV, LtRay& shadow) {
  Ray s;
  const float tMax = make_shadow_ray(lt_scene, position, rIndex, rU, rV, s);
  shadow.ox = s.ox; shadow.oy = s.oy; shadow.oz = s.oz;
  shadow.dx = s.dx; shadow.dy = s.dy; shadow.dz = s.dz;
  return tMax;
}

// progressive accumulator (accumulator.frag:10-19): pixel = frameCount > 0 ? (sample + pixel * frameCount) / (frameCount + 1) : sample
__device__ __forceinline__ void lt_accumulate(float* pixel, const float sample[3], unsigned frameCount) {
#pragma unroll
  for (int k = 0; k < 3; k++) {
    float v = sample[k];
    if (frameCount > 0) v = __fdiv_rn(__fadd_rn(v, __fmul_rn(pixel[k], (float)frameCount)), (float)(frameCount + 1u));
    pixel[k] = v;
  }
}

#endif  // plug-in API
