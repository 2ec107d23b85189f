// lens_trace_b200_device_cl.h -- the plug-in device API of lens_trace_b200_device.cuh, for OpenCL C kernel files.
//
// A user-written .cl file (include/lens_trace_b200.h: lt_plugin_load) opts in with exactly
//   #include "lens_trace_b200_device_cl.h"
// and may then call lt_trace() and the other functions below instead of walking the 32-byte node array on its own:
// the library's own traversal (the threaded tree for small scenes, the stack traversal in shared memory for large
// ones), RNG and sampling, as lens_trace_b200_device.cuh offers them to .cu plug-ins, under the same names and in
// OpenCL C types.  Each function is a thin conversion to that header's function; none adds arithmetic of its own.
//
// How it is compiled (lt_plugin.cu): the library replaces the include line with an empty line (the user's line numbers
// stay), compiles lens_trace_b200_device.cuh at global scope (its `lt_scene` constant is the one the library fills
// before every launch), then the OpenCL C runtime (lt_opencl_c.cuh), then this file and the user's text inside
// namespace lt_opencl.  So this file is C++ on the runtime's vector types, not OpenCL C, and is not meant to be
// compiled on its own.  The library launches such a file with the dynamic shared memory lt_trace needs for the
// work-group; the OpenCL C subset still has no __local memory, so nothing else claims it.
//
// The w components are those the reference's kernel text carries, so that the runtime's four-component dot()
// reproduces its expressions as written: positions and normals from lt_interpolate have w = 1, a hemisphere
// direction has w = hemisphere.y (global_illumination.cl:69-82; dot(previousNormal, direction) includes that term),
// ray origins w = 1 and ray directions w = 0.
#pragma once

// a ray as the reference's kernels hold it (origin and direction as float4)
typedef struct LtRay {
  float4 origin;
  float4 direction;
} LtRay;

// LtHit {t, u, v, primitiveIndex, hitType} and LT_EPSILON_BASIC / LT_EPSILON_GI are those of
// lens_trace_b200_device.cuh.

__device__ __forceinline__ ::LtRay lt_cl_ray(float4 origin, float4 direction) {
  ::LtRay r;
  r.ox = origin.x; r.oy = origin.y; r.oz = origin.z;
  r.dx = direction.x; r.dy = direction.y; r.dz = direction.z;
  return r;
}

__device__ __forceinline__ LtRay lt_cl_ray(const ::LtRay& r) {
  LtRay c;
  c.origin = float4(r.ox, r.oy, r.oz, 1.0f);
  c.direction = float4(r.dx, r.dy, r.dz, 0.0f);
  return c;
}

// intersect / intersectIgnorePrimitiveIndex of the reference (ignorePrimitiveIndex < 0: nothing ignored); anyHit != 0
// stops at the first accepted triangle (valid when only hitType is read)
__device__ __forceinline__ LtHit lt_trace(float4 origin, float4 direction, float tMax, int ignorePrimitiveIndex,
                                          int anyHit, float epsilon) {
  return ::lt_trace(lt_cl_ray(origin, direction), tMax, ignorePrimitiveIndex, anyHit != 0, epsilon);
}

// shadow query: is anything but `ignorePrimitiveIndex` hit before tMax?
__device__ __forceinline__ bool lt_occluded(float4 origin, float4 direction, float tMax, int ignorePrimitiveIndex,
                                            float epsilon) {
  return ::lt_occluded(lt_cl_ray(origin, direction), tMax, ignorePrimitiveIndex, epsilon);
}

// camera ray of pixel (x, y); `camera` is the kernel's own pointer to the reference's 28-byte camera record, *film
// receives the film position the hash RNG is keyed on
template <class Camera>
__device__ __forceinline__ LtRay lt_camera_ray(const Camera* camera, int x, int y, int width, int height, float2* film) {
  static_assert(sizeof(Camera) == sizeof(RefCamera), "lt_camera_ray takes the reference's 28-byte camera record");
  float fx, fy;
  const LtRay r = lt_cl_ray(::lt_camera_ray(*(const RefCamera*)camera, x, y, width, height, fx, fy));
  *film = float2(fx, fy);
  return r;
}

// random() of the reference's kernels, keyed on the film position
__device__ __forceinline__ float lt_random(float2 film, float seed) { return ::lt_random(film.x, film.y, seed); }

// light sample from three random numbers: *shadow is the ray from `position` towards the sampled point of the sampled
// light primitive (direction normalised); returns the ray's tMax (distance - 0.01)
__device__ __forceinline__ float lt_sample_light(float4 position, float r0, float r1, float r2, LtRay* shadow) {
  const float p[3] = {position.x, position.y, position.z};
  ::LtRay s;
  const float tMax = ::lt_sample_light(p, r0, r1, r2, s);
  *shadow = lt_cl_ray(s);
  shadow->origin = position;
  return tMax;
}

// uniformSampleHemisphere + alignHemisphereWithCoordinateSystem about `normal`; w = hemisphere.y
__device__ __forceinline__ float4 lt_sample_hemisphere(float u1, float u2, float4 normal) {
  const float up[3] = {normal.x, normal.y, normal.z};
  float d[4];
  ::lt_sample_hemisphere(u1, u2, up, d);
  return float4(d[0], d[1], d[2], d[3]);
}

// position and normal (not normalised) at barycentrics (u, v) of a primitive, both with w = 1
__device__ __forceinline__ void lt_interpolate(int primitiveIndex, float u, float v, float4* position, float4* normal) {
  float p[3], n[3];
  ::lt_interpolate(primitiveIndex, u, v, p, n);
  *position = float4(p[0], p[1], p[2], 1.0f);
  *normal = float4(n[0], n[1], n[2], 1.0f);
}

// the material of a primitive: diffuse[3], ior, dissolve, emission[3]
__device__ __forceinline__ const RefMaterial* lt_material_of(int primitiveIndex) {
  return &::lt_material_of(primitiveIndex);
}

__device__ __forceinline__ bool lt_is_light(int primitiveIndex) { return ::lt_is_light(primitiveIndex); }

// progressive running mean: pixel = frameCount > 0 ? (colour + pixel * frameCount) / (frameCount + 1) : colour
__device__ __forceinline__ void lt_accumulate(float* pixel, float3 colour, uint frameCount) {
  const float c[3] = {colour.x, colour.y, colour.z};
  ::lt_accumulate(pixel, c, frameCount);
}
