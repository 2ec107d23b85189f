// lt_opencl_c.cuh -- the subset of OpenCL C that user kernel files may use, as CUDA device code.
//
// A user's .cl file is compiled by NVRTC for sm_100a (lt_plugin.cu): the library hands this header over from
// memory, translates the file (vector literals `(float4)(...)` -> `float4(...)`, `__constant` at file scope ->
// device constant data, the other address-space qualifiers dropped, __kernel -> __device__, __local -> an undefined
// name, `#pragma OPENCL` lines dropped), and places the user's text inside namespace lt_opencl,
// after this header.  Entities without an execution-space qualifier are device code (-default-device).
// A file that includes lens_trace_b200_device_cl.h (the plug-in device API in OpenCL C types) has
// lens_trace_b200_device.cuh compiled at global scope before this header, and the OpenCL C view of it inside
// namespace lt_opencl after this header, ahead of the user's text.
//
// What is provided (OpenCL C 1.2, the part the reference's kernel files use):
//   - address spaces __global __constant __private (and the spellings without underscores), __kernel / kernel
//   - float2/3/4, int2/3/4, uint2/3/4: component-wise + - * /, unary -, += -= *= /=, scalar broadcast on either
//     side, .x .y .z .w and the .xy / .xyz swizzles.  sizeof and alignment of a 3-component vector are those of the
//     4-component one (16 bytes for float3), as the specification requires.  A float vector mixed with a double
//     scalar does not compile, as in OpenCL C.
//   - math built-ins on float and double by C++ overloading, which selects what OpenCL C's overloading selects
//     (sin cos sqrt fabs fmin fmax fmod floor ceil pow exp log come from CUDA's math library; min max clamp here),
//     and the component-wise float-vector forms of fabs floor ceil sqrt fmin fmax min max clamp
//   - geometric built-ins by the specification's formulae, FP32, one rounding per operation, left to right and never
//     contracted (whatever the file's FP_CONTRACT setting):
//       dot(a,b) = ((a.x*b.x + a.y*b.y) + a.z*b.z) + a.w*b.w;  cross(a,b) = (a.y*b.z - a.z*b.y, ..., 0)
//       length(a) = sqrt(dot(a,a));  distance(a,b) = length(a - b);  normalize(a) = a / length(a)
//   - work-item functions get_global_id/size, get_local_id/size, get_group_id, get_num_groups, dimensions 0..2
// Anything else -- __local memory, barriers, images, atomics, half -- is a compile error at the user's line.
#pragma once

namespace lt_opencl {

typedef unsigned int uint;
typedef unsigned short ushort;
typedef unsigned char uchar;
typedef unsigned long ulong;

// ---- work-item functions: an NDRange launch is a CUDA grid (global = grid * block, local = block) ----
__device__ __forceinline__ size_t get_local_id(uint d) {
  return d == 0 ? threadIdx.x : d == 1 ? threadIdx.y : d == 2 ? threadIdx.z : 0;
}
__device__ __forceinline__ size_t get_local_size(uint d) {
  return d == 0 ? blockDim.x : d == 1 ? blockDim.y : d == 2 ? blockDim.z : 1;
}
__device__ __forceinline__ size_t get_group_id(uint d) {
  return d == 0 ? blockIdx.x : d == 1 ? blockIdx.y : d == 2 ? blockIdx.z : 0;
}
__device__ __forceinline__ size_t get_num_groups(uint d) {
  return d == 0 ? gridDim.x : d == 1 ? gridDim.y : d == 2 ? gridDim.z : 1;
}
__device__ __forceinline__ size_t get_global_id(uint d) { return get_group_id(d) * get_local_size(d) + get_local_id(d); }
__device__ __forceinline__ size_t get_global_size(uint d) { return get_num_groups(d) * get_local_size(d); }
__device__ __forceinline__ uint get_work_dim() { return 2; }

// ---- scalar traits (NVRTC has no standard library) ----
template <class T> struct lt_scalar { enum { ok = 0, fp = 0 }; };
#define LT_SCALAR(T, F) template <> struct lt_scalar<T> { enum { ok = 1, fp = F }; };
LT_SCALAR(float, 1) LT_SCALAR(double, 2) LT_SCALAR(char, 0) LT_SCALAR(unsigned char, 0) LT_SCALAR(short, 0)
LT_SCALAR(unsigned short, 0) LT_SCALAR(int, 0) LT_SCALAR(unsigned int, 0) LT_SCALAR(long, 0)
LT_SCALAR(unsigned long, 0) LT_SCALAR(long long, 0) LT_SCALAR(unsigned long long, 0) LT_SCALAR(bool, 0)
#undef LT_SCALAR
template <bool B, class T = void> struct lt_enable_if {};
template <class T> struct lt_enable_if<true, T> { typedef T type; };

// element type E may take scalar S: an integer vector takes integers, a float vector integers and float, never double
template <class E, class S> struct lt_broadcast {
  enum { ok = lt_scalar<S>::ok && (lt_scalar<E>::fp ? lt_scalar<S>::fp != 2 : lt_scalar<S>::fp == 0) };
};

// ---- vector types ----
template <class T> struct lt_swz2 {  // .xy of a wider vector: reads as a 2-vector, takes one on assignment
  T x, y;
  template <class V> __device__ lt_swz2& operator=(const V& v) { x = v.x; y = v.y; return *this; }
};
template <class T> struct lt_swz3 {  // .xyz of a 4-component vector
  T x, y, z;
  template <class V> __device__ lt_swz3& operator=(const V& v) { x = v.x; y = v.y; z = v.z; return *this; }
};

#define LT_VEC_TYPES(T, P)                                                                                      \
  struct P##2 {                                                                                                  \
    T x, y;                                                                                                      \
    P##2() = default;                                                                                            \
    __device__ constexpr P##2(T a, T b) : x(a), y(b) {}                                                         \
    __device__ constexpr explicit P##2(T a) : x(a), y(a) {}                                                     \
    __device__ P##2(const lt_swz2<T>& s) : x(s.x), y(s.y) {}                                                    \
  };                                                                                                             \
  struct __align__(4 * sizeof(T)) P##3 {                                                                         \
    union {                                                                                                      \
      struct { T x, y, z; };                                                                                    \
      lt_swz2<T> xy;                                                                                             \
    };                                                                                                           \
    P##3() = default;                                                                                            \
    __device__ constexpr P##3(T a, T b, T c) : x(a), y(b), z(c) {}                                              \
    __device__ constexpr explicit P##3(T a) : x(a), y(a), z(a) {}                                               \
    __device__ constexpr P##3(P##2 a, T c) : x(a.x), y(a.y), z(c) {}                                            \
    __device__ constexpr P##3(T a, P##2 b) : x(a), y(b.x), z(b.y) {}                                            \
    __device__ P##3(const lt_swz3<T>& s) : x(s.x), y(s.y), z(s.z) {}                                            \
  };                                                                                                             \
  struct __align__(4 * sizeof(T)) P##4 {                                                                         \
    union {                                                                                                      \
      struct { T x, y, z, w; };                                                                                 \
      lt_swz2<T> xy;                                                                                             \
      lt_swz3<T> xyz;                                                                                            \
    };                                                                                                           \
    P##4() = default;                                                                                            \
    __device__ constexpr P##4(T a, T b, T c, T d) : x(a), y(b), z(c), w(d) {}                                   \
    __device__ constexpr explicit P##4(T a) : x(a), y(a), z(a), w(a) {}                                         \
    __device__ constexpr P##4(P##3 a, T d) : x(a.x), y(a.y), z(a.z), w(d) {}                                    \
    __device__ constexpr P##4(T a, P##3 b) : x(a), y(b.x), z(b.y), w(b.z) {}                                    \
    __device__ constexpr P##4(P##2 a, P##2 b) : x(a.x), y(a.y), z(b.x), w(b.y) {}                               \
    __device__ constexpr P##4(P##2 a, T c, T d) : x(a.x), y(a.y), z(c), w(d) {}                                 \
  };                                                                                                             \
  static_assert(sizeof(P##3) == 4 * sizeof(T) && alignof(P##3) == 4 * sizeof(T), "3-component vectors are padded");
LT_VEC_TYPES(float, float)
LT_VEC_TYPES(int, int)
LT_VEC_TYPES(uint, uint)
#undef LT_VEC_TYPES

// ---- component-wise operators, one set per vector type ----
#define LT_ZIP2(op) (a.x op b.x, a.y op b.y)
#define LT_ZIP3(op) (a.x op b.x, a.y op b.y, a.z op b.z)
#define LT_ZIP4(op) (a.x op b.x, a.y op b.y, a.z op b.z, a.w op b.w)
#define LT_NEG2 (-a.x, -a.y)
#define LT_NEG3 (-a.x, -a.y, -a.z)
#define LT_NEG4 (-a.x, -a.y, -a.z, -a.w)
#define LT_VEC_OPS(V, T, N)                                                                                         \
  __device__ __forceinline__ V operator+(V a, V b) { return V LT_ZIP##N(+); }                                      \
  __device__ __forceinline__ V operator-(V a, V b) { return V LT_ZIP##N(-); }                                      \
  __device__ __forceinline__ V operator*(V a, V b) { return V LT_ZIP##N(*); }                                      \
  __device__ __forceinline__ V operator/(V a, V b) { return V LT_ZIP##N(/); }                                      \
  __device__ __forceinline__ V operator-(V a) { return V LT_NEG##N; }                                              \
  __device__ __forceinline__ V operator+(V a) { return a; }                                                        \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V lt_bc(S s, V*) {                                                                    \
    static_assert(lt_broadcast<T, S>::ok,                                                                          \
                  "OpenCL C: a scalar of this type cannot be mixed with this vector type (e.g. float vector and "  \
                  "double scalar)");                                                                               \
    return V((T)s);                                                                                                \
  }                                                                                                                \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V operator+(V a, S s) { return a + lt_bc(s, (V*)0); }                                \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V operator+(S s, V a) { return lt_bc(s, (V*)0) + a; }                                \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V operator-(V a, S s) { return a - lt_bc(s, (V*)0); }                                \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V operator-(S s, V a) { return lt_bc(s, (V*)0) - a; }                                \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V operator*(V a, S s) { return a * lt_bc(s, (V*)0); }                                \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V operator*(S s, V a) { return lt_bc(s, (V*)0) * a; }                                \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V operator/(V a, S s) { return a / lt_bc(s, (V*)0); }                                \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V operator/(S s, V a) { return lt_bc(s, (V*)0) / a; }                                \
  __device__ __forceinline__ V& operator+=(V& a, V b) { return a = a + b; }                                        \
  __device__ __forceinline__ V& operator-=(V& a, V b) { return a = a - b; }                                        \
  __device__ __forceinline__ V& operator*=(V& a, V b) { return a = a * b; }                                        \
  __device__ __forceinline__ V& operator/=(V& a, V b) { return a = a / b; }                                        \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V& operator+=(V& a, S s) { return a = a + s; }                                        \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V& operator-=(V& a, S s) { return a = a - s; }                                        \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V& operator*=(V& a, S s) { return a = a * s; }                                        \
  template <class S, class = typename lt_enable_if<lt_scalar<S>::ok>::type>                                        \
  __device__ __forceinline__ V& operator/=(V& a, S s) { return a = a / s; }

#define LT_VEC_OPS_ALL(T, P) LT_VEC_OPS(P##2, T, 2) LT_VEC_OPS(P##3, T, 3) LT_VEC_OPS(P##4, T, 4)
LT_VEC_OPS_ALL(float, float)
LT_VEC_OPS_ALL(int, int)
LT_VEC_OPS_ALL(uint, uint)
#undef LT_VEC_OPS_ALL
#undef LT_VEC_OPS

// ---- math built-ins ----
// CUDA's math library already declares the float and double overloads of sin cos sqrt fabs fmin fmax fmod floor ceil
// pow exp log, and min / max for the scalar types; they are brought into this namespace so that the vector forms
// below do not hide them.
using ::ceil;
using ::cos;
using ::exp;
using ::fabs;
using ::floor;
using ::fmax;
using ::fmin;
using ::fmod;
using ::log;
using ::max;
using ::min;
using ::pow;
using ::sin;
using ::sqrt;

__device__ __forceinline__ float clamp(float x, float lo, float hi) { return fmin(fmax(x, lo), hi); }
__device__ __forceinline__ double clamp(double x, double lo, double hi) { return fmin(fmax(x, lo), hi); }
__device__ __forceinline__ int clamp(int x, int lo, int hi) { return min(max(x, lo), hi); }
__device__ __forceinline__ uint clamp(uint x, uint lo, uint hi) { return min(max(x, lo), hi); }

#define LT_MAP1(V, f, N) __device__ __forceinline__ V f(V a) { return V LT_MAP1_##N(f); }
#define LT_MAP1_2(f) (f(a.x), f(a.y))
#define LT_MAP1_3(f) (f(a.x), f(a.y), f(a.z))
#define LT_MAP1_4(f) (f(a.x), f(a.y), f(a.z), f(a.w))
#define LT_MAP2(V, f, N)                                                                 \
  __device__ __forceinline__ V f(V a, V b) { return V LT_MAP2_##N(f); }                  \
  __device__ __forceinline__ V f(V a, float s) { return f(a, V(s)); }
#define LT_MAP2_2(f) (f(a.x, b.x), f(a.y, b.y))
#define LT_MAP2_3(f) (f(a.x, b.x), f(a.y, b.y), f(a.z, b.z))
#define LT_MAP2_4(f) (f(a.x, b.x), f(a.y, b.y), f(a.z, b.z), f(a.w, b.w))
#define LT_FVEC_MATH(V, N)                                                                                       \
  LT_MAP1(V, fabs, N) LT_MAP1(V, floor, N) LT_MAP1(V, ceil, N) LT_MAP1(V, sqrt, N) LT_MAP2(V, fmin, N)          \
  LT_MAP2(V, fmax, N) LT_MAP2(V, min, N) LT_MAP2(V, max, N)                                                      \
  __device__ __forceinline__ V clamp(V x, V lo, V hi) { return fmin(fmax(x, lo), hi); }                          \
  __device__ __forceinline__ V clamp(V x, float lo, float hi) { return fmin(fmax(x, lo), hi); }
LT_FVEC_MATH(float2, 2)
LT_FVEC_MATH(float3, 3)
LT_FVEC_MATH(float4, 4)
#undef LT_FVEC_MATH

// ---- geometric built-ins: the specification's formulae, one rounding per operation, never contracted ----
__device__ __forceinline__ float dot(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float dot(float2 a, float2 b) { return __fadd_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)); }
__device__ __forceinline__ float dot(float3 a, float3 b) {
  return __fadd_rn(__fadd_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)), __fmul_rn(a.z, b.z));
}
__device__ __forceinline__ float dot(float4 a, float4 b) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)), __fmul_rn(a.z, b.z)),
                   __fmul_rn(a.w, b.w));
}
__device__ __forceinline__ float lt_diffprod(float p, float q, float r, float s) {
  return __fsub_rn(__fmul_rn(p, q), __fmul_rn(r, s));
}
__device__ __forceinline__ float3 cross(float3 a, float3 b) {
  return float3(lt_diffprod(a.y, b.z, a.z, b.y), lt_diffprod(a.z, b.x, a.x, b.z), lt_diffprod(a.x, b.y, a.y, b.x));
}
__device__ __forceinline__ float4 cross(float4 a, float4 b) {
  return float4(lt_diffprod(a.y, b.z, a.z, b.y), lt_diffprod(a.z, b.x, a.x, b.z), lt_diffprod(a.x, b.y, a.y, b.x),
                0.0f);
}
#define LT_GEOM(V)                                                                                               \
  __device__ __forceinline__ float length(V a) { return __fsqrt_rn(dot(a, a)); }                                \
  __device__ __forceinline__ float distance(V a, V b) { return length(a - b); }                                  \
  __device__ __forceinline__ V normalize(V a) { return a / length(a); }
LT_GEOM(float2)
LT_GEOM(float3)
LT_GEOM(float4)
#undef LT_GEOM

// ---- the reference's kernel arguments, converted to whatever pointer / integer types the user's kernel declares ----
struct lt_cl_pointer {
  void* p;
  template <class T> __device__ operator T*() const { return (T*)p; }
};
struct lt_cl_uint {
  unsigned v;
  template <class T, class = typename lt_enable_if<lt_scalar<T>::ok && lt_scalar<T>::fp == 0>::type>
  __device__ operator T() const { return (T)v; }
};

// ---- what the subset leaves out: a compile error at the user's line ----
void barrier(...) = delete;
void mem_fence(...) = delete;
void read_mem_fence(...) = delete;
void write_mem_fence(...) = delete;

}  // namespace lt_opencl

// The address-space qualifiers and __kernel are rewritten by the translation (lt_plugin.cu), not defined as macros
// here: CUDA's own __global__ and __shared__ expand to the words global and shared.
#define half lt_opencl_half_is_not_supported
#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif
#ifndef FLT_MAX
#define FLT_MAX 3.402823466e+38F
#endif
#define M_PI_F 3.14159265358979323846f
