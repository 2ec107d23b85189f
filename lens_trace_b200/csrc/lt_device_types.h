// lt_device_types.h -- launch descriptor and counters read by the device code (lt_device.cuh).  Device-safe: no host
// headers, so that NVRTC can compile it for plug-in kernels (it is handed to NVRTC from memory, like lt_device.cuh).
#pragma once
#include "lens_trace_b200_device.cuh"  // buffer layouts

// The values of enum lt_kernel and enum lt_flags (include/lens_trace_b200.h) that the device code tests: NVRTC cannot
// include the public header.  lt_plan.cpp checks that both agree.
constexpr int LT_DEV_KERNEL_BASIC_CU = 0;
constexpr int LT_DEV_KERNEL_BASIC_CL = 1;
constexpr int LT_DEV_KERNEL_CUSTOM_BARY = 2;
constexpr int LT_DEV_KERNEL_LIGHTING25 = 3;
constexpr int LT_DEV_KERNEL_ACCUMULATOR = 4;
constexpr int LT_DEV_KERNEL_GI25 = 5;
constexpr int LT_DEV_KERNEL_GI = 6;
constexpr int LT_DEV_FLAG_STATS = 1 << 0;
constexpr int LT_DEV_FLAG_CULL = 1 << 1;
constexpr int LT_DEV_FLAG_STATS_TRACED = 1 << 7;

#define LT_BLOCK 128     // threads per block of the library's traversal kernels
#define LT_MAX_BATCH 16  // leaf-list entries per thread (shared memory: [LT_MAX_BATCH][LT_BLOCK] ints)

// stack levels a stack traversal reserves for a tree of `stackDepth` levels (LtSceneDev, or the planner's scene facts)
template <class Scene>
__host__ __device__ inline int lt_stack_levels(const Scene& s) { return s.stackDepth < 1 ? 1 : s.stackDepth; }
// Dynamic shared memory of a traversal, ints laid out [level][thread]: `levels` stack levels, the LT_MAX_BATCH-entry
// leaf list / FIFO, and for culled launches `levels` entry distances (lt_device.cuh: LT_TRAV_SMEM carves it)
__host__ __device__ inline unsigned lt_traversal_smem(int levels, unsigned threads, bool cull) {
  return (unsigned)(levels * (cull ? 2 : 1) + LT_MAX_BATCH) * threads * 4u;
}

struct LtLaunch {
  int kernel;        // lt_kernel
  int kernelMode;    // 0 linear, 1 tile
  int width, height, depth;
  int maxRayDepth;
  int frames;
  unsigned frameStride;
  int accumMode;
  float accumWeight;
  int flags;
  // Row window of a tile split (multi-GPU): this launch renders `height` rows of an image of `fullHeight` rows;
  // local row j is image row ((j / rowBlock) * rowStride + rowPhase) * rowBlock + j % rowBlock (blocks of rowBlock
  // rows dealt round-robin to rowStride devices).  rowStride <= 1: the whole image (fullHeight == height).
  int fullHeight, rowBlock, rowStride, rowPhase;
  RefCamera cam;
};

// The pixels of a masked launch (lt_render_masked_device): `count` pixel indices (py * width + px) at `list`, in the
// order thread_pixel gives pixels to threads; m2: the Welford sums beside the running mean (M2Sink), or nullptr.
// The kernels' LIST / M2 variants read it; the others take it as an unused last argument.
struct LtList {
  const int* list;
  int count;
  float* m2;
};

struct LtCounters {
  unsigned long long rays, nodeTests, triTests;
};

