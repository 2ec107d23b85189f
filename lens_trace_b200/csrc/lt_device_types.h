// lt_device_types.h -- launch descriptor and counters read by the device code (lt_device.cuh).  Device-safe: no host
// headers, so that NVRTC can compile it for plug-in kernels (it is handed to NVRTC from memory, like lt_device.cuh).
#pragma once
#include "lens_trace_b200_device.cuh"  // buffer layouts

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

struct LtCounters {
  unsigned long long rays, nodeTests, triTests;
};

