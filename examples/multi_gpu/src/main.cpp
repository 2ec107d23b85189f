// multi_gpu -- the global-illumination example rendered by several GPUs of one box through the unchanged
// RendererOpenCL::render() surface: the RenderExtensionB200 on pNext names the device count and the split.
//   samples : GPU g renders frames g, g+G, ...; one NCCL all-reduce of the accumulators per call
//   tiles   : GPU g renders every G-th block of 8 image rows; no collective
// Prints the wall time of the call per device count and the largest difference from the one-GPU picture.
// --kernel names another kernel file: a user's own .cl or .cu file is compiled once and rendered by every GPU (sample
// split only; the file sets its own bounce count, --depth applies to the built-in kernel).
//
//   bin/multi_gpu [--devices N] [--size W H] [--frames F] [--depth D] [--split samples|tiles] [--model obj]
//                 [--kernel file] [--out file.pfm]
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <cmath>
#include <vector>

#include "lens_trace/acceleration_structure_explicit.h"
#include "lens_trace/camera.h"
#include "lens_trace/image_writer.h"
#include "lens_trace/model.h"
#include "lens_trace/opencl/renderer_opencl.h"
#include "lens_trace/structures.h"

int main(int argc, char** argv) {
  uint64_t width = 1920, height = 1080;
  uint32_t frames = 64, depth = 4, devices = 2, split = 1;
  const char* modelPath = "resources/models/cornell_box.obj";
  const char* outName = NULL;
  const char* kernelPath = "examples/global_illumination/resources/kernels/global_illumination.cl";
  for (int i = 1; i < argc; i++) {
    if (!strcmp(argv[i], "--size") && i + 2 < argc) { width = strtoull(argv[++i], NULL, 10); height = strtoull(argv[++i], NULL, 10); }
    else if (!strcmp(argv[i], "--frames") && i + 1 < argc) frames = (uint32_t)atoi(argv[++i]);
    else if (!strcmp(argv[i], "--depth") && i + 1 < argc) depth = (uint32_t)atoi(argv[++i]);
    else if (!strcmp(argv[i], "--devices") && i + 1 < argc) devices = (uint32_t)atoi(argv[++i]);
    else if (!strcmp(argv[i], "--split") && i + 1 < argc) split = !strcmp(argv[++i], "tiles") ? 2u : 1u;
    else if (!strcmp(argv[i], "--model") && i + 1 < argc) modelPath = argv[++i];
    else if (!strcmp(argv[i], "--out") && i + 1 < argc) outName = argv[++i];
    else if (!strcmp(argv[i], "--kernel") && i + 1 < argc) kernelPath = argv[++i];
  }
  Camera camera(0, 2.5, -50, 0);
  Model model(modelPath);
  AccelerationStructureExplicitProperties asProps = {};
  asProps.sType = STRUCTURE_TYPE_ACCELERATION_STRUCTURE_PROPERTIES;
  asProps.accelerationStructureExplicitType = ACCELERATION_STRUCTURE_TYPE_BVH;
  asProps.pModel = &model;
  AccelerationStructureExplicit accel(asProps);

  std::vector<float> one(width * height * 3), many(width * height * 3);
  RendererOpenCL renderer;
  RenderExtensionB200 ext = {};
  ext.sType = STRUCTURE_TYPE_RENDER_EXTENSION_B200;
  ext.frames = frames;
  ext.accumulate = 1;
  ext.maxRayDepth = depth;
  RenderPropertiesOpenCL props = {};
  props.sType = STRUCTURE_TYPE_RENDER_PROPERTIES_OPENCL;
  props.pNext = &ext;
  props.kernelFilePath = kernelPath;
  props.kernelMode = KERNEL_MODE_LINEAR;
  props.threadOrganizationMode = THREAD_ORGANIZATION_MODE_MAX_FIT;
  props.imageDimensions[0] = width;
  props.imageDimensions[1] = height;
  props.imageDimensions[2] = 3;
  props.outputBufferSize = one.size() * sizeof(float);
  props.pAccelerationStructureExplicit = &accel;
  props.pModel = &model;
  props.pCamera = &camera;

  double ms[2] = {0, 0};
  for (int pass = 0; pass < 2; pass++) {
    ext.deviceCount = pass == 0 ? 1 : devices;
    ext.splitMode = split;
    props.pOutputBuffer = pass == 0 ? one.data() : many.data();
    for (int rep = 0; rep < 3; rep++) {  // first call uploads the scene (and starts NCCL); time the last
      camera.resetFrameCount();
      auto t0 = std::chrono::steady_clock::now();
      renderer.render(&props);
      ms[pass] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
  }
  double maxRel = 0.0;
  size_t differing = 0;
  for (size_t i = 0; i < one.size(); i++) {
    double d = std::fabs((double)one[i] - many[i]) / std::fmax(std::fabs((double)one[i]), 1e-3);
    if (d > maxRel) maxRel = d;
    if (one[i] != many[i]) differing++;
  }
  printf("%s\n%llux%llu, %u frames, %u bounces, split = %s\n", kernelPath, (unsigned long long)width,
         (unsigned long long)height, frames, depth, split == 2 ? "tiles" : "samples");
  printf("1 GPU : %.2f ms per call\n%u GPUs: %.2f ms per call (%.2fx)\n", ms[0], devices, ms[1], ms[0] / ms[1]);
  printf("largest relative difference from the one-GPU picture: %.3g (%zu of %zu floats differ)\n", maxRel, differing,
         one.size());
  if (outName) {
    BufferToImageProperties out = {};
    out.sType = STRUCTURE_TYPE_BUFFER_TO_IMAGE_PROPERTIES;
    out.pBuffer = many.data();
    out.bufferSize = many.size() * sizeof(float);
    out.imageDimensions[0] = width;
    out.imageDimensions[1] = height;
    out.imageDimensions[2] = 3;
    out.imageType = IMAGE_TYPE_JPEG;
    out.filename = outName;
    ImageWriter::writeBufferToImage(out);
  }
  return maxRel <= 1e-4 ? 0 : 1;
}
