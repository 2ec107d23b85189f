// renderer_b200.cpp -- RendererCUDA / RendererOpenCL on top of the C-ABI (include/lens_trace_b200.h).
// Replaces src/cuda/renderer_cuda.cpp:41-140 and src/opencl/renderer_opencl.cpp:56-153.
#include <stdio.h>
#include <string.h>

#include "lens_trace/cuda/renderer_cuda.h"
#include "lens_trace/model.h"
#include "lens_trace/opencl/renderer_opencl.h"
#include "lens_trace/resource.h"
#include "lens_trace_b200.h"

#include <atomic>
#include <mutex>
#include <set>
#include <vector>

// ---- object identity for the device-scene cache (include/lens_trace/api.h) ----
namespace {
std::atomic<uint64_t> g_nextObjectId(1);
std::atomic<uint64_t> g_retireGeneration(0);
std::mutex g_retiredMutex;
std::set<uint64_t> g_retired;  // ids of destroyed objects; consulted only when the generation moved

// FNV-1a over the sizes, the whole light container, the materials (small) and up to 16 KB from both ends and the
// middle of the node and primitive arrays: cheap enough for every render() call (the reference re-uploads
// everything per call, src/cuda/renderer_cuda.cpp:90-104), and an in-place edit of a few records that it misses
// can be forced through forgetScenes().
uint64_t fnv(uint64_t h, const void* p, size_t n) {
  const unsigned char* b = (const unsigned char*)p;
  for (size_t i = 0; i < n; i++) h = (h ^ b[i]) * 1099511628211ull;
  return h;
}
uint64_t sample(uint64_t h, const void* p, uint64_t bytes) {
  const uint64_t chunk = 16 * 1024;
  h = fnv(h, &bytes, sizeof bytes);
  if (bytes <= 3 * chunk) return fnv(h, p, (size_t)bytes);
  const char* c = (const char*)p;
  h = fnv(h, c, chunk);
  h = fnv(h, c + ((bytes / 2) & ~(uint64_t)63), chunk);
  return fnv(h, c + bytes - chunk, chunk);
}
}  // namespace

uint64_t lt::newObjectId() { return g_nextObjectId.fetch_add(1); }
void lt::retireObjectId(uint64_t id) {
  std::lock_guard<std::mutex> lock(g_retiredMutex);
  g_retired.insert(id);
  g_retireGeneration.fetch_add(1);
}

RendererB200::RendererB200() : ctx(nullptr), groupCtx(nullptr), groupDevices(0), useCounter(0), seenRetireGeneration(0) {
  if (lt_ctx_create(0, &ctx) != LT_OK) {
    printf("ERROR: %s\n", lt_last_error(nullptr));
    ctx = nullptr;
  }
}

RendererB200::~RendererB200() {
  forgetScenes();
  if (groupCtx) lt_ctx_destroy(groupCtx);
  if (ctx) lt_ctx_destroy(ctx);
}

static void releaseCached(lt_ctx* ctx, lt_ctx* groupCtx, lt_scene* scene, lt_scene* groupScene) {
  if (scene) lt_scene_release(ctx, scene);
  if (groupScene) lt_scene_release(groupCtx, groupScene);
}

void RendererB200::forgetScenes() {
  for (size_t i = 0; i < sceneCache.size(); i++)
    releaseCached(ctx, groupCtx, sceneCache[i].scene, sceneCache[i].groupScene);
  sceneCache.clear();
}

void RendererB200::renderCommon(const std::string& kernelFilePath, KernelMode kernelMode, const uint64_t blockSize[2],
                                const uint64_t imageDimensions[3], void* pOutputBuffer, uint64_t outputBufferSize,
                                void* pAccelerationStructureExplicit, void* pModel, void* pCamera, void* pNext,
                                const uint64_t* workBlockSize) {
  if (!ctx) {
    printf("ERROR: no B200 context; nothing rendered (there is no CPU fallback)\n");
    return;
  }
  AccelerationStructureExplicit* as = (AccelerationStructureExplicit*)pAccelerationStructureExplicit;
  Model* model = (Model*)pModel;
  Camera* camera = (Camera*)pCamera;
  if (!as || !model || !camera || !pOutputBuffer) {
    printf("ERROR: render properties carry a NULL object\n");
    return;
  }

  int kernel;
  std::map<std::string, int>::iterator kc = kernelCache.find(kernelFilePath);
  if (kc != kernelCache.end()) {
    kernel = kc->second;
  } else {
    std::string resolved = Resource::findResource(kernelFilePath);
    kernel = lt_kernel_from_path(resolved == "INVALID RESOURCE" ? kernelFilePath.c_str() : resolved.c_str());
    kernelCache[kernelFilePath] = kernel;
  }
  // not one of the shipped kernels: a user-written .cu with the reference's CUDA kernel ABI, or a .cl with its
  // OpenCL one, is compiled (once) with NVRTC for sm_100a and launched like the reference launches it; anything
  // else is an error
  int plugin = -1;
  bool isCl = false;
  if (kernel < 0) {
    std::string resolved = Resource::findResource(kernelFilePath);
    bool isCu = resolved.size() > 3 && resolved.compare(resolved.size() - 3, 3, ".cu") == 0;
    isCl = resolved.size() > 3 && resolved.compare(resolved.size() - 3, 3, ".cl") == 0;
    std::map<std::string, int>::iterator pc = pluginCache.find(kernelFilePath);
    if (pc != pluginCache.end()) {
      plugin = pc->second;
    } else if (isCu || isCl) {
      if (lt_plugin_load(ctx, resolved.c_str(), &plugin) != LT_OK) {
        printf("%s\n", lt_last_error(ctx));
        plugin = -1;
      }
      pluginCache[kernelFilePath] = plugin;
    }
    if (plugin < 0) {
      printf("Kernel Error: '%s' is not a kernel this renderer provides (%s)\n", kernelFilePath.c_str(),
             isCu || isCl ? "plug-in compilation failed" : "only the shipped kernels and .cu / .cl plug-ins are supported");
      return;
    }
  }

  // device copy of this (acceleration structure, model) pair: see CachedScene in api.h
  const uint64_t generation = g_retireGeneration.load();
  if (generation != seenRetireGeneration) {  // some object was destroyed: drop what we hold for it
    std::lock_guard<std::mutex> lock(g_retiredMutex);
    for (size_t i = 0; i < sceneCache.size();) {
      if (g_retired.count(sceneCache[i].asId) || g_retired.count(sceneCache[i].modelId)) {
        releaseCached(ctx, groupCtx, sceneCache[i].scene, sceneCache[i].groupScene);
        sceneCache.erase(sceneCache.begin() + i);
      } else {
        i++;
      }
    }
    seenRetireGeneration = generation;
  }
  uint64_t checksum = 14695981039346656037ull;
  checksum = sample(checksum, as->getNodeBuffer(), as->getNodeBufferSize());
  checksum = sample(checksum, as->getOrderedPrimitiveBuffer(), as->getOrderedPrimitiveBufferSize());
  checksum = sample(checksum, model->getMaterialBuffer(), model->getMaterialBufferSize());
  checksum = sample(checksum, as->getLightContainerBuffer(), as->getLightContainerBufferSize());
  RenderExtensionB200* ext = nullptr;
  for (void* p = pNext; p;) {
    RenderExtensionB200* e = (RenderExtensionB200*)p;
    if (e->sType == STRUCTURE_TYPE_RENDER_EXTENSION_B200) {
      ext = e;
      break;
    }
    p = e->pNext;
  }

  // which context renders: the multi-GPU one when the extension asks for several devices (a plug-in splits samples
  // only, so it needs an accumulating call there)
  const uint32_t wantDevices = (ext && ext->deviceCount > 1 && (plugin < 0 || ext->accumulate)) ? ext->deviceCount : 1;
  if (wantDevices > 1 && (groupCtx == nullptr || groupDevices != wantDevices)) {
    groupPluginCache.clear();
    for (size_t i = 0; i < sceneCache.size(); i++)
      if (sceneCache[i].groupScene) {
        lt_scene_release(groupCtx, sceneCache[i].groupScene);
        sceneCache[i].groupScene = nullptr;
      }
    if (groupCtx) lt_ctx_destroy(groupCtx);
    groupCtx = nullptr;
    std::vector<int> devices(wantDevices);
    for (uint32_t d = 0; d < wantDevices; d++) devices[d] = (int)d;
    if (lt_ctx_create_multi(devices.data(), (int)wantDevices, &groupCtx) != LT_OK) {
      printf("ERROR: %s\n", lt_last_error(nullptr));
      groupCtx = nullptr;
      return;
    }
    groupDevices = wantDevices;
  }
  lt_ctx* useCtx = wantDevices > 1 ? groupCtx : ctx;
  if (plugin >= 0 && wantDevices > 1) {  // the same file, loaded on the devices of the group
    std::map<std::string, int>::iterator pc = groupPluginCache.find(kernelFilePath);
    if (pc != groupPluginCache.end()) {
      plugin = pc->second;
    } else {
      if (lt_plugin_load(groupCtx, Resource::findResource(kernelFilePath).c_str(), &plugin) != LT_OK) {
        printf("%s\n", lt_last_error(groupCtx));
        plugin = -1;
      }
      groupPluginCache[kernelFilePath] = plugin;
    }
    if (plugin < 0) {
      printf("Kernel Error: '%s' could not be loaded on %u devices\n", kernelFilePath.c_str(), wantDevices);
      return;
    }
  }
  CachedScene* entry = nullptr;
  for (size_t i = 0; i < sceneCache.size(); i++) {
    CachedScene& c = sceneCache[i];
    if (c.asId != as->getUniqueId() || c.modelId != model->getUniqueId()) continue;
    if (c.checksum == checksum) {
      entry = &c;
      c.lastUse = ++useCounter;
    } else {  // edited in place since the upload
      releaseCached(ctx, groupCtx, c.scene, c.groupScene);
      sceneCache.erase(sceneCache.begin() + i);
    }
    break;
  }
  if (!entry) {
    if (sceneCache.size() >= kMaxScenes) {  // bounded: the least recently used device copy goes
      size_t oldest = 0;
      for (size_t i = 1; i < sceneCache.size(); i++)
        if (sceneCache[i].lastUse < sceneCache[oldest].lastUse) oldest = i;
      releaseCached(ctx, groupCtx, sceneCache[oldest].scene, sceneCache[oldest].groupScene);
      sceneCache.erase(sceneCache.begin() + oldest);
    }
    CachedScene c = {as->getUniqueId(), model->getUniqueId(), checksum, ++useCounter, nullptr, nullptr};
    sceneCache.push_back(c);
    entry = &sceneCache.back();
  }
  lt_scene*& slot = wantDevices > 1 ? entry->groupScene : entry->scene;
  if (!slot) {
    int rc = lt_scene_upload(useCtx, as->getNodeBuffer(), as->getNodeBufferSize(), as->getOrderedPrimitiveBuffer(),
                             as->getOrderedPrimitiveBufferSize(), model->getMaterialBuffer(),
                             model->getMaterialBufferSize(), as->getLightContainerBuffer(),
                             as->getLightContainerBufferSize(), &slot);
    if (rc != LT_OK) {
      printf("ERROR: scene upload failed: %s\n", lt_last_error(useCtx));
      slot = nullptr;
      return;
    }
  }
  lt_scene* scene = slot;

  lt_render_params params;
  memset(&params, 0, sizeof params);
  params.struct_size = sizeof params;
  params.kernel = kernel;
  params.kernel_mode = kernelMode == KERNEL_MODE_TILE ? 1 : 0;
  params.width = (int)imageDimensions[0];
  params.height = (int)imageDimensions[1];
  params.depth = (int)imageDimensions[2];
  params.frames = 1;
  params.frame_stride = 1;
  params.block_x = blockSize ? (int)blockSize[0] : 0;
  params.block_y = blockSize ? (int)blockSize[1] : 0;
  if (ext) {
    params.frames = ext->frames ? (int)ext->frames : 1;
    params.accum_mode = ext->accumulate ? LT_ACCUM_RUNNING_MEAN : LT_ACCUM_NONE;
    params.max_ray_depth = (int)ext->maxRayDepth;
    if (ext->collectStats && wantDevices == 1 && plugin < 0) params.flags |= LT_FLAG_STATS;
    params.split_mode = (int)ext->splitMode;
  }
  const uint32_t views = ext && ext->viewCount >= 2 ? ext->viewCount : 1;
  uint64_t need = sizeof(float) * imageDimensions[0] * imageDimensions[1] * imageDimensions[2] * views;
  if (outputBufferSize < need) {
    printf("ERROR: output buffer is %llu bytes, %u image(s) need %llu\n", (unsigned long long)outputBufferSize, views,
           (unsigned long long)need);
    return;
  }
  std::vector<char> viewCameras;  // the views' 28-byte camera records, back to back
  if (views > 1) {
    if (plugin >= 0) {
      printf("ERROR: RenderExtensionB200::viewCount renders the built-in kernels only, not '%s'\n",
             kernelFilePath.c_str());
      return;
    }
    if (!ext->ppViewCameras) {
      printf("ERROR: RenderExtensionB200::viewCount is %u but ppViewCameras is NULL\n", views);
      return;
    }
    viewCameras.resize((size_t)views * 28);
    for (uint32_t v = 0; v < views; v++) {
      if (!ext->ppViewCameras[v]) {
        printf("ERROR: RenderExtensionB200::ppViewCameras[%u] is NULL\n", v);
        return;
      }
      memcpy(viewCameras.data() + (size_t)v * 28, ext->ppViewCameras[v]->getCameraBuffer(), 28);
    }
  }
  const bool adaptive = ext && ext->adaptiveError > 0.0f;
  if (adaptive) {  // the combinations lt_render_adaptive does not render: nothing is written
    const char* why = !ext->accumulate ? "needs accumulate"
                      : plugin >= 0    ? "renders the built-in kernels only"
                      : views > 1      ? "renders one view"
                      : ext->splitMode == LT_SPLIT_SAMPLES ? "divides the devices' work by rows, not samples"
                                                           : nullptr;
    if (why) {
      printf("ERROR: RenderExtensionB200::adaptiveError %s\n", why);
      return;
    }
  }
  int rc;
  if (adaptive) {
    lt_adaptive_params ap;
    memset(&ap, 0, sizeof ap);
    ap.struct_size = sizeof ap;
    ap.target = ext->adaptiveError;
    ap.round_frames = (int)ext->adaptiveRoundFrames;
    const int round = ap.round_frames ? ap.round_frames : params.frames;
    ap.max_frames = ext->adaptiveMaxFrames ? (int)ext->adaptiveMaxFrames : params.frames + 3 * round;  // INTEGRATION 5d
    lt_adaptive_result res;
    rc = lt_render_adaptive(useCtx, scene, camera->getCameraBuffer(), &params, &ap, (float*)pOutputBuffer,
                            ext->pPixelFrames, &res);
    if (rc == LT_OK) ext->adaptiveRounds = (uint32_t)res.rounds;
  } else if (views > 1)
    rc = lt_render_views(useCtx, scene, viewCameras.data(), (int)views, &params, (float*)pOutputBuffer);
  else if (plugin >= 0 && ext)  // frames, accumulation and devices as the extension asks
    rc = lt_render_plugin_frames(useCtx, scene, camera->getCameraBuffer(), plugin, &params,
                                 isCl && workBlockSize ? (int)workBlockSize[0] : 0,
                                 isCl && workBlockSize ? (int)workBlockSize[1] : 0,
                                 (float*)pOutputBuffer);
  else if (plugin >= 0 && isCl)
    rc = lt_render_plugin_cl(ctx, scene, camera->getCameraBuffer(), plugin, params.kernel_mode, params.width,
                             params.height, params.depth, workBlockSize ? (int)workBlockSize[0] : 0,
                             workBlockSize ? (int)workBlockSize[1] : 0, params.block_x, params.block_y,
                             (float*)pOutputBuffer);
  else if (plugin >= 0)
    rc = lt_render_plugin(ctx, scene, camera->getCameraBuffer(), plugin, params.kernel_mode, params.width,
                          params.height, params.depth, params.block_x, params.block_y, (float*)pOutputBuffer);
  else
    rc = lt_render(useCtx, scene, camera->getCameraBuffer(), &params, (float*)pOutputBuffer);
  if (rc != LT_OK) {
    printf("Kernel Error: %d (%s)\n", rc, lt_last_error(useCtx));
    return;
  }
  if (ext) {
    lt_stats st;
    lt_last_stats(useCtx, &st);
    ext->rays = st.rays;
    ext->nodeTests = st.node_tests;
    ext->triTests = st.tri_tests;
    ext->kernelMilliseconds = st.kernel_ms;
  }
}

RendererCUDA::RendererCUDA() : impl(new RendererB200()) {}
RendererCUDA::~RendererCUDA() { delete impl; }

void RendererCUDA::render(void* pRenderProperties) {
  RenderPropertiesCUDA* p = (RenderPropertiesCUDA*)pRenderProperties;
  if (p->sType != STRUCTURE_TYPE_RENDER_PROPERTIES_CUDA) printf("ERROR: RenderPropertiesCUDA sType\n");
  uint64_t block[2] = {32, 1};
  if (p->threadOrganizationMode == THREAD_ORGANIZATION_MODE_CUSTOM) {
    if (p->threadOrganization.sType != STRUCTURE_TYPE_THREAD_ORGANIZATION_CUDA)
      printf("ERROR: ThreadOrganizationCUDA sType\n");
    block[0] = p->threadOrganization.blockSize[0];
    block[1] = p->threadOrganization.blockSize[1];
  }
  impl->renderCommon(p->kernelFilePath, p->kernelMode, block, p->imageDimensions, p->pOutputBuffer, p->outputBufferSize,
                    p->pAccelerationStructureExplicit, p->pModel, p->pCamera, p->pNext);
}

RendererOpenCL::RendererOpenCL() : impl(new RendererB200()) {}
RendererOpenCL::~RendererOpenCL() { delete impl; }

void RendererOpenCL::render(void* pRenderProperties) {
  RenderPropertiesOpenCL* p = (RenderPropertiesOpenCL*)pRenderProperties;
  if (p->sType != STRUCTURE_TYPE_RENDER_PROPERTIES_OPENCL) printf("ERROR: RenderPropertiesOpenCL sType\n");
  uint64_t block[2] = {0, 0}, workBlock[2] = {0, 0};
  if (p->threadOrganizationMode == THREAD_ORGANIZATION_MODE_CUSTOM) {
    if (p->threadOrganization.sType != STRUCTURE_TYPE_THREAD_ORGANIZATION_OPENCL)
      printf("ERROR: ThreadOrganizationOpenCL sType\n");
    block[0] = p->threadOrganization.threadGroupSize[0];
    block[1] = p->threadOrganization.threadGroupSize[1];
    workBlock[0] = p->threadOrganization.workBlockSize[0];
    workBlock[1] = p->threadOrganization.workBlockSize[1];
  }
  // The reference splits the image into work blocks and drops the remainder (src/opencl/renderer_opencl.cpp:90).
  // The built-in pipelines render the whole image; a user's .cl kernel gets the reference's work blocks (whole image
  // for MAX_FIT), with the remainder written as 0.
  impl->renderCommon(p->kernelFilePath, p->kernelMode, block, p->imageDimensions, p->pOutputBuffer, p->outputBufferSize,
                    p->pAccelerationStructureExplicit, p->pModel, p->pCamera, p->pNext, workBlock);
}
