// lt_capi.cu -- the C-ABI of liblt_b200.so (include/lens_trace_b200.h): context, scene upload with
// device-side re-flatten, render entry points.  No CPU fallback: every compute call needs a CUDA
// device and fails with LT_ERR_NO_DEVICE / LT_ERR_CUDA otherwise.
#include "lens_trace_b200.h"
#include "lt_internal.h"

#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

static thread_local std::string g_error = "";

// Copier threads of lt_internal_download(): they sleep between jobs; a job is `chunks` pieces of a pinned staging
// buffer to be copied to the destination as soon as the owner has published them.
struct LtCopyPool {
  std::vector<std::thread> threads;
  std::mutex m;
  std::condition_variable wake;
  bool quit = false;
  unsigned long long job = 0;  // incremented per job (guards against spurious wake-ups)
  char* dst = nullptr;
  const char* src = nullptr;
  size_t bytes = 0, chunk = 0;
  int chunks = 0;
  std::atomic<int> ready{0}, next{0}, copied{0}, active{0};

  explicit LtCopyPool(int n) {
    for (int i = 0; i < n; i++) threads.emplace_back([this]() { run(); });
  }
  ~LtCopyPool() {
    {
      std::lock_guard<std::mutex> lock(m);
      quit = true;
    }
    wake.notify_all();
    for (std::thread& t : threads) t.join();
  }
  void copy_some() {
    while (true) {
      const int c = next.fetch_add(1);
      if (c >= chunks) return;
      while (ready.load(std::memory_order_acquire) <= c) std::this_thread::yield();
      const size_t off = (size_t)c * chunk, n = bytes - off < chunk ? bytes - off : chunk;
      memcpy(dst + off, src + off, n);
      copied.fetch_add(1, std::memory_order_release);
    }
  }
  void run() {
    unsigned long long seen = 0;
    while (true) {
      {
        std::unique_lock<std::mutex> lock(m);
        wake.wait(lock, [&]() { return quit || job != seen; });
        if (quit) return;
        seen = job;
        active++;  // under the lock: begin() never changes the job while a copier is inside copy_some()
      }
      copy_some();
      active.fetch_sub(1, std::memory_order_release);
    }
  }
  void begin(char* d, const char* s, size_t b, size_t c, int n) {
    {
      std::unique_lock<std::mutex> lock(m);
      while (active.load(std::memory_order_acquire) != 0) {  // a straggler of the previous job is still leaving
        lock.unlock();
        std::this_thread::yield();
        lock.lock();
      }
      dst = d; src = s; bytes = b; chunk = c; chunks = n;
      ready.store(0);
      next.store(0);
      copied.store(0);
      job++;
    }
    wake.notify_all();
  }
  void publish(int n) { ready.store(n, std::memory_order_release); }
  void finish() {  // the owner copies along, then waits for the stragglers
    copy_some();
    while (copied.load(std::memory_order_acquire) < chunks) std::this_thread::yield();
  }
};


static int fail(lt_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->error = msg;
  g_error = msg;
  return code;
}
int lt_internal_fail(lt_ctx* ctx, int code, const std::string& msg) { return fail(ctx, code, msg); }

#define CK(call)                                                                                     \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess)                                                                           \
      return fail(ctx, LT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));             \
  } while (0)

int lt_internal_ctx_device(const lt_ctx* ctx) { return ctx->device; }

// Host primitives of an upload, a device build or a refit: every material index in [0, matCount) and, with `finite`,
// every vertex coordinate finite.  `w` starts the error message.
static int check_prims(lt_ctx* ctx, const RefPrim* prims, uint64_t n, uint64_t matCount, bool finite,
                       const std::string& w) {
  for (uint64_t i = 0; i < n; i++)
    if (prims[i].materialIndex < 0 || (uint64_t)prims[i].materialIndex >= matCount)
      return fail(ctx, LT_ERR_INVALID, w + "primitive materialIndex out of range");
  if (finite)
    for (uint64_t i = 0; i < n; i++)
      for (int k = 0; k < 3; k++)
        if (!std::isfinite(prims[i].a[k]) || !std::isfinite(prims[i].b[k]) || !std::isfinite(prims[i].c[k]))
          return fail(ctx, LT_ERR_INVALID, w + "non-finite vertex coordinate");
  return LT_OK;
}

extern "C" int lt_api_version(void) { return LT_API_VERSION; }

extern "C" const char* lt_last_error(const lt_ctx* ctx) { return ctx ? ctx->error.c_str() : g_error.c_str(); }

extern "C" int lt_ctx_create(int device_ordinal, lt_ctx** out_ctx) {
  lt_ctx* ctx = nullptr;
  if (!out_ctx) return fail(nullptr, LT_ERR_INVALID, "lt_ctx_create: out_ctx is NULL");
  *out_ctx = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return fail(nullptr, LT_ERR_NO_DEVICE,
                std::string("lt_ctx_create: no CUDA device (") + cudaGetErrorString(e) +
                    "); liblt_b200 has no CPU fallback");
  }
  if (device_ordinal < 0 || device_ordinal >= n)
    return fail(nullptr, LT_ERR_INVALID, "lt_ctx_create: device ordinal out of range");
  CK(cudaSetDevice(device_ordinal));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device_ordinal));
  if (prop.major < 10)
    return fail(nullptr, LT_ERR_NO_DEVICE, "lt_ctx_create: device is not sm_100 (kernels are built for sm_100a only)");
  ctx = new lt_ctx();
  ctx->device = device_ordinal;
  ctx->stats.sm_count = prop.multiProcessorCount;
  ctx->totalMem = prop.totalGlobalMem;
  cudaError_t e2 = ctx->ownStream.create();
  ctx->stream = ctx->ownStream.get();
  if (e2 == cudaSuccess) e2 = ctx->ev.grow(2, cudaEventDefault);
  if (e2 == cudaSuccess) e2 = ctx->dCounters.grow(1);
  if (e2 == cudaSuccess) e2 = ctx->dWork.grow(64);  // 256 bytes
  if (e2 == cudaSuccess) e2 = ctx->wfExtra.create();
  if (e2 == cudaSuccess) e2 = ctx->wfEvents.grow(3, cudaEventDisableTiming);
  if (e2 != cudaSuccess) {
    std::string m = std::string("lt_ctx_create: ") + cudaGetErrorString(e2);
    delete ctx;
    return fail(nullptr, LT_ERR_CUDA, m);
  }
  *out_ctx = ctx;
  return LT_OK;
}

lt_ctx::lt_ctx() = default;

// A single-GPU context waits for its streams (the caller's one included) before its members release what they hold.
// A group context has no stream of its own and touches no device: lt_multi_destroy has released its members.
lt_ctx::~lt_ctx() {
  if (!ownStream.get()) return;
  cudaSetDevice(device);
  cudaStreamSynchronize(stream);
  if (wfExtra.get()) cudaStreamSynchronize(wfExtra.get());
  for (LtPlugin* p : plugins) lt_plugin_free(p);
}

extern "C" void lt_ctx_destroy(lt_ctx* ctx) {
  if (ctx && ctx->group) lt_multi_destroy(ctx);
  delete ctx;
}

extern "C" int lt_ctx_set_stream(lt_ctx* ctx, void* cuda_stream) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_ctx_set_stream: ctx is NULL");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_ctx_set_stream: a multi-GPU context renders on its own per-device streams");
  ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->ownStream.get();
  return LT_OK;
}

extern "C" void lt_scene_release(lt_ctx* ctx, lt_scene* s) {
  if (!s) return;
  if (!s->parts.empty()) {
    lt_multi_scene_release(ctx, s);
    return;
  }
  if (ctx) {
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
  }
  delete s;
}

extern "C" int lt_debug_scene_traversal_tree(const lt_scene* scene) {
  if (!scene) return fail(nullptr, LT_ERR_INVALID, "lt_debug_scene_traversal_tree: scene is NULL");
  if (!scene->parts.empty()) scene = scene->parts[0];
  return scene->dev.rank != nullptr ? 1 : 0;
}

// Where trav_begin_threaded starts the rays that may use pruned records: the pruned copies of dThread, or (no host-built
// copies, or `full`) the full copies, which are also the layout of the device-built dThreadBig.
static void set_pruned_copies(lt_scene* s, bool full) {
  LtSceneDev& d = s->dev;
  const bool pruned = s->dThread.get() != nullptr && !full;
  d.prunedBase = pruned ? 8 * d.nodeCount : 0;
  d.prunedStride = pruned ? s->threadStride : d.nodeCount;
}

extern "C" int lt_debug_scene_full_threaded(lt_scene* scene, int full) {
  if (!scene || !scene->parts.empty()) return fail(nullptr, LT_ERR_INVALID, "lt_debug_scene_full_threaded: bad scene");
  set_pruned_copies(scene, full != 0);
  return LT_OK;
}

// The buffers derived from dNodes and dPrims, written into the scene's allocations: the 64-byte child-pair nodes and
// 48-byte triangles (re-flatten through the inner-node ranks dInnerRank), the threaded copies the scene keeps
// (`copies`: built on the host for small trees, the one pass that may grow dThread or add dRank, or on the device for
// large ones), and the launch state.  Upload and refit share it, so a refitted scene is what an upload of its buffers
// makes.  ev[0] must already be recorded on the stream; records ev[1] and sets upload_ms.
static cudaError_t derive_scene(lt_ctx* ctx, lt_scene* s, const int* dInnerRank, LtTree copies, const RefNode& root) {
  LtSceneDev& d = s->dev;
  const int nNodes = d.nodeCount, nPrims = d.primCount;
  cudaError_t e = cudaSuccess;
  auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  cudaStream_t st = ctx->stream;
  lt_launch_reflatten(s->dNodes.get(), nNodes, s->dPrims.get(), nPrims, dInnerRank, s->dWide.get(), s->dTris.get(), st);
  A(cudaGetLastError());
  std::vector<int> hRank;
  if (e == cudaSuccess && copies == LT_TREE_HOST_THREADED) {
    std::vector<RefNode> hNodes((size_t)nNodes);
    std::vector<LtThreadNode> hThread;
    A(cudaMemcpyAsync(hNodes.data(), s->dNodes.get(), sizeof(RefNode) * (size_t)nNodes, cudaMemcpyDeviceToHost, st));
    A(cudaStreamSynchronize(st));
    if (e == cudaSuccess) {
      s->threadStride = lt_build_threaded(hNodes.data(), nNodes, nPrims, hThread, hRank);
      A(s->dThread.grow(hThread.size()));  // the pruned copies' size follows the boxes
      A(cudaMemcpyAsync(s->dThread.get(), hThread.data(), sizeof(LtThreadNode) * hThread.size(), cudaMemcpyHostToDevice,
                        st));
      if (!hRank.empty()) {
        A(s->dRank.grow(hRank.size()));
        A(cudaMemcpyAsync(s->dRank.get(), hRank.data(), sizeof(int) * hRank.size(), cudaMemcpyHostToDevice, st));
      }
      A(cudaStreamSynchronize(st));  // hThread and hRank are pageable and go out of scope
    }
  }
  // large trees: the threaded copies are built on the device and used by coherent-ray launches only (plan_tree)
  if (e == cudaSuccess && copies == LT_TREE_DEVICE_THREADED) {
    if (s->dThreadBig.grow(8 * (size_t)nNodes) != cudaSuccess)
      cudaGetLastError();  // no memory for the copies: the stack traversal serves every launch
    if (s->dThreadBig.get()) {
      lt_launch_build_threaded(s->dNodes.get(), nNodes, s->dThreadBig.get(), st);
      A(cudaGetLastError());
    }
  }
  A(cudaEventRecord(ctx->ev[1], st));
  A(cudaStreamSynchronize(st));
  if (e != cudaSuccess) return e;
  cudaEventElapsedTime(&ctx->stats.upload_ms, ctx->ev[0], ctx->ev[1]);
  d.wnodes = s->dWide.get();
  d.tris = s->dTris.get();
  for (int k = 0; k < 3; k++) {
    d.rootMin[k] = root.boundsMin[k];
    d.rootMax[k] = root.boundsMax[k];
  }
  d.rootRef = root.primitiveCount > 0 ? ~root.offset : 0;  // inner root is wide node 0
  d.rootCount = root.primitiveCount;
  d.tnodes = s->dThread.get();
  d.rank = hRank.empty() ? nullptr : s->dRank.get();
  set_pruned_copies(s, false);
  return cudaSuccess;
}

// Allocates the re-flattened buffers, derives them (derive_scene) and fills the device-side scene descriptor.  ev[0]
// must already be recorded on the stream; on failure the scene is released.
static int finish_scene(lt_ctx* ctx, lt_scene* s, int nNodes, int nPrims, int nMats, const RefNode& root,
                        int stackDepth, const char* who) {
  LtBuf<int> flags, rank;
  LtBuf<char> temp;
  int nInner = (nNodes - 1) / 2;  // a full binary tree with one primitive slot per leaf
  if (nNodes == 1) nInner = 0;
  size_t tempBytes = lt_scan_temp_bytes(nNodes);
  LtSceneDev& d = s->dev;
  d.prims = s->dPrims.get();
  d.mats = s->dMats.get();
  d.lights = s->dLights.get();
  d.stackDepth = stackDepth;
  d.nodeCount = nNodes;
  d.primCount = nPrims;
  d.matCount = nMats;
  cudaError_t e = cudaSuccess;
  auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  cudaStream_t st = ctx->stream;
  A(s->dWide.grow(nInner > 0 ? nInner : 1));
  A(s->dTris.grow(nPrims));
  A(flags.grow(nNodes));
  A(rank.grow(nNodes));
  A(temp.grow(tempBytes ? tempBytes : 16));
  if (e == cudaSuccess) {
    lt_launch_inner_flags(s->dNodes.get(), nNodes, flags.get(), st);
    lt_launch_exclusive_scan(temp.get(), tempBytes, flags.get(), rank.get(), nNodes, st);
    A(cudaGetLastError());
  }
  if (e == cudaSuccess)
    A(derive_scene(ctx, s, rank.get(), lt_plan_threaded_copies(nNodes, ctx->totalMem, ctx->limits), root));
  cudaStreamSynchronize(st);
  if (e != cudaSuccess) {
    lt_scene_release(ctx, s);
    return fail(ctx, LT_ERR_CUDA, std::string(who) + ": " + cudaGetErrorString(e));
  }
  return LT_OK;
}

// The device builders (lt_bvh.cu) behind lt_scene_build_lbvh and lt_scene_build_ploc: argument checks, upload of the
// inputs, build, depth check and re-flatten.  `who` names the entry point in error messages.
static int build_scene_on_device(lt_ctx* ctx, LtBvhBuilder builder, const char* who, const void* primitives,
                                 uint64_t primitive_bytes, const void* materials, uint64_t material_bytes,
                                 lt_scene** out_scene) {
  const std::string w = std::string(who) + ": ";
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, w + "ctx is NULL");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, w + "build on a single-GPU context, download, and upload to the multi-GPU context");
  if (!out_scene || !primitives || !materials) return fail(ctx, LT_ERR_INVALID, w + "NULL argument");
  *out_scene = nullptr;
  if (primitive_bytes == 0 || primitive_bytes % sizeof(RefPrim) || material_bytes == 0 ||
      material_bytes % sizeof(RefMaterial))
    return fail(ctx, LT_ERR_INVALID, w + "buffer size is not a multiple of the reference record size");
  uint64_t nPrims = primitive_bytes / sizeof(RefPrim), nMats = material_bytes / sizeof(RefMaterial);
  if (nPrims < 2) return fail(ctx, LT_ERR_UNSUPPORTED, w + "needs at least two primitives");
  if (nPrims > 0x3fffffffull) return fail(ctx, LT_ERR_INVALID, w + "too many primitives");
  // PLOC compares box areas; its progress argument needs every area to be a number
  if (int rc = check_prims(ctx, (const RefPrim*)primitives, nPrims, nMats, builder == LT_BVH_PLOC, w)) return rc;
  CK(cudaSetDevice(ctx->device));
  int n = (int)nPrims, nNodes = 2 * n - 1;
  lt_scene* s = new lt_scene();
  cudaError_t e = cudaSuccess;
  auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  A(s->dNodes.grow(nNodes));
  A(s->dPrims.grow(nPrims));
  A(s->dMats.grow(nMats));
  A(s->dLights.grow(1));
  int maxDepth = 0, launches = -1;
  RefNode root;
  memset(&root, 0, sizeof root);
  {  // the builder's input and scratch go before the re-flatten allocates
    LtBuf<RefPrim> input;
    LtBuf<char> scratch;
    A(input.grow(nPrims));
    A(scratch.grow(lt_bvh_scratch_bytes(n, builder)));
    cudaStream_t st = ctx->stream;
    A(cudaEventRecord(ctx->ev[0], st));
    A(cudaMemcpyAsync(input.get(), primitives, primitive_bytes, cudaMemcpyHostToDevice, st));
    A(cudaMemcpyAsync(s->dMats.get(), materials, material_bytes, cudaMemcpyHostToDevice, st));
    if (e == cudaSuccess)
      launches = lt_launch_bvh_build(builder, input.get(), n, s->dMats.get(), (int)nMats, s->dNodes.get(), s->dPrims.get(),
                                     s->dLights.get(), scratch.get(), scratch.count(), &maxDepth, st);
    if (e == cudaSuccess && launches >= 0) A(cudaMemcpy(&root, s->dNodes.get(), sizeof root, cudaMemcpyDeviceToHost));
  }
  if (e != cudaSuccess || launches < 0) {
    lt_scene_release(ctx, s);
    return fail(ctx, LT_ERR_CUDA, w + (e != cudaSuccess ? cudaGetErrorString(e) : "build failed"));
  }
  if (maxDepth > 64) {
    lt_scene_release(ctx, s);
    return fail(ctx, LT_ERR_UNSUPPORTED, w + "tree deeper than 64 (too many coincident centroids); use the host builder");
  }
  int rc = finish_scene(ctx, s, nNodes, n, (int)nMats, root, maxDepth, who);
  if (rc != LT_OK) return rc;
  *out_scene = s;
  return LT_OK;
}

extern "C" int lt_scene_build_lbvh(lt_ctx* ctx, const void* primitives, uint64_t primitive_bytes, const void* materials,
                                   uint64_t material_bytes, lt_scene** out_scene) {
  return build_scene_on_device(ctx, LT_BVH_LBVH, "lt_scene_build_lbvh", primitives, primitive_bytes, materials,
                               material_bytes, out_scene);
}

extern "C" int lt_scene_build_ploc(lt_ctx* ctx, const void* primitives, uint64_t primitive_bytes, const void* materials,
                                   uint64_t material_bytes, lt_scene** out_scene) {
  return build_scene_on_device(ctx, LT_BVH_PLOC, "lt_scene_build_ploc", primitives, primitive_bytes, materials,
                               material_bytes, out_scene);
}

extern "C" int lt_scene_download(lt_ctx* ctx, lt_scene* scene, void* nodes, uint64_t node_bytes, void* primitives,
                                 uint64_t primitive_bytes, void* light_container) {
  if (!ctx || !scene) return fail(ctx, LT_ERR_INVALID, "lt_scene_download: NULL argument");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_scene_download: not available on a multi-GPU context");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  if (nodes) {
    if (node_bytes != sizeof(RefNode) * (uint64_t)scene->dev.nodeCount) return fail(ctx, LT_ERR_INVALID, "lt_scene_download: node_bytes mismatch");
    CK(cudaMemcpy(nodes, scene->dNodes.get(), node_bytes, cudaMemcpyDeviceToHost));
  }
  if (primitives) {
    if (primitive_bytes != sizeof(RefPrim) * (uint64_t)scene->dev.primCount) return fail(ctx, LT_ERR_INVALID, "lt_scene_download: primitive_bytes mismatch");
    CK(cudaMemcpy(primitives, scene->dPrims.get(), primitive_bytes, cudaMemcpyDeviceToHost));
  }
  if (light_container) CK(cudaMemcpy(light_container, scene->dLights.get(), sizeof(RefLights), cudaMemcpyDeviceToHost));
  return LT_OK;
}

extern "C" int lt_scene_info(const lt_scene* scene, uint64_t* node_count, uint64_t* primitive_count, int32_t* stack_depth) {
  if (!scene) return LT_ERR_INVALID;
  if (!scene->parts.empty()) scene = scene->parts[0];
  if (node_count) *node_count = (uint64_t)scene->dev.nodeCount;
  if (primitive_count) *primitive_count = (uint64_t)scene->dev.primCount;
  if (stack_depth) *stack_depth = scene->dev.stackDepth;
  return LT_OK;
}

extern "C" int lt_scene_upload(lt_ctx* ctx, const void* nodes, uint64_t node_bytes, const void* primitives,
                               uint64_t primitive_bytes, const void* materials, uint64_t material_bytes,
                               const void* light_container, uint64_t light_bytes, lt_scene** out_scene) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_scene_upload: ctx is NULL");
  if (!out_scene) return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: out_scene is NULL");
  if (ctx->group)
    return lt_multi_scene_upload(ctx, nodes, node_bytes, primitives, primitive_bytes, materials, material_bytes,
                                 light_container, light_bytes, out_scene);
  *out_scene = nullptr;
  if (!nodes || !primitives || !materials || !light_container)
    return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: NULL buffer");
  if (node_bytes == 0 || node_bytes % sizeof(RefNode) || primitive_bytes == 0 ||
      primitive_bytes % sizeof(RefPrim) || material_bytes % sizeof(RefMaterial) ||
      light_bytes != sizeof(RefLights))
    return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: buffer size is not a multiple of the reference record size");
  uint64_t nNodes = node_bytes / sizeof(RefNode), nPrims = primitive_bytes / sizeof(RefPrim);
  uint64_t nMats = material_bytes / sizeof(RefMaterial);
  if (nNodes > 0x7fffffffull || nPrims > 0x7ffffffeull)
    return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: too many nodes/primitives for 32-bit indices");
  const RefNode* hNodes = (const RefNode*)nodes;
  const RefPrim* hPrims = (const RefPrim*)primitives;
  const RefLights* hLights = (const RefLights*)light_container;
  int stackDepth = 0;
  std::string why;
  if (lt_validate_tree(hNodes, (int)nNodes, (int)nPrims, &stackDepth, &why) != 0)
    return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: " + why);
  if (stackDepth > 64)
    return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: tree deeper than 64 (the reference's stack, basic.cu:162)");
  if (int rc = check_prims(ctx, hPrims, nPrims, nMats, false, "lt_scene_upload: ")) return rc;
  if (hLights->count > 64) return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: light count > 64");
  for (uint32_t i = 0; i < 64; i++)
    if (hLights->primitives[i] >= nPrims)
      return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: light primitive index out of range");

  CK(cudaSetDevice(ctx->device));
  lt_scene* s = new lt_scene();
  cudaError_t e = cudaSuccess;
  auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  A(s->dNodes.grow(nNodes));
  A(s->dPrims.grow(nPrims));
  A(s->dMats.grow(nMats ? nMats : 1));
  A(s->dLights.grow(1));
  cudaStream_t st = ctx->stream;
  A(cudaEventRecord(ctx->ev[0], st));
  A(cudaMemcpyAsync(s->dNodes.get(), nodes, node_bytes, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(s->dPrims.get(), primitives, primitive_bytes, cudaMemcpyHostToDevice, st));
  if (material_bytes) A(cudaMemcpyAsync(s->dMats.get(), materials, material_bytes, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(s->dLights.get(), light_container, sizeof(RefLights), cudaMemcpyHostToDevice, st));
  if (e != cudaSuccess) {
    lt_scene_release(ctx, s);
    return fail(ctx, LT_ERR_CUDA, std::string("lt_scene_upload: ") + cudaGetErrorString(e));
  }
  int rc = finish_scene(ctx, s, (int)nNodes, (int)nPrims, (int)nMats, hNodes[0], stackDepth, "lt_scene_upload");
  if (rc != LT_OK) return rc;
  *out_scene = s;
  return LT_OK;
}

static int check_params(lt_ctx* ctx, const lt_scene* scene, const void* camera28, const lt_render_params* p,
                        LtLaunch* L) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_render: ctx is NULL");
  if (!scene || !camera28 || !p) return fail(ctx, LT_ERR_INVALID, "lt_render: NULL argument");
  if (int rc = lt_params_to_launch(ctx, p, L)) return rc;
  memcpy(&L->cam, camera28, sizeof(RefCamera));
  return LT_OK;
}

static LtSceneFacts scene_facts(const lt_scene* s) {
  return {s->dev.nodeCount, s->dev.stackDepth,
          s->dThread.get() ? LT_TREE_HOST_THREADED : (s->dThreadBig.get() ? LT_TREE_DEVICE_THREADED : LT_TREE_CHILD_PAIR)};
}

// the scene as the plan's kernels see it: tnodes = the plan's threaded copies, NULL for the stack traversal
static LtSceneDev scene_for_plan(const lt_scene* s, const LtPlan& plan) {
  LtSceneDev d = s->dev;
  d.tnodes = plan.tree == LT_TREE_HOST_THREADED ? s->dThread.get()
             : plan.tree == LT_TREE_DEVICE_THREADED ? s->dThreadBig.get() : nullptr;
  return d;
}

// Is p memory of the context's device (device or managed memory), aligned to `align` bytes?  Fails with LT_ERR_INVALID
// naming `what` otherwise.
static int check_device_memory(lt_ctx* ctx, const void* p, size_t align, const std::string& w, const char* what) {
  cudaPointerAttributes pa;
  if (cudaPointerGetAttributes(&pa, p) != cudaSuccess ||
      (pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged) || pa.device != ctx->device) {
    cudaGetLastError();
    return fail(ctx, LT_ERR_INVALID, w + what + " is not device memory of the context's device");
  }
  if ((uintptr_t)p % align) return fail(ctx, LT_ERR_INVALID, w + what + " is not " + std::to_string(align) + "-byte aligned");
  return LT_OK;
}

// Both forms of lt_scene_refit, after the checks that need no device: `src` holds the scene's primitive count of new
// primitives in host memory, already checked, or in device memory (onDevice), checked here by a kernel.  Nothing of
// the scene is written before every check has passed.  The topology's parents and inner-node ranks are derived on the
// first refit that passes them, and kept.
static int refit_scene(lt_ctx* ctx, lt_scene* s, const void* src, bool onDevice, const char* who) {
  const std::string w = std::string(who) + ": ";
  CK(cudaSetDevice(ctx->device));
  const int n = s->dev.nodeCount, nPrims = s->dev.primCount;
  cudaStream_t st = ctx->stream;
  if (onDevice)
    if (int rc = check_device_memory(ctx, src, alignof(RefPrim), w, "device_primitives")) return rc;
  // The upload checks only a leaf's first primitive (the reference's leaves test no other, SURVEY H1); the refit reads
  // all of them, so every leaf's range must lie in the primitive buffer.
  if (s->refitLeaves == 0) {
    std::vector<RefNode> hNodes((size_t)n);
    CK(cudaMemcpyAsync(hNodes.data(), s->dNodes.get(), sizeof(RefNode) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    s->refitLeaves = 1;
    for (const RefNode& r : hNodes)
      if (r.primitiveCount > 0 && (long long)r.offset + r.primitiveCount > nPrims) s->refitLeaves = -1;
  }
  if (s->refitLeaves < 0)
    return fail(ctx, LT_ERR_INVALID, w + "a leaf's primitives run past the primitive buffer: the scene cannot be refitted");
  CK(s->dRefit.grow(3 * (size_t)n + 1));
  int *parent = s->dRefit.get(), *flags = parent + n, *rank = flags + n, *bad = rank + n;
  if (onDevice) {
    lt_launch_check_prims((const RefPrim*)src, nPrims, s->dev.matCount, bad, st);
    int why = 0;
    CK(cudaMemcpyAsync(&why, bad, sizeof why, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (why & 1) return fail(ctx, LT_ERR_INVALID, w + "primitive materialIndex out of range");
    if (why) return fail(ctx, LT_ERR_INVALID, w + "non-finite vertex coordinate");
  }
  if (!s->refitDerived) {  // the inner-node ranks as the upload computes them, with the arrival flags as the scan's input
    // Host-built copies: room for the largest pruned copies (8 n records besides the full ones) and for the tie-break
    // table, so that no later refit allocates whatever the boxes do to the traversal tree.
    if (s->dThread.get() && s->dThread.count() < 16 * (size_t)n) {
      CK(cudaStreamSynchronize(st));
      s->dev.tnodes = nullptr;
      CK(s->dThread.grow(16 * (size_t)n));
    }
    if (s->dThread.get()) CK(s->dRank.grow(8 * (size_t)nPrims));
    LtBuf<char> temp;
    const size_t tempBytes = lt_scan_temp_bytes(n);
    CK(temp.grow(tempBytes ? tempBytes : 16));
    lt_launch_refit_parents(s->dNodes.get(), n, parent, st);
    lt_launch_inner_flags(s->dNodes.get(), n, flags, st);
    lt_launch_exclusive_scan(temp.get(), tempBytes, flags, rank, n, st);
    CK(cudaStreamSynchronize(st));
    s->refitDerived = true;
  }
  CK(cudaEventRecord(ctx->ev[0], st));
  CK(cudaMemcpyAsync(s->dPrims.get(), src, sizeof(RefPrim) * (size_t)nPrims,
                     onDevice ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  lt_launch_refit(s->dNodes.get(), n, s->dPrims.get(), parent, flags, st);
  CK(cudaGetLastError());
  RefNode root;
  CK(cudaMemcpyAsync(&root, s->dNodes.get(), sizeof root, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));  // the root box travels in the launch state
  const cudaError_t e = derive_scene(ctx, s, rank, scene_facts(s).copies, root);
  if (e != cudaSuccess) return fail(ctx, LT_ERR_CUDA, w + cudaGetErrorString(e));
  return LT_OK;
}
int lt_internal_refit(lt_ctx* ctx, lt_scene* scene, const void* primitives) {
  return refit_scene(ctx, scene, primitives, false, "lt_scene_refit");
}

// the checks of both forms that need no device; prims: host primitives to check, or NULL
static int refit_args(lt_ctx* ctx, const lt_scene* scene, const void* prims, uint64_t primitive_bytes,
                      const RefPrim* hostPrims, const char* who) {
  const std::string w = std::string(who) + ": ";
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, w + "ctx is NULL");
  if (!scene || !prims) return fail(ctx, LT_ERR_INVALID, w + "NULL argument");
  if (!scene->parts.empty() != (ctx->group != nullptr))
    return fail(ctx, LT_ERR_INVALID, w + "the scene was not uploaded to this context");
  const lt_scene* one = scene->parts.empty() ? scene : scene->parts[0];
  const uint64_t nPrims = (uint64_t)one->dev.primCount;
  if (primitive_bytes != sizeof(RefPrim) * nPrims)
    return fail(ctx, LT_ERR_INVALID, w + "primitive_bytes is not the scene's primitive count x 76");
  return hostPrims ? check_prims(ctx, hostPrims, nPrims, (uint64_t)one->dev.matCount, true, w) : LT_OK;
}

extern "C" int lt_scene_refit(lt_ctx* ctx, lt_scene* scene, const void* primitives, uint64_t primitive_bytes) {
  const char* who = "lt_scene_refit";
  if (int rc = refit_args(ctx, scene, primitives, primitive_bytes, (const RefPrim*)primitives, who)) return rc;
  if (ctx->group) return lt_multi_scene_refit(ctx, scene, primitives);
  return refit_scene(ctx, scene, primitives, false, who);
}

extern "C" int lt_scene_refit_device(lt_ctx* ctx, lt_scene* scene, const void* device_primitives,
                                     uint64_t primitive_bytes) {
  const char* who = "lt_scene_refit_device";
  if (ctx && ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, std::string(who) + ": single-GPU contexts only");
  if (int rc = refit_args(ctx, scene, device_primitives, primitive_bytes, nullptr, who)) return rc;
  return refit_scene(ctx, scene, device_primitives, true, who);
}

static uint64_t scene_bytes(const lt_scene* s) {
  uint64_t bytes = s->dNodes.bytes() + s->dPrims.bytes() + s->dMats.bytes() + s->dLights.bytes() + s->dWide.bytes() +
                   s->dTris.bytes() + s->dThread.bytes() + s->dRank.bytes() + s->dThreadBig.bytes() + s->dRefit.bytes();
  for (const lt_scene* p : s->parts) bytes += scene_bytes(p);
  return bytes;
}

extern "C" int lt_debug_scene_bytes(const lt_scene* scene, uint64_t* out_bytes) {
  if (!scene || !out_bytes) return fail(nullptr, LT_ERR_INVALID, "lt_debug_scene_bytes: NULL argument");
  *out_bytes = scene_bytes(scene);
  return LT_OK;
}

extern "C" int lt_debug_ctx_limits(lt_ctx* ctx, int threaded_max_nodes, int stream_min_nodes) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_debug_ctx_limits: ctx is NULL");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_debug_ctx_limits: not available on a multi-GPU context");
  if (threaded_max_nodes < 0 || stream_min_nodes < 0) return fail(ctx, LT_ERR_INVALID, "lt_debug_ctx_limits: negative limit");
  ctx->limits.threadedMaxNodes = threaded_max_nodes;
  ctx->limits.streamMinNodes = stream_min_nodes;
  return LT_OK;
}

void lt_internal_stats_start(lt_ctx* ctx) {
  lt_stats s = {};
  s.sm_count = ctx->stats.sm_count;
  s.upload_ms = ctx->stats.upload_ms;
  ctx->stats = s;
}

// what one call adds to a sum of calls: counters, launches and per-kernel times (kernel_ms is the caller's to time)
static void stats_add(lt_stats* sum, const lt_stats& s) {
  sum->rays += s.rays;
  sum->node_tests += s.node_tests;
  sum->tri_tests += s.tri_tests;
  sum->kernel_launches += s.kernel_launches;
  sum->trace_ms += s.trace_ms;
  sum->trace_launches += s.trace_launches;
  sum->shade_ms += s.shade_ms;
  sum->primary_shade_ms += s.primary_shade_ms;
  sum->accumulate_ms += s.accumulate_ms;
  sum->shade_launches += s.shade_launches;
}

int lt_internal_ensure_out(lt_ctx* ctx, size_t floats) {
  if (ctx->dOut.count() >= floats) return LT_OK;
  CK(ctx->dOut.grow(floats));
  const cudaError_t e = cudaMemsetAsync(ctx->dOut.get(), 0, floats * sizeof(float), ctx->stream);
  if (e != cudaSuccess) ctx->dOut.reset();  // not zeroed: the next call allocates it anew
  CK(e);
  return LT_OK;
}

// cams: the cameras of a call of several views (viewCount >= 2, view v into dOut + v * W * H * depth); nullptr: L.cam
// list: the listed pixels of a masked call (lt_render_masked_device), or nullptr
static int render_common(lt_ctx* ctx, lt_scene* scene, const LtLaunch& L, float* dOut, bool sync,
                         const RefCamera* cams = nullptr, int viewCount = 1, const LtList* list = nullptr) {
  lt_internal_stats_start(ctx);
  CK(cudaSetDevice(ctx->device));
  const long long listed = list ? list->count : -1;
  LtPlan plan =
      lt_plan_render(L, scene_facts(scene), ctx->totalMem, ctx->stats.sm_count, ctx->limits, viewCount, listed);
  if (plan.error != LT_OK) return fail(ctx, plan.error, plan.message);
  const bool stats = plan.stats;
  if (stats) CK(cudaMemsetAsync(ctx->dCounters.get(), 0, sizeof(LtCounters), ctx->stream));
  if (plan.pipeline == LT_PIPE_WAVEFRONT && ctx->wfWorkspace.grow(plan.workspaceBytes) != cudaSuccess) {
    cudaGetLastError();
    if (plan.forced) return fail(ctx, LT_ERR_CUDA, "lt_render: cannot allocate the wavefront workspace");
    // not a fallback to other arithmetic: the megakernel is the same path per pixel
    LtLaunch mega = L;
    mega.flags |= LT_FLAG_MEGAKERNEL;
    plan = lt_plan_render(mega, scene_facts(scene), ctx->totalMem, ctx->stats.sm_count, ctx->limits, viewCount, listed);
  }
  const bool wavefront = plan.pipeline == LT_PIPE_WAVEFRONT;
  const int kMaxTracePairs = 8192;
  int tracePairs = 0;
  bool timeTrace = wavefront && (sync || stats);
  if (timeTrace) {
    CK(ctx->traceEvents.grow(2 * kMaxTracePairs, cudaEventDefault));
    ctx->pairKinds.resize(kMaxTracePairs);
  }
  // per-kernel times are only defined when one kernel runs at a time (LT_FLAG_SERIAL / stats launches)
  const bool timeKinds = timeTrace && plan.streams == 1;
  const LtSceneDev sc = scene_for_plan(scene, plan);
  LtViews views = {viewCount, cams, nullptr};
  if (wavefront && viewCount > 1) {  // the frameCount of every (view, frame) pair, for the shade kernels
    const size_t n = (size_t)viewCount * L.frames;
    std::vector<unsigned> fc(n);
    for (int v = 0; v < viewCount; v++)
      for (int f = 0; f < L.frames; f++) fc[(size_t)v * L.frames + f] = cams[v].frameCount + (unsigned)f * L.frameStride;
    CK(ctx->dViewFrameCounts.grow(n));
    // pageable source: staged before the call returns, so fc may go
    CK(cudaMemcpyAsync(ctx->dViewFrameCounts.get(), fc.data(), n * sizeof(unsigned), cudaMemcpyHostToDevice,
                       ctx->stream));
    views.dFrameCounts = ctx->dViewFrameCounts.get();
  }
  CK(cudaEventRecord(ctx->ev[0], ctx->stream));
  int launches = 0;
  if (wavefront) {
    const LtWfAux aux = {ctx->wfExtra.get(), ctx->wfEvents[0], {ctx->wfEvents[1], ctx->wfEvents[2]}};
    launches = lt_launch_render_wavefront(sc, plan, L, dOut, ctx->dCounters.get(), ctx->wfWorkspace.get(),
                                          ctx->stats.sm_count, ctx->stream,
                                          timeTrace ? ctx->traceEvents.data() : nullptr, kMaxTracePairs, &tracePairs,
                                          timeKinds ? ctx->pairKinds.data() : nullptr, &aux,
                                          viewCount > 1 ? &views : nullptr, list);
  } else if (viewCount > 1) {  // the megakernels: one launch per view, back to back on the stream
    for (int v = 0; v < viewCount; v++) {
      LtLaunch Lv = L;
      Lv.cam = cams[v];
      launches += lt_launch_render(sc, plan, Lv, dOut + (size_t)v * L.width * L.height * L.depth,
                                   ctx->dCounters.get(), ctx->dWork.get(), ctx->stream);
    }
  } else {
    launches = lt_launch_render(sc, plan, L, dOut, ctx->dCounters.get(), ctx->dWork.get(), ctx->stream, list);
  }
  CK(cudaGetLastError());
  CK(cudaEventRecord(ctx->ev[1], ctx->stream));
  ctx->stats.kernel_launches = launches;
  if (sync || stats) {
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaEventElapsedTime(&ctx->stats.kernel_ms, ctx->ev[0], ctx->ev[1]));
    if (!wavefront) {
      ctx->stats.trace_ms = ctx->stats.kernel_ms;
      ctx->stats.trace_launches = launches;
    }
    for (int i = 0; i < tracePairs; i++) {
      float ms = 0.0f;
      cudaEventElapsedTime(&ms, ctx->traceEvents[2 * i], ctx->traceEvents[2 * i + 1]);
      const int kind = timeKinds ? ctx->pairKinds[i] : LT_TIMED_TRAVERSAL;
      if (kind == LT_TIMED_TRAVERSAL) {
        ctx->stats.trace_ms += ms;
        ctx->stats.trace_launches++;
      } else if (kind == LT_TIMED_SHADE) {
        ctx->stats.shade_ms += ms;
        ctx->stats.shade_launches++;
      } else if (kind == LT_TIMED_PRIMARY_SHADE) {
        ctx->stats.primary_shade_ms += ms;
      } else {
        ctx->stats.accumulate_ms += ms;
      }
    }
  }
  if (stats) {
    LtCounters h;
    CK(cudaMemcpy(&h, ctx->dCounters.get(), sizeof(h), cudaMemcpyDeviceToHost));
    ctx->stats.rays = h.rays;
    ctx->stats.node_tests = h.nodeTests;
    ctx->stats.tri_tests = h.triTests;
  }
  return LT_OK;
}

extern "C" int lt_render_device(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                                float* device_out, int sync) {
  if (ctx && ctx->group)
    return fail(ctx, LT_ERR_UNSUPPORTED, "lt_render_device: a multi-GPU context renders into host memory (lt_render)");
  LtLaunch L;
  int rc = check_params(ctx, scene, camera28, params, &L);
  if (rc != LT_OK) return rc;
  if (!device_out) return fail(ctx, LT_ERR_INVALID, "lt_render_device: device_out is NULL");
  return render_common(ctx, scene, L, device_out, sync != 0);
}

// lt_render_masked_device: the pixel list in ctx->dMaskList, its count first, the list from kMaskListAt on (256 B).
// lt_render_adaptive: two lists (ping-pong between rounds), their counts at [0] and [1], the second list kListPad-aligned
static const size_t kMaskListAt = 64, kListPad = 64;

// The rendering of a masked call and of each adaptive round, given a ready list of `count` pixels in device memory: the
// test hook's reversal, then the plan and the launches for the listed pixels.  An empty list launches nothing.
static int render_listed(lt_ctx* ctx, lt_scene* scene, const LtLaunch& L, int* dList, int count, float* dOut,
                         float* dM2, bool sync) {
  if (count == 0) {  // nothing to render: no pixel is written
    lt_internal_stats_start(ctx);
    return LT_OK;
  }
  const int extra = ctx->reverseList ? lt_launch_list_reverse(dList, count, ctx->stream) : 0;
  const LtList list = {dList, count, dM2};
  const int rc = render_common(ctx, scene, L, dOut, sync, nullptr, 1, &list);
  ctx->stats.kernel_launches += extra;
  return rc;
}

extern "C" int lt_render_masked_device(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                                       const uint8_t* device_mask, float* device_out, float* device_m2, int sync) {
  const std::string w = "lt_render_masked_device: ";
  if (ctx && ctx->group)
    return fail(ctx, LT_ERR_UNSUPPORTED, w + "a multi-GPU context renders into host memory (lt_render)");
  LtLaunch L;
  if (int rc = check_params(ctx, scene, camera28, params, &L)) return rc;
  if (!device_out) return fail(ctx, LT_ERR_INVALID, w + "device_out is NULL");
  if (int rc = lt_masked_image_check(ctx, L, "lt_render_masked_device")) return rc;
  if (device_m2 && (L.accumMode != LT_ACCUM_RUNNING_MEAN || L.frameStride > 1))
    return fail(ctx, LT_ERR_INVALID, w + "device_m2 needs accum_mode LT_ACCUM_RUNNING_MEAN and frame_stride <= 1");
  if (device_mask)
    if (int rc = check_device_memory(ctx, device_mask, 1, w, "device_mask")) return rc;
  if (device_m2)
    if (int rc = check_device_memory(ctx, device_m2, alignof(float), w, "device_m2")) return rc;
  CK(cudaSetDevice(ctx->device));
  const size_t pixels = (size_t)L.width * L.height;
  CK(ctx->dMaskList.grow(kMaskListAt + pixels));
  int* dCount = ctx->dMaskList.get();
  int* dList = dCount + kMaskListAt;
  lt_launch_mask_compact(device_mask, L.width, L.height, dList, dCount, ctx->stream);
  CK(cudaGetLastError());
  // the plan sizes the launch by the listed pixels: their count comes back to the host (no mask: all of them)
  int count = (int)pixels;
  if (device_mask) {
    CK(cudaMemcpyAsync(&count, dCount, sizeof count, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  const int rc = render_listed(ctx, scene, L, dList, count, device_out, device_m2, sync != 0);
  ctx->stats.kernel_launches += 1;  // the compaction
  return rc;
}

// The adaptive loop on one device (arguments checked): round 1 over every pixel of the context's part of the image, then
// rounds over the pixels the selection kernel keeps, each continuing from the frames all its pixels hold.  dOut, dM2 and
// dFrames are full-size images.  One readback and stream synchronisation per round: the survivors' count, which the
// next round's plan needs; the count of the round that reaches max_frames is read only when readLast.
static int adaptive_loop(lt_ctx* ctx, lt_scene* scene, const LtLaunch& L, const LtAdaptive& A, float* dOut, float* dM2,
                         unsigned* dFrames, int parts, int part, bool readLast, bool sync, lt_adaptive_result* res) {
  CK(cudaSetDevice(ctx->device));
  *res = lt_adaptive_result{};
  const size_t pixels = (size_t)L.width * L.height, second = kMaskListAt + (pixels + kListPad - 1) / kListPad * kListPad;
  CK(ctx->dMaskList.grow(second + pixels));
  int* counts = ctx->dMaskList.get();
  int* lists[2] = {counts + kMaskListAt, counts + second};
  cudaStream_t st = ctx->stream;
  // round 1: a full image is the NULL-mask list of lt_render_masked_device, so it plans as the unmasked call
  int count = (int)pixels;
  if (parts <= 1) {
    lt_launch_mask_compact(nullptr, L.width, L.height, lists[0], &counts[0], st);
  } else {
    lt_launch_rows_compact(L.width, L.height, parts, part, lists[0], &counts[0], st);
    count = lt_tile_rows_of(L.height, parts, part) * L.width;
  }
  CK(cudaGetLastError());
  lt_internal_stats_start(ctx);
  lt_stats sum = ctx->stats;
  sum.kernel_launches = 1;
  int cur = 0, frames = L.frames, done = 0;
  bool waited = true;  // the device has finished every round counted in sum.kernel_ms
  while (count > 0) {
    LtLaunch Lr = L;
    Lr.frames = frames;
    Lr.cam.frameCount = L.cam.frameCount + (unsigned)done;
    if (int rc = render_listed(ctx, scene, Lr, lists[cur], count, dOut, dM2, false)) return rc;
    stats_add(&sum, ctx->stats);
    res->rounds++;
    res->pixel_frames += (uint64_t)count * (uint64_t)frames;
    done += frames;
    const int nextFrames = lt_adaptive_next_frames(A, done);
    const bool last = nextFrames == 0;
    int* next = last ? nullptr : lists[1 - cur];
    sum.kernel_launches += lt_launch_adaptive_select(lists[cur], count, dOut, L.depth, dM2, dFrames,
                                                     L.cam.frameCount + (unsigned)done, A.target, A.floor, next,
                                                     &counts[1 - cur], st);
    CK(cudaGetLastError());
    if (last && !readLast) {
      waited = false;
      break;
    }
    int kept = 0;
    CK(cudaMemcpyAsync(&kept, &counts[1 - cur], sizeof kept, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
    sum.kernel_ms += ms;
    if (last) {
      res->pixels_unconverged = (uint64_t)kept;
      break;
    }
    count = kept;
    cur = 1 - cur;
    frames = nextFrames;
  }
  if (!waited && sync) {
    CK(cudaStreamSynchronize(st));
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
    sum.kernel_ms += ms;
    waited = true;
  }
  if (!waited) sum.kernel_ms = 0.0f;  // not known before the work is done
  ctx->stats = sum;
  return LT_OK;
}

// the single-GPU checks of both adaptive forms (the multi-GPU form checks in lt_multi_render_adaptive)
static int adaptive_args(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                         const lt_adaptive_params* aparams, const char* who, LtLaunch* L, LtAdaptive* A) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, std::string(who) + ": ctx is NULL");
  if (!scene || !camera28 || !params) return fail(ctx, LT_ERR_INVALID, std::string(who) + ": NULL argument");
  if (int rc = lt_params_to_launch(ctx, params, L, who)) return rc;
  memcpy(&L->cam, camera28, sizeof(RefCamera));
  return lt_adaptive_check(ctx, *L, aparams, who, A);
}

int lt_internal_render_adaptive(lt_ctx* ctx, lt_scene* scene, const LtLaunch& L, const LtAdaptive& A, float* host_out,
                                uint32_t* host_frames, int parts, int part, lt_adaptive_result* res) {
  CK(cudaSetDevice(ctx->device));
  const size_t pixels = (size_t)L.width * L.height, meanFloats = pixels * L.depth;
  CK(ctx->dAdaptive.grow(meanFloats + 4 * pixels));
  float* dMean = ctx->dAdaptive.get();
  float* dM2 = dMean + meanFloats;
  unsigned* dFrames = (unsigned*)(dM2 + 3 * pixels);
  // from zero, as lt_accum_reset leaves the context accumulator
  CK(cudaMemsetAsync(dMean, 0, (meanFloats + 3 * pixels) * sizeof(float), ctx->stream));
  if (int rc = adaptive_loop(ctx, scene, L, A, dMean, dM2, host_frames ? dFrames : nullptr, parts, part, true, true, res))
    return rc;
  if (parts <= 1) {
    if (host_out)
      if (int rc = lt_internal_download(ctx, host_out, dMean, meanFloats * sizeof(float))) return rc;
    if (host_frames)
      if (int rc = lt_internal_download(ctx, (float*)host_frames, (const float*)dFrames, pixels * sizeof(unsigned)))
        return rc;
    return LT_OK;
  }
  // a part's rows only: the blocks of the row partition, out of the full-size buffers
  const int rows = lt_tile_rows_of(L.height, parts, part);
  const size_t meanRow = (size_t)L.width * L.depth * sizeof(float), frameRow = (size_t)L.width * sizeof(unsigned);
  const size_t blockRows = (size_t)parts * LT_TILE_ROWS, first = (size_t)part * LT_TILE_ROWS;
  cudaError_t e = cudaSuccess;
  if (host_out && rows > 0)
    e = lt_copy_row_blocks(host_out, (const char*)dMean + first * meanRow, blockRows * meanRow, meanRow, rows, parts,
                           part, ctx->stream);
  if (e == cudaSuccess && host_frames && rows > 0)
    e = lt_copy_row_blocks(host_frames, (const char*)dFrames + first * frameRow, blockRows * frameRow, frameRow, rows,
                           parts, part, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) return fail(ctx, LT_ERR_CUDA, std::string("lt_render_adaptive: row copy: ") + cudaGetErrorString(e));
  return LT_OK;
}

extern "C" int lt_render_adaptive(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                                  const lt_adaptive_params* aparams, float* host_out, uint32_t* host_frames,
                                  lt_adaptive_result* out_result) {
  if (ctx && ctx->group)
    return lt_multi_render_adaptive(ctx, scene, camera28, params, aparams, host_out, host_frames, out_result);
  LtLaunch L;
  LtAdaptive A;
  if (int rc = adaptive_args(ctx, scene, camera28, params, aparams, "lt_render_adaptive", &L, &A)) return rc;
  lt_adaptive_result res;
  const int rc =
      lt_internal_render_adaptive(ctx, scene, L, A, host_out, host_frames, ctx->adaptiveParts, ctx->adaptivePart, &res);
  if (rc == LT_OK && out_result) *out_result = res;
  return rc;
}

extern "C" int lt_render_adaptive_device(lt_ctx* ctx, lt_scene* scene, const void* camera28,
                                         const lt_render_params* params, const lt_adaptive_params* aparams,
                                         float* device_out, float* device_m2, uint32_t* device_frames,
                                         lt_adaptive_result* out_result, int sync) {
  const char* who = "lt_render_adaptive_device";
  const std::string w = std::string(who) + ": ";
  if (ctx && ctx->group)
    return fail(ctx, LT_ERR_UNSUPPORTED, w + "a multi-GPU context renders into host memory (lt_render_adaptive)");
  LtLaunch L;
  LtAdaptive A;
  if (int rc = adaptive_args(ctx, scene, camera28, params, aparams, who, &L, &A)) return rc;
  if (!device_out || !device_m2) return fail(ctx, LT_ERR_INVALID, w + "device_out and device_m2 are required");
  if (int rc = check_device_memory(ctx, device_out, alignof(float), w, "device_out")) return rc;
  if (int rc = check_device_memory(ctx, device_m2, alignof(float), w, "device_m2")) return rc;
  if (device_frames)
    if (int rc = check_device_memory(ctx, device_frames, alignof(uint32_t), w, "device_frames")) return rc;
  lt_adaptive_result res;
  const int rc = adaptive_loop(ctx, scene, L, A, device_out, device_m2, device_frames, ctx->adaptiveParts,
                               ctx->adaptivePart, out_result != nullptr, sync != 0, &res);
  if (rc == LT_OK && out_result) *out_result = res;
  return rc;
}

extern "C" int lt_debug_ctx_adaptive_part(lt_ctx* ctx, int parts, int part) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_debug_ctx_adaptive_part: ctx is NULL");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_debug_ctx_adaptive_part: not available on a multi-GPU context");
  if (parts < 1 || part < 0 || part >= parts)
    return fail(ctx, LT_ERR_INVALID, "lt_debug_ctx_adaptive_part: needs parts >= 1 and 0 <= part < parts");
  ctx->adaptiveParts = parts;
  ctx->adaptivePart = part;
  return LT_OK;
}

extern "C" int lt_debug_ctx_list_order(lt_ctx* ctx, int reversed) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_debug_ctx_list_order: ctx is NULL");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_debug_ctx_list_order: not available on a multi-GPU context");
  if (reversed != 0 && reversed != 1) return fail(ctx, LT_ERR_INVALID, "lt_debug_ctx_list_order: reversed must be 0 or 1");
  ctx->reverseList = reversed != 0;
  return LT_OK;
}

int lt_internal_render(lt_ctx* ctx, lt_scene* scene, const LtLaunch& L, float* device_out) {
  return render_common(ctx, scene, L, device_out, false);
}

// Result -> the caller's host buffer.  The reference hands render() a malloc'ed (pageable) pOutputBuffer
// (src/cuda/renderer_cuda.cpp:137-139: cuMemcpyDtoH); a plain cudaMemcpy into pageable memory runs at a third of the
// link rate because the driver stages it in small pieces.  Here: pinned or registered destinations get one DMA; a
// pageable destination is filled through the context's own pinned staging buffer in 1 MB chunks -- the DMA of chunk
// k+1 overlaps the host-side copy of chunk k, and the host side is spread over a few threads.  (Registering the
// caller's buffer behind its back is not an option: a cached registration outlives a free()/mmap() of the same
// address range and would then receive the frame in pages the caller no longer sees.)
int lt_internal_download(lt_ctx* ctx, float* host_out, const float* dSrc, size_t bytes) {
  cudaPointerAttributes attr;
  memset(&attr, 0, sizeof attr);
  const bool pinned = cudaPointerGetAttributes(&attr, host_out) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  const size_t kStagedMinBytes = 1u << 20;  // smaller frames: one plain copy
  if (pinned || bytes < kStagedMinBytes) {
    CK(cudaMemcpyAsync(host_out, dSrc, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return LT_OK;
  }
  // staging granularity; measured 256 KB .. 2 MB with 8 .. 16 copier threads: 1 MB and 8 threads are best (0.68 ms per 1080p call)
  const size_t kChunk = 1u << 20;
  const size_t kMaxStage = 256u << 20;
  if (!ctx->copyPool) {
    // threads copying (this one included); measured, 24.9 MB frame into a malloc'ed buffer: 2 threads 1.49 ms,
    // 4: 0.93 ms, 8: 0.76 ms per render() call
    const unsigned hw = std::thread::hardware_concurrency();
    const int threads = hw >= 16 ? 8 : (hw >= 8 ? 4 : 2);
    ctx->copyPool.reset(new LtCopyPool(threads - 1));
  }
  const size_t want = bytes < kMaxStage ? bytes : kMaxStage;
  if (ctx->stage.count() < want && ctx->stage.grow((want + kChunk - 1) / kChunk * kChunk) != cudaSuccess) {
    cudaGetLastError();  // no pinned memory to be had: the plain copy still works
    CK(cudaMemcpyAsync(host_out, dSrc, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return LT_OK;
  }
  const size_t room = ctx->stage.count();
  for (size_t done = 0; done < bytes;) {  // one pass unless the frame exceeds the staging buffer
    const size_t pass = bytes - done < room ? bytes - done : room;
    const int chunks = (int)((pass + kChunk - 1) / kChunk);
    CK(ctx->stageEvents.grow(chunks, cudaEventDisableTiming));
    for (int c = 0; c < chunks; c++) {
      const size_t off = (size_t)c * kChunk, n = pass - off < kChunk ? pass - off : kChunk;
      CK(cudaMemcpyAsync(ctx->stage.get() + off, (const char*)dSrc + done + off, n, cudaMemcpyDeviceToHost,
                         ctx->stream));
      CK(cudaEventRecord(ctx->stageEvents[c], ctx->stream));
    }
    // host side: a small pool of copier threads (no CUDA calls in them); this thread waits for the chunks' DMA and
    // publishes how many have landed, then copies along
    LtCopyPool& pool = *ctx->copyPool;
    pool.begin((char*)host_out + done, ctx->stage.get(), pass, kChunk, chunks);
    cudaError_t err = cudaSuccess;
    for (int c = 0; c < chunks; c++) {
      cudaError_t e = cudaEventSynchronize(ctx->stageEvents[c]);
      if (e != cudaSuccess && err == cudaSuccess) err = e;
      pool.publish(c + 1);
    }
    pool.finish();
    if (err != cudaSuccess) return fail(ctx, LT_ERR_CUDA, std::string("download: ") + cudaGetErrorString(err));
    done += pass;
  }
  return LT_OK;
}

extern "C" int lt_render(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                         float* host_out) {
  if (ctx && ctx->group) return lt_multi_render(ctx, scene, camera28, params, host_out, nullptr);
  LtLaunch L;
  int rc = check_params(ctx, scene, camera28, params, &L);
  if (rc != LT_OK) return rc;
  CK(cudaSetDevice(ctx->device));
  size_t floats = (size_t)L.width * L.height * L.depth;
  rc = lt_internal_ensure_out(ctx, floats);
  if (rc != LT_OK) return rc;
  rc = render_common(ctx, scene, L, ctx->dOut.get(), true);
  if (rc != LT_OK) return rc;
  if (host_out) return lt_internal_download(ctx, host_out, ctx->dOut.get(), floats * sizeof(float));
  return LT_OK;
}

// the cameras of a views call, with its argument checks (before any device is touched)
static int check_views(lt_ctx* ctx, const void* cameras28, int view_count, const char* who,
                       std::vector<RefCamera>* cams) {
  const std::string w = std::string(who) + ": ";
  if (view_count < 1) return fail(ctx, LT_ERR_INVALID, w + "view_count must be >= 1");
  if (!cameras28) return fail(ctx, LT_ERR_INVALID, w + "cameras28 is NULL");
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, w + "ctx is NULL");
  cams->resize((size_t)view_count);
  memcpy(cams->data(), cameras28, sizeof(RefCamera) * (size_t)view_count);
  return LT_OK;
}

int lt_internal_render_views(lt_ctx* ctx, lt_scene* scene, LtLaunch L, const RefCamera* cams, int count,
                             float* host_out, int hostFirst, int hostStride) {
  L.cam = cams[0];  // the camera of a single view
  CK(cudaSetDevice(ctx->device));
  const size_t image = (size_t)L.width * L.height * L.depth, floats = image * (size_t)count;
  CK(ctx->dViews.grow(floats));
  // every view accumulates from zero, as after lt_accum_reset
  CK(cudaMemsetAsync(ctx->dViews.get(), 0, floats * sizeof(float), ctx->stream));
  int rc = render_common(ctx, scene, L, ctx->dViews.get(), true, cams, count);
  if (rc != LT_OK || !host_out) return rc;
  if (hostStride == 1)
    return lt_internal_download(ctx, host_out + (size_t)hostFirst * image, ctx->dViews.get(), floats * sizeof(float));
  for (int k = 0; k < count && rc == LT_OK; k++)
    rc = lt_internal_download(ctx, host_out + (size_t)(hostFirst + (size_t)k * hostStride) * image,
                              ctx->dViews.get() + (size_t)k * image, image * sizeof(float));
  return rc;
}

extern "C" int lt_render_views(lt_ctx* ctx, lt_scene* scene, const void* cameras28, int view_count,
                               const lt_render_params* params, float* host_out) {
  std::vector<RefCamera> cams;
  if (int rc = check_views(ctx, cameras28, view_count, "lt_render_views", &cams)) return rc;
  if (ctx->group) {
    if (view_count == 1) return lt_multi_render(ctx, scene, cameras28, params, host_out, nullptr);
    return lt_multi_render_views(ctx, scene, cams.data(), view_count, params, host_out);
  }
  LtLaunch L;
  if (int rc = check_params(ctx, scene, cameras28, params, &L)) return rc;
  return lt_internal_render_views(ctx, scene, L, cams.data(), view_count, host_out, 0, 1);
}

extern "C" int lt_render_views_device(lt_ctx* ctx, lt_scene* scene, const void* cameras28, int view_count,
                                      const lt_render_params* params, float* device_out, int sync) {
  std::vector<RefCamera> cams;
  if (int rc = check_views(ctx, cameras28, view_count, "lt_render_views_device", &cams)) return rc;
  if (ctx->group)
    return fail(ctx, LT_ERR_UNSUPPORTED,
                "lt_render_views_device: a multi-GPU context renders into host memory (lt_render_views)");
  LtLaunch L;
  int rc = check_params(ctx, scene, cameras28, params, &L);
  if (rc != LT_OK) return rc;
  if (!device_out) return fail(ctx, LT_ERR_INVALID, "lt_render_views_device: device_out is NULL");
  return render_common(ctx, scene, L, device_out, sync != 0, cams.data(), view_count);
}

extern "C" int lt_plugin_load(lt_ctx* ctx, const char* kernel_file_path, int* out_plugin_id) {
  if (!ctx || !kernel_file_path || !out_plugin_id) return fail(ctx, LT_ERR_INVALID, "lt_plugin_load: NULL argument");
  std::string err;
  LtPluginImage img;
  if (!lt_plugin_compile(kernel_file_path, &img, &err)) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_plugin_load: " + err);
  if (ctx->group) return lt_multi_plugin_load(ctx, img, out_plugin_id);
  CK(cudaSetDevice(ctx->device));
  CK(cudaFree(0));  // make sure the primary context is current for the driver-API module load
  LtPlugin* p = lt_plugin_module_load(img, &err);
  if (!p) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_plugin_load: " + err);
  ctx->plugins.push_back(p);
  *out_plugin_id = (int)ctx->plugins.size() - 1;
  return LT_OK;
}

int lt_internal_render_plugin(lt_ctx* ctx, lt_scene* scene, const RefCamera& cam, const lt_render_params& P,
                              const LtPluginRun& run, bool sync, const char* who) {
  lt_internal_stats_start(ctx);
  CK(cudaSetDevice(ctx->device));
  LtPlugin* plugin = ctx->plugins[run.id];
  const bool cl = lt_plugin_is_opencl_c(plugin);
  std::string err;
  unsigned smem = 0;
  // a work-group whose traversal stacks do not fit is refused before anything is launched
  if (cl && !lt_plugin_smem(plugin, run.kernelMode, &scene->dev, (unsigned)(run.bx * run.by), &smem, &err))
    return fail(ctx, LT_ERR_INVALID, std::string(who) + ": " + err);
  const size_t floats = (size_t)P.width * P.height * P.depth;
  int rc = lt_internal_ensure_out(ctx, floats);
  if (rc != LT_OK) return rc;
  // LT_ACCUM_NONE: every frame into the output, in order (F consecutive single-frame calls); otherwise every frame into
  // the sample buffer, folded into the accumulator after it
  const bool fold = P.accum_mode != LT_ACCUM_NONE;
  if (fold) CK(ctx->dSample.grow(floats));
  float* dFrame = fold ? ctx->dSample.get() : ctx->dOut.get();
  CK(ctx->dCamera.grow(P.frames));
  // frame k reads its own record, frameCount = camera.frameCount + k * frame_stride
  const uint32_t stride = P.frame_stride ? P.frame_stride : 1u;
  std::vector<RefCamera> cams((size_t)P.frames, cam);
  for (int k = 0; k < P.frames; k++) cams[k].frameCount = cam.frameCount + (uint32_t)k * stride;
  CK(cudaMemcpyAsync(ctx->dCamera.get(), cams.data(), sizeof(RefCamera) * cams.size(), cudaMemcpyHostToDevice,
                     ctx->stream));
  if (lt_plugin_publish_scene(plugin, &scene->dev, ctx->stream, &err) != 0)
    return fail(ctx, LT_ERR_CUDA, std::string(who) + ": " + err);
  // pixels outside every work block (the remainder of W / wbx and H / wby) read 0; the reference leaves them undefined
  if (cl) CK(cudaMemsetAsync(dFrame, 0, floats * sizeof(float), ctx->stream));
  LtLaunch L = {};
  L.width = P.width;
  L.height = P.height;
  L.depth = P.depth;
  L.accumMode = P.accum_mode;
  L.accumWeight = P.accum_weight;
  CK(cudaEventRecord(ctx->ev[0], ctx->stream));
  int launches = 0;
  const lt_scene& sc = *scene;
  for (int k = 0; k < P.frames; k++) {
    const RefCamera* dCam = ctx->dCamera.get() + k;
    const int n = cl ? lt_plugin_launch_cl(plugin, run.kernelMode, &sc.dev, sc.dNodes.get(), sc.dPrims.get(),
                                           sc.dMats.get(), sc.dLights.get(), dCam, dFrame, P.width, P.height, P.depth,
                                           run.wbx, run.wby, run.bx, run.by, ctx->stream, &err)
                     : (lt_plugin_launch(plugin, run.kernelMode, &sc.dev, sc.dNodes.get(), sc.dPrims.get(),
                                         sc.dMats.get(), sc.dLights.get(), dCam, dFrame, P.width, P.height, P.depth,
                                         run.bx, run.by, ctx->stream, &err) == 0 ? 1 : -1);
    if (n < 0) return fail(ctx, LT_ERR_CUDA, std::string(who) + ": " + err);
    launches += n;
    if (fold) {
      L.cam = cams[k];
      launches += lt_launch_plugin_accumulate(L, dFrame, ctx->dOut.get(), ctx->stats.sm_count, ctx->stream);
    }
  }
  CK(cudaGetLastError());
  CK(cudaEventRecord(ctx->ev[1], ctx->stream));
  ctx->stats.kernel_launches = launches;
  if (sync) {
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaEventElapsedTime(&ctx->stats.kernel_ms, ctx->ev[0], ctx->ev[1]));
  }
  return LT_OK;
}

// Checks a plug-in id (and, for `cl` >= 0, its language) against the plug-ins of ctx; LT_ERR_INVALID otherwise.
static int check_plugin(lt_ctx* ctx, int plugin_id, int cl, const char* who) {
  const std::vector<LtPlugin*>& plugins = ctx->group ? lt_multi_plugins(ctx) : ctx->plugins;
  if (plugin_id < 0 || plugin_id >= (int)plugins.size())
    return fail(ctx, LT_ERR_INVALID, std::string(who) + ": bad argument");
  if (cl == 0 && lt_plugin_is_opencl_c(plugins[plugin_id]))
    return fail(ctx, LT_ERR_INVALID, std::string(who) + ": plug-in " + std::to_string(plugin_id) +
                                         " is an OpenCL C kernel; launch it with lt_render_plugin_cl");
  if (cl == 1 && !lt_plugin_is_opencl_c(plugins[plugin_id]))
    return fail(ctx, LT_ERR_INVALID, std::string(who) + ": plug-in " + std::to_string(plugin_id) +
                                         " is a CUDA kernel; launch it with lt_render_plugin");
  return LT_OK;
}

// One frame, no accumulation, into ctx->dOut, then to host_out: the two single-frame entry points
static int render_plugin_once(lt_ctx* ctx, lt_scene* scene, const void* camera28, const LtPluginRun& run, int width,
                              int height, int depth, float* host_out, const char* who) {
  lt_render_params P;
  memset(&P, 0, sizeof P);
  P.struct_size = sizeof P;
  P.width = width;
  P.height = height;
  P.depth = depth;
  P.frames = 1;
  RefCamera cam;
  memcpy(&cam, camera28, sizeof cam);
  int rc = lt_internal_render_plugin(ctx, scene, cam, P, run, true, who);
  if (rc != LT_OK) return rc;
  if (host_out)
    return lt_internal_download(ctx, host_out, ctx->dOut.get(), (size_t)width * height * depth * sizeof(float));
  return LT_OK;
}

extern "C" int lt_render_plugin(lt_ctx* ctx, lt_scene* scene, const void* camera28, int plugin_id, int kernel_mode,
                                int width, int height, int depth, int block_x, int block_y, float* host_out) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_render_plugin: ctx is NULL");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_render_plugin: plug-in kernels run on single-GPU contexts");
  if (!scene || !camera28 || width <= 0 || height <= 0 || depth < 1)
    return fail(ctx, LT_ERR_INVALID, "lt_render_plugin: bad argument");
  if (int rc = check_plugin(ctx, plugin_id, 0, "lt_render_plugin")) return rc;
  const LtPluginRun run = {plugin_id, kernel_mode ? 1 : 0, block_x, block_y, 0, 0};
  return render_plugin_once(ctx, scene, camera28, run, width, height, depth, host_out, "lt_render_plugin");
}

extern "C" int lt_render_plugin_cl(lt_ctx* ctx, lt_scene* scene, const void* camera28, int plugin_id, int kernel_mode,
                                   int width, int height, int depth, int work_block_x, int work_block_y, int group_x,
                                   int group_y, float* host_out) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_render_plugin_cl: ctx is NULL");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_render_plugin_cl: plug-in kernels run on single-GPU contexts");
  if (!scene || !camera28 || width <= 0 || height <= 0 || depth < 1)
    return fail(ctx, LT_ERR_INVALID, "lt_render_plugin_cl: bad argument");
  if (int rc = check_plugin(ctx, plugin_id, 1, "lt_render_plugin_cl")) return rc;
  std::string err;
  LtPluginRun run = {plugin_id, kernel_mode ? 1 : 0, group_x, group_y, work_block_x, work_block_y};
  if (!lt_plugin_cl_shape(width, height, &run.wbx, &run.wby, &run.bx, &run.by, &err))
    return fail(ctx, LT_ERR_INVALID, "lt_render_plugin_cl: " + err);
  return render_plugin_once(ctx, scene, camera28, run, width, height, depth, host_out, "lt_render_plugin_cl");
}

extern "C" int lt_render_plugin_frames(lt_ctx* ctx, lt_scene* scene, const void* camera28, int plugin_id,
                                       const lt_render_params* params, int work_block_x, int work_block_y,
                                       float* host_out) {
  const char* who = "lt_render_plugin_frames";
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_render_plugin_frames: ctx is NULL");
  if (!scene || !camera28 || !params) return fail(ctx, LT_ERR_INVALID, "lt_render_plugin_frames: NULL argument");
  // lt_render's checks; kernel and max_ray_depth do not apply (a plug-in is its own kernel, with its own bounce cap)
  lt_render_params P;
  if (int rc = lt_params_normalise(ctx, params, std::string(who) + ": ", &P)) return rc;
  P.kernel = 0;
  P.max_ray_depth = 0;
  LtLaunch L;
  if (int rc = lt_params_to_launch(ctx, &P, &L, who)) return rc;
  if (int rc = check_plugin(ctx, plugin_id, -1, who)) return rc;
  if (P.flags & (LT_FLAG_STATS | LT_FLAG_STATS_TRACED | LT_FLAG_CULL))
    return fail(ctx, LT_ERR_UNSUPPORTED, "lt_render_plugin_frames: a plug-in has no counters (LT_FLAG_STATS) and no "
                                         "culled traversal (LT_FLAG_CULL)");
  const bool cl = lt_plugin_is_opencl_c((ctx->group ? lt_multi_plugins(ctx) : ctx->plugins)[plugin_id]);
  LtPluginRun run = {plugin_id, P.kernel_mode ? 1 : 0, P.block_x, P.block_y, work_block_x, work_block_y};
  if (cl) {
    std::string err;
    if (!lt_plugin_cl_shape(P.width, P.height, &run.wbx, &run.wby, &run.bx, &run.by, &err))
      return fail(ctx, LT_ERR_INVALID, "lt_render_plugin_frames: " + err);
  } else if (work_block_x || work_block_y) {
    return fail(ctx, LT_ERR_INVALID, "lt_render_plugin_frames: a work block applies to OpenCL C plug-ins only");
  }
  if (ctx->group) return lt_multi_render(ctx, scene, camera28, &P, host_out, &run);
  RefCamera cam;
  memcpy(&cam, camera28, sizeof cam);
  int rc = lt_internal_render_plugin(ctx, scene, cam, P, run, true, who);
  if (rc != LT_OK) return rc;
  if (host_out)
    return lt_internal_download(ctx, host_out, ctx->dOut.get(), (size_t)P.width * P.height * P.depth * sizeof(float));
  return LT_OK;
}

extern "C" int64_t lt_debug_translate_cl(const char* text, char* out, uint64_t out_bytes, int32_t* contract_off) {
  if (!text) return fail(nullptr, LT_ERR_INVALID, "lt_debug_translate_cl: NULL text");
  bool off = false, deviceApi = false;
  std::vector<std::pair<std::string, int>> kernels;
  std::string t = lt_cl_translate(text, &off, &deviceApi, &kernels);
  if (contract_off) *contract_off = off ? 1 : 0;
  if (out && out_bytes > t.size()) memcpy(out, t.c_str(), t.size() + 1);
  return (int64_t)t.size() + 1;
}

extern "C" int lt_debug_compile_cl(const char* kernel_file_path, char* log, uint64_t log_bytes) {
  if (!kernel_file_path) return fail(nullptr, LT_ERR_INVALID, "lt_debug_compile_cl: NULL path");
  std::string err;
  bool ok = lt_plugin_compile_cl_only(kernel_file_path, &err);
  if (log && log_bytes) {
    size_t n = err.size() < log_bytes - 1 ? err.size() : (size_t)(log_bytes - 1);
    memcpy(log, err.data(), n);
    log[n] = 0;
  }
  if (!ok) return fail(nullptr, LT_ERR_UNSUPPORTED, "lt_debug_compile_cl: " + err);
  return LT_OK;
}

// Opt-in for applications that keep one output buffer alive across many render() calls (the progressive examples):
// a registered buffer receives the frame by a single DMA.  The caller owns the lifetime: unregister before free().
extern "C" int lt_host_register(void* host_buffer, uint64_t bytes) {
  if (!host_buffer || bytes == 0) return fail(nullptr, LT_ERR_INVALID, "lt_host_register: bad argument");
  cudaError_t e = cudaHostRegister(host_buffer, bytes, cudaHostRegisterPortable);
  if (e == cudaErrorHostMemoryAlreadyRegistered) {
    cudaGetLastError();
    return LT_OK;
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(nullptr, e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? LT_ERR_NO_DEVICE : LT_ERR_CUDA,
                std::string("lt_host_register: ") + cudaGetErrorString(e));
  }
  return LT_OK;
}

extern "C" int lt_host_unregister(void* host_buffer) {
  if (!host_buffer) return fail(nullptr, LT_ERR_INVALID, "lt_host_unregister: bad argument");
  cudaError_t e = cudaHostUnregister(host_buffer);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(nullptr, LT_ERR_CUDA, std::string("lt_host_unregister: ") + cudaGetErrorString(e));
  }
  return LT_OK;
}

extern "C" int lt_accum_reset(lt_ctx* ctx) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_accum_reset: ctx is NULL");
  if (ctx->group) return lt_multi_accum_reset(ctx);
  CK(cudaSetDevice(ctx->device));
  if (ctx->dOut.get()) CK(cudaMemsetAsync(ctx->dOut.get(), 0, ctx->dOut.bytes(), ctx->stream));
  return LT_OK;
}

extern "C" int lt_accum_read(lt_ctx* ctx, float* host_out, uint64_t float_count) {
  if (!ctx || !host_out) return fail(ctx, LT_ERR_INVALID, "lt_accum_read: NULL argument");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_accum_read: a multi-GPU context returns its accumulator through lt_render");
  if (!ctx->dOut.get() || float_count > ctx->dOut.count()) return fail(ctx, LT_ERR_INVALID, "lt_accum_read: no accumulator of that size");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(host_out, ctx->dOut.get(), float_count * sizeof(float), cudaMemcpyDeviceToHost));
  return LT_OK;
}

static int primary_hits_impl(lt_ctx* ctx, lt_scene* scene, const void* camera28, int kernel, int flags, int width,
                             int height, int32_t* ids, int32_t* hit, float* tuv) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_primary_hits: ctx is NULL");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_primary_hits: use a single-GPU context");
  if (!scene || !camera28 || width <= 0 || height <= 0 || kernel < 0 || kernel >= LT_KERNEL_COUNT)
    return fail(ctx, LT_ERR_INVALID, "lt_primary_hits: bad argument");
  CK(cudaSetDevice(ctx->device));
  size_t n = (size_t)width * height;
  LtBuf<int> all;  // one allocation: ids | hit | t,u,v
  CK(all.grow(5 * n));
  int *dIds = all.get(), *dHit = dIds + n;
  float* dTuv = reinterpret_cast<float*>(dIds + 2 * n);
  RefCamera cam;
  memcpy(&cam, camera28, sizeof(cam));
  const LtPlan plan = lt_plan_primary_hits(flags, width, height, scene_facts(scene));
  lt_launch_primary_hits(scene_for_plan(scene, plan), plan, cam, kernel, flags, width, height, dIds, dHit, dTuv,
                         ctx->stream);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e == cudaSuccess && ids) e = cudaMemcpy(ids, dIds, n * sizeof(int), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && hit) e = cudaMemcpy(hit, dHit, n * sizeof(int), cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && tuv) e = cudaMemcpy(tuv, dTuv, 3 * n * sizeof(float), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return fail(ctx, LT_ERR_CUDA, std::string("lt_primary_hits: ") + cudaGetErrorString(e));
  return LT_OK;
}

extern "C" int lt_primary_hits(lt_ctx* ctx, lt_scene* scene, const void* camera28, int kernel, int width, int height,
                               int32_t* ids, int32_t* hit, float* tuv) {
  return primary_hits_impl(ctx, scene, camera28, kernel, 0, width, height, ids, hit, tuv);
}

extern "C" int lt_primary_hits_flags(lt_ctx* ctx, lt_scene* scene, const void* camera28, int kernel, int flags,
                                     int width, int height, int32_t* ids, int32_t* hit, float* tuv) {
  return primary_hits_impl(ctx, scene, camera28, kernel, flags, width, height, ids, hit, tuv);
}

// parity hooks: evaluate device-side helper functions on host-supplied inputs
extern "C" int lt_debug_random(lt_ctx* ctx, const float* fx, const float* fy, const float* seed, int n, float* out) {
  if (!ctx || ctx->group || !fx || !fy || !seed || !out || n <= 0) return fail(ctx, LT_ERR_INVALID, "lt_debug_random: bad argument");
  CK(cudaSetDevice(ctx->device));
  LtBuf<float> buf;
  CK(buf.grow(4 * (size_t)n));
  float* d = buf.get();
  cudaError_t e = cudaMemcpy(d, fx, sizeof(float) * n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(d + n, fy, sizeof(float) * n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(d + 2 * (size_t)n, seed, sizeof(float) * n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    lt_launch_debug_random(d, d + n, d + 2 * (size_t)n, n, d + 3 * (size_t)n, ctx->stream);
    e = cudaStreamSynchronize(ctx->stream);
  }
  if (e == cudaSuccess) e = cudaMemcpy(out, d + 3 * (size_t)n, sizeof(float) * n, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return fail(ctx, LT_ERR_CUDA, std::string("lt_debug_random: ") + cudaGetErrorString(e));
  return LT_OK;
}

extern "C" int lt_debug_hemisphere(lt_ctx* ctx, const float* u1, const float* u2, const float* up3, int n, float* out4) {
  if (!ctx || ctx->group || !u1 || !u2 || !up3 || !out4 || n <= 0) return fail(ctx, LT_ERR_INVALID, "lt_debug_hemisphere: bad argument");
  CK(cudaSetDevice(ctx->device));
  LtBuf<float> buf;
  CK(buf.grow(9 * (size_t)n));
  float* d = buf.get();
  cudaError_t e = cudaMemcpy(d, u1, sizeof(float) * n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(d + n, u2, sizeof(float) * n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(d + 2 * (size_t)n, up3, sizeof(float) * 3 * n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    lt_launch_debug_hemisphere(d, d + n, d + 2 * (size_t)n, n, d + 5 * (size_t)n, ctx->stream);
    e = cudaStreamSynchronize(ctx->stream);
  }
  if (e == cudaSuccess) e = cudaMemcpy(out4, d + 5 * (size_t)n, sizeof(float) * 4 * n, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return fail(ctx, LT_ERR_CUDA, std::string("lt_debug_hemisphere: ") + cudaGetErrorString(e));
  return LT_OK;
}

extern "C" int lt_last_stats(const lt_ctx* ctx, lt_stats* out_stats) {
  if (!ctx || !out_stats) return LT_ERR_INVALID;
  *out_stats = ctx->stats;
  return LT_OK;
}

static const char* kKernelNames[LT_KERNEL_COUNT] = {"basic.cu",       "basic.cl",          "custom_opencl.cl",
                                                    "basic_lighting.cl", "accumulator.cl", "global_illumination.cl(25)",
                                                    "global_illumination.cl(1)"};

extern "C" const char* lt_kernel_name(int kernel) {
  return (kernel < 0 || kernel >= LT_KERNEL_COUNT) ? "unknown" : kKernelNames[kernel];
}

// kernelFilePath -> built-in pipeline, by CONTENT (the reference compiles whatever text the file holds,
// src/cuda/renderer_cuda.cpp:20-39,52-55, so the name alone must never select a pipeline):
//   * a descriptor file of this repository -- nothing but // comment lines, one of them "lt-pipeline: <tag>" -- or
//   * a file whose text is, byte for byte (CR dropped), one of the seven kernel files the reference ships
//     (lt_kernel_hashes.inc: FNV-1a-64 + length; only hashes are stored)
// maps to the hand-written pipeline that reproduces that kernel.  Anything else -- including an EDITED copy of a
// shipped kernel under its old name -- is a user kernel: LT_ERR_UNSUPPORTED here; the renderer then compiles it as a
// plug-in (lt_plugin_load): a .cu as CUDA, a .cl as OpenCL C on the runtime of lt_opencl_c.cuh.
struct LtKernelHash {
  unsigned long long hash;
  size_t bytes;
  int kernel;
};
static const LtKernelHash kShippedKernels[] = {
#include "lt_kernel_hashes.inc"
};

static bool read_file(const char* path, std::string* text) {
  FILE* f = fopen(path, "rb");
  if (!f) return false;
  char buf[4096];
  size_t n;
  while ((n = fread(buf, 1, sizeof buf, f)) > 0) text->append(buf, n);
  fclose(f);
  return true;
}

extern "C" int lt_kernel_from_path(const char* path) {
  if (!path) return LT_ERR_INVALID;
  std::string text;
  if (!read_file(path, &text)) {
    g_error = std::string("lt_kernel_from_path: cannot open kernel file '") + path + "'";
    return LT_ERR_UNSUPPORTED;
  }
  // descriptor: comment lines only, carrying a pipeline tag
  static const struct { const char* tag; int kernel; } kTags[] = {
      {"basic_cu", LT_KERNEL_BASIC_CU},     {"basic_cl", LT_KERNEL_BASIC_CL},       {"custom_bary", LT_KERNEL_CUSTOM_BARY},
      {"lighting25", LT_KERNEL_LIGHTING25}, {"accumulator", LT_KERNEL_ACCUMULATOR}, {"gi25", LT_KERNEL_GI25},
      {"gi", LT_KERNEL_GI}};
  bool commentsOnly = true;
  int tagged = -1;
  for (size_t pos = 0; pos < text.size();) {
    size_t end = text.find('\n', pos);
    if (end == std::string::npos) end = text.size();
    std::string line = text.substr(pos, end - pos);
    pos = end + 1;
    size_t b = line.find_first_not_of(" \t\r");
    if (b == std::string::npos) continue;
    if (line.compare(b, 2, "//") != 0) {
      commentsOnly = false;
      break;
    }
    size_t t = line.find("lt-pipeline:");
    if (t != std::string::npos && tagged < 0) {
      std::string tag = line.substr(t + 12);
      size_t tb = tag.find_first_not_of(" \t"), te = tag.find_last_not_of(" \t\r");
      tag = tb == std::string::npos ? "" : tag.substr(tb, te - tb + 1);
      for (size_t k = 0; k < sizeof kTags / sizeof kTags[0]; k++)
        if (tag == kTags[k].tag) tagged = kTags[k].kernel;
    }
  }
  if (commentsOnly && tagged >= 0) return tagged;
  // the reference's own shipped text
  unsigned long long h = 14695981039346656037ull;
  size_t bytes = 0;
  for (size_t i = 0; i < text.size(); i++) {
    if (text[i] == '\r') continue;
    h = (h ^ (unsigned char)text[i]) * 1099511628211ull;
    bytes++;
  }
  for (size_t k = 0; k < sizeof kShippedKernels / sizeof kShippedKernels[0]; k++)
    if (kShippedKernels[k].hash == h && kShippedKernels[k].bytes == bytes) return kShippedKernels[k].kernel;
  g_error = std::string("lt_kernel_from_path: '") + path + "' is neither a kernel descriptor nor the unmodified text of "
            "a shipped kernel (user kernels are compiled as plug-ins: lt_plugin_load)";
  return LT_ERR_UNSUPPORTED;
}
