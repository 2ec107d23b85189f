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

// Copier threads of download(): they sleep between jobs; a job is `chunks` pieces of a pinned staging buffer to be
// copied to the destination as soon as the owner has published them.
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

// cudaMalloc / cudaFree of a buffer the scene owns, counted in s->deviceBytes (lt_debug_scene_bytes)
template <class T>
static cudaError_t scene_alloc(lt_scene* s, T** p, size_t bytes) {
  const cudaError_t e = cudaMalloc((void**)p, bytes);
  if (e == cudaSuccess) s->deviceBytes += bytes;
  return e;
}
template <class T>
static void scene_free(lt_scene* s, T** p, size_t bytes) {
  if (*p) s->deviceBytes -= bytes;
  cudaFree(*p);
  *p = nullptr;
}

// ------------------------------------------------------------------------------------------------
// Launch plan: which kernels a call runs, on which tree, at which sizes.  Pure (no CUDA call, no allocation), so that
// lt_debug_plan shows it on a machine without a GPU.
// ------------------------------------------------------------------------------------------------
static_assert(LT_DEV_KERNEL_BASIC_CU == LT_KERNEL_BASIC_CU && LT_DEV_KERNEL_BASIC_CL == LT_KERNEL_BASIC_CL &&
                  LT_DEV_KERNEL_CUSTOM_BARY == LT_KERNEL_CUSTOM_BARY && LT_DEV_KERNEL_LIGHTING25 == LT_KERNEL_LIGHTING25 &&
                  LT_DEV_KERNEL_ACCUMULATOR == LT_KERNEL_ACCUMULATOR && LT_DEV_KERNEL_GI25 == LT_KERNEL_GI25 &&
                  LT_DEV_KERNEL_GI == LT_KERNEL_GI,
              "lt_device_types.h: kernel ids differ from enum lt_kernel");
static_assert(LT_DEV_FLAG_STATS == LT_FLAG_STATS && LT_DEV_FLAG_CULL == LT_FLAG_CULL &&
                  LT_DEV_FLAG_STATS_TRACED == LT_FLAG_STATS_TRACED,
              "lt_device_types.h: flags differ from enum lt_flags");

struct LtSceneFacts {
  int nodeCount, stackDepth;
  LtTree copies;  // the threaded copies the scene has (LT_TREE_CHILD_PAIR: none)
};

// Threaded copies lt_scene_upload makes of a tree of nNodes nodes: built on the host up to threadedMaxNodes (8 x 32 B
// x N for the full copies, at most as much again for the pruned ones, must stay cache resident); for larger trees the
// full copies built on the device, unless they would not fit the budget (4 GB and an eighth of the device) or 31-bit
// record indices.
static LtTree lt_plan_threaded_copies(int nNodes, size_t totalMem, const LtLimits& lim) {
  if (nNodes <= lim.threadedMaxNodes) return LT_TREE_HOST_THREADED;
  const size_t bytes = sizeof(LtThreadNode) * 8 * (size_t)nNodes;
  if (nNodes > 1 && bytes <= (4ull << 30) && bytes <= totalMem / 8 && (long long)nNodes * 8 < 0x7fffffffll)
    return LT_TREE_DEVICE_THREADED;
  return LT_TREE_CHILD_PAIR;
}

// The threaded copies serve the exact, uncounted kernels only: the stats kernels count in the stack traversal, whose
// tests are the same ones, the culled traversal has no threaded form, and LT_FLAG_NO_THREADED selects the stack
// traversal for comparison.  A large scene's device-built copies serve coherent launches only (camera rays and shadow
// rays towards a light: the two lighting kernels on the megakernel): 1 M triangles, 1080p, primary + shadow 0.96
// instead of 1.10 ms.  For the incoherent rays of GI they lose (56.8 instead of 42.6 ms per 16-spp frame: eight copies
// of the tree no longer fit in L2), and the tile-fetching k_flat_stream is faster on the child-pair tree (0.66 against
// 0.72 ms: half the dependent steps per ray).
static LtTree plan_tree(int flags, bool coherent, LtTree copies) {
  if (flags & (LT_FLAG_STATS | LT_FLAG_CULL | LT_FLAG_NO_THREADED)) return LT_TREE_CHILD_PAIR;
  if (copies == LT_TREE_DEVICE_THREADED && !coherent) return LT_TREE_CHILD_PAIR;
  return copies;
}

static int tile_blocks(int width, int height) { return ((width + 15) / 16) * ((height + 7) / 8); }

static LtPlan lt_plan_primary_hits(int flags, int width, int height, const LtSceneFacts& s) {
  LtPlan p = {};
  p.pipeline = LT_PIPE_FLAT;
  p.tree = plan_tree(flags, false, s.copies);
  p.cull = (flags & LT_FLAG_CULL) != 0;
  p.smemStack = p.smemTrace = lt_traversal_smem(lt_stack_levels(s), LT_BLOCK, p.cull);
  p.grid = tile_blocks(width, height);
  return p;
}

// Views of one call (lt_render_views) share no camera rays, so the frames' threshold does not carry over.  Measured
// (tools/views_timing.py, profiles/views_timing_b200.txt; NVIDIA B200 at its 1000 W power limit): one-frame 1080p GI
// views, 4 bounces, on the Cornell box, ms per view of the megakernel (one launch per view) against the wavefront over
// the views: V = 1 (2 073 600 paths) 0.705 against 0.787, V = 2 (4 147 200) 0.716 against 0.551, V = 4 0.799 against
// 0.485, V = 8 0.822 against 0.447, V = 16 0.796 against 0.403.  The crossover lies between 2.1 M and 4.1 M paths.
// The lighting kernels keep their factor of 4 (not measured for views).
static const long long kViewsMinPaths = 3ll << 20;

// views: a call of several views (lt_render_views) runs its (view, frame) pairs through one wavefront launch, or one
// megakernel launch per view
static LtPlan lt_plan_render(const LtLaunch& L, const LtSceneFacts& s, size_t totalMem, int smCount,
                             const LtLimits& lim, int views = 1) {
  LtPlan p = {};
  p.error = LT_OK;
  p.stats = (L.flags & LT_FLAG_STATS) != 0;
  p.cull = (L.flags & LT_FLAG_CULL) != 0;
  const long long pixels = (long long)L.width * L.height;
  const bool isGI = L.kernel == LT_KERNEL_GI25 || L.kernel == LT_KERNEL_GI;
  // stochastic kernels: wavefront pipeline for large launches, persistent megakernel for small ones
  p.pipeline = L.kernel >= LT_KERNEL_LIGHTING25 ? LT_PIPE_PATH : LT_PIPE_FLAT;
  if (p.pipeline == LT_PIPE_PATH && !(L.flags & LT_FLAG_MEGAKERNEL)) {
    // measured (tools/compare_pipelines.py): the wavefront wins once ~8M paths are in flight per batch; below that,
    // and for the two-ray lighting kernels on small scenes, its per-round launches and state traffic lose.  Second
    // measurement (shared camera rays, overlapped batches): the two-ray lighting kernels on a small scene win too
    // once a launch holds several batches (64 frames at 1080p: 1.31x); the 25-sample kernels stay on k_path
    const long long minPaths = views > 1 ? kViewsMinPaths : 1ll << 23;
    const long long need = (isGI || s.nodeCount > 100000) ? minPaths : 4 * minPaths;
    const bool forced = (L.flags & (LT_FLAG_WAVEFRONT | LT_FLAG_CULL)) != 0;
    const long long pairs = (long long)L.frames * views;  // (view, frame) pairs, view-major
    bool wavefront = forced || (pixels * pairs >= need && L.kernel != LT_KERNEL_GI25 &&
                                L.kernel != LT_KERNEL_LIGHTING25);
    // A queue entry carries the bounce depth in 5 bits (wf_pack_path): deeper bounce caps stay on the megakernel,
    // which is the same arithmetic per path (0 = the reference constant 16).  It carries its path id in 25 bits:
    // one frame must fit.
    const char* unsupported = nullptr;
    if (wavefront && isGI && L.maxRayDepth > 32)
      unsupported = "lt_render: the wavefront pipeline handles max_ray_depth <= 32 (use the default schedule)";
    else if (wavefront && pixels > (1ll << 25))
      unsupported = "lt_render: the wavefront pipeline handles at most 2^25 pixels per frame";
    if (unsupported && forced) {
      p.error = LT_ERR_UNSUPPORTED;
      p.message = unsupported;
      return p;
    }
    if (wavefront && !unsupported) {
      p.pipeline = LT_PIPE_WAVEFRONT;
      p.forced = forced;
      // paths in flight, both overlapped batches together (~200 B each), on at most 1/8 of the device
      long long cap = 1ll << 26;
      const long long memCap = (long long)(totalMem / 8) / 200;
      if (cap > memCap) cap = memCap;
      int batchFrames = (int)(cap / pixels);
      if (batchFrames < 1) batchFrames = 1;
      if (batchFrames > pairs) batchFrames = (int)pairs;
      // Two consecutive batches overlap on two streams (the trace kernel of one beside the shade kernel of the other:
      // L1 data pipe vs DRAM): half-size batches, one workspace each -- same memory.  LT_FLAG_SERIAL: one stream,
      // kernels run one at a time.  Measured: reserving room on the SMs for the other batch's blocks (fewer
      // persistent trace blocks) does not pay, nor do 3 or 4 batches in flight (profiles/r2u_overlap_sweep.txt).
      p.streams = !(L.flags & (LT_FLAG_SERIAL | LT_FLAG_STATS)) && pairs >= 2 ? 2 : 1;
      batchFrames = (batchFrames + p.streams - 1) / p.streams;
      long long perBatch = (1ll << 25) / pixels;  // a queue entry carries its path id in 25 bits
      if (perBatch < 1) perBatch = 1;
      p.batchFrames = batchFrames > perBatch ? (int)perBatch : batchFrames;
      p.samplesPerFrame = (L.kernel == LT_KERNEL_LIGHTING25 || L.kernel == LT_KERNEL_GI25) ? 25 : 1;
      p.rounds = isGI ? 2 + 2 * (L.maxRayDepth > 0 ? L.maxRayDepth : 16) : 2;
      p.sharedPrimary = !p.stats && !p.cull;  // the exact, uncounted pipelines
      p.classify = p.sharedPrimary && p.samplesPerFrame == 1;
      // primary records: one set per launch; with views, one set per view a batch touches, per batch workspace
      size_t records = lt_wf_primary_hits_bytes(pixels);
      if (views > 1)
        records = p.sharedPrimary ? lt_wf_view_records_bytes(pixels, lt_wf_views_per_batch(p.batchFrames, L.frames,
                                                                                            views)) * (size_t)p.streams
                                  : 0;
      p.workspaceBytes = lt_wf_workspace_bytes_padded((long long)p.batchFrames * pixels) * (size_t)p.streams + records;
    }
  }
  // camera rays and one shadow ray per hit: the two lighting kernels on the megakernel
  const bool coherent =
      p.pipeline == LT_PIPE_PATH && (L.kernel == LT_KERNEL_LIGHTING25 || L.kernel == LT_KERNEL_ACCUMULATOR);
  p.tree = plan_tree(L.flags, coherent, s.copies);
  p.smemStack = lt_traversal_smem(lt_stack_levels(s), LT_BLOCK, p.cull);
  p.smemTrace = p.tree == LT_TREE_CHILD_PAIR ? p.smemStack : lt_traversal_smem(0, LT_BLOCK, false);
  // shared memory is what limits residency of the persistent kernels (the threaded trace kernel's 8 KB: the cap of
  // 8); k_flat_stream measured at 4 .. 10: no difference (the longest tile bounds the kernel)
  p.blocksPerSm = (int)((200 * 1024) / p.smemTrace);
  if (p.blocksPerSm > 8) p.blocksPerSm = 8;
  if (p.blocksPerSm < 1) p.blocksPerSm = 1;
  // exact, uncounted launches of the deterministic pipelines on large scenes: persistent warps fetching tiles
  if (p.pipeline == LT_PIPE_FLAT && !(L.flags & (LT_FLAG_STATS | LT_FLAG_CULL | LT_FLAG_NO_STREAM)) &&
      p.tree == LT_TREE_CHILD_PAIR && s.nodeCount >= lim.streamMinNodes)
    p.pipeline = LT_PIPE_FLAT_STREAM;
  if (p.pipeline == LT_PIPE_FLAT_STREAM) {
    const int warpsNeeded = (((L.width + 7) >> 3) * ((L.height + 3) >> 2) + 3) / 4;  // blocks of 4 warps, one tile each
    p.grid = smCount * p.blocksPerSm < warpsNeeded ? smCount * p.blocksPerSm : warpsNeeded;
  } else if (p.pipeline == LT_PIPE_WAVEFRONT) {
    p.grid = smCount * p.blocksPerSm;
  } else {
    p.grid = tile_blocks(L.width, L.height);
  }
  return p;
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
  cudaError_t e2 = cudaStreamCreateWithFlags(&ctx->ownStream, cudaStreamNonBlocking);
  if (e2 == cudaSuccess) e2 = cudaEventCreate(&ctx->ev0);
  if (e2 == cudaSuccess) e2 = cudaEventCreate(&ctx->ev1);
  if (e2 == cudaSuccess) e2 = cudaMalloc(&ctx->dCounters, sizeof(LtCounters));
  if (e2 == cudaSuccess) e2 = cudaMalloc(&ctx->dWork, 256);
  if (e2 == cudaSuccess) e2 = cudaStreamCreateWithFlags(&ctx->wfAux.extra, cudaStreamNonBlocking);
  if (e2 == cudaSuccess) e2 = cudaEventCreateWithFlags(&ctx->wfAux.fork, cudaEventDisableTiming);
  for (int k = 0; k < 2; k++)
    if (e2 == cudaSuccess) e2 = cudaEventCreateWithFlags(&ctx->wfAux.order[k], cudaEventDisableTiming);
  if (e2 != cudaSuccess) {
    std::string m = std::string("lt_ctx_create: ") + cudaGetErrorString(e2);
    delete ctx;
    return fail(nullptr, LT_ERR_CUDA, m);
  }
  ctx->stream = ctx->ownStream;
  *out_ctx = ctx;
  return LT_OK;
}

extern "C" void lt_ctx_destroy(lt_ctx* ctx) {
  if (!ctx) return;
  if (ctx->group) {
    lt_multi_destroy(ctx);
    delete ctx;
    return;
  }
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->dOut) cudaFree(ctx->dOut);
  if (ctx->dCounters) cudaFree(ctx->dCounters);
  if (ctx->dWork) cudaFree(ctx->dWork);
  if (ctx->wfWorkspace) cudaFree(ctx->wfWorkspace);
  if (ctx->dCamera) cudaFree(ctx->dCamera);
  if (ctx->dSample) cudaFree(ctx->dSample);
  if (ctx->dViews) cudaFree(ctx->dViews);
  if (ctx->dViewFrameCounts) cudaFree(ctx->dViewFrameCounts);
  delete ctx->copyPool;
  if (ctx->stage) cudaFreeHost(ctx->stage);
  for (cudaEvent_t e : ctx->stageEvents) cudaEventDestroy(e);
  for (LtPlugin* p : ctx->plugins) lt_plugin_free(p);
  for (cudaEvent_t e : ctx->traceEvents) cudaEventDestroy(e);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->wfAux.extra) {
    cudaStreamSynchronize(ctx->wfAux.extra);
    cudaStreamDestroy(ctx->wfAux.extra);
  }
  if (ctx->wfAux.fork) cudaEventDestroy(ctx->wfAux.fork);
  for (cudaEvent_t e : ctx->wfAux.order)
    if (e) cudaEventDestroy(e);
  if (ctx->ownStream) cudaStreamDestroy(ctx->ownStream);
  delete ctx;
}

extern "C" int lt_ctx_set_stream(lt_ctx* ctx, void* cuda_stream) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_ctx_set_stream: ctx is NULL");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_ctx_set_stream: a multi-GPU context renders on its own per-device streams");
  ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->ownStream;
  return LT_OK;
}

// Host-side validation of the reference node array (bounds of every index the kernels will
// follow) and the depth the traversal stack needs.
static int validate_tree(const RefNode* nodes, int nodeCount, int primCount, int* stackDepth, std::string* why) {
  std::vector<std::pair<int, int>> todo;  // (node, number of inner ancestors)
  todo.reserve(128);
  todo.push_back({0, 0});
  long long visited = 0;
  int maxInner = 0;
  while (!todo.empty()) {
    std::pair<int, int> cur = todo.back();
    todo.pop_back();
    int i = cur.first, d = cur.second;
    if (++visited > nodeCount) { *why = "node array is not a tree (cycle or shared child)"; return -1; }
    const RefNode& n = nodes[i];
    if (n.primitiveCount > 0) {
      if (n.offset < 0 || n.offset >= primCount) { *why = "leaf primitivesOffset out of range"; return -1; }
    } else {
      if (i + 1 >= nodeCount || n.offset <= i + 1 || n.offset >= nodeCount) {
        *why = "inner node child index out of range";
        return -1;
      }
      if (n.axis > 2) { *why = "inner node axis > 2"; return -1; }
      if (d + 1 > maxInner) maxInner = d + 1;
      todo.push_back({n.offset, d + 1});
      todo.push_back({i + 1, d + 1});
    }
  }
  // every array entry must belong to the tree: the re-flatten kernels process all nodeCount entries and size their
  // output from the full-binary-tree count, so an unreachable entry would be followed unvalidated
  if (visited != nodeCount) { *why = "node array has entries that are not reachable from the root"; return -1; }
  *stackDepth = maxInner;
  return 0;
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
  cudaFree(s->dNodes);
  cudaFree(s->dPrims);
  cudaFree(s->dMats);
  cudaFree(s->dLights);
  cudaFree(s->dWide);
  cudaFree(s->dTris);
  cudaFree(s->dThread);
  cudaFree(s->dRank);
  cudaFree(s->dThreadBig);
  cudaFree(s->dRefit);
  delete s;
}

// Threaded form of the tree (LtThreadNode, lens_trace_b200_device.cuh): eight copies of the node array, copy o in
// the order the reference's traversal visits the nodes for rays of sign octant o, then eight pruned copies.  Built
// on the host, for small trees only (lt_plan_threaded_copies).

// The order in which the reference's traversal visits the nodes for rays of sign octant o (bit k: negative direction
// on axis k), whole tree, no culling.
static void visit_order(const RefNode* nodes, int o, std::vector<int>& order) {
  std::vector<int> stack(1, 0);
  order.clear();
  while (!stack.empty()) {
    int i = stack.back();
    stack.pop_back();
    order.push_back(i);
    const RefNode& r = nodes[i];
    if (r.primitiveCount == 0) {
      bool neg = (o >> r.axis) & 1;  // basic.cu:180-186: second child first when the direction is negative
      int nearC = neg ? r.offset : i + 1, farC = neg ? i + 1 : r.offset;
      stack.push_back(farC);
      stack.push_back(nearC);
    }
  }
}

// Appends eight copies of the threaded form to `out`, each in the visit order of its sign octant, leaving out the
// nodes with keep[i] == 0.  Copy o is records [base + o * stride, base + (o + 1) * stride), base = out.size() on
// entry, stride = the number of kept nodes; skip links are absolute record indices.  A link to a left-out node goes
// to the first kept record after it in the visit order (its first child, or that child's first child ...).
// Returns the stride.
static int append_threaded(const RefNode* nodes, int n, const std::vector<char>& keep, std::vector<LtThreadNode>& out) {
  const int base = (int)out.size();
  int stride = 0;
  for (char k : keep) stride += k ? 1 : 0;
  out.resize((size_t)base + 8 * (size_t)stride);
  std::vector<int> size(n), order, before(n + 1);
  for (int i = n - 1; i >= 0; i--)  // children follow their parent in the depth-first array
    size[i] = nodes[i].primitiveCount > 0 ? 1 : 1 + size[i + 1] + size[nodes[i].offset];
  auto bitsf = [](int v) { float f; memcpy(&f, &v, 4); return f; };
  for (int o = 0; o < 8; o++) {
    visit_order(nodes, o, order);
    // before[p]: kept nodes among the first p of the visit order = copy index of the first kept record at or after p
    // (every position has one: leaves are always kept, and a left-out node is followed by its subtree)
    for (int p = 0; p < n; p++) before[p + 1] = before[p] + (keep[order[p]] ? 1 : 0);
    const int copy = base + o * stride;
    for (int p = 0; p < n; p++) {
      const int i = order[p];
      if (!keep[i]) continue;
      const RefNode& r = nodes[i];
      const bool leaf = r.primitiveCount > 0;
      const float* lo[3];
      const float* hi[3];
      for (int k = 0; k < 3; k++) {
        bool neg = (o >> k) & 1;
        lo[k] = neg ? r.boundsMax : r.boundsMin;
        hi[k] = neg ? r.boundsMin : r.boundsMax;
      }
      const int end = p + size[i];
      const int skip = end >= n ? LT_DONE : copy + before[end];
      LtThreadNode& t = out[(size_t)copy + before[p]];
      t.a = make_float4(lo[0][0], lo[1][1], lo[2][2], hi[0][0]);
      t.b = make_float4(hi[1][1], hi[2][2], bitsf(leaf ? ~r.offset : 0), bitsf(skip));
    }
  }
  return stride;
}

// Nodes of the pruned copies.  Every builder here makes an inner box the exact min/max of its primitives, so a child
// box lies inside its parent box.  For a ray with finite, nonzero direction reciprocals and a finite origin,
// (b - o) * inv in round-to-nearest is monotonic in the bound b, so a contained child's entry is at least its
// parent's and its exit at most the parent's: a child is hit only if its parent is.  An inner node m whose two
// children lie inside its box can therefore be left out of the visit sequence.  If m would be hit, the walk goes on
// to its first child anyway.  If m would be missed, every record below it misses until a kept one misses, through the
// chain of left-out nodes, and the walk reaches m's old skip target.  Either way the same leaves are recorded in the
// same order.
// Leaving m out saves 2 p(m) - p(a) box tests per ray, p = probability that a box is hit and a = the nearest kept
// ancestor, so m goes when a ray that enters a usually enters m as well: surface area SA(m) > SA(a) / 2.  Box tests
// per ray (reference traversal order, no any-hit early exit, root excluded) for the GI kernel on the Cornell box
// (480x270, frames 0-1, depth 4, the 766 767 rays of an instrumented oracle): 26.70 with the full copies, 19.57 with
// this rule, 18.13 with per-node hit counts measured on those rays in place of the areas (an upper bound: it needs
// ray statistics); tools/threaded_prune_counts.py recounts the rule on a stand-in stream.  Leaves stay: a leaf box
// gates a triangle test, and a triangle can be hit a rounding step outside its box.  The rule does not depend on the
// octant, so all eight pruned copies have one length.  A tree that breaks containment (or has NaN or inverted
// bounds) keeps the records where it does; the comparisons below are false for NaN.
//
// Cost of the pruned walk: a kept record is tested exactly when the ray hits its nearest kept ancestor's box (the
// left-out nodes between them decide nothing), so the expected box tests per ray that hits the root are
// sum over kept records r != root of SA(keptAncestor(r)) / SA(root) -- the root's own test comes from the kernel
// parameters.  *cost receives it.  The octant changes neither the records nor the stride.
static double half_area(const float* mn, const float* mx) {
  double dx = (double)mx[0] - mn[0], dy = (double)mx[1] - mn[1], dz = (double)mx[2] - mn[2];
  return dx * dy + dy * dz + dz * dx;
}

// The rule above for a node m whose children lie inside its box, a = its nearest kept ancestor: leave m out.
static bool prune_contained(double areaM, double areaA) { return areaM > 0.5 * areaA; }

static std::vector<char> pruned_keep(const RefNode* nodes, int n, double* cost = nullptr) {
  std::vector<char> keep(n, 1);
  std::vector<int> anc(n, 0);  // nearest kept ancestor
  auto inside = [](const RefNode& c, const RefNode& m) {
    for (int k = 0; k < 3; k++)
      if (!(m.boundsMin[k] <= c.boundsMin[k] && c.boundsMin[k] <= c.boundsMax[k] && c.boundsMax[k] <= m.boundsMax[k]))
        return false;
    return true;
  };
  auto area = [](const RefNode& r) { return half_area(r.boundsMin, r.boundsMax); };
  for (int i = 0; i < n; i++) {  // parents precede their children in the depth-first array
    const RefNode& m = nodes[i];
    if (m.primitiveCount > 0) continue;
    if (i > 0)
      keep[i] = !(inside(nodes[i + 1], m) && inside(nodes[m.offset], m) &&
                  prune_contained(area(m), area(nodes[anc[i]])));
    anc[i + 1] = anc[m.offset] = keep[i] ? i : anc[i];
  }
  if (cost) {
    double sum = 0.0;
    for (int i = 1; i < n; i++)
      if (keep[i]) sum += area(nodes[anc[i]]);
    const double root = area(nodes[0]);
    *cost = root > 0.0 ? sum / root : sum;
  }
  return keep;
}

// Traversal tree (LtThreadNode).  By the argument above, applied to every ancestor of a leaf L, the reference reaches
// L exactly when L's own box is hit, provided L's box lies inside all its ancestors' boxes: which leaves a ray reaches
// is a property of the leaf boxes alone.  Any tree over the same leaves with containing inner boxes reaches the same
// ones and changes only the order of the triangle tests; the reference's result is the least (t, rank), rank = the
// leaf's position in the reference's visit order of the ray's octant (tri_test).  NaN t is never accepted, t == tInit
// without a hit stays rejected, and an any-hit ray only asks whether some reached triangle is accepted.
//
// Whether the reference's leaves allow one: every leaf box inside each of its ancestors' boxes, all bounds finite
// with lo <= hi (the builder below sorts centroids and sums areas), no primitive linked by two leaves (a rank per
// primitive), an inner root.  The tie-break table (8 ints per primitive) may take at most as much memory as the
// threaded copies (16 records per node): a small tree over a huge primitive array keeps the reference's copies.
static bool leaves_decide_reach(const RefNode* nodes, int n, int primCount) {
  if (n < 3 || nodes[0].primitiveCount > 0 || (long long)primCount > 16ll * n) return false;
  // lo, hi of node i: the intersection of its ancestors' boxes
  std::vector<float> lo((size_t)n * 3, -INFINITY), hi((size_t)n * 3, INFINITY);
  std::vector<char> linked((size_t)primCount, 0);
  for (int i = 0; i < n; i++) {  // parents precede their children in the depth-first array
    const RefNode& r = nodes[i];
    for (int k = 0; k < 3; k++)
      if (!(std::isfinite(r.boundsMin[k]) && std::isfinite(r.boundsMax[k]) && r.boundsMin[k] <= r.boundsMax[k]))
        return false;
    if (r.primitiveCount > 0) {
      for (int k = 0; k < 3; k++)
        if (r.boundsMin[k] < lo[(size_t)i * 3 + k] || r.boundsMax[k] > hi[(size_t)i * 3 + k]) return false;
      if (linked[r.offset]) return false;
      linked[r.offset] = 1;
      continue;
    }
    for (int c : {i + 1, r.offset})
      for (int k = 0; k < 3; k++) {
        lo[(size_t)c * 3 + k] = std::max(lo[(size_t)i * 3 + k], r.boundsMin[k]);
        hi[(size_t)c * 3 + k] = std::min(hi[(size_t)i * 3 + k], r.boundsMax[k]);
      }
  }
  return true;
}

// The traversal tree's builders share one form: a binary tree over the reference's leaf records.  Node j < m is leaf
// ordinal j (the j-th leaf of the reference's array), inner nodes follow, kid[0] = -1 for a leaf.  A leaf's box is its
// record's; an inner node's box is the exact float min/max of its children's, so every child lies inside its parent.
struct LeafTree {
  struct Node {
    int kid[2];
    float mn[3], mx[3];
  };
  std::vector<Node> node;
  int root = 0;

  LeafTree(const RefNode* nodes, const std::vector<int>& leaf) : node(leaf.size()) {
    node.reserve(2 * leaf.size() - 1);
    for (size_t j = 0; j < leaf.size(); j++) {
      node[j].kid[0] = node[j].kid[1] = -1;
      memcpy(node[j].mn, nodes[leaf[j]].boundsMin, sizeof node[j].mn);
      memcpy(node[j].mx, nodes[leaf[j]].boundsMax, sizeof node[j].mx);
    }
  }
  void fit(int i) {
    const Node &a = node[node[i].kid[0]], &b = node[node[i].kid[1]];
    for (int k = 0; k < 3; k++) {
      node[i].mn[k] = std::min(a.mn[k], b.mn[k]);
      node[i].mx[k] = std::max(a.mx[k], b.mx[k]);
    }
  }
  int join(int a, int b) {
    node.push_back(Node{{a, b}, {}, {}});
    fit((int)node.size() - 1);
    return (int)node.size() - 1;
  }
  double area(int i) const { return half_area(node[i].mn, node[i].mx); }
  // every node, children before their parent
  std::vector<int> postorder() const {
    std::vector<int> order, stack(1, root);
    while (!stack.empty()) {
      const int i = stack.back();
      stack.pop_back();
      order.push_back(i);
      if (node[i].kid[0] >= 0) {
        stack.push_back(node[i].kid[0]);
        stack.push_back(node[i].kid[1]);
      }
    }
    std::reverse(order.begin(), order.end());
    return order;
  }
};

// (a) SAH sweep: every split is a full sweep over the leaf-box centroids on each axis, minimising
// SA(first) * leaves(first) + SA(second) * leaves(second).
static LeafTree sah_leaf_tree(const RefNode* nodes, const std::vector<int>& leaf) {
  LeafTree t(nodes, leaf);
  const int m = (int)leaf.size();
  std::vector<double> cen((size_t)m * 3);
  for (int j = 0; j < m; j++)
    for (int k = 0; k < 3; k++) cen[(size_t)j * 3 + k] = (double)t.node[j].mn[k] + t.node[j].mx[k];
  std::vector<int> item(m);
  for (int j = 0; j < m; j++) item[j] = j;
  std::vector<double> secondCost(m);
  struct Box {
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    void grow(const LeafTree::Node& r) {
      for (int k = 0; k < 3; k++) {
        mn[k] = std::min(mn[k], r.mn[k]);
        mx[k] = std::max(mx[k], r.mx[k]);
      }
    }
    double area() const { return half_area(mn, mx); }
  };
  struct Task { int begin, end, parent, side; };
  std::vector<Task> todo = {{0, m, -1, 0}};
  while (!todo.empty()) {
    const Task tk = todo.back();
    todo.pop_back();
    const int b = tk.begin, e = tk.end;
    int id = item[b];
    if (e - b > 1) {
      int bestAxis = 0, bestCut = b + 1;
      double bestCost = INFINITY;
      for (int k = 0; k < 3; k++) {
        std::sort(item.begin() + b, item.begin() + e, [&](int x, int y) {
          double cx = cen[(size_t)x * 3 + k], cy = cen[(size_t)y * 3 + k];
          return cx < cy || (cx == cy && x < y);
        });
        Box second, first;
        for (int j = e - 1; j > b; j--) {
          second.grow(t.node[item[j]]);
          secondCost[j] = second.area() * (e - j);
        }
        for (int j = b + 1; j < e; j++) {  // cut j: first child [b, j), second [j, e)
          first.grow(t.node[item[j - 1]]);
          const double cost = first.area() * (j - b) + secondCost[j];
          if (cost < bestCost) {
            bestCost = cost;
            bestAxis = k;
            bestCut = j;
          }
        }
      }
      if (bestAxis != 2)
        std::sort(item.begin() + b, item.begin() + e, [&](int x, int y) {
          double cx = cen[(size_t)x * 3 + bestAxis], cy = cen[(size_t)y * 3 + bestAxis];
          return cx < cy || (cx == cy && x < y);
        });
      id = (int)t.node.size();
      t.node.push_back(LeafTree::Node{{-1, -1}, {}, {}});
      todo.push_back({bestCut, e, id, 1});
      todo.push_back({b, bestCut, id, 0});
    }
    if (tk.parent >= 0)
      t.node[tk.parent].kid[tk.side] = id;
    else
      t.root = id;
  }
  for (int i = (int)t.node.size() - 1; i >= m; i--) t.fit(i);  // inner children come after their parent
  return t;
}

// (b) PLOC over the leaf boxes, as lt_bvh.cu builds it over primitive boxes: clusters in the Morton order of their
// centroids (21 bits per axis over the centroids' bounds, stable), each one's nearest neighbour within kPlocRadius
// positions by the float half-area of the union, ties by (pair hash, lower position, higher position); mutual
// nearest neighbours merge into the lower position.  The smallest pair key is always mutual, so every round merges.
static LeafTree ploc_leaf_tree(const RefNode* nodes, const std::vector<int>& leaf) {
  constexpr int kPlocRadius = 8;
  LeafTree t(nodes, leaf);
  const int m = (int)leaf.size();
  std::vector<float> c((size_t)m * 3);
  float cmn[3] = {INFINITY, INFINITY, INFINITY}, cmx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int j = 0; j < m; j++)
    for (int k = 0; k < 3; k++) {
      const float v = 0.5f * t.node[j].mn[k] + 0.5f * t.node[j].mx[k];
      c[(size_t)j * 3 + k] = v;
      cmn[k] = std::min(cmn[k], v);
      cmx[k] = std::max(cmx[k], v);
    }
  auto spread21 = [](uint64_t x) {
    x &= 0x1FFFFF;
    x = (x | x << 32) & 0x1F00000000FFFFull;
    x = (x | x << 16) & 0x1F0000FF0000FFull;
    x = (x | x << 8) & 0x100F00F00F00F00Full;
    x = (x | x << 4) & 0x10C30C30C30C30C3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
  };
  std::vector<uint64_t> key(m);
  for (int j = 0; j < m; j++) {
    uint64_t q[3];
    for (int k = 0; k < 3; k++) {
      const float ext = cmx[k] - cmn[k];
      const float u = ext > 0.0f ? (c[(size_t)j * 3 + k] - cmn[k]) / ext : 0.0f;
      q[k] = (uint64_t)std::min(std::max(u * 2097152.0f, 0.0f), 2097151.0f);
    }
    key[j] = spread21(q[0]) << 2 | spread21(q[1]) << 1 | spread21(q[2]);
  }
  std::vector<int> cl(m);  // cluster at each position -> tree node
  for (int j = 0; j < m; j++) cl[j] = j;
  std::stable_sort(cl.begin(), cl.end(), [&](int x, int y) { return key[x] < key[y]; });
  auto pair_hash = [](uint32_t a, uint32_t b) {
    uint32_t h = a ^ (b * 0x9E3779B9u);
    h ^= h >> 16;
    h *= 0x85EBCA6Bu;
    h ^= h >> 13;
    h *= 0xC2B2AE35u;
    h ^= h >> 16;
    return h;
  };
  std::vector<int> nn(m), next;
  while (cl.size() > 1) {
    const int cnt = (int)cl.size();
    for (int i = 0; i < cnt; i++) {
      uint32_t bd = 0, bh = 0;
      int ba = 0, bb = 0, best = -1;
      for (int j = std::max(0, i - kPlocRadius); j <= std::min(cnt - 1, i + kPlocRadius); j++) {
        if (j == i) continue;
        const LeafTree::Node &p = t.node[cl[i]], &q = t.node[cl[j]];
        float e[3];
        for (int k = 0; k < 3; k++) e[k] = std::max(p.mx[k], q.mx[k]) - std::min(p.mn[k], q.mn[k]);
        const float area = (e[0] * e[1] + e[1] * e[2]) + e[2] * e[0];
        uint32_t d;
        memcpy(&d, &area, 4);
        const int a = std::min(i, j), b = std::max(i, j);
        const uint32_t h = pair_hash((uint32_t)a, (uint32_t)b);
        if (best < 0 || d < bd || (d == bd && (h < bh || (h == bh && (a < ba || (a == ba && b < bb)))))) {
          best = j;
          bd = d;
          bh = h;
          ba = a;
          bb = b;
        }
      }
      nn[i] = best;
    }
    next.clear();
    for (int i = 0; i < cnt; i++) {
      const int j = nn[i];
      if (nn[j] != i)
        next.push_back(cl[i]);
      else if (i < j)
        next.push_back(t.join(cl[i], cl[j]));
    }
    cl.swap(next);
  }
  t.root = cl[0];
  return t;
}

// (c) Treelet restructuring (Karras & Aila, "Fast Parallel Construction of High-Quality Bounding Volume
// Hierarchies", HPG 2013) with the pruned walk's cost as the objective.  One pass visits every inner node x, children
// before parents, grows a treelet below x to kTreeletLeaves leaves by expanding its largest inner leaf, and replaces
// the treelet by the topology over the same leaves with the least cost, found exhaustively by dynamic programming
// over leaf sets.  The cost is not a plain SAH: a node's keep decision and test probability depend on the area of its
// nearest kept ancestor, so a leaf set's optimum is taken per ancestor (x's own nearest kept ancestor, or any larger
// leaf set of the treelet), and the subtrees hanging below the treelet are costed by walking them down to their kept
// nodes, whose subtree costs `g` are kept up to date.  The box of x, and so everything outside the treelet, does not
// change, and every accepted treelet lowers the cost, so the build may stop after any treelet: at the end of a pass
// that improved none, or once its work (node walks and split evaluations) exceeds the budget it is given.
class TreeletRestructure {
 public:
  static constexpr int kTreeletLeaves = 7, kSets = 1 << kTreeletLeaves;

  TreeletRestructure(LeafTree& t, long long budget)
      : t_(t), area_(t.node.size()), g_(t.node.size()), budget_(budget),
        memo_((size_t)kSets * kSets), choice_((size_t)kSets * kSets), stamp_((size_t)kSets * kSets, 0),
        leafMemo_((size_t)kTreeletLeaves * kSets), leafStamp_((size_t)kTreeletLeaves * kSets, 0) {
    for (size_t i = 0; i < t.node.size(); i++) area_[i] = t.area((int)i);
    for (int x : t.postorder())
      if (t.node[x].kid[0] >= 0) regain(x);
  }

  // One bottom-up pass; whether some treelet improved.
  bool pass() {
    bool improved = false;
    struct Frame { int x; double a; bool down; };  // a: area of x's nearest kept ancestor
    std::vector<Frame> st = {{t_.root, 0.0, true}};
    while (!st.empty() && work_ <= budget_) {
      const Frame f = st.back();
      if (!f.down) {
        st.pop_back();
        improved |= treelet(f.x, f.a);
        continue;
      }
      const int k0 = t_.node[f.x].kid[0], k1 = t_.node[f.x].kid[1];
      if (k0 < 0) {
        st.pop_back();
        continue;
      }
      st.back().down = false;
      const double a = kept_area(f.x, f.a);
      st.push_back({k1, a, true});
      st.push_back({k0, a, true});
    }
    return improved;
  }
  bool exhausted() const { return work_ > budget_; }

 private:
  // the area that x's children see as their nearest kept ancestor's, when x's own is `a` (the root is always kept)
  double kept_area(int x, double a) const {
    return x == t_.root || !prune_contained(area_[x], a) ? area_[x] : a;
  }

  // cost of the records of x's subtree, x included, when x's nearest kept ancestor has area a
  double below(int x, double a) {
    double s = 0.0;
    walk_.assign(1, x);
    while (!walk_.empty()) {
      const int y = walk_.back();
      walk_.pop_back();
      work_++;
      const LeafTree::Node& nd = t_.node[y];
      if (nd.kid[0] >= 0 && prune_contained(area_[y], a)) {
        walk_.push_back(nd.kid[1]);
        walk_.push_back(nd.kid[0]);
      } else {
        s += a + (nd.kid[0] >= 0 ? g_[y] : 0.0);
      }
    }
    return s;
  }
  // g: cost of x's subtree below x when x is kept
  void regain(int x) { g_[x] = below(t_.node[x].kid[0], area_[x]) + below(t_.node[x].kid[1], area_[x]); }

  double set_area(int s) const { return s == full_ ? rootA_ : sarea_[s]; }  // full_: x's children's kept ancestor

  double leaf_cost(int s, int a) {
    const int j = __builtin_ctz(s);
    const size_t i = (size_t)j * kSets + a;
    if (leafStamp_[i] != gen_) {
      leafStamp_[i] = gen_;
      leafMemo_[i] = below(lv_[j], set_area(a));
    }
    return leafMemo_[i];
  }

  // least cost of a subtree over leaf set s (two or more leaves) below the children of the best split, given the
  // kept ancestor set a; *part receives that split's part holding s's lowest leaf
  double split(int s, int a, int* part) {
    const int low = s & -s;
    double best = INFINITY;
    for (int p = (s - 1) & s; p; p = (p - 1) & s) {
      if (!(p & low)) continue;
      work_++;
      const double c = opt(p, a) + opt(s ^ p, a);
      if (c < best) {
        best = c;
        *part = p;
      }
    }
    return best;
  }

  // least cost of a subtree over leaf set s whose nearest kept ancestor is set a
  double opt(int s, int a) {
    if (!(s & (s - 1))) return leaf_cost(s, a);
    const size_t i = (size_t)s * kSets + a;
    if (stamp_[i] != gen_) {
      const bool pruned = prune_contained(sarea_[s], set_area(a));
      stamp_[i] = gen_;
      memo_[i] = (pruned ? 0.0 : set_area(a)) + split(s, pruned ? a : s, &choice_[i]);
    }
    return memo_[i];
  }

  int mask_of(int x) const {
    for (int j = 0; j < nl_; j++)
      if (lv_[j] == x) return 1 << j;
    return mask_of(t_.node[x].kid[0]) | mask_of(t_.node[x].kid[1]);
  }

  // the same cost for the treelet's current topology below node x (leaf set s)
  double current(int x, int s, int a) {
    if (!(s & (s - 1))) return leaf_cost(s, a);
    const bool pruned = prune_contained(sarea_[s], set_area(a));
    return (pruned ? 0.0 : set_area(a)) + current_split(x, s, pruned ? a : s);
  }
  double current_split(int x, int s, int a) {
    const int k0 = t_.node[x].kid[0], k1 = t_.node[x].kid[1], s0 = mask_of(k0);
    const bool first0 = (s0 & s & -s) != 0;
    const double c0 = current(k0, s0, a), c1 = current(k1, s ^ s0, a);
    return first0 ? c0 + c1 : c1 + c0;
  }

  // rebuilds leaf set s with the optimum's splits on the treelet's inner nodes; returns its node
  int rebuild(int s, int a, int* next) {
    if (!(s & (s - 1))) return lv_[__builtin_ctz(s)];
    const size_t i = (size_t)s * kSets + a;
    const int cs = prune_contained(sarea_[s], set_area(a)) ? a : s;
    const int x = in_[(*next)++];
    const int k0 = rebuild(choice_[i], cs, next), k1 = rebuild(s ^ choice_[i], cs, next);
    t_.node[x].kid[0] = k0;
    t_.node[x].kid[1] = k1;
    t_.fit(x);
    area_[x] = t_.area(x);
    regain(x);
    return x;
  }

  bool treelet(int x, double a) {
    in_[0] = x;
    lv_[0] = t_.node[x].kid[0];
    lv_[1] = t_.node[x].kid[1];
    int ni = 1;
    nl_ = 2;
    while (nl_ < kTreeletLeaves) {
      int k = -1;
      for (int j = 0; j < nl_; j++)
        if (t_.node[lv_[j]].kid[0] >= 0 && (k < 0 || area_[lv_[j]] > area_[lv_[k]])) k = j;
      if (k < 0) break;
      in_[ni++] = lv_[k];
      lv_[nl_++] = t_.node[lv_[k]].kid[1];
      lv_[k] = t_.node[lv_[k]].kid[0];
    }
    bool improved = false;
    if (nl_ >= 3) {
      full_ = (1 << nl_) - 1;
      rootA_ = kept_area(x, a);
      gen_++;
      for (int s = 1; s <= full_; s++) {
        const int low = s & -s;
        if (s == low) {
          const LeafTree::Node& nd = t_.node[lv_[__builtin_ctz(s)]];
          memcpy(smn_[s], nd.mn, sizeof smn_[s]);
          memcpy(smx_[s], nd.mx, sizeof smx_[s]);
        } else {
          for (int k = 0; k < 3; k++) {
            smn_[s][k] = std::min(smn_[low][k], smn_[s ^ low][k]);
            smx_[s][k] = std::max(smx_[low][k], smx_[s ^ low][k]);
          }
        }
        sarea_[s] = half_area(smn_[s], smx_[s]);
      }
      const double now = current_split(x, full_, full_);
      int p = 0;
      const double best = split(full_, full_, &p);
      if (best < now - 1e-9 * now) {
        int next = 1;
        const int k0 = rebuild(p, full_, &next), k1 = rebuild(full_ ^ p, full_, &next);
        t_.node[x].kid[0] = k0;
        t_.node[x].kid[1] = k1;
        improved = true;
      }
    }
    regain(x);  // the subtrees below may have changed since x's g was last computed
    return improved;
  }

  LeafTree& t_;
  std::vector<double> area_, g_;
  long long work_ = 0, budget_;
  std::vector<int> walk_;
  // the current treelet: leaves, inner nodes (in_[0] = its root), leaf sets' boxes and areas
  int lv_[kTreeletLeaves], in_[kTreeletLeaves - 1], nl_ = 0, full_ = 0;
  double rootA_ = 0.0, sarea_[kSets];
  float smn_[kSets][3], smx_[kSets][3];
  // opt() per (leaf set, kept ancestor set), valid when stamp_ == gen_
  std::vector<double> memo_;
  std::vector<int> choice_, stamp_;
  std::vector<double> leafMemo_;
  std::vector<int> leafStamp_;
  int gen_ = 0;
};

// A leaf tree in the reference's depth-first layout, each leaf record copied as it is: its box gates its triangle
// test, and a multi-primitive leaf's box may be larger than the one triangle it tests.  `axis` is the axis on which
// the two children's box centroids lie farthest apart, the child with the lower centroid on it first (the child with
// the lower leaf ordinal when they are equal), as lt_bvh.cu orders PLOC's merges.  n = 2 m - 1 nodes again.
static std::vector<RefNode> emit_leaf_tree(const RefNode* nodes, const std::vector<int>& leaf, const LeafTree& t) {
  const int m = (int)leaf.size();
  std::vector<int> low(t.node.size());  // lowest leaf ordinal below each node
  for (int i : t.postorder())
    low[i] = t.node[i].kid[0] < 0 ? i : std::min(low[t.node[i].kid[0]], low[t.node[i].kid[1]]);
  std::vector<RefNode> out((size_t)(2 * m - 1));
  struct Task { int node, parent; };  // parent >= 0: this node is the second child of out[parent]
  std::vector<Task> todo = {{t.root, -1}};
  int next = 0;
  while (!todo.empty()) {
    const Task tk = todo.back();
    todo.pop_back();
    const int idx = next++;
    if (tk.parent >= 0) out[tk.parent].offset = idx;
    const LeafTree::Node& nd = t.node[tk.node];
    if (nd.kid[0] < 0) {
      out[idx] = nodes[leaf[tk.node]];
      continue;
    }
    const LeafTree::Node &a = t.node[nd.kid[0]], &b = t.node[nd.kid[1]];
    double d[3];
    int axis = 0;
    for (int k = 0; k < 3; k++) {
      d[k] = ((double)b.mn[k] + b.mx[k]) - ((double)a.mn[k] + a.mx[k]);
      if (std::fabs(d[k]) > std::fabs(d[axis])) axis = k;
    }
    const bool swap = d[axis] < 0.0 || (d[axis] == 0.0 && low[nd.kid[1]] < low[nd.kid[0]]);
    RefNode& r = out[idx];
    memset(&r, 0, sizeof r);
    memcpy(r.boundsMin, nd.mn, sizeof r.boundsMin);
    memcpy(r.boundsMax, nd.mx, sizeof r.boundsMax);
    r.axis = (uint8_t)axis;
    todo.push_back({nd.kid[swap ? 0 : 1], idx});  // second child, placed after the whole first subtree
    todo.push_back({nd.kid[swap ? 1 : 0], -1});   // first child: the next node, idx + 1
  }
  return out;
}

// The traversal tree: of (a) the SAH sweep tree, (b) the PLOC tree and (c) the better of the two after treelet
// restructuring, the one whose pruned copies cost the least (pruned_keep), the earlier one on equal cost.  costs
// (optional) receives the three costs.  Cornell box: 16.77 / 15.95 / 15.70 (box tests per ray on the stand-in stream of
// tools/threaded_prune_counts.py: SAH sweep 7.30, this tree 6.86); lens scene: 22.73 / 21.57 / 21.34 (11.52, 10.51).
// A pass costs about 330 work units per leaf on ordinary trees, and two or three passes reach the local optimum
// (passes after the third gained less than 0.05 % on a 64 539-node tree), hence at most kMaxPasses passes within
// kRestructureWork units per leaf: on that tree the build takes 0.63 s instead of the SAH tree's 0.19 s (one core of
// an x86-64 server CPU), and the budget bounds it where walks grow long (leaves with equal boxes).
static std::vector<RefNode> build_traversal_tree(const RefNode* nodes, int n, double* costs = nullptr) {
  constexpr int kMaxPasses = 3;
  constexpr long long kRestructureWork = 1024;
  std::vector<int> leaf;  // leaf ordinal -> reference node
  for (int i = 0; i < n; i++)
    if (nodes[i].primitiveCount > 0) leaf.push_back(i);
  auto cost_of = [](const std::vector<RefNode>& r) {
    double c = 0.0;
    pruned_keep(r.data(), (int)r.size(), &c);
    return c;
  };
  const LeafTree sah = sah_leaf_tree(nodes, leaf), ploc = ploc_leaf_tree(nodes, leaf);
  std::vector<RefNode> best = emit_leaf_tree(nodes, leaf, sah), other = emit_leaf_tree(nodes, leaf, ploc);
  const double costSah = cost_of(best), costPloc = cost_of(other);
  LeafTree tuned = costPloc < costSah ? ploc : sah;
  if (costPloc < costSah) best.swap(other);
  TreeletRestructure rs(tuned, kRestructureWork * (long long)leaf.size());
  for (int p = 0; p < kMaxPasses && !rs.exhausted(); p++)
    if (!rs.pass()) break;
  other = emit_leaf_tree(nodes, leaf, tuned);
  const double costTuned = cost_of(other);
  if (costs) {
    costs[0] = costSah;
    costs[1] = costPloc;
    costs[2] = costTuned;
  }
  if (costTuned < std::min(costSah, costPloc)) best.swap(other);
  return best;
}

// rank[o * primCount + p]: the position of the leaf linking primitive p among the leaves of octant o's reference visit
// order (the sequence of append_threaded's copy o).  Primitives no leaf links keep 0: they are never tested.
static std::vector<int> leaf_ranks(const RefNode* nodes, int primCount) {
  std::vector<int> rank((size_t)8 * primCount, 0), order;
  for (int o = 0; o < 8; o++) {
    visit_order(nodes, o, order);
    int pos = 0;
    for (int i : order)
      if (nodes[i].primitiveCount > 0) rank[(size_t)o * primCount + nodes[i].offset] = pos++;
  }
  return rank;
}

// Full copies of the reference tree (records [0, 8 n)), then the pruned copies (from record 8 n): of the traversal
// tree when the reference's leaves decide reach, with its tie-break table in `rank`; otherwise of the reference tree,
// and `rank` empty.  Returns the pruned stride.
static int build_threaded(const RefNode* nodes, int n, int primCount, std::vector<LtThreadNode>& out,
                          std::vector<int>& rank) {
  out.clear();
  rank.clear();
  append_threaded(nodes, n, std::vector<char>(n, 1), out);
  if (!leaves_decide_reach(nodes, n, primCount)) return append_threaded(nodes, n, pruned_keep(nodes, n), out);
  const std::vector<RefNode> trav = build_traversal_tree(nodes, n);
  rank = leaf_ranks(nodes, primCount);
  return append_threaded(trav.data(), (int)trav.size(), pruned_keep(trav.data(), (int)trav.size()), out);
}

static int debug_tree_arg(const void* nodes, uint64_t node_bytes, const char* who, int* n) {
  if (!nodes || node_bytes == 0 || node_bytes % sizeof(RefNode) || node_bytes / sizeof(RefNode) > 0x0fffffffull)
    return fail(nullptr, LT_ERR_INVALID, std::string(who) + ": bad arguments");
  int depth = 0;
  *n = (int)(node_bytes / sizeof(RefNode));
  std::string why;
  if (validate_tree((const RefNode*)nodes, *n, 0x7fffffff, &depth, &why) != 0)
    return fail(nullptr, LT_ERR_INVALID, std::string(who) + ": " + why);
  return LT_OK;
}

extern "C" int lt_debug_build_threaded(const void* nodes, uint64_t node_bytes, void* out_records) {
  int n = 0;
  if (!out_records) return fail(nullptr, LT_ERR_INVALID, "lt_debug_build_threaded: bad arguments");
  if (int rc = debug_tree_arg(nodes, node_bytes, "lt_debug_build_threaded", &n)) return rc;
  std::vector<LtThreadNode> out;
  append_threaded((const RefNode*)nodes, n, std::vector<char>(n, 1), out);
  memcpy(out_records, out.data(), out.size() * sizeof(LtThreadNode));
  return LT_OK;
}

extern "C" int lt_debug_build_threaded_pruned(const void* nodes, uint64_t node_bytes, void* out_records,
                                              int32_t* out_stride) {
  int n = 0;
  if (!out_stride) return fail(nullptr, LT_ERR_INVALID, "lt_debug_build_threaded_pruned: bad arguments");
  if (int rc = debug_tree_arg(nodes, node_bytes, "lt_debug_build_threaded_pruned", &n)) return rc;
  std::vector<LtThreadNode> out;
  *out_stride = append_threaded((const RefNode*)nodes, n, pruned_keep((const RefNode*)nodes, n), out);
  if (out_records) memcpy(out_records, out.data(), out.size() * sizeof(LtThreadNode));
  return LT_OK;
}

// What lt_scene_upload builds for a small tree: out_records (16 n records of room) receives the full copies and then the
// pruned ones, skip links as uploaded (absolute, from record 8 n); out_rank (8 x prim_count ints of room) the
// tie-break table when *out_traversal == 1, i.e. when the pruned copies are a traversal tree.
extern "C" int lt_debug_build_traversal_tree(const void* nodes, uint64_t node_bytes, int32_t prim_count,
                                             void* out_records, int32_t* out_stride, int32_t* out_rank,
                                             int32_t* out_traversal) {
  const char* who = "lt_debug_build_traversal_tree";
  int n = 0;
  if (!out_records || !out_stride || !out_rank || !out_traversal || prim_count < 1)
    return fail(nullptr, LT_ERR_INVALID, std::string(who) + ": bad arguments");
  if (int rc = debug_tree_arg(nodes, node_bytes, who, &n)) return rc;
  const RefNode* r = (const RefNode*)nodes;
  for (int i = 0; i < n; i++)
    if (r[i].primitiveCount > 0 && r[i].offset >= prim_count)
      return fail(nullptr, LT_ERR_INVALID, std::string(who) + ": leaf primitivesOffset out of range");
  std::vector<LtThreadNode> out;
  std::vector<int> rank;
  *out_stride = build_threaded(r, n, prim_count, out, rank);
  *out_traversal = rank.empty() ? 0 : 1;
  memcpy(out_records, out.data(), out.size() * sizeof(LtThreadNode));
  if (!rank.empty()) memcpy(out_rank, rank.data(), rank.size() * sizeof(int));
  return LT_OK;
}

// The traversal tree lt_scene_upload builds for a small tree, in the reference layout, and the costs it is chosen by.
extern "C" int lt_debug_traversal_tree(const void* nodes, uint64_t node_bytes, int32_t prim_count, void* out_nodes,
                                       double* out_costs) {
  const char* who = "lt_debug_traversal_tree";
  int n = 0;
  if (!out_nodes || !out_costs || prim_count < 1) return fail(nullptr, LT_ERR_INVALID, std::string(who) + ": bad arguments");
  if (int rc = debug_tree_arg(nodes, node_bytes, who, &n)) return rc;
  const RefNode* r = (const RefNode*)nodes;
  for (int i = 0; i < n; i++)
    if (r[i].primitiveCount > 0 && r[i].offset >= prim_count)
      return fail(nullptr, LT_ERR_INVALID, std::string(who) + ": leaf primitivesOffset out of range");
  pruned_keep(r, n, &out_costs[0]);
  out_costs[1] = out_costs[2] = out_costs[3] = NAN;
  if (leaves_decide_reach(r, n, prim_count)) {
    const std::vector<RefNode> trav = build_traversal_tree(r, n, out_costs + 1);
    memcpy(out_nodes, trav.data(), trav.size() * sizeof(RefNode));
  }
  return LT_OK;
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
  const bool pruned = s->dThread != nullptr && !full;
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
// makes.  ev0 must already be recorded on the stream; records ev1 and sets upload_ms.
static cudaError_t derive_scene(lt_ctx* ctx, lt_scene* s, const int* dInnerRank, LtTree copies, const RefNode& root) {
  LtSceneDev& d = s->dev;
  const int nNodes = d.nodeCount, nPrims = d.primCount;
  cudaError_t e = cudaSuccess;
  auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  cudaStream_t st = ctx->stream;
  lt_launch_reflatten(s->dNodes, nNodes, s->dPrims, nPrims, dInnerRank, s->dWide, s->dTris, st);
  A(cudaGetLastError());
  std::vector<int> hRank;
  if (e == cudaSuccess && copies == LT_TREE_HOST_THREADED) {
    std::vector<RefNode> hNodes((size_t)nNodes);
    std::vector<LtThreadNode> hThread;
    A(cudaMemcpyAsync(hNodes.data(), s->dNodes, sizeof(RefNode) * (size_t)nNodes, cudaMemcpyDeviceToHost, st));
    A(cudaStreamSynchronize(st));
    if (e == cudaSuccess) {
      s->threadStride = build_threaded(hNodes.data(), nNodes, nPrims, hThread, hRank);
      if (hThread.size() > s->threadRecords) {  // the pruned copies' size follows the boxes
        scene_free(s, &s->dThread, sizeof(LtThreadNode) * s->threadRecords);
        s->threadRecords = 0;
        A(scene_alloc(s, &s->dThread, sizeof(LtThreadNode) * hThread.size()));
        if (e == cudaSuccess) s->threadRecords = hThread.size();
      }
      A(cudaMemcpyAsync(s->dThread, hThread.data(), sizeof(LtThreadNode) * hThread.size(), cudaMemcpyHostToDevice, st));
      if (!hRank.empty()) {
        if (!s->dRank) A(scene_alloc(s, &s->dRank, sizeof(int) * hRank.size()));
        A(cudaMemcpyAsync(s->dRank, hRank.data(), sizeof(int) * hRank.size(), cudaMemcpyHostToDevice, st));
      }
      A(cudaStreamSynchronize(st));  // hThread and hRank are pageable and go out of scope
    }
  }
  // large trees: the threaded copies are built on the device and used by coherent-ray launches only (plan_tree)
  if (e == cudaSuccess && copies == LT_TREE_DEVICE_THREADED) {
    if (!s->dThreadBig && scene_alloc(s, &s->dThreadBig, sizeof(LtThreadNode) * 8 * (size_t)nNodes) != cudaSuccess) {
      cudaGetLastError();  // no memory for the copies: the stack traversal serves every launch
      s->dThreadBig = nullptr;
    }
    if (s->dThreadBig) {
      lt_launch_build_threaded(s->dNodes, nNodes, s->dThreadBig, st);
      A(cudaGetLastError());
    }
  }
  A(cudaEventRecord(ctx->ev1, st));
  A(cudaStreamSynchronize(st));
  if (e != cudaSuccess) return e;
  cudaEventElapsedTime(&ctx->stats.upload_ms, ctx->ev0, ctx->ev1);
  d.wnodes = s->dWide;
  d.tris = s->dTris;
  for (int k = 0; k < 3; k++) {
    d.rootMin[k] = root.boundsMin[k];
    d.rootMax[k] = root.boundsMax[k];
  }
  d.rootRef = root.primitiveCount > 0 ? ~root.offset : 0;  // inner root is wide node 0
  d.rootCount = root.primitiveCount;
  d.tnodes = s->dThread;
  d.rank = hRank.empty() ? nullptr : s->dRank;
  set_pruned_copies(s, false);
  return cudaSuccess;
}

// Allocates the re-flattened buffers, derives them (derive_scene) and fills the device-side scene descriptor.  ev0
// must already be recorded on the stream; on failure the scene is released.
static int finish_scene(lt_ctx* ctx, lt_scene* s, int nNodes, int nPrims, int nMats, const RefNode& root,
                        int stackDepth, const char* who) {
  int* dFlags = nullptr;
  int* dRank = nullptr;
  void* dTemp = nullptr;
  int nInner = (nNodes - 1) / 2;  // a full binary tree with one primitive slot per leaf
  if (nNodes == 1) nInner = 0;
  size_t tempBytes = lt_scan_temp_bytes(nNodes);
  LtSceneDev& d = s->dev;
  d.prims = s->dPrims;
  d.mats = s->dMats;
  d.lights = s->dLights;
  d.stackDepth = stackDepth;
  d.nodeCount = nNodes;
  d.primCount = nPrims;
  d.matCount = nMats;
  cudaError_t e = cudaSuccess;
  auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  cudaStream_t st = ctx->stream;
  A(scene_alloc(s, &s->dWide, sizeof(LtWideNode) * (size_t)(nInner > 0 ? nInner : 1)));
  A(scene_alloc(s, &s->dTris, sizeof(LtTri) * (size_t)nPrims));
  A(cudaMalloc(&dFlags, sizeof(int) * (size_t)nNodes));
  A(cudaMalloc(&dRank, sizeof(int) * (size_t)nNodes));
  A(cudaMalloc(&dTemp, tempBytes ? tempBytes : 16));
  if (e == cudaSuccess) {
    lt_launch_inner_flags(s->dNodes, nNodes, dFlags, st);
    lt_launch_exclusive_scan(dTemp, tempBytes, dFlags, dRank, nNodes, st);
    A(cudaGetLastError());
  }
  if (e == cudaSuccess) A(derive_scene(ctx, s, dRank, lt_plan_threaded_copies(nNodes, ctx->totalMem, ctx->limits), root));
  cudaStreamSynchronize(st);
  cudaFree(dFlags);
  cudaFree(dRank);
  cudaFree(dTemp);
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
  const RefPrim* hPrims = (const RefPrim*)primitives;
  for (uint64_t i = 0; i < nPrims; i++)
    if (hPrims[i].materialIndex < 0 || (uint64_t)hPrims[i].materialIndex >= nMats)
      return fail(ctx, LT_ERR_INVALID, w + "primitive materialIndex out of range");
  // PLOC compares box areas; its progress argument needs every area to be a number
  if (builder == LT_BVH_PLOC)
    for (uint64_t i = 0; i < nPrims; i++)
      for (int k = 0; k < 3; k++)
        if (!std::isfinite(hPrims[i].a[k]) || !std::isfinite(hPrims[i].b[k]) || !std::isfinite(hPrims[i].c[k]))
          return fail(ctx, LT_ERR_INVALID, w + "non-finite vertex coordinate");
  CK(cudaSetDevice(ctx->device));
  int n = (int)nPrims, nNodes = 2 * n - 1;
  lt_scene* s = new lt_scene();
  RefPrim* dInput = nullptr;
  void* scratch = nullptr;
  size_t scratchBytes = lt_bvh_scratch_bytes(n, builder);
  cudaError_t e = cudaSuccess;
  auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  A(scene_alloc(s, &s->dNodes, sizeof(RefNode) * (size_t)nNodes));
  A(scene_alloc(s, &s->dPrims, primitive_bytes));
  A(scene_alloc(s, &s->dMats, material_bytes));
  A(scene_alloc(s, &s->dLights, sizeof(RefLights)));
  A(cudaMalloc(&dInput, primitive_bytes));
  A(cudaMalloc(&scratch, scratchBytes));
  cudaStream_t st = ctx->stream;
  A(cudaEventRecord(ctx->ev0, st));
  A(cudaMemcpyAsync(dInput, primitives, primitive_bytes, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(s->dMats, materials, material_bytes, cudaMemcpyHostToDevice, st));
  int maxDepth = 0, launches = -1;
  if (e == cudaSuccess)
    launches = lt_launch_bvh_build(builder, dInput, n, s->dMats, (int)nMats, s->dNodes, s->dPrims, s->dLights, scratch,
                                   scratchBytes, &maxDepth, st);
  RefNode root;
  memset(&root, 0, sizeof root);
  if (e == cudaSuccess && launches >= 0) A(cudaMemcpy(&root, s->dNodes, sizeof root, cudaMemcpyDeviceToHost));
  cudaFree(dInput);
  cudaFree(scratch);
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
    CK(cudaMemcpy(nodes, scene->dNodes, node_bytes, cudaMemcpyDeviceToHost));
  }
  if (primitives) {
    if (primitive_bytes != sizeof(RefPrim) * (uint64_t)scene->dev.primCount) return fail(ctx, LT_ERR_INVALID, "lt_scene_download: primitive_bytes mismatch");
    CK(cudaMemcpy(primitives, scene->dPrims, primitive_bytes, cudaMemcpyDeviceToHost));
  }
  if (light_container) CK(cudaMemcpy(light_container, scene->dLights, sizeof(RefLights), cudaMemcpyDeviceToHost));
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
  if (validate_tree(hNodes, (int)nNodes, (int)nPrims, &stackDepth, &why) != 0)
    return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: " + why);
  if (stackDepth > 64)
    return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: tree deeper than 64 (the reference's stack, basic.cu:162)");
  for (uint64_t i = 0; i < nPrims; i++)
    if (hPrims[i].materialIndex < 0 || (uint64_t)hPrims[i].materialIndex >= nMats)
      return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: primitive materialIndex out of range");
  if (hLights->count > 64) return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: light count > 64");
  for (uint32_t i = 0; i < 64; i++)
    if (hLights->primitives[i] >= nPrims)
      return fail(ctx, LT_ERR_INVALID, "lt_scene_upload: light primitive index out of range");

  CK(cudaSetDevice(ctx->device));
  lt_scene* s = new lt_scene();
  cudaError_t e = cudaSuccess;
  auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  A(scene_alloc(s, &s->dNodes, node_bytes));
  A(scene_alloc(s, &s->dPrims, primitive_bytes));
  A(scene_alloc(s, &s->dMats, material_bytes ? material_bytes : sizeof(RefMaterial)));
  A(scene_alloc(s, &s->dLights, sizeof(RefLights)));
  cudaStream_t st = ctx->stream;
  A(cudaEventRecord(ctx->ev0, st));
  A(cudaMemcpyAsync(s->dNodes, nodes, node_bytes, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(s->dPrims, primitives, primitive_bytes, cudaMemcpyHostToDevice, st));
  if (material_bytes) A(cudaMemcpyAsync(s->dMats, materials, material_bytes, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(s->dLights, light_container, sizeof(RefLights), cudaMemcpyHostToDevice, st));
  if (e != cudaSuccess) {
    lt_scene_release(ctx, s);
    return fail(ctx, LT_ERR_CUDA, std::string("lt_scene_upload: ") + cudaGetErrorString(e));
  }
  int rc = finish_scene(ctx, s, (int)nNodes, (int)nPrims, (int)nMats, hNodes[0], stackDepth, "lt_scene_upload");
  if (rc != LT_OK) return rc;
  *out_scene = s;
  return LT_OK;
}

// lt_render_params -> the launch descriptor (all of it but the camera), with lt_render's checks; `who` names the entry
// point in error messages
static int launch_from_params(lt_ctx* ctx, const lt_render_params* p, LtLaunch* L, const char* who = "lt_render") {
  const std::string w = std::string(who) + ": ";
  // API version 1 callers pass the struct without its last field (split_mode)
  if (p->struct_size != sizeof(lt_render_params) && p->struct_size != offsetof(lt_render_params, split_mode))
    return fail(ctx, LT_ERR_INVALID, w + "params.struct_size mismatch");
  if (p->kernel < 0 || p->kernel >= LT_KERNEL_COUNT) return fail(ctx, LT_ERR_UNSUPPORTED, w + "unknown kernel id");
  if (p->width <= 0 || p->height <= 0 || p->depth < 3)
    return fail(ctx, LT_ERR_INVALID, w + "width/height must be > 0 and depth >= 3");
  if ((long long)p->width * p->height * p->depth > (1ll << 40)) return fail(ctx, LT_ERR_INVALID, w + "image too large");
  if (p->frames < 1) return fail(ctx, LT_ERR_INVALID, w + "frames must be >= 1");
  if (p->accum_mode < 0 || p->accum_mode > 2) return fail(ctx, LT_ERR_INVALID, w + "bad accum_mode");
  if (p->max_ray_depth < 0 || p->max_ray_depth > 255)
    return fail(ctx, LT_ERR_INVALID, w + "max_ray_depth must be in [0, 255]");
  L->kernel = p->kernel;
  L->kernelMode = p->kernel_mode ? 1 : 0;
  L->width = p->width;
  L->height = p->height;
  L->fullHeight = p->height;
  L->rowBlock = p->height;
  L->rowStride = 1;
  L->rowPhase = 0;
  L->depth = p->depth;
  L->maxRayDepth = p->max_ray_depth;
  L->frames = p->frames;
  L->frameStride = p->frame_stride ? p->frame_stride : 1u;
  L->accumMode = p->accum_mode;
  L->accumWeight = p->accum_weight;
  L->flags = p->flags;
  return LT_OK;
}

static int check_params(lt_ctx* ctx, const lt_scene* scene, const void* camera28, const lt_render_params* p,
                        LtLaunch* L) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_render: ctx is NULL");
  if (!scene || !camera28 || !p) return fail(ctx, LT_ERR_INVALID, "lt_render: NULL argument");
  if (int rc = launch_from_params(ctx, p, L)) return rc;
  memcpy(&L->cam, camera28, sizeof(RefCamera));
  return LT_OK;
}

static LtSceneFacts scene_facts(const lt_scene* s) {
  return {s->dev.nodeCount, s->dev.stackDepth,
          s->dThread ? LT_TREE_HOST_THREADED : (s->dThreadBig ? LT_TREE_DEVICE_THREADED : LT_TREE_CHILD_PAIR)};
}

// the scene as the plan's kernels see it: tnodes = the plan's threaded copies, NULL for the stack traversal
static LtSceneDev scene_for_plan(const lt_scene* s, const LtPlan& plan) {
  LtSceneDev d = s->dev;
  d.tnodes = plan.tree == LT_TREE_HOST_THREADED ? s->dThread
             : plan.tree == LT_TREE_DEVICE_THREADED ? s->dThreadBig : nullptr;
  return d;
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
  if (onDevice) {
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, src) != cudaSuccess ||
        (pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged) || pa.device != ctx->device) {
      cudaGetLastError();
      return fail(ctx, LT_ERR_INVALID, w + "device_primitives is not device memory of the context's device");
    }
    if ((uintptr_t)src % alignof(RefPrim))
      return fail(ctx, LT_ERR_INVALID, w + "device_primitives is not 4-byte aligned");
  }
  // The upload checks only a leaf's first primitive (the reference's leaves test no other, SURVEY H1); the refit reads
  // all of them, so every leaf's range must lie in the primitive buffer.
  if (s->refitLeaves == 0) {
    std::vector<RefNode> hNodes((size_t)n);
    CK(cudaMemcpyAsync(hNodes.data(), s->dNodes, sizeof(RefNode) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    s->refitLeaves = 1;
    for (const RefNode& r : hNodes)
      if (r.primitiveCount > 0 && (long long)r.offset + r.primitiveCount > nPrims) s->refitLeaves = -1;
  }
  if (s->refitLeaves < 0)
    return fail(ctx, LT_ERR_INVALID, w + "a leaf's primitives run past the primitive buffer: the scene cannot be refitted");
  if (!s->dRefit) CK(scene_alloc(s, &s->dRefit, sizeof(int) * (3 * (size_t)n + 1)));
  int *parent = s->dRefit, *flags = parent + n, *rank = flags + n, *bad = rank + n;
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
    if (s->dThread && s->threadRecords < 16 * (size_t)n) {
      CK(cudaStreamSynchronize(st));
      scene_free(s, &s->dThread, sizeof(LtThreadNode) * s->threadRecords);
      s->threadRecords = 0;
      s->dev.tnodes = nullptr;
      CK(scene_alloc(s, &s->dThread, sizeof(LtThreadNode) * 16 * (size_t)n));
      s->threadRecords = 16 * (size_t)n;
    }
    if (s->dThread && !s->dRank) CK(scene_alloc(s, &s->dRank, sizeof(int) * 8 * (size_t)nPrims));
    void* dTemp = nullptr;
    const size_t tempBytes = lt_scan_temp_bytes(n);
    CK(cudaMalloc(&dTemp, tempBytes ? tempBytes : 16));
    lt_launch_refit_parents(s->dNodes, n, parent, st);
    lt_launch_inner_flags(s->dNodes, n, flags, st);
    lt_launch_exclusive_scan(dTemp, tempBytes, flags, rank, n, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    cudaFree(dTemp);
    CK(e);
    s->refitDerived = true;
  }
  CK(cudaEventRecord(ctx->ev0, st));
  CK(cudaMemcpyAsync(s->dPrims, src, sizeof(RefPrim) * (size_t)nPrims,
                     onDevice ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  lt_launch_refit(s->dNodes, n, s->dPrims, parent, flags, st);
  CK(cudaGetLastError());
  RefNode root;
  CK(cudaMemcpyAsync(&root, s->dNodes, sizeof root, cudaMemcpyDeviceToHost, st));
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
  if (hostPrims) {
    for (uint64_t i = 0; i < nPrims; i++)
      if (hostPrims[i].materialIndex < 0 || hostPrims[i].materialIndex >= one->dev.matCount)
        return fail(ctx, LT_ERR_INVALID, w + "primitive materialIndex out of range");
    for (uint64_t i = 0; i < nPrims; i++)
      for (int k = 0; k < 3; k++)
        if (!std::isfinite(hostPrims[i].a[k]) || !std::isfinite(hostPrims[i].b[k]) || !std::isfinite(hostPrims[i].c[k]))
          return fail(ctx, LT_ERR_INVALID, w + "non-finite vertex coordinate");
  }
  return LT_OK;
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

static int debug_plan(const char* who, const lt_render_params* params, int views, uint64_t node_count,
                      int32_t stack_depth, uint64_t total_mem, int32_t sm_count, int64_t* out) {
  if (!params || !out || views < 1 || node_count < 1 || node_count > 0x7fffffffull || sm_count < 1)
    return fail(nullptr, LT_ERR_INVALID, std::string(who) + ": bad arguments");
  LtLaunch L = {};
  if (int rc = launch_from_params(nullptr, params, &L)) return rc;
  const LtLimits lim;
  const LtSceneFacts s = {(int)node_count, stack_depth, lt_plan_threaded_copies((int)node_count, total_mem, lim)};
  const LtPlan p = lt_plan_render(L, s, total_mem, sm_count, lim, views);
  const int64_t v[LT_PLAN_FIELDS] = {p.pipeline, p.tree, p.stats, p.cull, p.batchFrames, p.streams, p.rounds,
                                     p.samplesPerFrame, p.sharedPrimary, p.classify, (int64_t)p.smemStack,
                                     (int64_t)p.smemTrace, p.blocksPerSm, p.grid, (int64_t)p.workspaceBytes};
  memcpy(out, v, sizeof v);
  return p.error != LT_OK ? fail(nullptr, p.error, p.message) : LT_OK;
}

extern "C" int lt_debug_plan(const lt_render_params* params, uint64_t node_count, int32_t stack_depth,
                             uint64_t total_mem, int32_t sm_count, int64_t* out) {
  return debug_plan("lt_debug_plan", params, 1, node_count, stack_depth, total_mem, sm_count, out);
}

extern "C" int lt_debug_plan_views(const lt_render_params* params, int view_count, uint64_t node_count,
                                   int32_t stack_depth, uint64_t total_mem, int32_t sm_count, int64_t* out) {
  return debug_plan("lt_debug_plan_views", params, view_count, node_count, stack_depth, total_mem, sm_count, out);
}

extern "C" int lt_debug_scene_bytes(const lt_scene* scene, uint64_t* out_bytes) {
  if (!scene || !out_bytes) return fail(nullptr, LT_ERR_INVALID, "lt_debug_scene_bytes: NULL argument");
  uint64_t bytes = 0;
  for (const lt_scene* p : scene->parts) bytes += p->deviceBytes;
  *out_bytes = scene->parts.empty() ? scene->deviceBytes : bytes;
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

int lt_internal_ensure_out(lt_ctx* ctx, size_t floats);
static int ensure_out(lt_ctx* ctx, size_t floats) { return lt_internal_ensure_out(ctx, floats); }
int lt_internal_ensure_out(lt_ctx* ctx, size_t floats) {
  if (ctx->outFloats >= floats) return LT_OK;
  if (ctx->dOut) cudaFree(ctx->dOut);
  ctx->dOut = nullptr;
  ctx->outFloats = 0;
  CK(cudaMalloc(&ctx->dOut, floats * sizeof(float)));
  CK(cudaMemsetAsync(ctx->dOut, 0, floats * sizeof(float), ctx->stream));
  ctx->outFloats = floats;
  return LT_OK;
}

// cams: the cameras of a call of several views (viewCount >= 2, view v into dOut + v * W * H * depth); nullptr: L.cam
static int render_common(lt_ctx* ctx, lt_scene* scene, const LtLaunch& L, float* dOut, bool sync,
                         const RefCamera* cams = nullptr, int viewCount = 1) {
  CK(cudaSetDevice(ctx->device));
  LtPlan plan = lt_plan_render(L, scene_facts(scene), ctx->totalMem, ctx->stats.sm_count, ctx->limits, viewCount);
  if (plan.error != LT_OK) return fail(ctx, plan.error, plan.message);
  const bool stats = plan.stats;
  if (stats) CK(cudaMemsetAsync(ctx->dCounters, 0, sizeof(LtCounters), ctx->stream));
  if (plan.pipeline == LT_PIPE_WAVEFRONT && ctx->wfBytes < plan.workspaceBytes) {
    if (ctx->wfWorkspace) cudaFree(ctx->wfWorkspace);
    ctx->wfWorkspace = nullptr;
    ctx->wfBytes = 0;
    if (cudaMalloc(&ctx->wfWorkspace, plan.workspaceBytes) != cudaSuccess) {
      cudaGetLastError();
      if (plan.forced) return fail(ctx, LT_ERR_CUDA, "lt_render: cannot allocate the wavefront workspace");
      // not a fallback to other arithmetic: the megakernel is the same path per pixel
      LtLaunch mega = L;
      mega.flags |= LT_FLAG_MEGAKERNEL;
      plan = lt_plan_render(mega, scene_facts(scene), ctx->totalMem, ctx->stats.sm_count, ctx->limits, viewCount);
    } else {
      ctx->wfBytes = plan.workspaceBytes;
    }
  }
  const bool wavefront = plan.pipeline == LT_PIPE_WAVEFRONT;
  const int kMaxTracePairs = 8192;
  int tracePairs = 0;
  bool timeTrace = wavefront && (sync || stats);
  if (timeTrace && ctx->traceEvents.empty()) {
    ctx->traceEvents.resize(2 * kMaxTracePairs);
    ctx->pairKinds.resize(kMaxTracePairs);
    for (size_t i = 0; i < ctx->traceEvents.size(); i++) cudaEventCreate(&ctx->traceEvents[i]);
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
    if (ctx->viewFrameCountsSize < n) {
      if (ctx->dViewFrameCounts) cudaFree(ctx->dViewFrameCounts);
      ctx->dViewFrameCounts = nullptr;
      ctx->viewFrameCountsSize = 0;
      CK(cudaMalloc(&ctx->dViewFrameCounts, n * sizeof(unsigned)));
      ctx->viewFrameCountsSize = n;
    }
    // pageable source: staged before the call returns, so fc may go
    CK(cudaMemcpyAsync(ctx->dViewFrameCounts, fc.data(), n * sizeof(unsigned), cudaMemcpyHostToDevice, ctx->stream));
    views.dFrameCounts = ctx->dViewFrameCounts;
  }
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  int launches = 0;
  if (wavefront) {
    launches = lt_launch_render_wavefront(sc, plan, L, dOut, ctx->dCounters, ctx->wfWorkspace, ctx->stats.sm_count,
                                          ctx->stream, timeTrace ? ctx->traceEvents.data() : nullptr, kMaxTracePairs,
                                          &tracePairs, timeKinds ? ctx->pairKinds.data() : nullptr, &ctx->wfAux,
                                          viewCount > 1 ? &views : nullptr);
  } else if (viewCount > 1) {  // the megakernels: one launch per view, back to back on the stream
    for (int v = 0; v < viewCount; v++) {
      LtLaunch Lv = L;
      Lv.cam = cams[v];
      launches += lt_launch_render(sc, plan, Lv, dOut + (size_t)v * L.width * L.height * L.depth, ctx->dCounters,
                                   ctx->dWork, ctx->stream);
    }
  } else {
    launches = lt_launch_render(sc, plan, L, dOut, ctx->dCounters, ctx->dWork, ctx->stream);
  }
  CK(cudaGetLastError());
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->stats.kernel_launches = launches;
  if (sync || stats) {
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaEventElapsedTime(&ctx->stats.kernel_ms, ctx->ev0, ctx->ev1));
    ctx->stats.trace_ms = wavefront ? 0.0f : ctx->stats.kernel_ms;
    ctx->stats.trace_launches = wavefront ? 0 : launches;
    ctx->stats.shade_ms = ctx->stats.primary_shade_ms = ctx->stats.accumulate_ms = 0.0f;
    ctx->stats.shade_launches = 0;
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
  } else {
    ctx->stats.trace_ms = 0.0f;
    ctx->stats.trace_launches = 0;
    ctx->stats.shade_ms = ctx->stats.primary_shade_ms = ctx->stats.accumulate_ms = 0.0f;
    ctx->stats.shade_launches = 0;
  }
  if (stats) {
    LtCounters h;
    CK(cudaMemcpy(&h, ctx->dCounters, sizeof(h), cudaMemcpyDeviceToHost));
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

int lt_internal_render_rows(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                            float* device_out, int fullHeight, int rowBlock, int rowStride, int rowPhase, int sync) {
  LtLaunch L;
  int rc = check_params(ctx, scene, camera28, params, &L);
  if (rc != LT_OK) return rc;
  L.fullHeight = fullHeight;
  L.rowBlock = rowBlock;
  L.rowStride = rowStride;
  L.rowPhase = rowPhase;
  return render_common(ctx, scene, L, device_out, sync != 0);
}

// Result -> the caller's host buffer.  The reference hands render() a malloc'ed (pageable) pOutputBuffer
// (src/cuda/renderer_cuda.cpp:137-139: cuMemcpyDtoH); a plain cudaMemcpy into pageable memory runs at a third of the
// link rate because the driver stages it in small pieces.  Here: pinned or registered destinations get one DMA; a
// pageable destination is filled through the context's own pinned staging buffer in 1 MB chunks -- the DMA of chunk
// k+1 overlaps the host-side copy of chunk k, and the host side is spread over a few threads.  (Registering the
// caller's buffer behind its back is not an option: a cached registration outlives a free()/mmap() of the same
// address range and would then receive the frame in pages the caller no longer sees.)
int lt_internal_download(lt_ctx* ctx, float* host_out, const float* dSrc, size_t bytes);
static int download(lt_ctx* ctx, float* host_out, const float* dSrc, size_t bytes) {
  return lt_internal_download(ctx, host_out, dSrc, bytes);
}
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
    ctx->copyPool = new LtCopyPool(threads - 1);
  }
  if (ctx->stageBytes < (bytes < kMaxStage ? bytes : kMaxStage)) {
    if (ctx->stage) cudaFreeHost(ctx->stage);
    ctx->stage = nullptr;
    ctx->stageBytes = 0;
    size_t want = bytes < kMaxStage ? bytes : kMaxStage;
    want = (want + kChunk - 1) / kChunk * kChunk;
    if (cudaMallocHost(&ctx->stage, want) != cudaSuccess) {  // no pinned memory to be had: the plain copy still works
      cudaGetLastError();
      CK(cudaMemcpyAsync(host_out, dSrc, bytes, cudaMemcpyDeviceToHost, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
      return LT_OK;
    }
    ctx->stageBytes = want;
  }
  for (size_t done = 0; done < bytes;) {  // one pass unless the frame exceeds the staging buffer
    const size_t pass = bytes - done < ctx->stageBytes ? bytes - done : ctx->stageBytes;
    const int chunks = (int)((pass + kChunk - 1) / kChunk);
    while ((int)ctx->stageEvents.size() < chunks) {
      cudaEvent_t e;
      CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      ctx->stageEvents.push_back(e);
    }
    for (int c = 0; c < chunks; c++) {
      const size_t off = (size_t)c * kChunk, n = pass - off < kChunk ? pass - off : kChunk;
      CK(cudaMemcpyAsync(ctx->stage + off, (const char*)dSrc + done + off, n, cudaMemcpyDeviceToHost, ctx->stream));
      CK(cudaEventRecord(ctx->stageEvents[c], ctx->stream));
    }
    // host side: a small pool of copier threads (no CUDA calls in them); this thread waits for the chunks' DMA and
    // publishes how many have landed, then copies along
    LtCopyPool& pool = *ctx->copyPool;
    pool.begin((char*)host_out + done, ctx->stage, pass, kChunk, chunks);
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
  rc = ensure_out(ctx, floats);
  if (rc != LT_OK) return rc;
  rc = render_common(ctx, scene, L, ctx->dOut, true);
  if (rc != LT_OK) return rc;
  if (host_out) return download(ctx, host_out, ctx->dOut, floats * sizeof(float));
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

int lt_internal_render_views(lt_ctx* ctx, lt_scene* scene, const RefCamera* cams, int count,
                             const lt_render_params* params, float* host_out, int hostFirst, int hostStride) {
  LtLaunch L;
  int rc = check_params(ctx, scene, cams, params, &L);
  if (rc != LT_OK) return rc;
  CK(cudaSetDevice(ctx->device));
  const size_t image = (size_t)L.width * L.height * L.depth, floats = image * (size_t)count;
  if (ctx->viewsFloats < floats) {
    if (ctx->dViews) cudaFree(ctx->dViews);
    ctx->dViews = nullptr;
    ctx->viewsFloats = 0;
    CK(cudaMalloc(&ctx->dViews, floats * sizeof(float)));
    ctx->viewsFloats = floats;
  }
  // every view accumulates from zero, as after lt_accum_reset
  CK(cudaMemsetAsync(ctx->dViews, 0, floats * sizeof(float), ctx->stream));
  rc = render_common(ctx, scene, L, ctx->dViews, true, cams, count);
  if (rc != LT_OK || !host_out) return rc;
  if (hostStride == 1) return download(ctx, host_out + (size_t)hostFirst * image, ctx->dViews, floats * sizeof(float));
  for (int k = 0; k < count && rc == LT_OK; k++)
    rc = download(ctx, host_out + (size_t)(hostFirst + (size_t)k * hostStride) * image, ctx->dViews + (size_t)k * image,
                  image * sizeof(float));
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
  return lt_internal_render_views(ctx, scene, cams.data(), view_count, params, host_out, 0, 1);
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
  CK(cudaSetDevice(ctx->device));
  LtPlugin* plugin = ctx->plugins[run.id];
  const bool cl = lt_plugin_is_opencl_c(plugin);
  std::string err;
  unsigned smem = 0;
  // a work-group whose traversal stacks do not fit is refused before anything is launched
  if (cl && !lt_plugin_smem(plugin, run.kernelMode, &scene->dev, (unsigned)(run.bx * run.by), &smem, &err))
    return fail(ctx, LT_ERR_INVALID, std::string(who) + ": " + err);
  const size_t floats = (size_t)P.width * P.height * P.depth;
  int rc = ensure_out(ctx, floats);
  if (rc != LT_OK) return rc;
  // LT_ACCUM_NONE: every frame into the output, in order (F consecutive single-frame calls); otherwise every frame into
  // the sample buffer, folded into the accumulator after it
  const bool fold = P.accum_mode != LT_ACCUM_NONE;
  if (fold && ctx->sampleFloats < floats) {
    if (ctx->dSample) cudaFree(ctx->dSample);
    ctx->dSample = nullptr;
    ctx->sampleFloats = 0;
    CK(cudaMalloc(&ctx->dSample, floats * sizeof(float)));
    ctx->sampleFloats = floats;
  }
  float* dFrame = fold ? ctx->dSample : ctx->dOut;
  if (ctx->cameraCount < P.frames) {
    if (ctx->dCamera) cudaFree(ctx->dCamera);
    ctx->dCamera = nullptr;
    ctx->cameraCount = 0;
    CK(cudaMalloc(&ctx->dCamera, sizeof(RefCamera) * (size_t)P.frames));
    ctx->cameraCount = P.frames;
  }
  // frame k reads its own record, frameCount = camera.frameCount + k * frame_stride
  const uint32_t stride = P.frame_stride ? P.frame_stride : 1u;
  std::vector<RefCamera> cams((size_t)P.frames, cam);
  for (int k = 0; k < P.frames; k++) cams[k].frameCount = cam.frameCount + (uint32_t)k * stride;
  CK(cudaMemcpyAsync(ctx->dCamera, cams.data(), sizeof(RefCamera) * cams.size(), cudaMemcpyHostToDevice, ctx->stream));
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
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  int launches = 0;
  for (int k = 0; k < P.frames; k++) {
    const RefCamera* dCam = ctx->dCamera + k;
    const int n = cl ? lt_plugin_launch_cl(plugin, run.kernelMode, &scene->dev, scene->dNodes, scene->dPrims,
                                           scene->dMats, scene->dLights, dCam, dFrame, P.width, P.height, P.depth,
                                           run.wbx, run.wby, run.bx, run.by, ctx->stream, &err)
                     : (lt_plugin_launch(plugin, run.kernelMode, &scene->dev, scene->dNodes, scene->dPrims, scene->dMats,
                                         scene->dLights, dCam, dFrame, P.width, P.height, P.depth, run.bx, run.by,
                                         ctx->stream, &err) == 0 ? 1 : -1);
    if (n < 0) return fail(ctx, LT_ERR_CUDA, std::string(who) + ": " + err);
    launches += n;
    if (fold) {
      L.cam = cams[k];
      launches += lt_launch_plugin_accumulate(L, dFrame, ctx->dOut, ctx->stats.sm_count, ctx->stream);
    }
  }
  CK(cudaGetLastError());
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->stats.kernel_launches = launches;
  ctx->stats.rays = ctx->stats.node_tests = ctx->stats.tri_tests = 0;
  ctx->stats.trace_ms = ctx->stats.shade_ms = ctx->stats.primary_shade_ms = ctx->stats.accumulate_ms = 0.0f;
  ctx->stats.trace_launches = ctx->stats.shade_launches = 0;
  if (sync) {
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaEventElapsedTime(&ctx->stats.kernel_ms, ctx->ev0, ctx->ev1));
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
  if (host_out) return download(ctx, host_out, ctx->dOut, (size_t)width * height * depth * sizeof(float));
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
  memset(&P, 0, sizeof P);
  memcpy(&P, params, params->struct_size < sizeof P ? params->struct_size : sizeof P);
  P.kernel = 0;
  P.max_ray_depth = 0;
  LtLaunch L;
  if (int rc = launch_from_params(ctx, &P, &L, who)) return rc;
  P.struct_size = sizeof P;
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
  if (host_out) return download(ctx, host_out, ctx->dOut, (size_t)P.width * P.height * P.depth * sizeof(float));
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
  if (ctx->dOut) CK(cudaMemsetAsync(ctx->dOut, 0, ctx->outFloats * sizeof(float), ctx->stream));
  return LT_OK;
}

extern "C" int lt_accum_read(lt_ctx* ctx, float* host_out, uint64_t float_count) {
  if (!ctx || !host_out) return fail(ctx, LT_ERR_INVALID, "lt_accum_read: NULL argument");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_accum_read: a multi-GPU context returns its accumulator through lt_render");
  if (!ctx->dOut || float_count > ctx->outFloats) return fail(ctx, LT_ERR_INVALID, "lt_accum_read: no accumulator of that size");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(host_out, ctx->dOut, float_count * sizeof(float), cudaMemcpyDeviceToHost));
  return LT_OK;
}

static int primary_hits_impl(lt_ctx* ctx, lt_scene* scene, const void* camera28, int kernel, int flags, int width,
                             int height, int32_t* ids, int32_t* hit, float* tuv);

extern "C" int lt_primary_hits(lt_ctx* ctx, lt_scene* scene, const void* camera28, int kernel, int width, int height,
                               int32_t* ids, int32_t* hit, float* tuv) {
  return primary_hits_impl(ctx, scene, camera28, kernel, 0, width, height, ids, hit, tuv);
}

extern "C" int lt_primary_hits_flags(lt_ctx* ctx, lt_scene* scene, const void* camera28, int kernel, int flags,
                                     int width, int height, int32_t* ids, int32_t* hit, float* tuv) {
  return primary_hits_impl(ctx, scene, camera28, kernel, flags, width, height, ids, hit, tuv);
}

static int primary_hits_impl(lt_ctx* ctx, lt_scene* scene, const void* camera28, int kernel, int flags, int width,
                             int height, int32_t* ids, int32_t* hit, float* tuv) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_primary_hits: ctx is NULL");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_primary_hits: use a single-GPU context");
  if (!scene || !camera28 || width <= 0 || height <= 0 || kernel < 0 || kernel >= LT_KERNEL_COUNT)
    return fail(ctx, LT_ERR_INVALID, "lt_primary_hits: bad argument");
  CK(cudaSetDevice(ctx->device));
  size_t n = (size_t)width * height;
  int* dAll = nullptr;  // one allocation: ids | hit | t,u,v
  CK(cudaMalloc(&dAll, 5 * n * sizeof(int)));
  int *dIds = dAll, *dHit = dAll + n;
  float* dTuv = reinterpret_cast<float*>(dAll + 2 * n);
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
  cudaFree(dAll);
  if (e != cudaSuccess) return fail(ctx, LT_ERR_CUDA, std::string("lt_primary_hits: ") + cudaGetErrorString(e));
  return LT_OK;
}

// parity hooks: evaluate device-side helper functions on host-supplied inputs
extern "C" int lt_debug_random(lt_ctx* ctx, const float* fx, const float* fy, const float* seed, int n, float* out) {
  if (!ctx || ctx->group || !fx || !fy || !seed || !out || n <= 0) return fail(ctx, LT_ERR_INVALID, "lt_debug_random: bad argument");
  CK(cudaSetDevice(ctx->device));
  float* d = nullptr;
  CK(cudaMalloc(&d, sizeof(float) * 4 * (size_t)n));
  cudaMemcpy(d, fx, sizeof(float) * n, cudaMemcpyHostToDevice);
  cudaMemcpy(d + n, fy, sizeof(float) * n, cudaMemcpyHostToDevice);
  cudaMemcpy(d + 2 * (size_t)n, seed, sizeof(float) * n, cudaMemcpyHostToDevice);
  lt_launch_debug_random(d, d + n, d + 2 * (size_t)n, n, d + 3 * (size_t)n, ctx->stream);
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpy(out, d + 3 * (size_t)n, sizeof(float) * n, cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) return fail(ctx, LT_ERR_CUDA, std::string("lt_debug_random: ") + cudaGetErrorString(e));
  return LT_OK;
}

extern "C" int lt_debug_hemisphere(lt_ctx* ctx, const float* u1, const float* u2, const float* up3, int n, float* out4) {
  if (!ctx || ctx->group || !u1 || !u2 || !up3 || !out4 || n <= 0) return fail(ctx, LT_ERR_INVALID, "lt_debug_hemisphere: bad argument");
  CK(cudaSetDevice(ctx->device));
  float* d = nullptr;
  CK(cudaMalloc(&d, sizeof(float) * 9 * (size_t)n));
  cudaMemcpy(d, u1, sizeof(float) * n, cudaMemcpyHostToDevice);
  cudaMemcpy(d + n, u2, sizeof(float) * n, cudaMemcpyHostToDevice);
  cudaMemcpy(d + 2 * (size_t)n, up3, sizeof(float) * 3 * n, cudaMemcpyHostToDevice);
  lt_launch_debug_hemisphere(d, d + n, d + 2 * (size_t)n, n, d + 5 * (size_t)n, ctx->stream);
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpy(out4, d + 5 * (size_t)n, sizeof(float) * 4 * n, cudaMemcpyDeviceToHost);
  cudaFree(d);
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
