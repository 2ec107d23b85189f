// lt_capi.cu -- the C-ABI of liblt_b200.so (include/lens_trace_b200.h): context, scene upload with
// device-side re-flatten, render entry points.  No CPU fallback: every compute call needs a CUDA
// device and fails with LT_ERR_NO_DEVICE / LT_ERR_CUDA otherwise.
#include "lens_trace_b200.h"
#include "lt_internal.h"

#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

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
  cudaFree(s->dThreadBig);
  delete s;
}

// Threaded form of the tree (LtThreadNode, lens_trace_b200_device.cuh): eight copies of the node array, copy o in
// the order the reference's traversal visits the nodes for rays of sign octant o, then eight pruned copies.  Built
// on the host: it is only made for trees of at most lt_threaded_max_nodes() nodes (8 x 32 B x N for the full copies,
// at most as much again for the pruned ones, must stay cache resident).
static int lt_threaded_max_nodes() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("LT_THREADED_MAX_NODES");
    v = e ? atoi(e) : 65536;  // 16 MB of records at the limit
    if (v < 0) v = 0;
  }
  return v;
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
  std::vector<int> size(n), order, before(n + 1), stack;
  for (int i = n - 1; i >= 0; i--)  // children follow their parent in the depth-first array
    size[i] = nodes[i].primitiveCount > 0 ? 1 : 1 + size[i + 1] + size[nodes[i].offset];
  auto bitsf = [](int v) { float f; memcpy(&f, &v, 4); return f; };
  for (int o = 0; o < 8; o++) {
    order.clear();
    stack.clear();
    stack.push_back(0);
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
static std::vector<char> pruned_keep(const RefNode* nodes, int n) {
  std::vector<char> keep(n, 1);
  std::vector<int> anc(n, 0);  // nearest kept ancestor
  auto inside = [](const RefNode& c, const RefNode& m) {
    for (int k = 0; k < 3; k++)
      if (!(m.boundsMin[k] <= c.boundsMin[k] && c.boundsMin[k] <= c.boundsMax[k] && c.boundsMax[k] <= m.boundsMax[k]))
        return false;
    return true;
  };
  auto area = [](const RefNode& r) {
    double dx = (double)r.boundsMax[0] - r.boundsMin[0], dy = (double)r.boundsMax[1] - r.boundsMin[1],
           dz = (double)r.boundsMax[2] - r.boundsMin[2];
    return dx * dy + dy * dz + dz * dx;
  };
  for (int i = 0; i < n; i++) {  // parents precede their children in the depth-first array
    const RefNode& m = nodes[i];
    if (m.primitiveCount > 0) continue;
    if (i > 0)
      keep[i] = !(inside(nodes[i + 1], m) && inside(nodes[m.offset], m) && area(m) > 0.5 * area(nodes[anc[i]]));
    anc[i + 1] = anc[m.offset] = keep[i] ? i : anc[i];
  }
  return keep;
}

// Full copies (records [0, 8 n)), then the pruned copies (from record 8 n).  Returns the pruned stride.
static int build_threaded(const RefNode* nodes, int n, std::vector<LtThreadNode>& out) {
  out.clear();
  append_threaded(nodes, n, std::vector<char>(n, 1), out);
  return append_threaded(nodes, n, pruned_keep(nodes, n), out);
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

// Re-flatten on the device (inner-node ranks -> 64-byte child-pair nodes, 48-byte triangles) and fill the
// device-side scene descriptor.  ev0 must already be recorded on the stream; on failure the scene is released.
static int finish_scene(lt_ctx* ctx, lt_scene* s, int nNodes, int nPrims, int nMats, const RefNode& root,
                        int stackDepth, const char* who) {
  int* dFlags = nullptr;
  int* dRank = nullptr;
  void* dTemp = nullptr;
  int nInner = (nNodes - 1) / 2;  // a full binary tree with one primitive slot per leaf
  if (nNodes == 1) nInner = 0;
  size_t tempBytes = lt_scan_temp_bytes(nNodes);
  cudaError_t e = cudaSuccess;
  auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  cudaStream_t st = ctx->stream;
  A(cudaMalloc(&s->dWide, sizeof(LtWideNode) * (size_t)(nInner > 0 ? nInner : 1)));
  A(cudaMalloc(&s->dTris, sizeof(LtTri) * (size_t)nPrims));
  A(cudaMalloc(&dFlags, sizeof(int) * (size_t)nNodes));
  A(cudaMalloc(&dRank, sizeof(int) * (size_t)nNodes));
  A(cudaMalloc(&dTemp, tempBytes ? tempBytes : 16));
  if (e == cudaSuccess) {
    lt_launch_inner_flags(s->dNodes, nNodes, dFlags, st);
    lt_launch_exclusive_scan(dTemp, tempBytes, dFlags, dRank, nNodes, st);
    lt_launch_reflatten(s->dNodes, nNodes, s->dPrims, nPrims, dRank, s->dWide, s->dTris, st);
    A(cudaGetLastError());
  }
  if (e == cudaSuccess && nNodes <= lt_threaded_max_nodes()) {
    std::vector<RefNode> hNodes((size_t)nNodes);
    std::vector<LtThreadNode> hThread;
    A(cudaMemcpyAsync(hNodes.data(), s->dNodes, sizeof(RefNode) * (size_t)nNodes, cudaMemcpyDeviceToHost, st));
    A(cudaStreamSynchronize(st));
    if (e == cudaSuccess) {
      s->threadStride = build_threaded(hNodes.data(), nNodes, hThread);
      A(cudaMalloc(&s->dThread, sizeof(LtThreadNode) * hThread.size()));
      A(cudaMemcpyAsync(s->dThread, hThread.data(), sizeof(LtThreadNode) * hThread.size(), cudaMemcpyHostToDevice, st));
      A(cudaStreamSynchronize(st));  // hThread is pageable and goes out of scope
    }
  }
  // large trees: the threaded copies are built on the device and used by coherent-ray launches only (lt_kernels.cu:
  // scene_for_flags); skipped when they would not fit the budget (4 GB and an eighth of the device)
  if (e == cudaSuccess && nNodes > lt_threaded_max_nodes() && nNodes > 1) {
    const size_t kBudget = 4ull << 30;
    const size_t bytes = sizeof(LtThreadNode) * 8 * (size_t)nNodes;
    if (bytes <= kBudget && bytes <= ctx->totalMem / 8 && (long long)nNodes * 8 < 0x7fffffffll) {
      if (cudaMalloc(&s->dThreadBig, bytes) == cudaSuccess) {
        lt_launch_build_threaded(s->dNodes, nNodes, s->dThreadBig, st);
        A(cudaGetLastError());
      } else {
        cudaGetLastError();  // no memory for the copies: the stack traversal serves every launch
        s->dThreadBig = nullptr;
      }
    }
  }
  A(cudaEventRecord(ctx->ev1, st));
  A(cudaStreamSynchronize(st));
  cudaFree(dFlags);
  cudaFree(dRank);
  cudaFree(dTemp);
  if (e != cudaSuccess) {
    lt_scene_release(ctx, s);
    return fail(ctx, LT_ERR_CUDA, std::string(who) + ": " + cudaGetErrorString(e));
  }
  cudaEventElapsedTime(&ctx->stats.upload_ms, ctx->ev0, ctx->ev1);
  LtSceneDev& d = s->dev;
  d.wnodes = s->dWide;
  d.tris = s->dTris;
  d.prims = s->dPrims;
  d.mats = s->dMats;
  d.lights = s->dLights;
  for (int k = 0; k < 3; k++) {
    d.rootMin[k] = root.boundsMin[k];
    d.rootMax[k] = root.boundsMax[k];
  }
  d.rootRef = root.primitiveCount > 0 ? ~root.offset : 0;  // inner root is wide node 0
  d.rootCount = root.primitiveCount;
  d.stackDepth = stackDepth;
  d.nodeCount = nNodes;
  d.primCount = nPrims;
  d.matCount = nMats;
  d.tnodes = s->dThread;
  d.tnodesCoherent = s->dThreadBig;
  set_pruned_copies(s, false);
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
  A(cudaMalloc(&s->dNodes, sizeof(RefNode) * (size_t)nNodes));
  A(cudaMalloc(&s->dPrims, primitive_bytes));
  A(cudaMalloc(&s->dMats, material_bytes));
  A(cudaMalloc(&s->dLights, sizeof(RefLights)));
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
  A(cudaMalloc(&s->dNodes, node_bytes));
  A(cudaMalloc(&s->dPrims, primitive_bytes));
  A(cudaMalloc(&s->dMats, material_bytes ? material_bytes : sizeof(RefMaterial)));
  A(cudaMalloc(&s->dLights, sizeof(RefLights)));
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

static int check_params(lt_ctx* ctx, const lt_scene* scene, const void* camera28, const lt_render_params* p,
                        LtLaunch* L) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_render: ctx is NULL");
  if (!scene || !camera28 || !p) return fail(ctx, LT_ERR_INVALID, "lt_render: NULL argument");
  // API version 1 callers pass the struct without its last field (split_mode)
  if (p->struct_size != sizeof(lt_render_params) && p->struct_size != offsetof(lt_render_params, split_mode))
    return fail(ctx, LT_ERR_INVALID, "lt_render: params.struct_size mismatch");
  if (p->kernel < 0 || p->kernel >= LT_KERNEL_COUNT) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_render: unknown kernel id");
  if (p->width <= 0 || p->height <= 0 || p->depth < 3)
    return fail(ctx, LT_ERR_INVALID, "lt_render: width/height must be > 0 and depth >= 3");
  if ((long long)p->width * p->height * p->depth > (1ll << 40)) return fail(ctx, LT_ERR_INVALID, "lt_render: image too large");
  if (p->frames < 1) return fail(ctx, LT_ERR_INVALID, "lt_render: frames must be >= 1");
  if (p->accum_mode < 0 || p->accum_mode > 2) return fail(ctx, LT_ERR_INVALID, "lt_render: bad accum_mode");
  if (p->max_ray_depth < 0 || p->max_ray_depth > 255)
    return fail(ctx, LT_ERR_INVALID, "lt_render: max_ray_depth must be in [0, 255]");
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
  memcpy(&L->cam, camera28, sizeof(RefCamera));
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

static int render_common(lt_ctx* ctx, lt_scene* scene, const LtLaunch& L, float* dOut, bool sync) {
  CK(cudaSetDevice(ctx->device));
  bool stats = (L.flags & LT_FLAG_STATS) != 0;
  if (stats) CK(cudaMemsetAsync(ctx->dCounters, 0, sizeof(LtCounters), ctx->stream));
  // stochastic kernels: wavefront pipeline for large launches, persistent megakernel for small ones
  bool wavefront = false, overlapBatches = false;
  int batchFrames = 1;
  if (L.kernel >= 3 && !(L.flags & LT_FLAG_MEGAKERNEL)) {
    long long pixels = (long long)L.width * L.height;
    const long long minPaths = 1ll << 23;
    // paths in flight, both overlapped batches together (~200 B each); a queue entry carries its path id in 25 bits
    const long long maxPaths = 1ll << 26;
    // measured (tools/compare_pipelines.py): the wavefront wins once ~8M paths are in flight per batch; below
    // that, and for the two-ray lighting kernels on small scenes, its per-round launches and state traffic lose
    bool isGI = (L.kernel == 5 || L.kernel == 6);
    bool bigScene = scene->dev.nodeCount > 100000;
    // second measurement (shared camera rays, overlapped batches): the two-ray lighting kernels on a small scene win
    // too once a launch holds several batches (64 frames at 1080p: 1.31x); the 25-sample kernels stay on k_path
    long long need = (isGI || bigScene) ? minPaths : 4 * minPaths;
    wavefront = (L.flags & (LT_FLAG_WAVEFRONT | LT_FLAG_CULL)) ||
                (pixels * L.frames >= need && L.kernel != 5 && L.kernel != 3);
    // a queue entry carries the bounce depth in 5 bits (wf_pack_path): deeper bounce caps stay on the megakernel,
    // which is the same arithmetic per path (0 = the reference constant 16)
    if (wavefront && isGI && L.maxRayDepth > 32) {
      if (L.flags & (LT_FLAG_WAVEFRONT | LT_FLAG_CULL))
        return fail(ctx, LT_ERR_UNSUPPORTED, "lt_render: the wavefront pipeline handles max_ray_depth <= 32 (use the default schedule)");
      wavefront = false;
    }
    if (wavefront && pixels > (1ll << 25)) {  // a queue entry carries its path id in 25 bits: one frame must fit
      if (L.flags & (LT_FLAG_WAVEFRONT | LT_FLAG_CULL))
        return fail(ctx, LT_ERR_UNSUPPORTED, "lt_render: the wavefront pipeline handles at most 2^25 pixels per frame");
      wavefront = false;
    }
    if (wavefront) {
      long long cap = maxPaths;
      long long memCap = (long long)(ctx->totalMem / 8) / 200;  // at most 1/8 of the device for the workspace
      if (cap > memCap) cap = memCap;
      batchFrames = (int)(cap / pixels);
      if (batchFrames < 1) batchFrames = 1;
      if (batchFrames > L.frames) batchFrames = L.frames;
      // two consecutive batches overlap on two streams (trace of one beside shade of the other): half-size batches,
      // one workspace each -- same memory.  LT_FLAG_SERIAL: one stream, kernels run one at a time.
      overlapBatches = !(L.flags & (LT_FLAG_SERIAL | LT_FLAG_STATS)) && L.frames >= 2;
      const int nStreams = overlapBatches ? 2 : 1;
      batchFrames = (batchFrames + nStreams - 1) / nStreams;
      {  // a queue entry carries its path id in 25 bits: at most 2^25 paths per batch
        long long perBatch = (1ll << 25) / pixels;
        if (perBatch < 1) perBatch = 1;
        if (batchFrames > perBatch) batchFrames = (int)perBatch;
      }
      size_t need = lt_wf_workspace_bytes_padded((long long)batchFrames * pixels) * (size_t)nStreams +
                    lt_wf_primary_hits_bytes(pixels);
      if (ctx->wfBytes < need) {
        if (ctx->wfWorkspace) cudaFree(ctx->wfWorkspace);
        ctx->wfWorkspace = nullptr;
        ctx->wfBytes = 0;
        if (cudaMalloc(&ctx->wfWorkspace, need) != cudaSuccess) {
          cudaGetLastError();
          if (L.flags & (LT_FLAG_WAVEFRONT | LT_FLAG_CULL))
            return fail(ctx, LT_ERR_CUDA, "lt_render: cannot allocate the wavefront workspace");
          wavefront = false;  // not a fallback to other arithmetic: the megakernel is the same path per pixel
        } else {
          ctx->wfBytes = need;
        }
      }
    }
  }
  const int kMaxTracePairs = 8192;
  int tracePairs = 0;
  bool timeTrace = wavefront && (sync || stats);
  if (timeTrace && ctx->traceEvents.empty()) {
    ctx->traceEvents.resize(2 * kMaxTracePairs);
    ctx->pairKinds.resize(kMaxTracePairs);
    for (size_t i = 0; i < ctx->traceEvents.size(); i++) cudaEventCreate(&ctx->traceEvents[i]);
  }
  // per-kernel times are only defined when one kernel runs at a time (LT_FLAG_SERIAL / stats launches)
  const bool timeKinds = timeTrace && (!overlapBatches);
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  int launches = wavefront ? lt_launch_render_wavefront(scene->dev, L, dOut, ctx->dCounters, ctx->wfWorkspace,
                                                        batchFrames, ctx->stats.sm_count, ctx->stream,
                                                        timeTrace ? ctx->traceEvents.data() : nullptr, kMaxTracePairs,
                                                        &tracePairs, timeKinds ? ctx->pairKinds.data() : nullptr,
                                                        overlapBatches ? &ctx->wfAux : nullptr)
                           : lt_launch_render(scene->dev, L, dOut, ctx->dCounters, ctx->dWork, ctx->stats.sm_count,
                                              ctx->stream);
  CK(cudaGetLastError());
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->stats.kernel_launches = launches;
  if (sync || stats) {
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaEventElapsedTime(&ctx->stats.kernel_ms, ctx->ev0, ctx->ev1));
    ctx->stats.trace_ms = wavefront ? 0.0f : ctx->stats.kernel_ms;
    ctx->stats.trace_launches = wavefront ? 0 : 1;
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
  if (ctx && ctx->group) return lt_multi_render(ctx, scene, camera28, params, host_out);
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

extern "C" int lt_plugin_load(lt_ctx* ctx, const char* kernel_file_path, int* out_plugin_id) {
  if (!ctx || !kernel_file_path || !out_plugin_id) return fail(ctx, LT_ERR_INVALID, "lt_plugin_load: NULL argument");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_plugin_load: plug-in kernels run on single-GPU contexts");
  CK(cudaSetDevice(ctx->device));
  CK(cudaFree(0));  // make sure the primary context is current for the driver-API module load
  std::string err;
  LtPlugin* p = lt_plugin_compile(kernel_file_path, &err);
  if (!p) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_plugin_load: " + err);
  ctx->plugins.push_back(p);
  *out_plugin_id = (int)ctx->plugins.size() - 1;
  return LT_OK;
}

extern "C" int lt_render_plugin(lt_ctx* ctx, lt_scene* scene, const void* camera28, int plugin_id, int kernel_mode,
                                int width, int height, int depth, int block_x, int block_y, float* host_out) {
  if (!ctx) return fail(nullptr, LT_ERR_INVALID, "lt_render_plugin: ctx is NULL");
  if (ctx->group) return fail(ctx, LT_ERR_UNSUPPORTED, "lt_render_plugin: plug-in kernels run on single-GPU contexts");
  if (!scene || !camera28 || plugin_id < 0 || plugin_id >= (int)ctx->plugins.size() || width <= 0 || height <= 0 ||
      depth < 1)
    return fail(ctx, LT_ERR_INVALID, "lt_render_plugin: bad argument");
  CK(cudaSetDevice(ctx->device));
  size_t floats = (size_t)width * height * depth;
  int rc = ensure_out(ctx, floats);
  if (rc != LT_OK) return rc;
  if (!ctx->dCamera) CK(cudaMalloc(&ctx->dCamera, sizeof(RefCamera)));
  CK(cudaMemcpyAsync(ctx->dCamera, camera28, sizeof(RefCamera), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  std::string err;
  if (lt_plugin_launch(ctx->plugins[plugin_id], kernel_mode ? 1 : 0, &scene->dev, scene->dNodes, scene->dPrims, scene->dMats,
                       scene->dLights, ctx->dCamera, ctx->dOut, width, height, depth, block_x, block_y, ctx->stream,
                       &err) != 0)
    return fail(ctx, LT_ERR_CUDA, "lt_render_plugin: " + err);
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaEventElapsedTime(&ctx->stats.kernel_ms, ctx->ev0, ctx->ev1));
  ctx->stats.kernel_launches = 1;
  if (host_out) return download(ctx, host_out, ctx->dOut, floats * sizeof(float));
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
  lt_launch_primary_hits(scene->dev, cam, kernel, flags, width, height, dIds, dHit, dTuv, ctx->stream);
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
  return (kernel >= 0 && kernel < LT_KERNEL_COUNT) ? kKernelNames[kernel] : "unknown";
}

// kernelFilePath -> built-in pipeline, by CONTENT (the reference compiles whatever text the file holds,
// src/cuda/renderer_cuda.cpp:20-39,52-55, so the name alone must never select a pipeline):
//   * a descriptor file of this repository -- nothing but // comment lines, one of them "lt-pipeline: <tag>" -- or
//   * a file whose text is, byte for byte (CR dropped), one of the seven kernel files the reference ships
//     (lt_kernel_hashes.inc: FNV-1a-64 + length; only hashes are stored)
// maps to the hand-written pipeline that reproduces that kernel.  Anything else -- including an EDITED copy of a
// shipped kernel under its old name -- is a user kernel: LT_ERR_UNSUPPORTED here; the renderer then compiles a .cu
// as a plug-in (lt_plugin_load) and reports an error for a .cl (OpenCL C cannot be compiled for sm_100a here).
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
            "a shipped kernel (user kernels: .cu files are compiled as plug-ins, .cl files are not supported)";
  return LT_ERR_UNSUPPORTED;
}
