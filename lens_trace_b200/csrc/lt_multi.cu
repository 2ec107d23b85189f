// lt_multi.cu -- multi-GPU contexts of the C-ABI (lt_ctx_create_multi): one process, one single-GPU context per
// device, the scene replicated, one lt_render call divided among the devices (SURVEY.md 8(e); the reference renders
// on device 0 only, src/cuda/renderer_cuda.cpp:12).
//
//   sample split  device g renders frames g, g+G, ... of the call into its own FP32 accumulator as a weighted sum
//                 (LT_ACCUM_WEIGHTED_SUM, weight 1/N); the accumulators are combined by ONE all-reduce per call:
//                 ncclAllReduce over NVLink (single-process communicators, ncclCommInitAll; libnccl is loaded with
//                 dlopen on first use), or -- LT_MULTI_EXCHANGE=p2p, and whenever NCCL is unavailable -- this
//                 file's own kernel, in which every device sums all peers' accumulators through peer-mapped memory
//                 in a fixed order (deterministic) behind an event barrier.  The result differs from the sequential
//                 running mean of accumulator.frag:10-19 by FP32 summation order only.
//   tile split    device g renders every G-th block of 8 image rows (cost varies smoothly over the image, so the
//                 blocks balance); nothing is exchanged, every device copies its rows into the caller's buffer over
//                 its own PCIe link.
//
// The kernels of every device are launched from that device's own host thread: a 64-spp wavefront step is ~240
// launches, and eight devices' worth of them issued from one thread would cost more than the rendering.
#include <dlfcn.h>
#include <nccl.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <thread>
#include <vector>

#include "lt_internal.h"

namespace {

struct NcclApi {
  bool tried = false, ok = false;
  std::string why;
  ncclResult_t (*commInitAll)(ncclComm_t*, int, const int*);
  ncclResult_t (*commDestroy)(ncclComm_t);
  ncclResult_t (*allReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*groupStart)();
  ncclResult_t (*groupEnd)();
  const char* (*getErrorString)(ncclResult_t);
};
NcclApi g_nccl;

bool load_nccl() {
  NcclApi& a = g_nccl;
  if (a.tried) return a.ok;
  a.tried = true;
  void* lib = nullptr;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names)
    if ((lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break;
  if (!lib) {
    a.why = "libnccl.so.2 not found";
    return false;
  }
  a.commInitAll = (decltype(a.commInitAll))dlsym(lib, "ncclCommInitAll");
  a.commDestroy = (decltype(a.commDestroy))dlsym(lib, "ncclCommDestroy");
  a.allReduce = (decltype(a.allReduce))dlsym(lib, "ncclAllReduce");
  a.groupStart = (decltype(a.groupStart))dlsym(lib, "ncclGroupStart");
  a.groupEnd = (decltype(a.groupEnd))dlsym(lib, "ncclGroupEnd");
  a.getErrorString = (decltype(a.getErrorString))dlsym(lib, "ncclGetErrorString");
  a.ok = a.commInitAll && a.commDestroy && a.allReduce && a.groupStart && a.groupEnd && a.getErrorString;
  if (!a.ok) a.why = "libnccl lacks a needed symbol";
  return a.ok;
}

#define LT_MAX_DEVICES 16
struct PeerPointers {
  const float* p[LT_MAX_DEVICES];
};

// dst[i] = sum over the devices, in device order, of their accumulators (peer-mapped reads over NVLink)
__global__ void k_sum_peers(float* __restrict__ dst, PeerPointers src, int devices, size_t n) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const size_t n4 = n / 4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 s = reinterpret_cast<const float4*>(src.p[0])[i];
    for (int d = 1; d < devices; d++) {
      float4 v = reinterpret_cast<const float4*>(src.p[d])[i];
      s.x = __fadd_rn(s.x, v.x);
      s.y = __fadd_rn(s.y, v.y);
      s.z = __fadd_rn(s.z, v.z);
      s.w = __fadd_rn(s.w, v.w);
    }
    reinterpret_cast<float4*>(dst)[i] = s;
  }
  for (size_t i = n4 * 4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float s = src.p[0][i];
    for (int d = 1; d < devices; d++) s = __fadd_rn(s, src.p[d][i]);
    dst[i] = s;
  }
}

__global__ void k_scale(float* __restrict__ p, size_t n, float f) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) p[i] = __fmul_rn(p[i], f);
}

}  // namespace

enum { kRendered, kSummed };  // the events of a member of a group

struct LtGroup {
  std::vector<lt_ctx*> ctx;         // one single-GPU context per device
  std::vector<ncclComm_t> comms;    // sample split, NCCL exchange
  bool ncclTried = false, ncclReady = false;
  bool peersTried = false, peersReady = false;
  // per member, on its device: the p2p exchange's second accumulator (the kernel's destination), and its two events
  std::vector<LtBuf<float>> sumBuf;
  std::vector<LtEvents> events;  // [kRendered], [kSummed]
  int lastSplit = -1;               // split of the accumulators the devices hold (a change resets them)
  long long lastFloats = -1;
  bool sharesDevice = false;        // a device ordinal is listed more than once (lt_debug_ctx_create_shared)
};

extern "C" int lt_ctx_device_count(const lt_ctx* ctx) {
  if (!ctx) return 0;
  return ctx->group ? (int)ctx->group->ctx.size() : 1;
}

// The group context over `count` member contexts, member k on device ordinals[k].  An ordinal may repeat (shared
// groups, lt_debug_ctx_create_shared): every member is an ordinary single-GPU context with its own stream, buffers and
// host thread either way.  `who` names the entry point in error messages.
static int create_group(const int* ordinals, int count, const char* who, lt_ctx** out_ctx) {
  LtGroup* g = new LtGroup();
  lt_ctx* ctx = new lt_ctx();
  ctx->device = ordinals[0];
  ctx->group = g;
  for (int a = 0; a < count; a++)
    for (int b = a + 1; b < count; b++) g->sharesDevice |= ordinals[a] == ordinals[b];
  g->sumBuf.resize(count);
  g->events.resize(count);
  for (int k = 0; k < count; k++) {
    lt_ctx* c = nullptr;
    int rc = lt_ctx_create(ordinals[k], &c);
    if (rc != LT_OK) {
      lt_ctx_destroy(ctx);
      return rc;  // message already set by lt_ctx_create
    }
    g->ctx.push_back(c);
  }
  for (int k = 0; k < count; k++) {
    cudaError_t e = cudaSetDevice(g->ctx[k]->device);
    if (e == cudaSuccess) e = g->events[k].grow(2, cudaEventDisableTiming);
    if (e != cudaSuccess) {
      lt_ctx_destroy(ctx);
      return lt_internal_fail(nullptr, LT_ERR_CUDA, std::string(who) + ": " + cudaGetErrorString(e));
    }
  }
  ctx->stats.sm_count = g->ctx[0]->stats.sm_count;
  *out_ctx = ctx;
  return LT_OK;
}

extern "C" int lt_ctx_create_multi(const int* device_ordinals, int device_count, lt_ctx** out_ctx) {
  if (!out_ctx) return lt_internal_fail(nullptr, LT_ERR_INVALID, "lt_ctx_create_multi: out_ctx is NULL");
  *out_ctx = nullptr;
  if (!device_ordinals || device_count < 1 || device_count > LT_MAX_DEVICES)
    return lt_internal_fail(nullptr, LT_ERR_INVALID, "lt_ctx_create_multi: needs 1..16 device ordinals");
  for (int a = 0; a < device_count; a++)
    for (int b = a + 1; b < device_count; b++)
      if (device_ordinals[a] == device_ordinals[b])
        return lt_internal_fail(nullptr, LT_ERR_INVALID, "lt_ctx_create_multi: a device ordinal is listed twice");
  if (device_count == 1) return lt_ctx_create(device_ordinals[0], out_ctx);
  return create_group(device_ordinals, device_count, "lt_ctx_create_multi", out_ctx);
}

extern "C" int lt_debug_ctx_create_shared(int device_ordinal, int members, lt_ctx** out_ctx) {
  if (!out_ctx) return lt_internal_fail(nullptr, LT_ERR_INVALID, "lt_debug_ctx_create_shared: out_ctx is NULL");
  *out_ctx = nullptr;
  if (members < 2 || members > LT_MAX_DEVICES)
    return lt_internal_fail(nullptr, LT_ERR_INVALID, "lt_debug_ctx_create_shared: needs 2..16 members");
  const std::vector<int> ordinals(members, device_ordinal);
  return create_group(ordinals.data(), members, "lt_debug_ctx_create_shared", out_ctx);
}

void lt_multi_destroy(lt_ctx* ctx) {
  LtGroup* g = ctx->group;
  if (!g) return;
  for (size_t k = 0; k < g->ctx.size(); k++) {
    cudaSetDevice(g->ctx[k]->device);
    cudaDeviceSynchronize();
    if (k < g->comms.size() && g->comms[k] && g_nccl.ok) g_nccl.commDestroy(g->comms[k]);
    g->sumBuf[k].reset();
    g->events[k].reset();
  }
  for (lt_ctx* c : g->ctx) lt_ctx_destroy(c);
  delete g;
  ctx->group = nullptr;
}

// The one place that runs work on the devices of a group: fn(k) for the devices k = 0 .. n-1, each on a host thread of
// its own, joined before it returns.  Every device's statistics start first, so that a device with no share in the
// call reports zeros.  Returns LT_OK, or the code of the lowest-numbered device that failed, with that device's message
// copied to the group context.
template <class Fn>
static int fan_out(lt_ctx* ctx, int n, Fn fn) {
  LtGroup* g = ctx->group;
  for (lt_ctx* c : g->ctx) lt_internal_stats_start(c);
  std::vector<int> rcs(n, LT_OK);
  std::vector<std::thread> workers;
  for (int k = 0; k < n; k++) workers.emplace_back([&, k]() { rcs[k] = fn(k); });
  for (std::thread& t : workers) t.join();
  for (int k = 0; k < n; k++)
    if (rcs[k] != LT_OK) return lt_internal_fail(ctx, rcs[k], lt_last_error(g->ctx[k]));
  return LT_OK;
}

// c's device made current on the calling thread, or LT_ERR_CUDA with c's message
static int use_device(lt_ctx* c) {
  const cudaError_t e = cudaSetDevice(c->device);
  if (e == cudaSuccess) return LT_OK;
  return lt_internal_fail(c, LT_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
}

// upload and refit: the slowest device's time
static void merge_upload_ms(lt_ctx* ctx) {
  ctx->stats.upload_ms = 0.0f;
  for (const lt_ctx* c : ctx->group->ctx) ctx->stats.upload_ms = std::max(ctx->stats.upload_ms, c->stats.upload_ms);
}

// A render call's statistics: the slowest device's kernel time and every device's launches.  Leaves device 0 current
// on the calling thread.
static void merge_render_stats(lt_ctx* ctx) {
  lt_internal_stats_start(ctx);
  for (const lt_ctx* c : ctx->group->ctx) {
    ctx->stats.kernel_ms = std::max(ctx->stats.kernel_ms, c->stats.kernel_ms);
    ctx->stats.kernel_launches += c->stats.kernel_launches;
  }
  cudaSetDevice(ctx->group->ctx[0]->device);
}

int lt_multi_scene_upload(lt_ctx* ctx, const void* nodes, uint64_t node_bytes, const void* primitives,
                          uint64_t primitive_bytes, const void* materials, uint64_t material_bytes,
                          const void* light_container, uint64_t light_bytes, lt_scene** out_scene) {
  LtGroup* g = ctx->group;
  *out_scene = nullptr;
  lt_scene* s = new lt_scene();
  s->parts.resize(g->ctx.size(), nullptr);
  const int rc = fan_out(ctx, (int)g->ctx.size(), [&](int k) {
    return lt_scene_upload(g->ctx[k], nodes, node_bytes, primitives, primitive_bytes, materials, material_bytes,
                           light_container, light_bytes, &s->parts[k]);
  });
  merge_upload_ms(ctx);
  if (rc != LT_OK) {
    for (size_t j = 0; j < g->ctx.size(); j++)
      if (s->parts[j]) lt_scene_release(g->ctx[j], s->parts[j]);
    delete s;
    return rc;
  }
  *out_scene = s;
  return LT_OK;
}

int lt_multi_scene_refit(lt_ctx* ctx, lt_scene* scene, const void* primitives) {
  LtGroup* g = ctx->group;
  const int rc = fan_out(ctx, (int)g->ctx.size(),
                         [&](int k) { return lt_internal_refit(g->ctx[k], scene->parts[k], primitives); });
  merge_upload_ms(ctx);
  return rc;
}

void lt_multi_scene_release(lt_ctx* ctx, lt_scene* scene) {
  LtGroup* g = ctx ? ctx->group : nullptr;
  for (size_t k = 0; k < scene->parts.size(); k++)
    if (scene->parts[k]) lt_scene_release(g && k < g->ctx.size() ? g->ctx[k] : nullptr, scene->parts[k]);
  delete scene;
}

int lt_multi_accum_reset(lt_ctx* ctx) {
  LtGroup* g = ctx->group;
  for (lt_ctx* c : g->ctx) {
    int rc = lt_accum_reset(c);
    if (rc != LT_OK) return lt_internal_fail(ctx, rc, lt_last_error(c));
  }
  return LT_OK;
}

// One compiled image, loaded on every device in that device's thread (its primary context current there): each
// device's context holds the plug-in under the same id.
int lt_multi_plugin_load(lt_ctx* ctx, const LtPluginImage& img, int* out_plugin_id) {
  LtGroup* g = ctx->group;
  const int G = (int)g->ctx.size();
  std::vector<LtPlugin*> loaded(G, nullptr);
  const int rc = fan_out(ctx, G, [&](int k) {
    std::string err;
    if (cudaSetDevice(g->ctx[k]->device) != cudaSuccess || cudaFree(0) != cudaSuccess)
      err = "cannot make device " + std::to_string(g->ctx[k]->device) + " current";
    else
      loaded[k] = lt_plugin_module_load(img, &err);
    return loaded[k] ? LT_OK : lt_internal_fail(g->ctx[k], LT_ERR_UNSUPPORTED, "lt_plugin_load: " + err);
  });
  if (rc != LT_OK) {
    for (LtPlugin* p : loaded) lt_plugin_free(p);
    return rc;
  }
  for (int k = 0; k < G; k++) g->ctx[k]->plugins.push_back(loaded[k]);
  *out_plugin_id = (int)g->ctx[0]->plugins.size() - 1;
  return LT_OK;
}

const std::vector<LtPlugin*>& lt_multi_plugins(const lt_ctx* ctx) { return ctx->group->ctx[0]->plugins; }

static bool ensure_nccl(LtGroup* g, std::string* why) {
  if (g->ncclTried) return g->ncclReady;
  g->ncclTried = true;
  if (g->sharesDevice) {  // NCCL gives each rank a device of its own
    *why = "a device is listed more than once";
    return false;
  }
  if (!load_nccl()) {
    *why = g_nccl.why;
    return false;
  }
  std::vector<int> devs;
  for (lt_ctx* c : g->ctx) devs.push_back(c->device);
  g->comms.assign(devs.size(), nullptr);
  ncclResult_t r = g_nccl.commInitAll(g->comms.data(), (int)devs.size(), devs.data());
  if (r != ncclSuccess) {
    *why = std::string("ncclCommInitAll: ") + g_nccl.getErrorString(r);
    g->comms.clear();
    return false;
  }
  g->ncclReady = true;
  return true;
}

static bool ensure_peers(LtGroup* g, size_t floats, std::string* why) {
  if (!g->peersTried) {
    g->peersTried = true;
    g->peersReady = true;
    for (size_t a = 0; a < g->ctx.size() && g->peersReady; a++) {
      cudaSetDevice(g->ctx[a]->device);
      for (size_t b = 0; b < g->ctx.size(); b++) {
        // a device reads its own memory without peer mapping (members of a shared group)
        if (g->ctx[a]->device == g->ctx[b]->device) continue;
        int can = 0;
        cudaDeviceCanAccessPeer(&can, g->ctx[a]->device, g->ctx[b]->device);
        if (!can) {
          *why = "devices cannot access each other's memory (no peer access)";
          g->peersReady = false;
          break;
        }
        cudaError_t e = cudaDeviceEnablePeerAccess(g->ctx[b]->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
          *why = std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e);
          g->peersReady = false;
          break;
        }
        cudaGetLastError();
      }
    }
  }
  if (!g->peersReady) {
    if (why->empty()) *why = "peer access is unavailable";
    return false;
  }
  for (size_t k = 0; k < g->ctx.size(); k++) {
    if (g->sumBuf[k].count() >= floats) continue;
    cudaSetDevice(g->ctx[k]->device);
    if (g->sumBuf[k].grow(floats) != cudaSuccess) {
      *why = "cannot allocate the exchange buffer";
      return false;
    }
  }
  return true;
}

// rows of the image device g of G renders in a tile split: every G-th block of LT_TILE_ROWS rows
int lt_tile_rows_of(int height, int G, int g) {
  int rows = 0;
  for (int b = g; b * LT_TILE_ROWS < height; b += G) {
    int left = height - b * LT_TILE_ROWS;
    rows += left < LT_TILE_ROWS ? left : LT_TILE_ROWS;
  }
  return rows;
}

// Row blocks k, k + G, ... of an image (`rows` rows in all, LT_TILE_ROWS per block, the last block shorter when the image
// ends inside it) from device memory to their places in the host image dst: full blocks in one strided copy, a shorter
// last block on its own.  The source holds the blocks srcPitch bytes apart from src (a device's own rows, or its blocks
// inside a full-size image).  Asynchronous on `stream`.
cudaError_t lt_copy_row_blocks(void* dst, const void* src, size_t srcPitch, size_t rowBytes, int rows, int G, int k,
                               cudaStream_t stream) {
  const int fullBlocks = rows / LT_TILE_ROWS, tail = rows % LT_TILE_ROWS;
  const size_t dstPitch = (size_t)G * LT_TILE_ROWS * rowBytes;
  char* d = (char*)dst + (size_t)k * LT_TILE_ROWS * rowBytes;
  cudaError_t e = cudaSuccess;
  if (fullBlocks > 0)
    e = cudaMemcpy2DAsync(d, dstPitch, src, srcPitch, LT_TILE_ROWS * rowBytes, fullBlocks, cudaMemcpyDeviceToHost,
                          stream);
  if (e == cudaSuccess && tail > 0)
    e = cudaMemcpyAsync(d + (size_t)fullBlocks * dstPitch, (const char*)src + (size_t)fullBlocks * srcPitch,
                        tail * rowBytes, cudaMemcpyDeviceToHost, stream);
  return e;
}

// Host-only (no device needed): the image rows device `device` of `devices` renders in a tile split, in the order of
// its local rows -- the mapping the kernels apply (lt_device.cuh: lt_image_row) to the row count lt_multi_render hands
// them.  Exposed so that the partition can be checked on a machine without a GPU.
extern "C" int lt_debug_tile_rows(int height, int devices, int device, int32_t* out_rows, int capacity) {
  if (height < 1 || devices < 1 || device < 0 || device >= devices) return LT_ERR_INVALID;
  const int rows = lt_tile_rows_of(height, devices, device);
  if (out_rows) {
    if (capacity < rows) return LT_ERR_INVALID;
    for (int j = 0; j < rows; j++) {
      const int b = j / LT_TILE_ROWS;
      out_rows[j] = (b * devices + device) * LT_TILE_ROWS + (j - b * LT_TILE_ROWS);
    }
  }
  return rows;
}

// The checks of a multi-GPU render call, all before any device works: the arguments, the scene, and every check of the
// single-GPU call (lt_params_to_launch, under `who`).  Out: the normalised parameters and their launch, camera
// included.  Each entry point adds its own split_mode rules.
static int render_prologue(lt_ctx* ctx, const lt_scene* scene, const void* camera28, const lt_render_params* params,
                           const char* who, lt_render_params* P, LtLaunch* L) {
  const std::string w = std::string(who) + ": ";
  if (!scene || !camera28 || !params) return lt_internal_fail(ctx, LT_ERR_INVALID, w + "NULL argument");
  if (scene->parts.size() != ctx->group->ctx.size())
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "the scene was not uploaded through this multi-GPU context");
  if (int rc = lt_params_normalise(ctx, params, w, P)) return rc;
  if (int rc = lt_params_to_launch(ctx, P, L, who)) return rc;
  memcpy(&L->cam, camera28, sizeof(RefCamera));
  if (P->flags & LT_FLAG_STATS)
    return lt_internal_fail(ctx, LT_ERR_UNSUPPORTED, w + "LT_FLAG_STATS counts on a single-GPU context");
  return LT_OK;
}

int lt_multi_render(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params, float* host_out,
                    const LtPluginRun* run) {
  LtGroup* g = ctx->group;
  const char* who = run ? "lt_render_plugin_frames" : "lt_render";
  const std::string w = std::string(who) + ": ";
  lt_render_params P;
  LtLaunch L;
  if (int rc = render_prologue(ctx, scene, camera28, params, who, &P, &L)) return rc;
  const int G = (int)g->ctx.size();
  int split = P.split_mode;
  // a plug-in derives its pixel from blockIdx / get_global_id: it cannot be given a subset of the rows
  if (run && split == LT_SPLIT_TILES)
    return lt_internal_fail(ctx, LT_ERR_UNSUPPORTED, w + "a plug-in cannot render a tile split (use LT_SPLIT_SAMPLES)");
  if (split == LT_SPLIT_AUTO)
    split = (run || (L.frames >= 2 && L.accumMode != LT_ACCUM_NONE)) ? LT_SPLIT_SAMPLES : LT_SPLIT_TILES;
  if (split == LT_SPLIT_SAMPLES && L.accumMode == LT_ACCUM_NONE)
    return lt_internal_fail(ctx, LT_ERR_UNSUPPORTED,
                            w + "a sample split needs an accumulating call (LT_ACCUM_NONE keeps only the last frame)");
  if (split != LT_SPLIT_SAMPLES && split != LT_SPLIT_TILES) return lt_internal_fail(ctx, LT_ERR_INVALID, w + "bad split_mode");
  const bool mean = L.accumMode == LT_ACCUM_RUNNING_MEAN;
  const size_t fullFloats = (size_t)L.width * L.height * L.depth;
  bool useNccl = false;
  if (split == LT_SPLIT_SAMPLES) {
    if (mean && L.frameStride != 1u)
      return lt_internal_fail(ctx, LT_ERR_UNSUPPORTED, w + "a multi-GPU running mean needs frame_stride 1");
    std::string why;
    const char* ex = getenv("LT_MULTI_EXCHANGE");
    useNccl = !(ex && strcmp(ex, "p2p") == 0) && ensure_nccl(g, &why);
    if (!useNccl && !ensure_peers(g, fullFloats, &why))
      return lt_internal_fail(ctx, LT_ERR_UNSUPPORTED, w + "no way to combine the devices' accumulators: " + why);
  }
  // the devices' accumulators are only comparable while split and size stay the same
  if (g->lastSplit != split || g->lastFloats != (long long)fullFloats) {
    int rc = lt_multi_accum_reset(ctx);
    if (rc != LT_OK) return rc;
    g->lastSplit = split;
    g->lastFloats = (long long)fullFloats;
  }

  if (split == LT_SPLIT_TILES) {
    const size_t rowBytes = (size_t)L.width * L.depth * sizeof(float);
    const int rc = fan_out(ctx, G, [&](int k) -> int {
      lt_ctx* c = g->ctx[k];
      const int rows = lt_tile_rows_of(L.height, G, k);
      if (rows == 0) return LT_OK;
      if (int e = use_device(c)) return e;
      if (int e = lt_internal_ensure_out(c, (size_t)L.width * rows * L.depth)) return e;
      LtLaunch Lk = L;  // every G-th block of LT_TILE_ROWS rows from block k
      Lk.height = rows;
      Lk.rowBlock = LT_TILE_ROWS;
      Lk.rowStride = G;
      Lk.rowPhase = k;
      if (int e = lt_internal_render(c, scene->parts[k], Lk, c->dOut.get())) return e;
      if (!host_out) return LT_OK;
      cudaError_t e =
          lt_copy_row_blocks(host_out, c->dOut.get(), LT_TILE_ROWS * rowBytes, rowBytes, rows, G, k, c->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
      return e == cudaSuccess ? LT_OK : lt_internal_fail(c, LT_ERR_CUDA, std::string("tile copy: ") + cudaGetErrorString(e));
    });
    if (rc != LT_OK) return rc;
  } else {
    // ---- sample split ----
    // running mean: new = old * fc/(fc+F) + sum(samples)/(fc+F)  (fc = frames already in the accumulator; 0 discards it,
    // like frameCount == 0 in accumulator.frag:10-19)
    const double total = (double)L.cam.frameCount + (double)L.frames;
    const float weight = mean ? (float)(1.0 / total) : L.accumWeight;
    const float keep = mean ? (float)((double)L.cam.frameCount / total) : 1.0f;
    const int rc = fan_out(ctx, G, [&](int k) -> int {
      lt_ctx* c = g->ctx[k];
      if (int e = use_device(c)) return e;
      if (int e = lt_internal_ensure_out(c, fullFloats)) return e;
      // device 0 carries the accumulator that was there before this call, the others start from zero
      if (k == 0) {
        if (keep == 0.0f) cudaMemsetAsync(c->dOut.get(), 0, fullFloats * sizeof(float), c->stream);
        else if (keep != 1.0f) k_scale<<<c->stats.sm_count * 8, 256, 0, c->stream>>>(c->dOut.get(), fullFloats, keep);
      } else {
        cudaMemsetAsync(c->dOut.get(), 0, fullFloats * sizeof(float), c->stream);
      }
      int e = LT_OK;
      if (k < L.frames) {  // frames k, k+G, ... < L.frames, a weighted sum
        LtLaunch Lk = L;
        Lk.frames = (L.frames - k + G - 1) / G;
        Lk.frameStride = L.frameStride * (uint32_t)G;
        Lk.accumMode = LT_ACCUM_WEIGHTED_SUM;
        Lk.accumWeight = weight;
        Lk.cam.frameCount = L.cam.frameCount + (uint32_t)k * L.frameStride;
        if (run) {
          lt_render_params Pk = P;
          Pk.frames = Lk.frames;
          Pk.frame_stride = Lk.frameStride;
          Pk.accum_mode = Lk.accumMode;
          Pk.accum_weight = weight;
          e = lt_internal_render_plugin(c, scene->parts[k], Lk.cam, Pk, *run, false, who);
        } else {
          e = lt_internal_render(c, scene->parts[k], Lk, c->dOut.get());
        }
      }
      cudaEventRecord(g->events[k][kRendered], c->stream);
      return e;
    });
    if (rc != LT_OK) return rc;
    // ---- the exchange step: one all-reduce(sum) of W*H*depth floats ----
    if (useNccl) {
      g_nccl.groupStart();
      for (int k = 0; k < G; k++) {
        lt_ctx* c = g->ctx[k];
        ncclResult_t r =
            g_nccl.allReduce(c->dOut.get(), c->dOut.get(), fullFloats, ncclFloat, ncclSum, g->comms[k], c->stream);
        if (r != ncclSuccess) {
          g_nccl.groupEnd();
          return lt_internal_fail(ctx, LT_ERR_CUDA, std::string("ncclAllReduce: ") + g_nccl.getErrorString(r));
        }
      }
      ncclResult_t r = g_nccl.groupEnd();
      if (r != ncclSuccess) return lt_internal_fail(ctx, LT_ERR_CUDA, std::string("ncclGroupEnd: ") + g_nccl.getErrorString(r));
    } else {
      PeerPointers src;
      for (int k = 0; k < G; k++) src.p[k] = g->ctx[k]->dOut.get();
      for (int k = 0; k < G; k++) {
        lt_ctx* c = g->ctx[k];
        cudaSetDevice(c->device);
        for (int j = 0; j < G; j++)
          if (j != k) cudaStreamWaitEvent(c->stream, g->events[j][kRendered], 0);  // every device has finished rendering
        k_sum_peers<<<c->stats.sm_count * 4, 256, 0, c->stream>>>(g->sumBuf[k].get(), src, G, fullFloats);
        cudaEventRecord(g->events[k][kSummed], c->stream);
      }
      for (int k = 0; k < G; k++) {  // nobody overwrites its accumulator while a peer still reads it
        lt_ctx* c = g->ctx[k];
        cudaSetDevice(c->device);
        for (int j = 0; j < G; j++)
          if (j != k) cudaStreamWaitEvent(c->stream, g->events[j][kSummed], 0);
        cudaMemcpyAsync(c->dOut.get(), g->sumBuf[k].get(), fullFloats * sizeof(float), cudaMemcpyDeviceToDevice,
                        c->stream);
      }
    }
    lt_ctx* c0 = g->ctx[0];
    cudaSetDevice(c0->device);
    if (host_out)
      if (int e = lt_internal_download(c0, host_out, c0->dOut.get(), fullFloats * sizeof(float)))
        return lt_internal_fail(ctx, e, lt_last_error(c0));
  }
  // the devices rendered asynchronously: wait for each, then time the kernels of those that rendered
  for (lt_ctx* c : g->ctx) {
    cudaSetDevice(c->device);
    const cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess)
      return lt_internal_fail(ctx, LT_ERR_CUDA, std::string("multi-GPU render: ") + cudaGetErrorString(e));
    float ms = 0.0f;
    if (c->stats.kernel_launches > 0 && cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]) == cudaSuccess) c->stats.kernel_ms = ms;
    cudaGetLastError();
  }
  merge_render_stats(ctx);
  return LT_OK;
}

// Views of one call: device k renders views k, k + G, ... with the single-GPU path and copies each into its place in
// host_out.  Views are independent, so no collective is involved.
int lt_multi_render_views(lt_ctx* ctx, lt_scene* scene, const RefCamera* cams, int count, const lt_render_params* params,
                          float* host_out) {
  LtGroup* g = ctx->group;
  lt_render_params P;
  LtLaunch L;
  if (int rc = render_prologue(ctx, scene, cams, params, "lt_render_views", &P, &L)) return rc;
  if (P.split_mode != LT_SPLIT_AUTO)
    return lt_internal_fail(ctx, LT_ERR_INVALID,
                            "lt_render_views: views are dealt to the devices whole: split_mode must be LT_SPLIT_AUTO");
  const int G = (int)g->ctx.size();
  const int rc = fan_out(ctx, std::min(G, count), [&](int k) {
    std::vector<RefCamera> mine;
    for (int v = k; v < count; v += G) mine.push_back(cams[v]);
    return lt_internal_render_views(g->ctx[k], scene->parts[k], L, mine.data(), (int)mine.size(), host_out, k, G);
  });
  if (rc != LT_OK) return rc;
  merge_render_stats(ctx);
  return LT_OK;
}

// lt_render_adaptive on several devices: device k runs the whole adaptive loop on its own rows of the row partition (every
// G-th block of LT_TILE_ROWS rows from block k) in full-size buffers of its own context, and copies those rows of the
// mean and the frame counts into the host buffers.  Every pixel's rounds depend on that pixel alone, so the result is
// the single-GPU call's, and no collective is needed.
int lt_multi_render_adaptive(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                             const lt_adaptive_params* aparams, float* host_out, uint32_t* host_frames,
                             lt_adaptive_result* out_result) {
  LtGroup* g = ctx->group;
  const char* who = "lt_render_adaptive";
  lt_render_params P;
  LtLaunch L;
  if (int rc = render_prologue(ctx, scene, camera28, params, who, &P, &L)) return rc;
  if (P.split_mode != LT_SPLIT_AUTO && P.split_mode != LT_SPLIT_TILES)
    return lt_internal_fail(ctx, LT_ERR_INVALID, std::string(who) + ": the devices share the image by rows: split_mode "
                                                 "must be LT_SPLIT_AUTO or LT_SPLIT_TILES");
  LtAdaptive A;
  if (int rc = lt_adaptive_check(ctx, L, aparams, who, &A)) return rc;
  const int G = (int)g->ctx.size();
  std::vector<lt_adaptive_result> res(G, lt_adaptive_result{});
  const int rc = fan_out(ctx, G, [&](int k) {
    return lt_internal_render_adaptive(g->ctx[k], scene->parts[k], L, A, host_out, host_frames, G, k, &res[k]);
  });
  if (rc != LT_OK) return rc;
  lt_adaptive_result r = {};
  for (int k = 0; k < G; k++) {
    if (res[k].rounds > r.rounds) r.rounds = res[k].rounds;
    r.pixel_frames += res[k].pixel_frames;
    r.pixels_unconverged += res[k].pixels_unconverged;
  }
  if (out_result) *out_result = r;
  merge_render_stats(ctx);
  return LT_OK;
}
