// lt_internal.h -- types shared by the CUDA kernels and the C-ABI layer of liblt_b200.so.
// Host-visible mirrors of the reference buffer layouts plus the re-flattened device layouts.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "lens_trace_b200_device.cuh"  // buffer layouts shared with plug-in kernels

#include "lt_device_types.h"  // LtLaunch, LtCounters (shared with plug-in builds)

struct lt_ctx;
int lt_internal_ctx_device(const lt_ctx* ctx);  // lt_capi.cu

// launchers implemented in lt_kernels.cu (all asynchronous on `stream`; return launches made)
int lt_launch_reflatten(const RefNode* dNodes, int nodeCount, const RefPrim* dPrims, int primCount,
                        const int* dInnerRank, LtWideNode* dWide, LtTri* dTris, cudaStream_t stream);
int lt_launch_inner_flags(const RefNode* dNodes, int nodeCount, int* dFlags, cudaStream_t stream);
int lt_launch_build_threaded(const RefNode* dNodes, int nodeCount, LtThreadNode* dOut, cudaStream_t stream);
size_t lt_scan_temp_bytes(int n);
int lt_launch_exclusive_scan(void* dTemp, size_t tempBytes, const int* dIn, int* dOut, int n, cudaStream_t stream);
// dWork: one zero-initialisable int of device memory (work counter of the persistent kernels)
int lt_launch_render(const LtSceneDev& sc, const LtLaunch& L, float* dOut, LtCounters* dCounters, int* dWork,
                     int smCount, cudaStream_t stream);
int lt_launch_primary_hits(const LtSceneDev& sc, const RefCamera& cam, int kernel, int flags, int width, int height,
                           int* dIds, int* dHit, float* dTuv, cudaStream_t stream);
int lt_launch_debug_random(const float* fx, const float* fy, const float* seed, int n, float* out, cudaStream_t stream);
int lt_launch_debug_hemisphere(const float* u1, const float* u2, const float* up, int n, float* out,
                               cudaStream_t stream);

// wavefront pipeline (lt_wavefront.cu)
size_t lt_wf_workspace_bytes_padded(long long nPaths);
size_t lt_wf_primary_hits_bytes(long long pixels);  // per-launch primary hit records, kept behind the batch workspaces
// traceEvents: optional pool of 2*maxTraceLaunches events; when given, every traversal launch is bracketed by a
// pair of events and *traceLaunches receives the number of pairs recorded
// aux: a second stream + events (fork, one batch-order event per stream) for overlapping consecutive batches (the
// L1-bound trace kernel of one batch runs beside the DRAM-bound shade kernel of the other and fills the tail of the
// persistent kernels); `workspace` then holds two batch workspaces of
// lt_wf_workspace_bytes_padded(batchFrames * pixels) each.  aux == nullptr: one stream.
struct LtWfAux {
  cudaStream_t extra;  // odd batches; even batches run on the caller's stream
  cudaEvent_t fork, order[2];
};
// pairKinds: optional, one LT_TIMED_* per recorded pair; when given, the shade / primary-shade / accumulate launches
// are bracketed as well (per-kernel times of a serialised step)
enum { LT_TIMED_TRAVERSAL = 0, LT_TIMED_SHADE = 1, LT_TIMED_PRIMARY_SHADE = 2, LT_TIMED_ACCUMULATE = 3, LT_TIMED_KINDS = 4 };
int lt_launch_render_wavefront(const LtSceneDev& sc, const LtLaunch& L, float* dOut, LtCounters* dCounters,
                               void* workspace, int batchFrames, int smCount, cudaStream_t stream,
                               cudaEvent_t* traceEvents, int maxTraceLaunches, int* traceLaunches,
                               unsigned char* pairKinds, const LtWfAux* aux);

// user-written CUDA kernels with the reference's plug-in ABI (lt_plugin.cu)
#include <string>
struct LtPlugin;
LtPlugin* lt_plugin_compile(const char* path, std::string* err);
void lt_plugin_free(LtPlugin* p);
int lt_plugin_launch(LtPlugin* p, int kernelMode, const LtSceneDev* sceneDev, const void* dNodes, const void* dPrims,
                     const void* dMats, const void* dLights, const void* dCamera, float* dOut, int width, int height,
                     int depth, int bx, int by, cudaStream_t stream, std::string* err);

// ---- context and scene objects behind the C-ABI handles (lt_capi.cu; lt_multi.cu for multi-GPU contexts) ----
#include <vector>
#include "lens_trace_b200.h"
struct LtGroup;     // lt_multi.cu: the devices of a multi-GPU context
struct LtCopyPool;  // lt_capi.cu: host threads that copy staged chunks into a pageable destination

struct lt_ctx {
  int device = 0;
  LtGroup* group = nullptr;  // non-NULL: a multi-GPU context (lt_ctx_create_multi); the fields below are unused
  cudaStream_t ownStream = nullptr;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::string error;
  float* dOut = nullptr;  // context-owned output / accumulator
  size_t outFloats = 0;
  LtCounters* dCounters = nullptr;
  int* dWork = nullptr;  // work counters of the persistent kernels
  std::vector<cudaEvent_t> traceEvents;  // pairs of events around launches (timed when synchronous)
  std::vector<unsigned char> pairKinds;  // LT_TIMED_* of every pair
  std::vector<LtPlugin*> plugins;  // compiled user kernels, by id
  RefCamera* dCamera = nullptr;    // camera buffer for plug-in launches
  void* wfWorkspace = nullptr;  // wavefront path state / ray queues (two batch workspaces when batches overlap)
  size_t wfBytes = 0;
  LtWfAux wfAux = {};           // second stream + events for overlapping consecutive wavefront batches
  size_t totalMem = 0;
  char* stage = nullptr;  // pinned staging buffer of lt_render's copy into a pageable destination
  size_t stageBytes = 0;
  std::vector<cudaEvent_t> stageEvents;  // one per 2 MB chunk
  LtCopyPool* copyPool = nullptr;
  lt_stats stats = {};
};

struct lt_scene {
  std::vector<lt_scene*> parts;  // scene of a multi-GPU context: one uploaded copy per device (then nothing else is set)
  RefNode* dNodes = nullptr;
  RefPrim* dPrims = nullptr;
  RefMaterial* dMats = nullptr;
  RefLights* dLights = nullptr;
  LtWideNode* dWide = nullptr;
  LtTri* dTris = nullptr;
  LtThreadNode* dThread = nullptr;  // 8 octant copies in visit order, then 8 pruned ones, small scenes only
  int threadStride = 0;             // records per pruned copy
  LtThreadNode* dThreadBig = nullptr;  // the same for a large scene, built on the device, for coherent-ray launches
  LtSceneDev dev = {};
};


// multi-GPU contexts (lt_multi.cu); every entry point of lt_capi.cu forwards to these when ctx->group is set
int lt_multi_scene_upload(lt_ctx* ctx, const void* nodes, uint64_t node_bytes, const void* primitives,
                          uint64_t primitive_bytes, const void* materials, uint64_t material_bytes,
                          const void* light_container, uint64_t light_bytes, lt_scene** out_scene);
void lt_multi_scene_release(lt_ctx* ctx, lt_scene* scene);
int lt_multi_render(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params, float* host_out);
void lt_multi_destroy(lt_ctx* ctx);
int lt_multi_accum_reset(lt_ctx* ctx);
int lt_internal_fail(lt_ctx* ctx, int code, const std::string& msg);  // sets the context's (and the thread's) last error
int lt_internal_ensure_out(lt_ctx* ctx, size_t floats);
// device -> the caller's host buffer on ctx's stream, synchronous (staged through pinned memory when pageable)
int lt_internal_download(lt_ctx* ctx, float* host_out, const float* dSrc, size_t bytes);
// one device's share of a render call: like lt_render_device, with the row window of a tile split
int lt_internal_render_rows(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                            float* device_out, int fullHeight, int rowBlock, int rowStride, int rowPhase, int sync);

// device-side BVH construction in the reference's flattened layout (lt_bvh.cu)
enum LtBvhBuilder { LT_BVH_LBVH, LT_BVH_PLOC };
size_t lt_bvh_scratch_bytes(int n, LtBvhBuilder builder);
int lt_launch_bvh_build(LtBvhBuilder builder, const RefPrim* dPrims, int n, const RefMaterial* dMats, int matCount,
                        RefNode* dNodes, RefPrim* dOrderedPrims, RefLights* dLights, void* scratch, size_t scratchBytes,
                        int* outMaxDepth, cudaStream_t stream);
