// lt_internal.h -- types shared by the CUDA kernels and the C-ABI layer of liblt_b200.so.
// Host-visible mirrors of the reference buffer layouts plus the re-flattened device layouts.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "lens_trace_b200.h"
#include "lens_trace_b200_device.cuh"  // buffer layouts shared with plug-in kernels

#include "lt_device_types.h"  // LtLaunch, LtCounters (shared with plug-in builds)

struct lt_ctx;
int lt_internal_ctx_device(const lt_ctx* ctx);  // lt_capi.cu

// A row partition of an image into parts: part g owns every parts-th block of LT_TILE_ROWS rows from block g (the tile
// split of a multi-GPU context, lt_render_adaptive's partition of its devices).  lt_tile_rows_of: the rows part g owns.
#define LT_TILE_ROWS 8
int lt_tile_rows_of(int height, int parts, int g);  // lt_multi.cu

// ---- launch plan (lt_plan.cpp: lt_plan_render): every choice of which kernels run, on which tree, at which sizes ----
// k_flat, k_flat_stream, k_path, or the wavefront pipeline (lt_wavefront.cu)
enum LtPipeline { LT_PIPE_FLAT, LT_PIPE_FLAT_STREAM, LT_PIPE_PATH, LT_PIPE_WAVEFRONT };
// the tree the traversal kernels walk: child-pair nodes with a stack, or the host- or device-built threaded copies
enum LtTree { LT_TREE_CHILD_PAIR, LT_TREE_HOST_THREADED, LT_TREE_DEVICE_THREADED };
// Per-context limits of the plan and of the upload-time layout; lt_debug_ctx_limits changes them for tests.
struct LtLimits {
  int threadedMaxNodes = 65536;  // trees up to this size get host-built threaded copies (16 MB of records at the limit)
  int streamMinNodes = 100000;   // deterministic kernels on scenes this large: k_flat_stream
};
struct LtPlan {
  int error;            // LT_OK, or what lt_render returns (with `message`)
  const char* message;
  LtPipeline pipeline;
  LtTree tree;
  bool stats, cull;
  bool forced;          // the caller asked for the wavefront: no megakernel in its place when its workspace fails
  // wavefront only
  int batchFrames, streams, rounds, samplesPerFrame;
  bool sharedPrimary;   // camera rays traced once per pixel for all frames of the launch
  bool classify;        // ... and pixels without paths (background, light) skipped
  size_t workspaceBytes;
  // dynamic shared memory of the stack-traversal kernels, and of the trace kernel (threaded or stack)
  size_t smemStack, smemTrace;
  int blocksPerSm;      // persistent kernels (k_flat_stream, k_wf_trace)
  int grid;             // blocks: persistent grid, or one block per 16x8 tile (k_flat, k_path)
};
struct LtSceneFacts {
  int nodeCount, stackDepth;
  LtTree copies;  // the threaded copies the scene has (LT_TREE_CHILD_PAIR: none)
};
LtTree lt_plan_threaded_copies(int nNodes, size_t totalMem, const LtLimits& lim);
LtPlan lt_plan_primary_hits(int flags, int width, int height, const LtSceneFacts& s);
// listed >= 0: a masked launch (lt_render_masked_device) of that many listed pixels, planned for them instead of the
// width x height image
LtPlan lt_plan_render(const LtLaunch& L, const LtSceneFacts& s, size_t totalMem, int smCount, const LtLimits& lim,
                      int views = 1, long long listed = -1);
// The struct-size check of a caller's lt_render_params and its zero-filled copy at *P, which has the current
// struct_size; `w` starts the error message ("lt_render: ")
int lt_params_normalise(lt_ctx* ctx, const lt_render_params* params, const std::string& w, lt_render_params* P);
// lt_render_params -> the launch descriptor (all of it but the camera), with lt_render's checks; `who` names the entry
// point in error messages
int lt_params_to_launch(lt_ctx* ctx, const lt_render_params* params, LtLaunch* L, const char* who = "lt_render");
// LT_ERR_UNSUPPORTED (message set) for an image a masked call cannot number with 32-bit pixel indices
int lt_masked_image_check(lt_ctx* ctx, const LtLaunch& L, const char* who);
// lt_render_adaptive's parameters after their checks: defaults applied (floor 0 -> 1e-4, round_frames 0 -> frames)
struct LtAdaptive {
  float target, floor;
  int roundFrames, maxFrames;
};
// The checks of lt_render_adaptive that need no device, on the launch lt_params_to_launch made (camera included)
int lt_adaptive_check(lt_ctx* ctx, const LtLaunch& L, const lt_adaptive_params* a, const char* who, LtAdaptive* out);
// frames of the round that follows `done` frames of the call, 0 when max_frames is reached
inline int lt_adaptive_next_frames(const LtAdaptive& A, int done) {
  return A.maxFrames - done < A.roundFrames ? A.maxFrames - done : A.roundFrames;
}

// ---- host tree builders (lt_tree.cpp) ----
// Host-side validation of the reference node array (bounds of every index the kernels will follow) and the depth the
// traversal stack needs; nonzero with *why set when it fails.
int lt_validate_tree(const RefNode* nodes, int nodeCount, int primCount, int* stackDepth, std::string* why);
// The threaded copies lt_scene_upload makes of a small tree, and the rank table; returns the pruned stride.
int lt_build_threaded(const RefNode* nodes, int n, int primCount, std::vector<LtThreadNode>& out,
                      std::vector<int>& rank);

// launchers implemented in lt_kernels.cu (all asynchronous on `stream`; return launches made).  The launchers of the
// traversal kernels take the scene with the plan's tree in `tnodes`.
int lt_launch_reflatten(const RefNode* dNodes, int nodeCount, const RefPrim* dPrims, int primCount,
                        const int* dInnerRank, LtWideNode* dWide, LtTri* dTris, cudaStream_t stream);
int lt_launch_inner_flags(const RefNode* dNodes, int nodeCount, int* dFlags, cudaStream_t stream);
int lt_launch_build_threaded(const RefNode* dNodes, int nodeCount, LtThreadNode* dOut, cudaStream_t stream);
size_t lt_scan_temp_bytes(int n);
int lt_launch_exclusive_scan(void* dTemp, size_t tempBytes, const int* dIn, int* dOut, int n, cudaStream_t stream);
// dWork: one zero-initialisable int of device memory (work counter of the persistent kernels)
// list: the pixels of a masked launch (k_flat / k_path over the list, grid = plan.grid), or nullptr
int lt_launch_render(const LtSceneDev& sc, const LtPlan& plan, const LtLaunch& L, float* dOut, LtCounters* dCounters,
                     int* dWork, cudaStream_t stream, const LtList* list = nullptr);
// the set pixels of a width x height byte mask (nullptr: all) -> dList, their number -> *dCount (k_mask_compact)
int lt_launch_mask_compact(const unsigned char* dMask, int width, int height, int* dList, int* dCount,
                           cudaStream_t stream);
int lt_launch_list_reverse(int* dList, int count, cudaStream_t stream);  // the list in reverse order, in place
// lt_render_adaptive: the first list of part `part` of a `parts`-way row partition (k_rows_compact), and the selection
// after a round of `count` listed pixels with n frames each: pixels that go on -> dNext (nullptr: only counted), their
// number -> *dNextCount, n -> dFrames[pixel] when given (k_adaptive_select)
int lt_launch_rows_compact(int width, int height, int parts, int part, int* dList, int* dCount, cudaStream_t stream);
int lt_launch_adaptive_select(const int* dList, int count, const float* dMean, int depth, const float* dM2,
                              unsigned* dFrames, unsigned n, float target, float floor, int* dNext, int* dNextCount,
                              cudaStream_t stream);
int lt_launch_primary_hits(const LtSceneDev& sc, const LtPlan& plan, const RefCamera& cam, int kernel, int flags,
                           int width, int height, int* dIds, int* dHit, float* dTuv, cudaStream_t stream);
// Dynamic shared memory beyond 48 KB needs an opt-in per kernel and device: given once for every traversal kernel
// (both files), the first time a launch asks for more.
void lt_opt_in_traversal_smem(size_t smem);
extern const void* const lt_wf_traversal_kernels[10];  // lt_wavefront.cu
int lt_launch_debug_random(const float* fx, const float* fy, const float* seed, int n, float* out, cudaStream_t stream);
int lt_launch_debug_hemisphere(const float* u1, const float* u2, const float* up, int n, float* out,
                               cudaStream_t stream);

// wavefront pipeline (lt_wavefront.cu)
size_t lt_wf_workspace_bytes_padded(long long nPaths);
size_t lt_wf_primary_hits_bytes(long long pixels);  // per-launch primary hit records, kept behind the batch workspaces
// a call of several views: views a batch of batchFrames (view, frame) pairs touches at most, and the primary records of
// that many views, kept per batch workspace instead of the launch's one set
int lt_wf_views_per_batch(int batchFrames, int frames, int views);
size_t lt_wf_view_records_bytes(long long pixels, int viewsPerBatch);
// The views of one lt_render_views call on one device: view v renders camera cams[v] into dOut + v * W * H * depth.
struct LtViews {
  int count;
  const RefCamera* cams;         // host memory
  const unsigned* dFrameCounts;  // device memory: frameCount of each (view, frame) pair, view-major (count * frames)
};
// traceEvents: optional pool of 2*maxTraceLaunches events; when given, every traversal launch is bracketed by a
// pair of events and *traceLaunches receives the number of pairs recorded
// aux: a second stream + events (fork, one batch-order event per stream), used when the plan overlaps consecutive
// batches on two streams (the L1-bound trace kernel of one batch runs beside the DRAM-bound shade kernel of the other
// and fills the tail of the persistent kernels); `workspace` then holds two batch workspaces of
// lt_wf_workspace_bytes_padded(batchFrames * pixels) each.
struct LtWfAux {
  cudaStream_t extra;  // odd batches; even batches run on the caller's stream
  cudaEvent_t fork, order[2];
};
// pairKinds: optional, one LT_TIMED_* per recorded pair; when given, the shade / primary-shade / accumulate launches
// are bracketed as well (per-kernel times of a serialised step)
enum { LT_TIMED_TRAVERSAL = 0, LT_TIMED_SHADE = 1, LT_TIMED_PRIMARY_SHADE = 2, LT_TIMED_ACCUMULATE = 3, LT_TIMED_KINDS = 4 };
int lt_launch_render_wavefront(const LtSceneDev& sc, const LtPlan& plan, const LtLaunch& L, float* dOut,
                               LtCounters* dCounters, void* workspace, int smCount, cudaStream_t stream,
                               cudaEvent_t* traceEvents, int maxTraceLaunches, int* traceLaunches,
                               unsigned char* pairKinds, const LtWfAux* aux, const LtViews* views,
                               const LtList* list = nullptr);

// user-written CUDA kernels with the reference's plug-in ABI (lt_plugin.cu)
struct LtPlugin;
// A compiled plug-in, not yet loaded on a device: compiled once, loaded on every device of a multi-GPU context.
struct LtPluginImage {
  std::string path;
  bool openclC = false;
  std::vector<char> cubin;
};
bool lt_plugin_compile(const char* path, LtPluginImage* img, std::string* err);
LtPlugin* lt_plugin_module_load(const LtPluginImage& img, std::string* err);  // into the calling thread's current context
void lt_plugin_free(LtPlugin* p);
int lt_plugin_publish_scene(LtPlugin* p, const LtSceneDev* sceneDev, cudaStream_t stream, std::string* err);
int lt_plugin_launch(LtPlugin* p, int kernelMode, const LtSceneDev* sceneDev, const void* dNodes, const void* dPrims,
                     const void* dMats, const void* dLights, const void* dCamera, float* dOut, int width, int height,
                     int depth, int bx, int by, cudaStream_t stream, std::string* err);
// user-written OpenCL C kernels (.cl): translated onto lt_opencl_c.cuh, compiled by NVRTC, launched like the reference's
// OpenCL backend launches them
bool lt_plugin_is_opencl_c(const LtPlugin* p);
bool lt_plugin_compile_cl_only(const char* path, std::string* err);  // NVRTC only, no driver
std::string lt_cl_translate(const std::string& src, bool* contractOff, bool* deviceApi,
                            std::vector<std::pair<std::string, int>>* kernels);
bool lt_plugin_cl_shape(int width, int height, int* wbx, int* wby, int* gx, int* gy, std::string* err);
// dynamic shared memory of a block of `threads` threads of a plug-in on a scene (the device API's traversal stacks);
// false with `err` set when they do not fit
bool lt_plugin_smem(const LtPlugin* p, int kernelMode, const LtSceneDev* sceneDev, unsigned threads, unsigned* smem,
                    std::string* err);
int lt_plugin_launch_cl(LtPlugin* p, int kernelMode, const LtSceneDev* sceneDev, const void* dNodes, const void* dPrims,
                        const void* dMats, const void* dLights, const void* dCamera, float* dOut, int width, int height,
                        int depth, int wbx, int wby, int gx, int gy, cudaStream_t stream, std::string* err);
// k_plugin_accumulate (lt_kernels.cu): folds one plug-in frame (`sample`) into the accumulator `acc` with FrameSink, as
// L.accumMode / L.accumWeight / L.cam.frameCount say; 3 channels per pixel at stride L.depth
int lt_launch_plugin_accumulate(const LtLaunch& L, const float* sample, float* acc, int smCount, cudaStream_t stream);
// What a plug-in call launches besides its frames (host-side only).
struct LtPluginRun {
  int id;
  int kernelMode;
  int bx, by;    // CUDA block of a .cu plug-in, work-group of a .cl plug-in
  int wbx, wby;  // work block of a .cl plug-in (as normalised by lt_plugin_cl_shape)
};

// ---- owners of the CUDA resources of the C-ABI objects: each releases what it holds when it goes.  The device they
// were made on must be current then, as for the bare release calls. ----
// n elements of T in device memory, or (Pinned) in page-locked host memory
template <class T, bool Pinned = false>
class LtBuf {
 public:
  LtBuf() = default;
  LtBuf(LtBuf&& o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr, o.n_ = 0; }
  ~LtBuf() { reset(); }
  // At least n elements: when fewer are held, the old buffer is freed first and a new one allocated, which keeps
  // nothing of the old contents; empty (count 0) when the allocation fails.
  cudaError_t grow(size_t n) {
    if (n_ >= n) return cudaSuccess;
    reset();
    const cudaError_t e = Pinned ? cudaMallocHost((void**)&p_, n * sizeof(T)) : cudaMalloc((void**)&p_, n * sizeof(T));
    if (e != cudaSuccess) p_ = nullptr;
    else n_ = n;
    return e;
  }
  void reset() {
    if (!p_) return;
    if constexpr (Pinned) cudaFreeHost(p_);
    else cudaFree(p_);
    p_ = nullptr, n_ = 0;
  }
  T* get() const { return p_; }
  size_t count() const { return n_; }
  size_t bytes() const { return n_ * sizeof(T); }

 private:
  T* p_ = nullptr;
  size_t n_ = 0;
};
// events, handed to launchers as one contiguous array of raw handles
class LtEvents {
 public:
  LtEvents() = default;
  LtEvents(LtEvents&& o) noexcept : ev_(std::move(o.ev_)) { o.ev_.clear(); }
  ~LtEvents() { reset(); }
  // at least n events, the new ones made with `flags`; those made before a failed creation are kept
  cudaError_t grow(size_t n, unsigned flags) {
    while (ev_.size() < n) {
      cudaEvent_t e;
      const cudaError_t r = cudaEventCreateWithFlags(&e, flags);
      if (r != cudaSuccess) return r;
      ev_.push_back(e);
    }
    return cudaSuccess;
  }
  void reset() {
    for (cudaEvent_t e : ev_) cudaEventDestroy(e);
    ev_.clear();
  }
  cudaEvent_t operator[](size_t k) const { return ev_[k]; }
  cudaEvent_t* data() { return ev_.data(); }

 private:
  std::vector<cudaEvent_t> ev_;
};
// a non-blocking stream
class LtStream {
 public:
  LtStream() = default;
  LtStream(const LtStream&) = delete;
  LtStream& operator=(const LtStream&) = delete;
  ~LtStream() {
    if (s_) cudaStreamDestroy(s_);
  }
  cudaError_t create() {
    const cudaError_t e = cudaStreamCreateWithFlags(&s_, cudaStreamNonBlocking);
    if (e != cudaSuccess) s_ = nullptr;
    return e;
  }
  cudaStream_t get() const { return s_; }

 private:
  cudaStream_t s_ = nullptr;
};

// ---- context and scene objects behind the C-ABI handles (lt_capi.cu; lt_multi.cu for multi-GPU contexts) ----
struct LtGroup;     // lt_multi.cu: the devices of a multi-GPU context
struct LtCopyPool;  // lt_capi.cu: host threads that copy staged chunks into a pageable destination

struct lt_ctx {
  int device = 0;
  LtGroup* group = nullptr;  // non-NULL: a multi-GPU context (lt_ctx_create_multi); the fields below are unused
  LtStream ownStream;
  cudaStream_t stream = nullptr;  // ownStream, or the caller's (lt_ctx_set_stream), which is never destroyed here
  LtEvents ev;                    // [0], [1]: around the kernels of a call (timed)
  std::string error;
  LtBuf<float> dOut;  // context-owned output / accumulator
  LtBuf<LtCounters> dCounters;
  LtBuf<int> dWork;  // work counters of the persistent kernels
  LtEvents traceEvents;                  // pairs of events around launches (timed when synchronous)
  std::vector<unsigned char> pairKinds;  // LT_TIMED_* of every pair
  std::vector<LtPlugin*> plugins;  // compiled user kernels, by id
  LtBuf<RefCamera> dCamera;        // camera records of a plug-in call, one per frame
  LtBuf<float> dSample;            // one plug-in frame of an accumulating call, folded into dOut
  LtBuf<char> wfWorkspace;  // wavefront path state / ray queues (two batch workspaces when batches overlap)
  LtStream wfExtra;         // LtWfAux of the wavefront launches: the second stream, and its fork and order[2] events
  LtEvents wfEvents;
  LtBuf<float> dViews;  // the images of an lt_render_views call (not the accumulator dOut)
  LtBuf<unsigned> dViewFrameCounts;  // LtViews::dFrameCounts of a wavefront views launch
  LtBuf<int> dMaskList;  // lt_render_masked_device: the listed pixels' count, then (from kMaskListAt) the list
  bool reverseList = false;  // lt_debug_ctx_list_order: masked calls render their list in reverse order
  LtBuf<float> dAdaptive;  // host-form lt_render_adaptive: mean, m2 (3 per pixel), frame counts (one per pixel)
  int adaptiveParts = 1, adaptivePart = 0;  // lt_debug_ctx_adaptive_part: adaptive calls render this part's rows only
  size_t totalMem = 0;
  LtBuf<char, true> stage;  // pinned staging buffer of lt_render's copy into a pageable destination
  LtEvents stageEvents;     // one per staged chunk
  std::unique_ptr<LtCopyPool> copyPool;
  LtLimits limits;
  lt_stats stats = {};
  lt_ctx();  // both in lt_capi.cu, where LtCopyPool is complete
  ~lt_ctx();
};

struct lt_scene {
  std::vector<lt_scene*> parts;  // scene of a multi-GPU context: one uploaded copy per device (then nothing else is set)
  LtBuf<RefNode> dNodes;
  LtBuf<RefPrim> dPrims;
  LtBuf<RefMaterial> dMats;
  LtBuf<RefLights> dLights;
  LtBuf<LtWideNode> dWide;
  LtBuf<LtTri> dTris;
  LtBuf<LtThreadNode> dThread;  // 8 octant copies in visit order, then 8 pruned ones, small scenes only
  int threadStride = 0;         // records per pruned copy
  LtBuf<int> dRank;             // LtSceneDev::rank, when the pruned copies are a traversal tree
  LtBuf<LtThreadNode> dThreadBig;  // the same for a large scene, built on the device, for coherent-ray launches
  LtBuf<int> dRefit;  // from the first lt_scene_refit on: parents, arrival flags, inner-node ranks (n each), check flag
  bool refitDerived = false;  // dRefit holds the parents and the inner-node ranks
  int refitLeaves = 0;        // 1: every leaf's primitive range lies in the primitive buffer, -1: not, 0: not checked
  LtSceneDev dev = {};
};


// multi-GPU contexts (lt_multi.cu); every entry point of lt_capi.cu forwards to these when ctx->group is set
int lt_multi_scene_upload(lt_ctx* ctx, const void* nodes, uint64_t node_bytes, const void* primitives,
                          uint64_t primitive_bytes, const void* materials, uint64_t material_bytes,
                          const void* light_container, uint64_t light_bytes, lt_scene** out_scene);
void lt_multi_scene_release(lt_ctx* ctx, lt_scene* scene);
// lt_scene_refit on every device's copy (arguments already checked)
int lt_internal_refit(lt_ctx* ctx, lt_scene* scene, const void* primitives);  // one copy, host primitives checked
int lt_multi_scene_refit(lt_ctx* ctx, lt_scene* scene, const void* primitives);
// run: NULL renders the built-in kernel of params, otherwise the plug-in of run (loaded on every device)
int lt_multi_render(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params, float* host_out,
                    const LtPluginRun* run);
int lt_multi_plugin_load(lt_ctx* ctx, const LtPluginImage& img, int* out_plugin_id);
const std::vector<LtPlugin*>& lt_multi_plugins(const lt_ctx* ctx);  // device 0's; every device holds the same ids
void lt_multi_destroy(lt_ctx* ctx);
int lt_multi_accum_reset(lt_ctx* ctx);
int lt_internal_fail(lt_ctx* ctx, int code, const std::string& msg);  // sets the context's (and the thread's) last error
// The start of every call's statistics: all of ctx->stats zero but sm_count and upload_ms (the last upload or refit).
// A call then sets only what it measured.
void lt_internal_stats_start(lt_ctx* ctx);
int lt_internal_ensure_out(lt_ctx* ctx, size_t floats);
// device -> the caller's host buffer on ctx's stream, synchronous (staged through pinned memory when pageable)
int lt_internal_download(lt_ctx* ctx, float* host_out, const float* dSrc, size_t bytes);
// one device's share of a render call (L checked, camera and row window included): lt_render_device, asynchronous
int lt_internal_render(lt_ctx* ctx, lt_scene* scene, const LtLaunch& L, float* device_out);
// lt_render_views on one device (L checked; its camera is not used): view k (camera cams[k]) into the context's view
// buffer, from zero, and then (host_out != NULL) to host_out + (hostFirst + k * hostStride) * W * H * depth
int lt_internal_render_views(lt_ctx* ctx, lt_scene* scene, LtLaunch L, const RefCamera* cams, int count,
                             float* host_out, int hostFirst, int hostStride);
int lt_multi_render_views(lt_ctx* ctx, lt_scene* scene, const RefCamera* cams, int count, const lt_render_params* params,
                          float* host_out);
// lt_render_adaptive's host form on one device (arguments checked; L.cam is the camera): the rows of part `part` of a
// `parts`-way row partition, from zero in the context's buffers, copied to their places in host_out / host_frames
int lt_internal_render_adaptive(lt_ctx* ctx, lt_scene* scene, const LtLaunch& L, const LtAdaptive& A, float* host_out,
                                uint32_t* host_frames, int parts, int part, lt_adaptive_result* res);
int lt_multi_render_adaptive(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                             const lt_adaptive_params* aparams, float* host_out, uint32_t* host_frames,
                             lt_adaptive_result* out_result);
// Row blocks k, k + G, ... of a row partition (`rows` rows) from device memory, srcPitch bytes per block apart from src,
// to their places in the host image dst (rowBytes per image row); asynchronous on `stream`
cudaError_t lt_copy_row_blocks(void* dst, const void* src, size_t srcPitch, size_t rowBytes, int rows, int G, int k,
                               cudaStream_t stream);
// params->frames frames of a plug-in into ctx->dOut, combined by params->accum_mode (arguments already checked); `who`
// names the entry point in error messages
int lt_internal_render_plugin(lt_ctx* ctx, lt_scene* scene, const RefCamera& cam, const lt_render_params& P,
                              const LtPluginRun& run, bool sync, const char* who);

// device-side BVH construction in the reference's flattened layout (lt_bvh.cu)
enum LtBvhBuilder { LT_BVH_LBVH, LT_BVH_PLOC };
size_t lt_bvh_scratch_bytes(int n, LtBvhBuilder builder);
int lt_launch_bvh_build(LtBvhBuilder builder, const RefPrim* dPrims, int n, const RefMaterial* dMats, int matCount,
                        RefNode* dNodes, RefPrim* dOrderedPrims, RefLights* dLights, void* scratch, size_t scratchBytes,
                        int* outMaxDepth, cudaStream_t stream);
// refit of a tree in the reference layout (lt_scene_refit): dParent receives every node's parent (-1 for the root);
// the refit then fits every node's box to dPrims bottom-up, with one arrival flag per node in dFlags
int lt_launch_refit_parents(const RefNode* dNodes, int n, int* dParent, cudaStream_t stream);
int lt_launch_refit(RefNode* dNodes, int n, const RefPrim* dPrims, const int* dParent, int* dFlags,
                    cudaStream_t stream);
// *dBad = 0, then |= 1 for a materialIndex outside [0, matCount) and |= 2 for a non-finite vertex coordinate
int lt_launch_check_prims(const RefPrim* dPrims, int n, int matCount, int* dBad, cudaStream_t stream);
