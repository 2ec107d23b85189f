// lt_plan.cpp -- from what a render call asks for to what runs (no CUDA call, no allocation): the checks of
// lt_render_params, and the launch plan, which kernels a call runs, on which tree, at which sizes.  lt_debug_plan shows
// the plan on a machine without a GPU.
#include "lens_trace_b200.h"
#include "lt_internal.h"

#include <float.h>
#include <limits.h>
#include <stddef.h>
#include <string.h>

#include <string>

static_assert(LT_DEV_KERNEL_BASIC_CU == LT_KERNEL_BASIC_CU && LT_DEV_KERNEL_BASIC_CL == LT_KERNEL_BASIC_CL &&
                  LT_DEV_KERNEL_CUSTOM_BARY == LT_KERNEL_CUSTOM_BARY && LT_DEV_KERNEL_LIGHTING25 == LT_KERNEL_LIGHTING25 &&
                  LT_DEV_KERNEL_ACCUMULATOR == LT_KERNEL_ACCUMULATOR && LT_DEV_KERNEL_GI25 == LT_KERNEL_GI25 &&
                  LT_DEV_KERNEL_GI == LT_KERNEL_GI,
              "lt_device_types.h: kernel ids differ from enum lt_kernel");
static_assert(LT_DEV_FLAG_STATS == LT_FLAG_STATS && LT_DEV_FLAG_CULL == LT_FLAG_CULL &&
                  LT_DEV_FLAG_STATS_TRACED == LT_FLAG_STATS_TRACED,
              "lt_device_types.h: flags differ from enum lt_flags");

// Threaded copies lt_scene_upload makes of a tree of nNodes nodes: built on the host up to threadedMaxNodes (8 x 32 B
// x N for the full copies, at most as much again for the pruned ones, must stay cache resident); for larger trees the
// full copies built on the device, unless they would not fit the budget (4 GB and an eighth of the device) or 31-bit
// record indices.
LtTree lt_plan_threaded_copies(int nNodes, size_t totalMem, const LtLimits& lim) {
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

LtPlan lt_plan_primary_hits(int flags, int width, int height, const LtSceneFacts& s) {
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

// A masked call's list of scattered pixels (lt_render_masked_device with a partial mask) gives the megakernel no
// coherent camera rays, and its blocks wait for their longest thread over all frames.  Measured (tools/masked_timing.py,
// profiles/masked_timing_b200.txt; NVIDIA B200 at its 1000 W power limit): GI, 4 bounces, Cornell box, random masks of
// a 1080p image, ms of the megakernel against the wavefront: N = 2^12 .. 2^20 pixels at 1 frame 0.155 / 0.456 ..
// 0.869 / 0.760, at 4 frames 0.430 / 0.597 (2^12), 0.480 / 0.652 (2^16), 1.004 / 0.792 (2^18), at 16 frames
// 1.451 / 0.618 (2^12) .. 11.86 / 3.50 (2^20); a quarter of the image, 16 frames, 6.49 / 2.04, on the 1 M-triangle
// mesh 43.1 / 12.6.  So GI lists take the wavefront from 2^20 paths, and from 2^16 paths at 16 or more frames.
static const long long kMaskedMinPaths = 1ll << 20, kMaskedManyFramesMinPaths = 1ll << 16;
static const int kMaskedManyFrames = 16;

// views: a call of several views (lt_render_views) runs its (view, frame) pairs through one wavefront launch, or one
// megakernel launch per view
// listed >= 0: a masked call (lt_render_masked_device) renders that many listed pixels; every size below counts them
// where an unmasked call counts the image's pixels (the wavefront's threshold, frames per batch, the 2^25 paths per
// frame, its workspace and records, the grids), so a full mask plans as the unmasked call.  A partial GI list also
// takes the wavefront at the lower thresholds measured for scattered pixels (kMaskedMinPaths).  The deterministic
// kernels run k_flat over the list: k_flat_stream fetches whole 8x4 tiles (same output either way).
LtPlan lt_plan_render(const LtLaunch& L, const LtSceneFacts& s, size_t totalMem, int smCount, const LtLimits& lim,
                      int views, long long listed) {
  LtPlan p = {};
  p.error = LT_OK;
  p.stats = (L.flags & LT_FLAG_STATS) != 0;
  p.cull = (L.flags & LT_FLAG_CULL) != 0;
  const bool masked = listed >= 0;
  const long long pixels = masked ? listed : (long long)L.width * L.height;
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
    // a partial list (a full one plans as the image): the measured thresholds of scattered pixels above
    if (masked && pixels < (long long)L.width * L.height && L.kernel == LT_KERNEL_GI &&
        (pixels * pairs >= kMaskedMinPaths ||
         (L.frames >= kMaskedManyFrames && pixels * pairs >= kMaskedManyFramesMinPaths)))
      wavefront = true;
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
  if (p.pipeline == LT_PIPE_FLAT && !masked && !(L.flags & (LT_FLAG_STATS | LT_FLAG_CULL | LT_FLAG_NO_STREAM)) &&
      p.tree == LT_TREE_CHILD_PAIR && s.nodeCount >= lim.streamMinNodes)
    p.pipeline = LT_PIPE_FLAT_STREAM;
  if (p.pipeline == LT_PIPE_FLAT_STREAM) {
    const int warpsNeeded = (((L.width + 7) >> 3) * ((L.height + 3) >> 2) + 3) / 4;  // blocks of 4 warps, one tile each
    p.grid = smCount * p.blocksPerSm < warpsNeeded ? smCount * p.blocksPerSm : warpsNeeded;
  } else if (p.pipeline == LT_PIPE_WAVEFRONT) {
    p.grid = smCount * p.blocksPerSm;
  } else if (masked && pixels != (long long)L.width * L.height) {
    p.grid = (int)((pixels + LT_BLOCK - 1) / LT_BLOCK);  // one thread per listed pixel
  } else {
    p.grid = tile_blocks(L.width, L.height);  // (a full list: the blocks of the unmasked launch, the last ones idle)
  }
  return p;
}

int lt_params_normalise(lt_ctx* ctx, const lt_render_params* params, const std::string& w, lt_render_params* P) {
  // API version 1 callers pass the struct without its last field (split_mode)
  if (params->struct_size != sizeof(lt_render_params) && params->struct_size != offsetof(lt_render_params, split_mode))
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "params.struct_size mismatch");
  memset(P, 0, sizeof *P);
  memcpy(P, params, params->struct_size);
  P->struct_size = sizeof *P;
  return LT_OK;
}

int lt_params_to_launch(lt_ctx* ctx, const lt_render_params* params, LtLaunch* L, const char* who) {
  const std::string w = std::string(who) + ": ";
  lt_render_params P;
  if (int rc = lt_params_normalise(ctx, params, w, &P)) return rc;
  const lt_render_params* p = &P;
  if (p->kernel < 0 || p->kernel >= LT_KERNEL_COUNT)
    return lt_internal_fail(ctx, LT_ERR_UNSUPPORTED, w + "unknown kernel id");
  if (p->width <= 0 || p->height <= 0 || p->depth < 3)
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "width/height must be > 0 and depth >= 3");
  if ((long long)p->width * p->height * p->depth > (1ll << 40))
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "image too large");
  if (p->frames < 1) return lt_internal_fail(ctx, LT_ERR_INVALID, w + "frames must be >= 1");
  if (p->accum_mode < 0 || p->accum_mode > 2)
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "bad accum_mode");
  if (p->max_ray_depth < 0 || p->max_ray_depth > 255)
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "max_ray_depth must be in [0, 255]");
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

// A masked call numbers the image's pixels, the listed ones and its list slots with 32-bit ints: images of more than
// INT_MAX pixels are refused (lt_render_device renders them on the megakernels, which index with 64 bits)
int lt_masked_image_check(lt_ctx* ctx, const LtLaunch& L, const char* who) {
  if ((long long)L.width * L.height > (long long)INT_MAX)
    return lt_internal_fail(ctx, LT_ERR_UNSUPPORTED,
                            std::string(who) + ": a masked call handles at most 2^31 - 1 pixels (width * height)");
  return LT_OK;
}

// lt_render_adaptive's own checks, after those of lt_render (L) and before anything is launched; then the image size
int lt_adaptive_check(lt_ctx* ctx, const LtLaunch& L, const lt_adaptive_params* a, const char* who, LtAdaptive* out) {
  const std::string w = std::string(who) + ": ";
  if (!a) return lt_internal_fail(ctx, LT_ERR_INVALID, w + "aparams is NULL");
  if (a->struct_size != sizeof(lt_adaptive_params))
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "aparams.struct_size mismatch");
  // the stopping rule reads the Welford sums, which only a running mean over consecutive frames keeps
  if (L.accumMode != LT_ACCUM_RUNNING_MEAN || L.frameStride > 1)
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "needs accum_mode LT_ACCUM_RUNNING_MEAN and frame_stride <= 1");
  if ((long long)L.cam.frameCount + L.frames < 2)
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "camera.frameCount + frames must be >= 2 (a variance needs two frames)");
  if (!(a->target > 0.0f) || !(a->target <= FLT_MAX))
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "target must be finite and > 0");
  if (!(a->floor >= 0.0f) || !(a->floor <= FLT_MAX))
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "floor must be finite and >= 0");
  if (a->round_frames < 0) return lt_internal_fail(ctx, LT_ERR_INVALID, w + "round_frames must be >= 0");
  if (a->max_frames < L.frames) return lt_internal_fail(ctx, LT_ERR_INVALID, w + "max_frames must be >= frames");
  if ((long long)L.cam.frameCount + a->max_frames > (long long)UINT_MAX)
    return lt_internal_fail(ctx, LT_ERR_INVALID, w + "camera.frameCount + max_frames must fit 32 bits");
  if (int rc = lt_masked_image_check(ctx, L, who)) return rc;
  out->target = a->target;
  out->floor = a->floor == 0.0f ? 1e-4f : a->floor;
  out->roundFrames = a->round_frames ? a->round_frames : L.frames;
  out->maxFrames = a->max_frames;
  return LT_OK;
}

extern "C" int lt_debug_adaptive_rounds(const lt_render_params* params, const lt_adaptive_params* aparams,
                                        uint32_t first_frame_count, int32_t* out_frames, int capacity) {
  const char* who = "lt_render_adaptive";
  if (!params) return lt_internal_fail(nullptr, LT_ERR_INVALID, std::string(who) + ": NULL argument");
  LtLaunch L = {};
  if (int rc = lt_params_to_launch(nullptr, params, &L, who)) return rc;
  L.cam.frameCount = first_frame_count;
  LtAdaptive A;
  if (int rc = lt_adaptive_check(nullptr, L, aparams, who, &A)) return rc;
  int rounds = 0;
  for (int done = 0, f = L.frames; f > 0; done += f, f = lt_adaptive_next_frames(A, done)) {
    if (out_frames) {
      if (rounds >= capacity)
        return lt_internal_fail(nullptr, LT_ERR_INVALID, "lt_debug_adaptive_rounds: capacity is too small");
      out_frames[rounds] = f;
    }
    rounds++;
  }
  return rounds;
}

static int debug_plan(const char* who, const lt_render_params* params, int views, uint64_t node_count,
                      int32_t stack_depth, uint64_t total_mem, int32_t sm_count, int64_t* out, long long listed = -1) {
  if (!params || !out || views < 1 || node_count < 1 || node_count > 0x7fffffffull || sm_count < 1)
    return lt_internal_fail(nullptr, LT_ERR_INVALID, std::string(who) + ": bad arguments");
  LtLaunch L = {};
  if (int rc = lt_params_to_launch(nullptr, params, &L)) return rc;
  if (listed >= 0)
    if (int rc = lt_masked_image_check(nullptr, L, who)) return rc;
  if (listed >= 0 && (listed < 1 || listed > (long long)L.width * L.height))
    return lt_internal_fail(nullptr, LT_ERR_INVALID, std::string(who) + ": pixel_count must be in [1, width * height]");
  const LtLimits lim;
  const LtSceneFacts s = {(int)node_count, stack_depth, lt_plan_threaded_copies((int)node_count, total_mem, lim)};
  const LtPlan p = lt_plan_render(L, s, total_mem, sm_count, lim, views, listed);
  const int64_t v[LT_PLAN_FIELDS] = {p.pipeline, p.tree, p.stats, p.cull, p.batchFrames, p.streams, p.rounds,
                                     p.samplesPerFrame, p.sharedPrimary, p.classify, (int64_t)p.smemStack,
                                     (int64_t)p.smemTrace, p.blocksPerSm, p.grid, (int64_t)p.workspaceBytes};
  memcpy(out, v, sizeof v);
  return p.error != LT_OK ? lt_internal_fail(nullptr, p.error, p.message) : LT_OK;
}

extern "C" int lt_debug_plan(const lt_render_params* params, uint64_t node_count, int32_t stack_depth,
                             uint64_t total_mem, int32_t sm_count, int64_t* out) {
  return debug_plan("lt_debug_plan", params, 1, node_count, stack_depth, total_mem, sm_count, out);
}

extern "C" int lt_debug_plan_views(const lt_render_params* params, int view_count, uint64_t node_count,
                                   int32_t stack_depth, uint64_t total_mem, int32_t sm_count, int64_t* out) {
  return debug_plan("lt_debug_plan_views", params, view_count, node_count, stack_depth, total_mem, sm_count, out);
}

extern "C" int lt_debug_plan_masked(const lt_render_params* params, int64_t pixel_count, uint64_t node_count,
                                    int32_t stack_depth, uint64_t total_mem, int32_t sm_count, int64_t* out) {
  return debug_plan("lt_debug_plan_masked", params, 1, node_count, stack_depth, total_mem, sm_count, out,
                    pixel_count < 1 ? 0 : pixel_count);
}
