/*
 * lens_trace_b200.h -- C-ABI of the B200-native ray-scene hot path (liblt_b200.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++ or torch types.  The host-side
 * C++ classes in include/lens_trace/ (RendererCUDA / RendererOpenCL::render) call only these
 * entry points; a maintainer of the reference would bind the same calls from
 * src/cuda/renderer_cuda.cpp:41-140 (see INTEGRATION.md).
 *
 * Buffers are passed in the reference's own layouts so its AccelerationStructureExplicit, Model
 * and Camera objects can feed this library unchanged:
 *   nodes      LinearBVHNode[]  32 B  (include/lens_trace/acceleration_structure_explicit.h:20-32)
 *   primitives Primitive[]      76 B  (include/lens_trace/acceleration_structure_explicit.h:34-42)
 *   materials  Material[]       32 B  (include/lens_trace/model.h:26-31)
 *   lights     LightContainer  260 B  (include/lens_trace/acceleration_structure_explicit.h:44-47)
 *   camera     7 x 32-bit       28 B  (src/camera.cpp:14-19: pos[3], yaw, pitch, roll, frameCount)
 *
 * Error convention: 0 = ok, negative = error; message through lt_last_error().  There is no CPU
 * fallback: every compute entry point fails with LT_ERR_NO_DEVICE when no CUDA device is usable.
 */
#ifndef LENS_TRACE_B200_H
#define LENS_TRACE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LT_API_VERSION 2

enum lt_status {
  LT_OK = 0,
  LT_ERR_INVALID = -1,    /* bad argument / malformed buffer */
  LT_ERR_NO_DEVICE = -2,  /* no usable CUDA device (no fallback exists) */
  LT_ERR_CUDA = -3,       /* a CUDA call failed; see lt_last_error */
  LT_ERR_UNSUPPORTED = -4 /* unknown kernel file / option */
};

/* One id per kernel source file the reference ships (replaces the run-time compile of
 * RenderProperties*::kernelFilePath, src/cuda/renderer_cuda.cpp:20-39,52-55 and
 * src/opencl/renderer_opencl.cpp:22-54). */
enum lt_kernel {
  LT_KERNEL_BASIC_CU = 0,    /* resources/kernels/cuda/basic.cu */
  LT_KERNEL_BASIC_CL = 1,    /* resources/kernels/opencl/basic.cl */
  LT_KERNEL_CUSTOM_BARY = 2, /* examples/custom_kernel/resources/kernels/custom_opencl.cl */
  LT_KERNEL_LIGHTING25 = 3,  /* resources/kernels/opencl/basic_lighting.cl */
  LT_KERNEL_ACCUMULATOR = 4, /* examples/accumulator/resources/kernels/accumulator.cl */
  LT_KERNEL_GI25 = 5,        /* resources/kernels/opencl/global_illumination.cl */
  LT_KERNEL_GI = 6,          /* examples/global_illumination/resources/kernels/global_illumination.cl */
  LT_KERNEL_COUNT = 7
};

/* How successive frames of one lt_render call are combined. */
enum lt_accum_mode {
  LT_ACCUM_NONE = 0,         /* output = the last frame's sample (reference render() semantics) */
  LT_ACCUM_RUNNING_MEAN = 1, /* examples/accumulator/resources/shaders/accumulator.frag:10-19, FP32 */
  LT_ACCUM_WEIGHTED_SUM = 2  /* acc += weight * sample  (multi-GPU sample split: all-reduce(sum) gives the mean) */
};

enum lt_flags {
  LT_FLAG_STATS = 1 << 0, /* count rays / node tests / triangle tests in the reference's traversal order
                             (no any-hit early-out); results via lt_last_stats. Not for timed runs. */
  LT_FLAG_CULL = 1 << 1,  /* OPT-IN, off by default: closest-hit rays skip subtrees entered beyond the current hit
                             (+1e-4 relative margin).  Does less work than the reference's traversal; output is
                             identical on every tested scene but that is validated, not guaranteed (DESIGN.md). */
  LT_FLAG_MEGAKERNEL = 1 << 2, /* stochastic kernels: force the one-thread-per-pixel persistent kernel */
  LT_FLAG_WAVEFRONT = 1 << 3,  /* stochastic kernels: force the wavefront pipeline (default: chosen by size;
                                  both produce bit-identical output) */
  LT_FLAG_SERIAL = 1 << 5,     /* wavefront pipeline: one stream, one kernel at a time (default: consecutive batches
                                  overlap on two streams; identical output).  For timing kernels in isolation. */
  LT_FLAG_STATS_TRACED = 1 << 7, /* with LT_FLAG_STATS: count what the exact pipelines really trace -- an extension ray
                                    that hits a light is traced once, not once per remaining depth as the reference
                                    does (global_illumination.cl:314-331; the picture is the same) */
  LT_FLAG_NO_STREAM = 1 << 6,  /* deterministic kernels on large scenes: one thread per pixel (k_flat) instead of the
                                  persistent warps that fetch pixel tiles (identical output; kept for comparison) */
  LT_FLAG_NO_THREADED = 1 << 4 /* small scenes: traverse with the stack kernels instead of the stackless threaded
                                  tree (default for scenes whose 8 octant copies stay cache resident; identical
                                  output, kept selectable so tests can compare the two) */
};

/* How a multi-GPU context (lt_ctx_create_multi) divides one lt_render call among its devices. */
enum lt_split_mode {
  LT_SPLIT_AUTO = 0,    /* samples when the call accumulates two or more frames, tiles otherwise */
  LT_SPLIT_SAMPLES = 1, /* device g renders frames g, g+G, ...; the per-device accumulators are combined by one
                           all-reduce (NCCL over NVLink) per call */
  LT_SPLIT_TILES = 2    /* device g renders every G-th block of 8 image rows; no collective, every device copies
                           its rows to the host buffer */
};

typedef struct lt_ctx lt_ctx;
typedef struct lt_scene lt_scene;

typedef struct lt_render_params {
  uint32_t struct_size;   /* = sizeof(lt_render_params) */
  int32_t kernel;         /* enum lt_kernel */
  int32_t kernel_mode;    /* 0 = linearKernel, 1 = tileKernel (KernelMode, include/lens_trace/structures.h:20-23) */
  int32_t width;          /* imageDimensions[0] */
  int32_t height;         /* imageDimensions[1] */
  int32_t depth;          /* imageDimensions[2]; floats per pixel, 3 are written (basic.cu:344,361-363) */
  int32_t max_ray_depth;  /* GI bounce cap; 0 = the reference constant 16 (global_illumination.cl:308) */
  int32_t frames;         /* >= 1: frames rendered by this call; frame k uses frameCount = camera.frameCount + k*frame_stride */
  uint32_t frame_stride;  /* 0 is treated as 1 */
  int32_t accum_mode;     /* enum lt_accum_mode */
  float accum_weight;     /* LT_ACCUM_WEIGHTED_SUM only */
  int32_t flags;          /* enum lt_flags */
  int32_t block_x;        /* thread-block shape hint (ThreadOrganizationCUDA.blockSize); 0 = library default. */
  int32_t block_y;        /* Output never depends on it (tests/cuda_renderer_test.cc:51-115). */
  int32_t split_mode;     /* API version 2, multi-GPU contexts only: one of enum lt_split_mode; a struct_size without this
                             field is accepted and means LT_SPLIT_AUTO */
} lt_render_params;

/* Statistics of the context's last call (lt_last_stats).  Every field describes that call and reads 0 for what it did
 * not measure: the counters (rays, node_tests, tri_tests) on a call without LT_FLAG_STATS, and kernel_ms and the
 * per-kernel times on an asynchronous call (sync = 0 without LT_FLAG_STATS), which returns before its work is done.
 * upload_ms instead describes the last lt_scene_upload or lt_scene_refit, and sm_count the device. */
typedef struct lt_stats {
  uint64_t rays;        /* traversal calls (primary + shadow + extension + lens segments) */
  uint64_t node_tests;  /* boxes tested, reference traversal order */
  uint64_t tri_tests;   /* triangle tests executed, reference traversal order */
  float kernel_ms;      /* device time of the render kernels of the last lt_render* call (CUDA events) */
  float upload_ms;      /* device time of the last lt_scene_upload (H2D + re-flatten) or lt_scene_refit */
  int32_t kernel_launches; /* kernels launched by the last lt_render* call */
  int32_t sm_count;
  float trace_ms;       /* part of kernel_ms spent in the traversal kernels (k_wf_primary + k_wf_trace, or the
                           whole megakernel), CUDA events around each launch; 0 when the call was not synchronous */
  int32_t trace_launches;
  /* API version 2: per-kernel times of a wavefront step whose kernels ran one at a time (LT_FLAG_SERIAL or
     LT_FLAG_STATS, synchronous call), CUDA events around each launch; 0 otherwise */
  float shade_ms;          /* k_wf_shade launches */
  float primary_shade_ms;  /* k_wf_primary launches that shade shared camera-ray hits (no traversal) */
  float accumulate_ms;     /* k_wf_accumulate launches */
  int32_t shade_launches;
} lt_stats;

/* --- context: replaces RendererCUDA::RendererCUDA() (src/cuda/renderer_cuda.cpp:10-14). --- */
int lt_ctx_create(int device_ordinal, lt_ctx** out_ctx);
/* Multi-GPU context on the given devices of this process (SURVEY.md 8(b), 8(e); the reference renders on device 0
 * only, src/cuda/renderer_cuda.cpp:12).  lt_scene_upload replicates the scene on every device, lt_render divides the
 * call by params->split_mode and returns the combined frame in host_out.  device_count == 1 behaves like
 * lt_ctx_create.  The sample split needs NCCL (libnccl.so.2, loaded on first use). */
int lt_ctx_create_multi(const int* device_ordinals, int device_count, lt_ctx** out_ctx);
int lt_ctx_device_count(const lt_ctx* ctx);
void lt_ctx_destroy(lt_ctx* ctx);
/* Last error message of ctx (or of the failed lt_ctx_create when ctx == NULL). Never NULL. */
const char* lt_last_error(const lt_ctx* ctx);
/* Render on this CUDA stream (cudaStream_t as void*); NULL = the context's own stream. */
int lt_ctx_set_stream(lt_ctx* ctx, void* cuda_stream);

/* --- scene: replaces the per-call cuMemAlloc + cuMemcpyHtoD of nodes, primitives, materials and
 * the light container (src/cuda/renderer_cuda.cpp:90-104).  Uploads once and re-flattens on the
 * device into the 64-byte child-pair node / 48-byte triangle layout (DESIGN.md). --- */
int lt_scene_upload(lt_ctx* ctx, const void* nodes, uint64_t node_bytes, const void* primitives,
                    uint64_t primitive_bytes, const void* materials, uint64_t material_bytes,
                    const void* light_container, uint64_t light_bytes, lt_scene** out_scene);
void lt_scene_release(lt_ctx* ctx, lt_scene* scene);

/* --- optional device-side builder (replaces AccelerationStructureExplicit's host build,
 * src/acceleration_structure_explicit.cpp:3-41,47-137, for large scenes): an LBVH over `primitives` (Primitive[]
 * in any order, e.g. Model's face order) built on the GPU and emitted in the reference's flattened layout, then
 * uploaded like lt_scene_upload.  The tree differs from the median-split tree (same results except the winner of
 * exact ties); lt_scene_download returns the node / ordered-primitive / light buffers it produced (host
 * pointers, sizes in bytes: 32*(2n-1), 76*n, 260) so the CPU side can hold them. --- */
int lt_scene_build_lbvh(lt_ctx* ctx, const void* primitives, uint64_t primitive_bytes, const void* materials,
                        uint64_t material_bytes, lt_scene** out_scene);
/* The same contract with a PLOC tree (bottom-up clustering of mutual nearest neighbours over the Morton order,
 * Meister & Bittner 2018): about the surface-area cost of the host SAH builder's tree at about the LBVH's build
 * time (DESIGN.md section 4).  Deterministic.  Non-finite vertex coordinates -> LT_ERR_INVALID. */
int lt_scene_build_ploc(lt_ctx* ctx, const void* primitives, uint64_t primitive_bytes, const void* materials,
                        uint64_t material_bytes, lt_scene** out_scene);
int lt_scene_download(lt_ctx* ctx, lt_scene* scene, void* nodes, uint64_t node_bytes, void* primitives,
                      uint64_t primitive_bytes, void* light_container);
/* Replace the primitives of an uploaded scene and refit its tree on the device: moving geometry without a new upload.
 * primitives: the scene's primitive count of 76-byte Primitive records, in the order of the scene's primitive buffer
 * (the caller's order for an uploaded scene, the order lt_scene_download returns for a built one).  Materials, the
 * light container and the topology (child offsets, primitiveCount, axis, the DFS order) stay as they are.
 * Afterwards every node box is the exact union of its content: a leaf's box covers all primitiveCount triangles from
 * primitivesOffset, an inner node's box is the union of its two children, with std::min / std::max keeping the first
 * operand on ties (a triangle's vertices a, b, c in that order, a leaf's primitives in order, the first child before
 * the second).  The result is deterministic, and every render entry point on the scene then gives byte for byte what
 * it gives on a scene uploaded with lt_scene_upload from the refitted nodes (lt_scene_download), the new primitives
 * and the scene's materials and lights.
 * Rejected with LT_ERR_INVALID, the scene untouched: primitive_bytes other than the primitive count x 76, a
 * materialIndex out of range, a non-finite vertex coordinate; and a scene with a leaf whose primitiveCount primitives
 * from primitivesOffset run past its primitive buffer (lt_scene_upload checks only a leaf's first primitive, which
 * is all the reference's leaves test).  Synchronous: ordered after earlier work on the
 * context's stream, returns when the scene is ready; lt_stats.upload_ms reports the refit's device time.  On a
 * multi-GPU context every device's copy is refitted.  After LT_ERR_CUDA the scene is unusable: release it.
 * A refit keeps the topology: after large deformations a new build (lt_scene_build_ploc) gives a better tree. */
int lt_scene_refit(lt_ctx* ctx, lt_scene* scene, const void* primitives, uint64_t primitive_bytes);
/* The same with the primitives in device memory of the context's device (e.g. a torch tensor's data_ptr), checked by
 * a kernel before anything is overwritten; memory of another device, host memory or a pointer that is not 4-byte
 * aligned -> LT_ERR_INVALID.  Single-GPU contexts only (LT_ERR_UNSUPPORTED otherwise). */
int lt_scene_refit_device(lt_ctx* ctx, lt_scene* scene, const void* device_primitives, uint64_t primitive_bytes);
/* node and primitive counts of a scene */
int lt_scene_info(const lt_scene* scene, uint64_t* node_count, uint64_t* primitive_count, int32_t* stack_depth);

/* --- render: replaces cuLaunchKernel + cuCtxSynchronize + cuMemcpyDtoH
 * (src/cuda/renderer_cuda.cpp:113-139).  Synchronous.  host_out (may be NULL) receives
 * width*height*depth floats: the sample (LT_ACCUM_NONE) or the accumulator. --- */
int lt_render(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
              float* host_out);
/* Same, but the result stays in device memory (device_out: width*height*depth floats on ctx's
 * device, e.g. a torch tensor's data_ptr; used as the accumulator when accum_mode != NONE).
 * Asynchronous on the context stream unless sync != 0. */
int lt_render_device(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                     float* device_out, int sync);

/* Several camera views of one scene with the same params in one call.  cameras28: view_count >= 1 consecutive
 * 28-byte camera records.  View v equals lt_accum_reset followed by lt_render with camera v, bit for bit, in every
 * accum_mode: frame k of view v uses frameCount_v + k * frame_stride, and every view accumulates from zero within the
 * call.  The context accumulator of lt_render / lt_accum_read / lt_accum_reset is neither read nor changed, with one
 * exception: on a multi-GPU context view_count == 1 is lt_render (see below).  The views are rendered into a device
 * buffer the context owns (view_count images); like the wavefront workspace it keeps the largest size asked for until
 * lt_ctx_destroy.
 * host_out: view_count * width * height * depth floats, view v at v * width * height * depth (may be NULL).
 * Every kernel id and flag of lt_render is accepted and means the same; with LT_FLAG_STATS, lt_last_stats counts the
 * sum over the views.  The views of one call share one wavefront launch when they hold enough paths, otherwise each
 * runs the megakernel (lt_debug_plan_views).  view_count < 1 or NULL cameras28: LT_ERR_INVALID, nothing launched.
 * On a multi-GPU context with view_count >= 2, device g renders views g, g+G, ... on its own (no collective);
 * split_mode must be LT_SPLIT_AUTO (LT_ERR_INVALID otherwise).  There view_count == 1 is lt_render, with its split
 * and its per-device accumulators.  Synchronous. */
int lt_render_views(lt_ctx* ctx, lt_scene* scene, const void* cameras28, int view_count,
                    const lt_render_params* params, float* host_out);
/* Same, into device memory: device_out holds view_count images on ctx's device and is used as their view_count
 * accumulators when accum_mode != NONE: slice v equals lt_render_device(camera v, params, slice v) from the same
 * initial contents.  Asynchronous on the context stream unless sync != 0.  Single-GPU contexts only
 * (LT_ERR_UNSUPPORTED otherwise, as lt_render_device). */
int lt_render_views_device(lt_ctx* ctx, lt_scene* scene, const void* cameras28, int view_count,
                           const lt_render_params* params, float* device_out, int sync);

/* lt_render_device for the pixels of a mask only: spend samples where the image is still noisy.
 * device_mask: width * height bytes on ctx's device, row-major; a nonzero byte renders its pixel.  NULL: every pixel.
 * Every masked pixel gets exactly what lt_render_device gives it: frames camera.frameCount + k * frame_stride for
 * k < frames, combined by accum_mode into device_out from its current contents, bit for bit.  Pixels outside the mask
 * are not written: their bytes in device_out and device_m2 stay as they were.  Every kernel id, accum_mode and flag of
 * lt_render is accepted and means the same; with LT_FLAG_STATS the counters count the masked pixels' rays.
 * A pixel's frame count is the caller's bookkeeping: camera.frameCount must be the number of frames the running mean
 * of every masked pixel already holds.
 * device_m2 (may be NULL): 3 floats per pixel (width * height * 3, whatever depth is) on ctx's device, the per-channel
 * sum of squared deviations of the frame samples the running mean averages (Welford).  For a frame with frameCount n
 * and sample x, in FP32 with one rounding per operation: n == 0 sets m2 = 0; n > 0 computes d = x - mean_prev, the
 * running mean as always, then m2 = m2 + d * (x - mean).  The sample variance of a pixel of n frames is m2 / (n - 1).
 * Only with LT_ACCUM_RUNNING_MEAN and frame_stride <= 1 (LT_ERR_INVALID otherwise).
 * Checked before anything is launched: the parameters as lt_render; device_mask and device_m2 must be memory of ctx's
 * device (LT_ERR_INVALID otherwise, device_m2 4-byte aligned); a multi-GPU context returns LT_ERR_UNSUPPORTED, and so
 * does an image of more than 2^31 - 1 pixels (width * height): the pixel list holds 32-bit pixel indices.
 * A kernel compacts the mask into a list of pixels in the context's memory (grow-only, like the wavefront workspace),
 * and the launch plan is made for the listed pixels (lt_debug_plan_masked).  So with a mask the call reads the list's
 * length back -- one 4-byte copy and a synchronisation of the context stream, the call's only one; otherwise it is
 * asynchronous on the context stream unless sync != 0.  An empty mask launches nothing more and returns LT_OK.
 * lt_last_stats describes the call as for lt_render_device; kernel_launches counts the compaction.
 * Not provided: a host-memory form or the context accumulator, multi-GPU contexts, views, plug-ins, the C++ renderer
 * (RenderExtensionB200), and any policy that chooses the mask: the caller decides which pixels need more frames.
 * lt_render_adaptive (below) is one such policy inside the library, with a host form, multi-GPU contexts and the C++
 * renderer. */
int lt_render_masked_device(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                            const uint8_t* device_mask, float* device_out, float* device_m2, int sync);
/* Test hook (single-GPU contexts): reversed != 0 makes later lt_render_masked_device calls on ctx render their pixel
 * list, and lt_render_adaptive calls every list they render, in reverse order (one more kernel per list), 0 restores the
 * compaction's order.  The output is the same either way; tests
 * compare the two. */
int lt_debug_ctx_list_order(lt_ctx* ctx, int reversed);

/* Adaptive sampling inside the library: render to a noise target.  The stopping rule is the relative standard error of
 * each pixel's running mean (INTEGRATION.md section 5e); lt_render_masked_device stays the way to use a rule of one's
 * own. */
typedef struct lt_adaptive_params {
  uint32_t struct_size;  /* = sizeof(lt_adaptive_params) */
  float target;          /* a pixel stops once its relative standard error is <= target; finite, > 0 */
  float floor;           /* the error is relative to max(mean, floor); 0 -> 1e-4; finite, >= 0 */
  int32_t round_frames;  /* frames per round after the first; 0 -> params->frames; >= 0 */
  int32_t max_frames;    /* most frames one pixel gets in this call; >= params->frames */
} lt_adaptive_params;

typedef struct lt_adaptive_result {
  int32_t rounds;              /* rounds rendered, the first included (the maximum over devices) */
  uint64_t pixel_frames;       /* sum over pixels of the frames this call rendered */
  uint64_t pixels_unconverged; /* pixels that reached max_frames still above target */
} lt_adaptive_result;

/* Render every pixel, then keep rendering only the pixels whose relative standard error is above a target.
 * Round schedule: round 1 renders every pixel for F1 = params->frames frames; round r + 1 renders
 * min(round_frames, max_frames - (F1 + ... + Fr)) frames for the pixels that go on; the call stops when a round's list is
 * empty or max_frames is reached.  Every pixel of a round has the same frames behind it, camera.frameCount + F1 + ... +
 * Fr, so each round is a masked continuation (lt_render_masked_device) with m2.
 * Stopping rule, after a round, in FP32 with one IEEE round-to-nearest per operation: n = camera.frameCount + F1 + ... +
 * Fr, d = (float)n * (float)(n - 1), and per channel k < 3 e_k = sqrt(m2_k / d) / (mean_k < floor ? floor : mean_k).
 * A pixel goes on to the next round if it was in this round, no e_k is NaN and some e_k > target (what torch's sqrt, /,
 * clamp_min and amax(...) > target compute, NaN included).
 * Result: every pixel p with frame count n_p holds bit for bit the mean lt_render_device gives with frames = n_p -
 * camera.frameCount from the same starting contents, and the m2 lt_render_masked_device keeps; it depends neither on
 * the order of the pixel lists nor on the device count.
 * Checked before anything is launched (LT_ERR_INVALID): the parameters as lt_render; accum_mode other than
 * LT_ACCUM_RUNNING_MEAN; frame_stride > 1; camera.frameCount + frames < 2; target not finite or <= 0, floor not finite
 * or < 0, round_frames < 0, max_frames < frames.  An image of more than 2^31 - 1 pixels is LT_ERR_UNSUPPORTED.  Every
 * kernel id is accepted; the deterministic ones have m2 = 0 and stop after round 1.  With LT_FLAG_STATS (single-GPU)
 * the counters and kernel_launches are summed over the rounds; kernel_launches counts the list and selection kernels
 * too, kernel_ms sums the rounds' render kernels.
 * After each round a selection kernel writes the pixels that go on into the next list, and the call reads the list's
 * length back (one 4-byte copy and a synchronisation of the context stream per round, no others).
 * Host form: accumulates from zero (as lt_accum_reset + lt_render, per pixel) in buffers the context owns (grow-only:
 * mean, m2, frame counts); neither reads nor changes the context accumulator.  host_out receives width * height * depth
 * floats of means, host_frames (may be NULL) width * height frame counts n_p.  Synchronous.  On a multi-GPU context
 * device g owns every G-th block of 8 image rows (as LT_SPLIT_TILES) and runs the whole loop on its rows on its own (no
 * collective); split_mode must be LT_SPLIT_AUTO or LT_SPLIT_TILES (LT_ERR_INVALID otherwise), LT_FLAG_STATS is
 * LT_ERR_UNSUPPORTED there as for lt_render.  out_result (may be NULL) receives the result. */
int lt_render_adaptive(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                       const lt_adaptive_params* aparams, float* host_out, uint32_t* host_frames,
                       lt_adaptive_result* out_result);
/* The same in device memory of ctx's device (single-GPU contexts only, LT_ERR_UNSUPPORTED otherwise): device_out (width
 * * height * depth floats) and device_m2 (required, width * height * 3 floats, 4-byte aligned) are the running mean and
 * its Welford sums, continued from their contents: with camera.frameCount = c > 0 they must hold c frames for every
 * pixel.  device_frames (may be NULL, 4-byte aligned) receives n_p for every pixel.  Memory of another device or of the
 * host: LT_ERR_INVALID.  The count of the round that reaches max_frames is read back only when out_result is given;
 * work after the last readback is asynchronous on the context stream unless sync != 0. */
int lt_render_adaptive_device(lt_ctx* ctx, lt_scene* scene, const void* camera28, const lt_render_params* params,
                              const lt_adaptive_params* aparams, float* device_out, float* device_m2,
                              uint32_t* device_frames, lt_adaptive_result* out_result, int sync);
/* Host-only (no device needed): the argument checks of lt_render_adaptive with the same codes and messages, then the
 * frames of each round the call would render if every pixel kept going (F1, F2, ...), camera.frameCount being
 * first_frame_count.  Returns the number of rounds (out_frames may be NULL to ask for it; LT_ERR_INVALID when capacity
 * is too small), negative on error. */
int lt_debug_adaptive_rounds(const lt_render_params* params, const lt_adaptive_params* aparams,
                             uint32_t first_frame_count, int32_t* out_frames, int capacity);
/* Test hook (single-GPU contexts): later adaptive calls on ctx render only the rows device `part` of a `parts`-device
 * context would own (every parts-th block of 8 rows from block `part`) and leave the other pixels untouched, so that the
 * multi-GPU partition can be tested on one GPU.  parts = 1, part = 0 restores the whole image. */
int lt_debug_ctx_adaptive_part(lt_ctx* ctx, int parts, int part);

/* The output buffer of the reference API is the caller's malloc'ed memory (pOutputBuffer, structures.h:62,76).
 * lt_render copies into such pageable memory through its own pinned staging buffer; an application that reuses one
 * buffer for many calls can page-lock it once instead, and the frame then arrives by a single DMA.  Unregister
 * before freeing the buffer. */
int lt_host_register(void* host_buffer, uint64_t bytes);
int lt_host_unregister(void* host_buffer);

/* The context-owned accumulator used by lt_render (reset = next running-mean frame restarts). */
int lt_accum_reset(lt_ctx* ctx);
int lt_accum_read(lt_ctx* ctx, float* host_out, uint64_t float_count);

/* Hit record of the primary ray of every pixel (the payload of basic.cu:57-63 after intersect()):
 * ids = primitiveIndex, hit = hitType, tuv = t,u,v.  Any pointer may be NULL.  Host pointers. */
int lt_primary_hits(lt_ctx* ctx, lt_scene* scene, const void* camera28, int kernel, int width, int height,
                    int32_t* ids, int32_t* hit, float* tuv);

/* same, taking flags of enum lt_flags [LT_FLAG_CULL], to validate the opt-in culled traversal against the exact one */
int lt_primary_hits_flags(lt_ctx* ctx, lt_scene* scene, const void* camera28, int kernel, int flags, int width,
                          int height, int32_t* ids, int32_t* hit, float* tuv);

int lt_last_stats(const lt_ctx* ctx, lt_stats* out_stats);

/* Parity hooks (host pointers): the device's evaluation of random() (basic_lighting.cl:64-67) and of
 * alignHemisphereWithCoordinateSystem(uniformSampleHemisphere(u1,u2), up) (global_illumination.cl:69-82;
 * up3 = 3 floats per sample, out4 = 4 floats per sample), for tests that pin them against the oracle. */
int lt_debug_random(lt_ctx* ctx, const float* fx, const float* fy, const float* seed, int n, float* out);
int lt_debug_hemisphere(lt_ctx* ctx, const float* u1, const float* u2, const float* up3, int n, float* out4);

/* Measurement hook (no reference counterpart; SURVEY.md 8(d) asks for a measured ceiling of the node fetches): the
 * rate at which the device sustains per-lane 32-byte gathers (one ld.global.nc.v8.f32 per lane, the access a
 * traversal step makes) at pseudo-random records of a table of table_bytes.  dependent != 0: every lane chases
 * the index it just loaded (what one ray does); ilp = independent gathers per lane and iteration (1, 2 or 4);
 * persistent grid of blocks_per_sm x SMs blocks of 128 threads.  out_gbs = 32 B x gathers / best-of-3 time. */
int lt_debug_gather_peak(lt_ctx* ctx, uint64_t table_bytes, int dependent, int ilp, int blocks_per_sm, int iters,
                         double* out_gbs, double* out_ns_per_load);

/* Host-only (no device needed): the image rows device `device` of `devices` renders in a tile split (LT_SPLIT_TILES),
 * in the order of its local rows; returns their number (out_rows may be NULL to ask for it), negative on bad
 * arguments.  For tests of the partition on a machine without a GPU. */
int lt_debug_tile_rows(int height, int devices, int device, int32_t* out_rows, int capacity);
/* Test hook: a multi-GPU context of `members` (2..16) members that all render on device device_ordinal -- the group
 * lt_ctx_create_multi builds, each member an ordinary single-GPU context with its own stream, buffers, scene copy and
 * host thread -- so that the splits, the exchange kernel and the row copies run on a machine with one GPU.  Its sample
 * split always combines the members' accumulators with the library's own exchange kernel (no NCCL, no peer mapping).
 * Anything else than 2..16 members: LT_ERR_INVALID. */
int lt_debug_ctx_create_shared(int device_ordinal, int members, lt_ctx** out_ctx);

/* Host-only (no device needed): the threaded form of a reference node array that lt_scene_upload builds for
 * small trees -- 8 copies of node_count 32-byte records {lo.x lo.y lo.z hi.x | hi.y hi.z link skip}, copy o in
 * the order the reference's traversal (basic.cu:156-196) visits the nodes for rays whose direction signs are
 * the bits of o (LtThreadNode, include/lens_trace_b200_device.cuh).  out_records: 8 * node_count * 32 bytes.
 * Exposed so that the layout can be checked against the reference traversal on a machine without a GPU. */
int lt_debug_build_threaded(const void* nodes, uint64_t node_bytes, void* out_records);

/* Host-only: the eight pruned copies of the reference tree (same record format, inner nodes that cannot change which
 * leaves a ray reaches left out; skip links index out_records), which lt_scene_upload builds beside those when it
 * builds no traversal tree.  *out_stride receives the records per copy; out_records (8 * stride * 32 bytes, at most
 * 8 * node_count * 32) may be NULL to ask for it. */
int lt_debug_build_threaded_pruned(const void* nodes, uint64_t node_bytes, void* out_records, int32_t* out_stride);

/* Host-only: every threaded record lt_scene_upload builds for a small tree whose leaves link primitives below
 * prim_count.  out_records (16 * node_count * 32 bytes of room): the eight full copies, then the eight pruned copies
 * (*out_stride records each; skip links absolute, from record 8 * node_count).  When every leaf box lies inside all
 * its ancestors' boxes (bounds finite, lo <= hi, no primitive linked twice, inner root), the pruned copies are those
 * of a traversal tree: a tree over the reference's leaves, built for the cost of the pruned walk
 * (lt_debug_traversal_tree_costs), that reaches the same leaves in another order.  Then
 * *out_traversal = 1 and out_rank (8 * prim_count int32) receives the tie-break table rank[o][p] (LtSceneDev::rank);
 * otherwise *out_traversal = 0, the pruned copies are lt_debug_build_threaded_pruned's and out_rank is not written. */
int lt_debug_build_traversal_tree(const void* nodes, uint64_t node_bytes, int32_t prim_count, void* out_records,
                                  int32_t* out_stride, int32_t* out_rank, int32_t* out_traversal);

/* Host-only: the traversal tree lt_scene_upload builds for a small tree (see lt_debug_build_traversal_tree), in the
 * reference's node layout, and the cost model it is chosen by: the expected box tests of the pruned threaded walk per
 * ray that hits the root box, sum over the kept records r other than the root of SA(nearest kept ancestor of r) /
 * SA(root).  out_costs[0]: the reference tree's pruned copies; [1], [2], [3]: the candidates over the reference's
 * leaves -- SAH sweep, PLOC, the better of the two after treelet restructuring --, of which the cheapest is the
 * traversal tree, written to out_nodes (node_bytes of room).  Without a traversal tree [1..3] are NaN and out_nodes is
 * not written. */
int lt_debug_traversal_tree(const void* nodes, uint64_t node_bytes, int32_t prim_count, void* out_nodes,
                            double* out_costs);

/* Test hook: 1 when the pruned threaded copies of an uploaded scene are a traversal tree, 0 when not (also for
 * scenes without host-built copies), < 0 on error. */
int lt_debug_scene_traversal_tree(const lt_scene* scene);
/* Test hook: the bytes of device memory a scene holds (all devices' copies of a multi-GPU scene): the sum of the
 * buffers it holds at the time of the call. */
int lt_debug_scene_bytes(const lt_scene* scene, uint64_t* out_bytes);

/* Test hook: full != 0 makes launches on `scene` (single-GPU) walk the full threaded copies for every ray, 0 restores
 * the pruned ones.  The output is the same either way; tests compare the two. */
int lt_debug_scene_full_threaded(lt_scene* scene, int full);

/* Test hook (single-GPU contexts; LT_ERR_UNSUPPORTED on a multi-GPU one): the context's size limits.  Trees of at
 * most threaded_max_nodes nodes (default 65536) get threaded copies built on the host at upload, larger ones copies
 * built on the device; exact, uncounted launches of the deterministic kernels on scenes of at least stream_min_nodes
 * nodes (default 100000) run the tile-fetching kernel.  The output is the same either way; tests lower the limits so
 * that the small scenes the oracle can check run the large-scene paths. */
int lt_debug_ctx_limits(lt_ctx* ctx, int threaded_max_nodes, int stream_min_nodes);

/* Host-only (no device needed): the launch plan lt_render makes for `params` on a scene of node_count nodes whose
 * traversal stack needs stack_depth levels, uploaded to a device of total_mem bytes with sm_count SMs, under the
 * default limits; the scene has the threaded copies lt_scene_upload would make.  out receives LT_PLAN_FIELDS values:
 *   pipeline (0 k_flat, 1 k_flat_stream, 2 k_path megakernel, 3 wavefront), tree (0 child-pair stack traversal,
 *   1 host-built threaded copies, 2 device-built ones), stats, cull, then for the wavefront frames per batch,
 *   streams, rounds, samples per frame, shared primary hits, pixel classification, then dynamic shared memory of the
 *   stack-traversal kernels and of the trace kernel, blocks per SM of the persistent kernels, grid, and the wavefront
 *   workspace bytes.
 * Returns LT_OK, or the error lt_render would return (its message in lt_last_error(NULL)). */
#define LT_PLAN_FIELDS 15
int lt_debug_plan(const lt_render_params* params, uint64_t node_count, int32_t stack_depth, uint64_t total_mem,
                  int32_t sm_count, int64_t* out);
/* Host-only: the plan of an lt_render_views call of view_count views, as lt_debug_plan (view_count == 1: exactly
 * lt_debug_plan).  The wavefront's frames per batch then count (view, frame) pairs, and its workspace bytes include
 * the primary records of every view one batch touches. */
int lt_debug_plan_views(const lt_render_params* params, int view_count, uint64_t node_count, int32_t stack_depth,
                        uint64_t total_mem, int32_t sm_count, int64_t* out);
/* Host-only: the plan of an lt_render_masked_device call whose mask lists pixel_count pixels (1 .. width * height), as
 * lt_debug_plan.  Every size counts the listed pixels where lt_render counts the image's: the wavefront's threshold,
 * frames per batch, its limit of 2^25 paths per frame, workspace and primary records, and the grids.  The
 * deterministic kernels run k_flat over the list (pipeline 0, never k_flat_stream).  A partial list of the GI kernel
 * (LT_KERNEL_GI, pixel_count < width * height) takes the wavefront from 2^20 paths, and from 2^16 paths at 16 frames
 * or more: the crossovers measured for scattered pixels (DESIGN.md section 4).  Otherwise pixel_count = width *
 * height plans exactly as lt_debug_plan.  An image of more than 2^31 - 1 pixels returns LT_ERR_UNSUPPORTED, as
 * lt_render_masked_device does. */
int lt_debug_plan_masked(const lt_render_params* params, int64_t pixel_count, uint64_t node_count, int32_t stack_depth,
                         uint64_t total_mem, int32_t sm_count, int64_t* out);

/* --- plug-in kernels: a user-written .cu file with the reference's kernel ABI (extern "C" __global__
 * linearKernel / tileKernel(LinearBVHNode*, Primitive*, Material*, LightContainer*, Camera*, float* out,
 * int width, int height, int depth), resources/kernels/cuda/basic.cu:331-340).  Replaces the NVRTC compile
 * and launch of src/cuda/renderer_cuda.cpp:20-39,57-88,113-133 for files that are not one of the shipped
 * kernels: compiled once per context for sm_100a (once for all devices of a multi-GPU context, which loads it on
 * each), then launched on the scene's buffers in the reference layouts with the reference's launch shape
 * (block_x x block_y threads, 32x1 when 0).  lt_render_plugin and lt_render_plugin_cl render one frame on a
 * single-GPU context (LT_ERR_UNSUPPORTED on a multi-GPU one); lt_render_plugin_frames renders many, on either. --- */
int lt_plugin_load(lt_ctx* ctx, const char* kernel_file_path, int* out_plugin_id);
int lt_render_plugin(lt_ctx* ctx, lt_scene* scene, const void* camera28, int plugin_id, int kernel_mode, int width,
                     int height, int depth, int block_x, int block_y, float* host_out);

/* --- OpenCL C plug-ins: lt_plugin_load on a path ending in ".cl" translates the file onto this library's OpenCL C
 * runtime (the subset of INTEGRATION.md: vector types, math / geometric / work-item built-ins; no __local memory,
 * barriers, images, atomics or half) and compiles it with NVRTC for sm_100a, once per context.  Every
 * `__kernel void linearKernel` / `tileKernel` of the file must take the reference's OpenCL arguments
 *   (LinearBVHNode*, Primitive*, Material*, LightContainer*, Camera*, float* output, uint currentBlock, uint W,
 *    uint H, uint depth)
 * under the user's own struct names, or the file does not compile.  `#pragma OPENCL FP_CONTRACT OFF` anywhere in the
 * file compiles all of it without contraction (default: a * b + c may fuse, as OpenCL C allows).  A compile error
 * returns LT_ERR_UNSUPPORTED with the NVRTC log, which names the user's file and line.  A file that says exactly
 * `#include "lens_trace_b200_device_cl.h"` gets the plug-in device API of lens_trace_b200_device.cuh in OpenCL C
 * types (lt_trace, lt_occluded, lt_camera_ray, lt_random, lt_sample_light, lt_sample_hemisphere, lt_interpolate, ...)
 * and is launched with the dynamic shared memory lt_trace needs for its work-group; a work-group whose traversal
 * stacks do not fit a block returns LT_ERR_INVALID before anything is launched.
 * lt_render_plugin_cl launches it like the reference's OpenCL backend (src/opencl/renderer_opencl.cpp:84-146): one
 * launch per work block, (width / work_block_x) * (height / work_block_y) of them (integer division), global size =
 * the work block, local size = group, currentBlock = the block's index.  A work block of 0 is the whole image in that
 * dimension (what THREAD_ORGANIZATION_MODE_MAX_FIT renders); group 0 x 0 is the library's choice, any other group
 * must divide the work block (LT_ERR_INVALID otherwise).  Pixels no block covers are written as 0.  Synchronous;
 * lt_stats.kernel_ms and kernel_launches describe the call.  lt_render_plugin on a .cl plug-in and
 * lt_render_plugin_cl on a .cu plug-in return LT_ERR_INVALID. --- */
int lt_render_plugin_cl(lt_ctx* ctx, lt_scene* scene, const void* camera28, int plugin_id, int kernel_mode, int width,
                        int height, int depth, int work_block_x, int work_block_y, int group_x, int group_y,
                        float* host_out);
/* A plug-in (lt_plugin_load) rendered like lt_render renders a built-in kernel: params->frames frames, frame k with
 * camera frameCount + k * frame_stride, combined by params->accum_mode into the context's accumulator (the one lt_render,
 * lt_accum_reset and lt_accum_read use), divided among the devices of a multi-GPU context by the sample split.
 * work_block_x/y: .cl plug-ins only (as lt_render_plugin_cl; nonzero for a .cu plug-in is LT_ERR_INVALID);
 * params->block_x/y is the CUDA block of a .cu plug-in and the work-group of a .cl plug-in.  params->kernel and
 * max_ray_depth are ignored (a plug-in has its own bounce cap), as are the schedule flags; LT_FLAG_STATS,
 * LT_FLAG_STATS_TRACED and LT_FLAG_CULL return LT_ERR_UNSUPPORTED.  LT_ACCUM_NONE launches every frame into the output
 * in order, like consecutive lt_render_plugin calls; the accumulating modes launch every frame into a sample buffer
 * and fold it into the accumulator with the built-in pipelines' arithmetic (one extra kernel per frame).  A .cl
 * plug-in's uncovered pixels read 0.  On a multi-GPU context: LT_SPLIT_AUTO means samples, LT_SPLIT_TILES and
 * LT_ACCUM_NONE return LT_ERR_UNSUPPORTED, a running mean needs frame_stride 1.  Synchronous; lt_stats.kernel_ms
 * covers the call, kernel_launches counts the plug-in and fold launches, the counters are 0. */
int lt_render_plugin_frames(lt_ctx* ctx, lt_scene* scene, const void* camera28, int plugin_id,
                            const lt_render_params* params, int work_block_x, int work_block_y, float* host_out);
/* Host-only (NVRTC, no device or driver needed): translate and compile a .cl file as lt_plugin_load would.  Returns 0,
 * or LT_ERR_UNSUPPORTED with the reason / NVRTC log copied into log (NUL-terminated, truncated to log_bytes). */
int lt_debug_compile_cl(const char* kernel_file_path, char* log, uint64_t log_bytes);
/* Host-only: the translation of OpenCL C text that lt_debug_compile_cl compiles (before the runtime header and the
 * generated entry points are added).  Returns the bytes needed including the NUL; out receives the text when out_bytes
 * suffices.  *contract_off (may be NULL) = 1 when the text turns FP contraction off. */
int64_t lt_debug_translate_cl(const char* text, char* out, uint64_t out_bytes, int32_t* contract_off);

/* Maps RenderProperties*::kernelFilePath to an lt_kernel by the file's CONTENT: a descriptor file of this
 * repository (comment lines only, one reading "lt-pipeline: <tag>") or the unmodified text of one of the seven
 * kernel files the reference ships (content hash) selects the built-in pipeline that reproduces it.  Any other
 * file -- including an edited copy of a shipped kernel under its old name -- returns LT_ERR_UNSUPPORTED: the
 * renderer compiles such a file as a plug-in (lt_plugin_load), a .cu as CUDA and a .cl as OpenCL C. */
int lt_kernel_from_path(const char* kernel_file_path);
const char* lt_kernel_name(int kernel);

int lt_api_version(void);

#ifdef __cplusplus
}
#endif
#endif
