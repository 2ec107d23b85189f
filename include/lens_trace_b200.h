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

typedef struct lt_stats {
  uint64_t rays;        /* traversal calls (primary + shadow + extension + lens segments) */
  uint64_t node_tests;  /* boxes tested, reference traversal order */
  uint64_t tri_tests;   /* triangle tests executed, reference traversal order */
  float kernel_ms;      /* device time of the render kernels of the last lt_render* call (CUDA events) */
  float upload_ms;      /* device time of the last lt_scene_upload (H2D + re-flatten) */
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

/* Host-only (no device needed): the threaded form of a reference node array that lt_scene_upload builds for
 * small trees -- 8 copies of node_count 32-byte records {lo.x lo.y lo.z hi.x | hi.y hi.z link skip}, copy o in
 * the order the reference's traversal (basic.cu:156-196) visits the nodes for rays whose direction signs are
 * the bits of o (LtThreadNode, include/lens_trace_b200_device.cuh).  out_records: 8 * node_count * 32 bytes.
 * Exposed so that the layout can be checked against the reference traversal on a machine without a GPU. */
int lt_debug_build_threaded(const void* nodes, uint64_t node_bytes, void* out_records);

/* Host-only: the eight pruned copies lt_scene_upload builds beside those (same record format, inner nodes that
 * cannot change which leaves a ray reaches left out; skip links index out_records).  *out_stride receives the
 * records per copy; out_records (8 * stride * 32 bytes, at most 8 * node_count * 32) may be NULL to ask for it. */
int lt_debug_build_threaded_pruned(const void* nodes, uint64_t node_bytes, void* out_records, int32_t* out_stride);

/* Test hook: full != 0 makes launches on `scene` (single-GPU) walk the full threaded copies for every ray, 0 restores
 * the pruned ones.  The output is the same either way; tests compare the two. */
int lt_debug_scene_full_threaded(lt_scene* scene, int full);

/* --- plug-in kernels: a user-written .cu file with the reference's kernel ABI (extern "C" __global__
 * linearKernel / tileKernel(LinearBVHNode*, Primitive*, Material*, LightContainer*, Camera*, float* out,
 * int width, int height, int depth), resources/kernels/cuda/basic.cu:331-340).  Replaces the NVRTC compile
 * and launch of src/cuda/renderer_cuda.cpp:20-39,57-88,113-133 for files that are not one of the shipped
 * kernels: compiled once per context for sm_100a, then launched on the scene's buffers in the reference
 * layouts with the reference's launch shape (block_x x block_y threads, 32x1 when 0). --- */
int lt_plugin_load(lt_ctx* ctx, const char* kernel_file_path, int* out_plugin_id);
int lt_render_plugin(lt_ctx* ctx, lt_scene* scene, const void* camera28, int plugin_id, int kernel_mode, int width,
                     int height, int depth, int block_x, int block_y, float* host_out);

/* Maps RenderProperties*::kernelFilePath to an lt_kernel by the file's CONTENT: a descriptor file of this
 * repository (comment lines only, one reading "lt-pipeline: <tag>") or the unmodified text of one of the seven
 * kernel files the reference ships (content hash) selects the built-in pipeline that reproduces it.  Any other
 * file -- including an edited copy of a shipped kernel under its old name -- returns LT_ERR_UNSUPPORTED: the
 * renderer compiles such a .cu as a plug-in (lt_plugin_load) and reports an error for a .cl. */
int lt_kernel_from_path(const char* kernel_file_path);
const char* lt_kernel_name(int kernel);

int lt_api_version(void);

#ifdef __cplusplus
}
#endif
#endif
