// host_capi.h -- flat C entry points over the C++ host classes (Model, AccelerationStructureExplicit,
// Camera, RendererCUDA/RendererOpenCL, SceneParser), so scripts can drive the same objects the C++
// examples use.  Part of liblenstrace.so; tests/ and bench.py bind it with ctypes.
#pragma once
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

void* lth_model_create(const char* obj_path);
void lth_model_destroy(void* model);
int lth_model_ok(void* model);
uint64_t lth_model_primitive_count(void* model);
void* lth_model_material_buffer(void* model);
uint64_t lth_model_material_bytes(void* model);

void* lth_as_create(void* model);
/* type: 0 = host median-split (reference semantics), 100 = GPU LBVH (ACCELERATION_STRUCTURE_TYPE_LBVH_B200),
 * 101 = host binned SAH (ACCELERATION_STRUCTURE_TYPE_SAH_B200), 102 = GPU PLOC (ACCELERATION_STRUCTURE_TYPE_PLOC_B200) */
void* lth_as_create_typed(void* model, int type);
void lth_as_destroy(void* as);
void* lth_as_node_buffer(void* as);
uint64_t lth_as_node_bytes(void* as);
void* lth_as_primitive_buffer(void* as);
uint64_t lth_as_primitive_bytes(void* as);
void* lth_as_light_buffer(void* as);
uint64_t lth_as_light_bytes(void* as);

void* lth_camera_create(float x, float y, float z, float yaw);
void lth_camera_destroy(void* camera);
void* lth_camera_buffer(void* camera);
void lth_camera_set_frame_count(void* camera, uint32_t frame_count);
void lth_camera_increment_frame_count(void* camera);
void lth_camera_set_position(void* camera, float x, float y, float z);
void lth_camera_set_rotation(void* camera, float yaw, float pitch, float roll);

/* platform: 0 = RendererOpenCL, 1 = RendererCUDA */
void* lth_renderer_create(int platform);
void lth_renderer_destroy(void* renderer, int platform);
/* device scenes the renderer currently caches (one per live AccelerationStructureExplicit/Model pair, at most 8) */
uint64_t lth_renderer_cached_scenes(void* renderer, int platform);
/* Builds the RenderProperties{CUDA,OpenCL} struct and calls Renderer::render.  ext may be NULL
 * (a RenderExtensionB200*).  thread_org_mode 0 = MAX_FIT, 1 = CUSTOM with (bx, by). */
void lth_render(void* renderer, int platform, const char* kernel_file_path, int kernel_mode, int thread_org_mode,
                uint64_t bx, uint64_t by, uint64_t width, uint64_t height, uint64_t depth, float* out,
                uint64_t out_bytes, void* as, void* model, void* camera, void* ext);

uint64_t lth_write_synthetic_scene(const char* obj_path, uint32_t grid_n, uint64_t seed);

/* runs a .scene file end to end (SceneParser -> Renderer -> out); returns 0 on success */
int lth_run_scene_file(const char* scene_path, float* out, uint64_t out_bytes, uint64_t dims_out[3]);

#ifdef __cplusplus
}
#endif
