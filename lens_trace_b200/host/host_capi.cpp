// host_capi.cpp -- see include/lens_trace/b200/host_capi.h.
#include "lens_trace/b200/host_capi.h"

#include <string.h>

#include "lens_trace/b200/synthetic_scene.h"
#include "lens_trace/scene_parser.h"

extern "C" {

void* lth_model_create(const char* obj_path) { return new Model(obj_path); }
void lth_model_destroy(void* model) { delete (Model*)model; }
int lth_model_ok(void* model) { return ((Model*)model)->getPrimitiveInfoListP()->empty() ? 0 : 1; }
uint64_t lth_model_primitive_count(void* model) { return ((Model*)model)->getPrimitiveInfoListP()->size(); }
void* lth_model_material_buffer(void* model) { return ((Model*)model)->getMaterialBuffer(); }
uint64_t lth_model_material_bytes(void* model) { return ((Model*)model)->getMaterialBufferSize(); }

void* lth_as_create(void* model) {
  AccelerationStructureExplicitProperties props = {};
  props.sType = STRUCTURE_TYPE_ACCELERATION_STRUCTURE_PROPERTIES;
  props.pNext = NULL;
  props.accelerationStructureExplicitType = ACCELERATION_STRUCTURE_TYPE_BVH;
  props.pModel = model;
  return new AccelerationStructureExplicit(props);
}
void* lth_as_create_typed(void* model, int type) {
  AccelerationStructureExplicitProperties props = {};
  props.sType = STRUCTURE_TYPE_ACCELERATION_STRUCTURE_PROPERTIES;
  props.pNext = NULL;
  props.accelerationStructureExplicitType = (AccelerationStructureExplicitType)type;
  props.pModel = model;
  return new AccelerationStructureExplicit(props);
}
void lth_as_destroy(void* as) { delete (AccelerationStructureExplicit*)as; }
void* lth_as_node_buffer(void* as) { return ((AccelerationStructureExplicit*)as)->getNodeBuffer(); }
uint64_t lth_as_node_bytes(void* as) { return ((AccelerationStructureExplicit*)as)->getNodeBufferSize(); }
void* lth_as_primitive_buffer(void* as) { return ((AccelerationStructureExplicit*)as)->getOrderedPrimitiveBuffer(); }
uint64_t lth_as_primitive_bytes(void* as) {
  return ((AccelerationStructureExplicit*)as)->getOrderedPrimitiveBufferSize();
}
void* lth_as_light_buffer(void* as) { return ((AccelerationStructureExplicit*)as)->getLightContainerBuffer(); }
uint64_t lth_as_light_bytes(void* as) { return ((AccelerationStructureExplicit*)as)->getLightContainerBufferSize(); }

void* lth_camera_create(float x, float y, float z, float yaw) { return new Camera(x, y, z, yaw); }
void lth_camera_destroy(void* camera) { delete (Camera*)camera; }
void* lth_camera_buffer(void* camera) { return ((Camera*)camera)->getCameraBuffer(); }
void lth_camera_set_frame_count(void* camera, uint32_t frame_count) { ((Camera*)camera)->setFrameCount(frame_count); }
void lth_camera_increment_frame_count(void* camera) { ((Camera*)camera)->incrementFrameCount(); }
void lth_camera_set_position(void* camera, float x, float y, float z) { ((Camera*)camera)->setPosition(x, y, z); }
void lth_camera_set_rotation(void* camera, float yaw, float pitch, float roll) {
  ((Camera*)camera)->setRotation(yaw, pitch, roll);
}

void* lth_renderer_create(int platform) {
  if (platform == 1) return new RendererCUDA();
  return new RendererOpenCL();
}
void lth_renderer_destroy(void* renderer, int platform) {
  if (platform == 1) delete (RendererCUDA*)renderer;
  else delete (RendererOpenCL*)renderer;
}

uint64_t lth_renderer_cached_scenes(void* renderer, int platform) {
  RendererB200* r = platform == 1 ? ((RendererCUDA*)renderer)->b200() : ((RendererOpenCL*)renderer)->b200();
  return r ? r->cachedSceneCount() : 0;
}

void lth_render(void* renderer, int platform, const char* kernel_file_path, int kernel_mode, int thread_org_mode,
                uint64_t bx, uint64_t by, uint64_t width, uint64_t height, uint64_t depth, float* out,
                uint64_t out_bytes, void* as, void* model, void* camera, void* ext) {
  if (platform == 1) {
    RenderPropertiesCUDA p = {};
    p.sType = STRUCTURE_TYPE_RENDER_PROPERTIES_CUDA;
    p.pNext = ext;
    p.kernelFilePath = kernel_file_path;
    p.kernelMode = kernel_mode ? KERNEL_MODE_TILE : KERNEL_MODE_LINEAR;
    p.threadOrganizationMode = thread_org_mode ? THREAD_ORGANIZATION_MODE_CUSTOM : THREAD_ORGANIZATION_MODE_MAX_FIT;
    if (thread_org_mode) {
      p.threadOrganization.sType = STRUCTURE_TYPE_THREAD_ORGANIZATION_CUDA;
      p.threadOrganization.blockSize[0] = bx;
      p.threadOrganization.blockSize[1] = by;
    }
    p.imageDimensions[0] = width; p.imageDimensions[1] = height; p.imageDimensions[2] = depth;
    p.pOutputBuffer = out;
    p.outputBufferSize = out_bytes;
    p.pAccelerationStructureExplicit = as;
    p.pModel = model;
    p.pCamera = camera;
    ((RendererCUDA*)renderer)->render(&p);
  } else {
    RenderPropertiesOpenCL p = {};
    p.sType = STRUCTURE_TYPE_RENDER_PROPERTIES_OPENCL;
    p.pNext = ext;
    p.kernelFilePath = kernel_file_path;
    p.kernelMode = kernel_mode ? KERNEL_MODE_TILE : KERNEL_MODE_LINEAR;
    p.threadOrganizationMode = thread_org_mode ? THREAD_ORGANIZATION_MODE_CUSTOM : THREAD_ORGANIZATION_MODE_MAX_FIT;
    if (thread_org_mode) {
      p.threadOrganization.sType = STRUCTURE_TYPE_THREAD_ORGANIZATION_OPENCL;
      p.threadOrganization.workBlockSize[0] = bx;
      p.threadOrganization.workBlockSize[1] = by;
      p.threadOrganization.threadGroupSize[0] = bx;
      p.threadOrganization.threadGroupSize[1] = by;
    }
    p.imageDimensions[0] = width; p.imageDimensions[1] = height; p.imageDimensions[2] = depth;
    p.pOutputBuffer = out;
    p.outputBufferSize = out_bytes;
    p.pAccelerationStructureExplicit = as;
    p.pModel = model;
    p.pCamera = camera;
    ((RendererOpenCL*)renderer)->render(&p);
  }
}

void lth_render_opencl(void* renderer, const char* kernel_file_path, int kernel_mode, int thread_org_mode,
                       uint64_t work_bx, uint64_t work_by, uint64_t group_x, uint64_t group_y, uint64_t width,
                       uint64_t height, uint64_t depth, float* out, uint64_t out_bytes, void* as, void* model,
                       void* camera, void* ext) {
  RenderPropertiesOpenCL p = {};
  p.sType = STRUCTURE_TYPE_RENDER_PROPERTIES_OPENCL;
  p.pNext = ext;
  p.kernelFilePath = kernel_file_path;
  p.kernelMode = kernel_mode ? KERNEL_MODE_TILE : KERNEL_MODE_LINEAR;
  p.threadOrganizationMode = thread_org_mode ? THREAD_ORGANIZATION_MODE_CUSTOM : THREAD_ORGANIZATION_MODE_MAX_FIT;
  if (thread_org_mode) {
    p.threadOrganization.sType = STRUCTURE_TYPE_THREAD_ORGANIZATION_OPENCL;
    p.threadOrganization.workBlockSize[0] = work_bx;
    p.threadOrganization.workBlockSize[1] = work_by;
    p.threadOrganization.threadGroupSize[0] = group_x;
    p.threadOrganization.threadGroupSize[1] = group_y;
  }
  p.imageDimensions[0] = width; p.imageDimensions[1] = height; p.imageDimensions[2] = depth;
  p.pOutputBuffer = out;
  p.outputBufferSize = out_bytes;
  p.pAccelerationStructureExplicit = as;
  p.pModel = model;
  p.pCamera = camera;
  ((RendererOpenCL*)renderer)->render(&p);
}

uint64_t lth_write_synthetic_scene(const char* obj_path, uint32_t grid_n, uint64_t seed) {
  return lt::writeSyntheticScene(obj_path, grid_n, seed);
}

int lth_run_scene_file(const char* scene_path, float* out, uint64_t out_bytes, uint64_t dims_out[3]) {
  SceneParser parser(scene_path);
  if (!parser.ok()) return -1;
  if (parser.getOutputBufferSize() > out_bytes) return -2;
  Camera* camera = parser.createCamera();
  Model* model = parser.createModel();
  if (!model) return -3;
  AccelerationStructureExplicit* as = parser.createAccelerationStructure(model);
  RenderExtensionB200 ext = parser.getRenderExtensionB200();
  if (parser.getRenderPlatform() == RENDER_PLATFORM_CUDA) {
    RendererCUDA renderer;
    RenderPropertiesCUDA p = parser.getRenderPropertiesCUDA(out, as, model, camera);
    p.pNext = &ext;
    for (int k = 0; k < 3; k++) dims_out[k] = p.imageDimensions[k];
    renderer.render(&p);
  } else {
    RendererOpenCL renderer;
    RenderPropertiesOpenCL p = parser.getRenderPropertiesOpenCL(out, as, model, camera);
    p.pNext = &ext;
    for (int k = 0; k < 3; k++) dims_out[k] = p.imageDimensions[k];
    renderer.render(&p);
  }
  delete as;
  delete model;
  delete camera;
  return 0;
}

// the RenderExtensionB200 a .scene file gives the renderer (no device needed); 0 on success
int lth_scene_extension(const char* scene_path, void* ext_out) {
  SceneParser parser(scene_path);
  if (!parser.ok() || !ext_out) return -1;
  RenderExtensionB200 ext = parser.getRenderExtensionB200();
  memcpy(ext_out, &ext, sizeof ext);
  return 0;
}

}  // extern "C"
