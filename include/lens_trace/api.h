// api.h -- the complete public C++ surface of this repository in one header.
//
// It declares, with the reference's names, member order and enum values (they are the API contract: callers
// use designated initialisers and the reference's examples/tests compile against this header unchanged),
// everything the reference spreads over include/lens_trace/{structures,renderer,resource,camera,model,
// acceleration_structure_explicit,image_writer,scene_parser}.h and {cuda,opencl}/renderer_*.h.  Those file
// names still exist here as one-line forwarders to this header.  Implementations live in
// lens_trace_b200/host/*.cpp and, below the C-ABI (include/lens_trace_b200.h), in lens_trace_b200/csrc/.
#pragma once
#include <math.h>
#include <stdint.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <fstream>
#include <iostream>
#include <map>
#include <string>
#include <vector>

struct lt_ctx;
struct lt_scene;

// ================================================================================================
// enums and property structs (field order is API)
// structures.h -- public enums and property structs of the renderer surface.
// Field order is API: callers use designated initialisers in declaration order
// (reference: include/lens_trace/structures.h:5-95, tests/cuda_renderer_test.cc:30-43).
// B200 additions are opt-in and chained through the (so far unused) pNext pointer.
// ================================================================================================
enum StructureType {
  STRUCTURE_TYPE_RENDER_PROPERTIES_OPENCL,
  STRUCTURE_TYPE_THREAD_ORGANIZATION_OPENCL,
  STRUCTURE_TYPE_RENDER_PROPERTIES_CUDA,
  STRUCTURE_TYPE_THREAD_ORGANIZATION_CUDA,
  STRUCTURE_TYPE_BUFFER_TO_IMAGE_PROPERTIES,
  STRUCTURE_TYPE_ACCELERATION_STRUCTURE_PROPERTIES,
  // --- B200 extension (not in the reference) ---
  STRUCTURE_TYPE_RENDER_EXTENSION_B200 = 1000
};

enum RenderPlatform { RENDER_PLATFORM_OPENCL, RENDER_PLATFORM_CUDA, RENDER_PLATFORM_OPTIX };

enum KernelMode { KERNEL_MODE_LINEAR, KERNEL_MODE_TILE };

enum ThreadOrganizationMode { THREAD_ORGANIZATION_MODE_MAX_FIT, THREAD_ORGANIZATION_MODE_CUSTOM };

enum ImageType {
  IMAGE_TYPE_JPEG,
};

enum AccelerationStructureExplicitType {
  ACCELERATION_STRUCTURE_TYPE_BVH,
  // --- B200 extension (not in the reference): LBVH built on the GPU (lt_scene_build_lbvh), same flattened layout
  ACCELERATION_STRUCTURE_TYPE_LBVH_B200 = 100,
  // --- B200 extension: host builder with binned surface-area-heuristic splits, same flattened layout
  ACCELERATION_STRUCTURE_TYPE_SAH_B200 = 101,
  // --- B200 extension: PLOC tree built on the GPU (lt_scene_build_ploc), same flattened layout; without a usable
  // device the host SAH builder is used instead
  ACCELERATION_STRUCTURE_TYPE_PLOC_B200 = 102
};

struct ThreadOrganizationOpenCL {
  StructureType sType;
  void* pNext;
  uint64_t workBlockSize[2];
  uint64_t threadGroupSize[2];
};

struct ThreadOrganizationCUDA {
  StructureType sType;
  void* pNext;
  uint64_t blockSize[2];
};

struct RenderPropertiesOpenCL {
  StructureType sType;
  void* pNext;
  std::string kernelFilePath;
  KernelMode kernelMode;
  ThreadOrganizationMode threadOrganizationMode;
  ThreadOrganizationOpenCL threadOrganization;
  uint64_t imageDimensions[3];
  void* pOutputBuffer;
  uint64_t outputBufferSize;
  void* pAccelerationStructureExplicit;
  void* pModel;
  void* pCamera;
};

struct RenderPropertiesCUDA {
  StructureType sType;
  void* pNext;
  std::string kernelFilePath;
  KernelMode kernelMode;
  ThreadOrganizationMode threadOrganizationMode;
  ThreadOrganizationCUDA threadOrganization;
  uint64_t imageDimensions[3];
  void* pOutputBuffer;
  uint64_t outputBufferSize;
  void* pAccelerationStructureExplicit;
  void* pModel;
  void* pCamera;
};

struct BufferToImageProperties {
  StructureType sType;
  void* pNext;
  void* pBuffer;
  uint64_t bufferSize;
  uint64_t imageDimensions[3];
  ImageType imageType;
  const char* filename;
};

struct AccelerationStructureExplicitProperties {
  StructureType sType;
  void* pNext;
  AccelerationStructureExplicitType accelerationStructureExplicitType;
  void* pModel;
};

// Optional, chained on RenderProperties*::pNext.  Lets one render() call take several frames and
// keep the running mean of examples/accumulator/resources/shaders/accumulator.frag on the device.
struct RenderExtensionB200 {
  StructureType sType;     // STRUCTURE_TYPE_RENDER_EXTENSION_B200
  void* pNext;
  uint32_t frames;         // frames per render() call (0 -> 1); frame k uses frameCount + k
  uint32_t accumulate;     // 0: output = last sample; 1: running mean (accumulator.frag:10-19)
  uint32_t maxRayDepth;    // GI bounce cap (0 -> 16, global_illumination.cl:308)
  uint32_t collectStats;   // fill rays/nodeTests/triTests below (slower; not for timing)
  uint64_t rays;           // out
  uint64_t nodeTests;      // out
  uint64_t triTests;       // out
  float kernelMilliseconds;  // out: device time of the render kernels
  // --- multi-GPU (appended: older initialisers leave them 0 = one GPU) ---
  uint32_t deviceCount;    // GPUs 0 .. deviceCount-1 of this process render the call together (0, 1: device 0 only)
  uint32_t splitMode;      // 0 auto, 1 samples (one NCCL all-reduce per call), 2 tiles (blocks of 8 rows, no collective)
};

// ================================================================================================
// Renderer: the drop-in boundary
// renderer.h -- the drop-in boundary: one virtual render(void*) (reference: include/lens_trace/renderer.h:5-9).
// ================================================================================================
class Renderer {
protected:
public:
  virtual void render(void* pRenderProperties) = 0;
};

// ================================================================================================
// Resource: path lookup
// resource.h -- path lookup used for kernel and model files (reference: src/resource.cpp:3-16).
// ================================================================================================
class Resource {
public:
  // the path itself if it opens, else /usr/local/share/lens_trace/<path>, else "INVALID RESOURCE"
  static std::string findResource(std::string resourcePath);
};

// ================================================================================================
// Camera
// camera.h -- camera state + the 28-byte buffer the kernels read
// (reference: include/lens_trace/camera.h:10-41, src/camera.cpp:14-19: pos[3], yaw, pitch, roll, frameCount).
// ================================================================================================
class Camera {
private:
  struct Packed {  // the device-visible record, kept in sync by every setter
    float position[3];
    float yaw;
    float pitch;
    float roll;
    uint32_t frameCount;
  };
  Packed* packed;

public:
  Camera(float positionX, float positionY, float positionZ, float yaw = 0, float pitch = 0, float roll = 0);
  ~Camera();
  Camera(const Camera&) = delete;
  Camera& operator=(const Camera&) = delete;

  float getPositionX();
  float getPositionY();
  float getPositionZ();
  float getYaw();
  float getPitch();
  float getRoll();
  uint32_t getFrameCount();

  void setPosition(float x, float y, float z);
  void updatePosition(float x, float y, float z);

  void setRotation(float yaw, float pitch, float roll);
  void updateRotation(float yaw, float pitch, float roll);

  void incrementFrameCount();
  void resetFrameCount();
  void setFrameCount(uint32_t frameCount);  // B200 addition (multi-frame render calls)

  void* getCameraBuffer();
  uint64_t getCameraBufferSize();
};

// ================================================================================================
// OBJ/MTL reader types (namespace tinyobj for source compatibility)
// obj_loader.h -- small Wavefront OBJ/MTL reader (this project's own code).
// The type names live in namespace tinyobj only so that application code written against the
// reference's Model accessors (getAttrib/getShapes/getIndex) keeps compiling; nothing of
// tinyobjloader is included.  Behaviour that matters for parity (triangulation of quads by the
// shorter diagonal, decimal parsing, material defaults) follows tinyobjloader v2.0.0rc as vendored
// by the reference (include/tinyobjloader/tiny_obj_loader.h:837-960,1385-1500).
// ================================================================================================
namespace tinyobj {

struct index_t {
  int vertex_index;
  int normal_index;
  int texcoord_index;
};

struct attrib_t {
  std::vector<float> vertices;   // xyz
  std::vector<float> normals;    // xyz
  std::vector<float> texcoords;  // uv
};

struct mesh_t {
  std::vector<index_t> indices;
  std::vector<unsigned char> num_face_vertices;
  std::vector<int> material_ids;
};

struct shape_t {
  std::string name;
  mesh_t mesh;
};

struct material_t {
  std::string name;
  float ambient[3];
  float diffuse[3];
  float specular[3];
  float transmittance[3];
  float emission[3];
  float shininess;
  float ior;
  float dissolve;
  int illum;
};

// Reads `filename` (and the .mtl files it names, relative to its directory).  Faces are
// triangulated.  Returns false when the file cannot be opened; problems are appended to warn/err.
bool LoadObj(attrib_t* attrib, std::vector<shape_t>* shapes, std::vector<material_t>* materials, std::string* warn,
             std::string* err, const char* filename);

}  // namespace tinyobj

// ================================================================================================
// Model
// model.h -- OBJ/MTL model -> per-triangle PrimitiveInfo + 32-byte Material records
// (reference: include/lens_trace/model.h, src/model.cpp).  The loader is this project's own
// (lens_trace/obj_loader.h); it reproduces the triangulation and number parsing of the loader the
// reference vendors so primitive numbering and vertex floats come out identical.
// ================================================================================================
struct PrimitiveInfo {
  float positionA[3];
  float positionB[3];
  float positionC[3];

  float normalA[3];
  float normalB[3];
  float normalC[3];

  int materialIndex;

  float boundsMin[3];
  float boundsMax[3];
  float centroid[3];
};

struct Material {
  float diffuse[3];
  float ior;
  float dissolve;
  float emission[3];
};

// Identity of Model / AccelerationStructureExplicit objects for the renderer's device-scene cache: ids are never
// reused, and a destroyed object's id is retired so that a renderer drops the device copy it holds for it.
namespace lt {
uint64_t newObjectId();
void retireObjectId(uint64_t id);
}  // namespace lt

class Model {
private:
  uint64_t uniqueId;  // B200 addition
  std::vector<PrimitiveInfo> primitiveInfoList;
  std::vector<Material> materialList;

  std::string fileName;
  tinyobj::attrib_t attrib;
  std::vector<tinyobj::shape_t> shapes;
  std::vector<tinyobj::material_t> materials;

  std::string warning;
  std::string error;
  bool success;

public:
  Model(std::string fileName);
  ~Model();

  std::string getFileName();

  bool checkError();

  tinyobj::attrib_t getAttrib();
  std::vector<tinyobj::shape_t> getShapes();

  std::vector<PrimitiveInfo>* getPrimitiveInfoListP();

  uint64_t getMaterialBufferSize();
  void* getMaterialBuffer();

  float* getVertices();
  uint32_t getVertexCount();

  tinyobj::index_t getIndex(uint32_t index);
  uint32_t getIndexCount();

  uint64_t getUniqueId() const { return uniqueId; }  // B200 addition
};

// ================================================================================================
// AccelerationStructureExplicit
// acceleration_structure_explicit.h -- median-split BVH over a Model's triangles, flattened to the
// 32-byte DFS node array the kernels traverse (reference:
// include/lens_trace/acceleration_structure_explicit.h, src/acceleration_structure_explicit.cpp).
// Differences from the reference, all deliberate: centroid bounds are initialised (the reference
// reads them uninitialised, src/acceleration_structure_explicit.cpp:81-91, which makes its tree
// nondeterministic), primitives with coincident centroids are still split so every leaf holds one
// primitive (the kernels never test more than the first primitive of a leaf, basic.cu:168-172),
// nodes are emitted straight into the linear array, the light list is capped at its 64 slots, and
// the primitive buffer is freed.
// ================================================================================================
struct LinearBVHNode {
  float boundsMin[3];
  float boundsMax[3];

  union {
    int primitivesOffset;   // leaf
    int secondChildOffset;  // inner: first child is the next node
  };

  uint16_t primitiveCount;  // 0 = inner
  uint8_t axis;
  uint8_t pad[1];
};

struct Primitive {
  float positionA[3];
  float positionB[3];
  float positionC[3];
  float normalA[3];
  float normalB[3];
  float normalC[3];
  int materialIndex;
};

struct LightContainer {
  uint32_t count;
  uint32_t primitives[64];
};

class AccelerationStructureExplicit {
private:
  uint64_t uniqueId;  // B200 addition
  std::vector<LinearBVHNode> linearNodes;
  std::vector<Primitive> orderedPrimitives;
  LightContainer lightContainer;

public:
  AccelerationStructureExplicit(AccelerationStructureExplicitProperties accelerationStructureExplicitProperties);
  ~AccelerationStructureExplicit();

  uint64_t getNodeBufferSize();
  void* getNodeBuffer();

  uint64_t getOrderedPrimitiveBufferSize();
  void* getOrderedPrimitiveBuffer();

  uint64_t getLightContainerBufferSize();
  void* getLightContainerBuffer();

  uint64_t getUniqueId() const { return uniqueId; }  // B200 addition
};

// ================================================================================================
// ImageWriter
// image_writer.h -- float RGB buffer -> image file (reference: include/lens_trace/image_writer.h,
// src/image_writer.cpp:8-23).  JPEG encoding is out of scope here: the 8-bit conversion is the
// reference's (value * 255, no clamp) and the file is written as binary PPM; a ".pfm" filename
// writes the raw floats instead (lossless, for diffing).
// ================================================================================================
class ImageWriter {
public:
  static void writeBufferToImage(BufferToImageProperties bufferToImageProperties);
};

// ================================================================================================
// RendererB200: the one renderer behind both reference renderer classes
// renderer_b200.h -- the one renderer behind both RendererCUDA and RendererOpenCL.  Owns an lt_ctx
// (include/lens_trace_b200.h), uploads each AccelerationStructureExplicit once (cached by buffer
// identity) and maps kernelFilePath to a built-in pipeline.  Errors are printed and execution
// continues, as in the reference (src/cuda/renderer_cuda.cpp:44-46,134-136).
// ================================================================================================
struct lt_ctx;
struct lt_scene;

class RendererB200 {
private:
  // Device copy of one (AccelerationStructureExplicit, Model) pair.  Keyed by the objects' never-reused ids -- not
  // by buffer addresses, which a new object can inherit from a destroyed one -- and guarded by a sampled checksum
  // of the host buffers, so that a structure edited in place is uploaded again.  At most kMaxScenes entries (least
  // recently used goes first); entries of destroyed objects are dropped at the next render().
  struct CachedScene {
    uint64_t asId, modelId;
    uint64_t checksum;
    uint64_t lastUse;
    lt_scene* scene;
    lt_scene* groupScene;  // the same scene replicated on the devices of groupCtx, when it was rendered there
  };
  static const size_t kMaxScenes = 8;
  lt_ctx* ctx;
  std::vector<CachedScene> sceneCache;
  lt_ctx* groupCtx;      // multi-GPU context (lt_ctx_create_multi), made on first use of RenderExtensionB200::deviceCount
  uint32_t groupDevices;
  uint64_t useCounter;
  uint64_t seenRetireGeneration;
  std::map<std::string, int> kernelCache;
  std::map<std::string, int> pluginCache;  // user .cu kernels compiled for this context

public:
  RendererB200();
  ~RendererB200();
  RendererB200(const RendererB200&) = delete;
  RendererB200& operator=(const RendererB200&) = delete;

  bool valid() const { return ctx != nullptr; }
  void forgetScenes();  // drops every cached device scene
  size_t cachedSceneCount() const { return sceneCache.size(); }

  void renderCommon(const std::string& kernelFilePath, KernelMode kernelMode, const uint64_t blockSize[2],
                    const uint64_t imageDimensions[3], void* pOutputBuffer, uint64_t outputBufferSize,
                    void* pAccelerationStructureExplicit, void* pModel, void* pCamera, void* pNext);
};

// ================================================================================================
// RendererCUDA
// renderer_cuda.h -- RendererCUDA with the reference's interface
// (include/lens_trace/cuda/renderer_cuda.h:16-29); implemented on the B200 kernels, no NVRTC.
// ================================================================================================
class RendererCUDA final : public Renderer {
private:
  RendererB200* impl;  // behind a pointer: the class layout stays fixed for compiled applications

public:
  RendererCUDA();
  ~RendererCUDA();

  RendererCUDA(const RendererCUDA&) = delete;
  RendererCUDA& operator=(const RendererCUDA&) = delete;

  void render(void* pRenderProperties);
  RendererB200* b200() { return impl; }  // B200 addition: the shared implementation (scene cache control, tests)
};

// ================================================================================================
// RendererOpenCL
// renderer_opencl.h -- RendererOpenCL with the reference's interface
// (include/lens_trace/opencl/renderer_opencl.h:16-43).  There is no OpenCL dispatch: the kernel
// file named by RenderPropertiesOpenCL::kernelFilePath selects one of the built-in sm_100a
// pipelines; an unknown .cl is a reported error.
// ================================================================================================
class RendererOpenCL final : public Renderer {
private:
  RendererB200* impl;  // behind a pointer: the class layout stays fixed for compiled applications

public:
  RendererOpenCL();
  ~RendererOpenCL();

  RendererOpenCL(const RendererOpenCL&) = delete;
  RendererOpenCL& operator=(const RendererOpenCL&) = delete;

  void render(void* pRenderProperties);
  RendererB200* b200() { return impl; }  // B200 addition
};

// ================================================================================================
// SceneParser
// scene_parser.h -- JSON .scene file -> Camera / Model / AccelerationStructureExplicit / RenderProperties*
// (reference: include/lens_trace/scene_parser.h, src/scene_parser.cpp; same keys, same defaults).
// The JSON reader is this project's own (lens_trace_b200/host/scene_parser.cpp).  B200 additions,
// all optional, under "renderer": "frames", "accumulate", "max_ray_depth", "devices", "split".
// ================================================================================================
struct RendererParsed {
  RenderPlatform renderPlatform = RENDER_PLATFORM_OPENCL;
  std::string kernelFilePath = "resources/kernels/opencl/basic.cl";
  std::string kernelName = "basic";
  KernelMode kernelMode = KERNEL_MODE_LINEAR;
  ThreadOrganizationMode threadOrganizationMode = THREAD_ORGANIZATION_MODE_MAX_FIT;
  uint64_t workBlockSize[2] = {32, 32};
  uint64_t threadGroupSize[2] = {32, 32};
  uint64_t blockSize[2] = {32, 32};
  uint64_t imageDimensions[3] = {2048, 2048, 3};
  uint32_t frames = 1;        // B200
  uint32_t accumulate = 0;    // B200
  uint32_t maxRayDepth = 0;   // B200 (0 -> 16)
  uint32_t deviceCount = 0;   // B200: "devices" (GPUs 0..n-1 render each call together)
  uint32_t splitMode = 0;     // B200: "split": "samples" | "tiles" (default: chosen per call)
};

struct CameraParsed {
  float position[3] = {0, 0, 0};
  float pitch = 0;
  float yaw = 0;
  float roll = 0;
};

struct ModelParsed {
  std::string filePath;
};

struct WorldParsed {
  std::vector<ModelParsed> models;
};

struct OutputParsed {
  std::string filePath = "output.jpg";
};

class SceneParser {
private:
  RendererParsed rendererParsed;
  CameraParsed cameraParsed;
  WorldParsed worldParsed;
  OutputParsed outputParsed;
  bool parsedOk;

public:
  SceneParser(std::string filename);
  ~SceneParser();

  bool ok() const { return parsedOk; }

  uint64_t getOutputBufferSize();
  RenderPlatform getRenderPlatform();

  void* createOutputBuffer();

  Camera* createCamera();
  Model* createModel();
  AccelerationStructureExplicit* createAccelerationStructure(Model* model);

  RenderPropertiesOpenCL getRenderPropertiesOpenCL(void* outputBuffer,
                                                   AccelerationStructureExplicit* accelerationStructureExplicit,
                                                   Model* model, Camera* camera);
  RenderPropertiesCUDA getRenderPropertiesCUDA(void* outputBuffer,
                                               AccelerationStructureExplicit* accelerationStructureExplicit,
                                               Model* model, Camera* camera);
  BufferToImageProperties getBufferToImageProperties(void* outputBuffer);
  RenderExtensionB200 getRenderExtensionB200();
};

// ================================================================================================
// synthetic benchmark scenes
// synthetic_scene.h -- procedural benchmark meshes written as OBJ + MTL (BASELINE.json configs 3 and 5;
// SURVEY.md 8(d)).  Files, because Model only loads files (include/lens_trace/model.h).
// ================================================================================================
namespace lt {

// Room (floor, back, left, right, ceiling quads, non-emissive), one emissive quad under the ceiling
// (2 triangles <= the 64 light slots) and a displaced gridN x gridN height field (2*gridN^2
// triangles) inside x,z in [-2.5,2.5], y in [0,5].  Vertex heights come from a PCG32 stream seeded
// with `seed`.  Every face carries normals and a material.  Returns the triangle count, 0 on failure.
uint64_t writeSyntheticScene(const std::string& objPath, uint32_t gridN, uint64_t seed);

}  // namespace lt
