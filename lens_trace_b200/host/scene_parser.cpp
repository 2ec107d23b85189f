// scene_parser.cpp -- see include/lens_trace/scene_parser.h.
#include "lens_trace/scene_parser.h"

#include <ctype.h>
#include <stdio.h>
#include <stdlib.h>

#include <memory>
#include <sstream>

namespace {

// Minimal JSON value tree: enough for .scene files (objects keep key order sorted, as the
// reference's map-backed reader iterates "world" in key order, src/scene_parser.cpp:68-73).
struct JValue {
  enum Kind { NUL, BOOL, NUM, STR, ARR, OBJ } kind = NUL;
  bool b = false;
  double num = 0;
  std::string str;
  std::vector<JValue> arr;
  std::vector<std::pair<std::string, JValue>> obj;

  const JValue* get(const std::string& key) const {
    if (kind != OBJ) return nullptr;
    for (size_t i = 0; i < obj.size(); i++)
      if (obj[i].first == key) return obj[i].second.kind == NUL ? nullptr : &obj[i].second;
    return nullptr;
  }
  const JValue* at(size_t i) const { return (kind == ARR && i < arr.size()) ? &arr[i] : nullptr; }
};

struct JParser {
  const std::string& s;
  size_t i = 0;
  bool ok = true;
  explicit JParser(const std::string& text) : s(text) {}

  void ws() {
    while (i < s.size() && isspace((unsigned char)s[i])) i++;
  }
  bool eat(char c) {
    ws();
    if (i < s.size() && s[i] == c) {
      i++;
      return true;
    }
    return false;
  }
  std::string string() {
    std::string out;
    if (!eat('"')) {
      ok = false;
      return out;
    }
    while (i < s.size() && s[i] != '"') {
      if (s[i] == '\\' && i + 1 < s.size()) {
        char e = s[i + 1];
        i += 2;
        switch (e) {
          case 'n': out.push_back('\n'); break;
          case 't': out.push_back('\t'); break;
          case 'r': out.push_back('\r'); break;
          case 'b': out.push_back('\b'); break;
          case 'f': out.push_back('\f'); break;
          case 'u': i += 4; out.push_back('?'); break;
          default: out.push_back(e);
        }
      } else {
        out.push_back(s[i++]);
      }
    }
    if (i >= s.size()) ok = false;
    i++;
    return out;
  }
  JValue value() {
    JValue v;
    ws();
    if (i >= s.size()) {
      ok = false;
      return v;
    }
    char c = s[i];
    if (c == '{') {
      i++;
      v.kind = JValue::OBJ;
      if (eat('}')) return v;
      do {
        std::string k = string();
        if (!eat(':')) ok = false;
        JValue child = value();
        v.obj.push_back(std::make_pair(k, child));
      } while (ok && eat(','));
      if (!eat('}')) ok = false;
    } else if (c == '[') {
      i++;
      v.kind = JValue::ARR;
      if (eat(']')) return v;
      do v.arr.push_back(value());
      while (ok && eat(','));
      if (!eat(']')) ok = false;
    } else if (c == '"') {
      v.kind = JValue::STR;
      v.str = string();
    } else if (!s.compare(i, 4, "true")) {
      v.kind = JValue::BOOL; v.b = true; i += 4;
    } else if (!s.compare(i, 5, "false")) {
      v.kind = JValue::BOOL; v.b = false; i += 5;
    } else if (!s.compare(i, 4, "null")) {
      i += 4;
    } else {
      char* end = nullptr;
      v.num = strtod(s.c_str() + i, &end);
      if (end == s.c_str() + i) ok = false;
      v.kind = JValue::NUM;
      i = end - s.c_str();
    }
    return v;
  }
};

bool isStr(const JValue* v, const char* text) { return v && v->kind == JValue::STR && v->str == text; }
double numAt(const JValue* arr, size_t i, double def) {
  const JValue* v = arr ? arr->at(i) : nullptr;
  return (v && v->kind == JValue::NUM) ? v->num : def;
}

}  // namespace

SceneParser::SceneParser(std::string filename) : parsedOk(false) {
  std::ifstream ifs(filename.c_str());
  if (!ifs.good()) {
    printf("ERROR: cannot open scene file %s\n", filename.c_str());
    return;
  }
  std::stringstream ss;
  ss << ifs.rdbuf();
  std::string text = ss.str();
  JParser parser(text);
  JValue root = parser.value();
  if (!parser.ok || root.kind != JValue::OBJ) {
    printf("ERROR: scene file %s is not valid JSON\n", filename.c_str());
    return;
  }

  if (const JValue* r = root.get("renderer")) {
    const JValue* platform = r->get("render_platform");
    if (platform) {
      bool cl = isStr(platform, "RENDER_PLATFORM_OPENCL"), cu = isStr(platform, "RENDER_PLATFORM_CUDA");
      if (cl) rendererParsed.renderPlatform = RENDER_PLATFORM_OPENCL;
      if (cu) rendererParsed.renderPlatform = RENDER_PLATFORM_CUDA;
      const JValue* path = r->get("kernel_file_path");
      if ((cl || cu) && path && path->kind == JValue::STR) rendererParsed.kernelFilePath = path->str;
    }
    const JValue* mode = r->get("kernel_mode");
    if (isStr(mode, "KERNEL_MODE_LINEAR")) rendererParsed.kernelMode = KERNEL_MODE_LINEAR;
    if (isStr(mode, "KERNEL_MODE_TILE")) rendererParsed.kernelMode = KERNEL_MODE_TILE;
    const JValue* org = r->get("thread_organization_mode");
    if (isStr(org, "THREAD_ORGANIZATION_MODE_MAX_FIT"))
      rendererParsed.threadOrganizationMode = THREAD_ORGANIZATION_MODE_MAX_FIT;
    if (isStr(org, "THREAD_ORGANIZATION_MODE_CUSTOM")) {
      rendererParsed.threadOrganizationMode = THREAD_ORGANIZATION_MODE_CUSTOM;
      if (isStr(platform, "RENDER_PLATFORM_OPENCL")) {
        for (int k = 0; k < 2; k++) {
          rendererParsed.workBlockSize[k] = (uint64_t)numAt(r->get("work_block_size"), k, 32);
          rendererParsed.threadGroupSize[k] = (uint64_t)numAt(r->get("thread_group_size"), k, 32);
        }
      }
      if (isStr(platform, "RENDER_PLATFORM_CUDA"))
        for (int k = 0; k < 2; k++) rendererParsed.blockSize[k] = (uint64_t)numAt(r->get("block_size"), k, 32);
    }
    if (const JValue* dims = r->get("image_dimensions"))
      for (int k = 0; k < 3; k++)
        rendererParsed.imageDimensions[k] = (uint64_t)numAt(dims, k, (double)rendererParsed.imageDimensions[k]);
    if (const JValue* v = r->get("frames")) rendererParsed.frames = (uint32_t)v->num;
    if (const JValue* v = r->get("accumulate")) rendererParsed.accumulate = v->kind == JValue::BOOL ? v->b : (v->num != 0);
    if (const JValue* v = r->get("max_ray_depth")) rendererParsed.maxRayDepth = (uint32_t)v->num;
    if (const JValue* v = r->get("devices")) rendererParsed.deviceCount = (uint32_t)v->num;
    if (const JValue* v = r->get("split")) {
      if (isStr(v, "samples")) rendererParsed.splitMode = 1;
      else if (isStr(v, "tiles")) rendererParsed.splitMode = 2;
    }
    if (const JValue* v = r->get("adaptive_error")) rendererParsed.adaptiveError = (float)v->num;
    if (const JValue* v = r->get("adaptive_round_frames")) rendererParsed.adaptiveRoundFrames = (uint32_t)v->num;
    if (const JValue* v = r->get("adaptive_max_frames")) rendererParsed.adaptiveMaxFrames = (uint32_t)v->num;
  }

  if (const JValue* c = root.get("camera")) {
    if (const JValue* pos = c->get("position"))
      for (int k = 0; k < 3; k++) cameraParsed.position[k] = (float)numAt(pos, k, 0);
    if (const JValue* v = c->get("pitch")) cameraParsed.pitch = (float)v->num;
    if (const JValue* v = c->get("yaw")) cameraParsed.yaw = (float)v->num;
    if (const JValue* v = c->get("roll")) cameraParsed.roll = (float)v->num;
  }

  if (const JValue* w = root.get("world")) {
    std::vector<std::pair<std::string, std::string>> entries;
    for (size_t k = 0; k < w->obj.size(); k++) {
      const JValue* fp = w->obj[k].second.get("file_path");
      if (fp && fp->kind == JValue::STR) entries.push_back(std::make_pair(w->obj[k].first, fp->str));
    }
    std::sort(entries.begin(), entries.end());
    for (size_t k = 0; k < entries.size(); k++) {
      ModelParsed m;
      m.filePath = entries[k].second;
      worldParsed.models.push_back(m);
    }
  }

  if (const JValue* o = root.get("output"))
    if (const JValue* fp = o->get("file_path"))
      if (fp->kind == JValue::STR) outputParsed.filePath = fp->str;
  parsedOk = true;
}

SceneParser::~SceneParser() {}

uint64_t SceneParser::getOutputBufferSize() {
  return sizeof(float) * rendererParsed.imageDimensions[0] * rendererParsed.imageDimensions[1] *
         rendererParsed.imageDimensions[2];
}

RenderPlatform SceneParser::getRenderPlatform() { return rendererParsed.renderPlatform; }

void* SceneParser::createOutputBuffer() { return malloc(getOutputBufferSize()); }

Camera* SceneParser::createCamera() {
  // pitch and roll are parsed but not forwarded, as in the reference (src/scene_parser.cpp:101-103)
  return new Camera(cameraParsed.position[0], cameraParsed.position[1], cameraParsed.position[2], cameraParsed.yaw);
}

Model* SceneParser::createModel() {
  if (worldParsed.models.empty()) return nullptr;
  return new Model(worldParsed.models[0].filePath);
}

AccelerationStructureExplicit* SceneParser::createAccelerationStructure(Model* model) {
  AccelerationStructureExplicitProperties props = {};
  props.sType = STRUCTURE_TYPE_ACCELERATION_STRUCTURE_PROPERTIES;
  props.pNext = NULL;
  props.accelerationStructureExplicitType = ACCELERATION_STRUCTURE_TYPE_BVH;
  props.pModel = model;
  return new AccelerationStructureExplicit(props);
}

RenderPropertiesOpenCL SceneParser::getRenderPropertiesOpenCL(void* outputBuffer, AccelerationStructureExplicit* as,
                                                              Model* model, Camera* camera) {
  RenderPropertiesOpenCL p = {};
  p.sType = STRUCTURE_TYPE_RENDER_PROPERTIES_OPENCL;
  p.pNext = NULL;
  p.kernelFilePath = rendererParsed.kernelFilePath;
  p.kernelMode = rendererParsed.kernelMode;
  p.threadOrganizationMode = rendererParsed.threadOrganizationMode;
  for (int k = 0; k < 3; k++) p.imageDimensions[k] = rendererParsed.imageDimensions[k];
  p.pOutputBuffer = outputBuffer;
  p.outputBufferSize = getOutputBufferSize();
  p.pAccelerationStructureExplicit = as;
  p.pModel = model;
  p.pCamera = camera;
  if (rendererParsed.threadOrganizationMode == THREAD_ORGANIZATION_MODE_CUSTOM) {
    p.threadOrganization.sType = STRUCTURE_TYPE_THREAD_ORGANIZATION_OPENCL;
    p.threadOrganization.pNext = NULL;
    for (int k = 0; k < 2; k++) {
      p.threadOrganization.workBlockSize[k] = rendererParsed.workBlockSize[k];
      p.threadOrganization.threadGroupSize[k] = rendererParsed.threadGroupSize[k];
    }
  }
  return p;
}

RenderPropertiesCUDA SceneParser::getRenderPropertiesCUDA(void* outputBuffer, AccelerationStructureExplicit* as,
                                                          Model* model, Camera* camera) {
  RenderPropertiesCUDA p = {};
  p.sType = STRUCTURE_TYPE_RENDER_PROPERTIES_CUDA;
  p.pNext = NULL;
  p.kernelFilePath = rendererParsed.kernelFilePath;
  p.kernelMode = rendererParsed.kernelMode;
  p.threadOrganizationMode = rendererParsed.threadOrganizationMode;
  for (int k = 0; k < 3; k++) p.imageDimensions[k] = rendererParsed.imageDimensions[k];
  p.pOutputBuffer = outputBuffer;
  p.outputBufferSize = getOutputBufferSize();
  p.pAccelerationStructureExplicit = as;
  p.pModel = model;
  p.pCamera = camera;
  if (rendererParsed.threadOrganizationMode == THREAD_ORGANIZATION_MODE_CUSTOM) {
    p.threadOrganization.sType = STRUCTURE_TYPE_THREAD_ORGANIZATION_CUDA;
    p.threadOrganization.pNext = NULL;
    for (int k = 0; k < 2; k++) p.threadOrganization.blockSize[k] = rendererParsed.blockSize[k];
  }
  return p;
}

BufferToImageProperties SceneParser::getBufferToImageProperties(void* outputBuffer) {
  BufferToImageProperties p = {};
  p.sType = STRUCTURE_TYPE_BUFFER_TO_IMAGE_PROPERTIES;
  p.pNext = NULL;
  p.pBuffer = outputBuffer;
  p.bufferSize = getOutputBufferSize();
  for (int k = 0; k < 3; k++) p.imageDimensions[k] = rendererParsed.imageDimensions[k];
  p.imageType = IMAGE_TYPE_JPEG;
  p.filename = outputParsed.filePath.c_str();
  return p;
}

RenderExtensionB200 SceneParser::getRenderExtensionB200() {
  RenderExtensionB200 e = {};
  e.sType = STRUCTURE_TYPE_RENDER_EXTENSION_B200;
  e.pNext = NULL;
  e.frames = rendererParsed.frames;
  e.accumulate = rendererParsed.accumulate;
  e.maxRayDepth = rendererParsed.maxRayDepth;
  e.deviceCount = rendererParsed.deviceCount;
  e.splitMode = rendererParsed.splitMode;
  e.adaptiveError = rendererParsed.adaptiveError;
  e.adaptiveRoundFrames = rendererParsed.adaptiveRoundFrames;
  e.adaptiveMaxFrames = rendererParsed.adaptiveMaxFrames;
  return e;
}
