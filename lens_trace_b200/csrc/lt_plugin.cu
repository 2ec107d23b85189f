// lt_plugin.cu -- user-written CUDA kernels with the reference's plug-in ABI.
//
// The reference compiles the file named by RenderPropertiesCUDA::kernelFilePath at run time with NVRTC
// and launches its `linearKernel` / `tileKernel` entry point with
//   (LinearBVHNode*, Primitive*, Material*, LightContainer*, Camera*, float* out, int W, int H, int depth)
// (src/cuda/renderer_cuda.cpp:20-39,67-72,113-133; resources/kernels/cuda/basic.cu:331-340).  The seven
// shipped kernels map to built-in pipelines; any OTHER .cu file goes through here: compiled once per
// context for sm_100a (once for all devices of a multi-GPU context, which loads the cubin on each), cached, and
// launched on the buffers of the uploaded scene in the reference's layouts.  NVRTC and the driver API are loaded lazily with dlopen so that liblt_b200.so itself has no
// link-time dependency on them (it must load on machines without a GPU).
#include <cuda.h>
#include <dlfcn.h>
#include <nvrtc.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "lt_internal.h"

namespace {

struct Api {
  bool tried = false, ok = false, triedRtc = false, okRtc = false;
  std::string why, whyRtc;
  nvrtcResult (*createProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*);
  nvrtcResult (*compileProgram)(nvrtcProgram, int, const char* const*);
  nvrtcResult (*getProgramLogSize)(nvrtcProgram, size_t*);
  nvrtcResult (*getProgramLog)(nvrtcProgram, char*);
  nvrtcResult (*getCUBINSize)(nvrtcProgram, size_t*);
  nvrtcResult (*getCUBIN)(nvrtcProgram, char*);
  nvrtcResult (*destroyProgram)(nvrtcProgram*);
  CUresult (*moduleLoadData)(CUmodule*, const void*);
  CUresult (*moduleUnload)(CUmodule);
  CUresult (*moduleGetFunction)(CUfunction*, CUmodule, const char*);
  CUresult (*launchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, CUstream,
                           void**, void**);
  CUresult (*moduleGetGlobal)(CUdeviceptr*, size_t*, CUmodule, const char*);
  CUresult (*memcpyHtoDAsync)(CUdeviceptr, const void*, size_t, CUstream);
  CUresult (*funcSetAttribute)(CUfunction, CUfunction_attribute, int);
};

Api g_api;

template <class F>
bool sym(void* lib, const char* name, F& out, std::string& why) {
  out = (F)dlsym(lib, name);
  if (!out) why = std::string("missing symbol ") + name;
  return out != nullptr;
}

// NVRTC alone is enough to translate and compile (lt_debug_compile_cl); loading and launching needs the driver too
bool load_nvrtc() {
  Api& a = g_api;
  if (a.triedRtc) return a.okRtc;
  a.triedRtc = true;
  void* rtc = nullptr;
  const char* rtcNames[] = {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12",
                            "/usr/local/cuda/lib64/libnvrtc.so"};
  for (const char* n : rtcNames)
    if ((rtc = dlopen(n, RTLD_NOW | RTLD_LOCAL))) break;
  if (!rtc) {
    a.whyRtc = "libnvrtc not found";
    return false;
  }
  a.okRtc = sym(rtc, "nvrtcCreateProgram", a.createProgram, a.whyRtc) &&
            sym(rtc, "nvrtcCompileProgram", a.compileProgram, a.whyRtc) &&
            sym(rtc, "nvrtcGetProgramLogSize", a.getProgramLogSize, a.whyRtc) &&
            sym(rtc, "nvrtcGetProgramLog", a.getProgramLog, a.whyRtc) &&
            sym(rtc, "nvrtcGetCUBINSize", a.getCUBINSize, a.whyRtc) && sym(rtc, "nvrtcGetCUBIN", a.getCUBIN, a.whyRtc) &&
            sym(rtc, "nvrtcDestroyProgram", a.destroyProgram, a.whyRtc);
  return a.okRtc;
}

bool load_api() {
  Api& a = g_api;
  if (a.tried) return a.ok;
  a.tried = true;
  if (!load_nvrtc()) {
    a.why = a.whyRtc;
    return false;
  }
  void* drv = dlopen("libcuda.so.1", RTLD_NOW | RTLD_LOCAL);
  if (!drv) {
    a.why = "libcuda.so.1 not found";
    return false;
  }
  a.ok = sym(drv, "cuModuleLoadData", a.moduleLoadData, a.why) &&
         sym(drv, "cuModuleUnload", a.moduleUnload, a.why) && sym(drv, "cuModuleGetFunction", a.moduleGetFunction, a.why) &&
         sym(drv, "cuLaunchKernel", a.launchKernel, a.why) && sym(drv, "cuModuleGetGlobal_v2", a.moduleGetGlobal, a.why) &&
         sym(drv, "cuMemcpyHtoDAsync_v2", a.memcpyHtoDAsync, a.why) &&
         sym(drv, "cuFuncSetAttribute", a.funcSetAttribute, a.why);
  return a.ok;
}

}  // namespace

struct LtPlugin {
  std::string path;
  bool openclC = false;  // a .cl file: launched with the reference's OpenCL arguments (lt_plugin_launch_cl)
  CUmodule module = nullptr;
  CUfunction linear = nullptr, tile = nullptr;
  CUdeviceptr sceneSymbol = 0;  // address of the plug-in's `lt_scene` constant, 0 if it does not use the device API
};

// texts of include/lens_trace_b200_device.cuh, lt_device.cuh, lt_device_types.h, lt_opencl_c.cuh and
// include/lens_trace_b200_device_cl.h, handed to NVRTC as headers
#include "lt_device_api_embed.inc"

namespace {

bool read_text(const char* path, std::string* text, std::string* err) {
  FILE* f = fopen(path, "rb");
  if (!f) {
    *err = std::string("cannot open kernel file ") + path;
    return false;
  }
  char buf[4096];
  size_t n;
  while ((n = fread(buf, 1, sizeof buf, f)) > 0) text->append(buf, n);
  fclose(f);
  return true;
}

bool is_ident(char c) { return (c >= 'a' && c <= 'z') || (c >= 'A' && c <= 'Z') || (c >= '0' && c <= '9') || c == '_'; }

// `(T)(` with T one of the OpenCL vector types this library provides, spaces and tabs allowed inside; returns the
// length of the match (0: none) and the type in *type
size_t vector_literal_at(const std::string& s, size_t i, std::string* type) {
  static const char* kTypes[] = {"float2", "float3", "float4", "int2", "int3", "int4", "uint2", "uint3", "uint4"};
  size_t j = i + 1;
  while (j < s.size() && (s[j] == ' ' || s[j] == '\t')) j++;
  size_t b = j;
  while (j < s.size() && is_ident(s[j])) j++;
  std::string id = s.substr(b, j - b);
  bool known = false;
  for (const char* t : kTypes) known = known || id == t;
  if (!known) return 0;
  while (j < s.size() && (s[j] == ' ' || s[j] == '\t')) j++;
  if (j >= s.size() || s[j] != ')') return 0;
  j++;
  while (j < s.size() && (s[j] == ' ' || s[j] == '\t')) j++;
  if (j >= s.size() || s[j] != '(') return 0;
  *type = id;
  return j + 1 - i;
}

std::string vector_literals_only(const std::string& line) {
  std::string out, type;
  for (size_t i = 0; i < line.size();) {
    size_t m = line[i] == '(' ? vector_literal_at(line, i, &type) : 0;
    if (m) {
      out += type + "(";
      i += m;
    } else {
      out += line[i++];
    }
  }
  return out;
}

}  // namespace

// OpenCL C -> the C++ that lt_opencl_c.cuh makes of it.  One pass over the text that keeps every line where it was:
//   - `(floatN)(`, `(intN)(`, `(uintN)(` -> `floatN(` ... (vector literal -> constructor call), also in directives
//   - `__constant` / `constant` at file scope -> `__constant__ const` (device constant data), elsewhere `const`;
//     `__global`, `__private` and their spellings without underscores -> nothing; `__kernel` / `kernel` ->
//     `__device__` (entry points are generated apart); `__local` / `local` -> an undefined name, so that local memory
//     is a compile error at the user's line.  (Macros cannot do this: CUDA's own __global__ expands to `global`.)
//   - `#pragma OPENCL ...` lines are dropped; `#pragma OPENCL FP_CONTRACT OFF` anywhere turns contraction off for the
//     whole file (*contractOff)
//   - `#include "lens_trace_b200_device_cl.h"` is dropped and reported (*deviceApi): cl_source places the device API
//     ahead of the text; `#include "lens_trace_b200_device.cuh"` becomes an #error that names the OpenCL C header
//   - the `__kernel void <name>` declarations are recorded with their lines (*kernels)
// Comments, string and character literals are copied unchanged.
std::string lt_cl_translate(const std::string& src, bool* contractOff, bool* deviceApi,
                            std::vector<std::pair<std::string, int>>* kernels) {
  std::string out;
  out.reserve(src.size() + src.size() / 8);
  *contractOff = false;
  *deviceApi = false;
  int line = 1, braces = 0, parens = 0;
  bool lineStart = true;
  std::string type;
  for (size_t i = 0; i < src.size();) {
    char c = src[i];
    if (c == '\n') {
      out += c;
      line++;
      i++;
      lineStart = true;
      continue;
    }
    if (lineStart && (c == ' ' || c == '\t' || c == '\r')) {
      out += c;
      i++;
      continue;
    }
    if (lineStart && c == '#') {  // a directive, with its continuation lines
      size_t e = i;
      while (e < src.size() && src[e] != '\n') {
        if (src[e] == '\\' && e + 1 < src.size() && src[e + 1] == '\n') e++;
        e++;
      }
      std::string d = src.substr(i, e - i);
      std::string words;  // the directive's tokens, single-spaced
      for (size_t k = 1; k < d.size(); k++) {
        if (d[k] == ' ' || d[k] == '\t' || d[k] == '\\' || d[k] == '\n' || d[k] == '\r') {
          if (!words.empty() && words.back() != ' ') words += ' ';
        } else {
          words += d[k];
        }
      }
      const bool clApi = words == "include \"lens_trace_b200_device_cl.h\"";
      if (words.compare(0, 14, "pragma OPENCL ") == 0 || clApi) {
        if (words.compare(0, 30, "pragma OPENCL FP_CONTRACT OFF") == 0) *contractOff = true;
        *deviceApi = *deviceApi || clApi;
        for (char ch : d)
          if (ch == '\n') out += '\n';
      } else if (words == "include \"lens_trace_b200_device.cuh\"") {
        out += "#error \"an OpenCL C kernel file includes lens_trace_b200_device_cl.h for the device API\"";
        for (char ch : d)
          if (ch == '\n') out += '\n';
      } else {
        out += vector_literals_only(d);
      }
      for (char ch : d) line += ch == '\n';
      i = e;
      continue;
    }
    lineStart = false;
    if (c == '/' && i + 1 < src.size() && (src[i + 1] == '/' || src[i + 1] == '*')) {  // comment
      size_t e = src[i + 1] == '/' ? src.find('\n', i) : src.find("*/", i + 2);
      e = e == std::string::npos ? src.size() : (src[i + 1] == '/' ? e : e + 2);
      for (size_t k = i; k < e; k++) line += src[k] == '\n';
      out.append(src, i, e - i);
      i = e;
      continue;
    }
    if (c == '"' || c == '\'') {  // string or character literal
      size_t e = i + 1;
      while (e < src.size() && src[e] != c && src[e] != '\n') e += src[e] == '\\' ? 2 : 1;
      e = e < src.size() ? e + 1 : src.size();
      out.append(src, i, e - i);
      i = e;
      continue;
    }
    if (is_ident(c) && !(c >= '0' && c <= '9')) {
      size_t e = i;
      while (e < src.size() && is_ident(src[e])) e++;
      std::string id = src.substr(i, e - i);
      if (id == "__constant" || id == "constant") {
        out += braces == 0 && parens == 0 ? "__constant__ const" : "const";
      } else if (id == "__global" || id == "global" || id == "__private" || id == "private") {
        // the generic address space of CUDA: nothing to say
      } else if (id == "__local" || id == "local") {
        out += "lt_opencl_local_memory_is_not_supported";
      } else {
        const bool isKernel = id == "__kernel" || id == "kernel";
        out += isKernel ? "__device__" : id;
        if (isKernel) {  // record `__kernel void <name>`
          size_t k = e;
          while (k < src.size() && (src[k] == ' ' || src[k] == '\t' || src[k] == '\n' || src[k] == '\r')) k++;
          if (src.compare(k, 4, "void") == 0 && k + 4 < src.size() && !is_ident(src[k + 4])) {
            k += 4;
            int at = line;
            for (size_t q = e; q < k; q++) at += src[q] == '\n';
            while (k < src.size() && (src[k] == ' ' || src[k] == '\t' || src[k] == '\n' || src[k] == '\r'))
              at += src[k++] == '\n';
            size_t b = k;
            while (k < src.size() && is_ident(src[k])) k++;
            if (k > b) kernels->push_back(std::make_pair(src.substr(b, k - b), at));
          }
        }
      }
      i = e;
      continue;
    }
    if (is_ident(c)) {  // a number (keeps 1.0f, 0x1p3 ... whole)
      size_t e = i;
      while (e < src.size() && (is_ident(src[e]) || src[e] == '.' ||
                                ((src[e] == '+' || src[e] == '-') && (src[e - 1] == 'e' || src[e - 1] == 'E' ||
                                                                      src[e - 1] == 'p' || src[e - 1] == 'P'))))
        e++;
      out.append(src, i, e - i);
      i = e;
      continue;
    }
    if (c == '(') {
      size_t m = vector_literal_at(src, i, &type);
      out += m ? type + "(" : "(";
      i += m ? m : 1;
      parens++;
      continue;
    }
    if (c == ')') parens--;
    if (c == '{') braces++;
    if (c == '}') braces--;
    out += c;
    i++;
  }
  return out;
}

namespace {

std::string quoted(const std::string& s) {
  std::string q = "\"";
  for (char c : s) {
    if (c == '"' || c == '\\') q += '\\';
    q += c;
  }
  return q + "\"";
}

// The NVRTC source of a .cl file: the runtime, the translated text in namespace lt_opencl under the user's file name
// and line numbers, and one extern "C" entry point per reference entry point the file defines.  An entry point passes
// the reference's OpenCL arguments (renderer_opencl.cpp, SURVEY.md 8(b)):
//   (nodes, primitives, materials, lightContainer, camera, output, uint currentBlock, uint W, uint H, uint depth)
// as wrappers that convert to the pointer and integer types the user declared; a kernel whose parameters do not take
// them does not compile.  The call sits on the line of the user's declaration, so the error names it.
// A file that includes lens_trace_b200_device_cl.h gets the device API first: lens_trace_b200_device.cuh at global
// scope (so that `lt_scene` keeps the name lt_plugin_module_load looks up), its OpenCL C view inside lt_opencl.
bool cl_source(const char* path, std::string* program, bool* contractOff, std::vector<std::string>* entries,
               std::string* err) {
  std::string text;
  if (!read_text(path, &text, err)) return false;
  std::vector<std::pair<std::string, int>> kernels;
  bool deviceApi = false;
  std::string body = lt_cl_translate(text, contractOff, &deviceApi, &kernels);
  std::string p = deviceApi ? "#include \"lens_trace_b200_device.cuh\"\n" : "";
  p += "#include \"lt_opencl_c.cuh\"\nnamespace lt_opencl {\n";
  if (deviceApi) p += "#include \"lens_trace_b200_device_cl.h\"\n";
  p += "#line 1 " + quoted(path) + "\n" + body + "\n}\n";
  bool any = false;
  for (const char* entry : {"linearKernel", "tileKernel"}) {
    int at = 0;
    for (auto& k : kernels)
      if (k.first == entry) at = k.second;
    if (!at) continue;
    any = true;
    entries->push_back(entry);
    p += "#line " + std::to_string(at) + " " + quoted(path) + "\n";
    p += std::string("extern \"C\" __global__ void ") + entry +
         "(void* n, void* p, void* m, void* l, void* c, void* o, unsigned b, unsigned w, unsigned h, unsigned d) { "
         "using lt_opencl::lt_cl_pointer; using lt_opencl::lt_cl_uint; lt_opencl::" + entry +
         "(lt_cl_pointer{n}, lt_cl_pointer{p}, lt_cl_pointer{m}, lt_cl_pointer{l}, lt_cl_pointer{c}, "
         "lt_cl_pointer{o}, lt_cl_uint{b}, lt_cl_uint{w}, lt_cl_uint{h}, lt_cl_uint{d}); }\n";
  }
  if (!any) {
    *err = std::string(path) + " defines neither `__kernel void linearKernel` nor `__kernel void tileKernel`";
    return false;
  }
  *program = p;
  return true;
}

// NVRTC -> sm_100a cubin; on failure the log (which names the user's file and line) in `err`
bool nvrtc_cubin(const std::string& program, const char* path, bool openclC, bool contractOff, std::vector<char>* cubin,
                 std::string* err) {
  nvrtcProgram prog;
  const char* headerNames[] = {"lens_trace_b200_device.cuh", "lt_device.cuh", "lt_device_types.h", "lt_opencl_c.cuh",
                               "lens_trace_b200_device_cl.h"};
  const char* headerTexts[] = {kEmbedDeviceApi, kEmbedDeviceCode, kEmbedDeviceTypes, kEmbedOpenclC, kEmbedDeviceApiCl};
  if (g_api.createProgram(&prog, program.c_str(), path, 5, headerTexts, headerNames) != NVRTC_SUCCESS) {
    *err = "nvrtcCreateProgram failed";
    return false;
  }
  // NVRTC's defaults otherwise, as in the reference (renderer_cuda.cpp:28: no options): a user's a * b + c contracts
  // exactly as it would there.  The library's own device code is written with explicit rounding intrinsics and does
  // not depend on the contraction mode.  OpenCL C lets the implementation contract too, unless the file says
  // `#pragma OPENCL FP_CONTRACT OFF`; its functions are device code without a qualifier.
  std::vector<const char*> opts = {"--gpu-architecture=sm_100a", "--std=c++17"};
  if (openclC) opts.push_back("--device-as-default-execution-space");
  if (contractOff) opts.push_back("--fmad=false");
  nvrtcResult rc = g_api.compileProgram(prog, (int)opts.size(), opts.data());
  if (rc != NVRTC_SUCCESS) {
    size_t ls = 0;
    g_api.getProgramLogSize(prog, &ls);
    std::string log(ls, '\0');
    if (ls) g_api.getProgramLog(prog, &log[0]);
    *err = std::string("NVRTC could not compile ") + path + ":\n" + log;
    g_api.destroyProgram(&prog);
    return false;
  }
  size_t cs = 0;
  g_api.getCUBINSize(prog, &cs);
  cubin->resize(cs);
  g_api.getCUBIN(prog, cubin->data());
  g_api.destroyProgram(&prog);
  return true;
}

bool has_suffix(const char* path, const char* suffix) {
  size_t n = strlen(path), m = strlen(suffix);
  return n > m && strcmp(path + n - m, suffix) == 0;
}

}  // namespace

// Translates and compiles a .cl file to sm_100a without the driver; returns false with the reason / NVRTC log in err.
bool lt_plugin_compile_cl_only(const char* path, std::string* err) {
  if (!load_nvrtc()) {
    *err = "OpenCL C kernels need NVRTC: " + g_api.whyRtc;
    return false;
  }
  std::string program;
  bool contractOff = false;
  std::vector<std::string> entries;
  std::vector<char> cubin;
  if (!cl_source(path, &program, &contractOff, &entries, err) ||
      !nvrtc_cubin(program, path, true, contractOff, &cubin, err))
    return false;
  // the entry points must be in the cubin's symbol names (NUL-terminated in its string table)
  const std::string image(cubin.begin(), cubin.end());
  for (const std::string& e : entries)
    if (image.find(std::string(1, '\0') + e + std::string(1, '\0')) == std::string::npos) {
      *err = std::string("the compiled ") + path + " holds no entry point " + e;
      return false;
    }
  return true;
}

// Compiles `path` (a .cl file as OpenCL C, anything else as CUDA) to an sm_100a cubin; on failure returns false and
// the compiler log / reason in `err`.  No device is touched: a multi-GPU context loads the one image on every device.
bool lt_plugin_compile(const char* path, LtPluginImage* img, std::string* err) {
  if (!load_api()) {
    *err = "plug-in kernels need NVRTC and the CUDA driver: " + g_api.why;
    return false;
  }
  const bool openclC = has_suffix(path, ".cl");
  std::string program;
  bool contractOff = false;
  std::vector<std::string> entries;
  if (openclC ? !cl_source(path, &program, &contractOff, &entries, err) : !read_text(path, &program, err)) return false;
  img->path = path;
  img->openclC = openclC;
  return nvrtc_cubin(program, path, openclC, contractOff, &img->cubin, err);
}

// Loads a compiled image into the context current on the calling thread; nullptr with the reason in `err` on failure.
LtPlugin* lt_plugin_module_load(const LtPluginImage& img, std::string* err) {
  LtPlugin* p = new LtPlugin();
  p->path = img.path;
  p->openclC = img.openclC;
  if (g_api.moduleLoadData(&p->module, img.cubin.data()) != CUDA_SUCCESS) {
    *err = "cuModuleLoadData failed for the compiled plug-in";
    delete p;
    return nullptr;
  }
  g_api.moduleGetFunction(&p->linear, p->module, "linearKernel");
  g_api.moduleGetFunction(&p->tile, p->module, "tileKernel");
  size_t bytes = 0;
  CUdeviceptr addr = 0;
  if (g_api.moduleGetGlobal(&addr, &bytes, p->module, "lt_scene") == CUDA_SUCCESS && bytes == sizeof(LtSceneDev))
    p->sceneSymbol = addr;
  if (!p->linear && !p->tile) {
    *err = p->path + " exports neither linearKernel nor tileKernel (extern \"C\" __global__)";
    g_api.moduleUnload(p->module);
    delete p;
    return nullptr;
  }
  return p;
}

bool lt_plugin_is_opencl_c(const LtPlugin* p) { return p->openclC; }

void lt_plugin_free(LtPlugin* p) {
  if (!p) return;
  if (p->module && g_api.ok) g_api.moduleUnload(p->module);
  delete p;
}

// Sets the plug-in's `lt_scene` (if it uses the device API) to the scene the following launches render.  Returns 0, or
// -1 with `err` set.
int lt_plugin_publish_scene(LtPlugin* p, const LtSceneDev* sceneDev, cudaStream_t stream, std::string* err) {
  if (p->sceneSymbol && sceneDev &&
      g_api.memcpyHtoDAsync(p->sceneSymbol, sceneDev, sizeof(LtSceneDev), (CUstream)stream) != CUDA_SUCCESS) {
    *err = "cannot set lt_scene of plug-in " + p->path;
    return -1;
  }
  return 0;
}

// Dynamic shared memory of a launch of plug-in `p`'s kernelMode entry point with `threads` threads per block on the
// scene `sceneDev`: a plug-in that uses the device API traverses with per-thread stacks / leaf FIFOs there (lt_trace),
// any other gets none.  Above 48 KB the entry point's limit is raised to the size.  Returns false with `err` set when
// the stacks do not fit a block.
bool lt_plugin_smem(const LtPlugin* p, int kernelMode, const LtSceneDev* sceneDev, unsigned threads, unsigned* smem,
                    std::string* err) {
  *smem = 0;
  if (!p->sceneSymbol || !sceneDev) return true;
  *smem = lt_traversal_smem(sceneDev->tnodes ? 0 : lt_stack_levels(*sceneDev), threads, false);
  if (*smem > 200u * 1024u) {
    *err = "plug-in block too large for the traversal stacks of this scene (use a smaller block)";
    return false;
  }
  CUfunction fn = kernelMode ? p->tile : p->linear;
  if (fn && *smem > 48u * 1024u) g_api.funcSetAttribute(fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)*smem);
  return true;
}

// Launch shape of the reference: grid = ceil(W/bx) x ceil(H/by), block = bx x by (32x1 for MAX_FIT,
// src/cuda/renderer_cuda.cpp:74-88).  sceneDev (published by lt_plugin_publish_scene) sizes the traversal stacks.
// Returns 0, or -1 with `err` set.
int lt_plugin_launch(LtPlugin* p, int kernelMode, const LtSceneDev* sceneDev, const void* dNodes, const void* dPrims,
                     const void* dMats, const void* dLights, const void* dCamera, float* dOut, int width, int height,
                     int depth, int bx, int by, cudaStream_t stream, std::string* err) {
  CUfunction fn = kernelMode ? p->tile : p->linear;
  if (!fn) {
    *err = p->path + (kernelMode ? " has no tileKernel" : " has no linearKernel");
    return -1;
  }
  if (bx <= 0 || by <= 0) {
    bx = 32;
    by = 1;
  }
  if ((long long)bx * by > 1024) {
    *err = "plug-in block size exceeds 1024 threads";
    return -1;
  }
  unsigned smem = 0;
  if (!lt_plugin_smem(p, kernelMode, sceneDev, (unsigned)(bx * by), &smem, err)) return -1;
  void* args[] = {(void*)&dNodes, (void*)&dPrims, (void*)&dMats, (void*)&dLights, (void*)&dCamera,
                  (void*)&dOut,   (void*)&width,  (void*)&height, (void*)&depth};
  CUresult rc = g_api.launchKernel(fn, (unsigned)((width + bx - 1) / bx), (unsigned)((height + by - 1) / by), 1,
                                   (unsigned)bx, (unsigned)by, 1, smem, (CUstream)stream, args, nullptr);
  if (rc != CUDA_SUCCESS) {
    *err = "cuLaunchKernel failed for plug-in " + p->path + " (CUresult " + std::to_string((int)rc) + ")";
    return -1;
  }
  return 0;
}

// Work block and work-group size of an OpenCL-style launch.  A work block of 0 is the whole image in that dimension; a
// group of 0 x 0 is the library's choice: the largest group of at most 256 work-items that divides the work block,
// preferring 32 or more in x.  A given group must divide the work block (OpenCL 1.2).  Returns false with `err` set.
bool lt_plugin_cl_shape(int width, int height, int* wbx, int* wby, int* gx, int* gy, std::string* err) {
  if (*wbx < 0 || *wby < 0 || *gx < 0 || *gy < 0) {
    *err = "negative work block or group size";
    return false;
  }
  if (*wbx == 0) *wbx = width;
  if (*wby == 0) *wby = height;
  if (*gx == 0 || *gy == 0) {
    int bx = 1, by = 1;
    for (int x = 1; x <= 256 && x <= *wbx; x++) {
      if (*wbx % x) continue;
      for (int y = 1; x * y <= 256 && y <= *wby; y++) {
        if (*wby % y) continue;
        bool better = x * y > bx * by || (x * y == bx * by && (x <= 32 ? x : 32) > (bx <= 32 ? bx : 32));
        if (better) bx = x, by = y;
      }
    }
    *gx = bx;
    *gy = by;
  }
  if (*wbx % *gx || *wby % *gy) {
    *err = "the work-group size (" + std::to_string(*gx) + ", " + std::to_string(*gy) + ") does not divide the work block (" +
           std::to_string(*wbx) + ", " + std::to_string(*wby) + ")";
    return false;
  }
  if ((long long)*gx * *gy > 1024 || *wby / *gy > 65535) {
    *err = "work-group size or work block too large for a launch";
    return false;
  }
  return true;
}

// The reference's OpenCL launch loop (renderer_opencl.cpp:84-146, restated in oracle/cl_shim/ref_cl_host.cpp): one
// NDRange per work block, global size = the work block, local size = the group, currentBlock = the block's index, for
// (W / wbx) * (H / wby) blocks.  Arguments as normalised by lt_plugin_cl_shape; sceneDev sizes the traversal stacks of
// a file that uses the device API, as in lt_plugin_launch.  Returns launches made, or -1 with `err` set.
int lt_plugin_launch_cl(LtPlugin* p, int kernelMode, const LtSceneDev* sceneDev, const void* dNodes, const void* dPrims,
                        const void* dMats, const void* dLights, const void* dCamera, float* dOut, int width, int height,
                        int depth, int wbx, int wby, int gx, int gy, cudaStream_t stream, std::string* err) {
  CUfunction fn = kernelMode ? p->tile : p->linear;
  if (!fn) {
    *err = p->path + (kernelMode ? " has no tileKernel" : " has no linearKernel");
    return -1;
  }
  unsigned smem = 0;
  if (!lt_plugin_smem(p, kernelMode, sceneDev, (unsigned)(gx * gy), &smem, err)) return -1;
  const unsigned blocks = (unsigned)(width / wbx) * (unsigned)(height / wby);
  unsigned block = 0, w = (unsigned)width, h = (unsigned)height, d = (unsigned)depth;
  void* args[] = {(void*)&dNodes, (void*)&dPrims, (void*)&dMats, (void*)&dLights, (void*)&dCamera,
                  (void*)&dOut,   (void*)&block,  (void*)&w,     (void*)&h,       (void*)&d};
  for (block = 0; block < blocks; block++) {
    CUresult rc = g_api.launchKernel(fn, (unsigned)(wbx / gx), (unsigned)(wby / gy), 1, (unsigned)gx, (unsigned)gy, 1,
                                     smem, (CUstream)stream, args, nullptr);
    if (rc != CUDA_SUCCESS) {
      *err = "cuLaunchKernel failed for plug-in " + p->path + " (CUresult " + std::to_string((int)rc) + ")";
      return -1;
    }
  }
  return (int)blocks;
}
