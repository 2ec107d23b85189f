/*
 * cl_file_host.cpp -- runs ONE user-written OpenCL C kernel file on the host CPU, one work-item at a time, through
 * oracle/cl_shim/opencl_c_on_cpp.h.  TEST INFRASTRUCTURE ONLY: the oracle of tests/test_opencl_plugins.py, which
 * compiles this file with g++ at test time for each kernel under test.
 *
 * It generalises oracle/cl_shim/ref_cl_host.cpp from six fixed files to one given file: the test applies the same
 * mechanical rewrite (`(floatN)(` -> `floatN(`) and passes the result as LT_CL_FILE; LT_CL_LINEAR / LT_CL_TILE say
 * which entry points it defines.  The arguments reach the user's entry point through wrappers that convert to the
 * user's own struct names, as on the device.  The launch loop is ref_cl_host.cpp's, i.e. the reference's launcher
 * (src/opencl/renderer_opencl.cpp:84-146):
 *   blocks = (W / workBlock[0]) * (H / workBlock[1])       (integer division)
 *   for b in 0..blocks: NDRange(global = workBlock, local) with args (nodes, ..., output, b, W, H, depth)
 */
#include "opencl_c_on_cpp.h"

#include <atomic>
#include <thread>
#include <vector>

thread_local clshim_work_item clshim_wi;

namespace k_user {
#include LT_CL_FILE
}

namespace {

struct arg_pointer {
  void* p;
  template <class T> operator T*() const { return (T*)p; }
};
struct arg_uint {
  uint v;
  template <class T> operator T() const { return (T)v; }
};

struct launch {
  int mode;
  void *nodes, *prims, *mats, *lights, *cam;
  float* out;
  uint W, H, depth;
  size_t wbs[2], ls[2];
};

void run_item(const launch& L, uint block) {
  arg_pointer n{L.nodes}, p{L.prims}, m{L.mats}, l{L.lights}, c{L.cam}, o{L.out};
  arg_uint b{block}, w{L.W}, h{L.H}, d{L.depth};
#ifdef LT_CL_LINEAR
  if (L.mode == 0) k_user::linearKernel(n, p, m, l, c, o, b, w, h, d);
#endif
#ifdef LT_CL_TILE
  if (L.mode == 1) k_user::tileKernel(n, p, m, l, c, o, b, w, h, d);
#endif
}

}  // namespace

extern "C" int clfile_render(int mode, void* nodes, void* prims, void* mats, void* lights, void* cam, float* out, int W,
                             int H, int depth, int workBlockX, int workBlockY, int localX, int localY, int threads) {
  if ((mode != 0 && mode != 1) || W <= 0 || H <= 0 || depth < 1) return -1;
  if (workBlockX <= 0 || workBlockY <= 0 || localX <= 0 || localY <= 0) return -1;
  if (workBlockX % localX || workBlockY % localY) return -1;
  launch L{mode, nodes, prims, mats, lights, cam, out, (uint)W, (uint)H, (uint)depth,
           {(size_t)workBlockX, (size_t)workBlockY}, {(size_t)localX, (size_t)localY}};
  uint64_t blocks = (uint64_t)(W / workBlockX) * (uint64_t)(H / workBlockY);
  uint64_t rows = blocks * (uint64_t)workBlockY;
  if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
  if (threads < 1) threads = 1;
  std::atomic<uint64_t> next{0};
  auto worker = [&]() {
    for (;;) {
      uint64_t r = next.fetch_add(1);
      if (r >= rows) break;
      uint block = (uint)(r / L.wbs[1]);
      size_t gy = (size_t)(r % L.wbs[1]);
      for (size_t gx = 0; gx < L.wbs[0]; gx++) {
        clshim_work_item& wi = clshim_wi;
        wi.global_id[0] = gx; wi.global_id[1] = gy; wi.global_id[2] = 0;
        wi.global_size[0] = L.wbs[0]; wi.global_size[1] = L.wbs[1]; wi.global_size[2] = 1;
        wi.local_size[0] = L.ls[0]; wi.local_size[1] = L.ls[1]; wi.local_size[2] = 1;
        wi.local_id[0] = gx % L.ls[0]; wi.local_id[1] = gy % L.ls[1]; wi.local_id[2] = 0;
        wi.group_id[0] = gx / L.ls[0]; wi.group_id[1] = gy / L.ls[1]; wi.group_id[2] = 0;
        wi.num_groups[0] = L.wbs[0] / L.ls[0]; wi.num_groups[1] = L.wbs[1] / L.ls[1]; wi.num_groups[2] = 1;
        run_item(L, block);
      }
    }
  };
  if (threads == 1) {
    worker();
  } else {
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; t++) pool.emplace_back(worker);
    for (auto& t : pool) t.join();
  }
  return 0;
}
