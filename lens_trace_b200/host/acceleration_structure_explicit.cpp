// acceleration_structure_explicit.cpp -- deterministic median-split BVH, emitted directly in the
// reference's flattened DFS layout (see the header for the list of deliberate differences).
// Split rule, leaf rule and ordering follow src/acceleration_structure_explicit.cpp:47-137:
//   bounds = union of the primitive bounds; one primitive -> leaf; otherwise take the axis with the
//   strictly largest centroid extent (x if it beats both, else y if it beats z, else z);
//   std::nth_element at (start+end)/2 on the centroid of that axis, left = [start,mid),
//   right = [mid,end).  Equal centroids on that axis: see the comment in build().
#include "lens_trace/acceleration_structure_explicit.h"

#include <float.h>
#include <stdio.h>

#include "lens_trace_b200.h"

namespace {

struct BuildItem {
  float centroid[3];
  uint32_t source;  // index into the model's primitive list
};

struct Builder {
  const std::vector<PrimitiveInfo>& prims;
  std::vector<BuildItem> items;
  std::vector<LinearBVHNode>& nodes;
  std::vector<uint32_t> order;  // leaf order -> source primitive
  bool sah = false;             // ACCELERATION_STRUCTURE_TYPE_SAH_B200: binned surface-area-heuristic splits

  Builder(const std::vector<PrimitiveInfo>& p, std::vector<LinearBVHNode>& n) : prims(p), nodes(n) {
    items.resize(p.size());
    for (size_t i = 0; i < p.size(); i++) {
      memcpy(items[i].centroid, p[i].centroid, sizeof(float) * 3);
      items[i].source = (uint32_t)i;
    }
    nodes.reserve(p.size() * 2);
    order.reserve(p.size());
  }

  int emitLeaf(int self, int start, int end) {
    nodes[self].primitivesOffset = (int)order.size();
    nodes[self].primitiveCount = (uint16_t)(end - start);
    nodes[self].axis = 0;
    for (int i = start; i < end; i++) order.push_back(items[i].source);
    return self;
  }

  static float halfArea(const float lo[3], const float hi[3]) {
    float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    return dx * dy + dy * dz + dz * dx;
  }

  // Binned SAH (16 bins per axis over the centroid bounds, all three axes): the split that minimises
  // area(left) * count(left) + area(right) * count(right).  Partitions items[start, end) and returns the first index
  // of the right part, or -1 when no split separates the centroids (the caller then falls back to the median).
  // The lower-coordinate side becomes the first child, which is what the kernels' near/far ordering by the sign of
  // the ray direction on `dim` expects.
  int sahSplit(int start, int end, const float cmin[3], const float cmax[3], int* dimOut) {
    const int kBins = 16;
    float bestCost = FLT_MAX;
    int bestDim = -1, bestBin = -1;
    for (int dim = 0; dim < 3; dim++) {
      const float extent = cmax[dim] - cmin[dim];
      if (!(extent > 0.0f)) continue;
      const float scale = (float)kBins / extent;
      int count[kBins] = {0};
      float lo[kBins][3], hi[kBins][3];
      for (int b = 0; b < kBins; b++)
        for (int k = 0; k < 3; k++) {
          lo[b][k] = FLT_MAX;
          hi[b][k] = -FLT_MAX;
        }
      for (int i = start; i < end; i++) {
        int b = (int)((items[i].centroid[dim] - cmin[dim]) * scale);
        b = b < 0 ? 0 : (b >= kBins ? kBins - 1 : b);
        const PrimitiveInfo& p = prims[items[i].source];
        count[b]++;
        for (int k = 0; k < 3; k++) {
          lo[b][k] = std::min(lo[b][k], p.boundsMin[k]);
          hi[b][k] = std::max(hi[b][k], p.boundsMax[k]);
        }
      }
      // suffix boxes, then sweep the prefix
      float rArea[kBins];
      int rCount[kBins];
      float rl[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, rh[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
      int rc = 0;
      for (int b = kBins - 1; b >= 1; b--) {
        if (count[b])
          for (int k = 0; k < 3; k++) {
            rl[k] = std::min(rl[k], lo[b][k]);
            rh[k] = std::max(rh[k], hi[b][k]);
          }
        rc += count[b];
        rCount[b] = rc;
        rArea[b] = rc ? halfArea(rl, rh) : 0.0f;
      }
      float ll[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, lh[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
      int lc = 0;
      for (int b = 1; b < kBins; b++) {  // split between bins b-1 and b
        if (count[b - 1])
          for (int k = 0; k < 3; k++) {
            ll[k] = std::min(ll[k], lo[b - 1][k]);
            lh[k] = std::max(lh[k], hi[b - 1][k]);
          }
        lc += count[b - 1];
        if (lc == 0 || rCount[b] == 0) continue;
        const float cost = halfArea(ll, lh) * (float)lc + rArea[b] * (float)rCount[b];
        if (cost < bestCost) {
          bestCost = cost;
          bestDim = dim;
          bestBin = b;
        }
      }
    }
    if (bestDim < 0) return -1;
    const float scale = (float)kBins / (cmax[bestDim] - cmin[bestDim]);
    const float base = cmin[bestDim];
    const int dim = bestDim, bin = bestBin;
    BuildItem* mid = std::partition(items.data() + start, items.data() + end, [=](const BuildItem& a) {
      int b = (int)((a.centroid[dim] - base) * scale);
      b = b < 0 ? 0 : (b >= kBins ? kBins - 1 : b);
      return b < bin;
    });
    const int m = (int)(mid - items.data());
    if (m == start || m == end) return -1;
    *dimOut = dim;
    return m;
  }

  int build(int start, int end) {
    int self = (int)nodes.size();
    nodes.push_back(LinearBVHNode());
    {
      LinearBVHNode& n = nodes[self];
      memset(&n, 0, sizeof n);
      const PrimitiveInfo& first = prims[items[start].source];
      memcpy(n.boundsMin, first.boundsMin, sizeof(float) * 3);
      memcpy(n.boundsMax, first.boundsMax, sizeof(float) * 3);
      for (int i = start; i < end; i++) {
        const PrimitiveInfo& p = prims[items[i].source];
        for (int k = 0; k < 3; k++) {
          n.boundsMin[k] = std::min(n.boundsMin[k], p.boundsMin[k]);
          n.boundsMax[k] = std::max(n.boundsMax[k], p.boundsMax[k]);
        }
      }
    }
    if (end - start == 1) return emitLeaf(self, start, end);

    float cmin[3] = {FLT_MAX, FLT_MAX, FLT_MAX};
    float cmax[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int i = start; i < end; i++)
      for (int k = 0; k < 3; k++) {
        cmin[k] = std::min(cmin[k], items[i].centroid[k]);
        cmax[k] = std::max(cmax[k], items[i].centroid[k]);
      }
    float extent[3] = {cmax[0] - cmin[0], cmax[1] - cmin[1], cmax[2] - cmin[2]};
    int dim = (extent[0] > extent[1] && extent[0] > extent[2]) ? 0 : (extent[1] > extent[2] ? 1 : 2);
    int mid = (start + end) / 2;
    if (sah && end - start > 2) {
      int sahDim = dim;
      const int m = sahSplit(start, end, cmin, cmax, &sahDim);
      if (m > 0) {
        nodes[self].axis = (uint8_t)sahDim;
        nodes[self].primitiveCount = 0;
        build(start, m);
        int rightChild = build(m, end);
        nodes[self].secondChildOffset = rightChild;
        return self;
      }
    }
    // Coincident centroids: the reference text would emit one multi-primitive leaf here, but its
    // kernels only ever test the first primitive of such a leaf (basic.cu:168-172), so triangles
    // would vanish -- and with its uninitialised bounds the reference in practice keeps splitting
    // (its own known-answer test, tests/cuda_renderer_test.cc:182-225, needs both green_wall
    // triangles reachable).  Split by index order instead; every leaf holds one primitive.
    if (cmax[dim] != cmin[dim])
      std::nth_element(items.begin() + start, items.begin() + mid, items.begin() + end,
                       [dim](const BuildItem& a, const BuildItem& b) { return a.centroid[dim] < b.centroid[dim]; });
    nodes[self].axis = (uint8_t)dim;
    nodes[self].primitiveCount = 0;
    build(start, mid);
    int right = build(mid, end);
    nodes[self].secondChildOffset = right;
    return self;
  }
};

}  // namespace

AccelerationStructureExplicit::AccelerationStructureExplicit(
    AccelerationStructureExplicitProperties accelerationStructureExplicitProperties) {
  uniqueId = lt::newObjectId();
  Model* pModel = (Model*)accelerationStructureExplicitProperties.pModel;
  std::vector<PrimitiveInfo>& infos = *pModel->getPrimitiveInfoListP();
  const Material* materials = (const Material*)pModel->getMaterialBuffer();
  const size_t materialCount = pModel->getMaterialBufferSize() / sizeof(Material);
  memset(&lightContainer, 0, sizeof lightContainer);
  if (infos.empty()) return;

  // opt-in: build on the GPU (Morton-order LBVH or PLOC, lens_trace_b200/csrc/lt_bvh.cu) and keep the result in the
  // same host-side buffers; if no device is usable a host build below is used instead: the median split for the
  // LBVH, the binned SAH (the closest tree in kind) for PLOC
  const int type = accelerationStructureExplicitProperties.accelerationStructureExplicitType;
  const bool ploc = type == ACCELERATION_STRUCTURE_TYPE_PLOC_B200;
  if ((type == ACCELERATION_STRUCTURE_TYPE_LBVH_B200 || ploc) && infos.size() >= 2) {
    std::vector<Primitive> input(infos.size());
    for (size_t x = 0; x < infos.size(); x++) {
      memcpy(input[x].positionA, infos[x].positionA, sizeof(float) * 18);  // positions + normals are contiguous
      input[x].materialIndex = infos[x].materialIndex;
    }
    lt_ctx* ctx = nullptr;
    lt_scene* scene = nullptr;
    auto build = ploc ? lt_scene_build_ploc : lt_scene_build_lbvh;
    bool ok = lt_ctx_create(0, &ctx) == LT_OK &&
              build(ctx, input.data(), input.size() * sizeof(Primitive), materials, materialCount * sizeof(Material),
                    &scene) == LT_OK;
    if (ok) {
      linearNodes.resize(2 * infos.size() - 1);
      orderedPrimitives.resize(infos.size());
      ok = lt_scene_download(ctx, scene, linearNodes.data(), linearNodes.size() * sizeof(LinearBVHNode),
                             orderedPrimitives.data(), orderedPrimitives.size() * sizeof(Primitive),
                             &lightContainer) == LT_OK;
    }
    if (!ok)
      printf("WARNING: GPU BVH build unavailable (%s); using the host %sbuilder\n", lt_last_error(ctx), ploc ? "SAH " : "");
    if (scene) lt_scene_release(ctx, scene);
    if (ctx) lt_ctx_destroy(ctx);
    if (ok) return;
    linearNodes.clear();
    orderedPrimitives.clear();
    memset(&lightContainer, 0, sizeof lightContainer);
  }

  Builder b(infos, linearNodes);
  // opt-in: binned-SAH splits instead of the reference's median split (same layout, same kernels, fewer box tests
  // per ray; a different tree, so never the parity configuration)
  b.sah = type == ACCELERATION_STRUCTURE_TYPE_SAH_B200 || ploc;
  b.build(0, (int)infos.size());

  orderedPrimitives.resize(infos.size());
  std::vector<PrimitiveInfo> reordered(infos.size());
  for (size_t x = 0; x < b.order.size(); x++) {
    const PrimitiveInfo& src = infos[b.order[x]];
    reordered[x] = src;
    Primitive& dst = orderedPrimitives[x];
    memcpy(dst.positionA, src.positionA, sizeof(float) * 3);
    memcpy(dst.positionB, src.positionB, sizeof(float) * 3);
    memcpy(dst.positionC, src.positionC, sizeof(float) * 3);
    memcpy(dst.normalA, src.normalA, sizeof(float) * 3);
    memcpy(dst.normalB, src.normalB, sizeof(float) * 3);
    memcpy(dst.normalC, src.normalC, sizeof(float) * 3);
    dst.materialIndex = src.materialIndex;
    if (src.materialIndex >= 0 && (size_t)src.materialIndex < materialCount) {
      const Material& m = materials[src.materialIndex];
      if (m.emission[0] > 0 || m.emission[1] > 0 || m.emission[2] > 0) {
        if (lightContainer.count < 64) {
          lightContainer.primitives[lightContainer.count] = (uint32_t)x;
          lightContainer.count += 1;
        } else {
          static bool warned = false;
          if (!warned) printf("WARNING: more than 64 emissive primitives; extra lights ignored\n");
          warned = true;
        }
      }
    }
  }
  // like the reference's in-place nth_element, leave the model's list in leaf order
  infos.swap(reordered);
}

AccelerationStructureExplicit::~AccelerationStructureExplicit() { lt::retireObjectId(uniqueId); }

uint64_t AccelerationStructureExplicit::getNodeBufferSize() { return sizeof(LinearBVHNode) * linearNodes.size(); }
void* AccelerationStructureExplicit::getNodeBuffer() { return linearNodes.data(); }

uint64_t AccelerationStructureExplicit::getOrderedPrimitiveBufferSize() {
  return sizeof(Primitive) * orderedPrimitives.size();
}
void* AccelerationStructureExplicit::getOrderedPrimitiveBuffer() { return orderedPrimitives.data(); }

uint64_t AccelerationStructureExplicit::getLightContainerBufferSize() { return sizeof(LightContainer); }
void* AccelerationStructureExplicit::getLightContainerBuffer() { return &this->lightContainer; }

static_assert(sizeof(LinearBVHNode) == 32, "LinearBVHNode must stay 32 bytes");
static_assert(sizeof(Primitive) == 76, "Primitive must stay 76 bytes");
static_assert(sizeof(LightContainer) == 260, "LightContainer must stay 260 bytes");
