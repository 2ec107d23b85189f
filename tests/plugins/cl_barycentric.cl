// A user kernel in the style of examples/custom_kernel/resources/kernels/custom_opencl.cl: the colour of a pixel is
// the barycentric coordinates (u, v, 1 - u - v) of the first triangle its camera ray hits, black on a miss.
// Stack traversal of the 32-byte nodes, Moller-Trumbore, the reference's 10-argument entry points.
// FP_CONTRACT OFF: every operation rounds once, so the B200 and a CPU compute the same bits.
#pragma OPENCL FP_CONTRACT OFF
#pragma OPENCL EXTENSION cl_khr_fp64 : enable

#define EPSILON 0.0000001

typedef struct LinearBVHNode {
  float boundsMin[3];
  float boundsMax[3];
  int offset;  // primitivesOffset (leaf) | secondChildOffset (inner)
  ushort primitiveCount;
  uchar axis;
  uchar pad;
} LinearBVHNode;

typedef struct Primitive {
  float a[3], b[3], c[3];
  float na[3], nb[3], nc[3];
  int materialIndex;
} Primitive;

typedef struct Material {
  float diffuse[3];
  float ior;
  float dissolve;
  float emission[3];
} Material;

typedef struct LightContainer {
  uint count;
  uint primitives[64];
} LightContainer;

typedef struct Camera {
  float position[3];
  float yaw, pitch, roll;
  uint frameCount;
} Camera;

typedef struct Ray {
  float4 origin;
  float4 direction;
} Ray;

typedef struct Payload {
  float t, u, v;
  int primitiveIndex;
  int hitType;
} Payload;

__constant float4 FILM_CENTRE = (float4)(0.5f, 0.5f, 0.0f, 0.0f);

float4 toFloat4(__global const float* p, float w) { return (float4)(p[0], p[1], p[2], w); }

bool intersectTriangle(Payload* payload, Ray ray, __global Primitive* primitive) {
  const float epsilon = EPSILON;
  float4 a = toFloat4(primitive->a, 0.0f);
  float4 e1 = toFloat4(primitive->b, 0.0f) - a;
  float4 e2 = toFloat4(primitive->c, 0.0f) - a;
  float4 pvec = cross(ray.direction, e2);
  float det = dot(e1, pvec);
  if (fabs(det) < epsilon) return false;
  float invDet = 1.0f / det;
  float4 tvec = ray.origin - a;
  tvec.w = 0.0f;
  float u = dot(tvec, pvec) * invDet;
  if (u < 0 || u > 1) return false;
  float4 qvec = cross(tvec, e1);
  float v = dot(ray.direction, qvec) * invDet;
  if (v < 0 || u + v > 1) return false;
  float t = dot(e2, qvec) * invDet;
  if (t < payload->t) {
    payload->t = t;
    payload->u = u;
    payload->v = v;
    return true;
  }
  return false;
}

bool intersectBounds(Ray ray, float4 invDir, int dirIsNeg[3], __global LinearBVHNode* node) {
  float lo[3], hi[3];
  for (int k = 0; k < 3; k++) {
    lo[k] = dirIsNeg[k] ? node->boundsMax[k] : node->boundsMin[k];
    hi[k] = dirIsNeg[k] ? node->boundsMin[k] : node->boundsMax[k];
  }
  float tMin = (lo[0] - ray.origin.x) * invDir.x;
  float tMax = (hi[0] - ray.origin.x) * invDir.x;
  float tyMin = (lo[1] - ray.origin.y) * invDir.y;
  float tyMax = (hi[1] - ray.origin.y) * invDir.y;
  if (tMin > tyMax || tyMin > tMax) return false;
  if (tyMin > tMin) tMin = tyMin;
  if (tyMax < tMax) tMax = tyMax;
  float tzMin = (lo[2] - ray.origin.z) * invDir.z;
  float tzMax = (hi[2] - ray.origin.z) * invDir.z;
  if (tMin > tzMax || tzMin > tMax) return false;
  if (tzMin > tMin) tMin = tzMin;
  if (tzMax < tMax) tMax = tzMax;
  return tMax > 0;
}

void intersect(Payload* payload, Ray ray, __global LinearBVHNode* nodes, __global Primitive* primitives) {
  float4 invDir = (float4)(1.0f / ray.direction.x, 1.0f / ray.direction.y, 1.0f / ray.direction.z, 0.0f);
  int dirIsNeg[3] = {invDir.x < 0, invDir.y < 0, invDir.z < 0};
  int toVisitOffset = 0, currentNodeIndex = 0;
  int nodesToVisit[64];
  while (true) {
    __global LinearBVHNode* node = &nodes[currentNodeIndex];
    if (intersectBounds(ray, invDir, dirIsNeg, node)) {
      if (node->primitiveCount > 0) {
        for (int i = 0; i < node->primitiveCount; i++) {
          if (intersectTriangle(payload, ray, &primitives[node->offset])) {
            payload->primitiveIndex = node->offset;
            payload->hitType = 1;
          }
        }
        if (toVisitOffset == 0) break;
        currentNodeIndex = nodesToVisit[--toVisitOffset];
      } else if (dirIsNeg[node->axis]) {
        nodesToVisit[toVisitOffset++] = currentNodeIndex + 1;
        currentNodeIndex = node->offset;
      } else {
        nodesToVisit[toVisitOffset++] = node->offset;
        currentNodeIndex = currentNodeIndex + 1;
      }
    } else {
      if (toVisitOffset == 0) break;
      currentNodeIndex = nodesToVisit[--toVisitOffset];
    }
  }
}

Ray cameraRay(__global Camera* camera, int x, int y, uint width, uint height) {
  float4 film = (float4)((float)x / (float)width, (float)y / (float)height, 0.0f, 1.0f) - FILM_CENTRE;
  float c = cos(camera->yaw), s = sin(camera->yaw);
  float4 d = (float4)(0.0f, 0.0f, 5.0f, 1.0f) - film;
  Ray ray;
  ray.origin = (float4)(camera->position[0], camera->position[1], camera->position[2], 1.0f) + film;
  ray.direction = (float4)(c * d.x + s * d.z, d.y, -s * d.x + c * d.z, 0.0f);
  return ray;
}

void render(__global LinearBVHNode* nodes, __global Primitive* primitives, __global Camera* camera,
            __global float* output, int x, int y, uint width, uint height, uint depth) {
  if (x >= (int)width || y >= (int)height) return;
  Ray ray = cameraRay(camera, x, y, width, height);
  Payload payload = {FLT_MAX, 0.0f, 0.0f, 0, 0};
  intersect(&payload, ray, nodes, primitives);
  float4 colour = (float4)(0.0f);
  if (payload.hitType == 1) colour = (float4)(payload.u, payload.v, 1.0 - payload.u - payload.v, 1.0f);
  int id = (y * (int)width + x) * (int)depth;
  output[id + 0] = colour.x;
  output[id + 1] = colour.y;
  output[id + 2] = colour.z;
}

__kernel void linearKernel(__global LinearBVHNode* nodes, __global Primitive* primitives, __global Material* materials,
                           __global LightContainer* lightContainer, __global Camera* camera, __global float* output,
                           uint currentBlock, uint width, uint height, uint depth) {
  uint blocksX = width / get_global_size(0);
  int x = (currentBlock % blocksX) * get_global_size(0) + get_global_id(0);
  int y = (currentBlock / blocksX) * get_global_size(1) + get_global_id(1);
  render(nodes, primitives, camera, output, x, y, width, height, depth);
}

// the same picture, each work-item placed by its group and its position in the group
__kernel void tileKernel(__global LinearBVHNode* nodes, __global Primitive* primitives, __global Material* materials,
                         __global LightContainer* lightContainer, __global Camera* camera, __global float* output,
                         uint currentBlock, uint width, uint height, uint depth) {
  uint blocksX = width / (get_num_groups(0) * get_local_size(0));
  int x = (currentBlock % blocksX) * get_global_size(0) + get_group_id(0) * get_local_size(0) + get_local_id(0);
  int y = (currentBlock / blocksX) * get_global_size(1) + get_group_id(1) * get_local_size(1) + get_local_id(1);
  render(nodes, primitives, camera, output, x, y, width, height, depth);
}
