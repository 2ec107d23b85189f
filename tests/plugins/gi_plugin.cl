// The example's global-illumination kernel (examples/global_illumination/resources/kernels/global_illumination.cl:
// shade :242-376, linearKernel :378-412, and its tileKernel) ported to the device API of
// lens_trace_b200_device_cl.h: the traversal (intersect), the RNG (random), the light sample and the hemisphere sample
// are the library's calls; shade's structure, its float4 expressions and the entry points stay as the example has
// them.  One sample per launch, seeded by camera->frameCount; linearKernel clamps to [0, 1], tileKernel does not.
// The example's bounce cap is 16; this file uses 4, the cap of the built-in LT_KERNEL_GI workload it is compared with
// bit for bit (tests/test_opencl_device_api.py).
#pragma OPENCL FP_CONTRACT OFF
#pragma OPENCL EXTENSION cl_khr_fp64 : enable

#include "lens_trace_b200_device_cl.h"

#define MAX_RAY_DEPTH 4

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

float3 diffuseOf(int primitiveIndex) {
  const RefMaterial* material = lt_material_of(primitiveIndex);
  return (float3)(material->diffuse[0], material->diffuse[1], material->diffuse[2]);
}

float3 shade(LtRay ray, float2 filmPosition, uint sampleIndex) {
  float3 directColor = (float3)(0.0f, 0.0f, 0.0f);
  float3 indirectColor = (float3)(0.0f, 0.0f, 0.0f);

  LtHit payload = lt_trace(ray.origin, ray.direction, FLT_MAX, -1, 0, LT_EPSILON_GI);

  // a miss leaves primitiveIndex 0, which the light scan tests like a hit
  if (lt_is_light(payload.primitiveIndex)) {
    directColor = (float3)(1.0f, 1.0f, 1.0f);
  } else if (payload.hitType == 1) {
    float4 position, normal;
    lt_interpolate(payload.primitiveIndex, payload.u, payload.v, &position, &normal);
    float3 diffuse = diffuseOf(payload.primitiveIndex);

    LtRay shadowRay;
    float shadowT = lt_sample_light(position, lt_random(filmPosition, sampleIndex),
                                    lt_random(filmPosition, sampleIndex + 1), lt_random(filmPosition, sampleIndex + 2),
                                    &shadowRay);
    if (!lt_occluded(shadowRay.origin, shadowRay.direction, shadowT, payload.primitiveIndex, LT_EPSILON_GI)) {
      directColor = diffuse * dot(shadowRay.direction, normal);
    }

    LtRay extensionRay;
    extensionRay.origin = position;
    extensionRay.direction = lt_sample_hemisphere(lt_random(filmPosition, sampleIndex + 3),
                                                  lt_random(filmPosition, sampleIndex + 4), normal);
    float4 previousNormal = normal;
    int previousPrimitiveIndex = payload.primitiveIndex;

    bool active = true;
    for (int depth = 0; depth < MAX_RAY_DEPTH && active; depth++) {
      LtHit extension = lt_trace(extensionRay.origin, extensionRay.direction, FLT_MAX, previousPrimitiveIndex, 0,
                                 LT_EPSILON_GI);

      if (lt_is_light(extension.primitiveIndex)) {
        // the ray is not advanced: every remaining depth finds the light again
        float3 lightColor = (float3)(1.0f, 1.0f, 1.0f);
        float weight = 1.0 / (depth + 1);
        indirectColor += weight * lightColor * dot(previousNormal, extensionRay.direction);
      } else if (extension.hitType == 1) {
        lt_interpolate(extension.primitiveIndex, extension.u, extension.v, &position, &normal);
        diffuse = diffuseOf(extension.primitiveIndex);
        previousPrimitiveIndex = extension.primitiveIndex;

        uint lightIndex = sampleIndex + depth + 5;
        shadowT = lt_sample_light(position, lt_random(filmPosition, lightIndex),
                                  lt_random(filmPosition, lightIndex + 1), lt_random(filmPosition, lightIndex + 2),
                                  &shadowRay);
        if (!lt_occluded(shadowRay.origin, shadowRay.direction, shadowT, previousPrimitiveIndex, LT_EPSILON_GI)) {
          float weight = 1.0 / (depth + 1);
          indirectColor += weight * diffuse * dot(shadowRay.direction, normal);

          extensionRay.origin = position;
          extensionRay.direction = lt_sample_hemisphere(lt_random(filmPosition, sampleIndex + depth + 8),
                                                        lt_random(filmPosition, sampleIndex + depth + 9), normal);
          previousNormal = normal;
        } else {
          active = false;
        }
      } else {
        active = false;
      }
    }
  }

  return directColor + indirectColor;
}

__kernel void linearKernel(__global LinearBVHNode* nodes, __global Primitive* primitives, __global Material* materials,
                           __global LightContainer* lightContainer, __global Camera* camera, __global float* output,
                           uint currentBlock, uint width, uint height, uint depth) {
  uint blocksX = width / get_global_size(0);
  int x = (currentBlock % blocksX) * get_global_size(0) + get_global_id(0);
  int y = (currentBlock / blocksX) * get_global_size(1) + get_global_id(1);
  if (x >= (int)width || y >= (int)height) return;

  float2 filmPosition;
  LtRay ray = lt_camera_ray(camera, x, y, width, height, &filmPosition);
  float3 color = clamp(shade(ray, filmPosition, camera->frameCount), 0.0f, 1.0f);

  int id = (y * (int)width + x) * (int)depth;
  output[id + 0] = color.x;
  output[id + 1] = color.y;
  output[id + 2] = color.z;
}

__kernel void tileKernel(__global LinearBVHNode* nodes, __global Primitive* primitives, __global Material* materials,
                         __global LightContainer* lightContainer, __global Camera* camera, __global float* output,
                         uint currentBlock, uint width, uint height, uint depth) {
  uint blockWidth = get_num_groups(0) * get_local_size(0), blockHeight = get_num_groups(1) * get_local_size(1);
  uint blocksX = width / blockWidth;
  int x = (currentBlock % blocksX) * blockWidth + get_group_id(0) * get_local_size(0) + get_local_id(0);
  int y = (currentBlock / blocksX) * blockHeight + get_group_id(1) * get_local_size(1) + get_local_id(1);
  if (x >= (int)width || y >= (int)height) return;

  float2 filmPosition;
  LtRay ray = lt_camera_ray(camera, x, y, width, height, &filmPosition);
  float3 color = shade(ray, filmPosition, camera->frameCount);

  int id = (y * (int)width + x) * (int)depth;
  output[id + 0] = color.x;
  output[id + 1] = color.y;
  output[id + 2] = color.z;
}
