// Prints sizeof / offsetof of the launch-parameter structs as the reference's own headers declare them
// (`make ref` -> _ref/abi_layouts.txt); tests/test_abi.py compares them with the ctypes mirror.
#include <cstdio>
#include <cfloat>
#include <cstddef>
#define _USE_MATH_DEFINES
#include <cmath>
#include <cuda_runtime.h>
#include <curand_kernel.h>
#include "helper_math.h"
#include "kernel_params.h"
#include "atmosphere/definitions.h"
#include "gpu_vdb.h"
#include "camera.h"
#include "light.h"
#include "bvh/bvh.h"
#include "geometry/geometry.h"
int main(){ printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(camera), sizeof(light_list), sizeof(GPU_VDB), sizeof(sphere),
 sizeof(geometry_list), sizeof(BVHNode), sizeof(OCTNode), sizeof(AtmosphereParameters), sizeof(Kernel_params), sizeof(point_light), sizeof(VDB_INFO), sizeof(AABB));
 printf("%zu %zu %zu %zu\n", offsetof(Kernel_params, integrator), offsetof(Kernel_params, energy_inject), offsetof(OCTNode, bbox), offsetof(AtmosphereParameters, transmittance_texture)); }
