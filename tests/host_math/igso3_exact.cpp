// Host build of the exact IGSO(3) angle inversion in diffusion_extensions_b200/csrc/so3d_math.cuh -- TEST HARNESS ONLY.
// tests/test_igso3_angle_law.py compiles it with g++ (into a temporary directory) and checks the fp32 arithmetic the
// sm_100a sampler inlines against the fp64 law on the CPU.  Host exp / sin stand in for the device's, so the GPU tier
// repeats the check through the kernel.
#define SO3D_HOST_ONLY 1
#include "../../diffusion_extensions_b200/csrc/so3d_math.cuh"

extern "C" void hx_igso3_angle_icdf(const float* u, const float* eps, float* w, long n) {
  for (long i = 0; i < n; ++i) w[i] = so3d::igso3_angle_icdf(u[i], eps[i]);
}
