// Host build of the IGSO(3) entropy in diffusion_extensions_b200/csrc/so3d_math.cuh -- TEST HARNESS ONLY.
// tests/test_igso3_entropy_law.py compiles it with g++ (into a temporary directory) and checks the fp32 arithmetic the sm_100a
// entropy kernel inlines against the fp64 law on the CPU.  Host exp / log / sin stand in for the device's, so the GPU tier
// repeats the check through the kernel.
#define SO3D_HOST_ONLY 1
#include "../../diffusion_extensions_b200/csrc/so3d_math.cuh"

extern "C" void hr_igso3_entropy(const float* eps, float* H, float* dH, long n) {
  for (long i = 0; i < n; ++i) H[i] = so3d::igso3_entropy(eps[i], dH ? dH + i : nullptr);
}
