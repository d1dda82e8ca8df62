// Host build of the exact sampler's pathwise angle derivative in diffusion_extensions_b200/csrc/so3d_math.cuh -- TEST HARNESS
// ONLY.  tests/test_igso3_rsample_law.py compiles it with g++ (into a temporary directory) and checks the fp32 arithmetic the
// sm_100a backward kernel inlines against the fp64 law on the CPU.  Host exp / sin stand in for the device's, so the GPU tier
// repeats the check through the kernel.
#define SO3D_HOST_ONLY 1
#include "../../diffusion_extensions_b200/csrc/so3d_math.cuh"

extern "C" void hr_igso3_angle_icdf(const float* u, const float* eps, float* w, long n) {
  for (long i = 0; i < n; ++i) w[i] = so3d::igso3_angle_icdf(u[i], eps[i]);
}

// dw/deps at (w, eps); rows with eps == 0 take the eps -> 0+ limit from u, as the backward kernel does
extern "C" void hr_igso3_angle_deps(const float* w, const float* eps, const float* u, float* d, long n) {
  for (long i = 0; i < n; ++i) d[i] = eps[i] == 0.0f ? so3d::igso3_angle_deps_eps0(u[i]) : so3d::igso3_angle_deps(w[i], eps[i]);
}
