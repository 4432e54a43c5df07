// Test-only: compiles the Langevin noise generator of autoforce_b200/csrc/sgpr_math.cuh (Philox4x32-10 + Box-Muller,
// the code md.cu runs) with the host compiler so that tests/test_md_host.py can check it without a GPU.
#include "../../autoforce_b200/csrc/sgpr_math.cuh"

extern "C" void harness_philox(const uint32_t* ctr, uint32_t k0, uint32_t k1, uint32_t* out) {
    for (int i = 0; i < 4; ++i) out[i] = ctr[i];
    sgpr::philox4x32_10(out, k0, k1);
}

extern "C" void harness_langevin_normals(uint64_t seed, int n_atoms, uint64_t step, double* xi) {
    for (int i = 0; i < n_atoms; ++i) sgpr::langevin_normals(seed, (uint32_t)i, step, xi + 3 * i);
}
