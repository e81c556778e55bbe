// Test probe: the library's normal_pair (csrc/dexsim_core.cuh, included unchanged) applied to caller-given Philox words,
// so tests/test_normal_draws.py can sweep every input value.  Compiled by that test with the library's nvcc flags.
#include "../dexterous_rl_manipulation_b200/csrc/dexsim_core.cuh"

__global__ void normal_pair_probe_kernel(const uint32_t* __restrict__ wa, const uint32_t* __restrict__ wb,
                                         float* __restrict__ z0, float* __restrict__ z1, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        dexsim::normal_pair(wa[i], wb[i], z0[i], z1[i]);
}

extern "C" int normal_pair_probe(const uint32_t* wa, const uint32_t* wb, float* z0, float* z1, int64_t n, void* stream) {
    if (n <= 0) return 0;
    const int grid = (int)((n + 255) / 256 > 8192 ? 8192 : (n + 255) / 256);
    normal_pair_probe_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(wa, wb, z0, z1, n);
    return (int)cudaGetLastError();
}
