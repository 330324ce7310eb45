// Test harness of lr_poisson (lr_common.cuh), compiled by tests/test_gpu_predictive.py with the library's nvcc flags: one draw
// per (mean, counter) pair, applied elementwise on the legacy default stream.
#include "../literate_b200/csrc/lr_common.cuh"

__global__ void t_poisson_kernel(const double* mu, const uint32_t* ctr, uint32_t k0, uint32_t k1, long long* y, unsigned* exh, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned e = 0;
    y[i] = lr_poisson(mu[i], ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3], k0, k1, &e);
    exh[i] = e;
}

extern "C" int t_poisson(const double* mu, const uint32_t* ctr, unsigned long long seed, long long* y, unsigned* exh, long long n) {
    t_poisson_kernel<<<(unsigned)((n + 255) / 256), 256>>>(mu, ctr, (uint32_t)seed, (uint32_t)(seed >> 32), y, exh, n);
    return (int)cudaGetLastError();
}
