// Test-only harness of the shared sampler arithmetic in literate_b200/csrc/lr_common.cuh (tests/test_gpu_device_math.py,
// tests/test_device_math_host.py).  Not part of the library: the tests compile it into a temporary directory.
//
// Built as a shared library (-shared): one small kernel per helper, applied elementwise (per warp for the warp helpers), with an
// extern "C" launcher each that takes device pointers and a count, launches on the legacy default stream and returns the launch
// status.  Built with -DLR_HARNESS_HOST_MAIN: a host program that applies the __host__ __device__ philox4x32_10 to the
// (counter, key) tuples of stdin, six hexadecimal words a line, and prints the four output words of each.
#include "../literate_b200/csrc/lr_common.cuh"

#ifdef LR_HARNESS_HOST_MAIN
int main() {
    unsigned c0, c1, c2, c3, k0, k1;
    while (scanf("%x %x %x %x %x %x", &c0, &c1, &c2, &c3, &k0, &k1) == 6) {
        const Philox4 r = philox4x32_10(c0, c1, c2, c3, k0, k1);
        printf("%08x %08x %08x %08x\n", r.x, r.y, r.z, r.w);
    }
    return 0;
}
#else

namespace {
constexpr int THREADS = 256;
inline int blocks(long long n) { return (int)((n + THREADS - 1) / THREADS); }
}

// in[n][6] = (c0, c1, c2, c3, k0, k1) -> out[n][4]
__global__ void t_philox_kernel(const uint32_t* in, uint32_t* out, long long n) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t* a = in + 6 * i;
    const Philox4 r = philox4x32_10(a[0], a[1], a[2], a[3], a[4], a[5]);
    out[4 * i] = r.x; out[4 * i + 1] = r.y; out[4 * i + 2] = r.z; out[4 * i + 3] = r.w;
}

// hilo[n][2] = (hi, lo) -> u01(hi, lo)
__global__ void t_u01_kernel(const uint32_t* hilo, double* out, long long n) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = u01(hilo[2 * i], hilo[2 * i + 1]);
}

__global__ void t_exp_small_kernel(const double* x, double* out, long long n) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = exp_small(x[i]);
}

// the bracket of u[i] and the device's double log(u[i]): out[n][3] = (lo, hi, log u)
__global__ void t_bracket_kernel(const double* u, double* out, long long n) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    double lo, hi;
    mh_bracket(u[i], &lo, &hi);
    out[3 * i] = lo; out[3 * i + 1] = hi; out[3 * i + 2] = log(u[i]);
}

// the two accept decisions of (x[i], u[i]) and the double log(u[i]) of the same kernel: gt[i] = mh_accept_gt, ge[i] = K3's
// mh_accept_ge on the bracket of mh_bracket
__global__ void t_accept_kernel(const double* x, const double* u, int8_t* gt, int8_t* ge, double* logu, long long n) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    double lo, hi;
    mh_bracket(u[i], &lo, &hi);
    gt[i] = mh_accept_gt(x[i], u[i]);
    ge[i] = mh_accept_ge(x[i], u[i], lo, hi, [](double v) { return log(v); });
    logu[i] = log(u[i]);
}

__global__ void t_normal_kernel(const double* u1, const uint32_t* bits, double* out, long long n) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = normal_f32(u1[i], bits[i]);
}

// z[k] = normal_f32(u1, k << 8) for every angle code k = 0 .. 2^24 - 1
__global__ void t_normal_angles_kernel(double u1, double* z) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k < (1ll << 24)) z[k] = normal_f32(u1, (uint32_t)k << 8);
}

// one thread per sequence: out[s] = lr_sum over v[off[s] .. off[s + 1])
__global__ void t_lr_sum_kernel(const double* v, const long long* off, double* out, int n_seq) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seq) return;
    lr_sum acc;
    for (long long i = off[s]; i < off[s + 1]; ++i) acc.add(v[i]);
    out[s] = acc.value();
}

// key[i] = lr_key(x[i]), back[i] = lr_val(key[i])
__global__ void t_key_kernel(const double* x, unsigned long long* key, double* back, long long n) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    key[i] = lr_key(x[i]);
    back[i] = lr_val(key[i]);
}

// one warp per row of v[n_warps][32]: out[w][0][lane] = warp_sum, out[w][1][lane] = warp_sum_first(v, K[w])
__global__ void t_warp_sum_kernel(const double* v, const int* K, double* out, int n_warps) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n_warps) return;                          // warp-uniform: blockDim.x is a multiple of 32
    const double x = v[32 * w + lane];
    out[64 * w + lane] = warp_sum(x);
    out[64 * w + 32 + lane] = warp_sum_first(x, K[w]);
}

extern "C" {
int t_philox(const uint32_t* in, uint32_t* out, long long n) {
    t_philox_kernel<<<blocks(n), THREADS>>>(in, out, n);
    return (int)cudaGetLastError();
}
int t_u01(const uint32_t* hilo, double* out, long long n) {
    t_u01_kernel<<<blocks(n), THREADS>>>(hilo, out, n);
    return (int)cudaGetLastError();
}
int t_exp_small(const double* x, double* out, long long n) {
    t_exp_small_kernel<<<blocks(n), THREADS>>>(x, out, n);
    return (int)cudaGetLastError();
}
int t_bracket(const double* u, double* out, long long n) {
    t_bracket_kernel<<<blocks(n), THREADS>>>(u, out, n);
    return (int)cudaGetLastError();
}
int t_accept(const double* x, const double* u, int8_t* gt, int8_t* ge, double* logu, long long n) {
    t_accept_kernel<<<blocks(n), THREADS>>>(x, u, gt, ge, logu, n);
    return (int)cudaGetLastError();
}
int t_normal(const double* u1, const uint32_t* bits, double* out, long long n) {
    t_normal_kernel<<<blocks(n), THREADS>>>(u1, bits, out, n);
    return (int)cudaGetLastError();
}
int t_normal_angles(double u1, double* z) {
    t_normal_angles_kernel<<<blocks(1ll << 24), THREADS>>>(u1, z);
    return (int)cudaGetLastError();
}
int t_lr_sum(const double* v, const long long* off, double* out, int n_seq) {
    t_lr_sum_kernel<<<(n_seq + 31) / 32, 32>>>(v, off, out, n_seq);
    return (int)cudaGetLastError();
}
int t_key(const double* x, unsigned long long* key, double* back, long long n) {
    t_key_kernel<<<blocks(n), THREADS>>>(x, key, back, n);
    return (int)cudaGetLastError();
}
int t_warp_sum(const double* v, const int* K, double* out, int n_warps) {
    t_warp_sum_kernel<<<blocks(32ll * n_warps), THREADS>>>(v, K, out, n_warps);
    return (int)cudaGetLastError();
}
}
#endif
