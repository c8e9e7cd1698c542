// Test harness for the fp64 primitives of the metric epilogue (taxi2_b200/csrc/common.cuh):
// rcp_full / div_by, sqrt_pos, log_pos and count_to_double, compiled with the library's own flags and
// compared on the device with the IEEE operations they stand in for (tests/test_gpu_metric_arithmetic.py).
// The sweeps count mismatches on the device and keep the first few offending inputs; mp_apply returns
// the primitive's results for a list of operands, for references that live on the host.
#include <cstdint>
#include <cuda_runtime.h>

#include "../taxi2_b200/csrc/common.cuh"

using namespace taxi;

namespace {

constexpr int KEEP = 8;   // offending inputs kept per check

struct Report {
    unsigned long long count[2];
    double first[2][KEEP][2];
};

__device__ void note(Report* r, int check, double x, double y)
{
    const unsigned long long k = atomicAdd(&r->count[check], 1ull);
    if (k < KEEP) { r->first[check][k][0] = x; r->first[check][k][1] = y; }
}

__device__ bool same_bits(double x, double y) { return __double_as_longlong(x) == __double_as_longlong(y); }

// block b - 1 takes divisor b; its threads stride over every dividend 0 <= a <= b.
// check 0: a / b, check 1: u = 1 - 4p/3 of p = a / b as metrics_from_counts forms it.
__global__ void div_sweep_kernel(Report* r)
{
    const double b = (double)(blockIdx.x + 1), rb = rcp_full(b);
    for (int a = threadIdx.x; a <= (int)blockIdx.x + 1; a += blockDim.x) {
        const double p = __ddiv_rn((double)a, b);
        if (!same_bits(div_by((double)a, b, rb), p)) note(r, 0, a, b);
        const double u = 1.0 - div_by(4.0 * p, 3.0, 1.0 / 3.0);
        if (!same_bits(u, 1.0 - __ddiv_rn(4.0 * p, 3.0))) note(r, 1, a, b);
    }
}

// block n - 1 takes n; every b = 1 - 2 tv / n > 0 formed as in metrics_from_counts
__global__ void sqrt_sweep_kernel(Report* r)
{
    const int n = blockIdx.x + 1;
    const double nd = (double)n, rn = rcp_full(nd);
    for (int tv = threadIdx.x; 2 * tv < n; tv += blockDim.x) {
        const double b = 1.0 - 2.0 * div_by((double)tv, nd, rn);
        if (!same_bits(sqrt_pos(b), __dsqrt_rn(b))) note(r, 0, tv, n);
    }
}

__global__ void count_sweep_kernel(Report* r)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < (1ll << 31); k += stride)
        if (!same_bits(count_to_double((int)k), __int2double_rn((int)k))) note(r, 0, (double)k, 0.0);
}

__global__ void apply_kernel(int op, const double* a, const double* b, double* out, long long n)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const double x = a[k];
    double y;
    switch (op) {
    case 0: y = div_by(x, b[k], rcp_full(b[k])); break;
    case 1: y = 1.0 - div_by(4.0 * x, 3.0, 1.0 / 3.0); break;
    case 2: y = sqrt_pos(x); break;
    default: y = log_pos(x); break;
    }
    out[k] = y;
}

template <class Launch>
int run_sweep(Launch launch, unsigned long long* count, double* first)
{
    Report* d = nullptr;
    Report h;
    cudaError_t e = cudaMalloc(&d, sizeof(Report));
    if (e == cudaSuccess) e = cudaMemset(d, 0, sizeof(Report));
    if (e == cudaSuccess) { launch(d); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaMemcpy(&h, d, sizeof(Report), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return (int)e;
    for (int c = 0; c < 2; ++c) {
        count[c] = h.count[c];
        for (int k = 0; k < KEEP; ++k) { first[(c * KEEP + k) * 2] = h.first[c][k][0]; first[(c * KEEP + k) * 2 + 1] = h.first[c][k][1]; }
    }
    return 0;
}

}  // namespace

extern "C" {

// every 0 <= a <= b <= b_max: count[0] = div_by(a, b, rcp_full(b)) != a / b,
// count[1] = 1 - div_by(4p, 3, 1/3) != 1 - 4p / 3 (p = a / b); first = (a, b) of the first KEEP of each
int mp_div_sweep(int b_max, unsigned long long* count, double* first)
{
    return run_sweep([&](Report* d) { div_sweep_kernel<<<b_max, 256>>>(d); }, count, first);
}

// every n <= n_max and tv < n / 2: count[0] = sqrt_pos(b) != sqrt(b), b = 1 - 2 (tv / n); first = (tv, n)
int mp_sqrt_sweep(int n_max, unsigned long long* count, double* first)
{
    return run_sweep([&](Report* d) { sqrt_sweep_kernel<<<n_max, 256>>>(d); }, count, first);
}

// every 0 <= k < 2^31: count[0] = count_to_double(k) != (double)k; first = (k, 0)
int mp_count_sweep(unsigned long long* count, double* first)
{
    return run_sweep([&](Report* d) { count_sweep_kernel<<<148 * 16, 256>>>(d); }, count, first);
}

// out[k] = op(a[k], b[k]): 0 = div_by(a, b, rcp_full(b)), 1 = 1 - div_by(4a, 3, 1/3), 2 = sqrt_pos(a), 3 = log_pos(a)
int mp_apply(int op, const double* a, const double* b, double* out, long long n)
{
    if (n <= 0) return 0;
    double *da = nullptr, *db = nullptr, *dout = nullptr;
    const size_t bytes = (size_t)n * sizeof(double);
    cudaError_t e = cudaMalloc(&da, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&db, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&dout, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(da, a, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(db, b ? b : a, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        apply_kernel<<<(unsigned)((n + 255) / 256), 256>>>(op, da, db, dout, n);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out, dout, bytes, cudaMemcpyDeviceToHost);
    cudaFree(da);
    cudaFree(db);
    cudaFree(dout);
    return (int)e;
}

}  // extern "C"
