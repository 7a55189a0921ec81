// e_sat throughput: abd::e_sat (piecewise polynomial on [230, 330) K) against abd::e_sat_goff (the formula), timed
// with CUDA events over n temperatures in [260, 280) K, each evaluated at T + 3.7 k, k = 0..7 (the range of the
// synthetic ocean fields): eight calls per 16 bytes of HBM traffic keep both versions bound by the FP64 pipe, not by
// memory.  The arrays (2 x 8 n bytes) are far larger than L2; a kernel that copies them gives the memory floor.  Also
// prints the largest relative difference of the two.
// build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o esat_probe esat_probe.cu
// run:   ./esat_probe [n = 2^27] [reps = 20]
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../aerobulk_b200/csrc/ab_device.cuh"

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s at %d\n", cudaGetErrorString(e), __LINE__); exit(1); } } while (0)

__global__ void fill(double *T, long long n)
{
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) T[i] = 260. + 20. * (double)((i * 2654435761ull) & 0xffffffull) * 0x1p-24;
}
template <int MODE>   // 0: copy, 1: e_sat_goff, 2: e_sat
__global__ void __launch_bounds__(256) run(const double *T, double *out, long long n)
{
    abm::load_tables();
    const long long i = blockIdx.x * 256ll + threadIdx.x;
    if (i >= n) return;
    const double t = T[i];
    double s = 0.;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += MODE == 0 ? t : MODE == 1 ? abd::e_sat_goff(t + 3.7 * k) : abd::e_sat(t + 3.7 * k);
    out[i] = s;
}
__global__ void maxrel(const double *a, const double *b, long long n, unsigned long long *worst)
{
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) atomicMax(worst, (unsigned long long)__double_as_longlong(fabs(a[i] - b[i]) / fabs(b[i])));
}

template <int MODE>
static float time_ms(const double *T, double *out, long long n, int reps)
{
    const unsigned blocks = (unsigned)((n + 255) / 256);
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    run<MODE><<<blocks, 256>>>(T, out, n);   // warm-up
    CK(cudaEventRecord(e0));
    for (int r = 0; r < reps; ++r) run<MODE><<<blocks, 256>>>(T, out, n);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    return ms / reps;
}

int main(int argc, char **argv)
{
    const long long n = argc > 1 ? atoll(argv[1]) : (1ll << 27);
    const int reps = argc > 2 ? atoi(argv[2]) : 20;
    double *T, *a, *b;
    unsigned long long *worst;
    CK(cudaMalloc(&T, n * 8));
    CK(cudaMalloc(&a, n * 8));
    CK(cudaMalloc(&b, n * 8));
    CK(cudaMalloc(&worst, 8));
    CK(cudaMemset(worst, 0, 8));
    fill<<<(unsigned)((n + 255) / 256), 256>>>(T, n);
    CK(cudaGetLastError());
    const float copy = time_ms<0>(T, a, n, reps);
    const float goff = time_ms<1>(T, a, n, reps);
    const float table = time_ms<2>(T, b, n, reps);
    maxrel<<<(unsigned)((n + 255) / 256), 256>>>(b, a, n, worst);
    unsigned long long w;
    CK(cudaMemcpy(&w, worst, 8, cudaMemcpyDeviceToHost));
    double wd;
    memcpy(&wd, &w, 8);
    printf("n %lld, %d reps: copy %.3f ms | e_sat_goff %.3f ms (%.2f G calls/s) | e_sat %.3f ms (%.2f G calls/s) | speed-up %.2fx"
           " | max rel diff %.2e\n", n, reps, copy, goff, 8 * n / goff / 1e6, table, 8 * n / table / 1e6, goff / table, wd);
    return 0;
}
