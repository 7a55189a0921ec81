// Unstable psi throughput: the tables (abd::psi_mh_table, ab_math.cuh) against the formulas (abd::psi_mh_coare_formula, abd::psi_mh_ncar_unstable) for the
// COARE pair and the Paulson pair (NCAR's rounding), timed with CUDA events over n arguments zeta = -25 * 2^(-20 v), v
// uniform in [0, 1) per lane (|zeta| from 2.4e-5 to 25, neighbouring lanes on unrelated rows: the bank-conflict worst
// case), each evaluated at zeta (1 + k/8), k = 0..7: eight pairs per 16 bytes of HBM traffic keep every version bound by
// the FP64 pipe, not by memory.  The arrays (2 x 8 n bytes) are far larger than L2; a kernel that copies them gives the
// memory floor.  Also prints the largest |table - formula| / max(|formula|, 1) of the summed pairs.
// build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o psi_probe psi_probe.cu
// run:   ./psi_probe [n = 2^27] [reps = 20]
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../aerobulk_b200/csrc/ab_device.cuh"

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s at %d\n", cudaGetErrorString(e), __LINE__); exit(1); } } while (0)

__global__ void fill(double *Z, long long n)
{
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) Z[i] = -25. * exp2(-20. * (double)((i * 2654435761ull) & 0xffffffull) * 0x1p-24);
}
// 0: copy, 1: COARE formula, 2: COARE table, 3: Paulson formula, 4: Paulson table
template <int MODE>
__global__ void __launch_bounds__(256) run(const double *Z, double *out, long long n)
{
    abm::load_tables<MODE == 2 ? abm::PSI_TABLES_COARE : MODE == 4 ? abm::PSI_TABLES_PAULSON : abm::PSI_TABLES_NONE>();
    const long long i = blockIdx.x * 256ll + threadIdx.x;
    if (i >= n) return;
    const double t = Z[i];
    double s = 0.;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const double z = t * (1. + 0.125 * k);
        abd::PsiMH r = {z, 0.};
        if (MODE == 1) r = abd::psi_mh_coare_formula(z);
        if (MODE == 2) r = abd::psi_mh_table<abm::PSI_TABLES_COARE>(z);
        if (MODE == 3) r = abd::psi_mh_ncar_unstable(z);
        if (MODE == 4) r = abd::psi_mh_table<abm::PSI_TABLES_PAULSON>(z);
        s += r.m + r.h;
    }
    out[i] = s;
}
__global__ void maxdiff(const double *a, const double *b, long long n, unsigned long long *worst)
{
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) atomicMax(worst, (unsigned long long)__double_as_longlong(fabs(a[i] - b[i]) / fmax(fabs(b[i]), 1.)));
}

template <int MODE>
static float time_ms(const double *Z, double *out, long long n, int reps)
{
    const unsigned blocks = (unsigned)((n + 255) / 256);
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    run<MODE><<<blocks, 256>>>(Z, out, n);   // warm-up
    CK(cudaEventRecord(e0));
    for (int r = 0; r < reps; ++r) run<MODE><<<blocks, 256>>>(Z, out, n);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    CK(cudaEventDestroy(e0));
    CK(cudaEventDestroy(e1));
    return ms / reps;
}

static double worst_diff(const double *a, const double *b, long long n, unsigned long long *w_dev)
{
    CK(cudaMemset(w_dev, 0, 8));
    maxdiff<<<(unsigned)((n + 255) / 256), 256>>>(a, b, n, w_dev);
    unsigned long long w;
    CK(cudaMemcpy(&w, w_dev, 8, cudaMemcpyDeviceToHost));
    double wd;
    memcpy(&wd, &w, 8);
    return wd;
}

int main(int argc, char **argv)
{
    const long long n = argc > 1 ? atoll(argv[1]) : (1ll << 27);
    const int reps = argc > 2 ? atoi(argv[2]) : 20;
    double *Z, *a, *b;
    unsigned long long *w;
    CK(cudaMalloc(&Z, n * 8));
    CK(cudaMalloc(&a, n * 8));
    CK(cudaMalloc(&b, n * 8));
    CK(cudaMalloc(&w, 8));
    fill<<<(unsigned)((n + 255) / 256), 256>>>(Z, n);
    CK(cudaGetLastError());
    const float copy = time_ms<0>(Z, a, n, reps);
    const float cf = time_ms<1>(Z, a, n, reps);
    const float ct = time_ms<2>(Z, b, n, reps);
    const double cd = worst_diff(b, a, n, w);
    const float pf = time_ms<3>(Z, a, n, reps);
    const float pt = time_ms<4>(Z, b, n, reps);
    const double pd = worst_diff(b, a, n, w);
    printf("n %lld, %d reps, 8 pairs per argument: copy %.3f ms\n", n, reps, copy);
    printf("  COARE   formula %.3f ms (%.2f G pairs/s) | table %.3f ms (%.2f G pairs/s) | speed-up %.2fx | max diff %.2e\n",
           cf, 8 * n / cf / 1e6, ct, 8 * n / ct / 1e6, cf / ct, cd);
    printf("  Paulson formula %.3f ms (%.2f G pairs/s) | table %.3f ms (%.2f G pairs/s) | speed-up %.2fx | max diff %.2e\n",
           pf, 8 * n / pf / 1e6, pt, 8 * n / pt / 1e6, pf / pt, pd);
    CK(cudaFree(Z));
    CK(cudaFree(a));
    CK(cudaFree(b));
    CK(cudaFree(w));
    return 0;
}
