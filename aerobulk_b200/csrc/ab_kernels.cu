// ab_kernels.cu -- hand-written FP64 CUDA kernels for sm_100a.
//
//   flux_kernel<ALGO,SKIN,ZTEQ>  one thread per grid point: humidity conversion, scalar
//       wind, ssq, theta(zt), the nb_iter Monin-Obukhov iteration of one of the five bulk
//       algorithms (with cool-skin / warm-layer when SKIN), bulk formula and wind-stress
//       vector -- reference src/mod_aerobulk_compute.f90:22-213 fused into one launch.
//       All iteration state lives in registers; global memory is touched once per field
//       (6-8 coalesced 8-byte loads, 5-6 stores, 1-4 state words R+W).
//   classify_kernel              stability sort inside 2048-point windows (FP32 proxy, warp-scan prefix): whole thread
//       blocks of flux_kernel see one stability class.
//   stats_fast_kernel / stats_fix_kernel / stats_final   the field statistics AEROBULK_INIT needs
//       (src/mod_aerobulk.f90:104-153): mask, per-field masked sum/min/max, raw min/max; init_decide_kernel judges them
//       on the device (humidity type, unit checks) for asynchronous jt == 1 calls.
//   dfma_peak_kernel             dependent-chain DFMA microbenchmark (FP64 roofline denominator).
//   flux_io_kernel<T,ALGO,SKIN,ZTEQ>, classify_io_kernel<T>, stats_fast_io_kernel<T>, stats_fix_io_kernel<T>
//       the same for per-point arrays of element type T (float: aerobulk_gpu_model*_f32): the body is shared, only the
//       loads (widened exactly) and stores (rounded once to nearest) differ, and the arithmetic stays FP64.  The shared
//       bodies take threadIdx.x from the kernel: read in a __device__ function it would lose the range the kernel's
//       launch bounds give it, and the FP64 kernels' machine code would change.
//
// The path is FP64-pipe bound (no contraction -> no tensor cores): see DESIGN.md.
#include "ab_kernels.cuh"

#include <float.h>
#include <stdint.h>

namespace abk {

using namespace abd;

#ifndef AB_FLUX_BLOCK
#define AB_FLUX_BLOCK 256
#endif
// Resident blocks per SM (x 256 threads).  Skin kernels: 3 (24 warps/SM, <= 85 registers: the ~28 doubles they carry across
// the bulk iteration do not fit 64 registers without spilling into the loop).  Kernels without skin: 4 (32 warps/SM, 64
// registers; their few spills sit outside the loop).  Measured at 4320x2160 (profiles/exp_variants_r02i.txt, 256x3 ->
// 256x4): NCAR 0.900 -> 0.877 ms, ANDREAS 1.372 -> 1.322, COARE 3.6 1.900 -> 1.842; COARE 3.6 + skin 3.147 -> 3.204 (night),
// ECMWF + skin 4.126 -> 4.226.  128 x 7 (73 registers) loses everywhere but ANDREAS.
#ifndef AB_MIN_BLOCKS
#define AB_MIN_BLOCKS 3
#endif
#ifndef AB_MIN_BLOCKS_NOSKIN
#define AB_MIN_BLOCKS_NOSKIN 4
#endif
static constexpr int FLUX_BLOCK = AB_FLUX_BLOCK;

// Cheap proxy of the air-sea virtual potential temperature difference [K], whose sign is the stability class every
// psi_m / psi_h evaluation branches on.  Only used to GROUP points (performance); the physics never sees it.
// `skin_off`: what the skin schemes will do to the surface temperature before the first psi is evaluated (T_s starts at
// sst - 0.25 K, mod_blk_coare3p6.f90:254; plus the warm-layer increment carried from the previous step).
// |proxy| below the band [K]: class "uncertain" (own group, between the two sure ones).  Measured on B200 at 4320x2160
// (profiles/exp_sort_r02d.txt; band 0 / 0.1 / 0.25 / 0.5): COARE 3.6 2.146 / 2.080 / 2.099 / 2.136 ms, ECMWF 2.318 /
// 2.233 / 2.248 / 2.306 ms, COARE 3.6 + skin by day 4.495 / 4.459 / 4.411 / 4.377 ms and by night 3.635 / 3.538 / 3.449 /
// 3.419 ms, ECMWF + skin 4.731 / 4.631 / 4.555 / 4.535 ms: the skin schemes move T_s by a few tenths of a kelvin more.
#ifndef AB_SORT_BAND
#define AB_SORT_BAND 0.15
#endif
#ifndef AB_SORT_BAND_SKIN
#define AB_SORT_BAND_SKIN 0.5
#endif
#ifndef AB_SORT_BAND_NOQ
#define AB_SORT_BAND_NOQ 1.0 // the same when the humidity is rh / dp (the proxy ignores it)
#endif
// Per-point arrays of element type T (FluxArgs, StatsArgs): `ld` widens to FP64 (exact for float), `st` rounds once to
// nearest.  With T = double both are the plain load and store.
template <class T>
__device__ __forceinline__ double ld(const void *p, long long i) { return (double)__ldg(static_cast<const T *>(p) + i); }
template <class T>
__device__ __forceinline__ void st(void *p, long long i, double v) { static_cast<T *>(p)[i] = v; }
template <>
__device__ __forceinline__ void st<float>(void *p, long long i, double v) { static_cast<float *>(p)[i] = __double2float_rn(v); }

// The proxy only groups points, so it runs in FP32 (FP32 pipe and MUFU, both idle in this FP64 path): the temperature
// difference is taken in FP64 first (exact to 1e-13 K), the humidity correction 0.608 (T_a q - T_s q_s) ~ 1 K is good to
// 1e-6 K in FP32 -- against a band of 0.15 K.  classify_kernel is then bound by its 34 bytes per point.
template <class T>
__device__ __forceinline__ float stability_proxy(const FluxArgs &a, int ihum, double skin_off, long long i)
{
    const double sst = ld<T>(a.sst, i) + skin_off, ta = ld<T>(a.t_zt, i) + RGAMMA_DRY * a.u.zt;
    const float d0 = (float)(ta - sst);
    if (ihum != 0) return d0;
    const float q = (float)ld<T>(a.hum_zt, i), p = (float)ld<T>(a.slp, i);
    const float tc = (float)(sst - 273.15);
    const float es = 611.2f * __expf(17.67f * tc * __frcp_rn(tc + 243.5f));     // Magnus
    const float qs = 0.98f * 0.622f * es * __frcp_rn(p - 0.378f * es);
    return d0 + 0.608f * ((float)ta * q - (float)sst * qs);
}

// ---------------------------------------------------------------------------
// classify_kernel: stability sort inside windows of SORT_WIN consecutive points.
// The iteration branches on the stability class in every psi function (and the two sides differ a lot in cost); where
// stability is not spatially coherent a warp would execute both sides (23/32 active lanes in the round-1 profile).
// One block per window writes perm[] such that the window's slots hold, in this order, its surely-stable points, the
// uncertain ones (|proxy| < band: a misjudged point makes its whole warp run both sides, so the doubtful ones are kept
// to themselves) and the surely-unstable ones; flux_kernel then runs 256 consecutive SLOTS per block, so that all but two
// blocks per window are homogeneous -- and a homogeneous block retires as a whole (sorting inside a block left its fast
// warps idle behind the slow ones and was slower).  Accesses stay inside the window's 16 KB of each field.
// ---------------------------------------------------------------------------
static constexpr int SORT_WIN = 2048;
static constexpr int SORT_BLOCK = 256;
static constexpr int SORT_ITEMS = SORT_WIN / SORT_BLOCK;
static constexpr int SORT_CLASSES = 3;

template <class T>
__device__ __forceinline__ void classify_block(const FluxArgs &a, unsigned short *perm, int skin, int tid)
{
    constexpr int NW = SORT_BLOCK / 32, NG = SORT_ITEMS * NW;
    __shared__ unsigned short s_c[SORT_CLASSES][NG], s_off[SORT_CLASSES][NG];
    __shared__ int s_tot[SORT_CLASSES];
    const long long base = (long long)blockIdx.x * SORT_WIN;
    const int lane = tid & 31, w = tid >> 5;
    const int ihum = a.init_dev ? __ldg(a.init_dev) : a.ihum;
    const float band = (ihum != 0) ? (float)AB_SORT_BAND_NOQ : (skin ? (float)AB_SORT_BAND_SKIN : (float)AB_SORT_BAND);
    const bool wl = skin && !a.first_step && a.dT_wl != nullptr;
    int cls[SORT_ITEMS];
#pragma unroll
    for (int k = 0; k < SORT_ITEMS; ++k) {
        const long long i = base + k * SORT_BLOCK + tid;
        cls[k] = SORT_CLASSES;   // padding beyond n
        if (i < a.n) {
            const double off = skin ? (-0.25 + (wl ? a.dT_wl[i] : 0.)) : 0.;
            const float d = stability_proxy<T>(a, ihum, off, i);
            cls[k] = (d >= band) ? 0 : (d > -band) ? 1 : 2;
        }
    }
    // (the votes in a loop of their own: all 8 x 4 loads of a thread are in flight together)
    // group (k, w) = the 32 items warp w holds in round k, in item order g = k NW + w; per group and class: the count
    // (shared), and per thread its rank among the lanes of its class (`rank`) and among all real points (`real_rank`)
    const unsigned lt = (1u << lane) - 1u;
    int rank[SORT_ITEMS], real_rank[SORT_ITEMS];
#pragma unroll
    for (int k = 0; k < SORT_ITEMS; ++k) {
        unsigned any = 0u;
        rank[k] = 0;
#pragma unroll
        for (int c = 0; c < SORT_CLASSES; ++c) {
            const unsigned b = __ballot_sync(0xffffffffu, cls[k] == c);
            if (lane == 0) s_c[c][k * NW + w] = (unsigned short)__popc(b);
            if (cls[k] == c) rank[k] = __popc(b & lt);
            any |= b;
        }
        real_rank[k] = __popc(any & lt);
    }
    __syncthreads();
    // exclusive prefix of the counts over the NG = 64 groups, one warp per class (two groups per lane)
    static_assert(NG == 64 && SORT_CLASSES * 32 <= SORT_BLOCK, "prefix layout");
    if (w < SORT_CLASSES) {
        const int a0 = s_c[w][2 * lane], a1 = s_c[w][2 * lane + 1];
        int incl = a0 + a1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        const int excl = incl - (a0 + a1);
        s_off[w][2 * lane] = (unsigned short)excl;
        s_off[w][2 * lane + 1] = (unsigned short)(excl + a0);
        if (lane == 31) s_tot[w] = incl;
    }
    __syncthreads();
    const int tot0 = s_tot[0], tot1 = s_tot[1], tot2 = s_tot[2];
#pragma unroll
    for (int k = 0; k < SORT_ITEMS; ++k) {
        const int g = k * NW + w, item = k * SORT_BLOCK + tid;
        int slot;
        if (cls[k] < SORT_CLASSES) {
            const int before = (cls[k] > 0 ? tot0 : 0) + (cls[k] > 1 ? tot1 : 0);
            slot = before + s_off[cls[k]][g] + rank[k];
        } else {
            // padding: after all real points, in item order (item - number of real items before it)
            const int real_before = s_off[0][g] + s_off[1][g] + s_off[2][g] + real_rank[k];
            slot = tot0 + tot1 + tot2 + (item - real_before);
        }
        perm[base + slot] = (unsigned short)item;
    }
}

__global__ void __launch_bounds__(SORT_BLOCK) classify_kernel(const FluxArgs a, unsigned short *perm, int skin)
{
    classify_block<double>(a, perm, skin, threadIdx.x);
}

// the same for arrays of element type T
template <class T>
__global__ void __launch_bounds__(SORT_BLOCK) classify_io_kernel(const FluxArgs a, unsigned short *perm, int skin)
{
    classify_block<T>(a, perm, skin, threadIdx.x);
}

// warm-layer state of point i at the start of a step (*_INIT values at kt == nit000), and its write-back
template <int ALGO, class Args>
__device__ __forceinline__ void load_warm_layer(const Args &a, long long i, WarmLayer &wl)
{
    if (ALGO == ECMWF) {
        wl.Hz = 3.;                                            // rd0, mod_skin_ecmwf.f90:57 (constant)
        wl.dT = a.first_step ? 0. : a.dT_wl[i];
    } else if (a.first_step) {
        wl.Hz = 20.;                                           // Hwl_max, mod_blk_coare3p6.f90:84-87
    } else {
        wl.dT = a.dT_wl[i];
        wl.Hz = a.Hz_wl[i];
        wl.Qac = a.Qnt_ac[i];
        wl.Tac = a.Tau_ac[i];
    }
}
template <int ALGO, class Args>
__device__ __forceinline__ void store_warm_layer(const Args &a, long long i, const WarmLayer &wl)
{
    a.dT_wl[i] = wl.dT;
    if (ALGO != ECMWF) {
        a.Hz_wl[i] = wl.Hz;
        a.Qnt_ac[i] = wl.Qac;
        a.Tau_ac[i] = wl.Tac;
    }
}

// one thread's point of flux_kernel (T = double) and flux_io_kernel<T>: only the loads and stores depend on T
template <class T, int ALGO, bool SKIN, bool ZTEQ>
__device__ __forceinline__ void flux_point(const FluxArgs &a, unsigned tid)
{
    abm::load_tables();
    long long i = (long long)blockIdx.x * FLUX_BLOCK + tid;
    if (a.perm) i = (i / SORT_WIN) * SORT_WIN + a.perm[i];   // slot -> point (perm is padded to whole windows)
    if (i >= a.n) return;
    int ihum = a.ihum;
    if (a.init_dev) {   // asynchronous AEROBULK_INIT: its verdict is on the device, the host has not seen it yet
        if (__ldg(a.init_dev + 1) != 0) return;   // the reference would have stopped: nothing is computed
        ihum = __ldg(a.init_dev);
    }

    // ---- coalesced loads of the 6 (8) input fields
    const double sst = ld<T>(a.sst, i);
    const double t_air = ld<T>(a.t_zt, i);
    const double hum = ld<T>(a.hum_zt, i);
    const double U = ld<T>(a.U_zu, i);
    const double V = ld<T>(a.V_zu, i);
    const double slp = ld<T>(a.slp, i);

    PointIn p;
    p.sst = sst;
    p.slp = slp;
    // humidity -> specific humidity (mod_aerobulk_compute.f90:99-108); slp floored at 5e4 Pa by the caller
    if (ihum == 0) p.q_zt = hum;
    else if (ihum == 1) p.q_zt = q_air_dp(hum, abm::dmax(slp, 50000.));
    else p.q_zt = q_air_rh(hum, t_air, abm::dmax(slp, 50000.));
    // :111 -- no FMA contraction here: U*U+V*V must not depend on the order of the components
    p.wnd = sqrt(__dadd_rn(__dmul_rn(U, U), __dmul_rn(V, V)));
    p.ssq = RDCT_QSAT_SALT * q_sat(sst, slp);                      // :114
    p.theta_zt = theta_from_z_P0_T_q(a.u.zt, slp, t_air, p.q_zt);  // :118
    p.Qsw = 0.;
    p.rlw = 0.;
    p.lon = 0.;
    p.has_lon = false;

    WarmLayer wl = {0., 0., 0., 0.};
    if (SKIN) {
        p.Qsw = (1. - ROCE_ALB0) * ld<T>(a.rad_sw, i);             // :135,:146,:161
        p.rlw = ld<T>(a.rad_lw, i);
        if (a.lon) {
            p.lon = __ldg(a.lon + i);
            p.has_lon = true;
        }
        load_warm_layer<ALGO>(a, i, wl);
    }

    Diag dg;   // optional TURB_* outputs: unused here, eliminated by the compiler
    const Coeffs c = solve_ocean<ALGO, SKIN, SKIN, ZTEQ>(a.u, p, wl, dg);
    if (SKIN) store_warm_layer<ALGO>(a, i, wl);

    // ---- flux assembly (BULK_FORMULA, :184-185) and stress vector (:189-194)
    const Flux f = bulk_formula(air_at_zu(a.u.zu, c.t_zu, c.q_zu, slp), c.Ts, c.qs, c.t_zu, c.q_zu, c.Cd, c.Ch, c.Ce, p.wnd, c.Ub);
    if (f.tau > REF_TAU_MAX) atomicMin(a.bad_index, (unsigned long long)(a.index_offset + i));

    double tx = 0., ty = 0.;
    if (p.wnd > 1.E-3) {
        const double s = f.tau / p.wnd;
        tx = s * U;
        ty = s * V;
    }
    st<T>(a.QL, i, f.qlat);
    st<T>(a.QH, i, f.qsen);
    st<T>(a.Tau_x, i, tx);
    st<T>(a.Tau_y, i, ty);
    st<T>(a.Evap, i, f.evap);
    if (a.T_s) st<T>(a.T_s, i, c.Ts);
}

template <int ALGO, bool SKIN, bool ZTEQ>
__global__ void __launch_bounds__(FLUX_BLOCK, SKIN ? AB_MIN_BLOCKS : AB_MIN_BLOCKS_NOSKIN) flux_kernel(const FluxArgs a)
{
    flux_point<double, ALGO, SKIN, ZTEQ>(a, threadIdx.x);
}

// flux_kernel on per-point arrays of element type T, same launch bounds.  T is a type argument: the kernel-matrix
// census of the FP64 kernels takes the instantiations whose template arguments are all int or bool.
template <class T, int ALGO, bool SKIN, bool ZTEQ>
__global__ void __launch_bounds__(FLUX_BLOCK, SKIN ? AB_MIN_BLOCKS : AB_MIN_BLOCKS_NOSKIN) flux_io_kernel(const FluxArgs a)
{
    flux_point<T, ALGO, SKIN, ZTEQ>(a, threadIdx.x);
}

static auto flux_kernel_for(int algo, bool skin, bool zteq, size_t elem = ELEM_F64)
{
    return pick_ocean(algo, skin, zteq, [elem](auto A, auto S, auto Z) {
        return elem == ELEM_F64 ? flux_kernel<A(), S(), Z()> : elem == ELEM_F32 ? flux_io_kernel<float, A(), S(), Z()> : nullptr;
    });
}

cudaError_t launch_flux(int algo, bool skin, bool zteq, size_t elem, const FluxArgs &a, cudaStream_t s)
{
    const auto k = flux_kernel_for(algo, skin, zteq, elem);
    if (!k) return cudaErrorInvalidValue;
    if (a.n <= 0) return cudaSuccess;
    const long long span = a.perm ? (a.n + SORT_WIN - 1) / SORT_WIN * SORT_WIN : a.n;   // whole windows of slots
    k<<<(unsigned)((span + FLUX_BLOCK - 1) / FLUX_BLOCK), FLUX_BLOCK, 0, s>>>(a);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// turb_kernel<ALGO,CS,WL,ZTEQ>: the direct TURB_* entry (SURVEY.md 8f row 1) on the same solvers
// ---------------------------------------------------------------------------
template <int ALGO, bool CS, bool WL, bool ZTEQ>
__global__ void __launch_bounds__(FLUX_BLOCK, (CS || WL) ? AB_MIN_BLOCKS : AB_MIN_BLOCKS_NOSKIN) turb_kernel(const TurbArgs a)
{
    abm::load_tables();
    const long long i = (long long)blockIdx.x * FLUX_BLOCK + threadIdx.x;
    if (i >= a.n) return;
    constexpr bool SKIN = CS || WL;
    PointIn p;
    p.sst = a.T_s[i];
    p.ssq = a.q_s[i];
    p.theta_zt = __ldg(a.t_zt + i);
    p.q_zt = __ldg(a.q_zt + i);
    p.wnd = __ldg(a.U_zu + i);
    p.slp = 0.;
    p.Qsw = 0.;
    p.rlw = 0.;
    p.lon = 0.;
    p.has_lon = false;
    WarmLayer wl = {0., 0., 0., 0.};
    if (SKIN) {
        p.Qsw = __ldg(a.Qsw + i);
        p.rlw = __ldg(a.rad_lw + i);
        p.slp = __ldg(a.slp + i);
        if (a.lon) {
            p.lon = __ldg(a.lon + i);
            p.has_lon = true;
        }
    }
    if (WL) load_warm_layer<ALGO>(a, i, wl);
    Diag dg;
    const Coeffs c = solve_ocean<ALGO, CS, WL, ZTEQ>(a.u, p, wl, dg);
    if (WL) store_warm_layer<ALGO>(a, i, wl);
    if (SKIN) {
        a.T_s[i] = c.Ts;
        a.q_s[i] = c.qs;
    }
    a.Cd[i] = c.Cd; a.Ch[i] = c.Ch; a.Ce[i] = c.Ce;
    a.t_zu[i] = c.t_zu; a.q_zu[i] = c.q_zu; a.Ubzu[i] = c.Ub;
    if (a.opt[0]) a.opt[0][i] = dg.CdN;
    if (a.opt[1]) a.opt[1][i] = dg.ChN;
    if (a.opt[2]) a.opt[2][i] = dg.CeN;
    if (a.opt[3]) a.opt[3][i] = dg.z0;
    if (a.opt[4]) a.opt[4][i] = dg.us;
    if (a.opt[5]) a.opt[5][i] = dg.L;
    if (a.opt[6]) a.opt[6][i] = dg.UN10;
    if (CS && a.opt[7]) a.opt[7][i] = dg.dT_cs;
    if (WL && a.opt[8]) a.opt[8][i] = wl.dT;
    if (WL && a.opt[9]) a.opt[9][i] = wl.Hz;
}

// cool skin and warm layer are separate options here; NCAR and ANDREAS take neither
cudaError_t launch_turb(int algo, bool cs, bool wl, bool zteq, const TurbArgs &a, cudaStream_t s)
{
    const auto k = pick_ocean(algo, cs || wl, zteq, [cs, wl](auto A, auto S, auto Z) {
        if constexpr (!S()) return turb_kernel<A(), false, false, Z()>;
        else return cs ? (wl ? turb_kernel<A(), true, true, Z()> : turb_kernel<A(), true, false, Z()>)
                       : turb_kernel<A(), false, true, Z()>;
    });
    if (!k) return cudaErrorInvalidValue;
    if (a.n <= 0) return cudaSuccess;
    k<<<(unsigned)((a.n + FLUX_BLOCK - 1) / FLUX_BLOCK), FLUX_BLOCK, 0, s>>>(a);
    return cudaGetLastError();
}

int flux_block_size() { return FLUX_BLOCK; }

int sort_window() { return SORT_WIN; }

cudaError_t launch_classify(size_t elem, const FluxArgs &a, unsigned short *perm, bool skin, cudaStream_t s)
{
    const auto k = elem == ELEM_F64 ? classify_kernel : elem == ELEM_F32 ? classify_io_kernel<float> : nullptr;
    if (!k) return cudaErrorInvalidValue;
    if (a.n <= 0) return cudaSuccess;
    const long long nwin = (a.n + SORT_WIN - 1) / SORT_WIN;
    k<<<(unsigned)nwin, SORT_BLOCK, 0, s>>>(a, perm, skin ? 1 : 0);
    return cudaGetLastError();
}

cudaError_t flux_kernel_attributes(int algo, bool skin, bool zteq, cudaFuncAttributes *attr, int *blocks_per_sm)
{
    const auto k = flux_kernel_for(algo, skin, zteq);
    if (!k) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncGetAttributes(attr, k);
    if (e != cudaSuccess || !blocks_per_sm) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, k, FLUX_BLOCK, 0);
}

// ---------------------------------------------------------------------------
// AEROBULK_INIT statistics (src/mod_aerobulk.f90:104-153, src/mod_phymbl.f90:1851-2007)
// ---------------------------------------------------------------------------
static constexpr int STATS_BLOCK = 256;
static constexpr int STATS_MAX_BLOCKS = 148 * 8;   // x 256 threads: enough warps to hide the 7 loads per point (HBM-bound pass)

// sanity ranges, src/mod_const.f90:138-146
__device__ __forceinline__ bool point_unmasked(double sst, double ta, double slp, double wnd, bool rad, double rlw)
{
    bool m = true;
    if (sst < 270. || sst > 320.) m = false;
    if (ta < 180. || ta > 330.) m = false;
    if (slp < 80000. || slp > 110000.) m = false;
    if (wnd > 50.) m = false;
    if (rad) {
        if (rlw < 0. || rlw > 1500.) m = false;   // prsw=rad_lw (mod_aerobulk.f90:248): rad_lw vs the SW range
        if (rlw < 0. || rlw > 750.) m = false;
    }
    return m;
}

__device__ __forceinline__ double warp_reduce(double v, int op)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double w = __shfl_down_sync(0xffffffffu, v, o);
        v = (op == 0) ? v + w : (op == 1) ? fmin(v, w) : fmax(v, w);
    }
    return v;
}

__host__ __device__ inline int stat_op(int k)   // 0 sum, 1 min, 2 max
{
    if (k < 2) return 0;
    const int r = (k - 2) % 5;
    if (k >= 2 + 5 * NFIELDS) return 0;
    return (r == 0) ? 0 : (r == 1 || r == 3) ? 1 : 2;
}

// Slot of a block's partials row that tells stats_fix_kernel to redo the block (rows have NSTATS = 64 slots, 47 used).
static constexpr int STATS_REDO_SLOT = NSTATS - 1;

// stats_fast_kernel: the pass every jt == 1 call pays.  Where no point of a block is masked -- the normal case: the mask
// only removes values outside the sanity ranges of mod_const.f90:138-146 -- the masked statistics ARE the raw ones, so the
// fast pass keeps sum / min / max per field (27 accumulators instead of 47, no per-point mask tests) and derives "was any
// point of this block masked?" from the block's own raw minima and maxima at the end.  A block that may hold a masked
// point raises its redo flag and stats_fix_kernel recomputes that block's row with the full accumulator set (same points,
// same order: the row is bit-identical to what the one-kernel version produced).  NaNs: `x < lo || x > hi` is false for a
// NaN (the reference does not mask it) and the (v < acc ? v : acc) min / max skip it -- the derived test agrees.
// rad_lw is held against both radiation ranges (the reference's prsw=rad_lw slip): fields 7 and 8 are the same values.
template <class T, int UNROLL>
__device__ __forceinline__ void stats_fast_body(const StatsArgs &a, double (&sum)[8], double (&mn)[8], double (&mx)[8], double &cnt)
{
    const bool rad = (a.rad_lw != nullptr);
    const long long stride = (long long)gridDim.x * STATS_BLOCK;
    // UNROLL points per trip with all their loads issued first; a thread meets its points (base + k stride) in the same
    // order as in stats_fix_kernel whatever the unroll factor: the sums add up identically
    for (long long i0 = (long long)blockIdx.x * STATS_BLOCK + threadIdx.x; i0 < a.n; i0 += stride * UNROLL) {
        double in[UNROLL][7];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const long long i = i0 + u * stride;
            const long long j = (i < a.n) ? i : i0;
            in[u][0] = ld<T>(a.sst, j);
            in[u][1] = ld<T>(a.t_zt, j);
            in[u][2] = ld<T>(a.slp, j);
            in[u][3] = ld<T>(a.U_zu, j);
            in[u][4] = ld<T>(a.V_zu, j);
            in[u][5] = ld<T>(a.hum_zt, j);
            in[u][6] = rad ? ld<T>(a.rad_lw, j) : 0.;
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            if (i0 + u * stride >= a.n) break;
            double v[8];
            v[0] = in[u][0];
            v[1] = in[u][1];
            v[2] = in[u][2];
            v[3] = in[u][3];
            v[4] = in[u][4];
            v[5] = sqrt(__dadd_rn(__dmul_rn(v[3], v[3]), __dmul_rn(v[4], v[4])));
            v[6] = in[u][5];
            v[7] = in[u][6];
            cnt += 1.;
#pragma unroll
            for (int f = 0; f < 8; ++f) {
                sum[f] += v[f];
                mn[f] = abm::dmin(v[f], mn[f]);
                mx[f] = abm::dmax(v[f], mx[f]);
            }
        }
    }
}

#ifndef AB_STATS_UNROLL
#define AB_STATS_UNROLL 3   // 120 registers, no spills, 2 blocks/SM x 21 loads in flight per thread
#endif
template <class T>
__device__ __forceinline__ void stats_fast_block(const StatsArgs &a, unsigned tid)
{
    double sum[8], mn[8], mx[8], cnt = 0.;
#pragma unroll
    for (int f = 0; f < 8; ++f) {
        sum[f] = 0.;
        mn[f] = DBL_MAX;
        mx[f] = -DBL_MAX;
    }
    stats_fast_body<T, AB_STATS_UNROLL>(a, sum, mn, mx, cnt);   // a thread meets its points in the same order for any unroll
    // block reduction in the order of the one-kernel version: lanes by shuffle, then the warps in index order
    __shared__ double sm[STATS_BLOCK / 32][1 + 3 * 8];
    const int lane = tid & 31, warp = tid >> 5;
    {
        const double r = warp_reduce(cnt, 0);
        if (lane == 0) sm[warp][0] = r;
    }
#pragma unroll
    for (int f = 0; f < 8; ++f) {
        const double s = warp_reduce(sum[f], 0), lo = warp_reduce(mn[f], 1), hi = warp_reduce(mx[f], 2);
        if (lane == 0) {
            sm[warp][1 + 3 * f + 0] = s;
            sm[warp][1 + 3 * f + 1] = lo;
            sm[warp][1 + 3 * f + 2] = hi;
        }
    }
    __syncthreads();
    double *row = a.partials + (long long)blockIdx.x * NSTATS;
    if (tid < 1 + 3 * 8) {
        const int k = tid, op = (k == 0) ? 0 : (k - 1) % 3;
        double r = sm[0][k];
        for (int w = 1; w < STATS_BLOCK / 32; ++w)
            r = (op == 0) ? r + sm[w][k] : (op == 1) ? fmin(r, sm[w][k]) : fmax(r, sm[w][k]);
        sm[0][k] = r;
    }
    __syncthreads();
    if (tid == 0) {
        const double *b = sm[0];
        const bool rad = (a.rad_lw != nullptr);
        // min / max of field f: b[2 + 3 f], b[3 + 3 f]; field order sst t_zt slp U V wnd hum rad_lw
        bool masked = b[2] < 270. || b[3] > 320. || b[5] < 180. || b[6] > 330. || b[8] < 80000. || b[9] > 110000. || b[18] > 50.;
        if (rad) masked = masked || b[23] < 0. || b[24] > 750.;
        row[STATS_REDO_SLOT] = masked ? 1. : 0.;
        row[0] = b[0];
        row[1] = b[0];
        for (int f = 0; f < NFIELDS; ++f) {
            const int g = (f < 8) ? f : 7;   // field 8 = rad_lw again (checked against the short-wave range)
            row[2 + 5 * f + 0] = b[1 + 3 * g];
            row[2 + 5 * f + 1] = b[2 + 3 * g];
            row[2 + 5 * f + 2] = b[3 + 3 * g];
            row[2 + 5 * f + 3] = b[2 + 3 * g];
            row[2 + 5 * f + 4] = b[3 + 3 * g];
        }
    }
}

__global__ void __launch_bounds__(STATS_BLOCK, 2) stats_fast_kernel(const StatsArgs a) { stats_fast_block<double>(a, threadIdx.x); }

// the same for arrays of element type T
template <class T>
__global__ void __launch_bounds__(STATS_BLOCK, 2) stats_fast_io_kernel(const StatsArgs a) { stats_fast_block<T>(a, threadIdx.x); }

// the full accumulator set (masked and raw statistics side by side), for the blocks stats_fast_kernel flagged
template <class T>
__device__ __forceinline__ void stats_fix_block(const StatsArgs &a, unsigned tid)
{
    if (a.partials[(long long)blockIdx.x * NSTATS + STATS_REDO_SLOT] == 0.) return;
    double acc[2 + 5 * NFIELDS];
    acc[0] = 0.;
    acc[1] = 0.;
#pragma unroll
    for (int f = 0; f < NFIELDS; ++f) {
        acc[2 + 5 * f + 0] = 0.;
        acc[2 + 5 * f + 1] = DBL_MAX;
        acc[2 + 5 * f + 2] = -DBL_MAX;
        acc[2 + 5 * f + 3] = DBL_MAX;
        acc[2 + 5 * f + 4] = -DBL_MAX;
    }
    const bool rad = (a.rad_lw != nullptr);
    const long long stride = (long long)gridDim.x * STATS_BLOCK;
    // STATS_UNROLL points per trip with all their loads issued first: the pass is bound by memory latency, not by its
    // arithmetic (one point per trip ran at 1.5 TB/s: ~47 accumulators leave room for 2 blocks per SM only)
    constexpr int STATS_UNROLL = 4;
    for (long long i0 = (long long)blockIdx.x * STATS_BLOCK + tid; i0 < a.n; i0 += stride * STATS_UNROLL) {
        double in[STATS_UNROLL][7];
#pragma unroll
        for (int u = 0; u < STATS_UNROLL; ++u) {
            const long long i = i0 + u * stride;
            const bool ok = i < a.n;
            const long long j = ok ? i : i0;
            in[u][0] = ld<T>(a.sst, j);
            in[u][1] = ld<T>(a.t_zt, j);
            in[u][2] = ld<T>(a.slp, j);
            in[u][3] = ld<T>(a.U_zu, j);
            in[u][4] = ld<T>(a.V_zu, j);
            in[u][5] = ld<T>(a.hum_zt, j);
            in[u][6] = rad ? ld<T>(a.rad_lw, j) : 0.;
        }
#pragma unroll
        for (int u = 0; u < STATS_UNROLL; ++u) {
            if (i0 + u * stride >= a.n) break;
            double v[NFIELDS];
            v[0] = in[u][0];
            v[1] = in[u][1];
            v[2] = in[u][2];
            v[3] = in[u][3];
            v[4] = in[u][4];
            v[5] = sqrt(__dadd_rn(__dmul_rn(v[3], v[3]), __dmul_rn(v[4], v[4])));
            v[6] = in[u][5];
            v[7] = in[u][6];
            v[8] = v[7];
            const bool m = point_unmasked(v[0], v[1], v[2], v[5], rad, v[7]);
            acc[0] += m ? 1. : 0.;
            acc[1] += 1.;
#pragma unroll
            for (int f = 0; f < NFIELDS; ++f) {
                // (v < acc ? v : acc) keeps acc when v is a NaN, like fmin / fmax, in 3 instructions instead of their 8-9
                if (m) {
                    acc[2 + 5 * f + 0] += v[f];
                    acc[2 + 5 * f + 1] = abm::dmin(v[f], acc[2 + 5 * f + 1]);
                    acc[2 + 5 * f + 2] = abm::dmax(v[f], acc[2 + 5 * f + 2]);
                }
                acc[2 + 5 * f + 3] = abm::dmin(v[f], acc[2 + 5 * f + 3]);
                acc[2 + 5 * f + 4] = abm::dmax(v[f], acc[2 + 5 * f + 4]);
            }
        }
    }
    __shared__ double sm[STATS_BLOCK / 32][2 + 5 * NFIELDS];
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int k = 0; k < 2 + 5 * NFIELDS; ++k) {
        const double r = warp_reduce(acc[k], stat_op(k));
        if (lane == 0) sm[warp][k] = r;
    }
    __syncthreads();
    if (tid < 2 + 5 * NFIELDS) {
        const int k = tid, op = stat_op(k);
        double r = sm[0][k];
        for (int w = 1; w < STATS_BLOCK / 32; ++w)
            r = (op == 0) ? r + sm[w][k] : (op == 1) ? fmin(r, sm[w][k]) : fmax(r, sm[w][k]);
        a.partials[(long long)blockIdx.x * NSTATS + k] = r;
    }
}

__global__ void __launch_bounds__(STATS_BLOCK) stats_fix_kernel(const StatsArgs a) { stats_fix_block<double>(a, threadIdx.x); }

template <class T>
__global__ void __launch_bounds__(STATS_BLOCK) stats_fix_io_kernel(const StatsArgs a) { stats_fix_block<T>(a, threadIdx.x); }

// fixed-order final reduction (one block of 128 threads per statistic) -> results do not depend on scheduling
static constexpr int FINAL_BLOCK = 128;
__global__ void __launch_bounds__(FINAL_BLOCK) stats_final(const double *partials, int nblocks, double *out)
{
    const int k = blockIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (k >= 2 + 5 * NFIELDS) {
        if (threadIdx.x == 0) out[k] = 0.;
        return;
    }
    const int op = stat_op(k);
    double r = (op == 0) ? 0. : (op == 1) ? DBL_MAX : -DBL_MAX;
    for (int b = threadIdx.x; b < nblocks; b += FINAL_BLOCK) {
        const double x = partials[(long long)b * NSTATS + k];
        r = (op == 0) ? r + x : (op == 1) ? fmin(r, x) : fmax(r, x);
    }
    r = warp_reduce(r, op);
    __shared__ double sm[FINAL_BLOCK / 32];
    if (lane == 0) sm[w] = r;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = sm[0];
        for (int j = 1; j < FINAL_BLOCK / 32; ++j) t = (op == 0) ? t + sm[j] : (op == 1) ? fmin(t, sm[j]) : fmax(t, sm[j]);
        out[k] = t;
    }
}

int stats_max_blocks() { return STATS_MAX_BLOCKS; }

cudaError_t launch_stats(size_t elem, const StatsArgs &a, int nblocks, cudaStream_t s)
{
    const auto fast = elem == ELEM_F64 ? stats_fast_kernel : elem == ELEM_F32 ? stats_fast_io_kernel<float> : nullptr;
    const auto fix = elem == ELEM_F64 ? stats_fix_kernel : elem == ELEM_F32 ? stats_fix_io_kernel<float> : nullptr;
    if (!fast) return cudaErrorInvalidValue;
    fast<<<nblocks, STATS_BLOCK, 0, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    fix<<<nblocks, STATS_BLOCK, 0, s>>>(a);   // returns at once in every block that holds no masked point
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    stats_final<<<NSTATS, FINAL_BLOCK, 0, s>>>(a.partials, nblocks, a.out);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// init_decide_kernel: the stats-dependent half of AEROBULK_INIT on the device, so that jt == 1 of a device-resident
// session needs no host round trip (the host re-derives the same verdict, with its messages, when it next synchronises)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(NSTATS) init_decide_kernel(const double *all, int nranks, int have_rad, double *gstats, int *init)
{
    __shared__ double st[NSTATS];
    const int k = threadIdx.x;
    const int op = stat_op(k);
    double r = all[k];
    for (int d = 1; d < nranks; ++d) {
        const double w = all[(long long)d * NSTATS + k];
        r = (op == 0) ? r + w : (op == 1) ? fmin(r, w) : fmax(r, w);
    }
    st[k] = r;
    gstats[k] = r;
    __syncthreads();
    if (k != 0) return;
    const double np = st[0];
    int ihum = 0, err = 0;
    if (!(np > 0.)) {
        err = 4;   // AEROBULK_GPU_ERR_ALL_MASKED
    } else {
        // type_of_humidity, mod_phymbl.f90:1957-2007
        const double *h = st + 2 + 5 * 6;
        const double zmean = h[0] / np, zmin = h[1], zmax = h[2];
        double hlo = 0., hhi = 0.08;
        if (zmean >= 0. && zmean < 0.08 && zmin >= 0. && zmax < 0.08) { ihum = 0; }
        else if (zmean >= 150. && zmean < 330. && zmin >= 150. && zmax < 330.) { ihum = 1; hlo = 150.; hhi = 330.; }
        else if (zmean >= 0. && zmean <= 100. && zmin >= 0. && zmax <= 100.) { ihum = 2; hlo = 0.; hhi = 100.; }
        else err = 5;   // AEROBULK_GPU_ERR_HUMIDITY
        // check_unit_consistency, mod_phymbl.f90:1851-1954; field order of the statistics vector
        const double lo[9] = {270., 180., 80000., -50., -50., 0., hlo, 0., 0.};
        const double hi[9] = {320., 330., 110000., 50., 50., 50., hhi, 1500., 750.};
        for (int f = 0; f < (have_rad ? 9 : 7) && !err; ++f) {
            const double *s5 = st + 2 + 5 * f;
            const double m = s5[0] / np;
            if (s5[2] > hi[f] || s5[1] < lo[f] || m < lo[f] || m > hi[f]) err = 6;   // AEROBULK_GPU_ERR_UNITS
        }
    }
    init[0] = ihum;
    init[1] = err;
}

cudaError_t launch_init_decide(const double *all, int nranks, int have_rad, double *gstats, int *init, cudaStream_t s)
{
    init_decide_kernel<<<1, NSTATS, 0, s>>>(all, nranks, have_rad, gstats, init);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// flux diagnostics: sum / min / max of the output fields (the optional global reduction of SURVEY.md 8e)
// ---------------------------------------------------------------------------
__host__ __device__ inline int diag_op(int k) { return k == 0 ? 0 : (k - 1) % 3; }   // 0 sum, 1 min, 2 max

__global__ void __launch_bounds__(STATS_BLOCK) diag_kernel(const DiagArgs a)
{
    double acc[NDIAG];
    acc[0] = 0.;
#pragma unroll
    for (int f = 0; f < NDIAG_FIELDS; ++f) {
        acc[1 + 3 * f] = 0.;
        acc[2 + 3 * f] = DBL_MAX;
        acc[3 + 3 * f] = -DBL_MAX;
    }
    const long long stride = (long long)gridDim.x * STATS_BLOCK;
    for (long long i = (long long)blockIdx.x * STATS_BLOCK + threadIdx.x; i < a.n; i += stride) {
        acc[0] += 1.;
#pragma unroll
        for (int f = 0; f < NDIAG_FIELDS; ++f) {
            if (!a.field[f]) continue;
            const double v = __ldg(a.field[f] + i);
            acc[1 + 3 * f] += v;
            acc[2 + 3 * f] = fmin(acc[2 + 3 * f], v);
            acc[3 + 3 * f] = fmax(acc[3 + 3 * f], v);
        }
    }
    __shared__ double sm[STATS_BLOCK / 32][NDIAG];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NDIAG; ++k) {
        const double r = warp_reduce(acc[k], diag_op(k));
        if (lane == 0) sm[w][k] = r;
    }
    __syncthreads();
    if (threadIdx.x < NDIAG) {
        const int k = threadIdx.x, op = diag_op(k);
        double r = sm[0][k];
        for (int j = 1; j < STATS_BLOCK / 32; ++j) r = (op == 0) ? r + sm[j][k] : (op == 1) ? fmin(r, sm[j][k]) : fmax(r, sm[j][k]);
        a.partials[(long long)blockIdx.x * NDIAG + k] = r;
    }
}

__global__ void __launch_bounds__(32 * NDIAG) diag_final(const double *partials, int nblocks, double *out)
{
    const int k = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int op = diag_op(k);
    double r = (op == 0) ? 0. : (op == 1) ? DBL_MAX : -DBL_MAX;
    for (int b = lane; b < nblocks; b += 32) {
        const double w = partials[(long long)b * NDIAG + k];
        r = (op == 0) ? r + w : (op == 1) ? fmin(r, w) : fmax(r, w);
    }
    r = warp_reduce(r, op);
    if (lane == 0) out[k] = r;
}

cudaError_t launch_diag(const DiagArgs &a, int nblocks, cudaStream_t s)
{
    diag_kernel<<<nblocks, STATS_BLOCK, 0, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    diag_final<<<1, 32 * NDIAG, 0, s>>>(a.partials, nblocks, a.out);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// FP64 peak: 8 independent dependent-DFMA chains per thread
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dfma_peak_kernel(double *out, int iters, double a, double b)
{
    double x0 = threadIdx.x, x1 = x0 + 1., x2 = x0 + 2., x3 = x0 + 3., x4 = x0 + 4., x5 = x0 + 5., x6 = x0 + 6., x7 = x0 + 7.;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    out[(long long)blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

double measure_fp64_peak(cudaStream_t s)
{
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return -1.;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1.;
    const int blocks = sms * 8, threads = 256, iters = 4096;
    double *out = nullptr;
    if (cudaMalloc(&out, sizeof(double) * (size_t)blocks * threads) != cudaSuccess) return -1.;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    double best = 0.;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0, s);
        dfma_peak_kernel<<<blocks, threads, 0, s>>>(out, iters, 0.999999, 1.e-9);
        cudaEventRecord(e1, s);
        if (cudaEventSynchronize(e1) != cudaSuccess) { best = -1.; break; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double n = (double)blocks * threads * (double)iters * 64.;
        if (rep > 0 && ms > 0.f) best = fmax(best, n / (ms * 1e-3));
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    return best;
}

}  // namespace abk
