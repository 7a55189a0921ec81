// ab_kernels.cuh -- host-visible launch interface of the sm_100a kernels.
#pragma once

#include <cuda_runtime.h>

#include <type_traits>

#include "ab_device.cuh"
#include "ab_ice.cuh"

namespace abk {

template <int V> using IntC = std::integral_constant<int, V>;
template <bool V> using BoolC = std::bool_constant<V>;

// The instantiation an ocean launch runs: f(ALGO, SKIN, ZTEQ) with std::integral_constant arguments, nullptr for an
// unknown algorithm.  Skin schemes exist for COARE 3.x and ECMWF only: NCAR and ANDREAS ignore `skin`.
template <class F>
auto pick_ocean(int algo, bool skin, bool zteq, F f) -> decltype(f(IntC<abd::NCAR>{}, BoolC<false>{}, BoolC<false>{}))
{
    const auto z = [&](auto A, auto S) { return zteq ? f(A, S, BoolC<true>{}) : f(A, S, BoolC<false>{}); };
    const auto sz = [&](auto A) { return skin ? z(A, BoolC<true>{}) : z(A, BoolC<false>{}); };
    switch (algo) {
    case abd::COARE3P0: return sz(IntC<abd::COARE3P0>{});
    case abd::COARE3P6: return sz(IntC<abd::COARE3P6>{});
    case abd::ECMWF: return sz(IntC<abd::ECMWF>{});
    case abd::NCAR: return z(IntC<abd::NCAR>{}, BoolC<false>{});
    case abd::ANDREAS: return z(IntC<abd::ANDREAS>{}, BoolC<false>{});
    default: return nullptr;
    }
}

// Element type of the caller's per-point arrays in one aerobulk_model launch, given by its size in bytes:
// sizeof(double) runs the FP64 kernels (flux_kernel, classify_kernel, stats_*_kernel); sizeof(float) runs their
// *_io_kernel<float> twins, which widen every input exactly on load, compute in FP64 with the same code, and round every
// output once to nearest on store.  Anything else: cudaErrorInvalidValue.
constexpr size_t ELEM_F64 = sizeof(double);
constexpr size_t ELEM_F32 = sizeof(float);

// One fused launch = reference aerobulk_compute (src/mod_aerobulk_compute.f90:22-213)
// steps 1-9 for `n` consecutive grid points.
struct FluxArgs {
    // inputs (device), of the launch's element type
    const void *sst, *t_zt, *hum_zt, *U_zu, *V_zu, *slp;
    const void *rad_sw, *rad_lw;     // skin only
    const double *lon;               // optional longitudes [deg E]; NULL -> 0 (mod_aerobulk_compute.f90:126)
    // outputs (device), of the launch's element type; T_s may be NULL
    void *QL, *QH, *Tau_x, *Tau_y, *Evap, *T_s;
    // persistent warm-layer state (device); COARE: 4 arrays, ECMWF: dT_wl only
    double *dT_wl, *Hz_wl, *Qnt_ac, *Tau_ac;
    long long n;
    abd::Uniform u;
    int ihum;          // 0 'sh', 1 'dp', 2 'rh'   (mod_aerobulk_compute.f90:99-108)
    // device-side AEROBULK_INIT still in flight (asynchronous jt == 1 of a device-resident session): {humidity type,
    // error flag} written by init_decide_kernel earlier on the same stream; NULL: `ihum` above is final
    const int *init_dev;
    int first_step;    // kt == nit000: state starts from its *_INIT values, not from memory
    // first linear index whose wind stress exceeds 10 N/m^2 (mod_phymbl.f90:1250-1253), else ~0ull
    unsigned long long *bad_index;
    long long index_offset;   // global index of point 0 (chunked / sharded launches)
    // optional stability sort (classify_kernel): slot -> point inside windows of sort_window() points,
    // padded to a whole number of windows; NULL: identity
    const unsigned short *perm;
};

// One launch = one TURB_* call of the reference (SURVEY.md 8f row 1; interfaces
// src/mod_blk_coare3p6.f90:123-127, mod_blk_coare3p0.f90:54-59, mod_blk_ecmwf.f90:63-68, mod_blk_ncar.f90:57-59,
// mod_blk_andreas.f90:66-68): inputs are already potential temperature, specific humidity and scalar wind.
struct TurbArgs {
    double *T_s, *q_s;                        // in: bulk SST and its ssq; out: skin values when cs/wl are used
    const double *t_zt, *q_zt, *U_zu;
    const double *Qsw, *rad_lw, *slp, *lon;   // skin only; Qsw is the NET solar flux; lon may be NULL (-> 0)
    double *Cd, *Ch, *Ce, *t_zu, *q_zu, *Ubzu;
    double *opt[10];                          // CdN ChN CeN xz0 xu_star xL xUN10 pdT_cs pdT_wl pHz_wl (NULL: not wanted)
    double *dT_wl, *Hz_wl, *Qnt_ac, *Tau_ac;  // persistent warm-layer state
    long long n;
    abd::Uniform u;
    int first_step;
};
cudaError_t launch_turb(int algo, bool cs, bool wl, bool zt_eq_zu, const TurbArgs &a, cudaStream_t s);

// Station time series (SURVEY.md 8f row 3): the time loop of src/tests/test_aerobulk_buoy_series_oce.f90:364-537 for S
// independent stations in ONE launch -- one thread per station walks its Nt records with the warm-layer state in
// registers.  Records are [Nt][S] (station index fastest: coalesced).
constexpr int NSERIES_OUT = 28;
struct SeriesArgs {
    const int *isd;                  // [Nt] UTC seconds since midnight of each record
    const double *lon;               // [S]
    const double *sst, *t_zt, *hum_zt, *wnd, *slp, *rad_sw, *rad_lw;   // [Nt][S]
    // rho_zu QL QH Qlw QNS Qsw dT_cs dT_wl TAU dT Hz_wl Qnt_ac Tau_ac Cd Ce Ch theta_zu q_zu t_zu RiB z0 u_star L UN10
    // Ts Evap q_zt theta_zt  (NULL: not wanted)
    double *out[NSERIES_OUT];
    long long S;
    int Nt;
    int hum_kind;                    // 0 specific humidity, 1 dew-point [K], 2 relative humidity [%]
    abd::Uniform u;                  // isd / dawn are per record here and ignored
    unsigned long long *bad_index;   // first record*S + station whose stress exceeds 10 N/m^2, else ~0ull
};
cudaError_t launch_series(int algo, bool skin, bool zt_eq_zu, const SeriesArgs &a, cudaStream_t s);

// Sea ice (SURVEY.md 8f row 4).  One launch = one TURB_ICE_* call (src/ice/mod_blk_ice_*.f90).
struct IceTurbArgs {
    const double *Ts_i, *t_zt, *qs_i, *q_zt, *U_zu, *frice;   // frice: lu12 / lg15 only (else NULL)
    double *Cd, *Ch, *Ce, *t_zu, *q_zu, *Ubzu;
    double *opt[8];                  // CdN ChN CeN xz0 xu_star xL xUN10 CdN_frm (NULL: not wanted)
    long long n;
    long long form_index;            // point whose ice fraction drives the LG15 form drag (reference: n-1), -1: each its own
    abd::IceUniform u;
    unsigned long long *bad_rough;   // first point where rough_leng_tq would ctl_stop, else ~0ull
};
cudaError_t launch_ice_turb(int ialgo, bool zt_eq_zu, const IceTurbArgs &a, cudaStream_t s);

// Ice + leads workflow of src/ice/test_aerobulk_oce+ice.f90:225-412: ice_flux_kernel writes out[0..16], leads_kernel
// out[17..34] (the cell means read the four ice fluxes back from `ice_flux`).
constexpr int NOCEICE_OUT = 35;
struct OceIceArgs {
    const double *sit, *sst, *t_zt, *hum_zt, *wnd, *slp, *frice;
    double *out[NOCEICE_OUT];
    double *ice_flux[4];             // Tau, QH, QL, Evap over the ice (user arrays or scratch)
    long long n;
    long long form_index;
    int hum_kind;
    abd::IceUniform ui;
    abd::Uniform uo;
    unsigned long long *bad_tau, *bad_rough;
};
cudaError_t launch_ice_flux(int ialgo, bool zt_eq_zu, const OceIceArgs &a, cudaStream_t s);

// Sea-ice station series (src/ice/test_aerobulk_buoy_series_ice.f90:326-470), one thread per record.
// out: 0 rho_zu 1 QL 2 QH 3 Qlw 4 QNS 5 Qsw 6 TAU 7 SBLM 8 Cd_i 9 Ch_i 10 Ce_i 11 z0 12 RiB_zt 13 RiB_zu 14 CdN 15 u_star 16 L
//      17 UN10 18 theta_zu 19 q_zu 20 Ublk
constexpr int NICESERIES_OUT = 21;
struct IceSeriesArgs {
    const double *sic, *sit, *t_zt, *hum_zt, *wnd, *slp, *rad_sw, *rad_lw;
    double *out[NICESERIES_OUT];
    long long n;
    int hum_kind;
    abd::IceUniform ui;
    unsigned long long *bad_tau, *bad_rough;
};
cudaError_t launch_ice_series(int ialgo, bool zt_eq_zu, const IceSeriesArgs &a, cudaStream_t s);
cudaError_t launch_leads(int oalgo, bool zt_eq_zu, const OceIceArgs &a, cudaStream_t s);

// number of doubles in the statistics vector (see include/aerobulk_gpu.h)
constexpr int NSTATS = 64;
constexpr int NFIELDS = 9;

struct StatsArgs {
    const void *sst, *t_zt, *hum_zt, *U_zu, *V_zu, *slp, *rad_lw;   // of the launch's element type; rad_lw may be NULL
    long long n;
    double *partials;   // [gridDim.x][NSTATS]
    double *out;        // [NSTATS]
};

// Global flux diagnostics (SURVEY.md 8e: the optional reduction): sum / min / max of up to 6 fields.
// out[1 + 3 f + {0,1,2}] = sum, min, max of field f; out[0] = number of points.  Fixed-order reduction (deterministic).
constexpr int NDIAG_FIELDS = 6;
constexpr int NDIAG = 1 + 3 * NDIAG_FIELDS;
struct DiagArgs {
    const double *field[NDIAG_FIELDS];   // NULL: skipped (sum 0, min +DBL_MAX, max -DBL_MAX)
    long long n;
    double *partials;                    // [gridDim.x][NDIAG]
    double *out;                         // [NDIAG]
};
cudaError_t launch_diag(const DiagArgs &a, int nblocks, cudaStream_t s);

// `elem`: ELEM_F64 or ELEM_F32, the element type of the per-point arrays of `a`
cudaError_t launch_flux(int algo, bool skin, bool zt_eq_zu, size_t elem, const FluxArgs &a, cudaStream_t s);
// block size / register info for reports
int flux_block_size();
int sort_window();
// fills perm[] (ceil(n / sort_window()) * sort_window() entries) for the launch described by `a`
cudaError_t launch_classify(size_t elem, const FluxArgs &a, unsigned short *perm, bool skin, cudaStream_t s);
cudaError_t launch_stats(size_t elem, const StatsArgs &a, int nblocks, cudaStream_t s);
// AEROBULK_INIT's stats-dependent decisions on the device (src/mod_aerobulk.f90:104-153, src/mod_phymbl.f90:1851-2007):
// combines the statistics vectors of `nranks` row blocks (all[r][NSTATS], rank order: deterministic) into gstats[NSTATS]
// and writes init[0] = humidity type (0 'sh', 1 'dp', 2 'rh'), init[1] = 0 or the AEROBULK_GPU_ERR_* code the host will
// raise when it next synchronises (all masked / unknown humidity / unit check).
cudaError_t launch_init_decide(const double *all, int nranks, int have_rad, double *gstats, int *init, cudaStream_t s);
int stats_max_blocks();
// DFMA-chain microbenchmark: returns FP64 FMA instructions per second, <0 on error
double measure_fp64_peak(cudaStream_t s);
// blocks_per_sm (may be NULL): resident blocks per SM at the launch configuration
cudaError_t flux_kernel_attributes(int algo, bool skin, bool zt_eq_zu, cudaFuncAttributes *attr, int *blocks_per_sm);

// probe_kernel (ab_probe.cu): one __device__ building block per launch, for the per-function GPU unit tests.
// The numbering is part of the C ABI (aerobulk_gpu_probe, include/aerobulk_gpu.h).
enum ProbeFunc {
    PROBE_E_SAT = 1, PROBE_Q_SAT, PROBE_THETA, PROBE_RHO_AIR, PROBE_VISC_AIR, PROBE_L_VAP, PROBE_CP_AIR, PROBE_GAMMA_MOIST,
    PROBE_ALPHA_SW, PROBE_QLW_NET, PROBE_ONE_ON_L, PROBE_RI_BULK, PROBE_Q_AIR_RH, PROBE_Q_AIR_DP,
    PROBE_PSI_M_NCAR = 20, PROBE_PSI_H_NCAR, PROBE_PSI_M_COARE, PROBE_PSI_H_COARE, PROBE_PSI_M_ECMWF, PROBE_PSI_H_ECMWF,
    PROBE_PSI_M_ANDREAS, PROBE_PSI_H_ANDREAS,
    PROBE_Z0TQ_LKB = 30, PROBE_CD_N10_NCAR, PROBE_CHARN_COARE3P0, PROBE_CHARN_COARE3P6, PROBE_CS_COARE, PROBE_CS_ECMWF,
    PROBE_EXP = 40, PROBE_EXP10, PROBE_LOG, PROBE_ATAN, PROBE_SQRT, PROBE_RSQRT, PROBE_CBRT, PROBE_RCBRT, PROBE_POW075,
    PROBE_RCP, PROBE_POWR, PROBE_ATAN_GE1, PROBE_LOG10, PROBE_EXP_B, PROBE_EXP10_B,
    PROBE_E_SAT_ICE = 60, PROBE_Q_SAT_ICE, PROBE_PSI_M_ICE, PROBE_PSI_H_ICE, PROBE_F_M_LOUIS, PROBE_F_H_LOUIS,
    PROBE_ROUGH_LENG_M, PROBE_Z0T_AN87, PROBE_Z0Q_AN87, PROBE_CDN10_LU13, PROBE_CDN_LG15
};
cudaError_t launch_probe(int func, long long n, int nargs, const double *args, double *out, cudaStream_t s);

}  // namespace abk
