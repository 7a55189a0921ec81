/*
 * aerobulk_gpu.h -- C ABI of libaerobulk_gpu.so, the B200 (sm_100a) replacement
 * for the `aerobulk_model` hot path of brodeau/aerobulk.
 *
 * The library is a LINK-TIME DROP-IN for the two symbols the reference's C++
 * bridge binds (reference: src/aerobulk.cpp:5-19 declares them,
 * src/mod_aerobulk_cxx.f90:29-33,66-69 defines them with BIND(C)):
 *
 *     aerobulk_cxx_skin      aerobulk_cxx_no_skin
 *
 * plus `aerobulk_gpu_*` entry points that the Fortran shim
 * (aerobulk_b200/fortran/mod_aerobulk_gpu.f90, behind the unchanged
 * AEROBULK_MODEL signature of src/mod_aerobulk.f90:176-230) binds through
 * ISO_C_BINDING.  Plain pointers and sizes only; no C++/torch types.
 *
 * Arrays are FP64 (FP32 for the *_f32 calls), (Ni,Nj) column-major (Fortran order), contiguous.
 * Unless stated otherwise a call is blocking and returns 0 on success or an
 * AEROBULK_GPU_ERR_* code.  Error behaviour mirrors the reference: by default
 * (fail-stop mode) an error prints ' *** E R R O R :' + message on stdout and
 * terminates the process like `ctl_stop`/STOP does (src/mod_const.f90:238-278);
 * unlike Fortran STOP the exit status is 1.  aerobulk_gpu_set_error_mode(1)
 * makes the calls return the code instead (used by language bindings).
 *
 * There is NO CPU fallback: without a CUDA device every compute entry point fails.
 *
 * Host arrays (on_device = 0, and aerobulk_gpu_model / aerobulk_cxx_*): pageable memory is staged through device
 * buffers; aerobulk_gpu_model on 65536 points or more moves it instead through a pinned slab of its own on a few
 * persistent host threads, chunk by chunk around the kernel.  When EVERY array of a call is pinned
 * (cudaHostAlloc / cudaHostRegister) the kernels read and write the caller's memory directly over PCIe ("zero-copy":
 * same results, ~20 % faster end to end, no staging memory).
 * Environment: AEROBULK_GPU_DEVICE (or LOCAL_RANK) device ordinal; AEROBULK_GPU_ZEROCOPY=0 staged copies even for pinned
 * arrays (and no pinned slab for pageable ones); pageable arrays: AEROBULK_GPU_BOUNCE=0 driver-staged copies,
 * AEROBULK_GPU_HOST_THREADS copy threads (default: 3/4 of the CPUs the process may run on, at most 12),
 * AEROBULK_GPU_BOUNCE_CHUNK_POINTS, AEROBULK_GPU_COPY_STREAMING=0 plain instead of non-temporal stores,
 * AEROBULK_GPU_BOUNCE_MAX_MB largest pinned slab the library may allocate for them (default 12288; beyond it, or when the
 * host refuses the allocation, the driver-staged copies are used).
 */
#ifndef AEROBULK_GPU_H
#define AEROBULK_GPU_H

#include <stdbool.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- error codes ------------------------------------------------------- */
enum {
    AEROBULK_GPU_OK = 0,
    AEROBULK_GPU_ERR_JT = 1,          /* jt < 1                (mod_aerobulk.f90:244)            */
    AEROBULK_GPU_ERR_SKIN_ALGO = 2,   /* skin asked for ncar/andreas (mod_aerobulk.f90:69-70)    */
    AEROBULK_GPU_ERR_SKIN_NORAD = 3,  /* skin asked, no radiation    (mod_aerobulk.f90:72)       */
    AEROBULK_GPU_ERR_ALL_MASKED = 4,  /* whole domain masked         (mod_aerobulk.f90:122)      */
    AEROBULK_GPU_ERR_HUMIDITY = 5,    /* humidity type unidentified  (mod_phymbl.f90:1996-2003)  */
    AEROBULK_GPU_ERR_UNITS = 6,       /* unit-consistency check      (mod_phymbl.f90:1946-1950)  */
    AEROBULK_GPU_ERR_ALGO = 7,        /* unknown algorithm string    (mod_aerobulk_compute.f90:173-176) */
    AEROBULK_GPU_ERR_TAU = 8,         /* wind stress > 10 N/m^2      (mod_phymbl.f90:1250-1253)  */
    AEROBULK_GPU_ERR_STATE = 9,       /* warm-layer state (re)allocation (mod_blk_coare3p6.f90:82-83) */
    AEROBULK_GPU_ERR_ICE_ROUGH = 10,  /* rough_leng_tq ctl_stop  (src/ice/mod_blk_ice_an05.f90:296-297) */
    AEROBULK_GPU_ERR_CUDA = 100,      /* CUDA runtime failure / no device                         */
    AEROBULK_GPU_ERR_ARG = 101,       /* NULL / inconsistent argument                             */
    AEROBULK_GPU_ERR_IO = 102         /* series CSV: file cannot be opened / parsed               */
};

/* ---- the two symbols of the reference's C++ bridge ------------------------ */

/* Replaces SUBROUTINE aerobulk_cxx_skin BIND(c), src/mod_aerobulk_cxx.f90:29-62
 * (declared in src/aerobulk.cpp:7-11).  All scalars by pointer; `calgo` holds `*l`
 * characters (+NUL); every array has `*m` elements and is treated as (m,1).
 * l_skin is read as ONE byte (the reference reads a 4-byte LOGICAL through a
 * `const bool*`, a latent ABI bug: SURVEY 8a quirk 7). */
void aerobulk_cxx_skin(const int *jt, const int *Nt, const char *calgo, const double *zt, const double *zu,
                       const double *sst, const double *t_zt, const double *hum_zt, const double *U_zu,
                       const double *V_zu, const double *slp,
                       double *QL, double *QH, double *Tau_x, double *Tau_y, double *Evap,
                       const int *Niter, const bool *l_skin, const double *rad_sw, const double *rad_lw,
                       double *T_s, const int *l, const int *m);

/* Replaces SUBROUTINE aerobulk_cxx_no_skin BIND(c), src/mod_aerobulk_cxx.f90:66-95
 * (declared in src/aerobulk.cpp:13-17). */
void aerobulk_cxx_no_skin(const int *jt, const int *Nt, const char *calgo, const double *zt, const double *zu,
                          const double *sst, const double *t_zt, const double *hum_zt, const double *U_zu,
                          const double *V_zu, const double *slp,
                          double *QL, double *QH, double *Tau_x, double *Tau_y, double *Evap,
                          const int *Niter, const int *l, const int *m);

/* ---- AEROBULK_MODEL for 2-D fields (what mod_aerobulk_gpu.f90 binds) --------- */

/* Replaces SUBROUTINE AEROBULK_MODEL, src/mod_aerobulk.f90:176-269, HOST arrays.
 * Optional Fortran arguments: `Niter`/`l_use_skin` NULL when absent; `rad_sw`,
 * `rad_lw`, `T_s` NULL when absent (the skin path is taken iff rad_sw and rad_lw
 * are both present, mod_aerobulk.f90:242-246).  calgo is NUL-terminated. */
int aerobulk_gpu_model(int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj,
                       const double *sst, const double *t_zt, const double *hum_zt,
                       const double *U_zu, const double *V_zu, const double *slp,
                       double *QL, double *QH, double *Tau_x, double *Tau_y, double *Evap,
                       const int *Niter, const int *l_use_skin,
                       const double *rad_sw, const double *rad_lw, double *T_s);

/* Same contract, but every array pointer is a DEVICE pointer on the session's
 * device and the work is enqueued on the session's stream (see
 * aerobulk_gpu_set_stream).  At jt==1 the call synchronises (AEROBULK_INIT needs
 * the field statistics on the host); for jt>1 it returns after the launch and
 * the wind-stress check is deferred to aerobulk_gpu_synchronize(). */
int aerobulk_gpu_model_device(int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj,
                              const double *sst, const double *t_zt, const double *hum_zt,
                              const double *U_zu, const double *V_zu, const double *slp,
                              double *QL, double *QH, double *Tau_x, double *Tau_y, double *Evap,
                              const int *Niter, const int *l_use_skin,
                              const double *rad_sw, const double *rad_lw, double *T_s);

/* ---- AEROBULK_MODEL on float32 fields ---------------------------------------------------------------------------
 * aerobulk_gpu_model_f32 (host arrays) and aerobulk_gpu_model_device_f32 (device pointers) take the same arguments as
 * the two calls above, with EVERY array float32: the 6 (8) inputs and the 5 (6) outputs.  Inputs are widened exactly to
 * FP64, everything from there on is the FP64 call's own computation -- AEROBULK_INIT's statistics and verdicts, the
 * stability sort, the bulk solve, the tau > 10 N/m^2 test -- and every output is rounded once, to nearest:
 *
 *     f32_call(x) == (float) f64_call((double) x)     bit for bit, at every point and every step.
 *
 * The warm-layer state stays FP64 on the device and after every step is bit-identical to the FP64 session's on the
 * widened inputs, so FP32 and FP64 calls may alternate within one jt = 1..Nt session, and aerobulk_gpu_get_state /
 * aerobulk_gpu_set_state are unchanged.  Errors are the FP64 call's: same code, same AEROBULK_INIT message, same
 * (ji, jj) for tau > 10 (the stress it prints is computed from the float outputs).  Host arrays take the same paths as
 * FP64 ones (device staging, zero-copy on pinned arrays, the pinned slab for pageable ones, aerobulk_gpu_set_devices
 * splits) with half the bytes per point to move. */
int aerobulk_gpu_model_f32(int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj,
                           const float *sst, const float *t_zt, const float *hum_zt,
                           const float *U_zu, const float *V_zu, const float *slp,
                           float *QL, float *QH, float *Tau_x, float *Tau_y, float *Evap,
                           const int *Niter, const int *l_use_skin,
                           const float *rad_sw, const float *rad_lw, float *T_s);
int aerobulk_gpu_model_device_f32(int jt, int Nt, const char *calgo, double zt, double zu, int Ni, int Nj,
                                  const float *sst, const float *t_zt, const float *hum_zt,
                                  const float *U_zu, const float *V_zu, const float *slp,
                                  float *QL, float *QH, float *Tau_x, float *Tau_y, float *Evap,
                                  const int *Niter, const int *l_use_skin,
                                  const float *rad_sw, const float *rad_lw, float *T_s);

/* ---- direct TURB_* entry (what GCMs such as NEMO's sbcblk and the reference's test programs call) ------ */

/* Optional outputs of the TURB_* routines; any member may be NULL. */
typedef struct aerobulk_gpu_turb_optional {
    double *CdN, *ChN, *CeN;   /* neutral-stability transfer coefficients                      */
    double *xz0, *xu_star, *xL, *xUN10; /* roughness length [m], u* [m/s], Obukhov length [m], UN10 [m/s] */
    double *pdT_cs, *pdT_wl, *pHz_wl;   /* cool-skin / warm-layer increments [K], warm-layer depth [m]      */
} aerobulk_gpu_turb_optional;

/* Replaces TURB_COARE3P0 / TURB_COARE3P6 / TURB_ECMWF / TURB_NCAR / TURB_ANDREAS
 * (src/mod_blk_coare3p0.f90:54-59, mod_blk_coare3p6.f90:123-127, mod_blk_ecmwf.f90:63-68,
 * mod_blk_ncar.f90:57-59, mod_blk_andreas.f90:66-68), selected by calgo.
 * t_zt is the POTENTIAL air temperature, q_zt specific humidity, U_zu the scalar wind, Qsw the NET solar flux.
 * T_s / q_s: bulk SST and its saturation humidity in; skin values out when l_use_cs or l_use_wl.
 * Qsw, rad_lw, slp are needed with l_use_cs or l_use_wl, plong with l_use_wl (COARE) -- NULL otherwise.
 * kt is the time step (1: warm-layer state created; == nitend, see aerobulk_gpu_set_nitend: released);
 * the number of iterations is the nb_iter global (aerobulk_gpu_set_nb_iter).
 * on_device: 0 host arrays (blocking), 1 device pointers (asynchronous on the session stream). */
int aerobulk_gpu_turb(const char *calgo, int kt, double zt, double zu, int Ni, int Nj,
                      double *T_s, const double *t_zt, double *q_s, const double *q_zt, const double *U_zu,
                      int l_use_cs, int l_use_wl,
                      double *Cd, double *Ch, double *Ce, double *t_zu, double *q_zu, double *Ubzu,
                      const double *Qsw, const double *rad_lw, const double *slp,
                      int isecday_utc, const double *plong,
                      const aerobulk_gpu_turb_optional *opt, int on_device);
void aerobulk_gpu_set_nitend(int nitend);        /* mod_const.f90:22 (set by AEROBULK_INIT in the model path) */

/* ---- station time series (the reference's buoy-series workflow, without NetCDF) ------------------------ */

/* Output series of aerobulk_gpu_series, each [Nt][S] (station index fastest); any member may be NULL.
 * The first 16 are the variables src/tests/test_aerobulk_buoy_series_oce.f90:539-577 writes (Wind is an input). */
typedef struct aerobulk_gpu_series_out {
    double *rho_zu, *QL, *QH, *Qlw, *QNS, *Qsw, *dT_cs, *dT_wl, *TAU, *dT, *Hz_wl, *Qnt_ac, *Tau_ac, *Cd, *Ce, *Ch;
    double *theta_zu, *q_zu, *t_zu, *RiB, *z0, *u_star, *L, *UN10, *Ts, *Evap, *q_zt, *theta_zt;
} aerobulk_gpu_series_out;
#define AEROBULK_GPU_SERIES_NOUT 28

/* Runs the time loop of src/tests/test_aerobulk_buoy_series_oce.f90:364-537 for S independent stations in one
 * launch (one thread per station; warm-layer state in registers, created at record 1 and dropped after record Nt).
 * Inputs are [Nt][S]: sst [K], t_zt ABSOLUTE air temperature [K], hum_zt (hum_kind 0: specific humidity [kg/kg],
 * 1: dew-point [K], 2: relative humidity [%], capped at 99.999 as :227), wind scalar wind speed [m/s], slp [Pa],
 * rad_sw / rad_lw DOWNWELLING fluxes [W/m^2]; isecday_utc[Nt] (host memory, always) = hh*3600+mm*60 of each record
 * (:373), lon[S] station longitudes [deg E].  l_use_skin: cool-skin AND warm-layer on (as the program runs COARE
 * and ECMWF, :456-479); ignored for ncar / andreas.  The step between records is the rdt global
 * (aerobulk_gpu_set_rdt), the iteration count nb_iter (the program uses 20, :86).  'coare3p0' runs TURB_COARE3P0
 * (the program's slip of running 3.6 for that choice, :456, is not reproduced).
 * on_device: 0 host arrays, 1 device pointers (isecday_utc stays on the host); blocking either way. */
int aerobulk_gpu_series(const char *calgo, int Nt, long long S, double zt, double zu,
                        const int *isecday_utc, const double *lon,
                        const double *sst, const double *t_zt, const double *hum_zt, int hum_kind,
                        const double *wind, const double *slp, const double *rad_sw, const double *rad_lw,
                        int l_use_skin, const aerobulk_gpu_series_out *out, int on_device);

/* One station from / to CSV files: the whole program above (options -f/-r/-w, prompts for algorithm, zu, zt)
 * with CSV in place of NetCDF.  Input: one header line then one record per line; columns by the reference's
 * default names (src/mod_const.f90:208-220): time, lon, sst, t_air, one of q_air | rh_air | dp_air,
 * wndspd or u10 + v10, msl, ssrd, strd.  `time` is "YYYY-MM-DD hh:mm[:ss]" (also with 'T' or '/' '-' as in the
 * program's own date stamp); `lon` is read from the first record.  sst and t_air may be in deg C or K
 * (TO_KELVIN_3D rule of src/mod_phymbl.f90:1826-1847: series mean in ]-80,50[ -> deg C).
 * Output: time + the 16 series of the program + the inputs-derived extras, one line per record.
 * Returns 0, or an error code (AEROBULK_GPU_ERR_IO for file / format problems). */
int aerobulk_gpu_series_csv(const char *path_in, const char *path_out, const char *calgo, double zt, double zu,
                            int l_use_skin);

/* ---- sea ice (src/ice/) -------------------------------------------------------------------------------- */

/* Optional outputs of the TURB_ICE_* routines; any member may be NULL.  CdN_frm: neutral FORM drag (lu12, lg15,
 * lg15_io; 0 for the others). */
typedef struct aerobulk_gpu_turb_ice_optional {
    double *CdN, *ChN, *CeN, *xz0, *xu_star, *xL, *xUN10, *CdN_frm;
} aerobulk_gpu_turb_ice_optional;

/* Replaces TURB_ICE_NEMO / _EASY / _AN05 / _LU12 / _LG15 / _LG15_IO (src/ice/mod_blk_ice_nemo.f90:36-39,
 * mod_blk_ice_easy.f90:35-38, mod_blk_ice_an05.f90:41-43, mod_blk_ice_lu12.f90:50-52, mod_blk_ice_lg15.f90:53-55,
 * mod_blk_ice_lg15_io.f90:39-42 -- its over-ice outputs), selected by calgo = "nemo" | "easy" | "an05" | "lu12" | "lg15" |
 * "lg15_io".  t_zt is the POTENTIAL air temperature, qs_i the saturation humidity over ice at Ts_i, U_zu the scalar wind.
 * frice (ice fraction) is needed by lu12 / lg15 / lg15_io, CxN_easy[3] = CdN, ChN, CeN (host memory) by easy; NULL otherwise.
 * Iterations: the nb_iter global.  Not provided: TURB_ICE_BEST (reads an unset array in the reference,
 * mod_blk_ice_best.f90:154) and the over-water outputs of TURB_ICE_LG15_IO (never initialised there, :170-172).
 * Reference behaviour kept by default: the LG15 form drag of EVERY point is computed from the ice fraction of the LAST
 * point, because CdN_f_LG15_light assigns its whole result array inside the point loop (src/ice/mod_cdn_form_ice.f90:324);
 * aerobulk_gpu_set_ice_form_drag_per_point(1) uses each point's own fraction instead.
 * Error 10 where the reference's rough_leng_tq would ctl_stop (an05, roughness Reynolds number in ]2.49999, 2.5[). */
int aerobulk_gpu_turb_ice(const char *calgo, double zt, double zu, int Ni, int Nj,
                          const double *Ts_i, const double *t_zt, const double *qs_i, const double *q_zt,
                          const double *U_zu, const double *frice, const double *CxN_easy,
                          double *Cd, double *Ch, double *Ce, double *t_zu, double *q_zu, double *Ubzu,
                          const aerobulk_gpu_turb_ice_optional *opt, int on_device);
void aerobulk_gpu_set_ice_form_drag_per_point(int on);

/* Outputs of aerobulk_gpu_oce_ice; any member may be NULL.  _i over the ice, _w over the leads, no suffix: the
 * area-weighted cell mean A x_i + (1-A) x_w (the partition a model such as NEMO applies; the reference program prints the
 * two sides only). */
typedef struct aerobulk_gpu_oce_ice_out {
    double *Cd_i, *Ch_i, *Ce_i, *theta_zu_i, *q_zu_i, *t_zu_i, *Ub_i, *RiB_i, *z0_i, *u_star_i, *L_i, *UN10_i, *rho_zu_i;
    double *Tau_i, *QH_i, *QL_i, *Evap_i;
    double *Cd_w, *Ch_w, *Ce_w, *theta_zu_w, *q_zu_w, *Ub_w, *z0_w, *u_star_w, *L_w, *UN10_w, *Tau_w, *QH_w, *QL_w, *Evap_w;
    double *Tau, *QH, *QL, *Evap;
} aerobulk_gpu_oce_ice_out;

/* The ice + leads computation of src/ice/test_aerobulk_oce+ice.f90:225-412 (and test_aerobulk_ice.f90:186-370) on n
 * points: sit ice surface temperature [K], sst temperature of the leads [K], t_zt ABSOLUTE air temperature [K], hum_zt
 * (hum_kind 0 specific humidity, 1 dew-point [K], 2 RH [%]), wind [m/s], slp [Pa], frice ice fraction.  Over the ice:
 * siq = q_sat(sit, l_ice), theta_zt = t_zt + gamma_moist zt, TURB_ICE_<calgo_ice>, Ri_b, t_zu, rho_zu,
 * BULK_FORMULA(l_ice=.TRUE.) (sublimation heat, Evap = MIN(E, 0)).  Over the leads (calgo_oce NULL: skipped; the
 * program uses "ecmwf"): ssq = 0.98 q_sat(sst) (the program evaluates it at sit, :213 -- not reproduced),
 * TURB_<calgo_oce> without skin, BULK_FORMULA. */
int aerobulk_gpu_oce_ice(const char *calgo_ice, const char *calgo_oce, double zt, double zu, long long n,
                         const double *sit, const double *sst, const double *t_zt, const double *hum_zt, int hum_kind,
                         const double *wind, const double *slp, const double *frice, const double *CxN_easy,
                         const aerobulk_gpu_oce_ice_out *out, int on_device);

/* Outputs of aerobulk_gpu_series_ice, each n values; any member may be NULL. */
typedef struct aerobulk_gpu_series_ice_out {
    double *rho_zu, *QL, *QH, *Qlw, *QNS, *Qsw, *TAU, *SBLM;     /* SBLM: sublimation, kg/m^2/s (the program prints mm/day) */
    double *Cd_i, *Ch_i, *Ce_i, *z0, *RiB_zt, *RiB_zu, *CdN;
    double *u_star, *L, *UN10, *theta_zu, *q_zu, *Ublk;
} aerobulk_gpu_series_ice_out;

/* The sea-ice station series of src/ice/test_aerobulk_buoy_series_ice.f90:326-470 on n records (stations x time,
 * any order: nothing is carried from one record to the next): sic ice concentration, sit ice surface temperature [K],
 * t_zt ABSOLUTE air temperature [K], hum_zt (hum_kind as above), wind [m/s], slp [Pa], rad_sw / rad_lw downwelling
 * radiation [W/m^2].  calgo: "nemo", "an05", "lu12", "lg15" (the program's four choices; lg15 with the record's own
 * concentration, as its 1 x 1 arrays imply).  RiB_zt and Qsw = (1 - 0.8) rad_sw for every record; the bulk algorithm,
 * RiB_zu, BULK_FORMULA(l_ice), Qlw = 0.996 (rad_lw - sigma sit^4) and QNS = QH + QL + Qlw only where sic > 0.01 -- the
 * program skips the other records and leaves their values unset; here they are 0.  Iterations: the nb_iter global
 * (the program uses 20). */
int aerobulk_gpu_series_ice(const char *calgo, double zt, double zu, long long n, const double *sic, const double *sit,
                            const double *t_zt, const double *hum_zt, int hum_kind, const double *wind, const double *slp,
                            const double *rad_sw, const double *rad_lw, const aerobulk_gpu_series_ice_out *out,
                            int on_device);

/* Waits for the session stream and reports a deferred error (wind stress too strong). */
int aerobulk_gpu_synchronize(void);

/* ---- pinning helpers ------------------------------------------------------------------------------------ */
/* Page-lock / release an EXISTING host array (cudaHostRegister / cudaHostUnregister) so that callers that do not link
 * the CUDA runtime themselves (Fortran, ctypes ...) can give their fields the zero-copy path described at the top of
 * this file.  Register once, before the time loop; release before the array is freed.  Returns 0 or
 * AEROBULK_GPU_ERR_CUDA. */
int aerobulk_gpu_host_register(void *ptr, size_t bytes);
int aerobulk_gpu_host_unregister(void *ptr);
/* Self-test of the host copy threads used for PAGEABLE caller arrays (needs no device): copies n doubles through the
 * thread pool and back, `rounds` times; returns the number of rounds whose data came back changed (0 = pass). */
int aerobulk_gpu_selftest_host_copy(long long n, int rounds);
/* The row-block chunk plan aerobulk_gpu_model uses for n points (needs no device; for tests and tuning): kind 0 device or
 * pinned arrays (one chunk), 1 staged pipeline, 2 pageable arrays through the pinned slab.  Writes the nchunks + 1
 * boundaries into cstart (room for 17) and returns nchunks, or -1 for bad arguments.  kind 3: the staged pipeline of a
 * jt == 1 call (speculative AEROBULK_INIT: H2D and D2H overlap). */
int aerobulk_gpu_chunk_plan(long long n, int kind, long long *cstart);

/* ---- optional global flux diagnostics for sharded grids ---------------------------------------------- */
#define AEROBULK_GPU_NDIAG 19
/* Sum / min / max of the flux fields of this process's row block (any pointer may be NULL): stats[0] = number of points,
 * stats[1 + 3 f + {0,1,2}] = sum, min, max of field f in the order QL, QH, Tau_x, Tau_y, Evap, T_s (a skipped field
 * gives 0, +DBL_MAX, -DBL_MAX).  Deterministic (fixed-order) reduction on the device.  Ranks combine their vectors
 * element-wise with the operation aerobulk_gpu_diag_reduce_op(i) gives (0 sum, 1 min, 2 max): the one place a
 * collective (NCCL / MPI all-reduce of 19 doubles) appears besides the AEROBULK_INIT statistics below.  The reference
 * has no counterpart (its callers compute such diagnostics themselves). */
int aerobulk_gpu_flux_diagnostics(long long n, const double *QL, const double *QH, const double *Tau_x,
                                  const double *Tau_y, const double *Evap, const double *T_s, double *stats,
                                  int on_device);
int aerobulk_gpu_diag_reduce_op(int i);

/* ---- the reference's other two PUBLIC routines (src/mod_aerobulk.f90:20) ---------------------------------- */
/* AEROBULK_INIT (src/mod_aerobulk.f90:24-160) on HOST arrays, for callers that invoke it themselves: skin flag and its
 * two errors, nitend = Nt, the sanity mask, the humidity type and the unit checks -- with the reference's messages and
 * fail-stop.  As in the reference, AEROBULK_MODEL(jt == 1) runs the same initialisation again on its own arguments
 * (:255-262), so calling this first is never required.  rad_sw / rad_lw may be NULL (no radiation given). */
int aerobulk_gpu_init(int Nt, const char *calgo, int Ni, int Nj, const double *sst, const double *t_zt,
                      const double *hum_zt, const double *U_zu, const double *V_zu, const double *slp,
                      const int *l_use_skin, const double *rad_sw, const double *rad_lw);
/* AEROBULK_BYE (:162-170): prints the closing banner (AEROBULK_MODEL does it itself at jt == Nt). */
void aerobulk_gpu_bye(void);

/* ---- AEROBULK_INIT split for row-block sharded grids (one process per GPU) ---- */

#define AEROBULK_GPU_NSTATS 64
/* Field statistics of this rank's row block, DEVICE pointers (rad_lw may be NULL):
 * stats[0] = number of unmasked points, stats[1] = number of points, then for each
 * of the 9 checked fields f (sst,t_air,slp,u10,v10,wnd,hum,rad_lw-as-rad_sw,rad_lw;
 * mod_aerobulk.f90:143-153) 5 doubles at 2+5f: masked sum, masked min, masked max,
 * min, max.  Sums/counts combine by +, mins by min, maxes by max across ranks
 * (see aerobulk_gpu_stats_reduce_op). */
int aerobulk_gpu_init_local_stats(int Ni, int Nj, const double *sst, const double *t_zt, const double *hum_zt,
                                  const double *U_zu, const double *V_zu, const double *slp,
                                  const double *rad_lw, double *stats /* host, AEROBULK_GPU_NSTATS */);
/* 0: sum, 1: min, 2: max -- how stats[i] combines across ranks */
int aerobulk_gpu_stats_reduce_op(int i);
/* Runs AEROBULK_INIT's decisions (skin flag, nitend, humidity type, unit checks,
 * src/mod_aerobulk.f90:24-160) from globally reduced statistics.  After it, calls of
 * aerobulk_gpu_model*(jt==1, ...) on this rank skip their own local AEROBULK_INIT. */
int aerobulk_gpu_init_from_stats(int Nt, const char *calgo, const int *l_use_skin, int have_rad,
                                 const double *stats);

/* The same split WITHOUT a host round trip, for device-resident sessions (one collective, nothing copied to the host,
 * no synchronisation).  aerobulk_gpu_init_local_stats_device writes the row-block vector into DEVICE memory d_stats
 * (AEROBULK_GPU_NSTATS doubles) on the session stream.  The caller gathers the vectors of all ranks with ONE collective
 * (ncclAllGather / MPI_Allgather of 64 doubles per rank on that stream) into d_all[nranks][AEROBULK_GPU_NSTATS] and calls
 * aerobulk_gpu_init_from_gathered_stats: the argument-only decisions of AEROBULK_INIT (skin flag, nitend and their
 * errors) are taken at once; the statistics are combined in rank order and judged ON THE DEVICE (mask count, humidity
 * type, unit checks), and the flux kernels that follow read the verdict from device memory.  The host catches up -- and
 * raises an AEROBULK_INIT error with the reference's message -- at its next synchronisation (aerobulk_gpu_synchronize,
 * the jt == Nt call, any host-array call): the deferred-error rule the tau > 10 N/m^2 check already follows.  A kernel
 * launched after a failed device-side init computes nothing.  aerobulk_gpu_model_device(jt == 1) uses the same mechanism
 * on its own when the banners are off (aerobulk_gpu_set_verbose(0)). */
int aerobulk_gpu_init_local_stats_device(int Ni, int Nj, const double *sst, const double *t_zt, const double *hum_zt,
                                         const double *U_zu, const double *V_zu, const double *slp,
                                         const double *rad_lw, double *d_stats /* device, AEROBULK_GPU_NSTATS */);
int aerobulk_gpu_init_from_gathered_stats(int Nt, const char *calgo, const int *l_use_skin, int have_rad,
                                          const double *d_all /* device, [nranks][AEROBULK_GPU_NSTATS] */, int nranks);

/* ---- module globals of src/mod_const.f90:22-33 that callers may overwrite ------ */
void aerobulk_gpu_set_rdt(double rdt_seconds);   /* default 3600 */
void aerobulk_gpu_set_gdept(double depth_m);     /* default 1    */
void aerobulk_gpu_set_nb_iter(int nb_iter);      /* default 5    */
int aerobulk_gpu_get_nb_iter(void);
int aerobulk_gpu_get_use_skin(void);             /* sticky l_use_skin_schemes */
const char *aerobulk_gpu_get_humidity_type(void); /* "sh" | "rh" | "dp" */

/* ---- session plumbing ------------------------------------------------------ */
int aerobulk_gpu_set_device(int device);         /* default: $LOCAL_RANK or 0; before first compute call */
int aerobulk_gpu_get_device(void);
/* Multi-GPU inside ONE process (SURVEY.md 8b / 8e).  After aerobulk_gpu_set_devices(n), every host-array
 * AEROBULK_MODEL call (aerobulk_gpu_model, aerobulk_cxx_skin / _no_skin and the Fortran / C++ APIs on top of them) is
 * split by the library over GPUs device .. device+n-1: the flat point range of the caller's (Ni,Nj) fields is cut into
 * n contiguous shards (latitude row blocks, boundaries on multiples of 2048 points: aerobulk_gpu_shard_plan), each GPU
 * keeps the warm-layer state of its shard for the whole jt = 1..Nt session, and the field statistics AEROBULK_INIT needs
 * at jt == 1 (src/mod_aerobulk.f90:104-153) are combined over the shards inside the library.  Results are bit-identical
 * to the single-GPU call.  The caller still makes ONE call per time step, exactly as with the reference
 * (src/mod_aerobulk.f90:176-269).  Not combinable with aerobulk_gpu_set_stream; the device-pointer entry points and
 * the other entry points (turb, series, sea ice) stay on the first device.  n cannot change while a warm-layer session
 * is open.  aerobulk_gpu_get_state / _set_state gather / scatter the shards in point order. */
int aerobulk_gpu_set_devices(int n);             /* default 1 */
int aerobulk_gpu_get_devices(void);
/* The shard boundaries used for n points on n_dev devices (needs no device): writes the nshards + 1 boundaries into
 * start (room for 17) and returns nshards (<= n_dev: a tiny grid uses fewer devices), or -1 for bad arguments. */
int aerobulk_gpu_shard_plan(long long n, int n_dev, long long *start);
/* Run on a caller-owned cudaStream_t.  NULL selects the library's own non-blocking stream; to use the
 * legacy default stream pass cudaStreamLegacy ((cudaStream_t)0x1), cudaStreamPerThread is (cudaStream_t)0x2. */
int aerobulk_gpu_set_stream(void *cuda_stream);
/* 0: fail-stop like the reference (default), 1: return codes.  With return codes an error ENDS the session, as the
 * STOP of the reference ends the process: the warm-layer state is released and a skin flag set by the failed jt == 1
 * call is rolled back, so the next jt == 1 call starts clean (no aerobulk_gpu_reset needed). */
void aerobulk_gpu_set_error_mode(int return_codes);
/* Grouping of points of equal stability class into the same thread blocks (performance only; results
 * are bit-identical either way): 0 never, 1 (default) where it measured faster, 2 always. */
void aerobulk_gpu_set_sort(int mode);
void aerobulk_gpu_set_verbose(int on);           /* 1 (default): print the AeroBulk_init / _bye banners */
const char *aerobulk_gpu_last_error(void);
int aerobulk_gpu_last_error_code(void);
/* Drops every piece of session state (sticky globals, warm-layer arrays, buffers):
 * the equivalent of restarting the reference process. */
void aerobulk_gpu_reset(void);
/* The same for the reference-visible state only -- sticky nb_iter / skin flag / humidity type / nitend back to their
 * initial values, warm-layer arrays gone -- keeping the device buffers and this library's settings: what a program
 * that runs several independent AEROBULK_MODEL sessions in one process calls between them (the reference cannot:
 * its skin flag is sticky for the life of the process, src/mod_aerobulk.f90:74).  No device synchronisation. */
void aerobulk_gpu_new_session(void);

/* Persistent warm-layer state, device-resident between jt==1 and jt==Nt
 * (src/mod_skin_coare.f90:31-36, src/mod_skin_ecmwf.f90:52-55).
 * which: 0 dT_wl, 1 Hz_wl, 2 Qnt_ac, 3 Tau_ac of the COARE scheme while a COARE session is open, else dT_wl (0) and
 * the constant Hz_wl = 3 m (1) of the ECMWF scheme; 4 / 5 name the ECMWF pair explicitly (a COARE and an ECMWF session
 * can be open together, like the module arrays of the reference).  Returns the number of points copied (0 when the
 * state does not exist or n is not its size).
 * Restart protocol: the checkpoint holds the warm-layer arrays only.  The session globals set at jt == 1 (humidity type,
 * skin flag, nitend, nb_iter) are rebuilt by re-running the jt == 1 call with the step-1 inputs (or
 * aerobulk_gpu_init_from_stats), then aerobulk_gpu_set_state restores the arrays and the run continues at jt+1
 * (tests/test_gpu_checkpoint.py). */
long aerobulk_gpu_get_state(int which, double *host_out, long n);
long aerobulk_gpu_set_state(int which, const double *host_in, long n);

/* Fully asynchronous device-pointer calls (default off).  By default aerobulk_gpu_model_device synchronises at jt == Nt
 * (and at jt == 1 when the banners are on) so that a fail-stop caller sees every error before its session ends.  With
 * aerobulk_gpu_set_async(1) it never does: the caller collects deferred errors with aerobulk_gpu_synchronize(). */
void aerobulk_gpu_set_async(int on);

/* ---- measurement helpers --------------------------------------------------- */
/* CUDA events around every flux-kernel launch of aerobulk_gpu_model* on the stream it runs on (default off).
 * aerobulk_gpu_kernel_times waits for the stream, writes the durations [ms] of the launches recorded since the last call
 * (oldest first, at most max) and returns their number. */
void aerobulk_gpu_set_kernel_timing(int on);
int aerobulk_gpu_kernel_times(double *ms, int max);
/* Number of kernels this library has launched since load / reset of the counter. */
long aerobulk_gpu_launch_count(void);
void aerobulk_gpu_reset_launch_count(void);
/* Dependent-chain DFMA microbenchmark on the session device: returns FP64 FMA
 * instructions per second (all SMs), the denominator of the FP64 roofline. */
double aerobulk_gpu_measure_fp64_peak(void);
/* Algorithmic FP64-pipe work per point (SURVEY.md 8d: fx + nb_iter*it) and
 * algorithmic bytes per point for (algo, skin), of the FP64 calls.  A float32 call (aerobulk_gpu_model*_f32) does the
 * same work and moves half the per-point array bytes; these two functions do not describe it. */
double aerobulk_gpu_work_per_point(const char *calgo, int skin, int nb_iter);
double aerobulk_gpu_bytes_per_point(const char *calgo, int skin);
/* Resources of the flux kernel a call with (algo, skin, zt == zu) launches, on the session device: registers per thread,
 * local-memory (spill) bytes per thread, resident blocks per SM at the launch configuration (256 threads).  For reports
 * and regression tests: the skin kernels are built for 3 blocks/SM, the others for 4 (DESIGN.md 3.1).  0 on success.
 * It reports the FP64 kernel; the float32 twin a *_f32 call launches is listed in profiles/f32_kernels_r03b.txt. */
int aerobulk_gpu_kernel_info(const char *calgo, int skin, int zt_eq_zu, int *registers, int *local_bytes, int *blocks_per_sm);
const char *aerobulk_gpu_version(void);

/* ---- per-function probe (test support) ---------------------------------------
 * Evaluates ONE device building block of the hot path on n argument tuples (host arrays: args is
 * [nargs][n], argument-major; out is [n]) so that each can be checked against the CPU restatement of the
 * reference function it replaces.  func:
 *    1 e_sat(T)  2 q_sat(T,p)  3 Theta_from_z_P0_T_q(z,slp,T,q)  4 rho_air(T,q,p)  5 visc_air(T)  6 L_vap(T)
 *    7 cp_air(q)  8 gamma_moist(T,q)  9 alpha_sw(T)  10 qlw_net(rlw,Ts)  11 One_on_L(tha,qa,us,ts,qs)
 *    12 Ri_bulk(z,sst,tha,ssq,qa,ub)  13 q_air_rh(rh,T,p)  14 q_air_dp(dp,p)        (src/mod_phymbl.f90)
 *    20/21 psi_m/psi_h NCAR  22/23 COARE  24/25 ECMWF  26/27 ANDREAS  (zeta)
 *    30 z0tq_LKB(iflag,Rer,z0)  31 cd_n10_ncar(w)  32 charn_coare3p0(w)  33 charn_coare3p6(w)
 *    34 dT_cs of CS_COARE(alpha,Qsw,Qnsol,us,Qlat)  35 dT_cs of CS_ECMWF(alpha,Qsw,Qnsol,us)
 *    (21, 25 and 27 return NaN where the paired psi_m/psi_h evaluator the solvers use differs from the single psi_h)
 *    40 exp  41 exp10  42 log  43 atan  44 sqrt  45 x**-1/2  46 cbrt  47 x**-1/3  48 x**0.75  49 1/x  50 x**y
 *    51 atan(x), x >= 1  52 log10  53 exp, |x| <= 700  54 exp10, |x| <= 300
 *    60 e_sat_ice(T)  61 q_sat_ice(T,p)  62/63 psi_m_ice/psi_h_ice(zeta), |zeta| <= 50
 *    64/65 f_m_louis/f_h_louis(zu,Rib,Cxn,z0)  66 rough_leng_m(us,nu)
 *    67/68 z0t/z0q of rough_leng_tq(z0,us,nu), NaN where the reference stops  69 CdN10_f_LU13(A)
 *    70 CdN_f_LG15_light(LOG(10/z0w)/LOG(zu/z0w), A)          (src/ice/, SURVEY.md 8f row 4)
 * Returns 0, or an AEROBULK_GPU_ERR_* code. */
int aerobulk_gpu_probe(int func, long long n, int nargs, const double *args, double *out);

#ifdef __cplusplus
}
#endif
#endif /* AEROBULK_GPU_H */
