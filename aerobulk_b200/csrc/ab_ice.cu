// ab_ice.cu -- sea-ice kernels for sm_100a (SURVEY.md 8f row 4).
//
//   ice_turb_kernel<IALGO,ZTEQ>  one TURB_ICE_* call (src/ice/mod_blk_ice_{nemo,easy,an05,lu12,lg15,lg15_io}.f90).
//   ice_flux_kernel<IALGO,ZTEQ>  the over-ice half of src/ice/test_aerobulk_oce+ice.f90:225-412 fused per point:
//       humidity conversion, siq = q_sat(SIT, l_ice), theta_zt = t_zt + gamma_moist zt, TURB_ICE_*, Ri_b, t_zu,
//       rho_zu, BULK_FORMULA(l_ice=.TRUE.).
//   leads_kernel<OALGO,ZTEQ>     the over-water half (:297-304): TURB_<ocean algorithm> without skin + BULK_FORMULA,
//       and the area-weighted cell means A ice + (1-A) water.
// Same shape as the flux kernels: one thread per point, everything in registers, 256 x 3 blocks per SM.
#include "ab_kernels.cuh"

namespace abk {

using namespace abd;

static constexpr int ICE_BLOCK = 256;
static constexpr int ICE_MIN_BLOCKS = 3;

template <int IALGO, bool ZTEQ>
__global__ void __launch_bounds__(ICE_BLOCK, ICE_MIN_BLOCKS) ice_turb_kernel(const IceTurbArgs a)
{
    abm::load_tables<abm::PSI_TABLES_NONE>();
    const long long i = (long long)blockIdx.x * ICE_BLOCK + threadIdx.x;
    if (i >= a.n) return;
    double fr = 0., frf = 0.;
    if (IALGO == ICE_LU12) fr = __ldg(a.frice + i);
    if (IALGO == ICE_LG15) frf = __ldg(a.frice + (a.form_index >= 0 ? a.form_index : i));
    const IceOut o = solve_ice<IALGO, ZTEQ>(a.u, __ldg(a.Ts_i + i), __ldg(a.t_zt + i), __ldg(a.qs_i + i), __ldg(a.q_zt + i),
                                            __ldg(a.U_zu + i), fr, frf);
    if (IALGO == ICE_AN05 && o.bad) atomicMin(a.bad_rough, (unsigned long long)i);
    a.Cd[i] = o.Cd; a.Ch[i] = o.Ch; a.Ce[i] = o.Ce;
    a.t_zu[i] = o.t_zu; a.q_zu[i] = o.q_zu; a.Ubzu[i] = o.Ub;
    const double v[8] = {o.CdN, o.ChN, o.CeN, o.z0, o.us, o.L, o.UN10, o.CdN_frm};
#pragma unroll
    for (int k = 0; k < 8; ++k)
        if (a.opt[k]) a.opt[k][i] = v[k];
}

__device__ __forceinline__ double humidity_to_q(int kind, double hum, double T, double slp)
{
    if (kind == 2) return q_air_rh(hum, T, slp);
    if (kind == 1) return q_air_dp(hum, slp);
    return hum;
}

template <int IALGO, bool ZTEQ>
__global__ void __launch_bounds__(ICE_BLOCK, ICE_MIN_BLOCKS) ice_flux_kernel(const OceIceArgs a)
{
    abm::load_tables<abm::PSI_TABLES_NONE>();
    const long long i = (long long)blockIdx.x * ICE_BLOCK + threadIdx.x;
    if (i >= a.n) return;
    const double sit = __ldg(a.sit + i), T = __ldg(a.t_zt + i), slp = __ldg(a.slp + i), wnd = __ldg(a.wnd + i);
    const double q = humidity_to_q(a.hum_kind, __ldg(a.hum_zt + i), T, slp);
    const double siq = q_sat_ice(sit, slp);
    const double tha = T + gamma_moist(T, q) * a.ui.zt;
    double fr = 0., frf = 0.;
    if (IALGO == ICE_LU12) fr = __ldg(a.frice + i);
    if (IALGO == ICE_LG15) frf = __ldg(a.frice + (a.form_index >= 0 ? a.form_index : i));
    const IceOut o = solve_ice<IALGO, ZTEQ>(a.ui, sit, tha, siq, q, wnd, fr, frf);
    if (IALGO == ICE_AN05 && o.bad) atomicMin(a.bad_rough, (unsigned long long)i);

    double tz = o.t_zu;
#pragma unroll 1
    for (int jq = 0; jq < 4; ++jq) tz = o.t_zu - gamma_moist(0.5 * (tz + sit), o.q_zu) * a.ui.zu;
    double rho = rho_air(tz, o.q_zu, slp);
    rho = rho_air(tz, o.q_zu, slp - rho * GRAV * a.ui.zu);
    // BULK_FORMULA_SCLR with l_ice, mod_phymbl.f90:1149-1203
    const AirZu air = air_at_zu(a.ui.zu, o.t_zu, o.q_zu, slp);
    const double Urho = o.Ub * air.rho1;
    const double tau = Urho * o.Cd * wnd;
    const double evap = Urho * o.Ce * (o.q_zu - siq);
    const double qsen = Urho * o.Ch * (o.t_zu - sit) * air.cp;
    const double qlat = RLSUB * evap;
    const double ev = abm::dmin(evap, 0.);
    if (tau > 10.) atomicMin(a.bad_tau, (unsigned long long)i);
    const double v[17] = {o.Cd, o.Ch, o.Ce, o.t_zu, o.q_zu, tz, o.Ub, ri_bulk(a.ui.zu, sit, o.t_zu, siq, o.q_zu, o.Ub),
                          o.z0, o.us, o.L, o.UN10, rho, tau, qsen, qlat, ev};
#pragma unroll
    for (int k = 0; k < 17; ++k)
        if (a.out[k]) a.out[k][i] = v[k];
    if (a.ice_flux[0] && a.ice_flux[0] != a.out[13]) a.ice_flux[0][i] = tau;
    if (a.ice_flux[1] && a.ice_flux[1] != a.out[14]) a.ice_flux[1][i] = qsen;
    if (a.ice_flux[2] && a.ice_flux[2] != a.out[15]) a.ice_flux[2][i] = qlat;
    if (a.ice_flux[3] && a.ice_flux[3] != a.out[16]) a.ice_flux[3][i] = ev;
}

// One record of the sea-ice station series (src/ice/test_aerobulk_buoy_series_ice.f90:326-470): RiB at zt and the net
// solar flux for every record; TURB_ICE_*, RiB at zu, BULK_FORMULA(l_ice), net long-wave and non-solar flux only where
// the ice concentration exceeds 0.01 (:388) -- the other records read 0 (the program leaves them unset).  The program's
// arrays are 1 x 1, so the LG15 form drag follows the record's own concentration.
template <int IALGO, bool ZTEQ>
__global__ void __launch_bounds__(ICE_BLOCK, ICE_MIN_BLOCKS) ice_series_kernel(const IceSeriesArgs a)
{
    abm::load_tables<abm::PSI_TABLES_NONE>();
    const long long i = (long long)blockIdx.x * ICE_BLOCK + threadIdx.x;
    if (i >= a.n) return;
    const double sit = __ldg(a.sit + i), T = __ldg(a.t_zt + i), slp = __ldg(a.slp + i), wnd = __ldg(a.wnd + i);
    const double sic = __ldg(a.sic + i);
    const double q = humidity_to_q(a.hum_kind, __ldg(a.hum_zt + i), T, slp);
    const double siq = q_sat_ice(sit, slp);
    const double tha = T + gamma_moist(T, q) * a.ui.zt;
    double v[NICESERIES_OUT];
#pragma unroll
    for (int k = 0; k < NICESERIES_OUT; ++k) v[k] = 0.;
    v[12] = ri_bulk(a.ui.zt, sit, tha, siq, q, abm::dmax(wnd, WSPD_THRSHLD_ICE));   // :380
    v[5] = (1. - RICE_ALB0) * __ldg(a.rad_sw + i);                                  // :384
    if (sic > 0.01) {
        const IceOut o = solve_ice<IALGO, ZTEQ>(a.ui, sit, tha, siq, q, wnd, sic, sic);
        if (IALGO == ICE_AN05 && o.bad) atomicMin(a.bad_rough, (unsigned long long)i);
        // BULK_FORMULA_SCLR with l_ice, pEvap, prhoa: mod_phymbl.f90:1149-1203
        const AirZu air = air_at_zu(a.ui.zu, o.t_zu, o.q_zu, slp);
        const double Urho = o.Ub * air.rho1;
        const double tau = Urho * o.Cd * wnd;
        const double evap = Urho * o.Ce * (o.q_zu - siq);
        const double qsen = Urho * o.Ch * (o.t_zu - sit) * air.cp;
        const double qlat = RLSUB * evap;
        if (tau > 10.) atomicMin(a.bad_tau, (unsigned long long)i);
        const double t2 = sit * sit;
        const double qlw = EMISS_I * (__ldg(a.rad_lw + i) - STEFAN * t2 * t2);      // qlw_net(l_ice), :1306-1312
        v[0] = air.rho; v[1] = qlat; v[2] = qsen; v[3] = qlw; v[4] = qsen + qlat + qlw; v[6] = tau; v[7] = abm::dmin(evap, 0.);
        v[8] = o.Cd; v[9] = o.Ch; v[10] = o.Ce; v[11] = o.z0;
        v[13] = ri_bulk(a.ui.zu, sit, o.t_zu, siq, o.q_zu, o.Ub);
        v[14] = o.CdN; v[15] = o.us; v[16] = o.L; v[17] = o.UN10; v[18] = o.t_zu; v[19] = o.q_zu; v[20] = o.Ub;
    }
#pragma unroll
    for (int k = 0; k < NICESERIES_OUT; ++k)
        if (a.out[k]) a.out[k][i] = v[k];
}

template <int OALGO, bool ZTEQ>
__global__ void __launch_bounds__(ICE_BLOCK, ICE_MIN_BLOCKS) leads_kernel(const OceIceArgs a)
{
    abm::load_tables<PSI_TABLES_OF<OALGO>>();
    const long long i = (long long)blockIdx.x * ICE_BLOCK + threadIdx.x;
    if (i >= a.n) return;
    const double sst = __ldg(a.sst + i), T = __ldg(a.t_zt + i), slp = __ldg(a.slp + i), wnd = __ldg(a.wnd + i);
    const double q = humidity_to_q(a.hum_kind, __ldg(a.hum_zt + i), T, slp);
    PointIn p;
    p.sst = sst;
    p.ssq = RDCT_QSAT_SALT * q_sat(sst, slp);
    p.theta_zt = T + gamma_moist(T, q) * a.uo.zt;
    p.q_zt = q;
    p.wnd = wnd;
    p.slp = slp;
    p.Qsw = 0.; p.rlw = 0.; p.lon = 0.; p.has_lon = false;
    WarmLayer wl = {0., 0., 0., 0.};
    Diag dg;
    const Coeffs c = solve_ocean<OALGO, false, false, ZTEQ>(a.uo, p, wl, dg);
    const AirZu air = air_at_zu(a.uo.zu, c.t_zu, c.q_zu, slp);
    const Flux f = bulk_formula(air, sst, p.ssq, c.t_zu, c.q_zu, c.Cd, c.Ch, c.Ce, wnd, c.Ub);
    if (f.tau > 10.) atomicMin(a.bad_tau, (unsigned long long)i);
    const double A = __ldg(a.frice + i);
    const double v[18] = {c.Cd, c.Ch, c.Ce, c.t_zu, c.q_zu, c.Ub, dg.z0, dg.us, dg.L, dg.UN10, f.tau, f.qsen, f.qlat, f.evap,
                          A * a.ice_flux[0][i] + (1. - A) * f.tau, A * a.ice_flux[1][i] + (1. - A) * f.qsen,
                          A * a.ice_flux[2][i] + (1. - A) * f.qlat, A * a.ice_flux[3][i] + (1. - A) * f.evap};
#pragma unroll
    for (int k = 0; k < 18; ++k)
        if (a.out[17 + k]) a.out[17 + k][i] = v[k];
}

// The instantiation a sea-ice launch runs: f(IALGO, ZTEQ) with std::integral_constant arguments, nullptr for an unknown
// algorithm.
template <class F>
static auto pick_ice(int ialgo, bool zteq, F f) -> decltype(f(IntC<ICE_NEMO>{}, BoolC<false>{}))
{
    const auto z = [&](auto I) { return zteq ? f(I, BoolC<true>{}) : f(I, BoolC<false>{}); };
    switch (ialgo) {
    case ICE_NEMO: return z(IntC<ICE_NEMO>{});
    case ICE_EASY: return z(IntC<ICE_EASY>{});
    case ICE_AN05: return z(IntC<ICE_AN05>{});
    case ICE_LU12: return z(IntC<ICE_LU12>{});
    case ICE_LG15: return z(IntC<ICE_LG15>{});
    default: return nullptr;
    }
}

// every launch of this file: nothing to do for n <= 0 (whatever the algorithm), else one thread per point
template <class Args>
static cudaError_t launch_ice(void (*k)(Args), const Args &a, cudaStream_t s)
{
    if (a.n <= 0) return cudaSuccess;
    if (!k) return cudaErrorInvalidValue;
    k<<<(unsigned)((a.n + ICE_BLOCK - 1) / ICE_BLOCK), ICE_BLOCK, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_ice_turb(int ialgo, bool zteq, const IceTurbArgs &a, cudaStream_t s)
{
    return launch_ice(pick_ice(ialgo, zteq, [](auto I, auto Z) { return ice_turb_kernel<I(), Z()>; }), a, s);
}

cudaError_t launch_ice_flux(int ialgo, bool zteq, const OceIceArgs &a, cudaStream_t s)
{
    return launch_ice(pick_ice(ialgo, zteq, [](auto I, auto Z) { return ice_flux_kernel<I(), Z()>; }), a, s);
}

// the sea-ice station series has no EASY: ice_series_kernel<ICE_EASY, *> is never built
cudaError_t launch_ice_series(int ialgo, bool zteq, const IceSeriesArgs &a, cudaStream_t s)
{
    return launch_ice(pick_ice(ialgo, zteq, [](auto I, auto Z) -> void (*)(IceSeriesArgs) {
                          if constexpr (I() == ICE_EASY) return nullptr;
                          else return ice_series_kernel<I(), Z()>;
                      }), a, s);
}

// the leads run the ocean algorithm without skin
cudaError_t launch_leads(int oalgo, bool zteq, const OceIceArgs &a, cudaStream_t s)
{
    return launch_ice(pick_ocean(oalgo, false, zteq, [](auto A, auto, auto Z) { return leads_kernel<A(), Z()>; }), a, s);
}

}  // namespace abk
