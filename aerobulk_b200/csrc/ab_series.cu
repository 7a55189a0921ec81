// ab_series.cu -- station time series on sm_100a (SURVEY.md 8f row 3).
//
// series_kernel<ALGO,SKIN,ZTEQ>: one thread per station runs the whole time loop of the reference's
// buoy-series program (src/tests/test_aerobulk_buoy_series_oce.f90:364-537): per record the humidity conversion
// (:220-236), theta_zt = t_zt + gamma_moist*zt (:399), ssq (:413), Qsw (:447), TURB_<algo> with kt = record number
// (:450-491), then dT, t_zu (4 lapse-rate passes, :499-503), RiB (:506), BULK_FORMULA (:509-512), Qlw, QNS (:515-518).
// The time recursion of the warm layer is sequential per station, so the parallelism is across stations only; the
// warm-layer state never leaves the registers between records and there is one launch for the whole series instead
// of Nt.  Small blocks (64 threads) spread few stations over many SMs; 8 blocks per SM (16 warps, <= 128 registers)
// measured best over 64x1 / 64x8 / 64x12 / 128x6 both for one station (latency: 60 us per record at nb_iter = 20) and
// for 300 k stations, profiles/series_bench_r01i.txt.
#include "ab_kernels.cuh"

namespace abk {

using namespace abd;

#ifndef AB_SERIES_BLOCK
#define AB_SERIES_BLOCK 64
#endif
#ifndef AB_SERIES_MIN_BLOCKS
#define AB_SERIES_MIN_BLOCKS 8
#endif
static constexpr int SERIES_BLOCK = AB_SERIES_BLOCK;
static constexpr int SERIES_MIN_BLOCKS = AB_SERIES_MIN_BLOCKS;

template <int ALGO, bool SKIN, bool ZTEQ>
__global__ void __launch_bounds__(SERIES_BLOCK, SERIES_MIN_BLOCKS) series_kernel(const SeriesArgs a)
{
    abm::load_tables();
    const long long s = (long long)blockIdx.x * SERIES_BLOCK + threadIdx.x;
    if (s >= a.S) return;
    const double lon = __ldg(a.lon + s);
    WarmLayer wl = {0., 0., 0., 0.};
    if (SKIN) wl.Hz = (ALGO == ECMWF) ? 3. : 20.;     // *_INIT at kt == nit000
    Uniform u = a.u;
    u.dawn = 0;

#pragma unroll 1
    for (int jt = 0; jt < a.Nt; ++jt) {
        const long long i = (long long)jt * a.S + s;
        const double sst = __ldg(a.sst + i), T = __ldg(a.t_zt + i), hum = __ldg(a.hum_zt + i);
        const double wnd = __ldg(a.wnd + i), slp = __ldg(a.slp + i);
        const double rsw = __ldg(a.rad_sw + i), rlw = __ldg(a.rad_lw + i);
        u.isd = __ldg(a.isd + jt);

        double q = hum;
        if (a.hum_kind == 2) q = q_air_rh(abm::dmin(99.999, hum), T, slp);
        else if (a.hum_kind == 1) q = q_air_dp(hum, slp);

        PointIn p;
        p.sst = sst;
        p.q_zt = q;
        p.theta_zt = T + gamma_moist(T, q) * u.zt;
        p.ssq = RDCT_QSAT_SALT * q_sat(sst, slp);
        p.wnd = wnd;
        p.slp = slp;
        p.Qsw = (1. - ROCE_ALB0) * rsw;
        p.rlw = rlw;
        p.lon = lon;
        p.has_lon = true;

        Diag dg;
        dg.dT_cs = 0.;
        const Coeffs c = solve_ocean<ALGO, SKIN, SKIN, ZTEQ>(u, p, wl, dg);
        const double Ts = SKIN ? c.Ts : sst;
        const double qs = SKIN ? c.qs : p.ssq;

        double t_zu = c.t_zu;
#pragma unroll 1
        for (int jq = 0; jq < 4; ++jq) t_zu = c.t_zu - gamma_moist(t_zu, c.q_zu) * u.zu;
        const double rib = ri_bulk(u.zu, Ts, c.t_zu, qs, c.q_zu, c.Ub);
        const AirZu air = air_at_zu(u.zu, c.t_zu, c.q_zu, slp);
        const Flux f = bulk_formula(air, Ts, qs, c.t_zu, c.q_zu, c.Cd, c.Ch, c.Ce, wnd, c.Ub);
        if (f.tau > 10.) atomicMin(a.bad_index, (unsigned long long)i);   // BULK_FORMULA_VCTR, mod_phymbl.f90:1250-1253
        const double qlw = qlw_net(rlw, Ts);

        const double v[NSERIES_OUT] = {air.rho, f.qlat, f.qsen, qlw, f.qsen + f.qlat + qlw, p.Qsw,
                                       SKIN ? dg.dT_cs : 0., SKIN ? wl.dT : 0., f.tau, Ts - sst, SKIN ? wl.Hz : 0.,
                                       (SKIN && ALGO != ECMWF) ? wl.Qac : 0., (SKIN && ALGO != ECMWF) ? wl.Tac : 0.,
                                       c.Cd, c.Ce, c.Ch, c.t_zu, c.q_zu, t_zu, rib, dg.z0, dg.us, dg.L, dg.UN10, Ts,
                                       f.evap, q, p.theta_zt};
#pragma unroll
        for (int k = 0; k < NSERIES_OUT; ++k)
            if (a.out[k]) a.out[k][i] = v[k];
    }
}

cudaError_t launch_series(int algo, bool skin, bool zteq, const SeriesArgs &a, cudaStream_t s)
{
    const auto k = pick_ocean(algo, skin, zteq, [](auto A, auto S, auto Z) { return series_kernel<A(), S(), Z()>; });
    if (!k) return cudaErrorInvalidValue;
    if (a.S <= 0 || a.Nt <= 0) return cudaSuccess;
    k<<<(unsigned)((a.S + SERIES_BLOCK - 1) / SERIES_BLOCK), SERIES_BLOCK, 0, s>>>(a);
    return cudaGetLastError();
}

}  // namespace abk
