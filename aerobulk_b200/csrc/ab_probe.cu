// ab_probe.cu -- probe_kernel: evaluates ONE __device__ building block of ab_device.cuh / ab_ice.cuh / ab_math.cuh
// per launch on n argument tuples, so that every function of the hot path can be unit-tested on the GPU against the
// CPU restatement of the reference function it replaces (SURVEY.md 4: per-function unit tests; tests/test_gpu_functions.py,
// tests/test_gpu_ice_functions.py).  Test support inside the product library: nothing on the flux path calls it.
#include "ab_kernels.cuh"

namespace abk {

using namespace abd;

// args: [nargs][n] (argument-major, coalesced); out: [n]
__global__ void __launch_bounds__(256) probe_kernel(int func, long long n, int nargs, const double *args, double *out)
{
    abm::load_tables();
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    double a[6] = {0., 0., 0., 0., 0., 0.};
    for (int k = 0; k < nargs && k < 6; ++k) a[k] = args[(long long)k * n + i];
    double r = 0.;
    switch (func) {
    // ---- thermodynamics (src/mod_phymbl.f90), SURVEY 8a rows a4-a9
    case PROBE_E_SAT: r = e_sat(a[0]); break;
    case PROBE_Q_SAT: r = q_sat(a[0], a[1]); break;
    case PROBE_THETA: r = theta_from_z_P0_T_q(a[0], a[1], a[2], a[3]); break;
    case PROBE_RHO_AIR: r = rho_air(a[0], a[1], a[2]); break;
    case PROBE_VISC_AIR: r = visc_air(a[0]); break;
    case PROBE_L_VAP: r = L_vap(a[0]); break;
    case PROBE_CP_AIR: r = cp_air(a[0]); break;
    case PROBE_GAMMA_MOIST: r = gamma_moist(a[0], a[1]); break;
    case PROBE_ALPHA_SW: r = alpha_sw(a[0]); break;
    case PROBE_QLW_NET: r = qlw_net(a[0], a[1]); break;
    case PROBE_ONE_ON_L: r = one_on_L(a[0], a[1], a[2], a[3], a[4]); break;
    case PROBE_RI_BULK: r = ri_bulk(a[0], a[1], a[2], a[3], a[4], a[5]); break;
    case PROBE_Q_AIR_RH: r = q_air_rh(a[0], a[1], a[2]); break;
    case PROBE_Q_AIR_DP: r = q_air_dp(a[0], a[1]); break;
    // ---- stability functions, rows a15-a25 (the solvers call the one-sided evaluators; the sign selects the side
    //      exactly as `zstab = 0.5 + SIGN(0.5, zeta)` does in the reference)
    case PROBE_PSI_M_NCAR: r = psi_m_ncar(a[0]); break;
    case PROBE_PSI_H_NCAR:   // the solvers take psi_h(zeta_u) from the paired evaluator: NaN where it differs
        r = psi_h_ncar(a[0]);
        if (!nonneg(a[0]) && psi_mh_ncar_unstable(a[0]).h != r) r = nan("");
        break;
    case PROBE_PSI_M_COARE:
    case PROBE_PSI_H_COARE: {
        double m, h, ht;
        psi3_coare<false>(a[0], a[0], m, h, ht);
        r = (func == PROBE_PSI_M_COARE) ? m : ht;   // ht: the single-psi_h evaluator, h: the paired one (checked equal below)
        if (func == PROBE_PSI_H_COARE && h != ht) r = nan("");
        break;
    }
    case PROBE_PSI_M_ECMWF: r = nonneg(a[0]) ? psi_m_ecmwf_stable(a[0]) : psi_m_ecmwf_unstable(a[0]); break;
    case PROBE_PSI_H_ECMWF:
        r = nonneg(a[0]) ? psi_h_ecmwf_stable(a[0]) : psi_h_ecmwf_unstable(a[0]);
        if (!nonneg(a[0]) && psi_mh_ecmwf_unstable(a[0]).h != r) r = nan("");
        break;
    case PROBE_PSI_M_ANDREAS:
        r = nonneg(abm::dmin(a[0], 15.)) ? psi_m_andreas_stable(a[0]) : psi_mh_andreas_unstable(a[0]).m;
        break;
    case PROBE_PSI_H_ANDREAS:
        r = nonneg(abm::dmin(a[0], 15.)) ? psi_h_andreas_stable(a[0]) : psi_h_andreas_unstable(a[0]);
        if (!nonneg(abm::dmin(a[0], 15.)) && psi_mh_andreas_unstable(a[0]).h != r) r = nan("");
        break;
    // ---- roughness / neutral coefficients
    case PROBE_Z0TQ_LKB: {   // (iflag, Rer, z0) -> z0t or z0q; the device works in log space
        const double Rer = a[1], z0 = a[2];
        r = abm::dexp(log_z0tq_LKB((int)a[0], Rer, abm::dlog(abm::dmax(Rer, 1.E-300)), abm::dlog(z0)));
        break;
    }
    case PROBE_CD_N10_NCAR: r = cd_n10_ncar(a[0]); break;
    case PROBE_CHARN_COARE3P0: r = charn_coare3p0(a[0]); break;
    case PROBE_CHARN_COARE3P6: r = charn_coare3p6(a[0]); break;
    // ---- skin schemes: dT_cs of CS_COARE / CS_ECMWF (alpha, Qsw, Qnsol, u*, Qlat), rows a14, a20, a23
    case PROBE_CS_COARE: r = cool_skin_dT<true>(a[0], a[1], a[2], a[3], a[4]); break;
    case PROBE_CS_ECMWF: r = cool_skin_dT<false>(a[0], a[1], a[2], a[3], 0.); break;
    // ---- the kernels' own math (ab_math.cuh)
    case PROBE_EXP: r = abm::dexp(a[0]); break;
    case PROBE_EXP10: r = abm::dexp10(a[0]); break;
    case PROBE_LOG: r = abm::dlog(a[0]); break;
    case PROBE_ATAN: r = abm::datan(a[0]); break;
    case PROBE_SQRT: r = abm::fast_sqrt(a[0]); break;
    case PROBE_RSQRT: r = abm::fast_rsqrt(a[0]); break;
    case PROBE_CBRT: r = abm::fast_cbrt(a[0]); break;
    case PROBE_RCBRT: r = abm::fast_rcbrt(a[0]); break;
    case PROBE_POW075: r = abm::pow075(a[0]); break;
    case PROBE_RCP: r = abm::fast_rcp(a[0]); break;
    case PROBE_POWR: r = abm::dpowr(a[0], a[1]); break;
    case PROBE_ATAN_GE1: r = abm::datan_ge1(a[0]); break;
    case PROBE_LOG10: r = abm::dlog10(a[0]); break;
    case PROBE_EXP_B: r = abm::dexp_b(a[0]); break;
    case PROBE_EXP10_B: r = abm::dexp10_b(a[0]); break;
    // ---- sea ice (ab_ice.cuh)
    case PROBE_E_SAT_ICE: r = e_sat_ice(a[0]); break;
    case PROBE_Q_SAT_ICE: r = q_sat_ice(a[0], a[1]); break;
    case PROBE_PSI_M_ICE: r = psi_m_ice(a[0]); break;
    case PROBE_PSI_H_ICE: r = psi_h_ice(a[0]); break;
    case PROBE_F_M_LOUIS: r = f_m_louis(a[0], a[1], a[2], a[3]); break;
    case PROBE_F_H_LOUIS: r = f_h_louis(a[0], a[1], a[2], a[3]); break;
    case PROBE_ROUGH_LENG_M: r = rough_leng_m(a[0], a[1]); break;
    case PROBE_Z0T_AN87:
    case PROBE_Z0Q_AN87: {   // (z0, u*, nu) -> z0t or z0q as solve_ice computes them (log space); NaN where it sets `bad`
        double log_z0t, log_z0q;
        bool bad = false;
        log_rough_leng_tq(a[0], abm::dlog(a[0]), a[1], a[2], log_z0t, log_z0q, bad);
        r = bad ? nan("") : abm::dexp(func == PROBE_Z0T_AN87 ? log_z0t : log_z0q);
        break;
    }
    case PROBE_CDN10_LU13: r = CdN10_f_LU13(a[0]); break;
    case PROBE_CDN_LG15: r = CdN_f_LG15_light(a[0], a[1]); break;   // (LOG(10/z0w) / LOG(zu/z0w), A)
    default: r = nan(""); break;
    }
    out[i] = r;
}

cudaError_t launch_probe(int func, long long n, int nargs, const double *args, double *out, cudaStream_t s)
{
    if (n <= 0) return cudaSuccess;
    probe_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(func, n, nargs, args, out);
    return cudaGetLastError();
}

}  // namespace abk
