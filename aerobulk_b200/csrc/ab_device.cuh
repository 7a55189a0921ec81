// ab_device.cuh -- FP64 __device__ physics of the aerobulk_model hot path for sm_100a.
//
// Everything a grid point needs, register-resident: marine-boundary-layer
// thermodynamics (reference src/mod_phymbl.f90), the Monin-Obukhov stability
// functions and first guess (src/mod_common_coare.f90, src/mod_blk_*.f90), the
// cool-skin / warm-layer schemes (src/mod_skin_coare.f90, src/mod_skin_ecmwf.f90)
// and the five iterative solvers.  Written for the GPU, not transliterated:
//   * only the selected side of every `zstab*A + (1-zstab)*B` blend is evaluated
//     (same value: the unused side is finite by construction in the reference);
//   * loop invariants are hoisted (e_sat(T) out of the barometric loop,
//     alpha_sw(SST) and the Saunders constants out of the cool-skin loop, the
//     warm-layer "mess-o-constants" out of the bulk iteration, log(zu) & co. to
//     the host);
//   * `x**y` uses sqrt/cbrt/exp10 or exp(y*log x) instead of the ~90-instruction
//     pow(): a few ulp away from glibc, far inside the 1e-10 parity tolerance;
//   * FMA contraction is on.
// The reference's quirks (truncated literals 1.7320508/.3333/0.6667, grav=9.8 vs
// 9.80665 in rcst_cs, rt0 in e_sat, MOD(nb_iter,jit) commit rule, ECMWF warm layer
// stepping every iteration ...) are kept: they are part of the numbers.
#pragma once

#include <cuda_runtime.h>
#include <math.h>

#include "ab_math.cuh"

namespace abd {

#define ABD __device__ __forceinline__

// FP64 literals in the constant bank.  ptxas builds a double that does not fit a 32-bit immediate with two moves
// (UMOV / IMAD.MOV): ~20 % of the instructions the COARE + skin kernel executed in the round-1b profile.  KC(x) puts
// the value of the constant expression x into a __constant__ variable (one per distinct bit pattern; adjacent ones are
// fetched in pairs by LDCU.128) -- doubles whose low word is zero (0.5, 16., 1.25 ...) stay immediates.
// Wrap a WHOLE constant sub-expression, e.g. KC(1. / 0.014): the compiler cannot fold across a memory operand.
template <unsigned long long B>
static __constant__ double kc_bank = __builtin_bit_cast(double, B);
template <unsigned long long B>
__device__ __forceinline__ double kc_value()
{
    if constexpr ((B & 0xffffffffull) == 0ull) return __builtin_bit_cast(double, B);
    else return kc_bank<B>;
}
#define KC(x) (::abd::kc_value<__builtin_bit_cast(unsigned long long, static_cast<double>(x))>())

// ---------------------------------------------------------------------------
// constants, reference src/mod_const.f90:38-120 (derived ones folded in FP64
// operation by operation, as gfortran does for PARAMETERs)
// ---------------------------------------------------------------------------
constexpr double GRAV = 9.8;
constexpr double RPI = 3.141592653589793;
constexpr double ROCE_ALB0 = 0.066;
constexpr double EMISS_W = 0.98;
constexpr double STEFAN = 5.67E-8;
constexpr double RT0 = 273.15;
constexpr double RCP0_W = 4190.;
constexpr double RHO0_W = 1025.;
constexpr double RNU0_W = 1.e-6;
constexpr double RK0_W = 0.6;
constexpr double RCP_DRY = 1005.0;
constexpr double RCP_VAP = 1860.0;
constexpr double R_DRY = 287.05;
constexpr double R_VAP = 461.495;
constexpr double R_GAS = 8.314510;
constexpr double RMM_DRYAIR = 28.9647e-3;
constexpr double RMM_WATER = 18.0153e-3;
constexpr double RLEVAP = 2.46e+6;
constexpr double VKARMN = 0.4;
constexpr double VKARMN2 = 0.4 * 0.4;
constexpr double RDCT_QSAT_SALT = 0.98;
constexpr double Z0_SEA_MAX = 0.0025;
constexpr double CX_MIN = 0.1E-3;
constexpr double REF_TAU_MAX = 10.;
constexpr double RPOISS_DRY = R_DRY / RCP_DRY;
constexpr double RGAMMA_DRY = GRAV / RCP_DRY;
constexpr double REPS0 = R_DRY / R_VAP;
constexpr double RCTV0 = R_VAP / R_DRY - 1.;
constexpr double RCST_CS = -16. * 9.80665 * RHO0_W * RCP0_W * RNU0_W * RNU0_W * RNU0_W / (RK0_W * RK0_W);
constexpr double SQ_RADRW = 0x1.184c0ffddaa3cp-5;    // SQRT(1.2/1025.)           mod_const.f90:112
constexpr double RCP0W_POW15 = 0x1.08dce4ef23084p+18; // 4190.**1.5               mod_skin_coare.f90:156
constexpr double FLA_ECMWF = 0x1.1d9fee00723a0p+1;   // MAX(0.3**(-2./3.),1.)     mod_skin_ecmwf.f90:183-185
constexpr double SR3 = 0x1.bb67ae8584caap+0;         // SQRT(3.)                  mod_blk_andreas.f90:325
constexpr double SR5 = 0x1.1e3779b97f4a8p+1;         // SQRT(5.)                  mod_blk_andreas.f90:381
constexpr double ZBM_A = 5. / 6.5;                   // b_m                       mod_blk_andreas.f90:322
constexpr double ZBBM_A = 0x1.56bfea66ef78dp-1;      // ABS((1-b_m)/b_m)**(1/3)   mod_blk_andreas.f90:345

enum Algo { COARE3P0 = 1, COARE3P6 = 2, NCAR = 3, ECMWF = 4, ANDREAS = 5 };
// the psi tables an algorithm's solver reads (abm::load_tables<PSI_TABLES_OF<ALGO>>()); ECMWF starts from the COARE first
// guess, NCAR and ANDREAS read none.  A kernel that reads a table it does not load computes garbage: -Xptxas -v shows which tables a kernel's shared
// memory holds (7.7 KB without psi tables, 9.75 KB more per family)
template <int ALGO>
constexpr int PSI_TABLES_OF = (ALGO == COARE3P0 || ALGO == COARE3P6) ? abm::PSI_TABLES_COARE
                              : (ALGO == ECMWF)                      ? abm::PSI_TABLES_ALL
                                                                     : abm::PSI_TABLES_NONE;

// ---------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------
// SIGN(MIN(ABS(x),lim),x) and SIGN(MAX(ABS(x),lo),x)
ABD double clip_abs(double x, double lim) { return (fabs(x) <= lim) ? x : copysign(lim, x); }
ABD double floor_abs(double x, double lo) { return (fabs(x) >= lo) ? x : copysign(lo, x); }
// x**y for x >= 0 (0**y = 0 for y > 0); own exp/log/atan with constant-bank tables, see ab_math.cuh
ABD double powr(double x, double y) { return abm::dpowr(x, y); }
// zstab = 0.5 + SIGN(0.5, x) is 1 unless the sign bit of x is set
ABD bool nonneg(double x) { return !signbit(x); }
// a / b for normal-range operands: a * (1/b) with the reciprocal from MUFU.RCP64H + one refinement (<= 1.5 ulp; a
// residual correction to <= 1 ulp cost two more FP64 instructions per quotient, 5 % of the kernel's FP64 work, for
// nothing the 1e-10 parity metric can see).  CUDA's IEEE division spends as many non-FP64 instructions on its
// special-case guard as FP64 ones on the quotient; the physics never feeds it denormals, infinities or zero denominators.
ABD double fdiv(double a, double b) { return a * abm::fast_rcp(b); }
// natural logs of literals of the reference (glibc values), for roughness lengths handled in log space
constexpr double LOG_1EM9 = -0x1.4b927f32bffb8p+4;   // LOG(1.E-9)
constexpr double LOG_1EM8 = -18.420680743952367;     // LOG(1.E-8)
constexpr double LOG_0P05 = -0x1.7f7427b73e391p+1;   // LOG(0.05)
constexpr double LOG_1P6EM4 = -0x1.17b0d6ae41bdfp+3, LOG_5P8EM5 = -0x1.3829836acdc7ap+3;   // COARE 3.6 z0t
constexpr double LOG_1P1EM4 = -0x1.23ae53cc2dc88p+3, LOG_5P5EM5 = -0x1.39dc96cb28027p+3;   // COARE 3.0 z0t
constexpr double LOG_0P40 = -0x1.d5240f0e0e077p-1, LOG_0P62 = -0x1.e982378d782aap-2;       // ECMWF alpha_H, alpha_Q
constexpr double LOG_1EM3 = -0x1.ba18a998fffa0p+2;   // LOG(0.001)
constexpr double LOG_Z0_SEA_MAX = -0x1.7f7427b73e391p+2;   // LOG(0.0025)
constexpr double INV_VKARMN = 1. / VKARMN;
constexpr double INV_GRAV = 1. / GRAV;

// ---------------------------------------------------------------------------
// thermodynamics, reference src/mod_phymbl.f90
// ---------------------------------------------------------------------------
ABD double virt_temp(double T, double q) { return T * (1. + KC(RCTV0) * q); }           // :247-269

// Goff (1957) saturation vapour pressure [Pa], :777-800 (rt0, not the triple point)
ABD double e_sat_goff(double T)
{
    const double zta = abm::dmax(T, 180.);
    const double ztmp = fdiv(KC(RT0), zta);
    const double r = zta * KC(1. / RT0);
    const double a = KC(10.79574) * (1. - ztmp) - KC(5.028) * abm::dlog10(r)
                     + KC(1.50475 * 1.e-4) * (1. - abm::dexp10_b(KC(-8.2969) * (r - 1.)))
                     + KC(0.42873 * 1.e-3) * (abm::dexp10_b(KC(4.76955) * (1. - ztmp)) - 1.) + KC(0.78614);
    return 100. * abm::dexp10_b(a);   // T is floored at 180 K: every exponent of this function is inside [-4, 4]
}
// On [230, 330) K, every temperature of the ocean path, the same function from a piecewise polynomial
// (abm::esat_table, within 2 ulp of the formula; ~25 instructions instead of ~115); elsewhere, and for NaN, the formula.
ABD double e_sat(double T) { return (T >= 230. && T < 330.) ? abm::esat_table(T) : e_sat_goff(T); }
ABD double q_sat_from_e(double es, double p) { return fdiv(KC(REPS0) * es, p - KC(1. - REPS0) * es); }  // :903
ABD double q_sat(double T, double p) { return q_sat_from_e(e_sat(T), p); }                   // :881-904

// Theta_from_z_P0_T_q, :283-318 + :163-187 + :343-365; e_sat(T) is loop-invariant
ABD double theta_from_z_P0_T_q(double z, double slp, double T, double q)
{
    const double es = e_sat(T);
    double pa = slp;
#pragma unroll
    for (int it = 0; it < 3; ++it) {
        const double f = fdiv(q, q_sat_from_e(es, pa));
        const double xm = (1. - f) * RMM_DRYAIR + f * RMM_WATER;
        pa = slp * abm::dexp_b(fdiv(-GRAV * xm * z, R_GAS * T));
    }
    return T * powr(fdiv(slp, pa), RPOISS_DRY);
}

ABD double rho_air(double T, double q, double p) { return abm::dmax(fdiv(p, R_DRY * T * (1. + RCTV0 * q)), 0.8); }  // :522-537
ABD double visc_air(double T)                                                                              // :549-563
{
    const double tc = T - RT0, tc2 = tc * tc;
    return KC(1.326e-5) * (1. + KC(6.542E-3) * tc + KC(8.301e-6) * tc2 - KC(4.84e-9) * tc2 * tc);
}
ABD double L_vap(double T) { return (KC(2.501) - KC(0.00237) * (T - KC(RT0))) * 1.e6; }                               // :579-592
ABD double cp_air(double q) { return KC(RCP_DRY) + KC(RCP_VAP) * q; }                                             // :603-616
// moist adiabatic lapse rate [K/m], :627-649
ABD double gamma_moist(double T, double q)
{
    const double ta = abm::dmax(T, 180.);
    const double qa = abm::dmax(q, 1.E-6);
    const double wa = fdiv(qa, 1. - qa);
    const double iRT = abm::fast_rcp(R_DRY * ta);
    const double Lv = L_vap(T);
    return fdiv(GRAV * (1. + Lv * wa * iRT), RCP_DRY + fdiv(Lv * Lv * wa * REPS0 * iRT, ta));
}
ABD double alpha_sw(double T) { return 2.1e-5 * powr(abm::dmax(T - RT0 + 3.2, 0.), 0.79); }                    // :1267-1280
ABD double qlw_net(double rlw, double Ts) { const double t2 = Ts * Ts; return KC(EMISS_W) * (rlw - KC(STEFAN) * t2 * t2); }  // :1291-1314

// 1/L, :666-693
ABD double one_on_L(double tha, double qa, double us, double ts, double qs)
{
    const double zqa = 1. + KC(RCTV0) * qa;
    const double r = fdiv(KC(GRAV * VKARMN) * (ts * zqa + KC(RCTV0) * tha * qs), abm::dmax(us * us * tha * zqa, KC(1.E-9)));
    return clip_abs(r, 200.);
}

// bulk Richardson number, :712-747
ABD double ri_bulk(double z, double sst, double tha, double ssq, double qa, double ub)
{
    const double sstv = virt_temp(sst, ssq);
    const double dthv = virt_temp(tha, qa) - sstv;
    const double tv = 0.5 * (sstv + virt_temp(tha - KC(RGAMMA_DRY) * z, qa));
    return fdiv(KC(GRAV) * dthv * z, tv * ub * ub);
}

ABD double q_air_rh(double rh, double T, double p)  // :963-985
{
    const double ze = 0.01 * rh * e_sat(T);
    return fdiv(ze * REPS0, abm::dmax(p - (1. - REPS0) * ze, 1.));
}
ABD double q_air_dp(double dp, double p)            // :990-1000
{
    const double e = abm::dmax(e_sat(dp), 0.);
    return fdiv(e * REPS0, abm::dmax(p - (1. - REPS0) * e, 1.));
}

struct Flux {
    double tau, qsen, qlat, evap;
};

// Air column at zu, the part of BULK_FORMULA_SCLR (:1149-1203) that only depends on (theta_zu, q_zu, slp):
// density by the 2-pass estimate of :1182-1186 (MAX(rho,1) as used in zUrho) and cp of moist air.
// Computed once per iteration and shared by the two UPDATE_QNSOL_TAU calls and the final flux assembly.
struct AirZu {
    double rho1, cp;
    double rho;      // before the MAX(.,1): the prhoa output of BULK_FORMULA (dead in the flux kernels)
};
ABD AirZu air_at_zu(double zu, double tha, double qa, double slp)
{
    const double ta = tha - KC(RGAMMA_DRY) * zu;
    const double r = abm::fast_rcp(KC(R_DRY) * ta * (1. + KC(RCTV0) * qa));     // rho_air = MAX(p / (R T (1 + rctv0 q)), 0.8)
    double rho = abm::dmax(slp * r, KC(0.8));
    rho = abm::dmax((slp - rho * KC(GRAV) * zu) * r, KC(0.8));
    AirZu a;
    a.rho = rho;
    a.rho1 = abm::dmax(rho, 1.);
    a.cp = cp_air(qa);
    return a;
}

// BULK_FORMULA_SCLR, :1149-1203 (over water)
ABD Flux bulk_formula(const AirZu &air, double Ts, double qs, double tha, double qa, double Cd, double Ch, double Ce,
                      double wnd, double Ub)
{
    const double Urho = Ub * air.rho1;
    Flux f;
    f.tau = Urho * Cd * wnd;
    f.evap = Urho * Ce * (qa - qs);
    f.qsen = Urho * Ch * (tha - Ts) * air.cp;
    f.qlat = L_vap(Ts) * f.evap;
    return f;
}

// UPDATE_QNSOL_TAU_SCLR, :1059-1103 -> non-solar flux, stress and latent flux
ABD void update_qnsol_tau(const AirZu &air, double Ts, double qs, double tha, double qa, double us, double ts,
                          double qst, double wnd, double Ub, double rlw,
                          double &Qns, double &Tau, double &Qlat)
{
    const double dt = floor_abs(tha - Ts, KC(1.E-09));
    const double dq = floor_abs(qa - qs, KC(1.E-12));
    const double z0 = fdiv(us, Ub);
    const Flux f = bulk_formula(air, Ts, qs, tha, qa, z0 * z0, fdiv(z0 * ts, dt), fdiv(z0 * qst, dq), wnd, Ub);
    Qns = f.qlat + f.qsen + qlw_net(rlw, Ts);
    Tau = f.tau;
    Qlat = f.qlat;
}

// Liu-Katsaros-Businger z0t / z0q, :1635-1701 (iflag 1: temperature, 2: humidity), in log space:
// LOG(z0t) = LOG(XA) + (XB - 1) LOG(Rer) + LOG(z0), clipped to [LOG(1e-9), LOG(0.05)]; Rer outside
// ]0,1000[ gives the reference's ABS(-999.) -> 0.05.  (One log of Rer instead of two pow and two log.)
static __constant__ double LKB_T[2][8][2] = {
    {{-0x1.bb4a804765594p+0, 0.}, {0x1.46d750d6da9dbp-2, 0.929}, {0x1.a48a553637bd3p-6, -0.599}, {0x1.f128f5faf06edp-2, -1.018},
     {0x1.8a0afa79b6d2dp+0, -1.475}, {0x1.c6bba4d3499efp+1, -2.067}, {0x1.dacf2c5c04d22p+2, -2.907}, {0x1.a91a7a7897e05p+3, -3.935}},
    {{-0x1.3b22e9abd04f9p+0, 0.}, {0x1.2f37a01050599p-1, 0.826}, {0x1.536a2b94647bcp-2, -0.528}, {0x1.57806929d28c9p-1, -0.870},
     {0x1.9bb56ebf3d3b9p+0, -1.297}, {0x1.b657d7f0668f0p+1, -1.845}, {0x1.d1d1701b4f5c8p+2, -2.682}, {0x1.935aebcc59706p+3, -3.616}}};
ABD double log_z0tq_LKB(int iflag, double Rer, double log_Rer, double log_z0)
{
    if (!(Rer > 0. && Rer < 1000.)) return LOG_0P05;
    // interval of the table (upper bounds 0.11 0.825 3 10 30 100 300 1000) and its {LOG(XA), XB} from the constant bank
    int k = 0;
    k += (Rer > KC(0.11)) + (Rer > KC(0.825)) + (Rer > 3.0) + (Rer > 10.0) + (Rer > 30.0) + (Rer > 100.) + (Rer > 300.);
    const double la = LKB_T[iflag == 1 ? 0 : 1][k][0], b = LKB_T[iflag == 1 ? 0 : 1][k][1];
    return abm::dmin(abm::dmax(la + (b - 1.) * log_Rer + log_z0, KC(LOG_1EM9)), KC(LOG_0P05));
}

// ---------------------------------------------------------------------------
// stability functions.  Every algorithm evaluates psi_m and psi_h at several heights of the same
// sign of 1/L per iteration; the grouped evaluators below take ONE branch on the stability class and
// compute all of them inside it: independent dependency chains the scheduler can interleave
// ("wait" was the top stall with one branch per psi), shared sub-expressions computed once
// (exp(-0.35 zeta), sqrt(|1-15 zeta|), zeta^2/(1+zeta^2): bit-identical), fewer branches.
// ---------------------------------------------------------------------------
struct PsiMH {
    double m, h;
};

// Unstable psi_m / psi_h from the tables of ab_math.cuh (abm::psi_row): the COARE blend (COARE 3.x and the first guess
// of ECMWF) and the Paulson pair with coefficient 16 (ECMWF).  The COARE first guess does not clip zeta: below -50, and for
// NaN, psi_*_coare_formula runs.  NCAR and ANDREAS keep their Paulson formulas: the table's 96 bytes of coefficients per
// function are shared-memory bound where the formula is cheap (profiles/psi_probe_r03d.txt), and both kernels were
// slower with it (profiles/ab_psi_table_r03d.txt).
template <int FAM>
ABD PsiMH psi_mh_table(double z)
{
    const abm::PsiRow a = abm::psi_row(z);
    PsiMH r;
    r.m = abm::psi_poly<0>(abm::psi_coeffs<FAM>(), a);
    r.h = abm::psi_poly<1>(abm::psi_coeffs<FAM>(), a);
    return r;
}
template <int FAM>
ABD double psi_m_table(double z) { return abm::psi_poly<0>(abm::psi_coeffs<FAM>(), abm::psi_row(z)); }
template <int FAM>
ABD double psi_h_table(double z) { return abm::psi_poly<1>(abm::psi_coeffs<FAM>(), abm::psi_row(z)); }
ABD bool in_psi_table(double z) { return z >= -abm::PSI_ZMAX; }

// Large & Yeager, src/mod_blk_ncar.f90:333-407
ABD PsiMH psi_mh_ncar_unstable(double z)
{
    const double x2 = abm::dmax(abm::fast_sqrt_pos(fabs(1. - 16. * z)), 1.);
    const double x = abm::fast_sqrt_pos(x2);
    const double l2 = abm::dlog((1. + x2) * 0.5);
    PsiMH r;
    r.m = 2. * abm::dlog((1. + x) * 0.5) + l2 - 2. * abm::datan_ge1(x) + RPI * 0.5;
    r.h = 2. * l2;
    return r;
}
ABD double psi_h_ncar_unstable(double z)
{
    const double x2 = abm::dmax(abm::fast_sqrt_pos(fabs(1. - 16. * z)), 1.);
    return 2. * abm::dlog(0.5 * (1. + x2));
}
ABD double psi_m_ncar(double z) { return nonneg(z) ? -5. * z : psi_mh_ncar_unstable(z).m; }
ABD double psi_h_ncar(double z) { return nonneg(z) ? -5. * z : psi_h_ncar_unstable(z); }

// COARE 3.x, src/mod_common_coare.f90:217-254, :305-344.  Note psi(+0) = -4.524e-3:
// SIGN(0.5,+0.) selects the stable branch and the truncated literals do not cancel.
ABD double psi_coare_convective(double phi_c)
{
    return 1.5 * abm::dlog((1. + phi_c + phi_c * phi_c) * KC(1. / 3.)) - KC(1.7320508) * abm::datan_ge1((1. + 2. * phi_c) * KC(1. / 1.7320508)) + KC(1.813799447);
}
ABD PsiMH psi_mh_coare_stable(double z)
{
    const double e = abm::dexp_b(-abm::dmin(50., KC(0.35) * z));   // stable branch: z >= 0
    const double a = fabs(1. + 2. * z * KC(1. / 3.));
    PsiMH r;
    r.m = -(1. + 1. * z + KC(0.6667) * (z - KC(14.28)) * e + KC(8.525));
    r.h = -(a * abm::fast_sqrt_pos(a) + KC(.6667) * (z - KC(14.28)) * e + KC(8.525));                      // **1.5
    return r;
}
ABD double psi_h_coare_stable(double z)
{
    const double e = abm::dexp_b(-abm::dmin(50., KC(0.35) * z));   // stable branch: z >= 0
    const double a = fabs(1. + 2. * z * KC(1. / 3.));
    return -(a * abm::fast_sqrt_pos(a) + KC(.6667) * (z - KC(14.28)) * e + KC(8.525));
}
ABD PsiMH psi_mh_coare_formula(double z)
{
    const double phi_h = abm::fast_sqrt_pos(fabs(1. - 15. * z));                               // **.5
    const double phi_m = abm::fast_sqrt_pos(phi_h);                                            // **.25
    double f = z * z;
    f = fdiv(f, 1. + f);
    // LOG((1 + phi_m**2)/2) of psi_m is LOG((1 + phi_h)/2) of psi_h up to the rounding of phi_m**2 (phi_m = SQRT(phi_h)):
    // one logarithm serves both (the argument differs by <= 1 ulp: 1e-16 in the logarithm)
    const double lh = abm::dlog((1. + phi_h) * 0.5);
    const double km = 2. * abm::dlog((1. + phi_m) * 0.5) + lh - 2. * abm::datan_ge1(phi_m) + KC(0.5 * RPI);
    const double kh = 2. * lh;
    const double cm = psi_coare_convective(powr(fabs(1. - KC(10.15) * z), KC(.3333)));
    const double ch = psi_coare_convective(powr(fabs(1. - KC(34.15) * z), KC(.3333)));
    PsiMH r;
    r.m = (1. - f) * km + f * cm;
    r.h = (1. - f) * kh + f * ch;
    return r;
}
ABD PsiMH psi_mh_coare_unstable(double z) { return in_psi_table(z) ? psi_mh_table<abm::PSI_TABLES_COARE>(z) : psi_mh_coare_formula(z); }
ABD double psi_h_coare_formula(double z)
{
    const double phi_h = abm::fast_sqrt_pos(fabs(1. - 15. * z));
    double f = z * z;
    f = fdiv(f, 1. + f);
    const double kh = 2. * abm::dlog((1. + phi_h) * 0.5);
    const double ch = psi_coare_convective(powr(fabs(1. - KC(34.15) * z), KC(.3333)));
    return (1. - f) * kh + f * ch;
}
ABD double psi_h_coare_unstable(double z) { return in_psi_table(z) ? psi_h_table<abm::PSI_TABLES_COARE>(z) : psi_h_coare_formula(z); }
// psi_m(zeta_u), psi_h(zeta_u), psi_h(zeta_t); zeta_t has the sign of zeta_u
template <bool ZTEQ>
ABD void psi3_coare(double zeta_u, double zeta_t, double &m_u, double &h_u, double &h_t)
{
    h_t = 0.;
    if (nonneg(zeta_u)) {
        const PsiMH r = psi_mh_coare_stable(zeta_u);
        m_u = r.m;
        h_u = r.h;
        if (!ZTEQ) h_t = psi_h_coare_stable(zeta_t);
    } else {
        const PsiMH r = psi_mh_coare_unstable(zeta_u);
        m_u = r.m;
        h_u = r.h;
        if (!ZTEQ) h_t = psi_h_coare_unstable(zeta_t);
    }
}

// IFS, src/mod_blk_ecmwf.f90:441-564 (zeta capped to [-50, 5]; the cap keeps the sign)
ABD double cap_zeta(double zeta) { return abm::dmin(abm::dmax(zeta, -50.), 5.); }
ABD PsiMH psi_mh_ecmwf_stable(double zeta)
{
    constexpr double zc = 5. / 0.35;
    const double z = cap_zeta(zeta);
    const double t = KC(2. / 3.) * (z - KC(zc)) * abm::dexp_b(KC(-0.35) * z);   // zeta is capped to [-50, 5]
    const double a = fabs(1. + KC(2. / 3.) * z);
    PsiMH r;
    r.m = -t - z - KC(2. / 3. * zc);
    r.h = -t - a * abm::fast_sqrt_pos(a) - KC(2. / 3. * zc) + 1.;
    return r;
}
// unstable: the cap keeps zeta inside the Paulson table (a NaN zeta is capped to -50, as before)
ABD PsiMH psi_mh_ecmwf_unstable(double zeta) { return psi_mh_table<abm::PSI_TABLES_PAULSON>(cap_zeta(zeta)); }
ABD double psi_m_ecmwf_stable(double zeta) { return psi_mh_ecmwf_stable(zeta).m; }
ABD double psi_h_ecmwf_stable(double zeta) { return psi_mh_ecmwf_stable(zeta).h; }
ABD double psi_m_ecmwf_unstable(double zeta) { return psi_m_table<abm::PSI_TABLES_PAULSON>(cap_zeta(zeta)); }
ABD double psi_h_ecmwf_unstable(double zeta) { return psi_h_table<abm::PSI_TABLES_PAULSON>(cap_zeta(zeta)); }

// Andreas et al. 2015 (Paulson unstable / Grachev 2007 stable), src/mod_blk_andreas.f90:307-410
// the two terms of the stable functions that do not depend on zeta, as glibc evaluates them (the reference computes them
// at run time): ATAN((2 - b)/(SQRT(3) b)) and LOG(ABS((c - SQRT(5))/(c + SQRT(5)))), :353 / :384
constexpr double ATAN_A_STABLE = 0x1.b53ea749504d7p-1;
constexpr double LOG_A_STABLE = -0x1.ecc2caec5160ap+0;
ABD double psi_m_andreas_stable(double zeta)
{
    const double z = abm::dmin(zeta, 15.);
    constexpr double zam = 5.;
    const double x = abm::fast_cbrt(fabs(1. + z));
    return -(KC(3. * zam / ZBM_A) * (x - 1.))
           + KC(zam * ZBBM_A / (2. * ZBM_A))
                 * (2. * abm::dlog(fabs((x + KC(ZBBM_A)) * KC(1. / (1. + ZBBM_A))))
                    - abm::dlog(fabs((x * x - x * KC(ZBBM_A) + KC(ZBBM_A * ZBBM_A)) * KC(1. / (1. - ZBBM_A + ZBBM_A * ZBBM_A))))
                    + KC(2. * SR3) * (abm::datan_ge1((2. * x - KC(ZBBM_A)) * KC(1. / (SR3 * ZBBM_A))) - KC(ATAN_A_STABLE)));
}
ABD double psi_h_andreas_stable(double zeta)
{
    const double z = abm::dmin(zeta, 15.);
    constexpr double zah = 5., zbh = 5., zch = 3.;
    const double zz = 2. * z + zch;
    return -(KC(0.5 * zbh) * abm::dlog(fabs(1. + zch * z + z * z)))
           + KC(-zah / SR5 + 0.5 * zbh * zch / SR5)
                 * (abm::dlog(fabs(fdiv(zz - KC(SR5), zz + KC(SR5)))) - KC(LOG_A_STABLE));
}
ABD PsiMH psi_mh_andreas_unstable(double zeta)
{
    const double z = abm::dmin(zeta, 15.);
    const double x2 = abm::dmax(abm::fast_sqrt_pos(fabs(1. - 16. * z)), 1.);
    const double x = abm::fast_sqrt_pos(x2);
    PsiMH r;
    const double l2 = abm::dlog(0.5 * (1. + x2));   // x, x2 >= 1: the ABS of the reference is the identity
    r.m = 2. * abm::dlog((1. + x) * 0.5) + l2 - 2. * abm::datan_ge1(x) + KC(RPI * 0.5);
    r.h = 2. * l2;
    return r;
}
ABD double psi_h_andreas_unstable(double zeta)
{
    const double x2 = abm::dmax(abm::fast_sqrt_pos(fabs(1. - 16. * abm::dmin(zeta, 15.))), 1.);
    return 2. * abm::dlog(0.5 * (1. + x2));
}

// ---------------------------------------------------------------------------
// launch-uniform quantities computed once on the host (glibc libm, as the reference build uses)
// ---------------------------------------------------------------------------
struct Uniform {
    double zt, zu;
    double log_zt, log_zu, log_ztu, log_zu10, log_10;   // LOG(zt) LOG(zu) LOG(zt/zu) LOG(zu/10) LOG(10)
    double fg_c_a;                                     // 0.035*LOG(10/1e-4)/LOG(zu/1e-4)   mod_common_coare.f90:107
    double fg_1_o_Ribcu;                               // -0.004*600*1.2**3/zu              :108,:140
    double rdt, gdept;                                 // mod_const.f90:31-32
    int nb_iter;
    unsigned long long wl_commit_mask;                 // bit jit set iff MOD(nb_iter, jit) == 0, jit < 64 (host-computed)
    int isd;                                           // seconds since 00h UTC (12 in aerobulk_compute)
    int dawn;                                          // WL_COARE dawn reset for longitude 0 (host-computed)
};

// ---------------------------------------------------------------------------
// COARE first guess of u*, theta*, q*, z0 (also used by ECMWF),
// src/mod_common_coare.f90:33-179
// ---------------------------------------------------------------------------
struct Guess {
    double us, ts, qs, t_zu, q_zu, Ub, z0;
};

template <bool ZTEQ>
ABD Guess first_guess_coare(const Uniform &u, double sst, double t_zt, double ssq, double q_zt, double wnd, double charn)
{
    Guess g;
    g.t_zu = abm::dmax(t_zt, 180.);
    g.q_zu = abm::dmax(q_zt, 1.e-6);

    double dt = floor_abs(g.t_zu - sst, 1.E-09);
    double dq = floor_abs(g.q_zu - ssq, 1.E-12);

    const double nu_a = visc_air(g.t_zu);
    const double Ub = sqrt(wnd * wnd + 0.5 * 0.5);
    double us = u.fg_c_a * Ub;

    double z0 = charn * us * us * INV_GRAV + fdiv(0.11 * nu_a, us);
    z0 = abm::dmin(abm::dmax(fabs(z0), 1.E-8), 1.);
    const double log_z0 = abm::dlog(z0);

    const double sq = fdiv(VKARMN, u.log_zu - log_z0);
    const double Cd = sq * sq;
    const double r1_o_sqrt_Cd10 = (u.log_10 - log_z0) * INV_VKARMN;

    // z0t = 10 / EXP(k / (0.00115 r)) clipped to [1e-8, 1], only needed as LOG(z0t)
    const double log_z0t = abm::dmin(abm::dmax(u.log_10 - fdiv(VKARMN, 0.00115 * r1_o_sqrt_Cd10), LOG_1EM8), 0.);

    const double Rib = ri_bulk(u.zu, sst, g.t_zu, ssq, g.q_zu, Ub);

    const double cc = fdiv(VKARMN2, Cd * (u.log_zt - log_z0t));
    const double cc_ri = cc * Rib;
    const double zeta_u = nonneg(Rib) ? (cc_ri + 27. / 9. * Rib * Rib) : fdiv(cc_ri, 1. + Rib * u.fg_1_o_Ribcu);

    const double zeta_t = ZTEQ ? zeta_u : fdiv(u.zt * zeta_u, u.zu);
    double psi_m_u, psi_h_u, psi_h_t;
    psi3_coare<ZTEQ>(zeta_u, zeta_t, psi_m_u, psi_h_u, psi_h_t);
    us = abm::dmax(fdiv(Ub * VKARMN, u.log_zu - log_z0 - psi_m_u), 1.E-9);
    const double tmp = fdiv(VKARMN, u.log_zu - log_z0t - psi_h_u);
    double ts = dt * tmp;
    double qs = dq * tmp;

    if (!ZTEQ) {
        const double prf = u.log_ztu + psi_h_u - psi_h_t;
        g.t_zu = t_zt - ts * INV_VKARMN * prf;
        g.q_zu = q_zt - qs * INV_VKARMN * prf;
        g.q_zu = signbit(g.q_zu) ? 0. : g.q_zu;
        dt = floor_abs(g.t_zu - sst, 1.E-09);
        dq = floor_abs(g.q_zu - ssq, 1.E-12);
        ts = dt * tmp;
        qs = dq * tmp;
    }
    g.us = us;
    g.ts = ts;
    g.qs = qs;
    g.Ub = Ub;
    z0 = charn * us * us * INV_GRAV + fdiv(0.11 * nu_a, us);
    g.z0 = abm::dmin(abm::dmax(fabs(z0), 1.E-8), 1.);
    return g;
}

// ---------------------------------------------------------------------------
// cool skin (Fairall 1996 / Zeng-Beljaars 2005)
// src/mod_phymbl.f90:2010-2046, src/mod_skin_coare.f90:48-93, src/mod_skin_ecmwf.f90:68-110
// ---------------------------------------------------------------------------
// COARE_FORM: 0.137 coefficient and the latent-heat term in delta; else 0.065, no Qlat.
template <bool COARE_FORM>
ABD double cool_skin_dT(double alpha, double Qsw, double Qnsol, double us, double Qlat)
{
    // invariants of the five delta_skin_layer evaluations
    const double usw = abm::dmax(us, KC(1.E-4)) * KC(SQ_RADRW);
    const double usw2 = usw * usw;
    const double c_lamb = fdiv(alpha * KC(RCST_CS), usw2 * usw2);
    const double nu_o_usw = fdiv(KC(RNU0_W), usw);
    const double d_warm = abm::dmin(6. * nu_o_usw, KC(0.007));
    const double q_lat_term = COARE_FORM ? fdiv(KC(0.026) * abm::dmin(Qlat, 0.) * KC(RCP0_W * (1. / RLEVAP)), alpha) : 0.;

    auto delta = [&](double Qd) -> double {
        const double zQd = COARE_FORM ? Qd + q_lat_term : Qd;
        if (nonneg(zQd)) return d_warm;                                  // warming of the viscous layer
        // floored at 1e-30 instead of 0: x**0.75 < 4e-23 vanishes against the 1 it is added to (bit-identical), and
        // the root needs no zero guard
        const double x = abm::dmax(c_lamb * zQd, KC(1.e-30));
        const double x75 = abm::pow075_pos(x);                           // **0.75
        return 6. * abm::fast_rcbrt(1. + x75) * nu_o_usw;                 // **(-1./3.)
    };

    // delta(Qnsol), then 4 x { solar absorption fr(delta) -> Qabs -> delta(Qabs) }: one rolled loop so that
    // the delta code exists once (instruction-cache footprint)
    double Qabs = Qnsol, d = 0.;
#pragma unroll 1   // cool-skin passes rolled: the delta code exists once (instruction-cache footprint)
    for (int jc = 0; jc < 5; ++jc) {
        const double d_prev = d;
        if (jc > 0) {
            const double fr = abm::dmax((COARE_FORM ? KC(0.137) : KC(0.065)) + 11. * d - fdiv(KC(6.6E-5), d) * (1. - abm::dexp(-d * KC(1. / 8.E-4))), KC(0.01));
            Qabs = Qnsol + fr * Qsw;
        }
        d = delta(Qabs);
        // fixed point reached (typically d == d_warm while the skin warms): the remaining passes would reproduce
        // Qabs and d bit for bit
        if (jc > 0 && d == d_prev) break;
    }
    return Qabs * d * KC(1. / RK0_W);
}

// ---------------------------------------------------------------------------
// warm layer -- persistent per-point state kept in registers across the bulk
// iteration and device-resident across time steps
// ---------------------------------------------------------------------------
struct WarmLayer {
    double dT, Hz, Qac, Tac;   // dT_wl, Hz_wl, Qnt_ac, Tau_ac
};

// Per-point invariants of WL_COARE, src/mod_skin_coare.f90:146-156
struct WlCoareCtx {
    double cd1, cd2;
    bool dawn;     // local solar hour in ]4, 6.5]
};
// local solar time from longitude and UTC seconds, src/mod_skin_coare.f90:146-150,159
__host__ __device__ inline bool wl_coare_dawn(double lon, int isd)
{
    auto f_mod = [](double a, double p) {
        double r = fmod(a, p);
        if (r != 0. && ((r < 0.) != (p < 0.))) r += p;
        return r;
    };
    double lag = -1. * f_mod((360. - f_mod(lon, 360.)) / 15., 24.);
    lag = -1. * copysign(fmin(fabs(lag), fabs(f_mod(lag, 24.))), lag + 12.);
    const int ilag = (int)(lag * 3600.);
    int isol = (isd + ilag) % 86400;
    if (isol < 0) isol += 86400;
    const double hr = (double)isol / 3600.;
    return (hr > 4.) && (hr <= 6.5);
}
ABD WlCoareCtx wl_coare_ctx(double alpha, bool dawn)
{
    WlCoareCtx c;
    c.dawn = dawn;
    const double Rich0 = 0.65;
    c.cd1 = sqrt(2. * Rich0 * RCP0_W / (alpha * GRAV * RHO0_W));
    c.cd2 = sqrt(2. * alpha * GRAV / (Rich0 * RHO0_W)) / RCP0W_POW15;
    return c;
}
ABD double wl_coare_absorption(double H)   // solar absorption profile, :167-168 / :205-206
{
    // 1 - EXP(-x) is exactly 1 in FP64 once EXP(-x) < 2**-54, i.e. x > 37.43: the two short-wave bands
    // are only evaluated for shallow layers (H <= 0.53 m, H <= 13.4 m) -- bit-identical, fewer exps
    const double e1 = (H > KC(0.53)) ? 0. : abm::dexp_b(-H * KC(1. / 0.014));   // 0.1 <= H <= 20 (callers clamp)
    const double e2 = (H > KC(13.4)) ? 0. : abm::dexp_b(-H * KC(1. / 0.357));
    return 1. - fdiv(KC(0.28 * 0.014) * (1. - e1) + KC(0.27 * 0.357) * (1. - e2)
                     + KC(0.45 * 12.82) * (1 - abm::dexp_b(-H * KC(1. / 12.82))), H);
}
// WL_COARE, src/mod_skin_coare.f90:97-250; `commit` is (iwait == 0)
ABD void wl_coare(WarmLayer &w, const WlCoareCtx &c, double Qsw, double Qnsol, double Tau, double rdt,
                  double gdept, bool commit)
{
    const double Hwl_max = 20.;
    double dT = w.dT;
    double H = abm::dmax(abm::dmin(w.Hz, Hwl_max), 0.1);
    double qac = w.Qac;
    double tac = w.Tac;
    bool l_exit = c.dawn, destroy = c.dawn;
    double Qabs = 0.;

    if (!l_exit) {
        Qabs = wl_coare_absorption(H) * Qsw + Qnsol;
        if (fabs(dT) < 1.E-6 && Qabs <= 0.) l_exit = true;
    }
    if (!l_exit && (w.Qac + Qabs * rdt <= 0.)) {
        l_exit = true;
        destroy = true;
    }
    if (!l_exit) {
        tac = w.Tac + abm::dmax(.002, Tau) * rdt;
#pragma unroll 1
        for (int jl = 0; jl < 5; ++jl) {
            if (jl > 0) Qabs = wl_coare_absorption(H) * Qsw + Qnsol;   // jl == 0: H unchanged since the test above
            qac = w.Qac + Qabs * rdt;
            if (qac <= 0.) break;
            const double H_prev = H;
            H = abm::dmax(abm::dmin(Hwl_max, c.cd1 * tac * abm::fast_rsqrt(qac)), 0.1);
            if (H == H_prev) break;   // fixed point (usually a clamp): further passes are bit-identical
        }
        if (qac <= 0.) {
            destroy = true;
        } else {
            dT = fdiv(c.cd2 * (qac * (qac * abm::fast_rsqrt(qac))), tac);                       // qac > 0 here: MAX(qac/ABS(qac),0) = 1   // **1.5
            if (signbit(gdept - H)) dT = dT * fdiv(gdept, H);                       // flg = 0
        }
    }
    if (destroy) {
        dT = 0.;
        H = Hwl_max;
        qac = 0.;
        tac = 0.;
    }
    if (commit) {
        w.dT = dT;
        w.Hz = H;
        w.Qac = qac;
        w.Tac = tac;
    }
}

// Takaya et al. 2010 Eq.5, src/mod_skin_ecmwf.f90:233-253
ABD double phi_takaya(double z)
{
    const double z2 = z * z;
    if (nonneg(z)) return 1. + fdiv(5. * z + 4. * z2, 1. + 3. * z + 0.25 * z2);
    return abm::fast_rsqrt(1. - 16. * (-fabs(z)));
}
// WL_ECMWF, src/mod_skin_ecmwf.f90:113-230 -- advances dT_wl by rdt at EVERY call
// quantities of WL_ECMWF that only depend on the (constant) layer depth: hoisted out of the bulk iteration
struct WlEcmwfCtx {
    double fr, tcorr, r_tcorr;
};
ABD WlEcmwfCtx wl_ecmwf_ctx(double H, double gdept)
{
    WlEcmwfCtx c;
    c.tcorr = signbit(gdept - H) ? gdept / H : 1.;
    c.r_tcorr = 1. / c.tcorr;
    c.fr = 1. - 0.28 * abm::dexp(-71.5 * H) - 0.27 * abm::dexp(-2.8 * H) - 0.45 * abm::dexp(-0.07 * H);   // Eq. 8.157
    return c;
}
ABD void wl_ecmwf(WarmLayer &w, const WlEcmwfCtx &c, double alpha, double Qsw, double Qnsol, double us, double rdt)
{
    const double rNuwl0 = 0.5;
    const double RhoCp_w = RHO0_W * RCP0_W;
    const double H = w.Hz;
    const double tcorr = c.tcorr;
    const double dT_b = abm::dmax(w.dT * c.r_tcorr, 0.);

    const double Qabs = c.fr * Qsw + Qnsol;

    const double usw = abm::dmax(us, KC(1.E-4)) * KC(SQ_RADRW);
    const double usw2 = usw * usw;
    const bool warming = nonneg(Qabs);

    const double cst1 = KC(VKARMN * GRAV) * alpha;
    const double L2 = fdiv(cst1 * Qabs, RhoCp_w * usw2 * usw);
    const double cst2 = fdiv(cst1, 5. * H * usw2);
    const double cst0 = fdiv(rdt * (rNuwl0 + 1.), H);
    const double A = cst0 * Qabs * KC(1. / (rNuwl0 * RhoCp_w));
    const double cst3 = -cst0 * KC(VKARMN) * usw * KC(FLA_ECMWF);

    // while the layer warms zeta = H L2 does not depend on dT: B is the same in all ten passes
    const double B_warm = warming ? fdiv(cst3, phi_takaya(H * L2)) : 0.;
    double dT_n = dT_b;
#pragma unroll 2
    for (int jc = 0; jc < 10; ++jc) {
        const double prev = dT_n;
        dT_n = 0.5 * (dT_n + dT_b);
        const double B = warming ? B_warm : fdiv(cst3, phi_takaya(H * abm::fast_sqrt(dT_n * cst2)));
        dT_n = abm::dmax(dT_b + A + B * dT_n, 0.);
        if (dT_n == prev) break;   // fixed point of the pass (e.g. 0 at night): the remaining passes are bit-identical
    }
    w.dT = dT_n * tcorr;
}

// ---------------------------------------------------------------------------
// per-point problem and result
// ---------------------------------------------------------------------------
struct PointIn {
    double sst, theta_zt, ssq, q_zt, wnd, slp;   // after aerobulk_compute steps 1-5
    double Qsw, rlw, lon;                          // skin only
    bool has_lon;                                  // per-point longitude given (else Uniform::dawn)
};
struct Coeffs {
    double Cd, Ch, Ce, t_zu, q_zu, Ub, Ts, qs;
};
// optional outputs of the TURB_* routines (CdN, ChN, CeN, xz0, xu_star, xL, xUN10, pdT_cs); dead code in
// the aerobulk_model kernels, which do not read them
struct Diag {
    double CdN, ChN, CeN, z0, us, L, UN10, dT_cs;
};

// ---------------------------------------------------------------------------
// NCAR (Large & Yeager 2004/2008), src/mod_blk_ncar.f90:57-271
// ---------------------------------------------------------------------------
ABD double cd_n10_ncar(double w)
{
    double w6 = w * w * w;
    w6 = w6 * w6;
    const double r = nonneg(w - 33.) ? KC(1.e-3 * 2.34)
                                     : KC(1.e-3) * (fdiv(KC(2.7), w) + KC(0.142) + w * KC(1. / 13.09) - KC(3.14807E-10) * w6);
    return abm::dmax(r, KC(CX_MIN));
}

template <bool ZTEQ>
ABD Coeffs solve_ncar(const Uniform &u, const PointIn &p, Diag &dg)
{
    const double Ub = abm::dmax(0.5, p.wnd);
    const bool stable0 = nonneg(virt_temp(p.theta_zt, p.q_zt) - virt_temp(p.sst, p.ssq));
    double CdN = cd_n10_ncar(Ub);
    double sqrt_CdN = abm::fast_sqrt_pos(CdN);
    double Cd = CdN;
    double Ce = abm::dmax(1.e-3 * (34.6 * sqrt_CdN), CX_MIN);
    double Ch = abm::dmax(1.e-3 * sqrt_CdN * (stable0 ? 18. : 32.7), CX_MIN);
    double sqrt_Cd = sqrt_CdN;
    double t_zu = abm::dmax(p.theta_zt, 180.);
    double q_zu = abm::dmax(p.q_zt, 1.e-6);
    double us = 0., r1oL = 0., Un10 = 0., ChN = 0., CeN = 0.;

#pragma unroll 1
    for (int jit = 0; jit < u.nb_iter; ++jit) {
        const double dt = t_zu - p.sst;
        const double dq = q_zu - p.ssq;
        us = sqrt_Cd * Ub;
        const double r_sqrt_Cd = abm::fast_rcp(sqrt_Cd);
        const double ts = Ch * r_sqrt_Cd * dt;
        const double qs = Ce * r_sqrt_Cd * dq;
        r1oL = one_on_L(t_zu, q_zu, us, ts, qs);
        const double zeta_u = clip_abs(u.zu * r1oL, 10.);
        const double zeta_t = clip_abs(u.zt * r1oL, 10.);
        // psi_h(zeta_u) is used twice in the reference (:196,:217); one stability branch for all three
        double psi_m, psi_h_u, psi_h_t = 0.;
        if (nonneg(zeta_u)) {
            psi_m = psi_h_u = -5. * zeta_u;
            if (!ZTEQ) psi_h_t = -5. * zeta_t;
        } else {
            const PsiMH r = psi_mh_ncar_unstable(zeta_u);
            psi_m = r.m;
            psi_h_u = r.h;
            if (!ZTEQ) psi_h_t = psi_h_ncar_unstable(zeta_t);
        }
        if (!ZTEQ) {
            const double tmp = u.log_ztu + psi_h_u - psi_h_t;
            t_zu = p.theta_zt - ts * INV_VKARMN * tmp;
            q_zu = abm::dmax(0., p.q_zt - qs * INV_VKARMN * tmp);
        }
        // UN10_from_CD (mod_phymbl.f90:1532-1547) with z0_from_Cd(zu, Cd, psi) (:1335-1352); SQRT(Cd) is sqrt_Cd
        // z0 = zu EXP(-(k/SQRT(Cd) + psi_m)) only enters as LOG(10/z0) = k/SQRT(Cd) + psi_m - LOG(zu/10)
        Un10 = abm::dmax(0.25, sqrt_Cd * Ub * INV_VKARMN * (VKARMN * r_sqrt_Cd + psi_m - u.log_zu10));
        CdN = cd_n10_ncar(Un10);
        sqrt_CdN = abm::fast_sqrt_pos(CdN);
        double tmp = 1. + sqrt_CdN * INV_VKARMN * (u.log_zu10 - psi_m);
        Cd = abm::dmax(fdiv(CdN, tmp * tmp), CX_MIN);
        sqrt_Cd = abm::fast_sqrt_pos(Cd);
        const double r_sqrt_CdN = abm::fast_rcp(sqrt_CdN);
        tmp = (u.log_zu10 - psi_h_u) * INV_VKARMN * r_sqrt_CdN;
        const double tmp2 = sqrt_Cd * r_sqrt_CdN;
        ChN = 1.e-3 * sqrt_CdN * (nonneg(zeta_u) ? 18. : 32.7);
        CeN = 1.e-3 * (34.6 * sqrt_CdN);
        Ch = abm::dmax(fdiv(ChN * tmp2, 1. + ChN * tmp), CX_MIN);
        Ce = abm::dmax(fdiv(CeN * tmp2, 1. + CeN * tmp), CX_MIN);
    }
    Coeffs c;
    c.Cd = Cd; c.Ch = Ch; c.Ce = Ce; c.t_zu = t_zu; c.q_zu = q_zu; c.Ub = Ub; c.Ts = p.sst; c.qs = p.ssq;
    // optional outputs, src/mod_blk_ncar.f90:229-235
    dg.CdN = CdN; dg.ChN = ChN; dg.CeN = CeN; dg.UN10 = Un10; dg.L = 1. / r1oL; dg.us = us;
    dg.z0 = abm::dmin(u.zu * abm::dexp_b(-VKARMN * abm::fast_rsqrt(CdN)), Z0_SEA_MAX);
    dg.dT_cs = 0.;
    return c;
}

// ---------------------------------------------------------------------------
// COARE 3.0 (Fairall 2003) and 3.6 (Edson 2013)
// src/mod_blk_coare3p0.f90:54-447, src/mod_blk_coare3p6.f90:123-441
// ---------------------------------------------------------------------------
ABD double charn_coare3p0(double w)
{
    if (!nonneg(w - 10.)) return 0.011;
    if (nonneg(w - 18.)) return 0.018;
    return 0.011 + (0.018 - 0.011) * (w - 10.) * (1. / (18. - 10.));
}
ABD double charn_coare3p6(double w) { return abm::dmax(abm::dmin(KC(0.0017) * w - KC(0.005), KC(0.028)), 0.); }

// CS / WL: l_use_cs / l_use_wl of the reference (aerobulk_model switches both on together)
template <bool V36, bool CS, bool WL, bool ZTEQ>
ABD Coeffs solve_coare(const Uniform &u, const PointIn &p, WarmLayer &wl, Diag &dg)
{
    constexpr bool SKIN = CS || WL;
    constexpr double zi0 = 600., Beta0 = V36 ? 1.2 : 1.25, zeta_abs_max = 50.;

    double Ts = p.sst, qs_ = p.ssq;
    double alpha = 0.;
    WlCoareCtx wc = {};
    if (SKIN) {
        if (CS) Ts = Ts - 0.25;
        qs_ = RDCT_QSAT_SALT * q_sat(abm::dmax(Ts, 200.), p.slp);
        alpha = alpha_sw(p.sst);
        if (WL) wc = wl_coare_ctx(alpha, p.has_lon ? wl_coare_dawn(p.lon, u.isd) : (u.dawn != 0));
    }

    const Guess g = first_guess_coare<ZTEQ>(u, Ts, p.theta_zt, qs_, p.q_zt, p.wnd,
                                            V36 ? charn_coare3p6(p.wnd) : charn_coare3p0(p.wnd));
    double us = g.us, ts = g.ts, qst = g.qs, t_zu = g.t_zu, q_zu = g.q_zu, Ub = g.Ub;
    double log_z0 = abm::dlog(g.z0);
    // COARE 3.6 uses the first-guess t_zu, 3.0 the potential temperature at zt (SURVEY 8a quirk 5)
    const double nu_a = V36 ? visc_air(t_zu) : visc_air(p.theta_zt);

    double dt = floor_abs(t_zu - Ts, 1.E-09);
    double dq = floor_abs(q_zu - qs_, 1.E-12);
    double dT_cs = 0., r1oL = 0., z0 = g.z0, log_z0t = 0.;

#pragma unroll 1
    for (int jit = 1; jit <= u.nb_iter; ++jit) {
        const double us2 = us * us;
        r1oL = one_on_L(t_zu, q_zu, us, ts, qst);    // already clipped to +-200

        const double cv = abm::fast_cbrt(abm::dmax(KC(-zi0 * INV_VKARMN) * r1oL, 0.));
        const double gust2 = KC(Beta0 * Beta0) * us2 * (cv * cv);       // **(2./3.)
        Ub = abm::dmax(abm::fast_sqrt(p.wnd * p.wnd + gust2), KC(0.2));

        const double zeta_u = clip_abs(u.zu * r1oL, zeta_abs_max);

        const double Un10 = us * INV_VKARMN * (u.log_10 - log_z0);
        const double r_us = abm::fast_rcp(us);
        z0 = (V36 ? charn_coare3p6(Un10) : charn_coare3p0(Un10)) * us2 * KC(INV_GRAV) + KC(0.11) * nu_a * r_us;
        z0 = abm::dmin(abm::dmax(fabs(z0), KC(1.E-9)), 1.);
        log_z0 = abm::dlog(z0);

        // z0t = MIN(1.6e-4, 5.8e-5 (nu/(z0 u*))**0.72) [3.6] / MIN(1.1e-4, 5.5e-5 (..)**0.6) [3.0], floored at
        // 1e-9, is only needed as LOG(z0t): monotonic, so MIN / MAX act on the logarithms (no pow)
        const double log_rr = abm::dlog(nu_a * r_us) - log_z0;
        log_z0t = V36 ? abm::dmax(abm::dmin(KC(LOG_1P6EM4), KC(LOG_5P8EM5) + KC(0.72) * log_rr), KC(LOG_1EM9))
                      : abm::dmax(abm::dmin(KC(LOG_1P1EM4), KC(LOG_5P5EM5) + KC(0.6) * log_rr), KC(LOG_1EM9));

        const double zeta_t = clip_abs(u.zt * r1oL, zeta_abs_max);
        double psi_m_u, psi_h_u, psi_h_t;
        psi3_coare<ZTEQ>(zeta_u, zeta_t, psi_m_u, psi_h_u, psi_h_t);
        double tmp1 = fdiv(KC(VKARMN), u.log_zu - log_z0t - psi_h_u);
        ts = dt * tmp1;
        qst = dq * tmp1;
        us = abm::dmax(fdiv(Ub * KC(VKARMN), u.log_zu - log_z0 - psi_m_u), KC(1.E-9));

        if (!ZTEQ) {
            tmp1 = u.log_zt - u.log_zu + psi_h_u - psi_h_t;
            t_zu = p.theta_zt - ts * INV_VKARMN * tmp1;
            q_zu = p.q_zt - qst * INV_VKARMN * tmp1;
        } else if (!V36) {
            t_zu = p.theta_zt;   // zm_ztzu = 0 in COARE 3.0: t_zu <- t_zt, q_zu <- q_zt every iteration
            q_zu = p.q_zt;
        }

        if (SKIN) {
            // pass 0: cool skin, pass 1: warm layer (state committed whenever jit divides nb_iter, SURVEY 8a
            // quirk 1); rolled so that UPDATE_QNSOL_TAU and q_sat exist once in the loop body
            const AirZu air = air_at_zu(u.zu, t_zu, q_zu, p.slp);
            // WL_COARE only touches its state when iwait == 0 (mod_skin_coare.f90:239-248) and has no other output: at
            // the other iterations the reference computes it for nothing, here it is not called (nor the
            // UPDATE_QNSOL_TAU that feeds it).  T_s is still re-assembled in the warm-layer order of operations, and
            // q_s recomputed only if that changed a bit of T_s.
            // iwait = MOD(nb_iter, jit) == 0 (mod_blk_coare3p6.f90:370), from a host-computed bit mask: the integer
            // division cost 1.2 % of the kernel
            const bool commit = (jit < 64) ? ((u.wl_commit_mask >> jit) & 1ull) != 0ull : (u.nb_iter % jit) == 0;
#pragma unroll 1   // cool-skin pass and warm-layer pass rolled: UPDATE_QNSOL_TAU and q_sat exist once in the loop body
            for (int pass = CS ? 0 : 1; pass < (WL ? 2 : 1); ++pass) {
                const double Ts_q = Ts;
                if (CS && pass == 0) {
                    double Qns, Tau, Qlat;
                    update_qnsol_tau(air, Ts, qs_, t_zu, q_zu, us, ts, qst, p.wnd, Ub, p.rlw, Qns, Tau, Qlat);
                    dT_cs = cool_skin_dT<true>(alpha, p.Qsw, Qns, us, Qlat);
                    Ts = p.sst + dT_cs;
                    if (WL) Ts = Ts + wl.dT;
                } else {
                    if (commit) {
                        double Qns, Tau, Qlat;
                        update_qnsol_tau(air, Ts, qs_, t_zu, q_zu, us, ts, qst, p.wnd, Ub, p.rlw, Qns, Tau, Qlat);
                        wl_coare(wl, wc, p.Qsw, Qns, Tau, u.rdt, u.gdept, true);
                    }
                    Ts = p.sst + wl.dT;
                    if (CS) Ts = Ts + dT_cs;
                }
                if (Ts != Ts_q) qs_ = KC(RDCT_QSAT_SALT) * q_sat(abm::dmax(Ts, 200.), p.slp);
            }
        }
        if (SKIN || !ZTEQ || !V36) {
            dt = floor_abs(t_zu - Ts, KC(1.E-09));
            dq = floor_abs(q_zu - qs_, KC(1.E-12));
        }
    }
    Coeffs c;
    const double r = fdiv(us, Ub);
    c.Cd = abm::dmax(r * r, CX_MIN);
    c.Ch = abm::dmax(fdiv(r * ts, dt), CX_MIN);
    c.Ce = abm::dmax(fdiv(r * qst, dq), CX_MIN);
    c.t_zu = t_zu; c.q_zu = q_zu; c.Ub = Ub; c.Ts = Ts; c.qs = qs_;
    // optional outputs, src/mod_blk_coare3p6.f90:391-401
    const double t0 = 1. / (u.log_zu - log_z0);
    dg.CdN = abm::dmax(VKARMN2 * t0 * t0, CX_MIN);
    dg.ChN = dg.CeN = abm::dmax(VKARMN2 * t0 / (u.log_zu - log_z0t), CX_MIN);
    dg.z0 = z0; dg.us = us; dg.L = 1. / r1oL; dg.UN10 = us * INV_VKARMN * (u.log_10 - log_z0);
    dg.dT_cs = dT_cs;
    return c;
}

// ---------------------------------------------------------------------------
// ECMWF (IFS Cy40/45), src/mod_blk_ecmwf.f90:63-383
// ---------------------------------------------------------------------------
template <bool CS, bool WL, bool ZTEQ>
ABD Coeffs solve_ecmwf(const Uniform &u, const PointIn &p, WarmLayer &wl, Diag &dg)
{
    constexpr bool SKIN = CS || WL;
    constexpr double charn0 = 0.018, zi0 = 1000., Beta0 = 1., alpha_M = 0.11, alpha_H = 0.40, alpha_Q = 0.62;

    double Ts = p.sst, qs_ = p.ssq;
    double alpha = 0.;
    WlEcmwfCtx wec = {};
    if (SKIN) {
        if (CS) Ts = Ts - 0.25;
        qs_ = RDCT_QSAT_SALT * q_sat(abm::dmax(Ts, 200.), p.slp);
        alpha = alpha_sw(p.sst);
        if (WL) wec = wl_ecmwf_ctx(wl.Hz, u.gdept);
    }

    const Guess g = first_guess_coare<ZTEQ>(u, Ts, p.theta_zt, qs_, p.q_zt, p.wnd, charn0);
    double us = g.us, ts = g.ts, qst = g.qs, t_zu = g.t_zu, q_zu = g.q_zu, Ub = g.Ub;
    double z0 = g.z0;
    double log_z0 = abm::dlog(z0);
    const double nu_a = visc_air(p.theta_zt);

    double dt = floor_abs(t_zu - Ts, 1.E-09);
    double dq = floor_abs(q_zu - qs_, 1.E-12);

    double r1oL = one_on_L(t_zu, q_zu, us, ts, qst);
    const double x0 = fdiv(VKARMN, fdiv(0.00115, fdiv(VKARMN, u.log_10 - log_z0)));
    double z0t = abm::dmin(abm::dmax(10. * abm::dexp(-x0), 1.E-9), 1.);
    double log_z0t = abm::dmin(abm::dmax(u.log_10 - x0, LOG_1EM9), 0.);

    double Fm, Fh, psi_h_u;
    if (nonneg(r1oL)) {
        const PsiMH pu = psi_mh_ecmwf_stable(u.zu * r1oL);
        psi_h_u = pu.h;
        Fm = u.log_zu - log_z0 - pu.m + psi_m_ecmwf_stable(z0 * r1oL);
        Fh = u.log_zu - log_z0t - psi_h_u + psi_h_ecmwf_stable(z0t * r1oL);
    } else {
        const PsiMH pu = psi_mh_ecmwf_unstable(u.zu * r1oL);
        psi_h_u = pu.h;
        Fm = u.log_zu - log_z0 - pu.m + psi_m_ecmwf_unstable(z0 * r1oL);
        Fh = u.log_zu - log_z0t - psi_h_u + psi_h_ecmwf_unstable(z0t * r1oL);
    }
    double log_z0q = 0., psi_h_z0q = 0., dT_cs = 0.;

#pragma unroll 1
    for (int jit = 1; jit <= u.nb_iter; ++jit) {
        const double Rib = ri_bulk(u.zu, Ts, t_zu, qs_, q_zu, Ub);
        r1oL = clip_abs(fdiv(Rib * Fm * Fm, Fh * u.zu), 200.);

        // one stability branch for the four psi of this half-step (all arguments share the sign of 1/L)
        const bool stable = nonneg(r1oL);
        double psi_m_u, psi_h_t = 0., psi_m_z0old;
        if (stable) {
            const PsiMH pu = psi_mh_ecmwf_stable(u.zu * r1oL);
            psi_m_u = pu.m;
            psi_h_u = pu.h;
            if (!ZTEQ) psi_h_t = psi_h_ecmwf_stable(u.zt * r1oL);
            psi_m_z0old = psi_m_ecmwf_stable(z0 * r1oL);
        } else {
            const PsiMH pu = psi_mh_ecmwf_unstable(u.zu * r1oL);
            psi_m_u = pu.m;
            psi_h_u = pu.h;
            if (!ZTEQ) psi_h_t = psi_h_ecmwf_unstable(u.zt * r1oL);
            psi_m_z0old = psi_m_ecmwf_unstable(z0 * r1oL);
        }

        Fm = u.log_zu - log_z0 - psi_m_u + psi_m_z0old;

        us = fdiv(Ub * KC(VKARMN), Fm);
        const double us2 = us * us;
        double tmp0 = fdiv(nu_a, us);
        z0 = abm::dmin(fabs(KC(alpha_M) * tmp0 + KC(charn0) * us2 * KC(INV_GRAV)), KC(0.001));
        z0t = abm::dmin(fabs(KC(alpha_H) * tmp0), KC(0.001));
        const double z0q = abm::dmin(fabs(KC(alpha_Q) * tmp0), KC(0.001));
        log_z0 = abm::dlog(z0);
        const double log_t0 = abm::dlog(fabs(tmp0));          // LOG(alpha nu/u*) = LOG(alpha) + LOG(nu/u*)
        log_z0t = abm::dmin(KC(LOG_0P40) + log_t0, KC(LOG_1EM3));
        log_z0q = abm::dmin(KC(LOG_0P62) + log_t0, KC(LOG_1EM3));

        double psi_m_z0, psi_h_z0t;
        if (stable) {
            psi_m_z0 = psi_m_ecmwf_stable(z0 * r1oL);
            psi_h_z0t = psi_h_ecmwf_stable(z0t * r1oL);
            psi_h_z0q = psi_h_ecmwf_stable(z0q * r1oL);
        } else {
            psi_m_z0 = psi_m_ecmwf_unstable(z0 * r1oL);
            psi_h_z0t = psi_h_ecmwf_unstable(z0t * r1oL);
            psi_h_z0q = psi_h_ecmwf_unstable(z0q * r1oL);
        }

        const double cv = abm::fast_cbrt(abm::dmax(-zi0 * r1oL * INV_VKARMN, 0.));
        tmp0 = Beta0 * Beta0 * us2 * (cv * cv);
        Ub = abm::dmax(abm::fast_sqrt(p.wnd * p.wnd + tmp0), KC(0.2));

        tmp0 = psi_h_u - psi_h_z0t;
        double tmp1 = fdiv(KC(VKARMN), u.log_zu - log_z0t - tmp0);
        ts = dt * tmp1;
        if (!ZTEQ) {
            tmp1 = u.log_ztu + tmp0 - psi_h_t + psi_h_z0t;
            t_zu = p.theta_zt - ts * INV_VKARMN * tmp1;
        } else {
            t_zu = p.theta_zt;
        }
        tmp0 = psi_h_u - psi_h_z0q;
        tmp1 = fdiv(KC(VKARMN), u.log_zu - log_z0q - tmp0);
        qst = dq * tmp1;
        if (!ZTEQ) {
            tmp1 = u.log_ztu + tmp0 - psi_h_t + psi_h_z0q;
            q_zu = abm::dmax(p.q_zt - qst * INV_VKARMN * tmp1, 0.);
        } else {
            q_zu = abm::dmax(p.q_zt, 0.);
        }

        Fm = u.log_zu - log_z0 - psi_m_u + psi_m_z0;
        Fh = u.log_zu - log_z0t - psi_h_u + psi_h_z0t;

        if (SKIN) {
            // pass 0: cool skin, pass 1: warm layer -- advanced at every iteration (SURVEY 8a quirk 2)
            const AirZu air = air_at_zu(u.zu, t_zu, q_zu, p.slp);
#pragma unroll 1   // cool-skin pass and warm-layer pass rolled: UPDATE_QNSOL_TAU and q_sat exist once in the loop body
            for (int pass = CS ? 0 : 1; pass < (WL ? 2 : 1); ++pass) {
                double Qns, Tau, Qlat;
                update_qnsol_tau(air, Ts, qs_, t_zu, q_zu, us, ts, qst, p.wnd, Ub, p.rlw, Qns, Tau, Qlat);
                if (CS && pass == 0) {
                    dT_cs = cool_skin_dT<false>(alpha, p.Qsw, Qns, us, 0.);
                    Ts = p.sst + dT_cs;
                    if (WL) Ts = Ts + wl.dT;
                } else {
                    wl_ecmwf(wl, wec, alpha, p.Qsw, Qns, us, u.rdt);
                    Ts = p.sst + wl.dT;
                    if (CS) Ts = Ts + dT_cs;
                }
                qs_ = KC(RDCT_QSAT_SALT) * q_sat(abm::dmax(Ts, 200.), p.slp);
            }
        }
        dt = floor_abs(t_zu - Ts, KC(1.E-09));
        dq = floor_abs(q_zu - qs_, KC(1.E-12));
    }
    Coeffs c;
    const double Fq = u.log_zu - log_z0q - psi_h_u + psi_h_z0q;
    const double k2_o_Fm = fdiv(VKARMN2, Fm);
    c.Cd = abm::dmax(fdiv(k2_o_Fm, Fm), CX_MIN);
    c.Ch = abm::dmax(fdiv(k2_o_Fm, Fh), CX_MIN);
    c.Ce = abm::dmax(fdiv(k2_o_Fm, Fq), CX_MIN);
    c.t_zu = t_zu; c.q_zu = q_zu; c.Ub = Ub; c.Ts = Ts; c.qs = qs_;
    // optional outputs, src/mod_blk_ecmwf.f90:361-371
    const double t0 = 1. / (u.log_zu - log_z0);
    dg.CdN = abm::dmax(VKARMN2 * t0 * t0, CX_MIN);
    dg.ChN = dg.CeN = abm::dmax(VKARMN2 * t0 / (u.log_zu - log_z0t), CX_MIN);
    dg.z0 = z0; dg.us = us; dg.L = 1. / r1oL; dg.UN10 = us * INV_VKARMN * (u.log_10 - log_z0);
    dg.dT_cs = dT_cs;
    return c;
}

// ---------------------------------------------------------------------------
// ANDREAS (Andreas et al. 2015), src/mod_blk_andreas.f90:66-304
// ---------------------------------------------------------------------------
template <bool ZTEQ>
ABD Coeffs solve_andreas(const Uniform &u, const PointIn &p, Diag &dg)
{
    const double rRi_max = 0.15, rCs_min = 0.35E-3;
    const double Ub = abm::dmax(0.25, p.wnd);
    const double r_Ub = abm::fast_rcp(Ub);
    double UN10 = Ub;
    double t_zu = p.theta_zt, q_zu = p.q_zt;
    const double sq0 = sqrt(1.1E-3);
    double t_star = 1.1E-3 / sq0 * (t_zu - p.sst);
    double q_star = 1.1E-3 / sq0 * (q_zu - p.ssq);
    double RiB = ri_bulk(u.zu, p.sst, t_zu, p.ssq, q_zu, Ub);
    double u_star = 0., zeta_u = 0., z0 = 0., psi_m = 0.;

#pragma unroll 1
    for (int jit = 1; jit <= u.nb_iter; ++jit) {
        if (RiB < rRi_max) {
            const double za = UN10 - KC(8.271);
            u_star = KC(0.239) + KC(0.0433) * (za + abm::fast_sqrt_pos(KC(0.12) * za * za + KC(0.181)));   // :275-293
        } else {
            u_star = KC(0x1.47ae147ae147bp-7) * Ub;   // SQRT(Cx_min) = 0.01
        }
        zeta_u = u.zu * one_on_L(t_zu, q_zu, u_star, t_star, q_star);
        const double r = u_star * r_Ub;
        const double Cd = abm::dmax(r * r, CX_MIN);
        const double zeta_t = fdiv(zeta_u, u.zu) * u.zt;
        const bool adjust = !ZTEQ && jit > 1;
        double psi_h_u, psi_h_t = 0.;
        if (nonneg(abm::dmin(zeta_u, 15.))) {
            psi_m = psi_m_andreas_stable(zeta_u);
            psi_h_u = psi_h_andreas_stable(zeta_u);
            if (adjust) psi_h_t = psi_h_andreas_stable(zeta_t);
        } else {
            const PsiMH r = psi_mh_andreas_unstable(zeta_u);
            psi_m = r.m;
            psi_h_u = r.h;
            if (adjust) psi_h_t = psi_h_andreas_unstable(zeta_t);
        }
        // z0 = MIN(zu EXP(-(k/SQRT(Cd) + psi_m)), z0_sea_max), kept together with its logarithm
        const double log_z0 = abm::dmin(u.log_zu - (VKARMN * abm::fast_rsqrt(Cd) + psi_m), LOG_Z0_SEA_MAX);
        z0 = abm::dexp(log_z0);

        const double Rer = fdiv(z0 * u_star, visc_air(t_zu));
        const double log_Rer = abm::dlog(abm::dmax(Rer, 1.E-300));
        const double log_z0t = log_z0tq_LKB(1, Rer, log_Rer, log_z0);
        const double log_z0q = log_z0tq_LKB(2, Rer, log_Rer, log_z0);

        t_star = fdiv((t_zu - p.sst) * VKARMN, u.log_zu - log_z0t - psi_h_u);
        q_star = fdiv((q_zu - p.ssq) * VKARMN, u.log_zu - log_z0q - psi_h_u);

        if (adjust) {
            const double tmp = u.log_ztu + psi_h_u - psi_h_t;
            t_zu = p.theta_zt - t_star * INV_VKARMN * tmp;
            q_zu = p.q_zt - q_star * INV_VKARMN * tmp;
            RiB = ri_bulk(u.zu, p.sst, t_zu, p.ssq, q_zu, Ub);
        }
        UN10 = abm::dmax(0.1, Ub - u_star * INV_VKARMN * (u.log_zu10 - psi_m));   // UN10_from_ustar, mod_phymbl.f90:1498-1510
    }
    Coeffs c;
    const double r = u_star * r_Ub;
    c.Cd = abm::dmax(r * r, CX_MIN);
    const double d1 = floor_abs(t_zu - p.sst, 1.E-6);
    const double d2 = floor_abs(q_zu - p.ssq, 1.E-9);
    c.Ch = abm::dmax(fdiv(r * t_star, d1), rCs_min);
    c.Ce = abm::dmax(fdiv(r * q_star, d2), rCs_min);
    c.t_zu = t_zu; c.q_zu = q_zu; c.Ub = Ub; c.Ts = p.sst; c.qs = p.ssq;
    // optional outputs, src/mod_blk_andreas.f90:256-267
    const double log_z0 = abm::dlog(z0);
    const double t0 = 1. / (u.log_zu - log_z0);
    dg.CdN = abm::dmax(VKARMN2 * t0 * t0, CX_MIN);
    const double Rer = z0 * u_star / visc_air(t_zu);
    const double log_Rer = abm::dlog(abm::dmax(Rer, 1.E-300));
    dg.ChN = VKARMN2 * t0 / (u.log_zu - log_z0tq_LKB(1, Rer, log_Rer, log_z0));
    dg.CeN = VKARMN2 * t0 / (u.log_zu - log_z0tq_LKB(2, Rer, log_Rer, log_z0));
    dg.z0 = z0; dg.us = u_star; dg.L = u.zu / zeta_u;
    dg.UN10 = Ub - u_star * INV_VKARMN * (u.log_zu10 - psi_m);
    dg.dT_cs = 0.;
    return c;
}

// ---------------------------------------------------------------------------
// one TURB_<ALGO> call: the solver of the algorithm, with cool-skin (CS) / warm-layer (WL) where it has them
// ---------------------------------------------------------------------------
template <int ALGO, bool CS, bool WL, bool ZTEQ>
ABD Coeffs solve_ocean(const Uniform &u, const PointIn &p, WarmLayer &wl, Diag &dg)
{
    if (ALGO == NCAR) return solve_ncar<ZTEQ>(u, p, dg);
    else if (ALGO == ANDREAS) return solve_andreas<ZTEQ>(u, p, dg);
    else if (ALGO == ECMWF) return solve_ecmwf<CS, WL, ZTEQ>(u, p, wl, dg);
    else return solve_coare<ALGO == COARE3P6, CS, WL, ZTEQ>(u, p, wl, dg);
}

#undef ABD
}  // namespace abd
