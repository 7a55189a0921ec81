// ab_math.cuh -- the kernels' own FP64 exp / exp10 / log / log10 / atan / pow, and Goff's e_sat and the unstable stability
// functions as piecewise polynomials.
//
// Why not libdevice: ptxas builds every FP64 literal of CUDA's math functions with two 32-bit moves
// (UMOV / IMAD.MOV), which made ~35 % of the issued instructions of the flux kernels and a 188 KB
// code footprint (instruction-cache misses were the top stall in the round-1 ncu capture).  These
// versions read their coefficients from the constant bank (tools/gen_math_tables.py ->
// ab_math_tables.cuh; one LDCU.128 brings two coefficients), skip the denormal / NaN / huge-argument
// paths the physics never takes, and stay within ~2 ulp of the correctly rounded result -- five
// orders of magnitude inside the 1e-10 parity tolerance (tests/test_math_accuracy.py checks them
// against mpmath on the host, tests/test_gpu_parity.py end to end).
//
// Domain contract (asserted by the callers in ab_device.cuh):
//   dexp/dexp10 : any finite x; results below ~1e-304 flush to 0, x > 700 is not supported
//   dlog/dlog10 : x > 0 and normal
//   datan       : any finite x
//   dpowr       : x >= 0 (0**y = 0 for y > 0)
#pragma once

#ifdef ABM_HOST_TEST
// plain C++ build of the same source for the host-side accuracy tests
#include <cmath>
#include <cstdint>
#include <cstring>
#define ABM_FN static inline
#define ABM_BIG static inline
#define ABM_TABLE static const
#define ABM_GTABLE static const
#define ABM_LDG(p) (*(p))
struct double2 { double x, y; };
namespace abm {
static inline int hi_word(double x) { int64_t b; std::memcpy(&b, &x, 8); return (int)(b >> 32); }
static inline int lo_word(double x) { int64_t b; std::memcpy(&b, &x, 8); return (int)(b & 0xffffffff); }
static inline double make_double(int hi, int lo)
{
    int64_t b = ((int64_t)hi << 32) | (uint32_t)lo;
    double x; std::memcpy(&x, &b, 8); return x;
}
static inline double rcp_seed(double y) { return (double)(float)(1.0 / y); }   // ~24-bit seed like MUFU.RCP64H
static inline double dmax(double a, double b) { return (a > b) ? a : b; }
static inline double dmin(double a, double b) { return (a < b) ? a : b; }
// seeds of the root functions, degraded to the worst accuracy the device versions may have (2^-21)
static inline double rsqrt_seed(double y) { return (double)(float)(1.0 / std::sqrt(y)) * (1.0 + 0x1p-21); }
static inline double pow_seed(double y, float p) { return (double)(float)std::pow(y, (double)p) * (1.0 - 0x1p-21); }
}
#else
#include <cuda_runtime.h>
#define ABM_FN __device__ __forceinline__
#define ABM_LDG(p) __ldg(p)
// -DABM_NOINLINE=1 keeps exp/log/atan out of line (one body per kernel): smaller instruction footprint
// at the price of call overhead and less interleaving
#if defined(ABM_NOINLINE) && ABM_NOINLINE
#define ABM_BIG static __device__ __noinline__
#else
#define ABM_BIG __device__ __forceinline__
#endif
namespace abm {
ABM_FN int hi_word(double x) { return __double2hiint(x); }
ABM_FN int lo_word(double x) { return __double2loint(x); }
ABM_FN double make_double(int hi, int lo) { return __hiloint2double(hi, lo); }
ABM_FN double rcp_seed(double y)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(y));   // MUFU.RCP64H, rel. error <= 2^-23
    return r;
}
// MAX / MIN as the Fortran intrinsics define them (a > b ? a : b): one DSETP and two FSEL.  CUDA's fmax / fmin return
// the non-NaN operand, which ptxas lowers to 8-9 instructions per call (DSETP.MAX with a NaN predicate, moves, a
// predicated LOP3 that quiets the NaN ...): 8 % of what the COARE + skin kernel executed.  The setp / selp pair is
// written in PTX because NVVM canonicalises the C++ ternary back into max.f64.
ABM_FN double dmax(double a, double b)
{
    double d;
    asm("{\n\t.reg .pred p;\n\tsetp.gt.f64 p, %1, %2;\n\tselp.f64 %0, %1, %2, p;\n\t}" : "=d"(d) : "d"(a), "d"(b));
    return d;
}
ABM_FN double dmin(double a, double b)
{
    double d;
    asm("{\n\t.reg .pred p;\n\tsetp.lt.f64 p, %1, %2;\n\tselp.f64 %0, %1, %2, p;\n\t}" : "=d"(d) : "d"(a), "d"(b));
    return d;
}
ABM_FN double rsqrt_seed(double y)
{
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(y));   // MUFU.RSQ64H
    return r;
}
// y**p for y in the normal FP32 range through the FP32 special-function unit (MUFU.LG2, MUFU.EX2): ~2^-22,
// and off the FP64 pipe
ABM_FN double pow_seed(double y, float p)
{
    float l, r;
    const float f = (float)y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(f));
    l *= p;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(l));
    return (double)r;
}
}
#endif

#include "ab_math_tables.cuh"

namespace abm {

// 1/y for normal y: seed r0 (rel. error e <= 2^-23), then r1 = r0(1+e) and r2 = r1(1+e^2): the second
// step reuses e*e instead of a fresh residual (one dependent FMA less; ~1.5 ulp, corrected by callers
// that need a quotient, see abd::fdiv)
ABM_FN double fast_rcp(double y)
{
    const double r0 = rcp_seed(y);
    const double e = fma(-y, r0, 1.0);
    return fma(r0, fma(e, e, e), r0);            // r0 (1 + e + e^2): error e^3 <= 2^-69
}

// Roots: one seed of relative accuracy d <= 2^-21 and ONE step of cubic convergence.  With e = 1 - x y^n
// (~ n d) the exact root is y (1-e)^(-1/n) = y (1 + e/n + (n+1) e^2 / (2 n^2) + O(e^3)); the neglected term is
// below 2^-60.  About 1 ulp, for x > 0 in the normal range (callers guard zero).
// CUDA's rsqrt / rcbrt / cbrt cost 28 / 47 / 49 instructions here (special-case handling, FP64 seeds).
ABM_FN double fast_rsqrt(double x)              // x**(-1/2)
{
    const double y = rsqrt_seed(x);
    const double e = fma(-(x * y), y, 1.0);
    return fma(y * e, fma(0.375, e, 0.5), y);
}
// sqrt for x >= 0 in the normal range (0 and below 2^-962 -> 0): CUDA's sqrt is 12 instructions inline but up to 34
// where ptxas keeps its slow-path call (10 % of the ECMWF + skin kernel was the sqrt of the warm-layer inner loop)
ABM_FN double fast_sqrt(double x)
{
    const double r = fast_rsqrt(x);
    return (hi_word(x) >= 0x03d00000) ? x * r : 0.;   // x >= 2^-962
}
// the same for callers whose argument is provably positive and normal (no zero guard: 1 compare and 2 selects less)
ABM_FN double fast_sqrt_pos(double x) { return x * fast_rsqrt(x); }
ABM_FN double fast_rcbrt(double x)              // x**(-1/3), x in the normal FP32 range
{
    const double y = pow_seed(x, -1.0f / 3.0f);
    const double e = fma(-(x * y), y * y, 1.0);
    return fma(y * e, fma(MATH_K[K_TWO_NINTHS], e, MATH_K[K_ONE_THIRD]), y);
}
ABM_FN double fast_r4rt(double x)               // x**(-1/4), x in the normal FP32 range
{
    const double y = pow_seed(x, -0.25f);
    const double y2 = y * y;
    const double e = fma(-(x * y2), y2, 1.0);
    return fma(y * e, fma(5.0 / 32.0, e, 0.25), y);
}
// x**0.75 and x**(1/3) for x >= 0; below 2^-100 (where the FP32 seed would leave its range) the result is 0:
// the callers add it to 1 (delta_skin_layer) or to a squared wind speed (gustiness)
// (the guards compare the high word: x > 2^-100 without an FP64 compare or a 64-bit literal)
ABM_FN double pow075(double x) { return (hi_word(x) >= 0x39b00000) ? x * fast_r4rt(x) : 0.; }
ABM_FN double pow075_pos(double x) { return x * fast_r4rt(x); }   // x inside the normal FP32 range (caller's guarantee)
ABM_FN double fast_cbrt(double x)
{
    if (hi_word(x) < 0x39b00000) return 0.;
    const double r = fast_rcbrt(x);
    return x * (r * r);
}

// p(r) ~ exp(r) on |r| <= ln2/2 (Estrin: depth 5 instead of 11 dependent FMAs), then * 2^k through
// the exponent field
ABM_FN double exp_core(double r, int k)
{
    const double r2 = r * r, r4 = r2 * r2, r8 = r4 * r4;
    const double a0 = fma(EXP_C[1], r, EXP_C[0]), a1 = fma(EXP_C[3], r, EXP_C[2]), a2 = fma(EXP_C[5], r, EXP_C[4]);
    const double a3 = fma(EXP_C[7], r, EXP_C[6]), a4 = fma(EXP_C[9], r, EXP_C[8]), a5 = fma(EXP_C[11], r, EXP_C[10]);
    const double b0 = fma(a1, r2, a0), b1 = fma(a3, r2, a2), b2 = fma(a5, r2, a4);
    const double p = fma(b2, r8, fma(b1, r4, b0));
    return make_double(hi_word(p) + (k << 20), lo_word(p));
}

ABM_BIG double dexp_poly(double x)
{
    const double MAGIC = 6755399441055744.0;   // 1.5 * 2^52: adding it rounds to nearest integer
    const double t = fma(x, MATH_K[K_L2E], MAGIC);
    const int k = lo_word(t);
    const double kf = t - MAGIC;
    double r = fma(kf, -MATH_K[K_LN2_HI], x);
    r = fma(kf, -MATH_K[K_LN2_LO], r);
    const double v = exp_core(r, k);
    return (x < -700.) ? 0. : v;
}

ABM_BIG double dexp10_poly(double x)
{
    const double MAGIC = 6755399441055744.0;
    const double t = fma(x, MATH_K[K_L2T], MAGIC);
    const int k = lo_word(t);
    const double kf = t - MAGIC;
    double r = fma(kf, -MATH_K[K_LG2_HI], x);
    r = fma(kf, -MATH_K[K_LG2_LO], r);
    const double v = exp_core(r * MATH_K[K_LN10], k);
    return (x < -304.) ? 0. : v;
}

// log(x) = k ln2 + log(m), m in [sqrt(2)/2, sqrt(2)); log(m) = 2 atanh(s), s = (m-1)/(m+1)
ABM_BIG double dlog_poly(double x)
{
    int hx = hi_word(x);
    int k = (hx >> 20) - 1023;
    hx &= 0x000fffff;
    const int i = (hx + 0x95f64) & 0x100000;
    hx |= (i ^ 0x3ff00000);
    k += (i >> 20);
    const double f = make_double(hx, lo_word(x)) - 1.0;
    const double s = f * fast_rcp(2.0 + f);
    const double z = s * s;
    const double z2 = z * z;
    const double a0 = fma(LOG_C[1], z, LOG_C[0]), a1 = fma(LOG_C[3], z, LOG_C[2]), a2 = fma(LOG_C[5], z, LOG_C[4]);
    const double p = fma(fma(LOG_C[6], z2, a2), z2 * z2, fma(a1, z2, a0));
    const double R = z * p;
    const double hfsq = 0.5 * f * f;
    const double dk = (double)k;
    return dk * MATH_K[K_LN2_HI] - ((hfsq - fma(s, hfsq + R, dk * MATH_K[K_LN2_LO])) - f);
}

// ---------------------------------------------------------------------------
// Table-driven exp / log (default): a 64-entry table of 2^(j/64) and a 256-entry table of
// {1/c_j, -log(1/c_j)} (4.5 KB, copied to shared memory by each block) shrink the polynomials to degree 3 / 4:
// 10 FP64 instructions per exp instead of 18, 13 per log instead of 23 (no reciprocal).
// ---------------------------------------------------------------------------
#ifndef ABM_SMEM_TABLES
#define ABM_SMEM_TABLES 1   // measured 3 % faster than __ldg of the global tables (64-bit address arithmetic)
#endif
// which psi tables a kernel reads (psi_table): load_tables copies only those
enum { PSI_TABLES_NONE = 0, PSI_TABLES_COARE = 1, PSI_TABLES_PAULSON = 2, PSI_TABLES_ALL = 3 };
#if ABM_SMEM_TABLES && !defined(ABM_HOST_TEST)
// block-local copies of the tables in shared memory (4.5 KB, 3.2 KB of e_sat coefficients and 10 KB per family of psi
// coefficients; 32-bit addressing, LDS instead of LDG); every kernel must call abm::load_tables() (all threads) before the
// first exp/log/esat_table/psi_table, naming in PSI every psi family it evaluates from a table (a shared array a kernel
// does not reference takes no shared memory)
__shared__ double S_EXP_T[64];
__shared__ double S_LOG_T[512];
__shared__ __align__(16) double S_ESAT_T[8 * ESAT_ROWS];
__shared__ __align__(16) double S_PSI_COARE_T[2 * (PSI_DEG + 1) * PSI_ROWS];
__shared__ __align__(16) double S_PSI_PAULSON_T[2 * (PSI_DEG + 1) * PSI_ROWS];
ABM_FN void copy_table2(double *dst, const double *src, int n2)
{
    for (int i = threadIdx.x; i < n2; i += blockDim.x)
        reinterpret_cast<double2 *>(dst)[i] = reinterpret_cast<const double2 *>(src)[i];
}
template <int PSI = PSI_TABLES_ALL>
ABM_FN void load_tables()
{
    for (int i = threadIdx.x; i < 64; i += blockDim.x) S_EXP_T[i] = EXP_T[i];
    for (int i = threadIdx.x; i < 512; i += blockDim.x) S_LOG_T[i] = LOG_T[i];
    copy_table2(S_ESAT_T, ESAT_T, 4 * ESAT_ROWS);
    if (PSI & PSI_TABLES_COARE) copy_table2(S_PSI_COARE_T, PSI_COARE_T, (PSI_DEG + 1) * PSI_ROWS);
    if (PSI & PSI_TABLES_PAULSON) copy_table2(S_PSI_PAULSON_T, PSI_PAULSON_T, (PSI_DEG + 1) * PSI_ROWS);
    __syncthreads();
}
#define ABM_EXP_T(i) S_EXP_T[i]
#define ABM_LOG_T(i) S_LOG_T[i]
#define ABM_ESAT_T2(i) reinterpret_cast<const double2 *>(S_ESAT_T)[i]
#define ABM_PSI_T(fam) S_PSI_##fam##_T
#define ABM_PSI_T2(t, i) reinterpret_cast<const double2 *>(t)[i]
#else
template <int PSI = PSI_TABLES_ALL>
ABM_FN void load_tables() {}
#define ABM_EXP_T(i) ABM_LDG(&EXP_T[i])
#define ABM_LOG_T(i) ABM_LDG(&LOG_T[i])
#define ABM_ESAT_T2(i) ABM_LDG(reinterpret_cast<const double2 *>(ESAT_T) + (i))
#define ABM_PSI_T(fam) PSI_##fam##_T
#define ABM_PSI_T2(t, i) ABM_LDG(reinterpret_cast<const double2 *>(t) + (i))
#endif

// exp(r) for |r| <= ln2/128 times 2^(k/64), k = 64 m + j
ABM_FN double expt_core(double r, int k)
{
    const double T = ABM_EXP_T(k & 63);
    const double r2 = r * r;
    double q = fma(EXPT_C[3], r, EXPT_C[2]);
    q = fma(q, r, EXPT_C[1]);
    q = fma(q, r, EXPT_C[0]);
    const double v = fma(T, fma(r2, q, r), T);
    return make_double(hi_word(v) + ((k >> 6) << 20), lo_word(v));
}
ABM_BIG double dexp_table(double x)
{
    const double MAGIC = 6755399441055744.0;
    const double t = fma(x, MATH_K[K_L2E64], MAGIC);
    const int k = lo_word(t);
    const double kf = t - MAGIC;
    double r = fma(kf, -MATH_K[K_LN2_64_HI], x);
    r = fma(kf, -MATH_K[K_LN2_64_LO], r);
    const double v = expt_core(r, k);
    return (x < -700.) ? 0. : v;
}
// the same without the underflow guard, for call sites whose argument is provably inside [-700, 700]
ABM_BIG double dexp_table_bounded(double x)
{
    const double MAGIC = 6755399441055744.0;
    const double t = fma(x, MATH_K[K_L2E64], MAGIC);
    const int k = lo_word(t);
    const double kf = t - MAGIC;
    double r = fma(kf, -MATH_K[K_LN2_64_HI], x);
    r = fma(kf, -MATH_K[K_LN2_64_LO], r);
    return expt_core(r, k);
}
ABM_BIG double dexp10_table(double x)
{
    const double MAGIC = 6755399441055744.0;
    const double t = fma(x, MATH_K[K_L2T64], MAGIC);
    const int k = lo_word(t);
    const double kf = t - MAGIC;
    double r = fma(kf, -MATH_K[K_LG2_64_HI], x);
    r = fma(kf, -MATH_K[K_LG2_64_LO], r);
    const double v = expt_core(r * MATH_K[K_LN10], k);
    return (x < -304.) ? 0. : v;
}
ABM_BIG double dexp10_table_bounded(double x)   // |x| <= 300 guaranteed by the caller
{
    const double MAGIC = 6755399441055744.0;
    const double t = fma(x, MATH_K[K_L2T64], MAGIC);
    const int k = lo_word(t);
    const double kf = t - MAGIC;
    double r = fma(kf, -MATH_K[K_LG2_64_HI], x);
    r = fma(kf, -MATH_K[K_LG2_64_LO], r);
    return expt_core(r * MATH_K[K_LN10], k);
}
// log(x) = e ln2 + lc_j + log1p(m rc_j - 1), m in [0.708, 1.416) (so that x ~ 1 has e = 0 and the exact
// entry c = 1), j = interval of m's hi word
ABM_BIG double dlog_table(double x)
{
    const int hx = hi_word(x);
    const int e = (hx - 0x3fe6a800) >> 20;
    const int u = hx - (e << 20);
    const int j = (u - 0x3fe6a800) >> 12;
    const double m = make_double(u, lo_word(x));
    const double rc = ABM_LOG_T(2 * j), lc = ABM_LOG_T(2 * j + 1);
    const double r = fma(m, rc, -1.0);
    const double r2 = r * r;
    double q = fma(LOGT_C[4], r, LOGT_C[3]);
    q = fma(q, r, LOGT_C[2]);
    q = fma(q, r, LOGT_C[1]);
    q = fma(q, r, LOGT_C[0]);
    const double lp = fma(r2, q, r);
    const double de = (double)e;
    return fma(de, MATH_K[K_LN2_HI], lc) + fma(de, MATH_K[K_LN2_LO], lp);
}

#if defined(ABM_POLY_MATH) && ABM_POLY_MATH
ABM_FN double dexp(double x) { return dexp_poly(x); }
ABM_FN double dexp10(double x) { return dexp10_poly(x); }
ABM_FN double dexp_b(double x) { return dexp_poly(x); }
ABM_FN double dexp10_b(double x) { return dexp10_poly(x); }
ABM_FN double dlog(double x) { return dlog_poly(x); }
#else
ABM_FN double dexp(double x) { return dexp_table(x); }
ABM_FN double dexp10(double x) { return dexp10_table(x); }
ABM_FN double dexp_b(double x) { return dexp_table_bounded(x); }      // argument inside [-700, 700]
ABM_FN double dexp10_b(double x) { return dexp10_table_bounded(x); }  // argument inside [-300, 300]
ABM_FN double dlog(double x) { return dlog_table(x); }
#endif

ABM_FN double dlog10(double x) { return dlog(x) * MATH_K[K_LOG10E]; }

// Goff's saturation vapour pressure over water [Pa] for 229 <= T < 331 (the caller checks the range) from the
// piecewise polynomial ESAT_T: ~25 instructions instead of the quotient, log10 and three exp10 of the formula (~115),
// within 2 ulp of it.  Row m = rint(T / h) is centred on T_c = h m; T - T_c is exact (|T - T_c| <= h / 2 and h is a
// power of two), so the only rounding is the evaluation's.  Estrin form: e_sat sits on the dependent chain of the
// skin loops.  The four coefficient pairs of a row are ESAT_ROWS apart (tools/gen_math_tables.py: bank spread).
ABM_FN double esat_table(double T)
{
    const double MAGIC = 6755399441055744.0;   // 1.5 * 2^52: adding it rounds to nearest integer
    const double t = fma(T, 1. / ESAT_H, MAGIC);
    const double x = fma(t - MAGIC, -ESAT_H, T) * (2. / ESAT_H);
    const int i = lo_word(t) - ESAT_M0;
    const double2 c01 = ABM_ESAT_T2(i), c23 = ABM_ESAT_T2(i + ESAT_ROWS), c45 = ABM_ESAT_T2(i + 2 * ESAT_ROWS),
                  c67 = ABM_ESAT_T2(i + 3 * ESAT_ROWS);
    const double x2 = x * x;
    const double a0 = fma(c01.y, x, c01.x), a1 = fma(c23.y, x, c23.x), a2 = fma(c45.y, x, c45.x), a3 = fma(c67.y, x, c67.x);
    return fma(fma(a3, x2, a2), x2 * x2, fma(a1, x2, a0));
}

// Unstable psi_m / psi_h (zeta in [-PSI_ZMAX, 0], NaN excluded; the caller checks the range) from the piecewise
// polynomials PSI_COARE_T / PSI_PAULSON_T: ~25 instructions per function instead of the roots, logarithms, arctangents
// and powers of the formulas (two roots, three logs, three atans and two powr per COARE pair).  The row comes from the
// high word of |zeta| (its exponent and PSI_K mantissa bits, integer instructions only), u = |zeta| - c is exact (c, the
// row's centre, shares the binade of |zeta|), and row 0 (|zeta| < 2^PSI_E0, c = 0) has c_0 = 0: psi(-0) = 0.
struct PsiRow {
    int r;
    double u;
};
ABM_FN PsiRow psi_row(double z)
{
    constexpr int S = 20 - PSI_K;
    const int hx = hi_word(z) & 0x7fffffff;
    int d = hx - ((1023 + PSI_E0) << 20) + (1 << S);
    d = (d > 0) ? d : 0;
    const int r = d >> S;
    const int hc = (hx & -(1 << S)) | (1 << (S - 1));
    PsiRow a;
    a.r = r;
    a.u = -z - make_double(r ? hc : 0, 0);
    return a;
}
// F = 0: psi_m, 1: psi_h.  Estrin: depth 5 instead of 11 dependent FMAs
template <int F>
ABM_FN double psi_poly(const double *T, PsiRow a)
{
    constexpr int NP = (PSI_DEG + 1) / 2;
    double c[NP];
#pragma unroll
    for (int j = 0; j < NP; ++j) {
        const double2 p = ABM_PSI_T2(T, (F * NP + j) * PSI_ROWS + a.r);
        c[j] = fma(p.y, a.u, p.x);
    }
    double x = a.u * a.u;
#pragma unroll
    for (int n = NP; n > 1; n = (n + 1) / 2) {
#pragma unroll
        for (int j = 0; j < n / 2; ++j) c[j] = fma(c[2 * j + 1], x, c[2 * j]);
        if (n & 1) c[n / 2] = c[n - 1];
        x = x * x;
    }
    return c[0];
}
// the coefficients of one family (PSI_TABLES_COARE or PSI_TABLES_PAULSON)
template <int FAM>
ABM_FN const double *psi_coeffs()
{
    if constexpr (FAM == PSI_TABLES_COARE) return ABM_PSI_T(COARE);
    else return ABM_PSI_T(PAULSON);
}

// atan(t) for |t| <= tan(pi/8) (Estrin)
ABM_FN double atan_core(double t)
{
    const double z = t * t;
    const double z2 = z * z, z4 = z2 * z2;
    const double a0 = fma(ATAN_C[1], z, ATAN_C[0]), a1 = fma(ATAN_C[3], z, ATAN_C[2]), a2 = fma(ATAN_C[5], z, ATAN_C[4]);
    const double a3 = fma(ATAN_C[7], z, ATAN_C[6]), a4 = fma(ATAN_C[9], z, ATAN_C[8]);
    const double q = fma(fma(ATAN_C[10], z2, a4), z4 * z4, fma(fma(a3, z2, a2), z4, fma(a1, z2, a0)));
    return fma(t * z, q, t);
}
// atan: |x| <= tan(pi/8): poly; <= tan(3pi/8): pi/4 + atan((x-1)/(x+1)); else pi/2 - atan(1/x)
ABM_BIG double datan(double x)
{
    const double ax = fabs(x);
    double num = ax, den = 1.0, bhi = 0., blo = 0.;
    if (ax > MATH_K[K_TAN3PIO8]) {
        num = -1.0; den = ax; bhi = MATH_K[K_PIO2_HI]; blo = MATH_K[K_PIO2_LO];
    } else if (ax > MATH_K[K_TANPIO8]) {
        num = ax - 1.0; den = ax + 1.0; bhi = MATH_K[K_PIO4_HI]; blo = MATH_K[K_PIO4_LO];
    }
    const double a = atan_core(num * fast_rcp(den));
    return copysign(bhi + (a + blo), x);
}
// atan(x) for x >= 1 -- every atan of the stability functions: its argument is a root of (1 - g zeta) >= 1 or
// (1 + 2 phi) / sqrt(3) with phi >= 1.  With c = tan(3 pi/8), atan(x) = atan(c) + atan((x - c) / (1 + c x)) and the
// inner argument stays inside [-tan(pi/8), tan(pi/8)] for ALL x in [1, inf): the polynomial's range, one formula, no
// range selection (the three-way selection of datan cost 2 compares and ~10 predicated moves per call: 18 % of the
// register moves the COARE + skin kernel executed) and no sign handling.
ABM_BIG double datan_ge1(double x)
{
    const double c = MATH_K[K_TAN3PIO8];
    const double a = atan_core((x - c) * fast_rcp(fma(c, x, 1.0)));
    return MATH_K[K_ATANC_HI] + (a + MATH_K[K_ATANC_LO]);
}

// x**y, x >= 0
// (|y log x| <= 0.8 * 745 for the exponents of this path, all below 0.8 in magnitude: the bounded exp)
ABM_FN double dpowr(double x, double y) { return (x > 0.) ? dexp_b(y * dlog(x)) : 0.; }

}  // namespace abm
