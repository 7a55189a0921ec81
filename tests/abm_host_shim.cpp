// Host build of the kernels' own math (aerobulk_b200/csrc/ab_math.cuh) for tests/test_math_accuracy.py.
#define ABM_HOST_TEST 1
#include "../aerobulk_b200/csrc/ab_math.cuh"
extern "C" {
void abm_eval(int fn, const double *x, const double *y, double *out, long n)
{
    for (long i = 0; i < n; ++i) {
        switch (fn) {
        case 0: out[i] = abm::dexp(x[i]); break;
        case 1: out[i] = abm::dexp10(x[i]); break;
        case 2: out[i] = abm::dlog(x[i]); break;
        case 3: out[i] = abm::dlog10(x[i]); break;
        case 4: out[i] = abm::datan(x[i]); break;
        case 5: out[i] = abm::dpowr(x[i], y[i]); break;
        case 6: out[i] = abm::fast_rcp(x[i]); break;
        case 10: out[i] = abm::fast_rsqrt(x[i]); break;
        case 11: out[i] = abm::fast_rcbrt(x[i]); break;
        case 12: out[i] = abm::fast_r4rt(x[i]); break;
        case 13: out[i] = abm::pow075(x[i]); break;
        case 14: out[i] = abm::fast_cbrt(x[i]); break;
        case 15: out[i] = abm::fast_sqrt(x[i]); break;
        case 16: out[i] = abm::datan_ge1(x[i]); break;
        case 17: out[i] = abm::fast_sqrt_pos(x[i]); break;
        case 18: out[i] = abm::pow075_pos(x[i]); break;
        }
    }
}
}
