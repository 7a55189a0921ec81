// Host build of abm::esat_table (aerobulk_b200/csrc/ab_math.cuh) for tests/test_esat_table.py.
#define ABM_HOST_TEST 1
#include "../aerobulk_b200/csrc/ab_math.cuh"
extern "C" {
void esat_table_eval(const double *T, double *out, long n)
{
    for (long i = 0; i < n; ++i) out[i] = abm::esat_table(T[i]);
}
}
