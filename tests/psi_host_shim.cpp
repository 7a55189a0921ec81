// Host build of abm::psi_row / abm::psi_poly (aerobulk_b200/csrc/ab_math.cuh) for tests/test_psi_tables.py.
#define ABM_HOST_TEST 1
#include "../aerobulk_b200/csrc/ab_math.cuh"
extern "C" {
// fam: 0 COARE, 1 Paulson; which: 0 psi_m, 1 psi_h
void psi_table_eval(int fam, int which, const double *z, double *out, long n)
{
    const double *T = fam ? abm::psi_coeffs<abm::PSI_TABLES_PAULSON>() : abm::psi_coeffs<abm::PSI_TABLES_COARE>();
    for (long i = 0; i < n; ++i) {
        const abm::PsiRow a = abm::psi_row(z[i]);
        out[i] = which ? abm::psi_poly<1>(T, a) : abm::psi_poly<0>(T, a);
    }
}
}
