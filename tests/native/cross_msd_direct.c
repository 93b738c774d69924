/*
 * Direct long-double definition of the all-origins cross MSD of channel groups that mdp_cross_msd_fft computes
 * (csrc/msdfft.cu).  An extension with no reference implementation: this direct sum is its definition.  TEST
 * INFRASTRUCTURE ONLY (tests/einstein_oracle.py builds and loads it).
 *
 * out[g][tau] = sum_{c in group g} (1/(T-tau)) sum_{t < T-tau} (a_c(t+tau) - a_c(t)) * (b_c(t+tau) - b_c(t)),  tau < nlags.
 * a, b are [nchan][T] (b == NULL: b = a); group_off [ngroups+1]; every product and sum in long double.
 */
#include <stdint.h>

void orc_cross_msd_direct(const double *a, const double *b, int64_t T, const int64_t *group_off, int64_t ngroups,
                          int64_t nlags, double *out)
{
    if (!b) b = a;
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t tau = 0; tau < nlags; ++tau)
        for (int64_t g = 0; g < ngroups; ++g) {
            long double s = 0.0L;
            for (int64_t c = group_off[g]; c < group_off[g + 1]; ++c) {
                const double *x = a + c * T, *y = b + c * T;
                long double sc = 0.0L;
                for (int64_t t = 0; t + tau < T; ++t)
                    sc += ((long double)x[t + tau] - (long double)x[t]) * ((long double)y[t + tau] - (long double)y[t]);
                s += sc / (long double)(T - tau);
            }
            out[g * nlags + tau] = (double)s;
        }
}
