// Host build of the per-term body of the structure-factor kernel (mdproptools_b200/csrc/sk_phase.h): fixed-point fractional
// coordinates, the integer phase, the angle, and rho_c(k) summed in fp32 chunks of MDP_SK_CHUNK terms and fp64 beyond, as
// k_sk_rho sums them.  sin and cos are the host's (fp64 of the fp32 angle, rounded to fp32), so the device's __sincosf bound
// is the one part of the contract this build does not exercise.  TEST INFRASTRUCTURE ONLY.  Built with -ffp-contract=off.
#include <math.h>
#include <stdint.h>

#include "../../mdproptools_b200/csrc/sk_phase.h"

extern "C" {

int sk_consts(double *out)
{
    out[0] = MDP_SK_NLIM;
    out[1] = MDP_SK_EPS;
    out[2] = MDP_SK_MAX_CLASSES;
    out[3] = MDP_SK_CHUNK;
    return 0;
}

// s[n][3] fractional coordinates of positions r[n][3] in cell[6]
void sk_frac(const double *cell, const double *r, long long n, double *s)
{
    for (long long i = 0; i < n; ++i) mdp_sk_frac(cell, r[3 * i], r[3 * i + 1], r[3 * i + 2], s + 3 * i);
}

void sk_fix(const double *s, long long n, uint32_t *u)
{
    for (long long i = 0; i < n; ++i) u[i] = mdp_sk_fix(s[i]);
}

// p[k][j] for triplets miller[nk][3] and fixed-point atoms u[n][3]
void sk_phase(const int32_t *miller, long long nk, const uint32_t *u, long long n, uint32_t *p)
{
    for (long long k = 0; k < nk; ++k)
        for (long long j = 0; j < n; ++j)
            p[k * n + j] = mdp_sk_phase(miller[3 * k], miller[3 * k + 1], miller[3 * k + 2], u[3 * j], u[3 * j + 1], u[3 * j + 2]);
}

// terms[k][j] = (cos, sin) of the angle of p, negated (exp(2 pi i p / 2^32) = -exp(i angle))
void sk_terms(const uint32_t *p, long long m, float *cs)
{
    for (long long i = 0; i < m; ++i) {
        const float a = mdp_sk_angle(p[i]);
        cs[2 * i] = -(float)cos((double)a);
        cs[2 * i + 1] = -(float)sin((double)a);
    }
}

// rho[k] = sum_j exp(2 pi i n_k.s_j) for atoms given by fractional coordinates s[n][3], in the kernel's summation order
void sk_rho(const int32_t *miller, long long nk, const double *s, long long n, double *rho)
{
    for (long long k = 0; k < nk; ++k) {
        double sr = 0.0, si = 0.0;
        for (long long j0 = 0; j0 < n; j0 += MDP_SK_CHUNK) {
            float cr = 0.f, ci = 0.f;
            for (long long j = j0; j < n && j < j0 + MDP_SK_CHUNK; ++j) {
                const uint32_t p = mdp_sk_phase(miller[3 * k], miller[3 * k + 1], miller[3 * k + 2], mdp_sk_fix(s[3 * j]),
                                                mdp_sk_fix(s[3 * j + 1]), mdp_sk_fix(s[3 * j + 2]));
                const float a = mdp_sk_angle(p);
                cr += (float)cos((double)a);
                ci += (float)sin((double)a);
            }
            sr += (double)cr;
            si += (double)ci;
        }
        rho[2 * k] = 0.0 - sr;
        rho[2 * k + 1] = 0.0 - si;
    }
}

} // extern "C"
