// Host emulation of the FFT all-origins MSD of mdproptools_b200/csrc/msdfft.cu: the same mean centring, unit pairing,
// butterflies, spectrum combination (self and cross), group accumulation, two-groups-per-inverse transform and
// prefix/suffix epilogue (csrc/msd_fft.h, csrc/fft_corr.h).  TEST INFRASTRUCTURE ONLY.  Built with -ffp-contract=off.
#include <stdint.h>
#include <vector>

#include "../../mdproptools_b200/csrc/msd_fft.h"
#include "fft_host.h"

namespace {

double mean(const double *x, long long T)
{
    double lanes[MDP_MSD_MEAN_LANES];
    for (int l = 0; l < MDP_MSD_MEAN_LANES; ++l) lanes[l] = mdp_msd_lane_sum(x, T, l);
    return mdp_msd_mean_tree(lanes, T);
}

} // namespace

// b == NULL: self case.  centre == 0 skips the mean subtraction (to show what it is for).  Returns log2 N.
extern "C" int emulate_cross_msd(const double *a, const double *b, long long T, const long long *group_off, int ngroups,
                                 long long nlags, int centre, double *out)
{
    const int self = b == nullptr;
    if (self) b = a;
    const int p = mdp_fft_log2_size(T, nlags);
    const long long n = 1ll << p, H = n / 2 + 1;
    const long long nchan = group_off[ngroups];
    std::vector<mdp_c64> W((size_t)n / 2), x((size_t)n), y((size_t)n);
    for (long long k = 0; k < n / 2; ++k) W[(size_t)k] = mdp_twiddle(k, n);
    std::vector<double> ma((size_t)nchan), mb((size_t)nchan);
    for (long long c = 0; c < nchan; ++c) {
        ma[(size_t)c] = centre ? mean(a + c * T, T) : 0.0;
        mb[(size_t)c] = self ? ma[(size_t)c] : centre ? mean(b + c * T, T) : 0.0;
    }
    std::vector<double> acc((size_t)(ngroups * H), 0.0), pre((size_t)(ngroups * (T + 1))), suf((size_t)(ngroups * (T + 1)));
    for (int g = 0; g < ngroups; ++g) {
        std::vector<double> pg((size_t)T, 0.0);
        for (long long c = group_off[g]; c < group_off[g + 1]; ++c)
            for (long long t = 0; t < T; ++t) pg[(size_t)t] += (a[c * T + t] - ma[(size_t)c]) * (b[c * T + t] - mb[(size_t)c]);
        double *P = &pre[(size_t)(g * (T + 1))], *S = &suf[(size_t)(g * (T + 1))];
        P[0] = 0.0;
        for (long long t = 0; t < T; ++t) P[t + 1] = P[t] + pg[(size_t)t];
        S[T] = 0.0;
        for (long long t = T - 1; t >= 0; --t) S[t] = S[t + 1] + pg[(size_t)t];
        for (long long c = group_off[g]; c < group_off[g + 1]; c += self ? 2 : 1) {
            const long long c1 = self ? (c + 1 < group_off[g + 1] ? c + 1 : -1) : c;
            for (long long i = 0; i < n; ++i) {
                x[(size_t)i].re = i < T ? a[c * T + i] - ma[(size_t)c] : 0.0;
                x[(size_t)i].im = i < T && c1 >= 0 ? b[c1 * T + i] - mb[(size_t)c1] : 0.0;
            }
            const mdp_c64 *Z = fft_fused(x.data(), y.data(), W.data(), p, n);
            for (long long k = 0; k < H; ++k)
                acc[(size_t)(g * H + k)] += self ? mdp_msd_spectrum_self(Z, k, n) : mdp_msd_spectrum_cross(Z, k, n);
        }
    }
    for (long long j = 0; j < mdp_fft_transforms_per_bin(ngroups); ++j) {
        const mdp_fft_group_pair gp = mdp_fft_pair_groups(j, ngroups);
        const long long g = gp.first;
        for (long long k = 0; k < n; ++k) {
            const long long kk = mdp_fft_fold(k, n);
            x[(size_t)k].re = acc[(size_t)(g * H + kk)];
            x[(size_t)k].im = gp.partner ? acc[(size_t)((g + 1) * H + kk)] : 0.0;
        }
        const mdp_c64 *r = fft_fused(x.data(), y.data(), W.data(), p, n);
        for (long long tau = 0; tau < nlags; ++tau) {
            out[g * nlags + tau] = group_off[g + 1] == group_off[g] ? 0.0
                : mdp_msd_epilogue(&suf[(size_t)(g * (T + 1))], &pre[(size_t)(g * (T + 1))], T, tau, r[tau].re / (double)n);
            if (gp.partner)
                out[(g + 1) * nlags + tau] = group_off[g + 2] == group_off[g + 1] ? 0.0
                    : mdp_msd_epilogue(&suf[(size_t)((g + 1) * (T + 1))], &pre[(size_t)((g + 1) * (T + 1))], T, tau,
                                       r[tau].im / (double)n);
        }
    }
    return p;
}
