// Host emulation of the FFT all-origins MSD of mdproptools_b200/csrc/msdfft.cu: the same mean centring, unit pairing,
// butterflies, spectrum combination (self and cross), group accumulation, two-groups-per-inverse transform and
// prefix/suffix epilogue (csrc/msd_fft.h, csrc/fft_corr.h).  TEST INFRASTRUCTURE ONLY.  Built with -ffp-contract=off.
#include <stdint.h>
#include <vector>

#include "../../mdproptools_b200/csrc/msd_fft.h"

namespace {

struct HostIn {
    const mdp_c64 *x;
    mdp_c64 operator()(long long i) const { return x[i]; }
};
struct HostOut {
    mdp_c64 *y;
    void operator()(long long i, const mdp_c64 &v) const { y[i] = v; }
};

mdp_c64 *fft_fused(mdp_c64 *src, mdp_c64 *dst, const mdp_c64 *W, int p, long long n)
{
    for (int t = 0; t < p;) {
        const int R = mdp_fft_pass_radix(t, p);
        for (long long i = 0; i < (n >> R); ++i) {
            if (R == 3) mdp_fft_radix_pass<3>(HostIn{src}, HostOut{dst}, W, i, t, n);
            else if (R == 2) mdp_fft_radix_pass<2>(HostIn{src}, HostOut{dst}, W, i, t, n);
            else mdp_fft_radix_pass<1>(HostIn{src}, HostOut{dst}, W, i, t, n);
        }
        mdp_c64 *tmp = src; src = dst; dst = tmp;
        t += R;
    }
    return src;
}

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
    for (int g = 0; g < ngroups; g += 2) {
        for (long long k = 0; k < n; ++k) {
            const long long kk = mdp_msd_fold(k, n);
            x[(size_t)k].re = acc[(size_t)(g * H + kk)];
            x[(size_t)k].im = g + 1 < ngroups ? acc[(size_t)((g + 1) * H + kk)] : 0.0;
        }
        const mdp_c64 *r = fft_fused(x.data(), y.data(), W.data(), p, n);
        for (long long tau = 0; tau < nlags; ++tau) {
            out[g * nlags + tau] = group_off[g + 1] == group_off[g] ? 0.0
                : mdp_msd_epilogue(&suf[(size_t)(g * (T + 1))], &pre[(size_t)(g * (T + 1))], T, tau, r[tau].re / (double)n);
            if (g + 1 < ngroups)
                out[(g + 1) * nlags + tau] = group_off[g + 2] == group_off[g + 1] ? 0.0
                    : mdp_msd_epilogue(&suf[(size_t)((g + 1) * (T + 1))], &pre[(size_t)((g + 1) * (T + 1))], T, tau,
                                       r[tau].im / (double)n);
        }
    }
    return p;
}
