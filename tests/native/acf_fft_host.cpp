// Host emulation of the grouped FFT autocorrelation of mdproptools_b200/csrc/msdfft.cu (mdp_group_acf_fft): the same
// self-case unit pairing (two channels of a group per transform, an odd last one with zero), butterflies, group spectrum
// accumulation, two-groups-per-inverse transform and epilogue (csrc/msd_fft.h, csrc/fft_corr.h), with no centring.
// TEST INFRASTRUCTURE ONLY.  Built with -ffp-contract=off.
#include <stdint.h>
#include <vector>

#include "../../mdproptools_b200/csrc/msd_fft.h"
#include "fft_host.h"

// Returns log2 N.
extern "C" int emulate_group_acf(const double *a, long long T, const long long *group_off, int ngroups, long long nlags, double *out)
{
    const int p = mdp_fft_log2_size(T, nlags);
    const long long n = 1ll << p, H = n / 2 + 1;
    std::vector<mdp_c64> W((size_t)n / 2), x((size_t)n), y((size_t)n);
    for (long long k = 0; k < n / 2; ++k) W[(size_t)k] = mdp_twiddle(k, n);
    std::vector<double> acc((size_t)(ngroups * H), 0.0);
    for (int g = 0; g < ngroups; ++g) {
        for (long long c = group_off[g]; c < group_off[g + 1]; c += 2) {
            const long long c1 = c + 1 < group_off[g + 1] ? c + 1 : -1;
            for (long long i = 0; i < n; ++i) {
                x[(size_t)i].re = i < T ? a[c * T + i] : 0.0;
                x[(size_t)i].im = i < T && c1 >= 0 ? a[c1 * T + i] : 0.0;
            }
            const mdp_c64 *Z = fft_fused(x.data(), y.data(), W.data(), p, n);
            for (long long k = 0; k < H; ++k) acc[(size_t)(g * H + k)] += mdp_msd_spectrum_self(Z, k, n);
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
            out[g * nlags + tau] = group_off[g + 1] == group_off[g] ? 0.0 : mdp_acf_epilogue(r[tau].re, n, T, tau);
            if (gp.partner)
                out[(g + 1) * nlags + tau] = group_off[g + 2] == group_off[g + 1] ? 0.0 : mdp_acf_epilogue(r[tau].im, n, T, tau);
        }
    }
    return p;
}
