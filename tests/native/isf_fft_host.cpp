// Host emulation of the binned FFT correlation of mdproptools_b200/csrc/isffft.cu: the same butterflies, symmetrised pair
// spectrum, per-(pair, bin) accumulation in k order, within-bin pairing of groups in the inverse transforms, fold and
// epilogue (csrc/isf_fft.h, csrc/fft_corr.h).  TEST INFRASTRUCTURE ONLY.  Built with -ffp-contract=off.
#include <stdint.h>
#include <vector>

#include "../../mdproptools_b200/csrc/isf_fft.h"
#include "fft_host.h"

// rho = (re, im) [nchan][nk][T]; pairs [npairs][2]; bin_off [nbins+1]; out [npairs][nbins][nlags].  Returns log2 N.
extern "C" int emulate_isf_fft(const double *rho, int nchan, long long nk, long long T, const int *pairs, int npairs,
                               const long long *bin_off, int nbins, long long nlags, double *out)
{
    const int p = mdp_fft_log2_size(T, nlags);
    const long long n = 1ll << p, H = n / 2 + 1;
    std::vector<mdp_c64> W((size_t)n / 2), x((size_t)n), y((size_t)n);
    for (long long k = 0; k < n / 2; ++k) W[(size_t)k] = mdp_twiddle(k, n);
    std::vector<double> acc((size_t)npairs * nbins * H, 0.0);
    std::vector<mdp_c64> Z((size_t)nchan * n);
    for (int b = 0; b < nbins; ++b)
        for (long long k = bin_off[b]; k < bin_off[b + 1]; ++k) {
            for (int c = 0; c < nchan; ++c) {
                for (long long i = 0; i < n; ++i) {
                    x[(size_t)i].re = i < T ? rho[2 * ((c * nk + k) * T + i)] : 0.0;
                    x[(size_t)i].im = i < T ? rho[2 * ((c * nk + k) * T + i) + 1] : 0.0;
                }
                const mdp_c64 *r = fft_fused(x.data(), y.data(), W.data(), p, n);
                for (long long i = 0; i < n; ++i) Z[(size_t)(c * n + i)] = r[i];
            }
            for (int q = 0; q < npairs; ++q) {
                double *a = &acc[(size_t)((b * (long long)npairs + q) * H)];
                for (long long w = 0; w < H; ++w) a[w] += mdp_isf_spectrum(&Z[(size_t)(pairs[2 * q] * n)], &Z[(size_t)(pairs[2 * q + 1] * n)], w, n);
            }
        }
    for (int b = 0; b < nbins; ++b)
        for (long long j = 0; j < mdp_fft_transforms_per_bin(npairs); ++j) {
            const mdp_fft_group_pair gp = mdp_fft_pair_groups(j, npairs);
            const long long q = gp.first, g = b * (long long)npairs + q;
            for (long long w = 0; w < n; ++w) {
                const long long ww = mdp_fft_fold(w, n);
                x[(size_t)w].re = acc[(size_t)(g * H + ww)];
                x[(size_t)w].im = gp.partner ? acc[(size_t)((g + 1) * H + ww)] : 0.0;
            }
            const mdp_c64 *r = fft_fused(x.data(), y.data(), W.data(), p, n);
            for (long long tau = 0; tau < nlags; ++tau) {
                out[(q * nbins + b) * nlags + tau] = mdp_fft_unbiased(r[tau].re, n, T, tau);
                if (gp.partner) out[((q + 1) * nbins + b) * nlags + tau] = mdp_fft_unbiased(r[tau].im, n, T, tau);
            }
        }
    return p;
}
