// Host emulation of the FFT correlation of mdproptools_b200/csrc/fftcorr.cu: the same butterflies, cross spectrum and
// normalisation (csrc/fft_corr.h), stage after stage.  TEST INFRASTRUCTURE ONLY.  Built with -ffp-contract=off.
#include <stdint.h>
#include <vector>

#include "fft_host.h"

// the fused passes against p single radix-2 stages on the same data: number of values that differ in any bit
extern "C" long long fft_fused_vs_radix2(const double *re, const double *im, int p)
{
    const long long n = 1ll << p;
    std::vector<mdp_c64> W((size_t)n / 2), x((size_t)n), y((size_t)n), u((size_t)n), v((size_t)n);
    for (long long k = 0; k < n / 2; ++k) W[(size_t)k] = mdp_twiddle(k, n);
    for (long long i = 0; i < n; ++i) {
        x[(size_t)i].re = u[(size_t)i].re = re[i];
        x[(size_t)i].im = u[(size_t)i].im = im[i];
    }
    mdp_c64 *src = x.data(), *dst = y.data();
    for (int t = 0; t < p; ++t) {
        for (long long i = 0; i < n / 2; ++i) mdp_fft_butterfly(src, dst, W.data(), i, t, n);
        mdp_c64 *tmp = src; src = dst; dst = tmp;
    }
    const mdp_c64 *f = fft_fused(u.data(), v.data(), W.data(), p, n);
    long long bad = 0;
    for (long long i = 0; i < n; ++i) {
        union { double d; uint64_t b; } a0{src[i].re}, a1{f[i].re}, b0{src[i].im}, b1{f[i].im};
        bad += (a0.b != a1.b) + (b0.b != b1.b);
    }
    return bad;
}

extern "C" int emulate_fft_xcorr(const double *a, const double *b, long long T, long long nlags, double *out)
{
    const int p = mdp_fft_log2_size(T, nlags);
    const long long n = 1ll << p;
    std::vector<mdp_c64> W((size_t)n / 2), x((size_t)n), y((size_t)n);
    for (long long k = 0; k < n / 2; ++k) W[(size_t)k] = mdp_twiddle(k, n);
    for (long long i = 0; i < n; ++i) {
        x[(size_t)i].re = i < T ? a[i] : 0.0;
        x[(size_t)i].im = i < T ? b[i] : 0.0;
    }
    mdp_c64 *src = fft_fused(x.data(), y.data(), W.data(), p, n);
    mdp_c64 *dst = src == x.data() ? y.data() : x.data();
    for (long long k = 0; k < n; ++k) dst[k] = mdp_cross_spectrum_conj(src, k, n);
    src = fft_fused(dst, src, W.data(), p, n);
    // src = FFT(conj(P)) = N * conj(corr); corr is real
    for (long long tau = 0; tau < nlags; ++tau) out[tau] = mdp_fft_unbiased(src[tau].re, n, T, tau);
    return p;
}
