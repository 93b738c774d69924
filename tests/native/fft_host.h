// The transform of the FFT calls (csrc/fft_pass.cuh: mdp_fft_transform) on the host, for the emulators of fftcorr.cu,
// msdfft.cu and isffft.cu: the same fused passes, in the same schedule, between two arrays.  TEST INFRASTRUCTURE ONLY.
#pragma once
#include "../../mdproptools_b200/csrc/fft_corr.h"

struct HostIn {
    const mdp_c64 *x;
    mdp_c64 operator()(long long i) const { return x[i]; }
};
struct HostOut {
    mdp_c64 *y;
    void operator()(long long i, const mdp_c64 &v) const { y[i] = v; }
};

// one transform of src in fused passes; returns the array that holds the result
inline mdp_c64 *fft_fused(mdp_c64 *src, mdp_c64 *dst, const mdp_c64 *W, int p, long long n)
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
