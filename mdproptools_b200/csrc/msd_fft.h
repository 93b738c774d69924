// msd_fft.h -- mean-square displacement over all time origins through the Stockham FFT of fft_corr.h (host/device shared
// bodies of the kernels in msdfft.cu; exercised on the host by tests/native/msd_fft_host.cpp and acf_fft_host.cpp).
//
// out[g][tau] = sum_{c in group g} (1/(T-tau)) sum_{t < T-tau} (a_c(t+tau) - a_c(t)) * (b_c(t+tau) - b_c(t)),  tau < nlags
//
// Expanding the product with p(t) = a(t) b(t), the lag-tau sum is
//     sum_{t >= tau} p(t) + sum_{t < T-tau} p(t) - [xc_ab(tau) + xc_ba(tau)],      xc_ab(tau) = sum_t a(t+tau) b(t).
// Zero-padded to N = 2^p >= T + nlags (mdp_fft_log2_size), the bracket is IFFT(2 Re(A conj B))[tau] (self case b = a:
// IFFT(2 |A|^2)[tau]).  That spectrum is real and even, and it is linear in the channel, so it is summed per group in the
// frequency domain and only one inverse transform runs per group; two groups share one complex transform (the forward FFT
// of R_g + i R_{g+1} is N (r_g + i r_{g+1}) for real even R).  Every channel's mean is subtracted first: the result does
// not change, and the cancellation between the p sums and the bracket shrinks from the squared offset of unwrapped
// coordinates to the squared fluctuation.
//
// Accuracy: agreement with the direct long-double sum (tests/native/cross_msd_direct.c) to 1e-10 of
// max_tau |out[g]| for T <= 10^5 -- the contract of the FFT correlation.  The error is absolute: the p sums and the
// bracket are of the size of T times the series' variance and cancel at small lags, so lags where out is small relative
// to its maximum (the first few lags of a long diffusive series) carry that absolute error and nothing tighter.
#pragma once
#include "fft_corr.h"

// self case: one transform Z of a_c + i a_{c'} carries two channels of the group; their summed spectrum
// 2 (|A|^2 + |B|^2) = |Z[k]|^2 + |Z[N-k]|^2
MDP_HD double mdp_msd_spectrum_self(const mdp_c64 *Z, long long k, long long n)
{
    const mdp_c64 z = Z[k], zc = Z[(n - k) & (n - 1)];
    return (z.re * z.re + z.im * z.im) + (zc.re * zc.re + zc.im * zc.im);
}

// cross case: Z = FFT(a + i b); 2 Re(A conj B) (the real part of mdp_cross_spectrum_conj, doubled)
MDP_HD double mdp_msd_spectrum_cross(const mdp_c64 *Z, long long k, long long n)
{
    return 2.0 * mdp_cross_spectrum_conj(Z, k, n).re;
}

// out[tau] from the group's suffix sum suf[tau] = sum_{t >= tau} p(t), prefix sum pre[T - tau] = sum_{t < T-tau} p(t) and
// the bracket xc = xc_ab(tau) + xc_ba(tau) (the inverse transform divided by N)
MDP_HD double mdp_msd_epilogue(const double *suf, const double *pre, long long T, long long tau, double xc)
{
    return ((suf[tau] + pre[T - tau]) - xc) / (double)(T - tau);
}

// Grouped autocorrelation (mdp_group_acf_fft, the self case without centring; emulated by tests/native/acf_fft_host.cpp):
//   out[g][tau] = sum_{c in group g} (1/(T-tau)) sum_{t < T-tau} a_c(t+tau) * a_c(t)
// The group's summed self spectrum is 2 sum_c |A_c|^2 (mdp_msd_spectrum_self), whose inverse transform is N times twice
// the lag-tau sum: out = 0.5 * x / N / (T - tau) of element tau (x = its real or imaginary part).  The series are not
// centred: a mean (a velocity drift) is part of this result.  Same contract as the MSD: 1e-10 of max_tau |out[g]|, which
// is out[g][0], for T <= 10^5.
MDP_HD double mdp_acf_epilogue(double x, long long n, long long T, long long tau)
{
    return 0.5 * x / (double)n / (double)(T - tau);
}

// the mean of a channel in a fixed order: lane l of MDP_MSD_MEAN_LANES sums t = l, l + lanes, ... (mdp_msd_lane_sum),
// then the lanes are added pairwise, halving (mdp_msd_mean_tree on the host, the same loop in shared memory on the device)
#define MDP_MSD_MEAN_LANES 256

MDP_HD double mdp_msd_lane_sum(const double *x, long long T, int lane)
{
    double s = 0.0;
    for (long long t = lane; t < T; t += MDP_MSD_MEAN_LANES) s += x[t];
    return s;
}

#if !defined(__CUDA_ARCH__)
inline double mdp_msd_mean_tree(double *lanes, long long T)
{
    for (int h = MDP_MSD_MEAN_LANES / 2; h > 0; h >>= 1)
        for (int l = 0; l < h; ++l) lanes[l] += lanes[l + h];
    return lanes[0] / (double)T;
}
#endif
