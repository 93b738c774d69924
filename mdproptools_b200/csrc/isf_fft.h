// isf_fft.h -- binned, symmetrised time correlation of complex series through the Stockham FFT of fft_corr.h: the coherent
// intermediate scattering function (host/device shared bodies of the kernels in isffft.cu; exercised on the host by
// tests/native/isf_fft_host.cpp).
//
// For channels a, b of complex series z_c(k, t) (t < T; rho_c(k, t) of mdp_sk_rho) and a bin's k-vectors:
//     out[p][bin][tau] = sum_{k in bin} C_ab(k, tau),
//     C_ab(k, tau) = 1/(T-tau) sum_{t < T-tau} 1/2 Re( z_a(k,t+tau) z_b(k,t)* + z_b(k,t+tau) z_a(k,t)* ),   tau < nlags.
// Zero-padded to N = 2^p >= T + nlags (mdp_fft_log2_size), with Z_c = FFT(z_c) and S = Z_a conj(Z_b),
//     sum_t z_a(t+tau) z_b(t)* = IFFT(S)[tau],   sum_t z_b(t+tau) z_a(t)* = IFFT(conj S)[tau],
// so the bracket is IFFT(2 Re S)[tau], and its real part is the transform of the even part of Re S:
//     G(w) = 1/2 (Re S(w) + Re S(-w))      (self pair a = b: 1/2 (|Z_a(w)|^2 + |Z_a(-w)|^2)).
// G is real and even and linear in the k-vector, so it is summed over the bin's k-vectors (in k order) in the frequency
// domain and one inverse transform serves a (pair, bin) group; two groups of the same bin share one complex transform
// (mdp_fft_pair_groups, mdp_fft_fold).  rho is not centred: its time mean is physical (Bragg peaks).
//
// G is computed as 1/2 ((a.re b.re + a.im b.im) + (a'.re b'.re + a'.im b'.im)): products commute, so the pairs (a, b) and
// (b, a) give the same bits.
//
// Accuracy: agreement with the long-double direct sum (tests/isf_oracle.py) to 1e-10 of max_tau |out[p][bin]| for
// T <= 10^5 -- the contract of the FFT correlation (fft_corr.h, msd_fft.h).
#pragma once
#include "fft_corr.h"

// G at frequency k of the pair whose spectra are Za, Zb (Za == Zb for a self pair)
MDP_HD double mdp_isf_spectrum(const mdp_c64 *Za, const mdp_c64 *Zb, long long k, long long n)
{
    const long long kc = (n - k) & (n - 1);                // -k mod N
    const mdp_c64 a = Za[k], b = Zb[k], ac = Za[kc], bc = Zb[kc];
    return 0.5 * ((a.re * b.re + a.im * b.im) + (ac.re * bc.re + ac.im * bc.im));
}

// the earlier names of the shared helpers for the ISF's bins and epilogue, kept for host code written against them
MDP_HD long long mdp_isf_transforms_per_bin(long long npairs)
{
    return mdp_fft_transforms_per_bin(npairs);
}

MDP_HD double mdp_isf_epilogue(double x, long long n, long long T, long long tau)
{
    return mdp_fft_unbiased(x, n, T, tau);
}
