// fft_corr.h -- unbiased time correlation through a Stockham FFT in fp64: radix-2 butterflies, three stages per pass
// (host/device shared bodies of fft_pass.cuh and fftcorr.cu, also used by msd_fft.h and isf_fft.h; exercised on the host
// by tests/native/fft_corr_host.cpp).
//
// out[tau] = (sum_{t < T - tau} a[t + tau] * b[t]) / (T - tau)       (conductivity.py:97-114, viscosity.py:86-120)
//
// The reference evaluates this with a zero-padded FFT (numpy); the direct kernel k_xcorr costs T^2/2 FMAs per channel,
// which is fine at 10^5 steps (13 ms for 30 channels) and hopeless at the 10^6..10^7 thermo steps a viscosity run
// produces.  Here: z = a + i*b zero-padded to N = 2^p >= T + nlags, ONE forward FFT gives both spectra
// (A[k] = (Z[k] + conj(Z[N-k]))/2, B[k] = (Z[k] - conj(Z[N-k]))/(2i)), P = A * conj(B), and one more forward FFT of
// conj(P) gives N * conj(corr).  Stockham autosort: every stage reads one array and writes the other, no bit reversal, all
// N/2 butterflies of a stage independent (one thread each).  Twiddles come from a table W[k] = exp(-2 pi i k / N),
// k < N/2, computed once per call with sincospi (full fp64 accuracy: the result agrees with the direct sum to ~1e-15 of
// max|corr| times log2 N).
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define MDP_HD __host__ __device__ __forceinline__
#else
#ifndef MDP_HD
#define MDP_HD inline
#endif
#endif

struct alignas(16) mdp_c64 {
    double re, im;
};

MDP_HD mdp_c64 mdp_twiddle(long long k, long long n)   // exp(-2 pi i k / n)
{
    mdp_c64 w;
    const double x = 2.0 * (double)k / (double)n;
#if defined(__CUDA_ARCH__)
    double s, c;
    sincospi(x, &s, &c);
    w.re = c;
    w.im = -s;
#else
    w.re = cos(M_PI * x);
    w.im = -sin(M_PI * x);
#endif
    return w;
}

// butterfly i (0 <= i < n/2) of stage t (0 <= t < log2 n): x -> y
MDP_HD void mdp_fft_butterfly(const mdp_c64 *x, mdp_c64 *y, const mdp_c64 *W, long long i, int t, long long n)
{
    const long long m = 1ll << t, l = n >> (t + 1);
    const long long k = i & (m - 1), j = i >> t;
    const mdp_c64 c0 = x[k + j * m], c1 = x[k + j * m + l * m];
    const mdp_c64 w = W[j << t];                       // exp(-2 pi i j / (2 l)) = W_n[j * m]
    mdp_c64 s, d, r;
    s.re = c0.re + c1.re;
    s.im = c0.im + c1.im;
    d.re = c0.re - c1.re;
    d.im = c0.im - c1.im;
    r.re = d.re * w.re - d.im * w.im;
    r.im = d.re * w.im + d.im * w.re;
    y[k + 2 * j * m] = s;
    y[k + 2 * j * m + m] = r;
}

// 2^R butterflies of R consecutive stages t .. t+R-1 in registers: one pass over the data instead of R.  Thread i
// (0 <= i < n >> R) owns the points i + q * (n >> R); after every stage the two results of a butterfly stay in the
// registers of its two inputs, and the positions they WOULD have in the Stockham array are carried along (pos[]), so the
// arithmetic is, operation for operation, that of R calls of mdp_fft_butterfly -- bit-identical results (checked on the
// host by tests/native/fft_corr_host.cpp).  in(pos) reads a point, out(pos, v) writes one: the first pass of a transform
// can read the real series directly and the last one can write the normalised correlation (fft_pass.cuh).
// Requires t + R <= log2 n.
template <int R, class In, class Out>
MDP_HD void mdp_fft_radix_pass(const In in, const Out out, const mdp_c64 *W, long long i, int t, long long n)
{
    constexpr int Q = 1 << R;
    mdp_c64 v[Q];
    long long pos[Q];
    const long long step = n >> R;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int q = 0; q < Q; ++q) {
        pos[q] = i + q * step;
        v[q] = in(pos[q]);
    }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int s = 0; s < R; ++s) {
        const int ts = t + s, h = Q >> (s + 1);
        const long long ms = 1ll << ts;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int a = 0; a < Q; ++a) {
            if (a & h) continue;
            const int b = a + h;                           // pos[b] == pos[a] + n/2: the butterfly of index pos[a]
            const long long k = pos[a] & (ms - 1), j = pos[a] >> ts;
            const mdp_c64 w = W[j << ts];
            const mdp_c64 c0 = v[a], c1 = v[b];
            mdp_c64 sum, d, r;
            sum.re = c0.re + c1.re;
            sum.im = c0.im + c1.im;
            d.re = c0.re - c1.re;
            d.im = c0.im - c1.im;
            r.re = d.re * w.re - d.im * w.im;
            r.im = d.re * w.im + d.im * w.re;
            v[a] = sum;
            v[b] = r;
            pos[a] = k + 2 * j * ms;
            pos[b] = pos[a] + ms;
        }
    }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int q = 0; q < Q; ++q) out(pos[q], v[q]);
}

MDP_HD int mdp_fft_pass_radix(int t, int p)               // stages fused by the pass that starts at stage t: 3, then what is left
{
    return p - t >= 3 ? 3 : p - t;
}

// element k (0 <= k < n) of conj(P), P = A * conj(B), from the spectrum Z of z = a + i*b
MDP_HD mdp_c64 mdp_cross_spectrum_conj(const mdp_c64 *Z, long long k, long long n)
{
    const mdp_c64 z = Z[k], zc = Z[(n - k) & (n - 1)];      // Z[N - k] with Z[N] = Z[0]
    // A = (z + conj(zc)) / 2, B = (z - conj(zc)) / (2i) = (-i/2) (z - conj(zc))
    const double ar = 0.5 * (z.re + zc.re), ai = 0.5 * (z.im - zc.im);
    const double dr = z.re - zc.re, di = z.im + zc.im;      // z - conj(zc)
    const double br = 0.5 * di, bi = -0.5 * dr;
    mdp_c64 p;                                              // conj(A * conj(B)) = conj(A) * B
    p.re = ar * br + ai * bi;
    p.im = ar * bi - ai * br;
    return p;
}

MDP_HD int mdp_fft_log2_size(long long T, long long nlags)   // smallest p with 2^p >= T + nlags (no circular wrap below nlags)
{
    int p = 1;
    while ((1ll << p) < T + nlags) ++p;
    return p;
}

// lag tau of the unbiased correlation from element tau of a transform of N points (x = its real or imaginary part)
MDP_HD double mdp_fft_unbiased(double x, long long n, long long T, long long tau)
{
    return x / (double)n / (double)(T - tau);
}

// element k (0 <= k < n) of a real even spectrum held as its half acc[0 .. n/2]
MDP_HD long long mdp_fft_fold(long long k, long long n)
{
    return k <= n / 2 ? k : n - k;
}

// the earlier name of mdp_fft_fold (msd_fft.h and isf_fft.h both offered it), kept for host code written against it
MDP_HD long long mdp_msd_fold(long long k, long long n)
{
    return mdp_fft_fold(k, n);
}

// A real even spectrum transforms to a real series, so one complex inverse transform serves two groups of spectra.
// Groups come in bins of per_bin (the MSD's groups are one bin, an ISF bin holds one group per pair), and groups of
// different bins never share a transform, so a bin's bits depend on its own groups only.  A bin takes
// mdp_fft_transforms_per_bin(per_bin) transforms; its transform j carries group `first` of the bin in its real part and,
// when `partner`, group first + 1 in its imaginary part (an odd last group is paired with zero).
MDP_HD long long mdp_fft_transforms_per_bin(long long per_bin)
{
    return (per_bin + 1) / 2;
}

struct mdp_fft_group_pair {
    long long first;
    bool partner;
};

MDP_HD mdp_fft_group_pair mdp_fft_pair_groups(long long j, long long per_bin)
{
    mdp_fft_group_pair r;
    r.first = 2 * j;
    r.partner = r.first + 1 < per_bin;
    return r;
}
