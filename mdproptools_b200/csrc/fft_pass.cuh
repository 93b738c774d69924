// fft_pass.cuh -- how a batch of fp64 Stockham transforms runs on the device, shared by the FFT correlation (fftcorr.cu),
// the FFT MSD (msdfft.cu) and the ISF correlation (isffft.cu): the twiddle table, the pass kernel k_fft_pass, the host
// driver mdp_fft_transform with the pass schedule, and the load of the inverse transforms' input from half spectra.
//
// A pass is one launch over all units of the batch (grid (ceil((n >> R) / MDP_FFT_THREADS), units)) that covers R
// butterfly stages in registers (fft_corr.h: mdp_fft_radix_pass).  Unit u of a pass reads its points through
// in(u, i, n) and writes them through out(u, i, n, v).  The passes between the first and the last of a transform use
// FftArrayIn / FftArrayOut on the two work arrays; a call supplies its own functors for the first pass (reading its
// series in place of an array) or the last one (writing its result), so there is no copy in or out.  Each call names
// its functors, so a pass kernel in a trace says which call it belongs to.
//
// Everything here is static: every .cu file that includes it owns its own kernels.
#pragma once
#include <algorithm>
#include <type_traits>
#include <utility>

#include "common.cuh"
#include "fft_corr.h"

constexpr int MDP_FFT_THREADS = 256;

struct FftArrayIn {
    const mdp_c64 *x;
    __device__ __forceinline__ mdp_c64 operator()(long long u, long long i, long long n) const { return x[u * n + i]; }
};

struct FftArrayOut {
    mdp_c64 *y;
    __device__ __forceinline__ void operator()(long long u, long long i, long long n, const mdp_c64 &v) const { y[u * n + i] = v; }
};

static __global__ void __launch_bounds__(MDP_FFT_THREADS) k_fft_twiddle(mdp_c64 *__restrict__ W, long long n)
{
    const long long k = (long long)blockIdx.x * MDP_FFT_THREADS + threadIdx.x;
    if (k < n / 2) W[k] = mdp_twiddle(k, n);
}

// n follows the functors: ptxas allocates registers by parameter layout, and in this order no pass needs more than the
// 64 registers of four blocks per SM where it did not before (IsfRhoIn at R = 3 takes 70 with n last).
template <int R, class In, class Out>
static __global__ void __launch_bounds__(MDP_FFT_THREADS) k_fft_pass(const In in, const Out out, long long n,
                                                                      const mdp_c64 *__restrict__ W, int t)
{
    const long long i = (long long)blockIdx.x * MDP_FFT_THREADS + threadIdx.x;
    if (i >= (n >> R)) return;
    const long long u = blockIdx.y;
    mdp_fft_radix_pass<R>([&](long long j) { return in(u, j, n); }, [&](long long j, const mdp_c64 &v) { out(u, j, n, v); }, W, i,
                          t, n);
}

// grid (ceil(n / MDP_FFT_THREADS), transforms): x[j][k] = acc[g][fold k] + i acc[g + 1][fold k] for inverse transform j0 + j,
// which is transform j' of bin b (mdp_fft_pair_groups; acc [bins][per_bin][n/2 + 1])
static __global__ void __launch_bounds__(MDP_FFT_THREADS) k_fft_spec_load(const double *__restrict__ acc, long long n, int per_bin,
                                                                          long long j0, mdp_c64 *__restrict__ x)
{
    const long long k = (long long)blockIdx.x * MDP_FFT_THREADS + threadIdx.x;
    if (k >= n) return;
    const long long tpb = mdp_fft_transforms_per_bin(per_bin), j = j0 + blockIdx.y, b = j / tpb;
    const mdp_fft_group_pair gp = mdp_fft_pair_groups(j % tpb, per_bin);
    const long long H = n / 2 + 1, g = b * per_bin + gp.first, kk = mdp_fft_fold(k, n);
    mdp_c64 v;
    v.re = acc[g * H + kk];
    v.im = gp.partner ? acc[(g + 1) * H + kk] : 0.0;
    x[(long long)blockIdx.y * n + k] = v;
}

static inline void mdp_fft_twiddles(mdp_ctx *ctx, mdp_c64 *W, long long n, cudaStream_t st)   // W[k] = exp(-2 pi i k / n), k < n/2
{
    k_fft_twiddle<<<(unsigned)ceil_div<long long>(std::max<long long>(n / 2, 1), MDP_FFT_THREADS), MDP_FFT_THREADS, 0, st>>>(W, n);
    MDP_LAUNCHED(ctx);
}

template <class In, class Out>
static void mdp_fft_launch_pass(int R, const In &in, const Out &out, const mdp_c64 *W, int t, long long n, int units, cudaStream_t st)
{
    const dim3 g((unsigned)ceil_div<long long>(std::max<long long>(n >> R, 1), MDP_FFT_THREADS), (unsigned)units);
    if (R == 3) k_fft_pass<3><<<g, MDP_FFT_THREADS, 0, st>>>(in, out, n, W, t);
    else if (R == 2) k_fft_pass<2><<<g, MDP_FFT_THREADS, 0, st>>>(in, out, n, W, t);
    else k_fft_pass<1><<<g, MDP_FFT_THREADS, 0, st>>>(in, out, n, W, t);
}

// One forward transform of 2^p points per unit, in passes of mdp_fft_pass_radix stages (one launch each) between the work
// arrays x (the input, unless first_in reads it from elsewhere) and y.  The first pass reads through first_in, the last
// writes through last_out; an FftArrayOut as last_out writes the work array that pass writes.  Returns that array.
template <class In, class Out>
static mdp_c64 *mdp_fft_transform(mdp_ctx *ctx, const In &first_in, Out last_out, mdp_c64 *x, mdp_c64 *y, const mdp_c64 *W, int p,
                                  int units, cudaStream_t st)
{
    const long long n = 1ll << p;
    for (int t = 0; t < p;) {
        const int R = mdp_fft_pass_radix(t, p);
        if constexpr (std::is_same<Out, FftArrayOut>::value) last_out.y = y;
        if (t == 0 && t + R == p) mdp_fft_launch_pass(R, first_in, last_out, W, t, n, units, st);
        else if (t == 0) mdp_fft_launch_pass(R, first_in, FftArrayOut{y}, W, t, n, units, st);
        else if (t + R == p) mdp_fft_launch_pass(R, FftArrayIn{x}, last_out, W, t, n, units, st);
        else mdp_fft_launch_pass(R, FftArrayIn{x}, FftArrayOut{y}, W, t, n, units, st);
        MDP_LAUNCHED(ctx);
        std::swap(x, y);
        t += R;
    }
    return x;
}
