// fftcorr.cu -- unbiased time correlation through a Stockham FFT (the default for series of >= 2048 steps,
// ops.XCORR_FFT_MIN_T; shorter ones and MDP_XCORR_FFT=0 take the direct fp64 sum k_xcorr of corr.cu).
//
// Same result as mdp_xcorr_unbiased (Conductivity.correlate conductivity.py:97-114, Viscosity.autocorrelate
// viscosity.py:86-120) to the round-off of an FFT -- which is how the reference itself computes it -- at N log N instead of
// T^2/2: method in fft_corr.h.  Every pass is one launch over all channels and covers THREE butterfly stages in registers
// (N/8 threads per channel, eight points each, coalesced 16-byte complex loads); the first pass reads the series and the
// last one writes the normalised correlation, so a 2^18-point correlation is 13 passes over the work arrays instead of
// 39.  HBM-bound: 32 B per point and pass.  Channels are processed in groups that keep the two work arrays within the
// scratch arena.
#include <algorithm>

#include "common.cuh"
#include "fft_corr.h"
#include "scratch_plan.h"

namespace {

constexpr int FC_THREADS = 256;

__global__ void __launch_bounds__(FC_THREADS) k_fft_twiddle(mdp_c64 *__restrict__ W, long long n)
{
    const long long k = (long long)blockIdx.x * FC_THREADS + threadIdx.x;
    if (k < n / 2) W[k] = mdp_twiddle(k, n);
}

// One pass = R fused stages (fft_corr.h: mdp_fft_radix_pass).  IO 0: array -> array; 1: the first pass of the first
// transform reads z = a + i*b (0 beyond T) straight from the series; 2: the last pass of the second transform writes
// out[tau] = Re X[tau] / N / (T - tau) for tau < nlags and nothing else.  grid (ceil((n >> R) / FC_THREADS), channels)
struct FftIo {
    const mdp_c64 *x;
    mdp_c64 *y;
    const double *a, *b;
    double *out;
    long long T, nlags, n;
};

template <int IO>
struct FftIn {
    const FftIo &io;
    long long c;
    __device__ __forceinline__ mdp_c64 operator()(long long i) const
    {
        if (IO != 1) return io.x[c * io.n + i];
        mdp_c64 v;
        v.re = i < io.T ? __ldg(io.a + c * io.T + i) : 0.0;
        v.im = i < io.T ? __ldg(io.b + c * io.T + i) : 0.0;
        return v;
    }
};

template <int IO>
struct FftOut {
    const FftIo &io;
    long long c;
    __device__ __forceinline__ void operator()(long long i, const mdp_c64 &v) const
    {
        if (IO != 2) io.y[c * io.n + i] = v;
        else if (i < io.nlags) io.out[c * io.nlags + i] = v.re / (double)io.n / (double)(io.T - i);
    }
};

template <int R, int IO>
__global__ void __launch_bounds__(FC_THREADS) k_fft_pass(const FftIo io, const mdp_c64 *__restrict__ W, int t)
{
    const long long i = (long long)blockIdx.x * FC_THREADS + threadIdx.x;
    if (i >= (io.n >> R)) return;
    const long long c = blockIdx.y;
    mdp_fft_radix_pass<R>(FftIn<IO>{io, c}, FftOut<IO>{io, c}, W, i, t, io.n);
}

template <int IO>
void launch_fft_pass(int R, const FftIo &io, const mdp_c64 *W, int t, int chans, cudaStream_t st)
{
    const dim3 g((unsigned)ceil_div<long long>(std::max<long long>(io.n >> R, 1), FC_THREADS), (unsigned)chans);
    if (R == 3) k_fft_pass<3, IO><<<g, FC_THREADS, 0, st>>>(io, W, t);
    else if (R == 2) k_fft_pass<2, IO><<<g, FC_THREADS, 0, st>>>(io, W, t);
    else k_fft_pass<1, IO><<<g, FC_THREADS, 0, st>>>(io, W, t);
}

__global__ void __launch_bounds__(FC_THREADS) k_fft_cross(const mdp_c64 *__restrict__ Z, mdp_c64 *__restrict__ P, long long n)
{
    const long long k = (long long)blockIdx.x * FC_THREADS + threadIdx.x;
    if (k >= n) return;
    const long long c = blockIdx.y;
    P[c * n + k] = mdp_cross_spectrum_conj(Z + c * n, k, n);
}

} // namespace

extern "C" {

int mdp_xcorr_fft(mdp_ctx *ctx, int nchan, int64_t T, const double *a, const double *b, int64_t nlags, double *out, void *stream)
{
    MDP_REQUIRE(ctx && a && b && out, "mdp_xcorr_fft: NULL argument");
    MDP_REQUIRE(nchan > 0 && T > 0 && nlags > 0 && nlags <= T, "mdp_xcorr_fft: bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    MDP_CUDA(cudaSetDevice(ctx->device));
    const int p = mdp_fft_log2_size(T, nlags);
    MDP_REQUIRE(p <= 30, "mdp_xcorr_fft: %lld steps need a transform of 2^%d points", (long long)T, p);
    const long long n = 1ll << p;
    const size_t per_chan = (size_t)n * sizeof(mdp_c64);
    const size_t wbytes = align256((size_t)(n / 2) * sizeof(mdp_c64));
    // two work arrays per channel of the group; groups sized to 2 GiB of scratch (at least one channel), on the whole
    // request and what arena_reserve adds to it (scratch_plan.h)
    const size_t budget = std::min<size_t>(ctx->slab_limit, (size_t)2 << 30);
    const size_t fixed_req = wbytes + 4096, per_chan_req = 2 * align256(per_chan);
    const int group = (int)mdp_scratch_units(budget, fixed_req, per_chan_req, (size_t)std::min(nchan, 65535));
    int rc = ctx->arena_reserve(fixed_req + (size_t)group * per_chan_req);
    if (rc) return rc;
    ctx->arena_reset();
    mdp_c64 *W = (mdp_c64 *)ctx->arena_take((size_t)(n / 2) * sizeof(mdp_c64));
    mdp_c64 *x = (mdp_c64 *)ctx->arena_take((size_t)group * per_chan);
    mdp_c64 *y = (mdp_c64 *)ctx->arena_take((size_t)group * per_chan);
    if (!W || !x || !y) {
        mdp_set_error("internal: scratch arena exhausted (fft correlation)");
        return MDP_ERR_OOM;
    }
    cudaEvent_t tk = ctx->timer_begin(3, st);
    k_fft_twiddle<<<(unsigned)ceil_div<long long>(std::max<long long>(n / 2, 1), FC_THREADS), FC_THREADS, 0, st>>>(W, n);
    MDP_LAUNCHED(ctx);
    for (int c0 = 0; c0 < nchan; c0 += group) {
        const int g = std::min(group, nchan - c0);
        const dim3 gn((unsigned)ceil_div<long long>(n, FC_THREADS), (unsigned)g);
        FftIo io{nullptr, nullptr, a + (size_t)c0 * T, b + (size_t)c0 * T, out + (size_t)c0 * nlags, T, nlags, n};
        mdp_c64 *src = x, *dst = y;
        for (int t = 0; t < p;) {                                   // Z = FFT(a + i*b)
            const int R = mdp_fft_pass_radix(t, p);
            io.x = src;
            io.y = dst;
            if (t == 0) launch_fft_pass<1>(R, io, W, t, g, st);
            else launch_fft_pass<0>(R, io, W, t, g, st);
            MDP_LAUNCHED(ctx);
            std::swap(src, dst);
            t += R;
        }
        k_fft_cross<<<gn, FC_THREADS, 0, st>>>(src, dst, n);
        MDP_LAUNCHED(ctx);
        std::swap(src, dst);
        for (int t = 0; t < p;) {                                   // FFT(conj(P)) = N * conj(corr)
            const int R = mdp_fft_pass_radix(t, p);
            io.x = src;
            io.y = dst;
            if (t + R == p) launch_fft_pass<2>(R, io, W, t, g, st);
            else launch_fft_pass<0>(R, io, W, t, g, st);
            MDP_LAUNCHED(ctx);
            std::swap(src, dst);
            t += R;
        }
    }
    ctx->timer_end(tk, st);
    return mdp_check_launch("k_fft_pass");
}

} // extern "C"
