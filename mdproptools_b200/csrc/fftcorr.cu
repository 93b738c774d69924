// fftcorr.cu -- unbiased time correlation through a Stockham FFT (the default for series of >= 2048 steps,
// ops.XCORR_FFT_MIN_T; shorter ones and MDP_XCORR_FFT=0 take the direct fp64 sum k_xcorr of corr.cu).
//
// Same result as mdp_xcorr_unbiased (Conductivity.correlate conductivity.py:97-114, Viscosity.autocorrelate
// viscosity.py:86-120) to the round-off of an FFT -- which is how the reference itself computes it -- at N log N instead of
// T^2/2: method in fft_corr.h.  The transforms run through the shared passes of fft_pass.cuh: every pass is one launch
// over all channels and covers THREE butterfly stages in registers (N/8 threads per channel, eight points each, coalesced
// 16-byte complex loads); the first pass reads the series (XcorrSeriesIn) and the last one writes the normalised
// correlation (XcorrNormOut), so a 2^18-point correlation is 13 passes over the work arrays instead of 39.  HBM-bound:
// 32 B per point and pass.  Channels are processed in groups that keep the two work arrays within the scratch arena.
#include <algorithm>

#include "common.cuh"
#include "fft_pass.cuh"
#include "scratch_plan.h"

namespace {

constexpr int FC_THREADS = 256;

// the first pass of the first transform reads z = a + i*b of channel u (0 beyond T) straight from the series
struct XcorrSeriesIn {
    const double *a, *b;
    long long T;
    __device__ __forceinline__ mdp_c64 operator()(long long u, long long i, long long) const
    {
        mdp_c64 v;
        v.re = i < T ? __ldg(a + u * T + i) : 0.0;
        v.im = i < T ? __ldg(b + u * T + i) : 0.0;
        return v;
    }
};

// the last pass of the second transform writes out[u][tau] = Re X[tau] / N / (T - tau) for tau < nlags and nothing else
struct XcorrNormOut {
    double *out;
    long long T, nlags;
    __device__ __forceinline__ void operator()(long long u, long long i, long long n, const mdp_c64 &v) const
    {
        if (i < nlags) out[u * nlags + i] = mdp_fft_unbiased(v.re, n, T, i);
    }
};

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
    mdp_fft_twiddles(ctx, W, n, st);
    for (int c0 = 0; c0 < nchan; c0 += group) {
        const int g = std::min(group, nchan - c0);
        const dim3 gn((unsigned)ceil_div<long long>(n, FC_THREADS), (unsigned)g);
        // Z = FFT(a + i*b), then FFT(conj(P)) = N * conj(corr)
        mdp_c64 *Z = mdp_fft_transform(ctx, XcorrSeriesIn{a + (size_t)c0 * T, b + (size_t)c0 * T, T}, FftArrayOut{}, x, y, W, p, g, st);
        mdp_c64 *P = Z == x ? y : x;
        k_fft_cross<<<gn, FC_THREADS, 0, st>>>(Z, P, n);
        MDP_LAUNCHED(ctx);
        mdp_fft_transform(ctx, FftArrayIn{P}, XcorrNormOut{out + (size_t)c0 * nlags, T, nlags}, P, Z, W, p, g, st);
    }
    ctx->timer_end(tk, st);
    return mdp_check_launch("k_fft_pass");
}

} // extern "C"
