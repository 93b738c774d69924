// msdfft.cu -- all-origins (cross) mean-square displacement of channel groups through the Stockham FFT (method and
// accuracy contract in msd_fft.h).  Conductivity.einstein (the translational-dipole MSD) and Conductivity.nernst (the
// per-type centre-of-mass MSD) use it; it costs N log N per channel where mdp_msd_all_origins costs T * max_lag.
//
// One call:
//   k_msd_mean      channel means, fixed order (one CTA per channel);
//   k_msd_psum      p_g(t) = sum over the group's channels (fixed order) of the centred a(t) * b(t);
//   k_msd_scan      per group the prefix sums pre[t] = sum_{s<t} p and suffix sums suf[t] = sum_{s>=t} p (one CTA, fixed
//                   order: per-thread chunks, a serial scan of the chunk sums, then the chunks);
//   per sub-batch of transforms ("units": channel a_c + i b_c in the cross case, two channels a_c + i a_c' of the same
//   group in the self case, an odd last channel paired with zero):
//     k_fft_pass      the forward transform, three butterfly stages per pass (fft_pass.cuh; the first pass reads the
//                     centred series through MsdSeriesIn);
//     k_msd_spec_acc  acc_g[k] += the unit spectra of group g, units in order, k <= N/2 (the spectrum is even).  The
//                     accumulator lives across sub-batches, so a group may span several of them and the summation order
//                     -- hence every bit of the result -- does not depend on the scratch limit;
//   per sub-batch of group pairs:
//     k_fft_spec_load acc_g + i acc_{g+1} unfolded to N points (the groups are one bin of mdp_fft_pair_groups);
//     k_fft_pass      the inverse transform (a forward FFT of a real even spectrum); its last pass writes out[g] and
//                     out[g+1] through MsdEpilogueOut (mdp_msd_epilogue).
// HBM traffic: 32 B per point and pass of the transforms (as fftcorr.cu), plus 16 B per point for the spectrum
// accumulation and 8-16 B per series point for the mean and p sums.  No atomics: results are run-to-run identical.
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "fft_pass.cuh"
#include "msd_fft.h"
#include "scratch_plan.h"

namespace {

constexpr int MF_THREADS = 256;
constexpr int MF_SCAN_THREADS = 1024;

// grid (nchan, 1 or 2): mean of channel blockIdx.x of a (y = 0) or b (y = 1)
__global__ void __launch_bounds__(MDP_MSD_MEAN_LANES) k_msd_mean(const double *__restrict__ a, const double *__restrict__ b,
                                                                 long long T, double *__restrict__ ma, double *__restrict__ mb)
{
    __shared__ double sh[MDP_MSD_MEAN_LANES];
    const long long c = blockIdx.x;
    const double *x = (blockIdx.y ? b : a) + c * T;
    sh[threadIdx.x] = mdp_msd_lane_sum(x, T, (int)threadIdx.x);
    __syncthreads();
    for (int h = MDP_MSD_MEAN_LANES / 2; h > 0; h >>= 1) {
        if ((int)threadIdx.x < h) sh[threadIdx.x] += sh[threadIdx.x + h];
        __syncthreads();
    }
    if (threadIdx.x == 0) (blockIdx.y ? mb : ma)[c] = sh[0] / (double)T;
}

// grid (ceil(T / MF_THREADS), ngroups): p[g][t] = sum_{c in g} (a_c(t) - ma_c) * (b_c(t) - mb_c), channels in order
__global__ void __launch_bounds__(MF_THREADS) k_msd_psum(const double *__restrict__ a, const double *__restrict__ b,
                                                         const double *__restrict__ ma, const double *__restrict__ mb,
                                                         const long long *__restrict__ goff, long long T, double *__restrict__ p)
{
    const long long t = (long long)blockIdx.x * MF_THREADS + threadIdx.x;
    if (t >= T) return;
    const int g = blockIdx.y;
    const long long c0 = goff[g], c1 = goff[g + 1];
    double s = 0.0;
#pragma unroll 4
    for (long long c = c0; c < c1; ++c) s += (__ldg(a + c * T + t) - __ldg(ma + c)) * (__ldg(b + c * T + t) - __ldg(mb + c));
    p[(long long)g * T + t] = s;
}

// grid ngroups: pre[g][0..T] and suf[g][0..T] of p[g][0..T-1]
__global__ void __launch_bounds__(MF_SCAN_THREADS) k_msd_scan(const double *__restrict__ p, long long T, double *__restrict__ pre,
                                                              double *__restrict__ suf)
{
    __shared__ double part[MF_SCAN_THREADS], base_lo[MF_SCAN_THREADS], base_hi[MF_SCAN_THREADS];
    const long long g = blockIdx.x;
    const double *x = p + g * T;
    double *P = pre + g * (T + 1), *S = suf + g * (T + 1);
    const long long L = (T + MF_SCAN_THREADS - 1) / MF_SCAN_THREADS;
    const long long t0 = min(T, (long long)threadIdx.x * L), t1 = min(T, t0 + L);
    double s = 0.0;
    for (long long t = t0; t < t1; ++t) s += x[t];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = 0.0;
        for (int j = 0; j < MF_SCAN_THREADS; ++j) {
            base_lo[j] = r;
            r += part[j];
        }
        r = 0.0;
        for (int j = MF_SCAN_THREADS - 1; j >= 0; --j) {
            base_hi[j] = r;
            r += part[j];
        }
        P[0] = 0.0;
        S[T] = 0.0;
    }
    __syncthreads();
    double r = base_lo[threadIdx.x];
    for (long long t = t0; t < t1; ++t) {
        r += x[t];
        P[t + 1] = r;
    }
    r = base_hi[threadIdx.x];
    for (long long t = t1 - 1; t >= t0; --t) {
        r += x[t];
        S[t] = r;
    }
}

// the first forward pass reads the centred series of unit u (utab = {c0, c1, group}, c1 = -1 for zero)
struct MsdSeriesIn {
    const double *a, *b, *ma, *mb;
    const int *utab;
    long long T;
    int self;
    __device__ __forceinline__ mdp_c64 operator()(long long u, long long i, long long) const
    {
        mdp_c64 v;
        v.re = 0.0;
        v.im = 0.0;
        if (i < T) {
            const int c0 = utab[3 * u], c1 = utab[3 * u + 1];
            v.re = __ldg(a + (long long)c0 * T + i) - __ldg(ma + c0);
            if (!self) v.im = __ldg(b + (long long)c0 * T + i) - __ldg(mb + c0);
            else if (c1 >= 0) v.im = __ldg(a + (long long)c1 * T + i) - __ldg(ma + c1);
        }
        return v;
    }
};

// the last inverse pass writes out[g][tau], out[g+1][tau] of inverse transform j0 + u, tau < nlags (the groups are one bin
// of mdp_fft_pair_groups)
struct MsdEpilogueOut {
    const long long *goff;
    const double *pre, *suf;
    double *out;
    long long T, nlags;
    int ngroups, j0;
    __device__ __forceinline__ void operator()(long long u, long long i, long long n, const mdp_c64 &v) const
    {
        if (i >= nlags) return;
        // an empty group is exactly zero (its transform partner would leave round-off in its half of the transform)
        const mdp_fft_group_pair gp = mdp_fft_pair_groups(j0 + u, ngroups);
        const long long g = gp.first, T1 = T + 1;
        out[g * nlags + i] = goff[g + 1] == goff[g] ? 0.0 : mdp_msd_epilogue(suf + g * T1, pre + g * T1, T, i, v.re / (double)n);
        if (gp.partner)
            out[(g + 1) * nlags + i] = goff[g + 2] == goff[g + 1] ? 0.0
                : mdp_msd_epilogue(suf + (g + 1) * T1, pre + (g + 1) * T1, T, i, v.im / (double)n);
    }
};

// grid (ceil((n/2 + 1) / MF_THREADS), groups g_lo + blockIdx.y): acc[g][k] += spectra of the units of g in [u0, u1)
__global__ void __launch_bounds__(MF_THREADS) k_msd_spec_acc(const mdp_c64 *__restrict__ Z, long long n, const long long *__restrict__ uoff,
                                                             int g_lo, long long u0, long long u1, int self, double *__restrict__ acc)
{
    const long long k = (long long)blockIdx.x * MF_THREADS + threadIdx.x;
    const long long H = n / 2 + 1;
    if (k >= H) return;
    const long long g = g_lo + blockIdx.y;
    const long long ua = max(uoff[g], u0), ub = min(uoff[g + 1], u1);
    if (ua >= ub) return;
    double s = acc[g * H + k];
    for (long long u = ua; u < ub; ++u) {
        const mdp_c64 *z = Z + (u - u0) * n;
        s += self ? mdp_msd_spectrum_self(z, k, n) : mdp_msd_spectrum_cross(z, k, n);
    }
    acc[g * H + k] = s;
}

} // namespace

extern "C" {

int mdp_cross_msd_fft(mdp_ctx *ctx, int nchan, int64_t T, const double *a, const double *b, int ngroups, const int64_t *group_off,
                      int64_t nlags, double *out, void *stream)
{
    MDP_REQUIRE(ctx && a && group_off && out, "mdp_cross_msd_fft: NULL argument");
    MDP_REQUIRE(nchan > 0 && T > 0 && nlags > 0 && nlags <= T, "mdp_cross_msd_fft: bad sizes (nchan %d, T %lld, nlags %lld)",
                nchan, (long long)T, (long long)nlags);
    MDP_REQUIRE(ngroups >= 1 && ngroups <= 65535, "mdp_cross_msd_fft: ngroups %d outside [1, 65535]", ngroups);
    MDP_REQUIRE(group_off[0] == 0 && group_off[ngroups] == nchan,
                "mdp_cross_msd_fft: group_off must run from 0 to nchan = %d", nchan);
    for (int g = 0; g < ngroups; ++g)
        MDP_REQUIRE(group_off[g + 1] >= group_off[g], "mdp_cross_msd_fft: group_off decreases at group %d", g);
    const int p = mdp_fft_log2_size(T, nlags);
    MDP_REQUIRE(p <= 30, "mdp_cross_msd_fft: %lld steps need a transform of 2^%d points", (long long)T, p);
    const int self = b == nullptr || b == a;
    if (self) b = a;
    cudaStream_t st = (cudaStream_t)stream;
    MDP_CUDA(cudaSetDevice(ctx->device));
    const long long n = 1ll << p, H = n / 2 + 1;

    // units: cross -> one per channel; self -> channels (c, c+1) of a group, an odd last one alone
    std::vector<int> utab;
    std::vector<long long> uoff((size_t)ngroups + 1, 0), goff(group_off, group_off + ngroups + 1);
    for (int g = 0; g < ngroups; ++g) {
        for (long long c = group_off[g]; c < group_off[g + 1]; c += self ? 2 : 1) {
            utab.push_back((int)c);
            utab.push_back(self && c + 1 < group_off[g + 1] ? (int)(c + 1) : -1);
            utab.push_back(g);
        }
        uoff[(size_t)g + 1] = (long long)(utab.size() / 3);
    }
    const long long U = (long long)(utab.size() / 3);

    // group accumulators and everything else that does not scale with the sub-batch; sub-batches of units sized to 2 GiB
    // of scratch on the whole request (scratch_plan.h)
    const size_t wbytes = align256((size_t)(n / 2) * sizeof(mdp_c64));
    const size_t mbytes = align256((size_t)nchan * sizeof(double));
    const size_t fixed_req = wbytes + 2 * mbytes + align256(utab.size() * sizeof(int)) + 2 * align256(uoff.size() * 8) +
                             align256((size_t)ngroups * H * 8) + align256((size_t)ngroups * T * 8) +
                             2 * align256((size_t)ngroups * (T + 1) * 8) + 4096;
    const size_t per_unit = (size_t)n * sizeof(mdp_c64), per_unit_req = 2 * align256(per_unit);
    MDP_REQUIRE(mdp_scratch_reserved(fixed_req) <= ctx->slab_limit,
                "mdp_cross_msd_fft: the group accumulators of %d groups over 2^%d points (%zu B) exceed the context limit %zu B",
                ngroups, p, fixed_req, ctx->slab_limit);
    const size_t budget = std::min<size_t>(ctx->slab_limit, (size_t)2 << 30);
    const long long batch = (long long)mdp_scratch_units(budget, fixed_req, per_unit_req, (size_t)std::min<long long>(U, 65535));
    int rc = ctx->arena_reserve(fixed_req + (size_t)batch * per_unit_req);
    if (rc) return rc;
    ctx->arena_reset();
    mdp_c64 *W = (mdp_c64 *)ctx->arena_take((size_t)(n / 2) * sizeof(mdp_c64));
    double *ma = (double *)ctx->arena_take((size_t)nchan * sizeof(double));
    double *mb = self ? ma : (double *)ctx->arena_take((size_t)nchan * sizeof(double));
    int *d_utab = (int *)ctx->arena_take(utab.size() * sizeof(int));
    long long *d_uoff = (long long *)ctx->arena_take(uoff.size() * 8);
    long long *d_goff = (long long *)ctx->arena_take(goff.size() * 8);
    double *acc = (double *)ctx->arena_take((size_t)ngroups * H * 8);
    double *psum = (double *)ctx->arena_take((size_t)ngroups * T * 8);
    double *pre = (double *)ctx->arena_take((size_t)ngroups * (T + 1) * 8);
    double *suf = (double *)ctx->arena_take((size_t)ngroups * (T + 1) * 8);
    mdp_c64 *x = (mdp_c64 *)ctx->arena_take((size_t)batch * per_unit);
    mdp_c64 *y = (mdp_c64 *)ctx->arena_take((size_t)batch * per_unit);
    if (!W || !ma || !mb || !d_utab || !d_uoff || !d_goff || !acc || !psum || !pre || !suf || !x || !y) {
        mdp_set_error("internal: scratch arena exhausted (fft msd)");
        return MDP_ERR_OOM;
    }
    cudaEvent_t tk = ctx->timer_begin(7, st);
    if (U > 0) MDP_CUDA(cudaMemcpyAsync(d_utab, utab.data(), utab.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    MDP_CUDA(cudaMemcpyAsync(d_uoff, uoff.data(), uoff.size() * 8, cudaMemcpyHostToDevice, st));
    MDP_CUDA(cudaMemcpyAsync(d_goff, goff.data(), goff.size() * 8, cudaMemcpyHostToDevice, st));
    MDP_CUDA(cudaMemsetAsync(acc, 0, (size_t)ngroups * H * 8, st));
    mdp_fft_twiddles(ctx, W, n, st);
    k_msd_mean<<<dim3((unsigned)nchan, self ? 1 : 2), MDP_MSD_MEAN_LANES, 0, st>>>(a, b, T, ma, mb);
    MDP_LAUNCHED(ctx);
    k_msd_psum<<<dim3((unsigned)ceil_div<long long>(T, MF_THREADS), (unsigned)ngroups), MF_THREADS, 0, st>>>(a, b, ma, mb, d_goff, T,
                                                                                                          psum);
    MDP_LAUNCHED(ctx);
    k_msd_scan<<<(unsigned)ngroups, MF_SCAN_THREADS, 0, st>>>(psum, T, pre, suf);
    MDP_LAUNCHED(ctx);

    int g_lo = 0;
    for (long long u0 = 0; u0 < U; u0 += batch) {                    // forward transforms and spectrum accumulation
        const long long u1 = std::min(U, u0 + batch);
        const mdp_c64 *Z = mdp_fft_transform(ctx, MsdSeriesIn{a, b, ma, mb, d_utab + 3 * u0, T, self}, FftArrayOut{}, x, y, W, p,
                                             (int)(u1 - u0), st);
        while (uoff[(size_t)g_lo + 1] <= u0) ++g_lo;                 // first group with a unit in [u0, u1)
        int g_hi = g_lo;
        while (uoff[(size_t)g_hi + 1] < u1) ++g_hi;                  // last one
        k_msd_spec_acc<<<dim3((unsigned)ceil_div<long long>(H, MF_THREADS), (unsigned)(g_hi - g_lo + 1)), MF_THREADS, 0, st>>>(
            Z, n, d_uoff, g_lo, u0, u1, self, acc);
        MDP_LAUNCHED(ctx);
    }
    const int pairs = (int)mdp_fft_transforms_per_bin(ngroups);
    for (int j0 = 0; j0 < pairs; j0 += (int)batch) {                 // inverse transforms, two groups each
        const int nj = (int)std::min<long long>(batch, pairs - j0);
        k_fft_spec_load<<<dim3((unsigned)ceil_div<long long>(n, MDP_FFT_THREADS), (unsigned)nj), MDP_FFT_THREADS, 0, st>>>(acc, n, ngroups,
                                                                                                                     j0, x);
        MDP_LAUNCHED(ctx);
        mdp_fft_transform(ctx, FftArrayIn{x}, MsdEpilogueOut{d_goff, pre, suf, out, T, nlags, ngroups, j0}, x, y, W, p, nj, st);
    }
    ctx->timer_end(tk, st);
    return mdp_check_launch("k_fft_pass");
}

} // extern "C"
