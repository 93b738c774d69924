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
//     k_msd_fft_pass  the forward transform, three butterfly stages per pass (the first pass reads the centred series);
//     k_msd_spec_acc  acc_g[k] += the unit spectra of group g, units in order, k <= N/2 (the spectrum is even).  The
//                     accumulator lives across sub-batches, so a group may span several of them and the summation order
//                     -- hence every bit of the result -- does not depend on the scratch limit;
//   per sub-batch of group pairs:
//     k_msd_spec_load acc_g + i acc_{g+1} unfolded to N points;
//     k_msd_fft_pass  the inverse transform (a forward FFT of a real even spectrum); its last pass writes out[g] and
//                     out[g+1] through mdp_msd_epilogue.
// HBM traffic: 32 B per point and pass of the transforms (as fftcorr.cu), plus 16 B per point for the spectrum
// accumulation and 8-16 B per series point for the mean and p sums.  No atomics: results are run-to-run identical.
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "msd_fft.h"
#include "scratch_plan.h"

namespace {

constexpr int MF_THREADS = 256;
constexpr int MF_SCAN_THREADS = 1024;

__global__ void __launch_bounds__(MF_THREADS) k_msd_twiddle(mdp_c64 *__restrict__ W, long long n)
{
    const long long k = (long long)blockIdx.x * MF_THREADS + threadIdx.x;
    if (k < n / 2) W[k] = mdp_twiddle(k, n);
}

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

// IO 0: array -> array; 1: the first forward pass reads the centred series of unit blockIdx.y (utab = {c0, c1, group},
// c1 = -1 for zero); 2: the last inverse pass writes out[g][tau], out[g+1][tau] (g = 2 * (pair0 + blockIdx.y)), tau < nlags
struct MsdIo {
    const mdp_c64 *x;
    mdp_c64 *y;
    const double *a, *b, *ma, *mb;
    const int *utab;
    const long long *goff;
    const double *pre, *suf;
    double *out;
    long long T, nlags, n;
    int self, ngroups, pair0;
};

template <int IO>
struct MsdIn {
    const MsdIo &io;
    long long u;
    __device__ __forceinline__ mdp_c64 operator()(long long i) const
    {
        if (IO != 1) return io.x[u * io.n + i];
        mdp_c64 v;
        v.re = 0.0;
        v.im = 0.0;
        if (i < io.T) {
            const int c0 = io.utab[3 * u], c1 = io.utab[3 * u + 1];
            v.re = __ldg(io.a + (long long)c0 * io.T + i) - __ldg(io.ma + c0);
            if (!io.self) v.im = __ldg(io.b + (long long)c0 * io.T + i) - __ldg(io.mb + c0);
            else if (c1 >= 0) v.im = __ldg(io.a + (long long)c1 * io.T + i) - __ldg(io.ma + c1);
        }
        return v;
    }
};

template <int IO>
struct MsdOut {
    const MsdIo &io;
    long long u;
    __device__ __forceinline__ void operator()(long long i, const mdp_c64 &v) const
    {
        if (IO != 2) {
            io.y[u * io.n + i] = v;
            return;
        }
        if (i >= io.nlags) return;
        // an empty group is exactly zero (its transform partner would leave round-off in its half of the transform)
        const long long g = 2 * (io.pair0 + u), T1 = io.T + 1;
        io.out[g * io.nlags + i] = io.goff[g + 1] == io.goff[g] ? 0.0
            : mdp_msd_epilogue(io.suf + g * T1, io.pre + g * T1, io.T, i, v.re / (double)io.n);
        if (g + 1 < io.ngroups)
            io.out[(g + 1) * io.nlags + i] = io.goff[g + 2] == io.goff[g + 1] ? 0.0
                : mdp_msd_epilogue(io.suf + (g + 1) * T1, io.pre + (g + 1) * T1, io.T, i, v.im / (double)io.n);
    }
};

template <int R, int IO>
__global__ void __launch_bounds__(MF_THREADS) k_msd_fft_pass(const MsdIo io, const mdp_c64 *__restrict__ W, int t)
{
    const long long i = (long long)blockIdx.x * MF_THREADS + threadIdx.x;
    if (i >= (io.n >> R)) return;
    const long long u = blockIdx.y;
    mdp_fft_radix_pass<R>(MsdIn<IO>{io, u}, MsdOut<IO>{io, u}, W, i, t, io.n);
}

template <int IO>
void launch_msd_pass(int R, const MsdIo &io, const mdp_c64 *W, int t, int units, cudaStream_t st)
{
    const dim3 g((unsigned)ceil_div<long long>(std::max<long long>(io.n >> R, 1), MF_THREADS), (unsigned)units);
    if (R == 3) k_msd_fft_pass<3, IO><<<g, MF_THREADS, 0, st>>>(io, W, t);
    else if (R == 2) k_msd_fft_pass<2, IO><<<g, MF_THREADS, 0, st>>>(io, W, t);
    else k_msd_fft_pass<1, IO><<<g, MF_THREADS, 0, st>>>(io, W, t);
}

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

// grid (ceil(n / MF_THREADS), pairs): x[j][k] = acc[2 (pair0 + j)][fold k] + i acc[2 (pair0 + j) + 1][fold k]
__global__ void __launch_bounds__(MF_THREADS) k_msd_spec_load(const double *__restrict__ acc, long long n, int ngroups, int pair0,
                                                              mdp_c64 *__restrict__ x)
{
    const long long k = (long long)blockIdx.x * MF_THREADS + threadIdx.x;
    if (k >= n) return;
    const long long H = n / 2 + 1, g = 2 * ((long long)pair0 + blockIdx.y), kk = mdp_msd_fold(k, n);
    mdp_c64 v;
    v.re = acc[g * H + kk];
    v.im = g + 1 < ngroups ? acc[(g + 1) * H + kk] : 0.0;
    x[(long long)blockIdx.y * n + k] = v;
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
    k_msd_twiddle<<<(unsigned)ceil_div<long long>(std::max<long long>(n / 2, 1), MF_THREADS), MF_THREADS, 0, st>>>(W, n);
    MDP_LAUNCHED(ctx);
    k_msd_mean<<<dim3((unsigned)nchan, self ? 1 : 2), MDP_MSD_MEAN_LANES, 0, st>>>(a, b, T, ma, mb);
    MDP_LAUNCHED(ctx);
    k_msd_psum<<<dim3((unsigned)ceil_div<long long>(T, MF_THREADS), (unsigned)ngroups), MF_THREADS, 0, st>>>(a, b, ma, mb, d_goff, T,
                                                                                                          psum);
    MDP_LAUNCHED(ctx);
    k_msd_scan<<<(unsigned)ngroups, MF_SCAN_THREADS, 0, st>>>(psum, T, pre, suf);
    MDP_LAUNCHED(ctx);

    MsdIo io{nullptr, nullptr, a, b, ma, mb, d_utab, d_goff, pre, suf, out, T, nlags, n, self, ngroups, 0};
    int g_lo = 0;
    for (long long u0 = 0; u0 < U; u0 += batch) {                    // forward transforms and spectrum accumulation
        const long long u1 = std::min(U, u0 + batch);
        io.utab = d_utab + 3 * u0;
        mdp_c64 *src = x, *dst = y;
        for (int t = 0; t < p;) {
            const int R = mdp_fft_pass_radix(t, p);
            io.x = src;
            io.y = dst;
            if (t == 0) launch_msd_pass<1>(R, io, W, t, (int)(u1 - u0), st);
            else launch_msd_pass<0>(R, io, W, t, (int)(u1 - u0), st);
            MDP_LAUNCHED(ctx);
            std::swap(src, dst);
            t += R;
        }
        while (uoff[(size_t)g_lo + 1] <= u0) ++g_lo;                 // first group with a unit in [u0, u1)
        int g_hi = g_lo;
        while (uoff[(size_t)g_hi + 1] < u1) ++g_hi;                  // last one
        k_msd_spec_acc<<<dim3((unsigned)ceil_div<long long>(H, MF_THREADS), (unsigned)(g_hi - g_lo + 1)), MF_THREADS, 0, st>>>(
            src, n, d_uoff, g_lo, u0, u1, self, acc);
        MDP_LAUNCHED(ctx);
    }
    const int pairs = (ngroups + 1) / 2;
    for (int j0 = 0; j0 < pairs; j0 += (int)batch) {                 // inverse transforms, two groups each
        const int nj = (int)std::min<long long>(batch, pairs - j0);
        k_msd_spec_load<<<dim3((unsigned)ceil_div<long long>(n, MF_THREADS), (unsigned)nj), MF_THREADS, 0, st>>>(acc, n, ngroups, j0, x);
        MDP_LAUNCHED(ctx);
        io.pair0 = j0;
        mdp_c64 *src = x, *dst = y;
        for (int t = 0; t < p;) {
            const int R = mdp_fft_pass_radix(t, p);
            io.x = src;
            io.y = dst;
            if (t + R == p) launch_msd_pass<2>(R, io, W, t, nj, st);
            else launch_msd_pass<0>(R, io, W, t, nj, st);
            MDP_LAUNCHED(ctx);
            std::swap(src, dst);
            t += R;
        }
    }
    ctx->timer_end(tk, st);
    return mdp_check_launch("k_msd_fft_pass");
}

} // extern "C"
