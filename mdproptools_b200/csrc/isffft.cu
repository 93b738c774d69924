// isffft.cu -- binned, symmetrised all-origins correlation of complex per-k series through the Stockham FFT: the coherent
// intermediate scattering function (method and accuracy contract in isf_fft.h, ABI in include/mdprop_b200.h).
//
// One call:
//   per sub-batch of whole k-vectors (all channels that a pair uses, "units" = (k, channel) series):
//     k_isf_fft_pass  the forward transform, three butterfly stages per pass (the first pass reads rho[c][k][0..T) and
//                     zero-pads it);
//     k_isf_spec_acc  acc_g[w] += G_k(w) of every group g = (bin, pair) over the bin's k-vectors in the sub-batch, in k
//                     order, w <= N/2 (G is even).  The accumulator lives across sub-batches, so the summation order -- hence
//                     every bit of the result -- does not depend on the scratch limit;
//   k_isf_flag        per group: does its half spectrum hold a nonzero value (an empty bin or a pair of empty channels comes
//                     out exactly zero instead of carrying round-off of its transform partner);
//   per sub-batch of inverse transforms (two groups of the same bin each):
//     k_isf_spec_load acc_g + i acc_{g+1} unfolded to N points;
//     k_isf_fft_pass  the inverse transform (a forward FFT of a real even spectrum); its last pass writes out[p][bin] and
//                     out[p+1][bin] through mdp_isf_epilogue.
// HBM traffic: 32 B per point and pass of the transforms, plus 16 B per point and pair for the spectrum accumulation.  No
// atomics: run-to-run bit-identical.
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "isf_fft.h"
#include "scratch_plan.h"

namespace {

constexpr int IF_THREADS = 256;

__global__ void __launch_bounds__(IF_THREADS) k_isf_twiddle(mdp_c64 *__restrict__ W, long long n)
{
    const long long k = (long long)blockIdx.x * IF_THREADS + threadIdx.x;
    if (k < n / 2) W[k] = mdp_twiddle(k, n);
}

// IO 0: array -> array; 1: the first forward pass reads unit blockIdx.y = (k0 + u / nused, channel used[u % nused]) of
// rho; 2: the last inverse pass writes transform j0 + blockIdx.y to out, tau < nlags
struct IsfIo {
    const mdp_c64 *x;
    mdp_c64 *y;
    const mdp_c64 *rho;
    const int *used, *flag;
    double *out;
    long long T, nk, nlags, n, k0, j0;
    int nused, npairs, nbins;
};

template <int IO>
struct IsfIn {
    const IsfIo &io;
    long long u;
    __device__ __forceinline__ mdp_c64 operator()(long long i) const
    {
        if (IO != 1) return io.x[u * io.n + i];
        mdp_c64 v;
        v.re = 0.0;
        v.im = 0.0;
        if (i < io.T) {
            const long long k = io.k0 + u / io.nused, c = io.used[u % io.nused];
            const double2 z = __ldg((const double2 *)io.rho + (c * io.nk + k) * io.T + i);
            v.re = z.x;
            v.im = z.y;
        }
        return v;
    }
};

template <int IO>
struct IsfOut {
    const IsfIo &io;
    long long u;
    __device__ __forceinline__ void operator()(long long i, const mdp_c64 &v) const
    {
        if (IO != 2) {
            io.y[u * io.n + i] = v;
            return;
        }
        if (i >= io.nlags) return;
        const long long tpb = mdp_isf_transforms_per_bin(io.npairs), j = io.j0 + u;
        const long long b = j / tpb, p = 2 * (j % tpb), g = b * io.npairs + p;
        io.out[(p * io.nbins + b) * io.nlags + i] = io.flag[g] ? mdp_isf_epilogue(v.re, io.n, io.T, i) : 0.0;
        if (p + 1 < io.npairs)
            io.out[((p + 1) * io.nbins + b) * io.nlags + i] = io.flag[g + 1] ? mdp_isf_epilogue(v.im, io.n, io.T, i) : 0.0;
    }
};

template <int R, int IO>
__global__ void __launch_bounds__(IF_THREADS) k_isf_fft_pass(const IsfIo io, const mdp_c64 *__restrict__ W, int t)
{
    const long long i = (long long)blockIdx.x * IF_THREADS + threadIdx.x;
    if (i >= (io.n >> R)) return;
    const long long u = blockIdx.y;
    mdp_fft_radix_pass<R>(IsfIn<IO>{io, u}, IsfOut<IO>{io, u}, W, i, t, io.n);
}

template <int IO>
void launch_isf_pass(int R, const IsfIo &io, const mdp_c64 *W, int t, int units, cudaStream_t st)
{
    const dim3 g((unsigned)ceil_div<long long>(std::max<long long>(io.n >> R, 1), IF_THREADS), (unsigned)units);
    if (R == 3) k_isf_fft_pass<3, IO><<<g, IF_THREADS, 0, st>>>(io, W, t);
    else if (R == 2) k_isf_fft_pass<2, IO><<<g, IF_THREADS, 0, st>>>(io, W, t);
    else k_isf_fft_pass<1, IO><<<g, IF_THREADS, 0, st>>>(io, W, t);
}

// grid (ceil((n/2 + 1) / IF_THREADS), <= 65535): groups g_lo + blockIdx.y, + gridDim.y, ... below g_hi;
// acc[g][w] += sum over the k-vectors of g's bin in [k0, k1), in k order, of G_k(w).  Z = [k - k0][nused][n]
__global__ void __launch_bounds__(IF_THREADS) k_isf_spec_acc(const mdp_c64 *__restrict__ Z, long long n, int nused,
                                                             const long long *__restrict__ boff, const int *__restrict__ pidx,
                                                             int npairs, long long g_lo, long long g_hi, long long k0, long long k1,
                                                             double *__restrict__ acc)
{
    const long long w = (long long)blockIdx.x * IF_THREADS + threadIdx.x;
    const long long H = n / 2 + 1;
    if (w >= H) return;
    for (long long g = g_lo + blockIdx.y; g < g_hi; g += gridDim.y) {
        const long long b = g / npairs, p = g % npairs;
        const long long ka = max(boff[b], k0), kb = min(boff[b + 1], k1);
        if (ka >= kb) continue;
        const long long ia = pidx[2 * p], ib = pidx[2 * p + 1];
        double s = acc[g * H + w];
        for (long long k = ka; k < kb; ++k) {
            const mdp_c64 *z = Z + (k - k0) * nused * n;
            s += mdp_isf_spectrum(z + ia * n, z + ib * n, w, n);
        }
        acc[g * H + w] = s;
    }
}

// grid ngroups: flag[g] = some acc[g][w] != 0
__global__ void __launch_bounds__(IF_THREADS) k_isf_flag(const double *__restrict__ acc, long long H, int *__restrict__ flag)
{
    const long long g = blockIdx.x;
    int nz = 0;
    for (long long w = threadIdx.x; w < H; w += IF_THREADS) nz |= acc[g * H + w] != 0.0;
    nz = __syncthreads_or(nz);
    if (threadIdx.x == 0) flag[g] = nz;
}

// grid (ceil(n / IF_THREADS), transforms): x[j][w] = acc[g][fold w] + i acc[g + 1][fold w] for transform j0 + j
__global__ void __launch_bounds__(IF_THREADS) k_isf_spec_load(const double *__restrict__ acc, long long n, int npairs, long long j0,
                                                              mdp_c64 *__restrict__ x)
{
    const long long w = (long long)blockIdx.x * IF_THREADS + threadIdx.x;
    if (w >= n) return;
    const long long H = n / 2 + 1, tpb = mdp_isf_transforms_per_bin(npairs), j = j0 + blockIdx.y;
    const long long b = j / tpb, p = 2 * (j % tpb), g = b * npairs + p, ww = mdp_msd_fold(w, n);
    mdp_c64 v;
    v.re = acc[g * H + ww];
    v.im = p + 1 < npairs ? acc[(g + 1) * H + ww] : 0.0;
    x[(long long)blockIdx.y * n + w] = v;
}

} // namespace

extern "C" {

int mdp_isf_fft(mdp_ctx *ctx, int nchan, int64_t nk, int64_t T, const double *rho, int npairs, const int32_t *pairs, int nbins,
                const int64_t *bin_off, int64_t nlags, double *out, void *stream)
{
    MDP_REQUIRE(ctx && bin_off, "mdp_isf_fft: NULL argument");
    MDP_REQUIRE(nchan >= 1 && nk >= 0 && T >= 1 && nlags >= 1 && nlags <= T && npairs >= 0 && nbins >= 0,
                "mdp_isf_fft: bad sizes (nchan %d, nk %lld, T %lld, nlags %lld, npairs %d, nbins %d)", nchan, (long long)nk,
                (long long)T, (long long)nlags, npairs, nbins);
    MDP_REQUIRE(npairs == 0 || pairs, "mdp_isf_fft: NULL pairs with npairs = %d", npairs);
    for (int q = 0; q < 2 * npairs; ++q)
        MDP_REQUIRE(pairs[q] >= 0 && pairs[q] < nchan, "mdp_isf_fft: pair %d names channel %d outside [0, %d)", q / 2,
                    (int)pairs[q], nchan);
    MDP_REQUIRE(bin_off[0] == 0 && bin_off[nbins] == nk, "mdp_isf_fft: bin_off must run from 0 to nk = %lld", (long long)nk);
    for (int b = 0; b < nbins; ++b) MDP_REQUIRE(bin_off[b + 1] >= bin_off[b], "mdp_isf_fft: bin_off decreases at bin %d", b);
    const int p = mdp_fft_log2_size(T, nlags);
    MDP_REQUIRE(p <= 30, "mdp_isf_fft: %lld steps need a transform of 2^%d points", (long long)T, p);
    if (npairs == 0 || nbins == 0) return 0;
    MDP_REQUIRE(out && (nk == 0 || rho), "mdp_isf_fft: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    MDP_CUDA(cudaSetDevice(ctx->device));
    const long long n = 1ll << p, H = n / 2 + 1;

    // the channels some pair uses (ascending), and each pair's two positions in that list
    std::vector<int> used;
    for (int q = 0; q < 2 * npairs; ++q) used.push_back(pairs[q]);
    std::sort(used.begin(), used.end());
    used.erase(std::unique(used.begin(), used.end()), used.end());
    std::vector<int> pidx((size_t)2 * npairs);
    for (int q = 0; q < 2 * npairs; ++q) pidx[(size_t)q] = (int)(std::lower_bound(used.begin(), used.end(), pairs[q]) - used.begin());
    const int nused = (int)used.size();
    const long long ngroups = (long long)npairs * nbins, tpb = mdp_isf_transforms_per_bin(npairs), U2 = nbins * tpb;

    // group accumulators and everything else that does not scale with the sub-batch; sub-batches of whole k-vectors (nused
    // transforms each, two buffers) sized to 2 GiB of scratch on the whole request (scratch_plan.h).  The inverse transforms
    // reuse the buffers, nused * (k-vectors per sub-batch) at a time
    const size_t wbytes = align256((size_t)(n / 2) * sizeof(mdp_c64));
    const size_t fixed_req = wbytes + align256((size_t)ngroups * H * 8) + align256((size_t)ngroups * 4) +
                             align256(pidx.size() * 4) + align256(used.size() * 4) + align256((size_t)(nbins + 1) * 8) + 2 * 256;
    const size_t per_unit = (size_t)nused * n * sizeof(mdp_c64), per_unit_req = 2 * per_unit;
    MDP_REQUIRE(mdp_scratch_reserved(fixed_req) <= ctx->slab_limit,
                "mdp_isf_fft: the accumulators of %d pairs x %d bins over 2^%d points (%zu B) exceed the context limit %zu B",
                npairs, nbins, p, fixed_req, ctx->slab_limit);
    const long long want = std::max<long long>(nk, ceil_div<long long>(U2, nused));
    const size_t budget = std::min<size_t>(ctx->slab_limit, (size_t)2 << 30);
    const long long batch =
        (long long)mdp_scratch_units(budget, fixed_req, per_unit_req, (size_t)std::max<long long>(1, std::min<long long>(want, 65535 / nused)));
    int rc = ctx->arena_reserve(fixed_req + (size_t)batch * per_unit_req);
    if (rc) return rc;
    ctx->arena_reset();
    mdp_c64 *W = (mdp_c64 *)ctx->arena_take((size_t)(n / 2) * sizeof(mdp_c64));
    double *acc = (double *)ctx->arena_take((size_t)ngroups * H * 8);
    int *flag = (int *)ctx->arena_take((size_t)ngroups * 4);
    int *d_pidx = (int *)ctx->arena_take(pidx.size() * 4);
    int *d_used = (int *)ctx->arena_take(used.size() * 4);
    long long *d_boff = (long long *)ctx->arena_take((size_t)(nbins + 1) * 8);
    mdp_c64 *x = (mdp_c64 *)ctx->arena_take((size_t)batch * per_unit);
    mdp_c64 *y = (mdp_c64 *)ctx->arena_take((size_t)batch * per_unit);
    if (!W || !acc || !flag || !d_pidx || !d_used || !d_boff || !x || !y) {
        mdp_set_error("internal: scratch arena exhausted (isf fft)");
        return MDP_ERR_OOM;
    }
    cudaEvent_t tk = ctx->timer_begin(9, st);
    MDP_CUDA(cudaMemcpyAsync(d_pidx, pidx.data(), pidx.size() * 4, cudaMemcpyHostToDevice, st));
    MDP_CUDA(cudaMemcpyAsync(d_used, used.data(), used.size() * 4, cudaMemcpyHostToDevice, st));
    MDP_CUDA(cudaMemcpyAsync(d_boff, bin_off, (size_t)(nbins + 1) * 8, cudaMemcpyHostToDevice, st));
    MDP_CUDA(cudaMemsetAsync(acc, 0, (size_t)ngroups * H * 8, st));
    k_isf_twiddle<<<(unsigned)ceil_div<long long>(std::max<long long>(n / 2, 1), IF_THREADS), IF_THREADS, 0, st>>>(W, n);
    MDP_LAUNCHED(ctx);

    IsfIo io{nullptr, nullptr, (const mdp_c64 *)rho, d_used, flag, out, T, nk, nlags, n, 0, 0, nused, npairs, nbins};
    int b_lo = 0;
    for (long long k0 = 0; k0 < nk; k0 += batch) {                   // forward transforms and spectrum accumulation
        const long long k1 = std::min<long long>(nk, k0 + batch);
        const int units = (int)((k1 - k0) * nused);
        io.k0 = k0;
        mdp_c64 *src = x, *dst = y;
        for (int t = 0; t < p;) {
            const int R = mdp_fft_pass_radix(t, p);
            io.x = src;
            io.y = dst;
            if (t == 0) launch_isf_pass<1>(R, io, W, t, units, st);
            else launch_isf_pass<0>(R, io, W, t, units, st);
            MDP_LAUNCHED(ctx);
            std::swap(src, dst);
            t += R;
        }
        while (bin_off[b_lo + 1] <= k0) ++b_lo;                      // first bin with a k-vector in [k0, k1)
        int b_hi = b_lo;
        while (b_hi + 1 < nbins && bin_off[b_hi + 1] < k1) ++b_hi;   // last one
        const long long g_lo = (long long)b_lo * npairs, g_hi = (long long)(b_hi + 1) * npairs;
        k_isf_spec_acc<<<dim3((unsigned)ceil_div<long long>(H, IF_THREADS), (unsigned)std::min<long long>(g_hi - g_lo, 65535)),
                         IF_THREADS, 0, st>>>(src, n, nused, d_boff, d_pidx, npairs, g_lo, g_hi, k0, k1, acc);
        MDP_LAUNCHED(ctx);
    }
    k_isf_flag<<<(unsigned)ngroups, IF_THREADS, 0, st>>>(acc, H, flag);
    MDP_LAUNCHED(ctx);
    const long long ibatch = batch * nused;
    for (long long j0 = 0; j0 < U2; j0 += ibatch) {                  // inverse transforms, two groups of a bin each
        const int nj = (int)std::min<long long>(ibatch, U2 - j0);
        k_isf_spec_load<<<dim3((unsigned)ceil_div<long long>(n, IF_THREADS), (unsigned)nj), IF_THREADS, 0, st>>>(acc, n, npairs, j0, x);
        MDP_LAUNCHED(ctx);
        io.j0 = j0;
        mdp_c64 *src = x, *dst = y;
        for (int t = 0; t < p;) {
            const int R = mdp_fft_pass_radix(t, p);
            io.x = src;
            io.y = dst;
            if (t + R == p) launch_isf_pass<2>(R, io, W, t, nj, st);
            else launch_isf_pass<0>(R, io, W, t, nj, st);
            MDP_LAUNCHED(ctx);
            std::swap(src, dst);
            t += R;
        }
    }
    ctx->timer_end(tk, st);
    return mdp_check_launch("k_isf_fft_pass");
}

} // extern "C"
