// sk.cu -- static structure factor by the direct sum over reciprocal-lattice vectors (definition, accuracy contract and ABI in
// include/mdprop_b200.h; per-term body in sk_phase.h).
//
// rho_c(k) = sum_{j in c} exp(2 pi i n.s_j) costs N * N_k complex exponentials per frame: a dense workload bound by the
// sin/cos throughput.  One call, per sub-batch of frames (sized to the context's scratch, scratch_plan.h):
//   k_sk_sort  one CTA per frame: fractional coordinates in 32-bit fixed point (uint4 per atom, the fourth word unused so
//              that a tile row is one 16-byte shared load), placed in a stable counting sort by class, with the class
//              offsets; the main loop then walks contiguous class ranges and never branches on a class per term;
//   k_sk_rho   one CTA per (frame, block of SK_KBLOCK k-vectors), SK_KPT triplets per thread in registers; the frame's
//              atoms stream through shared memory in tiles of SK_TILE; every MDP_SK_CHUNK terms are summed in fp32 and
//              then added to fp64 class sums; rho_c(k) is written as fp64 complex at (class, k, frame) strides: to scratch
//              as [F][ncls][nk] for k_sk_bins, or straight into the caller's [ncls][nk][T] series (mdp_sk_rho);
//   k_sk_bins  one thread per (frame, class-pair row, bin): sum over the bin's contiguous k range of Re(rho_a rho_b*), in k
//              order, into sums_out.
// No atomics and a fixed summation order: run-to-run bit-identical, and a frame's result does not depend on the sub-batch it
// falls in (hence not on the scratch limit or on how frames are dealt to ranks).
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "scratch_plan.h"
#include "sk_phase.h"

namespace {

constexpr int SK_THREADS = 128;
constexpr int SK_KPT = 4;                                   // Miller triplets per thread
constexpr int SK_KBLOCK = SK_THREADS * SK_KPT;              // k-vectors per CTA
constexpr int SK_TILE = 512;                                // atoms per shared-memory tile
constexpr int SK_SORT_THREADS = 1024;
constexpr int SK_BIN_THREADS = 128;

struct SkCell {
    double c[6];
};

// block-wide exclusive scan of one int per thread (SK_SORT_THREADS threads); returns the prefix, *total the sum
__device__ int sk_block_scan(int v, int *warp_sums, int *total)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int x = v;
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) warp_sums[w] = x;
    __syncthreads();
    if (w == 0) {
        int s = warp_sums[lane];
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += y;
        }
        warp_sums[lane] = s;                                // inclusive over warps
    }
    __syncthreads();
    const int r = x - v + (w ? warp_sums[w - 1] : 0);
    *total = warp_sums[31];
    __syncthreads();                                        // warp_sums is reused by the next call
    return r;
}

// grid Fb: frame blockIdx.x of the sub-batch.  Atoms whose class lies outside [0, ncls) belong to no class and are left out.
__global__ void __launch_bounds__(SK_SORT_THREADS) k_sk_sort(const double *__restrict__ xyz, const int32_t *__restrict__ cls,
                                                             long long cls_stride, long long n, int ncls, SkCell cell,
                                                             uint4 *__restrict__ u, int *__restrict__ coff)
{
    __shared__ int warp_sums[32];
    const long long f = blockIdx.x;
    const double *x = xyz + f * 3 * n;
    const int32_t *cl = cls ? cls + f * cls_stride : nullptr;
    uint4 *uf = u + f * n;
    int *co = coff + f * (ncls + 1);
    const long long L = (n + SK_SORT_THREADS - 1) / SK_SORT_THREADS;
    const long long i0 = min(n, (long long)threadIdx.x * L), i1 = min(n, i0 + L);
    int base = 0;
    for (int c = 0; c < ncls; ++c) {
        int cnt = 0;
        for (long long i = i0; i < i1; ++i) cnt += (cl ? __ldg(cl + i) : 0) == c;
        int total;
        int pos = base + sk_block_scan(cnt, warp_sums, &total);
        if (cnt)
            for (long long i = i0; i < i1; ++i) {
                if ((cl ? __ldg(cl + i) : 0) != c) continue;
                double s[3];
                mdp_sk_frac(cell.c, __ldg(x + i), __ldg(x + n + i), __ldg(x + 2 * n + i), s);
                uf[pos++] = make_uint4(mdp_sk_fix(s[0]), mdp_sk_fix(s[1]), mdp_sk_fix(s[2]), 0u);
            }
        if (threadIdx.x == 0) co[c] = base;
        base += total;
    }
    if (threadIdx.x == 0) co[ncls] = base;
}

// where k_sk_rho writes rho_c(k) of frame f: rho[c * sc + k * sk + f * sf]
struct SkRhoOut {
    double2 *rho;
    long long sc, sk, sf;
};

// grid (ceil(nk / SK_KBLOCK), Fb)
__global__ void __launch_bounds__(SK_THREADS) k_sk_rho(const uint4 *__restrict__ u, const int *__restrict__ coff, long long n,
                                                       int ncls, const int4 *__restrict__ miller, long long nk, const SkRhoOut o)
{
    __shared__ uint4 tile[SK_TILE];
    const long long f = blockIdx.y;
    const long long k0 = (long long)blockIdx.x * SK_KBLOCK + threadIdx.x;
    int h[SK_KPT], kk[SK_KPT], l[SK_KPT];
#pragma unroll
    for (int j = 0; j < SK_KPT; ++j) {
        const long long k = k0 + (long long)j * SK_THREADS;
        const int4 m = k < nk ? __ldg(miller + k) : make_int4(0, 0, 0, 0);
        h[j] = m.x;
        kk[j] = m.y;
        l[j] = m.z;
    }
    const uint4 *uf = u + f * n;
    const int *co = coff + f * (ncls + 1);
    for (int c = 0; c < ncls; ++c) {
        const int a0 = __ldg(co + c), a1 = __ldg(co + c + 1);
        double sr[SK_KPT], si[SK_KPT];
#pragma unroll
        for (int j = 0; j < SK_KPT; ++j) sr[j] = si[j] = 0.0;
        for (int t0 = a0; t0 < a1; t0 += SK_TILE) {
            const int m = min(SK_TILE, a1 - t0);
            __syncthreads();
            for (int i = threadIdx.x; i < m; i += SK_THREADS) tile[i] = uf[t0 + i];
            __syncthreads();
            for (int j0 = 0; j0 < m; j0 += MDP_SK_CHUNK) {
                const int je = min(m, j0 + MDP_SK_CHUNK);
                float cr[SK_KPT], ci[SK_KPT];
#pragma unroll
                for (int j = 0; j < SK_KPT; ++j) cr[j] = ci[j] = 0.f;
#pragma unroll 4
                for (int a = j0; a < je; ++a) {
                    const uint4 q = tile[a];
#pragma unroll
                    for (int j = 0; j < SK_KPT; ++j) {
                        float s, cs;
                        __sincosf(mdp_sk_angle(mdp_sk_phase(h[j], kk[j], l[j], q.x, q.y, q.z)), &s, &cs);
                        cr[j] += cs;
                        ci[j] += s;
                    }
                }
#pragma unroll
                for (int j = 0; j < SK_KPT; ++j) {
                    sr[j] += (double)cr[j];
                    si[j] += (double)ci[j];
                }
            }
        }
        double2 *out = o.rho + c * o.sc + f * o.sf;
#pragma unroll
        for (int j = 0; j < SK_KPT; ++j) {
            const long long k = k0 + (long long)j * SK_THREADS;
            if (k < nk) out[k * o.sk] = make_double2(0.0 - sr[j], 0.0 - si[j]);     // exp(2 pi i p / 2^32) = -exp(2 pi i f)
        }
    }
}

// grid (ceil(rows * nbins / SK_BIN_THREADS), Fb): out[f][row(a,b)][bin] = sum_{k in bin} Re(rho_a(k) conj(rho_b(k)))
__global__ void __launch_bounds__(SK_BIN_THREADS) k_sk_bins(const double2 *__restrict__ rho, int ncls, long long nk,
                                                            const long long *__restrict__ bin_off, int nbins,
                                                            double *__restrict__ out)
{
    const int rows = ncls * (ncls + 1) / 2;
    const long long idx = (long long)blockIdx.x * SK_BIN_THREADS + threadIdx.x;
    if (idx >= (long long)rows * nbins) return;
    const long long f = blockIdx.y;
    const int row = (int)(idx / nbins), b = (int)(idx % nbins);
    int a = 0, r = row;                                      // row(a <= b) = a ncls - a (a - 1) / 2 + (b - a)
    while (r >= ncls - a) {
        r -= ncls - a;
        ++a;
    }
    const double2 *ra = rho + (f * ncls + a) * nk, *rb = rho + (f * ncls + a + r) * nk;
    double s = 0.0;
    for (long long k = bin_off[b]; k < bin_off[b + 1]; ++k) {
        const double2 x = ra[k], y = rb[k];
        s += x.x * y.x + x.y * y.y;
    }
    out[(f * rows + row) * nbins + b] = s;
}

// the checks mdp_structure_factor and mdp_sk_rho share (sizes, classes, cell, Miller bound)
int sk_check(const char *who, int nframes, int64_t n, int64_t cls_stride, int ncls, const double *cell, int64_t nk,
             const int32_t *miller)
{
    MDP_REQUIRE(nframes >= 0 && n >= 0 && n < (1ll << 31) && nk >= 0 && cls_stride >= 0,
                "%s: bad sizes (nframes %d, n %lld, nk %lld, cls_stride %lld)", who, nframes, (long long)n, (long long)nk,
                (long long)cls_stride);
    MDP_REQUIRE(ncls >= 1 && ncls <= MDP_SK_MAX_CLASSES, "%s: ncls %d outside [1, %d]", who, ncls, MDP_SK_MAX_CLASSES);
    for (int i = 0; i < 3; ++i)
        MDP_REQUIRE(cell[i] > 0.0 && isfinite(cell[i]), "%s: cell length %d is %g (must be positive)", who, i, cell[i]);
    for (int i = 3; i < 6; ++i) MDP_REQUIRE(isfinite(cell[i]), "%s: tilt %d is %g", who, i - 3, cell[i]);
    MDP_REQUIRE(nk == 0 || miller, "%s: NULL miller with nk = %lld", who, (long long)nk);
    for (int64_t k = 0; k < 3 * nk; ++k)
        MDP_REQUIRE(miller[k] >= -MDP_SK_NLIM && miller[k] <= MDP_SK_NLIM,
                    "%s: Miller component %d of vector %lld is beyond the accuracy bound %d", who, (int)miller[k],
                    (long long)(k / 3), MDP_SK_NLIM);
    return 0;
}

// Miller triplets padded to int4 (one 16-byte load per k-vector)
std::vector<int> sk_miller4(int64_t nk, const int32_t *miller)
{
    std::vector<int> m4((size_t)4 * nk, 0);
    for (int64_t k = 0; k < nk; ++k)
        for (int i = 0; i < 3; ++i) m4[(size_t)4 * k + i] = miller[3 * k + i];
    return m4;
}

} // namespace

extern "C" {

int mdp_structure_factor(mdp_ctx *ctx, int nframes, int64_t n, const double *xyz, const int32_t *cls, int64_t cls_stride,
                         int ncls, const double *cell, int64_t nk, const int32_t *miller, int nbins, const int64_t *bin_off,
                         double *sums_out, void *stream)
{
    MDP_REQUIRE(ctx && cell && bin_off, "mdp_structure_factor: NULL argument");
    MDP_REQUIRE(nbins >= 0, "mdp_structure_factor: bad sizes (nbins %d)", nbins);
    if (int rc = sk_check("mdp_structure_factor", nframes, n, cls_stride, ncls, cell, nk, miller)) return rc;
    MDP_REQUIRE(bin_off[0] == 0 && bin_off[nbins] == nk, "mdp_structure_factor: bin_off must run from 0 to nk = %lld",
                (long long)nk);
    for (int b = 0; b < nbins; ++b)
        MDP_REQUIRE(bin_off[b + 1] >= bin_off[b], "mdp_structure_factor: bin_off decreases at bin %d", b);
    const int rows = ncls * (ncls + 1) / 2;
    if (nframes == 0 || nbins == 0) return 0;
    MDP_REQUIRE(sums_out && (n == 0 || xyz), "mdp_structure_factor: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    MDP_CUDA(cudaSetDevice(ctx->device));

    // the k-set and the bin table are shared by every frame of the call; per frame the fixed-point atoms, the class offsets
    // and rho.  Sub-batches of frames sized to 2 GiB of scratch on the whole request (scratch_plan.h)
    const std::vector<int> m4 = sk_miller4(nk, miller);
    const size_t mbytes = (size_t)nk * sizeof(int4), bbytes = (size_t)(nbins + 1) * 8;
    const size_t fixed_req = align256(mbytes) + align256(bbytes) + 3 * 256;
    const size_t per_frame = (size_t)n * sizeof(uint4) + (size_t)(ncls + 1) * sizeof(int) + (size_t)ncls * nk * sizeof(double2);
    const size_t budget = std::min<size_t>(ctx->slab_limit, (size_t)2 << 30);
    const int batch = (int)mdp_scratch_units(budget, fixed_req, per_frame, (size_t)std::min(nframes, 65535));
    int rc = ctx->arena_reserve(fixed_req + (size_t)batch * per_frame);
    if (rc) return rc;
    ctx->arena_reset();
    int4 *d_miller = (int4 *)ctx->arena_take(mbytes);
    long long *d_boff = (long long *)ctx->arena_take(bbytes);
    uint4 *u = (uint4 *)ctx->arena_take((size_t)batch * n * sizeof(uint4));
    int *coff = (int *)ctx->arena_take((size_t)batch * (ncls + 1) * sizeof(int));
    double2 *rho = (double2 *)ctx->arena_take((size_t)batch * ncls * nk * sizeof(double2));
    if (!d_miller || !d_boff || !u || !coff || !rho) {
        mdp_set_error("internal: scratch arena exhausted (structure factor)");
        return MDP_ERR_OOM;
    }
    cudaEvent_t tk = ctx->timer_begin(8, st);
    if (nk > 0) MDP_CUDA(cudaMemcpyAsync(d_miller, m4.data(), mbytes, cudaMemcpyHostToDevice, st));
    MDP_CUDA(cudaMemcpyAsync(d_boff, bin_off, bbytes, cudaMemcpyHostToDevice, st));
    SkCell c;
    for (int i = 0; i < 6; ++i) c.c[i] = cell[i];
    const SkRhoOut ro{rho, nk, 1, (long long)ncls * nk};
    for (int f0 = 0; f0 < nframes; f0 += batch) {
        const int fb = std::min(batch, nframes - f0);
        k_sk_sort<<<(unsigned)fb, SK_SORT_THREADS, 0, st>>>(xyz + (size_t)f0 * 3 * n, cls ? cls + (size_t)f0 * cls_stride : nullptr,
                                                            cls_stride, n, ncls, c, u, coff);
        MDP_LAUNCHED(ctx);
        if (nk > 0) {
            k_sk_rho<<<dim3((unsigned)ceil_div<long long>(nk, SK_KBLOCK), (unsigned)fb), SK_THREADS, 0, st>>>(u, coff, n, ncls, d_miller,
                                                                                                          nk, ro);
            MDP_LAUNCHED(ctx);
        }
        k_sk_bins<<<dim3((unsigned)ceil_div<long long>((long long)rows * nbins, SK_BIN_THREADS), (unsigned)fb), SK_BIN_THREADS, 0,
                    st>>>(rho, ncls, nk, d_boff, nbins, sums_out + (size_t)f0 * rows * nbins);
        MDP_LAUNCHED(ctx);
    }
    ctx->timer_end(tk, st);
    return mdp_check_launch("k_sk_rho");
}

int mdp_sk_rho(mdp_ctx *ctx, int nframes, int64_t n, const double *xyz, const int32_t *cls, int64_t cls_stride, int ncls,
               const double *cell, int64_t nk, const int32_t *miller, double *rho_out, int64_t out_stride, int64_t frame0,
               void *stream)
{
    MDP_REQUIRE(ctx && cell, "mdp_sk_rho: NULL argument");
    if (int rc = sk_check("mdp_sk_rho", nframes, n, cls_stride, ncls, cell, nk, miller)) return rc;
    MDP_REQUIRE(frame0 >= 0 && out_stride >= frame0 + nframes,
                "mdp_sk_rho: frames [%lld, %lld) do not fit a series of out_stride %lld", (long long)frame0,
                (long long)(frame0 + nframes), (long long)out_stride);
    if (nframes == 0 || nk == 0) return 0;
    MDP_REQUIRE(rho_out && (n == 0 || xyz), "mdp_sk_rho: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    MDP_CUDA(cudaSetDevice(ctx->device));

    // as mdp_structure_factor without the rho scratch: k_sk_rho writes the caller's series directly
    const std::vector<int> m4 = sk_miller4(nk, miller);
    const size_t mbytes = (size_t)nk * sizeof(int4);
    const size_t fixed_req = align256(mbytes) + 2 * 256;
    const size_t per_frame = (size_t)n * sizeof(uint4) + (size_t)(ncls + 1) * sizeof(int);
    const size_t budget = std::min<size_t>(ctx->slab_limit, (size_t)2 << 30);
    const int batch = (int)mdp_scratch_units(budget, fixed_req, per_frame, (size_t)std::min(nframes, 65535));
    int rc = ctx->arena_reserve(fixed_req + (size_t)batch * per_frame);
    if (rc) return rc;
    ctx->arena_reset();
    int4 *d_miller = (int4 *)ctx->arena_take(mbytes);
    uint4 *u = (uint4 *)ctx->arena_take((size_t)batch * n * sizeof(uint4));
    int *coff = (int *)ctx->arena_take((size_t)batch * (ncls + 1) * sizeof(int));
    if (!d_miller || !u || !coff) {
        mdp_set_error("internal: scratch arena exhausted (sk rho)");
        return MDP_ERR_OOM;
    }
    cudaEvent_t tk = ctx->timer_begin(8, st);
    MDP_CUDA(cudaMemcpyAsync(d_miller, m4.data(), mbytes, cudaMemcpyHostToDevice, st));
    SkCell c;
    for (int i = 0; i < 6; ++i) c.c[i] = cell[i];
    for (int f0 = 0; f0 < nframes; f0 += batch) {
        const int fb = std::min(batch, nframes - f0);
        k_sk_sort<<<(unsigned)fb, SK_SORT_THREADS, 0, st>>>(xyz + (size_t)f0 * 3 * n, cls ? cls + (size_t)f0 * cls_stride : nullptr,
                                                            cls_stride, n, ncls, c, u, coff);
        MDP_LAUNCHED(ctx);
        const SkRhoOut ro{(double2 *)rho_out + frame0 + f0, (long long)nk * out_stride, out_stride, 1};
        k_sk_rho<<<dim3((unsigned)ceil_div<long long>(nk, SK_KBLOCK), (unsigned)fb), SK_THREADS, 0, st>>>(u, coff, n, ncls, d_miller,
                                                                                                      nk, ro);
        MDP_LAUNCHED(ctx);
    }
    ctx->timer_end(tk, st);
    return mdp_check_launch("k_sk_rho");
}

} // extern "C"
