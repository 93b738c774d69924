// orient.cu -- channels of molecule-fixed unit vectors for the reorientation correlations (definition and ABI in
// include/mdprop_b200.h; per-(vector, frame) body in orient.h).
//
// Memory-bound: per vector and frame 2-3 atom positions are read (24 B each) and 8 fp64 channels written (64 B), into a
// [8][nvec][out_stride] series whose rows are time.  k_orient takes a tile of OR_TV vectors x OR_TF frames: the threads of
// a warp compute 32 consecutive vectors of one frame (their atoms lie close together in each coordinate row), the channels
// are staged in shared memory, and then every half-warp writes OR_TF consecutive columns of one row, so each store
// instruction fills whole 32-byte sectors instead of putting 8 bytes in each.
#include <algorithm>

#include "common.cuh"
#include "orient.h"

namespace {

constexpr int OR_TV = 32;                                   // vectors per tile
constexpr int OR_TF = 16;                                   // frames per tile
constexpr int OR_THREADS = 256;
constexpr int OR_PITCH = OR_TF + 1;                         // staged row pitch (doubles)
constexpr int OR_MAX_TILES_Y = 65535;

// grid (ceil(nvec / OR_TV), frame tiles of this launch); frame tile blockIdx.y covers frames f_base + blockIdx.y * OR_TF + ...
__global__ void __launch_bounds__(OR_THREADS) k_orient(const double *__restrict__ xyz, long long n, int nframes,
                                                       const double *__restrict__ cell, int kind, long long nvec,
                                                       const int *__restrict__ atoms, double *__restrict__ out,
                                                       long long out_stride, long long frame0, int f_base)
{
    __shared__ double s[MDP_ORIENT_CHANNELS * OR_TV * OR_PITCH];
    const long long v0 = (long long)blockIdx.x * OR_TV;
    const int f0 = f_base + blockIdx.y * OR_TF;
    const int lane = threadIdx.x & 31;
    const long long v = v0 + lane;
    int ia = 0, ja = 0, ka = 0;
    if (v < nvec) {
        ia = __ldg(atoms + 3 * v);
        ja = __ldg(atoms + 3 * v + 1);
        ka = kind ? __ldg(atoms + 3 * v + 2) : ia;
    }
    for (int fl = threadIdx.x >> 5; fl < OR_TF; fl += OR_THREADS / 32) {
        const int f = f0 + fl;
        if (v >= nvec || f >= nframes) continue;
        const double *x = xyz + (long long)f * 3 * n;
        double c[6], ri[3], rj[3], rk[3], ch[MDP_ORIENT_CHANNELS];
#pragma unroll
        for (int q = 0; q < 6; ++q) c[q] = __ldg(cell + 6 * f + q);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            ri[a] = __ldg(x + a * n + ia);
            rj[a] = __ldg(x + a * n + ja);
            rk[a] = __ldg(x + a * n + ka);
        }
        mdp_orient_channels(c, kind, ri, rj, rk, ch);
#pragma unroll
        for (int q = 0; q < MDP_ORIENT_CHANNELS; ++q) s[(q * OR_TV + lane) * OR_PITCH + fl] = ch[q];
    }
    __syncthreads();
    // row r = (channel, vector) of the tile; a half-warp stores its OR_TF columns
    const int col = threadIdx.x % OR_TF;
    const int f = f0 + col;
    for (int r = threadIdx.x / OR_TF; r < MDP_ORIENT_CHANNELS * OR_TV; r += OR_THREADS / OR_TF) {
        const int q = r / OR_TV, vl = r % OR_TV;
        if (v0 + vl >= nvec || f >= nframes) continue;
        out[((long long)q * nvec + v0 + vl) * out_stride + frame0 + f] = s[r * OR_PITCH + col];
    }
}

} // namespace

extern "C" {

int mdp_orient_series(mdp_ctx *ctx, int nframes, int64_t n, const double *xyz, const double *cell, int kind, int64_t nvec,
                      const int32_t *atoms, double *out, int64_t out_stride, int64_t frame0, void *stream)
{
    MDP_REQUIRE(ctx, "mdp_orient_series: NULL context");
    MDP_REQUIRE(nframes >= 0 && n >= 0 && n < (1ll << 31) && nvec >= 0, "mdp_orient_series: bad sizes (nframes %d, n %lld, nvec %lld)",
                nframes, (long long)n, (long long)nvec);
    MDP_REQUIRE(kind >= 0 && kind < MDP_ORIENT_KINDS, "mdp_orient_series: kind %d outside [0, %d)", kind, MDP_ORIENT_KINDS);
    MDP_REQUIRE(frame0 >= 0 && out_stride >= frame0 + nframes,
                "mdp_orient_series: frames [%lld, %lld) do not fit a series of out_stride %lld", (long long)frame0,
                (long long)(frame0 + nframes), (long long)out_stride);
    MDP_REQUIRE(nframes == 0 || cell, "mdp_orient_series: NULL cell");
    for (int f = 0; f < nframes; ++f) {
        const double *c = cell + 6 * (size_t)f;
        for (int i = 0; i < 3; ++i)
            MDP_REQUIRE(c[i] > 0.0 && isfinite(c[i]), "mdp_orient_series: cell length %d of frame %d is %g (must be positive)", i,
                        f, c[i]);
        for (int i = 3; i < 6; ++i) MDP_REQUIRE(isfinite(c[i]), "mdp_orient_series: tilt %d of frame %d is %g", i - 3, f, c[i]);
    }
    MDP_REQUIRE(nvec == 0 || atoms, "mdp_orient_series: NULL atoms");
    const int na = kind ? 3 : 2;
    for (int64_t v = 0; v < nvec; ++v) {
        const int32_t *a = atoms + 3 * v;
        for (int i = 0; i < na; ++i)
            MDP_REQUIRE(a[i] >= 0 && a[i] < n, "mdp_orient_series: atom %d of vector %lld is %d, outside [0, %lld)", i,
                        (long long)v, (int)a[i], (long long)n);
        MDP_REQUIRE(a[0] != a[1] && (na == 2 || (a[0] != a[2] && a[1] != a[2])),
                    "mdp_orient_series: vector %lld repeats an atom", (long long)v);
    }
    if (nframes == 0 || nvec == 0) return 0;
    MDP_REQUIRE(xyz && out, "mdp_orient_series: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    MDP_CUDA(cudaSetDevice(ctx->device));

    const size_t cbytes = (size_t)nframes * 6 * sizeof(double), abytes = (size_t)nvec * 3 * sizeof(int32_t);
    int rc = ctx->arena_reserve(align256(cbytes) + align256(abytes) + 256);
    if (rc) return rc;
    ctx->arena_reset();
    double *d_cell = (double *)ctx->arena_take(cbytes);
    int *d_atoms = (int *)ctx->arena_take(abytes);
    if (!d_cell || !d_atoms) {
        mdp_set_error("internal: scratch arena exhausted (orient series)");
        return MDP_ERR_OOM;
    }
    cudaEvent_t tk = ctx->timer_begin(11, st);
    MDP_CUDA(cudaMemcpyAsync(d_cell, cell, cbytes, cudaMemcpyHostToDevice, st));
    MDP_CUDA(cudaMemcpyAsync(d_atoms, atoms, abytes, cudaMemcpyHostToDevice, st));
    const long long ftiles = ceil_div<long long>(nframes, OR_TF);
    for (long long t0 = 0; t0 < ftiles; t0 += OR_MAX_TILES_Y) {
        const unsigned ty = (unsigned)std::min<long long>(OR_MAX_TILES_Y, ftiles - t0);
        k_orient<<<dim3((unsigned)ceil_div<long long>(nvec, OR_TV), ty), OR_THREADS, 0, st>>>(
            xyz, n, nframes, d_cell, kind, nvec, d_atoms, out, out_stride, frame0, (int)(t0 * OR_TF));
        MDP_LAUNCHED(ctx);
    }
    ctx->timer_end(tk, st);
    return mdp_check_launch("k_orient");
}

} // extern "C"
