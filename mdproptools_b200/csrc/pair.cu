// pair.cu -- minimum-image pair-distance engine for sm_100a.
//
// Replaces the numba loops of mdproptools/structural/rdf_cn.py:35-162 (_calc_rsq, _remove_outliers,
// _rdf_loop, _cn_loop, _rdf_mol_loop, _cn_mol_loop) and the cutoff searches that call _calc_rsq
// (cluster_analysis.py:150-161, hydration_number.py:16-19, residence_time.py:100-104).
//
// Design (B200-first, not a translation of the row-by-row reference loop):
//   1. per frame the point set is binned on a grid of cells ordered along a Hilbert curve by a counting sort and written out
//      group-blocked (32 points = one contiguous 1 KB block of double2: 32 x (x, y), then 32 x (z, class|index)), padded to
//      256-point tiles; every 32-point group gets a float box rounded outward, every tile an fp64 box;
//   2. tile pairs whose boxes cannot contain a pair inside the cutoff (under the REFERENCE's single-shift minimum image,
//      evaluated with interval arithmetic that is monotone w.r.t. the fp64 operation order) are dropped when the work list
//      is built, per tile row.  The set of pairs with rsq < rcut2 is unchanged by any culling level;
//   3. persistent CTAs walk the frames of the batch (each starts at a different frame); inside a frame every WARP pulls
//      units -- one 32-point i group (one point per lane) against the whole tile row of its tile -- from the frame's
//      counter, so there is no CTA barrier on the pair path.  Chunk level: 32 lanes test 32 j-chunk boxes at a time (fp32,
//      directed rounding) and classify the image per axis; point level: the points of a needed chunk are filtered against
//      the i group's box; the survivors queue up in a per-warp ring and are evaluated 32 at a time;
//   4. TWO pair kernels share all of that:
//        k_pair_fast (pair_fast.cuh, the default for uniform bins): distances and bins in fp32 relative to the group
//          centre, every pair within a proven error bound of a bin edge re-evaluated in the reference's fp64 arithmetic
//          and corrected -- counts identical to the reference's, 1.6x faster than the all-fp64 kernel;
//        k_pair (this file): the reference's unfused fp64 chain for every evaluated pair (8-14 FP64-pipe ops); the hits
//          are compacted into a per-warp queue and binned from there (uniform bins: fp32 estimate + one exact fp64 edge
//          pair).  It serves table bins (coordination numbers), the neighbour list (clusters, hydration, residence
//          searches), MDP_PAIR_F64, MDP_PAIR_NO_CULL and every shape the fast kernel declines.
//      The per-CTA uint32 histogram is flushed to the per-frame uint64 global histogram when the CTA leaves a frame (the
//      only barrier) and whenever the CTA has evaluated 2^30 pairs since the last flush (overflow guard).
#include <float.h>
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "scratch_plan.h"

namespace {

constexpr int TS = 256;        // points per tile
constexpr int GS = 32;         // points per group (one warp's i points / one j chunk)
constexpr int GPT = TS / GS;   // groups per tile
constexpr int NWARP = 8;       // warps per CTA of the pair kernel
constexpr int QCAP = 160;      // queue entries per warp (32 carried + 4 steps x 32)
constexpr int MAX_CLS = 64;
constexpr int CTAS_PER_SM = 2;   // resident CTAs of the pair kernel per SM (register budget 65536 / (CTAS_PER_SM * 256))

// Sorted points are stored group-blocked: group g (32 points) occupies 64 consecutive double2,
//   [g*64 + l]      = (x, y)  of point l
//   [g*64 + 32 + l] = (z, meta), meta = the bit pattern {lo: class, hi: row in the caller's order or -1 for padding}
// so that one 32-point chunk is a single contiguous 1 KB block and both halves are bank-conflict free.
constexpr int GREC = 64;       // double2 per group
constexpr int RING = 64;       // candidate ring of the pair kernel: entries per warp
__host__ __device__ __forceinline__ int64_t rec_xy(int64_t pos) { return (pos >> 5) * GREC + (pos & 31); }
__host__ __device__ __forceinline__ int64_t rec_zw(int64_t pos) { return (pos >> 5) * GREC + 32 + (pos & 31); }
constexpr size_t REC_BYTES = 32;   // bytes per point

enum { MODE_HIST_UNIFORM = 0, MODE_HIST_TABLE = 1, MODE_LIST = 2 };
// the flag bits mdp_pair_hist and mdp_pair_list accept (include/mdprop_b200.h)
constexpr int PAIR_FLAGS = MDP_PAIR_NO_CULL | MDP_PAIR_NO_SORT | MDP_PAIR_TRICLINIC | MDP_PAIR_F64;

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_min(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__device__ __forceinline__ uint32_t spread3(uint32_t v)
{
    // spread the low 10 bits of v so that there are two zero bits between each
    v &= 0x3ffu;
    v = (v | (v << 16)) & 0x030000ffu;
    v = (v | (v << 8)) & 0x0300f00fu;
    v = (v | (v << 4)) & 0x030c30c3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}

// Lower bound of |f(d)| over d in [dlo, dhi], f = the reference's single-shift minimum image
// (rdf_cn.py:50-55): f(d) = d - l if d > h, d + l if d < -h, else d  (h = l/2).  Because fp64
// subtraction/addition are monotone, evaluating the pieces at the interval end points with the same
// operations the pair loop uses gives a bound that no pair of the two boxes can undercut.
// general <- true when some d of the interval needs a shift.
__device__ __forceinline__ double axis_lower_bound(double alo, double ahi, double blo, double bhi, double l, double h,
                                                   bool &general)
{
    const double dlo = __dsub_rn(alo, bhi), dhi = __dsub_rn(ahi, blo);
    double best = DBL_MAX;
    {
        const double lo = fmax(dlo, -h), hi = fmin(dhi, h);
        if (lo <= hi) best = (lo <= 0.0 && hi >= 0.0) ? 0.0 : fmin(fabs(lo), fabs(hi));
    }
    if (dhi > h) {
        general = true;
        const double lo = __dsub_rn(fmax(dlo, h), l), hi = __dsub_rn(dhi, l);
        best = fmin(best, (lo <= 0.0 && hi >= 0.0) ? 0.0 : fmin(fabs(lo), fabs(hi)));
    }
    if (dlo < -h) {
        general = true;
        const double lo = __dadd_rn(dlo, l), hi = __dadd_rn(fmin(dhi, -h), l);
        best = fmin(best, (lo <= 0.0 && hi >= 0.0) ? 0.0 : fmin(fabs(lo), fabs(hi)));
    }
    return best;
}

// box-pair test: returns true when some pair of the two boxes may have rsq < rcut2
__device__ __forceinline__ bool boxes_may_interact(const double *a, const double *b, double lx, double ly, double lz,
                                                   double rcut2, bool &general)
{
    if (a[0] > a[3] || b[0] > b[3]) return false;   // empty box (padding only)
    general = false;
    const double bx = axis_lower_bound(a[0], a[3], b[0], b[3], lx, lx * 0.5, general);
    const double by = axis_lower_bound(a[1], a[4], b[1], b[4], ly, ly * 0.5, general);
    const double bz = axis_lower_bound(a[2], a[5], b[2], b[5], lz, lz * 0.5, general);
    const double lb = __dadd_rn(__dadd_rn(__dmul_rn(bx, bx), __dmul_rn(by, by)), __dmul_rn(bz, bz));
    return lb < rcut2;
}

// ---- chunk-level test in fp32 with directed rounding ------------------------------------------------
// Group boxes are also kept as floats rounded OUTWARD (lo down, hi up), box lengths as (down, up) pairs.
// Every bound below is rounded towards "keep the pair", so the test can only err on the side of evaluating
// a chunk pair that has no hit; the per-axis classification is exact in the same sense:
//   AX_NONE   every pair of the two boxes has |d| <= l/2           -> no minimum-image work
//   AX_SHIFT  every pair has |d| > l/2                              -> d' = |d| - l for all of them
//   AX_MIXED  undecided                                            -> d' = min(|d|, ||d| - l|), which has the
//             same magnitude as the reference's strict single shift (rdf_cn.py:50-55) for every d
enum { AX_NONE = 0, AX_SHIFT = 1, AX_MIXED = 2 };

struct AxisF {
    float l_dn, l_up, h_dn, h_up;
};

__device__ __forceinline__ AxisF make_axis(double l)
{
    AxisF a;
    a.l_dn = __double2float_rd(l);
    a.l_up = __double2float_ru(l);
    const double h = l * 0.5;
    a.h_dn = __double2float_rd(h);
    a.h_up = __double2float_ru(h);
    return a;
}

__device__ __forceinline__ float interval_min_abs(float lo, float hi)
{
    return (lo <= 0.f && hi >= 0.f) ? 0.f : fminf(fabsf(lo), fabsf(hi));
}

// lower bound of the wrapped |d| over the two intervals + the class of the axis
__device__ __forceinline__ float axis_test_f32(float alo, float ahi, float blo, float bhi, const AxisF &ax, int &cls)
{
    const float dlo = __fsub_rd(alo, bhi), dhi = __fsub_ru(ahi, blo);
    const bool may_plus = dhi > ax.h_dn, may_minus = dlo < -ax.h_dn;
    float best = 3.0e38f;
    if (dlo > ax.h_up) {
        cls = AX_SHIFT;
        best = interval_min_abs(__fsub_rd(dlo, ax.l_up), __fsub_ru(dhi, ax.l_dn));
    } else if (dhi < -ax.h_up) {
        cls = AX_SHIFT;
        best = interval_min_abs(__fadd_rd(dlo, ax.l_dn), __fadd_ru(dhi, ax.l_up));
    } else {
        cls = (may_plus || may_minus) ? AX_MIXED : AX_NONE;
        {
            const float lo = fmaxf(dlo, -ax.h_up), hi = fminf(dhi, ax.h_up);
            if (lo <= hi) best = interval_min_abs(lo, hi);
        }
        if (may_plus) best = fminf(best, interval_min_abs(__fsub_rd(fmaxf(dlo, ax.h_dn), ax.l_up), __fsub_ru(dhi, ax.l_dn)));
        if (may_minus) best = fminf(best, interval_min_abs(__fadd_rd(dlo, ax.l_dn), __fadd_ru(fminf(dhi, -ax.h_dn), ax.l_up)));
    }
    return best;
}

// a, b: float[6] outward-rounded boxes.  Returns need; code = cls_x | cls_y << 2 | cls_z << 4
__device__ __forceinline__ bool chunk_test_f32(const float *a, const float *b, const AxisF &X, const AxisF &Y, const AxisF &Z,
                                               float rcut2_up, int &code)
{
    code = 0;
    if (a[0] > a[3] || b[0] > b[3]) return false;   // empty box (padding only)
    int cx, cy, cz;
    const float bx = axis_test_f32(a[0], a[3], b[0], b[3], X, cx);
    const float by = axis_test_f32(a[1], a[4], b[1], b[4], Y, cy);
    const float bz = axis_test_f32(a[2], a[5], b[2], b[5], Z, cz);
    code = cx | (cy << 2) | (cz << 4);
    const float lb = __fadd_rd(__fadd_rd(__fmul_rd(bx, bx), __fmul_rd(by, by)), __fmul_rd(bz, bz));
    return lb < rcut2_up;
}

// ---- general triclinic cells (MDP_PAIR_TRICLINIC) -----------------------------------------------------
// Image convention (an extension -- the reference has no triclinic image; defined by oracle/oracle.c
// pair_rsq_tri): sequential single shifts in the order z, y, x for the restricted triclinic cell a=(lx,0,0),
// b=(xy,ly,0), c=(xz,yz,lz):  kz from dz; dy -= kz*yz, dx -= kz*xz;  ky from dy; dx -= ky*xy;  kx from dx.
// The box tests enumerate the image vectors (kz, ky, kx) that some pair of the two boxes can take, with
// every operation rounded outward, so (i) the lower bound on rsq can only be too small and (ii) a box pair
// is called uniform only when a single image vector is possible for every pair in it.
struct DirF64 {
    typedef double T;
    static __device__ __forceinline__ T sub_dn(T a, T b) { return __dsub_rd(a, b); }
    static __device__ __forceinline__ T sub_up(T a, T b) { return __dsub_ru(a, b); }
    static __device__ __forceinline__ T add_dn(T a, T b) { return __dadd_rd(a, b); }
    static __device__ __forceinline__ T add_up(T a, T b) { return __dadd_ru(a, b); }
    static __device__ __forceinline__ T mul_dn(T a, T b) { return __dmul_rd(a, b); }
    static __device__ __forceinline__ T dn(double v) { return v; }
    static __device__ __forceinline__ T up(double v) { return v; }
    static __device__ __forceinline__ T big() { return DBL_MAX; }
};
struct DirF32 {
    typedef float T;
    static __device__ __forceinline__ T sub_dn(T a, T b) { return __fsub_rd(a, b); }
    static __device__ __forceinline__ T sub_up(T a, T b) { return __fsub_ru(a, b); }
    static __device__ __forceinline__ T add_dn(T a, T b) { return __fadd_rd(a, b); }
    static __device__ __forceinline__ T add_up(T a, T b) { return __fadd_ru(a, b); }
    static __device__ __forceinline__ T mul_dn(T a, T b) { return __fmul_rd(a, b); }
    static __device__ __forceinline__ T dn(double v) { return __double2float_rd(v); }
    static __device__ __forceinline__ T up(double v) { return __double2float_ru(v); }
    static __device__ __forceinline__ T big() { return 3.0e38f; }
};

template <class D>
struct TriConst {
    typename D::T l_dn[3], l_up[3], h_dn[3], h_up[3];   // x, y, z lengths and half lengths
    typename D::T c_dn[3], c_up[3];                     // xy, xz, yz
    __device__ __forceinline__ void set(const double *cell)
    {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            l_dn[a] = D::dn(cell[a]);
            l_up[a] = D::up(cell[a]);
            h_dn[a] = D::dn(cell[a] * 0.5);
            h_up[a] = D::up(cell[a] * 0.5);
            c_dn[a] = D::dn(cell[3 + a]);
            c_up[a] = D::up(cell[3 + a]);
        }
    }
};

template <class T>
__device__ __forceinline__ T iv_min_abs(T lo, T hi)
{
    return (lo <= (T)0 && hi >= (T)0) ? (T)0 : (fabs(lo) < fabs(hi) ? fabs(lo) : fabs(hi));
}

// part of [lo, hi] whose image index is k, after the shift by k*l: [ol, oh]; false when no d of the interval has index k
template <class D>
__device__ __forceinline__ bool tri_region(typename D::T lo, typename D::T hi, int k, typename D::T l_dn, typename D::T l_up,
                                           typename D::T h_dn, typename D::T h_up, typename D::T &ol, typename D::T &oh)
{
    typedef typename D::T T;
    if (k == 0) {
        if (lo > h_up || hi < -h_up) return false;
        ol = lo > -h_up ? lo : -h_up;
        oh = hi < h_up ? hi : h_up;
        return true;
    }
    if (k > 0) {
        if (!(hi > h_dn)) return false;
        const T c = lo > h_dn ? lo : h_dn;
        ol = D::sub_dn(c, l_up);
        oh = D::sub_up(hi, l_dn);
        return true;
    }
    if (!(lo < -h_dn)) return false;
    const T c = hi < -h_dn ? hi : -h_dn;
    ol = D::add_dn(lo, l_dn);
    oh = D::add_up(c, l_up);
    return true;
}

// [lo, hi] -= k * c, c in [c_dn, c_up]
template <class D>
__device__ __forceinline__ void tri_shift(typename D::T &lo, typename D::T &hi, int k, typename D::T c_dn, typename D::T c_up)
{
    if (k > 0) {
        lo = D::sub_dn(lo, c_up);
        hi = D::sub_up(hi, c_dn);
    } else if (k < 0) {
        lo = D::add_dn(lo, c_dn);
        hi = D::add_up(hi, c_up);
    }
}

constexpr int TRI_MIXED = 0x3f;
__device__ __forceinline__ int tri_enc(int k) { return k == 0 ? 0 : (k > 0 ? 1 : 2); }
__device__ __forceinline__ double tri_dec(int c2, double v) { return c2 == 0 ? 0.0 : (c2 == 1 ? v : -v); }

// a, b: boxes {lo[3], hi[3]} (supersets of the points).  Returns true when some pair may have rsq < rcut2_up;
// code = enc(kx) | enc(ky) << 2 | enc(kz) << 4 when one image vector serves every pair, TRI_MIXED otherwise.
template <class D>
__device__ __forceinline__ bool tri_box_test(const typename D::T *a, const typename D::T *b, const TriConst<D> &C,
                                             typename D::T rcut2_up, int &code)
{
    typedef typename D::T T;
    code = 0;
    if (a[0] > a[3] || b[0] > b[3]) return false;   // empty box (padding only)
    const T x0lo = D::sub_dn(a[0], b[3]), x0hi = D::sub_up(a[3], b[0]);
    const T y0lo = D::sub_dn(a[1], b[4]), y0hi = D::sub_up(a[4], b[1]);
    const T z0lo = D::sub_dn(a[2], b[5]), z0hi = D::sub_up(a[5], b[2]);
    T best = D::big();
    int nfeas = 0;
#pragma unroll 1
    for (int kz = 1; kz >= -1; --kz) {
        T zl, zh;
        if (!tri_region<D>(z0lo, z0hi, kz, C.l_dn[2], C.l_up[2], C.h_dn[2], C.h_up[2], zl, zh)) continue;
        const T bz = iv_min_abs(zl, zh);
        const T bz2 = D::mul_dn(bz, bz);
        T y1lo = y0lo, y1hi = y0hi, x1lo = x0lo, x1hi = x0hi;
        tri_shift<D>(y1lo, y1hi, kz, C.c_dn[2], C.c_up[2]);   // yz
        tri_shift<D>(x1lo, x1hi, kz, C.c_dn[1], C.c_up[1]);   // xz
#pragma unroll 1
        for (int ky = 1; ky >= -1; --ky) {
            T yl, yh;
            if (!tri_region<D>(y1lo, y1hi, ky, C.l_dn[1], C.l_up[1], C.h_dn[1], C.h_up[1], yl, yh)) continue;
            const T by = iv_min_abs(yl, yh);
            const T byz2 = D::add_dn(D::mul_dn(by, by), bz2);
            T x2lo = x1lo, x2hi = x1hi;
            tri_shift<D>(x2lo, x2hi, ky, C.c_dn[0], C.c_up[0]);   // xy
#pragma unroll 1
            for (int kx = 1; kx >= -1; --kx) {
                T xl, xh;
                if (!tri_region<D>(x2lo, x2hi, kx, C.l_dn[0], C.l_up[0], C.h_dn[0], C.h_up[0], xl, xh)) continue;
                const T bx = iv_min_abs(xl, xh);
                const T lb = D::add_dn(D::mul_dn(bx, bx), byz2);
                best = lb < best ? lb : best;
                ++nfeas;
                code = tri_enc(kx) | (tri_enc(ky) << 2) | (tri_enc(kz) << 4);
            }
        }
    }
    if (nfeas != 1) code = TRI_MIXED;
    return best < rcut2_up;
}

// ---- point-level test ----------------------------------------------------------------------------------
// One j point against the box of an i group, for a chunk pair whose image class (code) is already known from
// the box-box test.  Same rounding discipline as chunk_test_f32: every bound errs towards "keep".
// code == 0 (no axis needs the minimum image for any pair of the two boxes) is the common, cheap case.
__device__ __forceinline__ bool point_test_f32(const float *a, double x, double y, double z, const AxisF &X, const AxisF &Y,
                                               const AxisF &Z, float rcut2_up, int code)
{
    const float xd = __double2float_rd(x), xu = __double2float_ru(x);
    const float yd = __double2float_rd(y), yu = __double2float_ru(y);
    const float zd = __double2float_rd(z), zu = __double2float_ru(z);
    float bx, by, bz;
    if (code == 0) {
        bx = fmaxf(fmaxf(__fsub_rd(a[0], xu), __fsub_rd(xd, a[3])), 0.f);
        by = fmaxf(fmaxf(__fsub_rd(a[1], yu), __fsub_rd(yd, a[4])), 0.f);
        bz = fmaxf(fmaxf(__fsub_rd(a[2], zu), __fsub_rd(zd, a[5])), 0.f);
    } else {
        int cls;
        bx = axis_test_f32(a[0], a[3], xd, xu, X, cls);
        by = axis_test_f32(a[1], a[4], yd, yu, Y, cls);
        bz = axis_test_f32(a[2], a[5], zd, zu, Z, cls);
    }
    const float lb = __fadd_rd(__fadd_rd(__fmul_rd(bx, bx), __fmul_rd(by, by)), __fmul_rd(bz, bz));
    return lb < rcut2_up;
}

// triclinic, single image vector (kx, ky, kz) for every pair of the chunk pair (code != TRI_MIXED)
__device__ __forceinline__ bool tri_point_test_f32(const float *a, double x, double y, double z, const double *cell,
                                                   float rcut2_up, int code)
{
    typedef DirF32 D;
    float xl = __fsub_rd(a[0], __double2float_ru(x)), xh = __fsub_ru(a[3], __double2float_rd(x));
    float yl = __fsub_rd(a[1], __double2float_ru(y)), yh = __fsub_ru(a[4], __double2float_rd(y));
    float zl = __fsub_rd(a[2], __double2float_ru(z)), zh = __fsub_ru(a[5], __double2float_rd(z));
    if (code != 0) {
        const int ex = code & 3, ey = (code >> 2) & 3, ez = (code >> 4) & 3;
        const int kx = ex == 0 ? 0 : (ex == 1 ? 1 : -1), ky = ey == 0 ? 0 : (ey == 1 ? 1 : -1), kz = ez == 0 ? 0 : (ez == 1 ? 1 : -1);
        if (kz) {
            tri_shift<D>(zl, zh, kz, D::dn(cell[2]), D::up(cell[2]));
            tri_shift<D>(yl, yh, kz, D::dn(cell[5]), D::up(cell[5]));   // yz
            tri_shift<D>(xl, xh, kz, D::dn(cell[4]), D::up(cell[4]));   // xz
        }
        if (ky) {
            tri_shift<D>(yl, yh, ky, D::dn(cell[1]), D::up(cell[1]));
            tri_shift<D>(xl, xh, ky, D::dn(cell[3]), D::up(cell[3]));   // xy
        }
        if (kx) tri_shift<D>(xl, xh, kx, D::dn(cell[0]), D::up(cell[0]));
    }
    const float bx = iv_min_abs(xl, xh), by = iv_min_abs(yl, yh), bz = iv_min_abs(zl, zh);
    const float lb = __fadd_rd(__fadd_rd(__fmul_rd(bx, bx), __fmul_rd(by, by)), __fmul_rd(bz, bz));
    return lb < rcut2_up;
}

// ---------------------------------------------------------------------------------------------
// preparation kernels
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_minmax(const double *__restrict__ xyz, int64_t n, double *__restrict__ mm)
{
    const int f = blockIdx.x;
    const double *p = xyz + (int64_t)f * 3 * n;
    double lo[3] = {DBL_MAX, DBL_MAX, DBL_MAX}, hi[3] = {-DBL_MAX, -DBL_MAX, -DBL_MAX};
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double v = p[c * n + i];
            lo[c] = fmin(lo[c], v);
            hi[c] = fmax(hi[c], v);
        }
    }
    __shared__ double s[32][6];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        lo[c] = warp_min(lo[c]);
        hi[c] = warp_max(hi[c]);
    }
    if (lane == 0) {
        for (int c = 0; c < 3; ++c) {
            s[w][c] = lo[c];
            s[w][3 + c] = hi[c];
        }
    }
    __syncthreads();
    if (w == 0) {
        const int nw = blockDim.x >> 5;
        for (int c = 0; c < 3; ++c) {
            double a = lane < nw ? s[lane][c] : DBL_MAX, b = lane < nw ? s[lane][3 + c] : -DBL_MAX;
            a = warp_min(a);
            b = warp_max(b);
            if (lane == 0) {
                mm[f * 6 + c] = a;
                mm[f * 6 + 3 + c] = b;
            }
        }
    }
}

__global__ void __launch_bounds__(256) k_cell_count(const double *__restrict__ xyz, int64_t n, const double *__restrict__ mm,
                                                    int bits, uint32_t *__restrict__ code, uint32_t *__restrict__ rank,
                                                    uint32_t *__restrict__ cnt)
{
    const int f = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (bits == 0) {   // MDP_PAIR_NO_SORT (or a tiny set): keep the caller's order, single cell
        code[(int64_t)f * n + i] = 0u;
        rank[(int64_t)f * n + i] = (uint32_t)i;
        return;
    }
    uint32_t c = 0;
    {
        const double *p = xyz + (int64_t)f * 3 * n;
        const int nc = 1 << bits;
        uint32_t q[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const double lo = mm[f * 6 + a], hi = mm[f * 6 + 3 + a];
            const double ext = hi - lo;
            int v = ext > 0.0 ? (int)((p[a * n + i] - lo) / ext * (double)nc) : 0;
            v = v < 0 ? 0 : (v >= nc ? nc - 1 : v);
            q[a] = (uint32_t)v;
        }
        // Hilbert index of the cell (Skilling's transpose algorithm): consecutive indices are face-adjacent
        // cells, so 32 consecutive points form a compact blob; a Morton order jumps across the box at every
        // octant boundary, which gave 6 % of the groups boxes that interact with everything.
        {
            const uint32_t M = 1u << (bits - 1);
            for (uint32_t Q = M; Q > 1u; Q >>= 1) {
                const uint32_t P = Q - 1u;
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    if (q[a] & Q) {
                        q[0] ^= P;
                    } else {
                        const uint32_t t = (q[0] ^ q[a]) & P;
                        q[0] ^= t;
                        q[a] ^= t;
                    }
                }
            }
            q[1] ^= q[0];
            q[2] ^= q[1];
            uint32_t t = 0;
            for (uint32_t Q = M; Q > 1u; Q >>= 1)
                if (q[2] & Q) t ^= Q - 1u;
            q[0] ^= t;
            q[1] ^= t;
            q[2] ^= t;
        }
        c = (spread3(q[0]) << 2) | (spread3(q[1]) << 1) | spread3(q[2]);
    }
    const int64_t ncode = (int64_t)1 << (3 * bits);
    code[(int64_t)f * n + i] = c;
    rank[(int64_t)f * n + i] = atomicAdd(&cnt[(int64_t)f * ncode + c], 1u);
}

// exclusive scan of ncode counters per frame, in place (one CTA per frame)
__global__ void __launch_bounds__(1024) k_cell_scan(uint32_t *__restrict__ cnt, int64_t ncode)
{
    uint32_t *c = cnt + (int64_t)blockIdx.x * ncode;
    const int t = threadIdx.x, nt = blockDim.x;
    const int64_t per = (ncode + nt - 1) / nt;
    const int64_t b = (int64_t)t * per, e = b + per < ncode ? b + per : ncode;
    uint32_t s = 0;
    for (int64_t k = b; k < e; ++k) s += c[k];
    __shared__ uint32_t ws[32];
    const int lane = t & 31, w = t >> 5;
    uint32_t inc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) ws[w] = inc;
    __syncthreads();
    if (w == 0) {
        uint32_t v = lane < (nt >> 5) ? ws[lane] : 0u;
        uint32_t iv = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, iv, o);
            if (lane >= o) iv += u;
        }
        ws[lane] = iv - v;
    }
    __syncthreads();
    uint32_t run = ws[w] + inc - s;
    for (int64_t k = b; k < e; ++k) {
        const uint32_t v = c[k];
        c[k] = run;
        run += v;
    }
}

__global__ void __launch_bounds__(256) k_scatter(const double *__restrict__ xyz, const int32_t *__restrict__ cls,
                                                 int64_t cls_stride, int64_t n, int64_t npad, int bits,
                                                 const uint32_t *__restrict__ code, const uint32_t *__restrict__ rank,
                                                 const uint32_t *__restrict__ cnt, double pad_sign, double2 *__restrict__ rec)
{
    const int f = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npad) return;
    double x, y, z;
    int32_t c, idx;
    int64_t pos;
    if (i < n) {
        const double *p = xyz + (int64_t)f * 3 * n;
        const int64_t ncode = (int64_t)1 << (3 * bits);
        pos = (int64_t)cnt[(int64_t)f * ncode + code[(int64_t)f * n + i]] + rank[(int64_t)f * n + i];
        x = p[i];
        y = p[n + i];
        z = p[2 * n + i];
        c = cls ? cls[(int64_t)f * cls_stride + i] : 0;
        idx = (int32_t)i;
    } else {
        // padding: far away, pairwise distinct, opposite sign for the two sets so that no pad-pad
        // pair of a rectangular call can coincide
        pos = i;
        x = pad_sign * (1.0e30 + (double)(i - n) * 1.0e25);
        y = 0.0;
        z = 0.0;
        c = 0;
        idx = -1;
    }
    double2 *r = rec + (int64_t)f * npad * 2;
    r[rec_xy(pos)] = make_double2(x, y);
    r[rec_zw(pos)] = make_double2(z, __hiloint2double(idx, c));
}

// group (32 points) and tile (256 points) bounding boxes over the valid points; one CTA per tile
__global__ void __launch_bounds__(TS) k_aabb(const double2 *__restrict__ rec, int64_t npad, int ngroups, int ntiles,
                                             double *__restrict__ taabb, float4 *__restrict__ gbox32)
{
    const int f = blockIdx.y, t = blockIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const double2 *r = rec + (int64_t)f * npad * 2;
    const int64_t pos = (int64_t)t * TS + threadIdx.x;
    const double2 xy = r[rec_xy(pos)], zw = r[rec_zw(pos)];
    const bool valid = __double2hiint(zw.y) >= 0;
    double lo[3] = {valid ? xy.x : DBL_MAX, valid ? xy.y : DBL_MAX, valid ? zw.x : DBL_MAX};
    double hi[3] = {valid ? xy.x : -DBL_MAX, valid ? xy.y : -DBL_MAX, valid ? zw.x : -DBL_MAX};
    __shared__ double s[GPT][6];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        lo[c] = warp_min(lo[c]);
        hi[c] = warp_max(hi[c]);
    }
    if (lane == 0) {
        for (int c = 0; c < 3; ++c) {
            s[w][c] = lo[c];
            s[w][3 + c] = hi[c];
        }
        // outward-rounded float copy for the chunk-level test of the pair kernel (empty group: lo > hi survives)
        float4 *g32 = gbox32 + ((int64_t)f * ngroups + (int64_t)t * GPT + w) * 2;
        g32[0] = make_float4(__double2float_rd(lo[0]), __double2float_rd(lo[1]), __double2float_rd(lo[2]), 0.f);
        g32[1] = make_float4(__double2float_ru(hi[0]), __double2float_ru(hi[1]), __double2float_ru(hi[2]), 0.f);
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        const int c = threadIdx.x;
        double v = s[0][c];
        for (int k = 1; k < GPT; ++k) v = c < 3 ? fmin(v, s[k][c]) : fmax(v, s[k][c]);
        taabb[((int64_t)f * ntiles + t) * 6 + c] = v;
    }
}

// one warp per (frame, ta) row: count (FILL=false) or emit (FILL=true) the tile pairs that may interact
template <bool FILL>
__global__ void __launch_bounds__(256) k_items(const double *__restrict__ taabbA, const double *__restrict__ taabbB, int ntA,
                                               int ntB, bool symm, bool nocull, bool tric, const double *__restrict__ box,
                                               double rcut2, int nframes, uint32_t *__restrict__ rowcnt,
                                               const uint32_t *__restrict__ rowoff, uint64_t *__restrict__ items)
{
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= (int64_t)nframes * ntA) return;
    const int f = (int)(row / ntA), ta = (int)(row % ntA);
    const double lx = box[f * 6 + 0], ly = box[f * 6 + 1], lz = box[f * 6 + 2];
    TriConst<DirF64> TC;
    if (tric) TC.set(box + f * 6);
    double a[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) a[c] = taabbA[((int64_t)f * ntA + ta) * 6 + c];
    uint32_t count = 0;
    const uint32_t base = FILL ? rowoff[row] : 0u;
    for (int tb0 = symm ? ta : 0; tb0 < ntB; tb0 += 32) {
        const int tb = tb0 + lane;
        bool ok = false;
        if (tb < ntB) {
            double b[6];
#pragma unroll
            for (int c = 0; c < 6; ++c) b[c] = taabbB[((int64_t)f * ntB + tb) * 6 + c];
            bool general;
            if (tric) {
                int code;
                ok = tri_box_test<DirF64>(a, b, TC, rcut2, code);
            } else {
                ok = boxes_may_interact(a, b, lx, ly, lz, rcut2, general);
            }
            if (nocull) ok = !(a[0] > a[3] || b[0] > b[3]);
        }
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (FILL && ok) {
            const uint32_t pos = base + count + __popc(m & ((1u << lane) - 1u));
            items[pos] = ((uint64_t)f << 44) | ((uint64_t)ta << 22) | (uint64_t)tb;
        }
        count += __popc(m);
    }
    if (!FILL && lane == 0) rowcnt[row] = count;
}

// exclusive scan over the rows (single CTA); also resets the work counter and records the totals
__global__ void __launch_bounds__(1024) k_row_scan(const uint32_t *__restrict__ rowcnt, uint32_t *__restrict__ rowoff,
                                                   int64_t nrows, unsigned long long *__restrict__ total,
                                                   unsigned int *__restrict__ counter, unsigned long long *__restrict__ stats,
                                                   unsigned long long nominal)
{
    const int t = threadIdx.x, nt = blockDim.x;
    const int64_t per = (nrows + nt - 1) / nt;
    const int64_t b = (int64_t)t * per, e = b + per < nrows ? b + per : nrows;
    uint32_t s = 0;
    for (int64_t k = b; k < e; ++k) s += rowcnt[k];
    __shared__ uint32_t ws[32];
    const int lane = t & 31, w = t >> 5;
    uint32_t inc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) ws[w] = inc;
    __syncthreads();
    if (w == 0) {
        const uint32_t v = lane < (nt >> 5) ? ws[lane] : 0u;
        uint32_t iv = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, iv, o);
            if (lane >= o) iv += u;
        }
        ws[lane] = iv - v;
        if (lane == 31) {
            *total = (unsigned long long)iv;
            *counter = 0u;
            atomicAdd(&stats[0], (unsigned long long)iv);
            atomicAdd(&stats[1], nominal);
        }
    }
    __syncthreads();
    uint32_t run = ws[w] + inc - s;
    for (int64_t k = b; k < e; ++k) {
        const uint32_t v = rowcnt[k];
        rowoff[k] = run;
        run += v;
    }
}

// ---------------------------------------------------------------------------------------------
// the pair kernel
// ---------------------------------------------------------------------------------------------
struct PairParams {
    const double2 *recA, *recB;      // group-blocked records, [F][npad*2] double2
    const float4 *gboxA, *gboxB;     // outward-rounded float boxes of the 32-point groups, 2 x float4 each
    int64_t npadA, npadB;
    int ngA, ngB;
    int ntA;                         // tiles of set A per frame (rows of the work list per frame)
    int nframes;
    const double *box;               // device [F][3]
    const uint64_t *items;           // tile pairs, grouped by frame
    const uint32_t *rowoff;          // [F*ntA] exclusive offsets into items
    const unsigned long long *total; // number of items
    unsigned int *counters;          // [F] per-frame warp-item counters (zeroed before launch)
    unsigned long long *stats;
    double rcut2;                    // pre-filter cutoff (max of all cutoffs)
    // histogram modes
    int nbins, nrows, nclsB, ncp;
    const double2 *edges2;           // device [nbins+1]: {e[k], e[k+1]}, e[nbins+1] = +inf
    const int *cptab;                // device [nclsA*nclsB] -> histogram row
    float inv_ddr;
    unsigned long long *hist;        // device [F][nrows][nbins]
    int edges_in_smem;
    // list mode
    double rin2, rout2;
    int shell_mode, exclude_same;
    int swap_out;                    // list mode: sets A and B were exchanged by the host, write (frame, j, i)
    int32_t *list;
    double *list_rsq;
    long long capacity;
    unsigned long long *list_count;
    int frame0;                      // global index of the first frame of this sub-batch
    int nocull;                      // MDP_PAIR_NO_CULL: evaluate every chunk pair on the general path
    // k_pair_fast (pair_fast.cuh): error-bound terms in bins, already times the 1.5 safety factor
    float f_rc;                      // cutoff radius, rounded up
    float f_c1;                      // 1.5 * sqrt(3) * 2^-24 / ddr: bins per A of coordinate error
    float f_rel;                     // 1.5 * (nbins + 1) * RHO: the relative part
    float f_rc2t;                    // point-filter threshold: rcut2 rounded up, times (1 + 2^-18) rounded up
    int f_smax;                      // most fraction bits the 2^23 trick leaves room for
};

struct Shared {
    const double2 *edges_s;          // shared-memory copy of the edge table (valid when edges_in_smem)
    const int *cptab;
    unsigned int *hist;
};

// bytes of the warp-private region: two chunk stages + the hit queue (+ its metadata)
__host__ __device__ constexpr size_t warp_region_bytes(bool meta)
{
    return 2 * RING * sizeof(double2) + QCAP * sizeof(double) + (meta ? QCAP * sizeof(uint2) : 0);
}

// shared-memory bytes of the edge table: nbins + 1 (lo, hi) pairs
__host__ __device__ constexpr size_t edge_region_bytes(int nbins) { return (size_t)(nbins + 1) * 16; }

template <int MODE, bool MULTICLS>
__device__ __forceinline__ void drain(const PairParams &p, const Shared &sh, int lane, int m, const double *qr,
                                      const uint2 *qm, int base, int frame)
{
    __syncwarp();
    if (MODE == MODE_LIST) {
        bool ok = false;
        double r2 = 0.0;
        uint2 me = make_uint2(0u, 0u);
        if (lane < m) {
            r2 = qr[base + lane];
            me = qm[base + lane];
            ok = p.shell_mode ? (r2 > p.rin2 && r2 <= p.rout2) : (r2 < p.rout2);
            if (p.exclude_same && me.x == me.y) ok = false;
        }
        const unsigned mask = __ballot_sync(0xffffffffu, ok);
        if (mask) {
            unsigned long long b0 = 0;
            if (lane == 0) b0 = atomicAdd(p.list_count, (unsigned long long)__popc(mask));
            b0 = __shfl_sync(0xffffffffu, b0, 0);
            if (ok) {
                const long long pos = (long long)b0 + __popc(mask & ((1u << lane) - 1u));
                if (pos < p.capacity) {
                    p.list[pos * 3 + 0] = frame;
                    p.list[pos * 3 + 1] = (int32_t)(p.swap_out ? me.y : me.x);
                    p.list[pos * 3 + 2] = (int32_t)(p.swap_out ? me.x : me.y);
                    if (p.list_rsq) p.list_rsq[pos] = r2;
                }
            }
        }
    } else {
        if (lane < m) {
            const double r2 = qr[base + lane];
            if (r2 < p.rcut2) {
                int k;
                if (MODE == MODE_HIST_UNIFORM) {
                    // fp32 estimate of sqrt(rsq)/ddr is within +-1 of the reference bin; the exact fp64
                    // edge pair {e[k], e[k+1]} settles it (see mdp_bin_edges)
                    float s;
                    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(__double2float_rz(r2)));
                    s *= p.inv_ddr;
                    k = (int)s;
                    k = k < 0 ? 0 : (k > p.nbins ? p.nbins : k);
                    const double2 e = p.edges_in_smem ? sh.edges_s[k] : p.edges2[k];
                    k += (r2 >= e.y) ? 1 : 0;
                    k -= (r2 < e.x) ? 1 : 0;
                } else {
                    k = 0;
                    for (int j = 1; j <= p.nbins; ++j) k += ((p.edges_in_smem ? sh.edges_s[j].x : p.edges2[j].x) <= r2) ? 1 : 0;
                }
                if (k >= 0 && k < p.nbins) {
                    const int row = MULTICLS ? sh.cptab[qm[base + lane].x] : 0;
                    atomicAdd(&sh.hist[row * p.nbins + k], 1u);
                }
            }
        }
    }
    __syncwarp();
}

// one 32 x 32 chunk pair: lane = i point, loop over the 32 j points of the staged chunk, four at a time so that
// four independent fp64 chains are in flight; the hits of the four steps are compacted with one branch.
//   VAR_FAST   no axis needs the minimum image           8 fp64 ops / pair
//   VAR_SHIFT  per axis d' = |d| - s, s = 0 or l          11 fp64 ops / pair (|d| - 0 is exact)
//   VAR_MIXED  per axis d' = min(|d|, ||d| - l|)          14 fp64 ops / pair (see AX_MIXED)
// In every variant only the square of d' is used and it equals the reference's (rdf_cn.py:50-56) bit for bit.
//   VAR_TSHIFT triclinic, one image vector for the chunk    14 fp64 ops / pair (sequential shifts, oracle order)
//   VAR_TMIXED triclinic, image vector decided per pair      14 fp64 ops + selects
enum { VAR_FAST = 0, VAR_SHIFT = 1, VAR_MIXED = 2, VAR_TSHIFT = 3, VAR_TMIXED = 4 };

// shifts of one chunk pair.  Orthogonal variants use x, y, z only (0 or l).  VAR_TSHIFT: x = kx*lx, y = ky*ly,
// z = kz*lz, xy = ky*xy, xz = kz*xz, yz = kz*yz.  VAR_TMIXED: the cell itself (lx, ly, lz, xy, xz, yz).
struct Shift {
    double x, y, z, xy, xz, yz;
};

// squared minimum-image distance of one pair from the raw differences (ax, ay, az) = (xi - xj, ...), in the operation
// order of the reference (rdf_cn.py:50-56) / of oracle.c pair_rsq_tri for the triclinic variants
template <int VAR>
__device__ __forceinline__ double image_r2(double ax, double ay, double az, const Shift &S, double hx, double hy, double hz)
{
    const double sx = S.x, sy = S.y, sz = S.z;
    if (VAR == VAR_SHIFT) {
        ax = __dsub_rn(fabs(ax), sx);
        ay = __dsub_rn(fabs(ay), sy);
        az = __dsub_rn(fabs(az), sz);
    } else if (VAR == VAR_MIXED) {
        ax = fmin(fabs(ax), fabs(__dsub_rn(fabs(ax), sx)));
        ay = fmin(fabs(ay), fabs(__dsub_rn(fabs(ay), sy)));
        az = fmin(fabs(az), fabs(__dsub_rn(fabs(az), sz)));
    } else if (VAR == VAR_TSHIFT) {
        az = __dsub_rn(az, sz);
        ay = __dsub_rn(__dsub_rn(ay, S.yz), sy);
        ax = __dsub_rn(__dsub_rn(__dsub_rn(ax, S.xz), S.xy), sx);
    } else if (VAR == VAR_TMIXED) {
        const bool pz = az > hz, nz = az < -hz;
        az = __dsub_rn(az, pz ? sz : (nz ? -sz : 0.0));
        ay = __dsub_rn(ay, pz ? S.yz : (nz ? -S.yz : 0.0));
        ax = __dsub_rn(ax, pz ? S.xz : (nz ? -S.xz : 0.0));
        const bool py = ay > hy, ny = ay < -hy;
        ay = __dsub_rn(ay, py ? sy : (ny ? -sy : 0.0));
        ax = __dsub_rn(ax, py ? S.xy : (ny ? -S.xy : 0.0));
        const bool px = ax > hx, nx = ax < -hx;
        ax = __dsub_rn(ax, px ? sx : (nx ? -sx : 0.0));
    }
    return __dadd_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)), __dmul_rn(az, az));
}

template <int MODE, bool MULTICLS, int VAR, bool TRI>
__device__ __forceinline__ void chunk_loop(const PairParams &p, const Shared &sh, const double2 *__restrict__ jb, int nj, double xi,
                                           double yi, double zi, uint32_t mi, const Shift S, int rc_hi,
                                           int lane, int &qn, double *qr, uint2 *qm, int frame)
{
    const double hx = S.x * 0.5, hy = S.y * 0.5, hz = S.z * 0.5;   // VAR_TMIXED only
    constexpr bool META = MULTICLS || MODE == MODE_LIST;
    const unsigned lt = (1u << lane) - 1u;
#pragma unroll 1
    for (int j0 = 0; j0 < nj; j0 += 4) {   // nj is a multiple of 4 (candidate batches are padded with +inf points)
        double r2[4];
        double meta[4];
        bool hit[4];
        unsigned m[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int jj = j0 + u;
            const double2 xy = jb[jj];
            const double2 zw = jb[RING + jj];
            r2[u] = image_r2<VAR>(__dsub_rn(xi, xy.x), __dsub_rn(yi, xy.y), __dsub_rn(zi, zw.x), S, hx, hy, hz);
            hit[u] = __double2hiint(r2[u]) <= rc_hi;   // superset of rsq < rcut2; settled exactly in drain()
            if (TRI) hit[u] = hit[u] && (jj > lane);
            if (META) meta[u] = zw.y;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) m[u] = __ballot_sync(0xffffffffu, hit[u]);
        if (m[0] | m[1] | m[2] | m[3]) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (hit[u]) {
                    const int pos = qn + __popc(m[u] & lt);
                    qr[pos] = r2[u];
                    if (META) {
                        if (MODE == MODE_LIST)
                            qm[pos] = make_uint2(mi, (uint32_t)__double2hiint(meta[u]));
                        else
                            qm[pos] = make_uint2(mi + (uint32_t)__double2loint(meta[u]), 0u);
                    }
                }
                qn += __popc(m[u]);
            }
            while (qn >= 32) {
                qn -= 32;
                drain<MODE, MULTICLS>(p, sh, lane, 32, qr, qm, qn, frame);
            }
        }
    }
}

// evaluate the nj queued j points at jb (a multiple of 4; (x,y) at jb[k], (z,meta) at jb[RING + k]) against the 32 i points
// of the warp, under the image class `cc` of the chunk pair they came from
template <int MODE, bool MULTICLS, bool TRICL>
__device__ __forceinline__ void run_batch(const PairParams &p, const Shared &sh, const double2 *jb, int nj, int cc, bool tri,
                                          double xi, double yi, double zi, uint32_t mi, double lx, double ly, double lz,
                                          const double *cell, int rc_hi, int lane, int &qn, double *qr, uint2 *qm, int frame)
{
    const Shift Z0 = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    if (cc == 0) {
        if (tri)
            chunk_loop<MODE, MULTICLS, VAR_FAST, true>(p, sh, jb, nj, xi, yi, zi, mi, Z0, rc_hi, lane, qn, qr, qm, frame);
        else
            chunk_loop<MODE, MULTICLS, VAR_FAST, false>(p, sh, jb, nj, xi, yi, zi, mi, Z0, rc_hi, lane, qn, qr, qm, frame);
    } else if (TRICL) {
        if (cc != TRI_MIXED && !tri) {
            const int kx = cc & 3, ky = (cc >> 2) & 3, kz = (cc >> 4) & 3;
            const Shift S = {tri_dec(kx, lx), tri_dec(ky, ly), tri_dec(kz, lz), tri_dec(ky, cell[3]), tri_dec(kz, cell[4]),
                             tri_dec(kz, cell[5])};
            chunk_loop<MODE, MULTICLS, VAR_TSHIFT, false>(p, sh, jb, nj, xi, yi, zi, mi, S, rc_hi, lane, qn, qr, qm, frame);
        } else {
            const Shift S = {lx, ly, lz, cell[3], cell[4], cell[5]};
            if (tri)
                chunk_loop<MODE, MULTICLS, VAR_TMIXED, true>(p, sh, jb, nj, xi, yi, zi, mi, S, rc_hi, lane, qn, qr, qm, frame);
            else
                chunk_loop<MODE, MULTICLS, VAR_TMIXED, false>(p, sh, jb, nj, xi, yi, zi, mi, S, rc_hi, lane, qn, qr, qm, frame);
        }
    } else {
        const bool mixed = ((cc | (cc >> 2) | (cc >> 4)) & AX_MIXED) != 0;
        if (!mixed && !tri) {
            const Shift S = {(cc & 1) ? lx : 0.0, (cc & 4) ? ly : 0.0, (cc & 16) ? lz : 0.0, 0.0, 0.0, 0.0};
            chunk_loop<MODE, MULTICLS, VAR_SHIFT, false>(p, sh, jb, nj, xi, yi, zi, mi, S, rc_hi, lane, qn, qr, qm, frame);
        } else {
            // undecided axes (small boxes, huge groups) and the rare wrapped diagonal chunk: exact for every d
            const Shift S = {lx, ly, lz, 0.0, 0.0, 0.0};
            if (tri)
                chunk_loop<MODE, MULTICLS, VAR_MIXED, true>(p, sh, jb, nj, xi, yi, zi, mi, S, rc_hi, lane, qn, qr, qm, frame);
            else
                chunk_loop<MODE, MULTICLS, VAR_MIXED, false>(p, sh, jb, nj, xi, yi, zi, mi, S, rc_hi, lane, qn, qr, qm, frame);
        }
    }
}

template <int MODE, bool MULTICLS, bool SYMM, bool TRICL>
__global__ void __launch_bounds__(NWARP * 32, CTAS_PER_SM) k_pair(const PairParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr bool META = MULTICLS || MODE == MODE_LIST;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;

    // warp-private region
    unsigned char *wp = smem_raw + (size_t)w * warp_region_bytes(META);
    double2 *ring = reinterpret_cast<double2 *>(wp);                       // [RING] (x,y) then [RING] (z,meta)
    double *qr = reinterpret_cast<double *>(wp + 2 * RING * sizeof(double2));
    uint2 *qm = reinterpret_cast<uint2 *>(wp + 2 * RING * sizeof(double2) + QCAP * sizeof(double));
    // CTA-shared region
    unsigned char *sp = smem_raw + (size_t)NWARP * warp_region_bytes(META);
    Shared sh;
    double2 *edges_s = reinterpret_cast<double2 *>(sp);
    if (MODE != MODE_LIST && p.edges_in_smem) sp += edge_region_bytes(p.nbins);
    int *cptab_s = reinterpret_cast<int *>(sp);
    if (MULTICLS) sp += (size_t)((p.ncp * 4 + 15) & ~15);
    unsigned int *evals_s = reinterpret_cast<unsigned int *>(sp);   // 32-pair steps since the CTA histogram was last flushed
    if (MODE != MODE_LIST) sp += 16;                                // (list mode has no histogram region at all)
    sh.hist = reinterpret_cast<unsigned int *>(sp);
    sh.edges_s = edges_s;
    sh.cptab = p.cptab;

    const int nhist = MODE == MODE_LIST ? 0 : p.nrows * p.nbins;
    if (MODE != MODE_LIST) {
        if (p.edges_in_smem)
            for (int k = tid; k <= p.nbins; k += blockDim.x) edges_s[k] = p.edges2[k];
        for (int k = tid; k < nhist; k += blockDim.x) sh.hist[k] = 0u;
    }
    if (MODE != MODE_LIST && tid == 0) *evals_s = 0u;
    if (MULTICLS) {
        for (int k = tid; k < p.ncp; k += blockDim.x) cptab_s[k] = p.cptab[k];
        sh.cptab = cptab_s;
    }
    __syncthreads();

    int qn = 0;
    const int rc_hi = __double2hiint(p.rcut2);
    const float rcut2_up = __double2float_ru(p.rcut2);
    const unsigned long long total = *p.total;
    unsigned long long my_evals = 0;   // 32-pair evaluation steps executed by this warp
    const int F = p.nframes;
    // every CTA starts at a different frame and walks all of them, so the frames' tails do not line up
    const int fstart = (int)(((long long)blockIdx.x * F) / gridDim.x);

    // Histogram modes: a CTA works on one frame at a time (its shared-memory histogram belongs to that frame) and its
    // warps pull units from the frame's counter.  List mode has no per-frame state, so every warp pulls from ONE counter
    // over all (frame, unit) pairs -- with thousands of small frames (residence-time searches) walking every frame
    // from every CTA would cost more than the search itself.
    const unsigned int nunits = (unsigned int)p.ntA * GPT;   // work units per frame: one per 32-point i group
    const unsigned int all_units = MODE == MODE_LIST ? nunits * (unsigned int)F : 0u;
    unsigned int gq = 0;
    if (MODE == MODE_LIST) {
        if (lane == 0) gq = atomicAdd(&p.counters[0], 1u);
        gq = __shfl_sync(0xffffffffu, gq, 0);
    }
#pragma unroll 1
    for (int fk = 0;; ++fk) {
        int f;
        if (MODE == MODE_LIST) {
            if (gq >= all_units) break;
            f = (int)(gq / nunits);
        } else {
            if (fk >= F) break;
            f = fstart + fk;
            if (f >= F) f -= F;
        }
        const double lx = p.box[f * 6 + 0], ly = p.box[f * 6 + 1], lz = p.box[f * 6 + 2];
        const AxisF AX = make_axis(lx), AY = make_axis(ly), AZ = make_axis(lz);
        const int frame = p.frame0 + f;
        const double2 *rA = p.recA + (int64_t)f * p.npadA * 2;
        const double2 *rB = p.recB + (int64_t)f * p.npadB * 2;
        const float4 *gbB = p.gboxB + (int64_t)f * p.ngB * 2;
        bool did = false;

        unsigned int q = 0;
        if (MODE == MODE_LIST) {
            q = gq - (unsigned int)f * nunits;
        } else {
            if (lane == 0) q = atomicAdd(&p.counters[f], 1u);
            q = __shfl_sync(0xffffffffu, q, 0);
        }
#pragma unroll 1
        while (q < nunits) {
            unsigned int qnext = 0;
            if (lane == 0) qnext = atomicAdd(&p.counters[MODE == MODE_LIST ? 0 : f], 1u);   // prefetch the next work index
            did = true;
            const unsigned long long unit_evals0 = my_evals;
            // One unit = one i group (32 points, one per lane) against every j tile of its tile row of the work list.
            const int ta = (int)(q >> 3), wi = (int)(q & 7u);
            const int64_t row = (int64_t)f * p.ntA + ta;
            unsigned int t0 = p.rowoff[row];
            const unsigned int tend = row + 1 < (int64_t)F * p.ntA ? p.rowoff[row + 1] : (unsigned int)total;
            const int64_t gi = (int64_t)ta * GPT + wi;
            const double2 ixy = rA[gi * GREC + lane], izw = rA[gi * GREC + 32 + lane];
            const float4 *ga4 = p.gboxA + ((int64_t)f * p.ngA + gi) * 2;
            const float4 alo = ga4[0], ahi = ga4[1];
            const float ga[6] = {alo.x, alo.y, alo.z, ahi.x, ahi.y, ahi.z};
            const uint32_t mi = MODE == MODE_LIST ? (uint32_t)__double2hiint(izw.y)
                                                  : (uint32_t)(__double2loint(izw.y) * p.nclsB);

            // Chunk level: 32 lanes test the boxes of 32 j chunks (4 tiles x 8 chunks) against my group's box at a time.
            // Point level: the needed chunks are filtered point by point -- lane l keeps j point l of the chunk only if
            // it can be inside the cutoff of SOME point of my group's box (fp32, rounded outward, under the chunk pair's
            // image class).  The survivors are appended to a 64-entry ring; whenever 32 are queued they are evaluated
            // against the 32 i points with the 4-way unrolled loop.  A change of image class, the triangular self chunk
            // and the end of the unit flush the ring (padded to a multiple of 4 with +inf points, which can never be
            // inside the cutoff).  One chunk is always in flight (registers) while the previous one is processed.
            unsigned needmask = 0;
            int tbl = -1, code = 0;                       // per lane: tile and image class of "my" chunk of the current 32
            int head = 0, tail = 0, cur = 0;              // ring state; cur = image class of the queued candidates
            bool cvalid = false, nvalid = false, cself = false, nself = false;
            int ccode = 0, ncode = 0;
            double2 jxy = make_double2(0.0, 0.0), jzw = jxy, nxy = jxy, nzw = jxy;
#pragma unroll 1
            while (true) {
                // promote the prefetched chunk and fetch its successor in the same round; the first round of a unit has
                // nothing to promote yet and takes a second pass
#pragma unroll 1
                for (int pass = 0; pass < 2; ++pass) {
                    if (!cvalid && nvalid) {
                        cvalid = true;
                        nvalid = false;
                        ccode = ncode;
                        cself = nself;
                        jxy = nxy;
                        jzw = nzw;
                    }
                    if (!nvalid) {
                        // fetch: next needed chunk of the row into the "next" registers
#pragma unroll 1
                        while (needmask == 0u && t0 < tend) {
                            const unsigned int it = t0 + (unsigned)(lane >> 3);
                            const int cj = lane & 7;
                            tbl = it < tend ? (int)(p.items[it] & 0x3fffffu) : -1;
                            bool need = false;
                            code = 0;
                            if (tbl >= 0 && !(SYMM && tbl == ta && cj < wi)) {
                                const float4 *gb4 = gbB + ((int64_t)tbl * GPT + cj) * 2;
                                const float4 blo = gb4[0], bhi = gb4[1];
                                const float gb[6] = {blo.x, blo.y, blo.z, bhi.x, bhi.y, bhi.z};
                                if (TRICL) {
                                    TriConst<DirF32> TC;
                                    TC.set(p.box + f * 6);
                                    need = tri_box_test<DirF32>(ga, gb, TC, rcut2_up, code);
                                } else {
                                    need = chunk_test_f32(ga, gb, AX, AY, AZ, rcut2_up, code);
                                }
                                if (p.nocull) {
                                    need = !(ga[0] > ga[3] || gb[0] > gb[3]);
                                    code = TRICL ? TRI_MIXED : (AX_MIXED | (AX_MIXED << 2) | (AX_MIXED << 4));
                                }
                            }
                            needmask = __ballot_sync(0xffffffffu, need);
                            t0 += 4;
                        }
                        if (needmask) {
                            const int l = __ffs(needmask) - 1;
                            needmask &= needmask - 1;
                            const int tb = __shfl_sync(0xffffffffu, tbl, l);
                            ncode = __shfl_sync(0xffffffffu, code, l);
                            nself = SYMM && tb == ta && (l & 7) == wi;
                            const double2 *jsrc = rB + ((int64_t)tb * GPT + (l & 7)) * GREC;
                            nxy = __ldg(&jsrc[lane]);
                            nzw = __ldg(&jsrc[32 + lane]);
                            nvalid = true;
                        }
                    }
                    if (cvalid || !nvalid) break;
                }
                int run_n = 0, run_base = 0, run_code = cur;
                bool run_tri = false;
                if (!cvalid) {
                    if (tail == head) break;   // nothing prefetched either (a prefetched chunk was promoted above)
                    run_n = -1;   // end of the unit: flush
                } else if ((cself || ccode != cur) && tail != head) {
                    run_n = -1;   // flush first; the chunk is looked at again in the next round
                } else if (cself) {
                    ring[lane] = jxy;
                    ring[RING + lane] = jzw;
                    run_n = 32;
                    run_code = ccode;
                    run_tri = true;
                    cvalid = false;
                } else {
                    cur = ccode;
                    run_code = ccode;
                    bool ok;
                    if (TRICL)
                        ok = (ccode == TRI_MIXED) || tri_point_test_f32(ga, jxy.x, jxy.y, jzw.x, p.box + f * 6, rcut2_up, ccode);
                    else
                        ok = point_test_f32(ga, jxy.x, jxy.y, jzw.x, AX, AY, AZ, rcut2_up, ccode);
                    if (p.nocull) ok = true;
                    const unsigned m = __ballot_sync(0xffffffffu, ok);
                    if (ok) {
                        const int pos = (tail + __popc(m & ((1u << lane) - 1u))) & (RING - 1);
                        ring[pos] = jxy;
                        ring[RING + pos] = jzw;
                    }
                    tail += __popc(m);
                    cvalid = false;
                    if (tail - head >= 32) {
                        run_n = 32;
                        run_base = head & 32;
                    }
                }
                if (run_n == 0) continue;
                const bool flush = run_n < 0;
                if (flush) {
                    const int n = tail - head;
                    run_n = (n + 3) & ~3;
                    run_base = head & 32;
                    if (lane < run_n - n) {
                        const int pos = (tail + lane) & (RING - 1);
                        ring[pos] = make_double2(INFINITY, 0.0);
                        ring[RING + pos] = make_double2(0.0, 0.0);
                    }
                }
                __syncwarp();
                my_evals += (unsigned long long)run_n;
                run_batch<MODE, MULTICLS, TRICL>(p, sh, ring + run_base, run_n, run_code, run_tri, ixy.x, ixy.y, izw.x, mi, lx, ly, lz,
                                                 p.box + f * 6, rc_hi, lane, qn, qr, qm, frame);
                __syncwarp();   // everyone is done with the batch before the ring is written again
                if (flush || run_tri) {
                    head = 0;
                    tail = 0;
                } else {
                    head += 32;
                }
            }
            if (MODE != MODE_LIST) {
                // overflow guard of the uint32 shared histogram (a frame of N >~ 90 000 points has more than 2^32 pairs and a
                // CTA may own a whole frame): the CTA counts its 32-pair steps; the warp that crosses a multiple of 2^25
                // steps (2^30 pairs) moves the histogram to the global one word by word with atomicExch -- race free without
                // a barrier; a unit adds at most 32 x npad pairs (npad < 2^22: 8 warps stay below 2^31 in between)
                const unsigned add = (unsigned)(my_evals - unit_evals0);
                unsigned old_ = 0;
                if (lane == 0) old_ = atomicAdd(evals_s, add);
                old_ = __shfl_sync(0xffffffffu, old_, 0);
                if (((old_ + add) >> 25) != (old_ >> 25)) {
                    unsigned long long *hg = p.hist + (int64_t)frame * nhist;
                    for (int k = lane; k < nhist; k += 32) {
                        const unsigned int v = atomicExch(&sh.hist[k], 0u);
                        if (v) atomicAdd(&hg[k], (unsigned long long)v);
                    }
                }
            }
            q = __shfl_sync(0xffffffffu, qnext, 0);
            if (MODE == MODE_LIST) {
                gq = q;                                   // global index; beyond this frame it ends the unit loop
                q -= (unsigned int)f * nunits;
            }
        }

        // this warp is done with frame f: empty its queue, then the CTA flushes its histogram
        if (qn > 0) {
            drain<MODE, MULTICLS>(p, sh, lane, qn, qr, qm, 0, frame);
            qn = 0;
        }
        if (MODE != MODE_LIST) {
            if (__syncthreads_or(did ? 1 : 0)) {
                unsigned long long *hg = p.hist + (int64_t)frame * nhist;
                for (int k = tid; k < nhist; k += blockDim.x) {
                    const unsigned int v = sh.hist[k];
                    if (v) {
                        atomicAdd(&hg[k], (unsigned long long)v);
                        sh.hist[k] = 0u;
                    }
                }
                if (tid == 0) *evals_s = 0u;
                __syncthreads();
            }
        }
    }
    if (lane == 0 && my_evals) atomicAdd(&p.stats[2], my_evals * (unsigned long long)GS);
}

} // namespace

#include "pair_fast.cuh"

namespace {

// out[f][r][b] = sum_rows w[r][row] * (cumulative ? prefix : value) hist[f][row][b]
__global__ void __launch_bounds__(256) k_hist_reduce(const unsigned long long *__restrict__ hist, int rows, int nbins,
                                                     int nout, const int *__restrict__ wts, int cumulative,
                                                     unsigned long long *__restrict__ out)
{
    const int f = blockIdx.y;
    const int r = blockIdx.x;
    const unsigned long long *h = hist + (int64_t)f * rows * nbins;
    unsigned long long *o = out + ((int64_t)f * nout + r) * nbins;
    if (!cumulative) {
        for (int b = threadIdx.x; b < nbins; b += blockDim.x) {
            unsigned long long s = 0;
            for (int q = 0; q < rows; ++q) {
                const int wv = wts[r * rows + q];
                if (wv) s += (unsigned long long)wv * h[(int64_t)q * nbins + b];
            }
            o[b] = s;
        }
    } else if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (int b = 0; b < nbins; ++b) {
            for (int q = 0; q < rows; ++q) {
                const int wv = wts[r * rows + q];
                if (wv) run += (unsigned long long)wv * h[(int64_t)q * nbins + b];
            }
            o[b] = run;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host orchestration
// ---------------------------------------------------------------------------------------------
struct SetPlan {
    int64_t n = 0, npad = 0;
    int ntiles = 0, ngroups = 0, bits = 0;
    int64_t ncode = 1;
    // device scratch (per sub-batch)
    double2 *rec = nullptr;
    float4 *gbox32 = nullptr;
    double *taabb = nullptr, *mm = nullptr;
    uint32_t *code = nullptr, *rank = nullptr, *cnt = nullptr;
};

static void plan_set(SetPlan &s, int64_t n, bool nosort)
{
    s.n = n;
    s.ntiles = (int)ceil_div<int64_t>(n, TS);
    s.npad = (int64_t)s.ntiles * TS;
    s.ngroups = s.ntiles * GPT;
    // ~4 points per cell
    int bits = 0;
    if (!nosort) {
        while (bits < 7 && ((int64_t)1 << (3 * (bits + 1))) * 4 <= n * 2) ++bits;
    }
    s.bits = bits;
    s.ncode = (int64_t)1 << (3 * bits);
}

static size_t set_bytes_per_frame(const SetPlan &s)
{
    return align256(s.npad * REC_BYTES) + align256(s.ngroups * 32) + align256(s.ntiles * 48) + align256(48) +
           2 * align256(s.n * 4) + align256(s.ncode * 4) + 4096;
}

static int carve_set(mdp_ctx *ctx, SetPlan &s, int F)
{
    s.rec = (double2 *)ctx->arena_take((size_t)F * s.npad * REC_BYTES);
    s.gbox32 = (float4 *)ctx->arena_take((size_t)F * s.ngroups * 32);
    s.taabb = (double *)ctx->arena_take((size_t)F * s.ntiles * 48);
    s.mm = (double *)ctx->arena_take((size_t)F * 48);
    s.code = (uint32_t *)ctx->arena_take((size_t)F * s.n * 4);
    s.rank = (uint32_t *)ctx->arena_take((size_t)F * s.n * 4);
    s.cnt = (uint32_t *)ctx->arena_take((size_t)F * s.ncode * 4);
    if (!s.rec || !s.gbox32 || !s.taabb || !s.mm || !s.code || !s.rank || !s.cnt) {
        mdp_set_error("internal: scratch arena exhausted while carving a point set");
        return MDP_ERR_OOM;
    }
    return 0;
}

static int sort_set(mdp_ctx *ctx, SetPlan &s, int F, const double *xyz, const int32_t *cls, int64_t cls_stride,
                    double pad_sign, cudaStream_t st)
{
    if (s.bits > 0) {
        k_minmax<<<F, 1024, 0, st>>>(xyz, s.n, s.mm);
        MDP_LAUNCHED(ctx);
    }
    MDP_CUDA(cudaMemsetAsync(s.cnt, 0, (size_t)F * s.ncode * 4, st));
    dim3 g1((unsigned)ceil_div<int64_t>(s.n, 256), F);
    k_cell_count<<<g1, 256, 0, st>>>(xyz, s.n, s.mm, s.bits, s.code, s.rank, s.cnt);
    MDP_LAUNCHED(ctx);
    k_cell_scan<<<F, 1024, 0, st>>>(s.cnt, s.ncode);
    MDP_LAUNCHED(ctx);
    dim3 g2((unsigned)ceil_div<int64_t>(s.npad, 256), F);
    k_scatter<<<g2, 256, 0, st>>>(xyz, cls, cls_stride, s.n, s.npad, s.bits, s.code, s.rank, s.cnt, pad_sign, s.rec);
    MDP_LAUNCHED(ctx);
    dim3 g3(s.ntiles, F);
    k_aabb<<<g3, TS, 0, st>>>(s.rec, s.npad, s.ngroups, s.ntiles, s.taabb, s.gbox32);
    MDP_LAUNCHED(ctx);
    return mdp_check_launch("pair prep");
}

typedef void (*pair_kernel_t)(const PairParams);

template <int MODE, bool MULTICLS>
static pair_kernel_t pick_kernel2(bool symm, bool tric)
{
    if (tric) return symm ? k_pair<MODE, MULTICLS, true, true> : k_pair<MODE, MULTICLS, false, true>;
    return symm ? k_pair<MODE, MULTICLS, true, false> : k_pair<MODE, MULTICLS, false, false>;
}
template <int MODE>
static pair_kernel_t pick_kernel(bool multicls, bool symm, bool tric)
{
    return multicls ? pick_kernel2<MODE, true>(symm, tric) : pick_kernel2<MODE, false>(symm, tric);
}

static pair_kernel_t pick_fast(bool multicls, bool symm, bool tric)
{
    if (tric) {
        if (multicls) return symm ? k_pair_fast<true, true, true> : k_pair_fast<true, false, true>;
        return symm ? k_pair_fast<false, true, true> : k_pair_fast<false, false, true>;
    }
    if (multicls) return symm ? k_pair_fast<true, true, false> : k_pair_fast<true, false, false>;
    return symm ? k_pair_fast<false, true, false> : k_pair_fast<false, false, false>;
}

struct PairCall {
    int mode = MODE_HIST_UNIFORM;
    int nframes = 0;
    int64_t n_a = 0, n_b = 0;
    const double *xyz_a = nullptr, *xyz_b = nullptr;
    const int32_t *cls_a = nullptr, *cls_b = nullptr;
    int64_t cls_stride_a = 0, cls_stride_b = 0;
    int ncls_a = 1, ncls_b = 1;
    const double *box = nullptr;   // host
    double rcut2 = 0;
    const double *edges = nullptr; // host
    int nbins = 0;
    double uniform_ddr = 0;
    uint64_t *hist_out = nullptr;
    int flags = 0;
    // list
    double rin2 = 0, rout2 = 0;
    int shell_mode = 0, exclude_same = 0, swap_out = 0;
    int32_t *list = nullptr;
    double *list_rsq = nullptr;
    int64_t capacity = 0;
    int64_t *list_count = nullptr;
};

static int run_pair_call(mdp_ctx *ctx, const PairCall &c, cudaStream_t st)
{
    MDP_CUDA(cudaSetDevice(ctx->device));
    const bool symm = c.xyz_b == nullptr;
    const bool nosort = (c.flags & MDP_PAIR_NO_SORT) != 0;
    const bool nocull = (c.flags & MDP_PAIR_NO_CULL) != 0;
    const bool tric = (c.flags & MDP_PAIR_TRICLINIC) != 0;
    const bool hist_mode = c.mode != MODE_LIST;
    const int nclsB = symm ? c.ncls_a : c.ncls_b;
    const int nrows = symm ? c.ncls_a * (c.ncls_a + 1) / 2 : c.ncls_a * c.ncls_b;
    const bool multicls = hist_mode && nrows > 1;

    SetPlan A, B;
    plan_set(A, c.n_a, nosort);
    if (!symm) plan_set(B, c.n_b, nosort);
    const SetPlan &Bp = symm ? A : B;
    MDP_REQUIRE(A.ntiles < (1 << 22) && Bp.ntiles < (1 << 22), "pair: too many tiles");
    MDP_REQUIRE(!hist_mode || Bp.npad < ((int64_t)1 << 22),
                "pair: histogram calls are limited to 2^22 points per frame and set (the overflow guard of the per-CTA uint32 "
                "histogram assumes a work unit adds fewer than 2^27 pairs)");

    // shared memory budget of the pair kernel
    const bool meta = multicls || !hist_mode;
    size_t smem = NWARP * warp_region_bytes(meta);
    const int ncp = c.ncls_a * nclsB;
    int edges_in_smem = 0;
    if (hist_mode) {
        const size_t hist_bytes = (size_t)nrows * c.nbins * 4;
        const size_t edge_bytes = edge_region_bytes(c.nbins);
        if (multicls) smem += (size_t)((ncp * 4 + 15) & ~15);
        const size_t cap = std::min<size_t>(ctx->smem_optin, (216 / CTAS_PER_SM) * 1024);   // keep CTAS_PER_SM CTAs per SM
        MDP_REQUIRE(smem + hist_bytes + 16 <= ctx->smem_optin,
                    "pair: histogram of %d rows x %d bins does not fit in shared memory (%zu B needed); "
                    "reduce the number of distinct classes or bins per call",
                    nrows, c.nbins, smem + hist_bytes);
        if (smem + hist_bytes + 16 + edge_bytes <= cap) {
            edges_in_smem = 1;
            smem += edge_bytes;
        }
        smem += hist_bytes + 16;   // + the overflow guard's counter
    }

    // sub-batching over frames so that scratch stays bounded
    const size_t items_worst = symm ? (size_t)A.ntiles * (A.ntiles + 1) / 2 : (size_t)A.ntiles * Bp.ntiles;
    const size_t per_frame = set_bytes_per_frame(A) + (symm ? 0 : set_bytes_per_frame(B)) + align256(items_worst * 8) +
                             2 * align256((size_t)A.ntiles * 4) + 64 + 4;
    const size_t fixed = align256((size_t)(c.nbins + 2) * sizeof(double2)) + align256(MAX_CLS * MAX_CLS * 4) + 8192;
    const size_t target = std::min<size_t>(ctx->slab_limit, (size_t)3 << 29);   // 1.5 GiB working set
    // the request is the fixed part + 64 KB of headroom + per frame its scratch and its box (48 B); Fsub is sized on all
    // of it, and on what arena_reserve adds, so that a limit Fsub frames fit in is never exceeded (scratch_plan.h)
    const size_t fixed_req = fixed + 65536, per_frame_req = per_frame + 48;
    const int Fsub = (int)mdp_scratch_units(target, fixed_req, per_frame_req, (size_t)std::min(c.nframes, 1 << 19));
    MDP_REQUIRE((size_t)Fsub * items_worst < ((size_t)1 << 32), "pair: work list too long");
    int rc = ctx->arena_reserve(fixed_req + (size_t)Fsub * per_frame_req);
    if (rc) return rc;

    // edge pairs / class-pair table (host side staging)
    std::vector<double2> e2;
    std::vector<int> cpt(MAX_CLS * MAX_CLS, 0);
    if (hist_mode) {
        e2.resize(c.nbins + 2);
        for (int k = 0; k <= c.nbins; ++k) {
            const double lo = k == 0 ? 0.0 : c.edges[k];
            const double hi = k + 1 <= c.nbins ? c.edges[k + 1] : INFINITY;
            e2[k] = make_double2(lo, hi);
        }
        e2[c.nbins + 1] = make_double2(INFINITY, INFINITY);
        if (symm) {
            for (int i = 0; i < c.ncls_a; ++i)
                for (int j = 0; j < c.ncls_a; ++j) {
                    const int a = std::min(i, j), b = std::max(i, j);
                    cpt[i * c.ncls_a + j] = a * c.ncls_a - a * (a - 1) / 2 + (b - a);
                }
        } else {
            for (int i = 0; i < c.ncls_a; ++i)
                for (int j = 0; j < c.ncls_b; ++j) cpt[i * c.ncls_b + j] = i * c.ncls_b + j;
        }
    }

    // the fp32-filtered kernel (pair_fast.cuh) serves the uniform-bin histograms unless the caller asks for the fp64 one
    int f_smax = 0;
    {
        int bits = 0;
        while ((1 << bits) <= c.nbins + FAST_XROW) ++bits;
        f_smax = std::min(12, 22 - bits);
    }
    const size_t fast_smem = NWARP * FAST_WARP_BYTES + ((sizeof(FrameConst) + 15) & ~(size_t)15) +
                             (multicls ? (size_t)((ncp * 4 + 15) & ~15) : 0) + 32 + (size_t)nrows * (c.nbins + FAST_XROW) * 4;
    const bool fast = c.mode == MODE_HIST_UNIFORM && !nocull && c.edges[c.nbins] <= c.rcut2 && f_smax >= 6 &&
                      !(c.flags & MDP_PAIR_F64) && Bp.npad < ((int64_t)1 << 22) && fast_smem <= ctx->smem_optin &&
                      !getenv("MDP_PAIR_F64");
    if (fast) smem = fast_smem;
    pair_kernel_t kern = fast                          ? pick_fast(multicls, symm, tric)
                         : c.mode == MODE_HIST_UNIFORM ? pick_kernel<MODE_HIST_UNIFORM>(multicls, symm, tric)
                         : c.mode == MODE_HIST_TABLE   ? pick_kernel<MODE_HIST_TABLE>(multicls, symm, tric)
                                                       : pick_kernel2<MODE_LIST, false>(symm, tric);
    MDP_CUDA(cudaFuncSetAttribute((const void *)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int ctas_per_sm = CTAS_PER_SM;
    if (fast) {
        MDP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, (const void *)kern, NWARP * 32, smem));
        ctas_per_sm = std::max(1, std::min(ctas_per_sm, FAST_CTAS_PER_SM));
    }

    MDP_CUDA(cudaMemsetAsync(ctx->d_stats, 0, 4 * sizeof(unsigned long long), st));

    for (int f0 = 0; f0 < c.nframes; f0 += Fsub) {
        const int F = std::min(Fsub, c.nframes - f0);
        ctx->arena_reset();
        double2 *d_e2 = (double2 *)ctx->arena_take((size_t)(c.nbins + 2) * sizeof(double2));
        int *d_cpt = (int *)ctx->arena_take(MAX_CLS * MAX_CLS * 4);
        double *d_box = (double *)ctx->arena_take((size_t)F * 48);
        unsigned long long *d_total = (unsigned long long *)ctx->arena_take(16);
        unsigned int *d_counter = (unsigned int *)(d_total + 1);
        unsigned int *d_fcount = (unsigned int *)ctx->arena_take((size_t)F * 4);
        rc = carve_set(ctx, A, F);
        if (rc) return rc;
        if (!symm) {
            rc = carve_set(ctx, B, F);
            if (rc) return rc;
        }
        uint32_t *rowcnt = (uint32_t *)ctx->arena_take((size_t)F * A.ntiles * 4);
        uint32_t *rowoff = (uint32_t *)ctx->arena_take((size_t)F * A.ntiles * 4);
        uint64_t *items = (uint64_t *)ctx->arena_take((size_t)F * items_worst * 8);
        if (!d_e2 || !d_cpt || !d_box || !d_total || !d_fcount || !rowcnt || !rowoff || !items) {
            mdp_set_error("internal: scratch arena exhausted");
            return MDP_ERR_OOM;
        }
        if (hist_mode) {
            MDP_CUDA(cudaMemcpyAsync(d_e2, e2.data(), e2.size() * sizeof(double2), cudaMemcpyHostToDevice, st));
            MDP_CUDA(cudaMemcpyAsync(d_cpt, cpt.data(), cpt.size() * 4, cudaMemcpyHostToDevice, st));
        }
        // device cell rows are always {lx, ly, lz, xy, xz, yz} (pageable source: the copy is staged before it returns)
        {
            const int bs = tric ? 6 : 3;
            std::vector<double> hb((size_t)F * 6, 0.0);
            for (int f = 0; f < F; ++f)
                for (int k = 0; k < bs; ++k) hb[(size_t)f * 6 + k] = c.box[(size_t)(f0 + f) * bs + k];
            MDP_CUDA(cudaMemcpyAsync(d_box, hb.data(), (size_t)F * 48, cudaMemcpyHostToDevice, st));
        }

        cudaEvent_t tp = ctx->timer_begin(1, st);
        rc = sort_set(ctx, A, F, c.xyz_a + (size_t)f0 * 3 * c.n_a, c.cls_a ? c.cls_a + (size_t)f0 * c.cls_stride_a : nullptr,
                      c.cls_stride_a, +1.0, st);
        if (rc) return rc;
        if (!symm) {
            rc = sort_set(ctx, B, F, c.xyz_b + (size_t)f0 * 3 * c.n_b,
                          c.cls_b ? c.cls_b + (size_t)f0 * c.cls_stride_b : nullptr, c.cls_stride_b, -1.0, st);
            if (rc) return rc;
        }
        const SetPlan &Bs = symm ? A : B;
        const int64_t nrows_items = (int64_t)F * A.ntiles;
        const unsigned gi = (unsigned)ceil_div<int64_t>(nrows_items * 32, 256);
        k_items<false><<<gi, 256, 0, st>>>(A.taabb, Bs.taabb, A.ntiles, Bs.ntiles, symm, nocull, tric, d_box, c.rcut2, F, rowcnt,
                                           rowoff, items);
        MDP_LAUNCHED(ctx);
        k_row_scan<<<1, 1024, 0, st>>>(rowcnt, rowoff, nrows_items, d_total, d_counter, ctx->d_stats,
                                       (unsigned long long)F * (unsigned long long)items_worst);
        MDP_LAUNCHED(ctx);
        k_items<true><<<gi, 256, 0, st>>>(A.taabb, Bs.taabb, A.ntiles, Bs.ntiles, symm, nocull, tric, d_box, c.rcut2, F, rowcnt,
                                          rowoff, items);
        MDP_LAUNCHED(ctx);
        ctx->timer_end(tp, st);

        PairParams p;
        memset(&p, 0, sizeof(p));
        p.recA = A.rec;
        p.recB = Bs.rec;
        p.gboxA = A.gbox32;
        p.gboxB = Bs.gbox32;
        p.npadA = A.npad;
        p.npadB = Bs.npad;
        p.ngA = A.ngroups;
        p.ngB = Bs.ngroups;
        p.ntA = A.ntiles;
        p.nframes = F;
        p.box = d_box;
        p.items = items;
        p.rowoff = rowoff;
        p.total = d_total;
        p.counters = d_fcount;
        p.ncp = ncp;
        p.stats = ctx->d_stats;
        p.rcut2 = c.rcut2;
        p.nbins = c.nbins;
        p.nrows = nrows;
        p.nclsB = nclsB;
        p.edges2 = d_e2;
        p.cptab = d_cpt;
        p.inv_ddr = c.uniform_ddr > 0 ? (float)(1.0 / c.uniform_ddr) : 0.f;
        p.hist = (unsigned long long *)c.hist_out;
        p.edges_in_smem = edges_in_smem;
        p.rin2 = c.rin2;
        p.rout2 = c.rout2;
        p.shell_mode = c.shell_mode;
        p.exclude_same = c.exclude_same;
        p.swap_out = c.swap_out;
        p.list = c.list;
        p.list_rsq = c.list_rsq;
        p.capacity = c.capacity;
        p.list_count = (unsigned long long *)c.list_count;
        p.frame0 = f0;
        p.nocull = nocull ? 1 : 0;
        if (fast) {
            const double rho = 1.0 / 4194304.0 + 3.5 / 16777216.0, safety = 1.5 * 1.02;
            const double rcd = sqrt(c.rcut2);
            p.f_rc = (float)(rcd * (1.0 + 1e-6));
            p.f_c1 = (float)(safety * sqrt(3.0) / 16777216.0 / c.uniform_ddr);
            p.f_rel = (float)(safety * (c.nbins + 1) * rho);
            p.f_smax = f_smax;
            p.f_rc2t = nextafterf(nextafterf((float)c.rcut2, INFINITY) * (1.0f + 1.0f / 262144.0f), INFINITY);
        }
        MDP_CUDA(cudaMemsetAsync(d_fcount, 0, (size_t)F * 4, st));
        cudaEvent_t tk = ctx->timer_begin(0, st);
        kern<<<ctx->sm_count * ctas_per_sm, NWARP * 32, smem, st>>>(p);
        ctx->timer_end(tk, st);
        MDP_LAUNCHED(ctx);
        rc = mdp_check_launch("k_pair");
        if (rc) return rc;
    }
    return 0;
}

} // namespace

extern "C" {

int mdp_bin_edges(double ddr, int nb, double *edges)
{
    MDP_REQUIRE(ddr > 0 && nb > 0 && edges, "mdp_bin_edges: bad argument");
    // bin(rsq) = (int64)(sqrt(rsq)/ddr) is monotone non-decreasing in rsq (IEEE sqrt and divide are
    // monotone), so the smallest rsq reaching bin k is found by bisection on the (ordered) bit pattern.
    auto bin_of = [ddr](double rsq) -> long long {
        volatile double s = sqrt(rsq);
        volatile double q = s / ddr;
        return (long long)q;
    };
    edges[0] = 0.0;
    for (int k = 1; k <= nb; ++k) {
        uint64_t lo = 0;   // bin(lo) < k   (bin(0) = 0 < k)
        double hi_d = ((double)k * ddr) * ((double)k * ddr) * 1.0000001 + 1e-300;
        while (bin_of(hi_d) < k) hi_d *= 2.0;
        uint64_t hi;
        memcpy(&hi, &hi_d, 8);   // bin(hi) >= k
        while (hi - lo > 1) {
            const uint64_t mid = lo + (hi - lo) / 2;
            double md;
            memcpy(&md, &mid, 8);
            if (bin_of(md) >= k)
                hi = mid;
            else
                lo = mid;
        }
        memcpy(&edges[k], &hi, 8);
    }
    return 0;
}

int mdp_pair_hist(mdp_ctx *ctx, int nframes, int64_t n_a, const double *xyz_a, const int32_t *cls_a, int64_t cls_stride_a,
                  int ncls_a, int64_t n_b, const double *xyz_b, const int32_t *cls_b, int64_t cls_stride_b, int ncls_b,
                  const double *box, double rcut2, const double *edges, int nbins, double uniform_ddr, uint64_t *hist_out,
                  int flags, void *stream)
{
    MDP_REQUIRE(ctx && xyz_a && box && edges && hist_out, "mdp_pair_hist: NULL argument");
    MDP_REQUIRE(nframes > 0 && n_a > 0 && nbins > 0, "mdp_pair_hist: nframes, n_a and nbins must be positive");
    MDP_REQUIRE(n_a < ((int64_t)1 << 30) && n_b < ((int64_t)1 << 30), "mdp_pair_hist: point sets limited to 2^30 points");
    MDP_REQUIRE(ncls_a >= 1 && ncls_a <= MAX_CLS && (xyz_b == nullptr || (ncls_b >= 1 && ncls_b <= MAX_CLS)),
                "mdp_pair_hist: class count must be in [1, %d]", MAX_CLS);
    MDP_REQUIRE(xyz_b == nullptr || n_b > 0, "mdp_pair_hist: n_b must be positive when set B is given");
    MDP_REQUIRE(rcut2 > 0, "mdp_pair_hist: rcut2 must be positive");
    MDP_REQUIRE(uniform_ddr == 0.0 || nbins <= (1 << 18), "mdp_pair_hist: uniform binning limited to 2^18 bins");
    MDP_REQUIRE(uniform_ddr > 0.0 || nbins <= 64, "mdp_pair_hist: table binning limited to 64 thresholds");
    MDP_REQUIRE((flags & ~PAIR_FLAGS) == 0, "mdp_pair_hist: unknown flag bits 0x%x", flags & ~PAIR_FLAGS);
    PairCall c;
    c.mode = uniform_ddr > 0 ? MODE_HIST_UNIFORM : MODE_HIST_TABLE;
    c.nframes = nframes;
    c.n_a = n_a;
    c.xyz_a = xyz_a;
    c.cls_a = cls_a;
    c.cls_stride_a = cls_stride_a;
    c.ncls_a = ncls_a;
    c.n_b = n_b;
    c.xyz_b = xyz_b;
    c.cls_b = cls_b;
    c.cls_stride_b = cls_stride_b;
    c.ncls_b = ncls_b;
    c.box = box;
    c.rcut2 = rcut2;
    c.edges = edges;
    c.nbins = nbins;
    c.uniform_ddr = uniform_ddr;
    c.hist_out = hist_out;
    c.flags = flags;
    return run_pair_call(ctx, c, (cudaStream_t)stream);
}

int mdp_pair_list(mdp_ctx *ctx, int nframes, int64_t n_a, const double *xyz_a, int64_t n_b, const double *xyz_b,
                  const double *box, double rin2, double rout2, int shell_mode, int exclude_same_index, int32_t *list_out,
                  double *rsq_out, int64_t capacity, int64_t *count_out, int flags, void *stream)
{
    MDP_REQUIRE(ctx && xyz_a && xyz_b && box && list_out && count_out, "mdp_pair_list: NULL argument");
    MDP_REQUIRE(nframes > 0 && n_a > 0 && n_b > 0 && capacity > 0, "mdp_pair_list: sizes must be positive");
    MDP_REQUIRE(n_a < ((int64_t)1 << 30) && n_b < ((int64_t)1 << 30), "mdp_pair_list: point sets limited to 2^30 points");
    MDP_REQUIRE(rout2 > 0, "mdp_pair_list: rout2 must be positive");
    MDP_REQUIRE((flags & ~PAIR_FLAGS) == 0, "mdp_pair_list: unknown flag bits 0x%x", flags & ~PAIR_FLAGS);
    PairCall c;
    c.mode = MODE_LIST;
    c.nframes = nframes;
    // The lanes of a warp hold 32 points of set A and stream candidates of set B past them; culling works on the box of
    // those 32 points, so the denser (larger) set belongs on the lanes: 2 000 ions spread over the cell make 30 A boxes
    // that touch everything, 60 000 solvent atoms make 10 A boxes.  Swapping the roles only swaps the output columns.
    const bool swap = n_a < n_b;
    c.swap_out = swap ? 1 : 0;
    c.n_a = swap ? n_b : n_a;
    c.xyz_a = swap ? xyz_b : xyz_a;
    c.n_b = swap ? n_a : n_b;
    c.xyz_b = swap ? xyz_a : xyz_b;
    c.box = box;
    // pre-filter must pass rsq <= rout2 too: use the next double above rout2 as the strict cutoff
    c.rcut2 = nextafter(rout2, INFINITY);
    c.rin2 = rin2;
    c.rout2 = rout2;
    c.shell_mode = shell_mode;
    c.exclude_same = exclude_same_index;
    c.list = list_out;
    c.list_rsq = rsq_out;
    c.capacity = capacity;
    c.list_count = count_out;
    c.flags = flags;
    return run_pair_call(ctx, c, (cudaStream_t)stream);
}

int mdp_hist_reduce(mdp_ctx *ctx, int nframes, int rows, int nbins, const uint64_t *hist, int nout, const int32_t *weights,
                    int cumulative, uint64_t *out, void *stream)
{
    MDP_REQUIRE(ctx && hist && weights && out, "mdp_hist_reduce: NULL argument");
    MDP_REQUIRE(nframes > 0 && rows > 0 && nbins > 0 && nout > 0, "mdp_hist_reduce: sizes must be positive");
    cudaStream_t st = (cudaStream_t)stream;
    MDP_CUDA(cudaSetDevice(ctx->device));
    int rc = ctx->arena_reserve((size_t)nout * rows * 4 + 4096);
    if (rc) return rc;
    ctx->arena_reset();
    int *d_w = (int *)ctx->arena_take((size_t)nout * rows * 4);
    MDP_CUDA(cudaMemcpyAsync(d_w, weights, (size_t)nout * rows * 4, cudaMemcpyHostToDevice, st));
    dim3 g(nout, nframes);
    k_hist_reduce<<<g, 256, 0, st>>>((const unsigned long long *)hist, rows, nbins, nout, d_w, cumulative,
                                     (unsigned long long *)out);
    MDP_LAUNCHED(ctx);
    return mdp_check_launch("k_hist_reduce");
}

} // extern "C"
