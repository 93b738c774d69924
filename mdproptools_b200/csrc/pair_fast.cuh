// pair_fast.cuh -- the uniform-bin histogram kernel of the pair engine: fp32 classification, fp64 only where it decides.
// Included by pair.cu (shares its records, boxes, work list and PairParams).
//
// What the reference computes per pair (rdf_cn.py:46-68, 85): rsq in unfused fp64, then bin = int64(sqrt(rsq) / ddr).
// Only the INTEGER bin reaches the result.  The fp64 kernel k_pair pays the whole fp64 chain (8-14 ops on the FP64 pipe
// + F2F + an fp64 edge compare from shared memory) for every evaluated pair although for all but a few pairs in ten
// thousand the bin is already decided by a distance known to six digits.  k_pair_fast therefore
//   1. expresses the j candidates of one i group (32 points, one per lane) RELATIVE TO THE GROUP'S BOX CENTRE, image shift
//      applied, as fp32 (the subtraction and the shift are done in fp64 BEFORE the single rounding to fp32, so the fp32
//      values are small -- |j_rel| <= half extent + r_cut -- and carry an absolute error of ~1e-6 A);
//   2. evaluates d^2 in fp32 (3 FADD + FMUL + 2 FFMA), x = sqrt(d^2) * 2^s / ddr with MUFU.SQRT and one FFMA.RM that
//      also floors (2^23 trick), so that one integer Y = floor(x * 2^s) + 1 holds the bin (Y >> s) and s fraction bits;
//      the FP32 operations run two candidates at a time as packed FP32x2 instructions (FADD2, FMUL2, FFMA2), each half
//      rounded exactly as the scalar operation, so nothing below depends on the packing;
//   3. increments histogram word (Y >> s) unconditionally (misses are clamped to a per-lane scratch word behind the row,
//      as in k_pair), and flags the pair as UNDECIDED when the fraction bits are all zero or all one, i.e. when x is
//      within 2^-s of a bin edge.  s is chosen per unit from a rigorous bound E on |x_fp32 - x_exact| (below) such that
//      2^-s >= 1.5 E: an unflagged pair is provably in the reference's bin;
//   4. undecided pairs (about 1 in 1000) go to a per-warp queue and are settled by the exact path: the reference's own
//      fp64 arithmetic (image_r2, the code k_pair uses) on the fp64 records, the exact edge table (mdp_bin_edges), and
//      a correction -1/+1 of the shared histogram when the exact bin differs from the one already incremented.
// Counts are therefore bit-identical to k_pair's and to the reference's; tests/test_gpu_parity.py runs both kernels
// against the oracle (pairs planted exactly on bin edges and on the cutoff included).
//
// Error bound (per axis k, all quantities in A).  g = centre of the i group's box, ext = its half extent, S = image shift of
// the chunk pair (0, +-l, or the triclinic image vector), both subtractions in fp64 (relative error 2^-53, ignored
// against 2^-24 but covered by the 1.5 safety factor):
//   i_rel = fl32(X_i - g)            |err| <= 2^-24 |i_rel|        <= 2^-24 ext
//   j_rel = fl32(X_j + S - g)        |err| <= 2^-24 |j_rel|        <= 2^-24 (ext + rc)    (the point filter keeps only such j)
//   d     = fl32(i_rel - j_rel)      |err| <= 2^-24 |d|            <= 2^-24 (2 ext + rc)
// so |d_fp32 - d_exact| <= 2^-24 (4 ext + 2 rc) =: delta, and | ||d_fp32|| - ||d_exact|| | <= sqrt(3) delta.  The sum of
// squares (FMUL, FFMA, FFMA: all terms positive) has relative error <= 3 * 2^-24, MUFU.SQRT <= 2^-22 (PTX documents
// 2^-23 for sqrt.approx.f32; tools/peaks.cu checks every fp32 input on the device), fl32(2^s/ddr) 2^-24; the FFMA.RM
// is exact.  Together, in units of bins,  E = (nbins + 1) * RHO + sqrt(3) * delta / ddr,  RHO = 2^-22 + 3.5 * 2^-24.
// Chunk pairs whose image is not uniform (small cells) take the MIXED variant: j is NOT shifted, the loop computes
// min(|d|, ||d| - l|) per axis (the magnitude of the reference's single shift for every d, see AX_MIXED in pair.cu) and
// delta = 2^-24 (4 l + 6 ext + 3 rc).  Triclinic chunk pairs without a single image vector are evaluated in fp64
// outright (the image decision is discontinuous there).
#pragma once

namespace {

#ifndef MDP_FAST_CTAS
#define MDP_FAST_CTAS 3
#endif
constexpr int FAST_CTAS_PER_SM = MDP_FAST_CTAS;
#ifndef MDP_FAST_UNROLL
#define MDP_FAST_UNROLL 4
#endif
constexpr int FU = MDP_FAST_UNROLL;           // candidates per round of the pair loop (ring runs are padded to a multiple of it)
static_assert(FU % 2 == 0, "the pair loop evaluates candidates two at a time");
constexpr int FRING = 64;                     // candidate ring: 16-byte entries per warp
constexpr int FQ_CAP = 64;                    // undecided-pair queue: entries per warp
constexpr unsigned FMAGIC_BITS = 0x4b400000u; // bits of 12582912.0f = 1.5 * 2^23
constexpr float FAST_PAD = 1.0e18f;           // coordinate of a padding candidate: d^2 = 1e36 stays finite, bin clamps to a miss
constexpr unsigned FAST_PADMETA = 0xffffffc0u; // w of a padding candidate: class bits 0 (a valid row lookup), position all ones
constexpr int FAST_XROW = 32;                 // scratch words behind every histogram row (one per lane, for misses)
constexpr unsigned FAST_FLUSH_EVALS = 1u << 30;   // a CTA re-bases its uint32 histogram after this many evaluated pairs

struct FastBin {
    float inv_s;       // 2^s / ddr
    unsigned mask;     // 2^s - 2 (0: every pair takes the exact path)
    unsigned clampv;   // FMAGIC_BITS + (((nbins + lane) << s) | 2): misses land on word nbins + lane and are never flagged
    unsigned base;     // hist_a - ((FMAGIC_BITS >> s) << 2): base + ((bits >> s) << 2) is the byte address of the bin word
    int s;
};

__device__ __forceinline__ FastBin make_fastbin(float e15, int smax, float inv_ddr, unsigned nb, int lane, unsigned hist_a)
{
    // largest s with 2^-s >= e15 (e15 = m * 2^e, 1 <= m < 2  ->  s = -e - 1), clamped to [1, smax]; s = 1 gives mask 0
    const int e = (int)((__float_as_uint(e15) >> 23) & 255u) - 127;
    int s = -e - 1;
    s = s < 1 ? 1 : (s > smax ? smax : s);
    FastBin fb;
    fb.s = s;
    fb.inv_s = inv_ddr * (float)(1u << s);
    fb.mask = (1u << s) - 2u;
    fb.clampv = FMAGIC_BITS + (((nb + (unsigned)lane) << s) | 2u);
    fb.base = hist_a - ((FMAGIC_BITS >> s) << 2);
    return fb;
}

// per-axis class of a chunk pair in the orthogonal (reference) image, d = a - b:
//   0 every pair has |d| <= l/2; 1 every pair has d > l/2 (j is shifted by +l); 2 every pair has d < -l/2 (j shifted by
//   -l); 3 undecided.  Returns the lower bound of the wrapped |d| (rounded towards "keep").
__device__ __forceinline__ float axis_class_f32(float alo, float ahi, float blo, float bhi, const AxisF &ax, int &cls)
{
    const float dlo = __fsub_rd(alo, bhi), dhi = __fsub_ru(ahi, blo);
    float best = 3.0e38f;
    if (dlo > ax.h_up) {
        cls = 1;
        best = interval_min_abs(__fsub_rd(dlo, ax.l_up), __fsub_ru(dhi, ax.l_dn));
    } else if (dhi < -ax.h_up) {
        cls = 2;
        best = interval_min_abs(__fadd_rd(dlo, ax.l_dn), __fadd_ru(dhi, ax.l_up));
    } else {
        const bool may_plus = dhi > ax.h_dn, may_minus = dlo < -ax.h_dn;
        cls = (may_plus || may_minus) ? 3 : 0;
        {
            const float lo = fmaxf(dlo, -ax.h_up), hi = fminf(dhi, ax.h_up);
            if (lo <= hi) best = interval_min_abs(lo, hi);
        }
        if (may_plus) best = fminf(best, interval_min_abs(__fsub_rd(fmaxf(dlo, ax.h_dn), ax.l_up), __fsub_ru(dhi, ax.l_dn)));
        if (may_minus) best = fminf(best, interval_min_abs(__fadd_rd(dlo, ax.l_dn), __fadd_ru(fminf(dhi, -ax.h_dn), ax.l_up)));
    }
    return best;
}

__device__ __forceinline__ bool chunk_class_f32(const float *a, const float *b, const AxisF &X, const AxisF &Y, const AxisF &Z,
                                                float rcut2_up, int &code)
{
    code = 0;
    if (a[0] > a[3] || b[0] > b[3]) return false;   // empty box (padding only)
    int cx, cy, cz;
    const float bx = axis_class_f32(a[0], a[3], b[0], b[3], X, cx);
    const float by = axis_class_f32(a[1], a[4], b[1], b[4], Y, cy);
    const float bz = axis_class_f32(a[2], a[5], b[2], b[5], Z, cz);
    code = cx | (cy << 2) | (cz << 4);
    const float lb = __fadd_rd(__fadd_rd(__fmul_rd(bx, bx), __fmul_rd(by, by)), __fmul_rd(bz, bz));
    return lb < rcut2_up;
}

// lower bound of the wrapped distance of a point at distance a >= 0 from the box centre (half extent e, already inflated)
// under min(|d|, ||d| - l|): the raw |d| ranges over [a - e, a + e]
__device__ __forceinline__ float mixed_axis_lb(float a, float e, float l_dn, float l_up)
{
    const float lo = a - e, hi = a + e;
    const float lb1 = fmaxf(lo, 0.f);
    const float lb2 = fmaxf(fmaxf(l_dn - hi, lo - l_up), 0.f);
    return fminf(lb1, lb2);
}

// ---- shared-memory layout ----------------------------------------------------------------------------------------------
// per warp:  ring   float[FRING][4]      candidates (x, y, z relative to the group centre, w = sorted j position [<< 6 | class]),
//                                        interleaved in pairs (ring_put)
//            xq     uint2[FQ_CAP]        undecided pairs: (w of the candidate, lane << 16 | bin already incremented)
//            jst    double2[2][64]       two staged j chunks (1 KB each, filled by cp.async one chunk ahead of their use)
//            gs     double[3][3]         g - S for the three uniform image classes of each axis (0: none, 1: j + l, 2: j - l);
//                   double[27][3]        triclinic: g - S for the 27 image vectors (index ex + 3 ey + 9 ez, e = 0 / 1 / 2 for k = 0 / +1 / -1)
//            ga     float[8]             box of the i group (lo.xyz, -, hi.xyz, -), for the chunk-level test
// per CTA:   fc     FrameConst           box lengths of the current frame in the forms the tests need
//            cptab, evals, totals, hist
constexpr size_t FW_RING = 0, FW_XQ = FW_RING + FRING * 16, FW_JST = FW_XQ + FQ_CAP * 8, FW_GS = FW_JST + 2 * 1024,
                 FW_GA = FW_GS + 656, FAST_WARP_BYTES = FW_GA + 32;
static_assert(FAST_WARP_BYTES % 16 == 0, "warp region must keep 16-byte alignment");

struct FrameConst {
    float ax[3][4];        // per axis: l_dn, l_up, h_dn, h_up   (read as float4: keep at offset 0, 16-byte aligned)
    float l32[3];          // fl32(l): the MIXED variant's shift
    float lmax_up;
    double cell[6];        // lx, ly, lz, xy, xz, yz
    const double2 *rB;     // records of set B of the current frame (kept here: the pointer is needed once per chunk, and
                           // re-deriving it from the parameter block costs a 64-bit multiply chain in an issue-bound loop)
};

struct FastShared {
    unsigned hist_a, cptab_a;
    unsigned *hist;
    const unsigned *cptab;       // MULTICLS: byte offset of the histogram row of class pair (ci * nclsB + cj)
};

// The candidate ring is interleaved in pairs: candidate c is half (c & 1) of the 32-byte block c >> 1, laid out
// {x0, x1, y0, y1}{z0, z1, w0, w1}.  Two LDS.128 then hand the pair loop each coordinate of two candidates as one register
// pair, the operand of the packed FP32x2 instructions (one float4 per candidate would need a MOV per coordinate to pair
// them).  These three functions are the only code that knows the layout.
__device__ __forceinline__ void ring_put(float *ring, int c, float x, float y, float z, unsigned w)
{
    float *e = ring + (c >> 1) * 8 + (c & 1);
    e[0] = x;
    e[2] = y;
    e[4] = z;
    e[6] = __uint_as_float(w);
}

// candidates c and c + 1 (c even) of the run at shared address ja
__device__ __forceinline__ void ring_get2(unsigned ja, int c, float2 &x, float2 &y, float2 &z, uint2 &w)
{
    const unsigned a = ja + (unsigned)(c >> 1) * 32u;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(y.x), "=f"(y.y) : "r"(a));
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=f"(z.x), "=f"(z.y), "=r"(w.x), "=r"(w.y) : "r"(a + 16u));
}

// shared address of the w of candidate c of the run at ja
__device__ __forceinline__ unsigned ring_w_addr(unsigned ja, int c)
{
    return ja + (unsigned)(c >> 1) * 32u + 24u + (unsigned)(c & 1) * 4u;
}

__device__ __forceinline__ void pf_mbar_init(unsigned bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void pf_mbar_expect_tx(unsigned bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void pf_mbar_wait(unsigned bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void pf_bulk_g2s(unsigned dst, const void *src, unsigned bytes, unsigned bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar) : "memory");
}

// the exact path: settle the queued pairs with the reference's arithmetic and correct the shared histogram.
// rAg = records of my i group (the i point of an entry is re-read from them: lane index in the entry)
// (scalar arguments only: a struct, or the kernel's parameter block, passed by address to an out-of-line function would
// force it -- and with it much of the caller's loop state -- into local memory)
template <bool MULTICLS, bool TRICL>
__device__ __noinline__ void fast_settle(int nb, const double2 *__restrict__ edges2, int nclsB, unsigned *hist, const unsigned *cptab,
                                         int lane, int qn, const uint2 *xq, const double2 *__restrict__ rAg,
                                         const double2 *__restrict__ rB, const double *cell)
{
    const double lx = cell[0], ly = cell[1], lz = cell[2];
    const Shift S = {lx, ly, lz, TRICL ? cell[3] : 0.0, TRICL ? cell[4] : 0.0, TRICL ? cell[5] : 0.0};
    const double hx = lx * 0.5, hy = ly * 0.5, hz = lz * 0.5;
    for (int b0 = lane; b0 < qn; b0 += 32) {
        const uint2 e = xq[b0];
        const int il = (int)(e.y >> 16);
        const int ka = (int)(e.y & 0xffffu);
        const double2 ixy = rAg[il], izw = rAg[32 + il];
        const uint32_t jpos = MULTICLS ? (e.x >> 6) : e.x;
        const double2 jxy = rB[rec_xy((int64_t)jpos)], jzw = rB[rec_zw((int64_t)jpos)];
        const double r2 = TRICL ? image_r2<VAR_TMIXED>(__dsub_rn(ixy.x, jxy.x), __dsub_rn(ixy.y, jxy.y), __dsub_rn(izw.x, jzw.x), S, hx, hy, hz)
                                : image_r2<VAR_MIXED>(__dsub_rn(ixy.x, jxy.x), __dsub_rn(ixy.y, jxy.y), __dsub_rn(izw.x, jzw.x), S, hx, hy, hz);
        // exact bin: bin(rsq) >= k  <=>  rsq >= edge[k] (mdp_bin_edges); edges2[k] = {edge[k], edge[k+1]}, edge[nb+1] = +inf
        int k = ka < nb ? ka : nb;
        while (k < nb && r2 >= edges2[k].y) ++k;
        while (k > 0 && r2 < edges2[k].x) --k;
        if (k != ka) {
            const unsigned row = MULTICLS ? cptab[(uint32_t)(__double2loint(izw.y) * nclsB) + (e.x & 63u)] : 0u;   // byte offset
            unsigned *h = hist + (row >> 2);
            if (ka < nb) atomicSub(&h[ka], 1u);
            if (k < nb) atomicAdd(&h[k], 1u);
        }
    }
    __syncwarp();
}

// every pair of one 32 x 32 chunk pair in fp64 (triclinic chunk pairs without a single image vector): lane = i point
template <bool MULTICLS>
__device__ __noinline__ void fast_exact_chunk(int nb, const double2 *__restrict__ edges2, int nclsB, double rcut2, float inv_ddr,
                                              unsigned *hist, const unsigned *cptab, int lane, double jx_, double jy_, double jz_,
                                              double jm_, bool tri, const double2 *__restrict__ rAg, const double *cell)
{
    const Shift S = {cell[0], cell[1], cell[2], cell[3], cell[4], cell[5]};
    const double hx = cell[0] * 0.5, hy = cell[1] * 0.5, hz = cell[2] * 0.5;
    const double2 jxy = make_double2(jx_, jy_), jzw = make_double2(jz_, jm_);
    const double2 ixy = rAg[lane], izw = rAg[32 + lane];
    const bool ipad = __double2hiint(izw.y) < 0;
    const uint32_t mi = (uint32_t)(__double2loint(izw.y) * nclsB);
#pragma unroll 1
    for (int jj = 0; jj < 32; ++jj) {
        const double bx = __shfl_sync(0xffffffffu, jxy.x, jj), by = __shfl_sync(0xffffffffu, jxy.y, jj);
        const double bz = __shfl_sync(0xffffffffu, jzw.x, jj), bm = __shfl_sync(0xffffffffu, jzw.y, jj);
        if (__double2hiint(bm) < 0 || ipad) continue;        // padding point
        if (tri && jj <= lane) continue;
        const double r2 = image_r2<VAR_TMIXED>(__dsub_rn(ixy.x, bx), __dsub_rn(ixy.y, by), __dsub_rn(izw.x, bz), S, hx, hy, hz);
        if (!(r2 < rcut2)) continue;
        float sq;
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(__double2float_rz(r2)));
        int k = (int)(sq * inv_ddr);
        k = k < 0 ? 0 : (k > nb ? nb : k);
        while (k < nb && r2 >= edges2[k].y) ++k;
        while (k > 0 && r2 < edges2[k].x) --k;
        if (k < nb) {
            const unsigned row = MULTICLS ? cptab[mi + (uint32_t)__double2loint(bm)] : 0u;
            atomicAdd(&hist[(row >> 2) + k], 1u);
        }
    }
}

// triclinic chunk-level test, out of line (scalar arguments): its 27-image enumeration needs ~40 registers of its own, which
// inlined would be taken from the pair loop of the whole kernel.  Returns code | need << 8.
__device__ __noinline__ int fast_tri_chunk_test(float a0, float a1, float a2, float a3, float a4, float a5, float b0, float b1, float b2,
                                                float b3, float b4, float b5, const double *cell, float rcut2_up)
{
    const float a[6] = {a0, a1, a2, a3, a4, a5}, b[6] = {b0, b1, b2, b3, b4, b5};
    TriConst<DirF32> TC;
    TC.set(cell);
    int code = 0;
    const bool need = tri_box_test<DirF32>(a, b, TC, rcut2_up, code);
    return code | (need ? 256 : 0);
}

struct FastExact {              // what the exact path needs (per unit); all warp-uniform
    const double2 *rAg, *rB, *edges2;
    const double *cell;
    unsigned *hist;
    const unsigned *cptab;
    int nb, nclsB;
};

struct FastRunP {               // per-unit constants of the pair loop
    float inv_s;                // 2^s / ddr
    unsigned mask, clampv, base;
    int s;
    unsigned cptab_mi_a;        // shared address of my class's row of the class-pair table (MULTICLS)
    float xi, yi, zi;           // my i point relative to the group centre
};

// nj (a multiple of FU) queued candidates at shared address ja against my i point.  MIXED: min(|d|, ||d| - l|) per axis on
// unshifted candidates (l32*).  TRI: the self chunk, only j > lane counts.
template <bool MULTICLS, bool TRICL, bool MIXED, bool TRI>
__device__ __forceinline__ void fast_run(const FastRunP &R, const FastExact &ex, const unsigned ja, const int nj,
                                         const float l32x, const float l32y, const float l32z, const int lane, int &qn, uint2 *xq,
                                         unsigned &uex)
{
    const float2 xi = make_float2(R.xi, R.xi), yi = make_float2(R.yi, R.yi), zi = make_float2(R.zi, R.zi);
    const float2 inv_s = make_float2(R.inv_s, R.inv_s), magic = make_float2(12582913.0f, 12582913.0f);
    const unsigned mask = R.mask, clampv = R.clampv, base = R.base;
    const int s = R.s;
    const auto wrap = [](float d, float l) { return fminf(fabsf(d), fabsf(fabsf(d) - l)); };
#pragma unroll 1
    for (int j0 = 0; j0 < nj; j0 += FU) {
        unsigned b[FU];
        bool unc = false;
        float2 jx[FU / 2], jy[FU / 2], jz[FU / 2];
        uint2 jm[FU / 2];
        // all candidates of the round first (back-to-back loads, nothing depends on the previous one), then the arithmetic
#pragma unroll
        for (int k = 0; k < FU / 2; ++k) ring_get2(ja, j0 + 2 * k, jx[k], jy[k], jz[k], jm[k]);
        // candidates 2k and 2k + 1 share every FP32 instruction; each half is the scalar operation with its rounding, so Y,
        // the histogram word and the undecided flag of every pair are what scalar code computes
#pragma unroll
        for (int k = 0; k < FU / 2; ++k) {
            float2 dx = __fadd2_rn(xi, make_float2(-jx[k].x, -jx[k].y)), dy = __fadd2_rn(yi, make_float2(-jy[k].x, -jy[k].y)),
                   dz = __fadd2_rn(zi, make_float2(-jz[k].x, -jz[k].y));
            if (MIXED) {
                dx = make_float2(wrap(dx.x, l32x), wrap(dx.y, l32x));
                dy = make_float2(wrap(dy.x, l32y), wrap(dy.y, l32y));
                dz = make_float2(wrap(dz.x, l32z), wrap(dz.y, l32z));
            }
            float2 r2 = __ffma2_rn(dz, dz, __ffma2_rn(dy, dy, __fmul2_rn(dx, dx)));
            if (TRI) {
                r2.x = (j0 + 2 * k > lane) ? r2.x : 1.0e36f;
                r2.y = (j0 + 2 * k + 1 > lane) ? r2.y : 1.0e36f;
            }
            float2 sq;
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq.x) : "f"(r2.x));
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq.y) : "f"(r2.y));
            const float2 y = __ffma2_rd(sq, inv_s, magic);   // FMAGIC_BITS + floor(x * 2^s) + 1
            unsigned v0 = __float_as_uint(y.x), v1 = __float_as_uint(y.y);
            v0 = v0 < clampv ? v0 : clampv;
            v1 = v1 < clampv ? v1 : clampv;
            b[2 * k] = v0;
            b[2 * k + 1] = v1;
            unc = unc || ((v0 & mask) == 0u) || ((v1 & mask) == 0u);
        }
#pragma unroll
        for (int u = 0; u < FU; ++u) {
            unsigned a = base + ((b[u] >> s) << 2);
            if (MULTICLS) {
                const unsigned w = (u & 1) ? jm[u / 2].y : jm[u / 2].x;
                unsigned row;
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(row) : "r"(R.cptab_mi_a + ((w & 63u) << 2)));
                a += row;
            }
            asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(a) : "memory");
        }
        if (__any_sync(0xffffffffu, unc)) {
            const unsigned lt = (1u << lane) - 1u;
#pragma unroll
            for (int u = 0; u < FU; ++u) {   // unrolled: b[] stays in registers; the candidate's w is re-read from the ring
                unsigned jm;
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(jm) : "r"(ring_w_addr(ja, j0 + u)));
                bool f = (b[u] & mask) == 0u && jm < FAST_PADMETA;
                if (TRI) f = f && (j0 + u > lane);
                const unsigned m = __ballot_sync(0xffffffffu, f);
                if (m == 0u) continue;
                const int c = __popc(m);
                if (qn + c > FQ_CAP) {
                    __syncwarp();
                    uex += (unsigned)qn;
                    fast_settle<MULTICLS, TRICL>(ex.nb, ex.edges2, ex.nclsB, ex.hist, ex.cptab, lane, qn, xq, ex.rAg, ex.rB, ex.cell);
                    qn = 0;
                }
                if (f) xq[qn + __popc(m & lt)] = make_uint2(jm, ((unsigned)lane << 16) | ((b[u] >> s) - (FMAGIC_BITS >> s)));
                qn += c;
            }
        }
    }
}

// the ring holds n pending candidates from `base`: pad to a multiple of FU and evaluate them (uniform-image variant)
template <bool MULTICLS, bool TRICL>
__device__ __forceinline__ void fast_flush(const FastRunP &R, const FastExact &ex, float *ring, unsigned ring_a, int head, int tail,
                                           int lane, int &qn, uint2 *xq, unsigned &uex)
{
    const int n = tail - head;
    const int np = (n + FU - 1) & ~(FU - 1);
    if (lane < np - n) ring_put(ring, (tail + lane) & (FRING - 1), FAST_PAD, 0.f, 0.f, FAST_PADMETA);
    __syncwarp();
    fast_run<MULTICLS, TRICL, false, false>(R, ex, ring_a + (unsigned)(head & 32) * 16u, np, 0.f, 0.f, 0.f, lane, qn, xq, uex);
    __syncwarp();
}

// A chunk that is not the common case -- the triangular self chunk, or (orthogonal cells) a chunk pair whose image is not
// uniform -- after the ring has been flushed: filter (not for the self chunk), compact into ring[0..], evaluate at once.
// (jx, jy, jz) = my j point relative to the centre, unshifted when `mixed`.  Returns the 32-pair steps evaluated.
template <bool MULTICLS, bool TRICL>
__device__ __forceinline__ unsigned fast_special(int f_smax, float inv_ddr, const FastRunP &R, const FastExact &ex, const FrameConst *fc,
                                                 float *ring, unsigned ring_a, float jx, float jy, float jz, unsigned jmeta, bool self,
                                                 bool mixed, float extx, float exty, float extz, float rc2t, float e15m,
                                                 unsigned hist_a, int lane, int &qn, uint2 *xq, unsigned &uex)
{
    int n = 32;
    if (self) {
        ring_put(ring, lane, jx, jy, jz, jmeta);
    } else {
        const float bx = mixed_axis_lb(fabsf(jx), extx, fc->ax[0][0], fc->ax[0][1]), by = mixed_axis_lb(fabsf(jy), exty, fc->ax[1][0], fc->ax[1][1]),
                    bz = mixed_axis_lb(fabsf(jz), extz, fc->ax[2][0], fc->ax[2][1]);
        const bool ok = __fmaf_rn(bz, bz, __fmaf_rn(by, by, bx * bx)) < rc2t && jmeta < FAST_PADMETA;
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (ok) ring_put(ring, __popc(m & ((1u << lane) - 1u)), jx, jy, jz, jmeta);
        const int c = __popc(m);
        n = (c + FU - 1) & ~(FU - 1);
        if (lane < n - c) ring_put(ring, c + lane, FAST_PAD, 0.f, 0.f, FAST_PADMETA);
    }
    __syncwarp();
    if (n > 0) {
        if (!mixed) {
            fast_run<MULTICLS, TRICL, false, true>(R, ex, ring_a, n, 0.f, 0.f, 0.f, lane, qn, xq, uex);    // (only the self chunk gets here)
        } else if (!TRICL) {
            const FastBin fbM = make_fastbin(e15m, f_smax, inv_ddr, (unsigned)ex.nb, lane, hist_a);
            FastRunP RM = R;
            RM.inv_s = fbM.inv_s;
            RM.mask = fbM.mask;
            RM.clampv = fbM.clampv;
            RM.base = fbM.base;
            RM.s = fbM.s;
            if (self)
                fast_run<MULTICLS, TRICL, true, true>(RM, ex, ring_a, n, fc->l32[0], fc->l32[1], fc->l32[2], lane, qn, xq, uex);
            else
                fast_run<MULTICLS, TRICL, true, false>(RM, ex, ring_a, n, fc->l32[0], fc->l32[1], fc->l32[2], lane, qn, xq, uex);
        }
    }
    __syncwarp();
    return (unsigned)n;
}

template <bool MULTICLS, bool SYMM, bool TRICL, int NCTA>
__global__ void __launch_bounds__(NWARP * 32, NCTA) k_pair_fast(const PairParams p)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    unsigned char *wp = smem_raw + (size_t)(threadIdx.x >> 5) * FAST_WARP_BYTES;
    float *ring = reinterpret_cast<float *>(wp + FW_RING);
    uint2 *xq = reinterpret_cast<uint2 *>(wp + FW_XQ);
    double *gs = reinterpret_cast<double *>(wp + FW_GS);
    float4 *gas = reinterpret_cast<float4 *>(wp + FW_GA);
    const unsigned wp_a = (unsigned)__cvta_generic_to_shared(wp);
    unsigned char *sp = smem_raw + (size_t)NWARP * FAST_WARP_BYTES;
    FrameConst *fc = reinterpret_cast<FrameConst *>(sp);
    sp += (sizeof(FrameConst) + 15) & ~(size_t)15;
    unsigned *cptab_s = reinterpret_cast<unsigned *>(sp);
    if (MULTICLS) sp += (size_t)((p.ncp * 4 + 15) & ~15);
    unsigned *evals_s = reinterpret_cast<unsigned *>(sp);                         // 32-pair steps since the histogram was last re-based
    unsigned long long *tot_s = reinterpret_cast<unsigned long long *>(sp + 8);   // [2]: 32-pair steps, exact-path pairs of this CTA
    sp += 32;
    unsigned *hist = reinterpret_cast<unsigned *>(sp);
    const unsigned hist_a = (unsigned)__cvta_generic_to_shared(hist);
    const unsigned cptab_a = (unsigned)__cvta_generic_to_shared(cptab_s);
    const int nb = p.nbins;
    const int rowstride = nb + FAST_XROW;
    const int nwords = p.nrows * rowstride;
    for (int k = threadIdx.x; k < nwords; k += blockDim.x) hist[k] = 0u;
    if (MULTICLS)
        for (int k = threadIdx.x; k < p.ncp; k += blockDim.x) cptab_s[k] = (unsigned)(p.cptab[k] * rowstride) * 4u;
    if (threadIdx.x == 0) {
        *evals_s = 0u;
        tot_s[0] = 0ull;
        tot_s[1] = 0ull;
    }
    int qn = 0;
    const float rcut2_up = __double2float_ru(p.rcut2);
    const float rc2t = p.f_rc2t;   // point filter threshold: rcut2 rounded up x (1 + 2^-18), covers the fp32 rounding of its own sums
    const int F = p.nframes;
    const int fstart = (int)(((long long)blockIdx.x * F) / gridDim.x);
    const unsigned int nunits = (unsigned int)p.ntA * GPT;

    // flush = re-base: every word is exchanged for 0 and added to the frame's global histogram as a SIGNED 32-bit value
    // (a correction of the exact path may arrive after the word it corrects was flushed), so it needs no barrier and
    // any warp may do it at any time
    auto flush_words = [&](int frame, int k0, int kstep) {
        unsigned long long *hg = p.hist + (int64_t)frame * p.nrows * nb;
        for (int k = k0; k < nwords; k += kstep) {
            const int r = k / rowstride, c = k - r * rowstride;
            if (c >= nb) continue;
            const unsigned v = atomicExch(&hist[k], 0u);
            if (v) atomicAdd(&hg[(int64_t)r * nb + c], (unsigned long long)(long long)(int)v);
        }
    };

#pragma unroll 1
    for (int fk = 0; fk < F; ++fk) {
        int f = fstart + fk;
        if (f >= F) f -= F;
        const double *cell = p.box + f * 6;
        // frame constants -> shared memory (everybody is past the previous frame: barrier at its end)
        if (threadIdx.x < 3) {
            const int a = threadIdx.x;
            const AxisF A = make_axis(cell[a]);
            fc->ax[a][0] = A.l_dn;
            fc->ax[a][1] = A.l_up;
            fc->ax[a][2] = A.h_dn;
            fc->ax[a][3] = A.h_up;
            fc->l32[a] = __double2float_rn(cell[a]);
        } else if (threadIdx.x < 9) {
            fc->cell[threadIdx.x - 3] = cell[threadIdx.x - 3];
        } else if (threadIdx.x == 9) {
            fc->lmax_up = __double2float_ru(fmax(fmax(cell[0], cell[1]), cell[2]));
            fc->rB = p.recB + (int64_t)f * p.npadB * 2;
        }
        __syncthreads();
        const int frame = p.frame0 + f;
        const double2 *rA = p.recA + (int64_t)f * p.npadA * 2;
        const double2 *rB = p.recB + (int64_t)f * p.npadB * 2;
        const float4 *gbB = p.gboxB + (int64_t)f * p.ngB * 2;
        bool did = false;

        unsigned int q = 0;
        if (lane == 0) q = atomicAdd(&p.counters[f], 1u);
        q = __shfl_sync(0xffffffffu, q, 0);
#pragma unroll 1
        while (q < nunits) {
            unsigned int qnext = 0;
            if (lane == 0) qnext = atomicAdd(&p.counters[f], 1u);   // prefetch the next work index
            did = true;
            unsigned uev = 0, uex = 0;                              // this unit: 32-pair steps evaluated, pairs settled in fp64
            const int ta = (int)(q >> 3), wi = (int)(q & 7u);
            const int64_t row = (int64_t)f * p.ntA + ta;
            unsigned int t0 = p.rowoff[row];
            const unsigned int tend = row + 1 < (int64_t)F * p.ntA ? p.rowoff[row + 1] : (unsigned int)*p.total;
            const int64_t gi = (int64_t)ta * GPT + wi;
            FastExact ex;
            ex.rAg = rA + gi * GREC;
            ex.rB = rB;
            ex.cell = cell;
            ex.hist = hist;
            ex.cptab = cptab_s;
            ex.edges2 = p.edges2;
            ex.nb = nb;
            ex.nclsB = p.nclsB;
            FastRunP R;
            R.cptab_mi_a = cptab_a;
            float extx, exty, extz;
            float e15m;                                              // error bound of the MIXED variant (its bins are made on demand)
            {
                const float4 *ga4 = p.gboxA + ((int64_t)f * p.ngA + gi) * 2;
                const float4 alo = ga4[0], ahi = ga4[1];
                const bool iempty = alo.x > ahi.x;                    // a group of padding only
                // group centre (exact in fp64) and half extents, rounded up and inflated by the rounding of the filter's own
                // arithmetic (2^-21 (ext + rc) >> 2^-24 |j_rel| + 2^-24 | |j_rel| - ext |)
                const float gcx = iempty ? 0.f : 0.5f * alo.x + 0.5f * ahi.x, gcy = iempty ? 0.f : 0.5f * alo.y + 0.5f * ahi.y,
                            gcz = iempty ? 0.f : 0.5f * alo.z + 0.5f * ahi.z;
                float ex_ = fmaxf(__fsub_ru(ahi.x, gcx), __fsub_ru(gcx, alo.x)), ey_ = fmaxf(__fsub_ru(ahi.y, gcy), __fsub_ru(gcy, alo.y)),
                      ez_ = fmaxf(__fsub_ru(ahi.z, gcz), __fsub_ru(gcz, alo.z));
                if (iempty) ex_ = ey_ = ez_ = 0.f;
                const float extm = fmaxf(fmaxf(ex_, ey_), ez_);
                const float infl = 1.0f / 2097152.0f;
                extx = __fmaf_ru(infl, ex_ + p.f_rc, ex_);
                exty = __fmaf_ru(infl, ey_ + p.f_rc, ey_);
                extz = __fmaf_ru(infl, ez_ + p.f_rc, ez_);
                __syncwarp();                                        // the previous unit's readers of gs / ga are done
                if (lane == 0) {
                    gas[0] = alo;
                    gas[1] = ahi;
                }
                if (TRICL) {
                    if (lane < 27) {
                        // gs[t][axis] = g - S(image vector t): S = (kx lx + ky xy + kz xz, ky ly + kz yz, kz lz)
                        const int ez = lane / 9, r9 = lane - ez * 9, ey = r9 / 3, ex3 = r9 - ey * 3;
                        const double kx = tri_dec(ex3, 1.0), ky = tri_dec(ey, 1.0), kz = tri_dec(ez, 1.0);
                        const double *c6 = fc->cell;
                        gs[lane * 3 + 0] = __dsub_rn((double)gcx, __dadd_rn(__dadd_rn(__dmul_rn(kx, c6[0]), __dmul_rn(ky, c6[3])), __dmul_rn(kz, c6[4])));
                        gs[lane * 3 + 1] = __dsub_rn((double)gcy, __dadd_rn(__dmul_rn(ky, c6[1]), __dmul_rn(kz, c6[5])));
                        gs[lane * 3 + 2] = __dsub_rn((double)gcz, __dmul_rn(kz, c6[2]));
                    }
                } else if (lane < 9) {
                    // gs[axis][cls] = g - S(cls): the j point's coordinate relative to the centre is X_j - gs (one DADD)
                    const int a = lane / 3, c = lane - a * 3;
                    const double g = (double)(a == 0 ? gcx : (a == 1 ? gcy : gcz));
                    const double l = fc->cell[a];
                    gs[lane] = c == 0 ? g : (c == 1 ? __dsub_rn(g, l) : __dadd_rn(g, l));
                }
                const double2 ixy = ex.rAg[lane], izw = ex.rAg[32 + lane];
                const bool ipad = __double2hiint(izw.y) < 0;           // padding lanes: far away, never inside any cutoff
                R.xi = ipad ? -FAST_PAD : __double2float_rn(__dsub_rn(ixy.x, (double)gcx));
                R.yi = ipad ? 0.f : __double2float_rn(__dsub_rn(ixy.y, (double)gcy));
                R.zi = ipad ? 0.f : __double2float_rn(__dsub_rn(izw.x, (double)gcz));
                if (MULTICLS) R.cptab_mi_a = cptab_a + (unsigned)(__double2loint(izw.y) * p.nclsB) * 4u;
                // bin parameters of this unit: s from the error bound (header)
                const FastBin fbS = make_fastbin(__fmaf_ru(p.f_c1, 4.f * extm + 2.f * p.f_rc, p.f_rel), p.f_smax, p.inv_ddr, (unsigned)nb, lane,
                                                 hist_a);
                R.inv_s = fbS.inv_s;
                R.mask = fbS.mask;
                R.clampv = fbS.clampv;
                R.base = fbS.base;
                R.s = fbS.s;
                e15m = __fmaf_ru(p.f_c1, 4.f * fc->lmax_up + 6.f * extm + 3.f * p.f_rc, p.f_rel);
                __syncwarp();
            }

            unsigned needmask = 0;
            int tbl = -1, code = 0;
            int head = 0, tail = 0;
            unsigned stage = 0;
            bool have = false, cself = false;
            int ccode = 0;
            unsigned cbase = 0;                       // sorted position of the current chunk's first point
#pragma unroll 1
            for (;;) {
                // ---- A: the next needed chunk of the row; its 1 KB of records starts travelling to stage buffer `stage`
                // (two 16-byte cp.async per lane: every lane copies, and later reads, its own two entries)
                bool nvalid = false, nself = false;
                int ncode = 0;
                unsigned nbase = 0;
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
                        const float4 alo = gas[0], ahi = gas[1];
                        const float ga[6] = {alo.x, alo.y, alo.z, ahi.x, ahi.y, ahi.z};
                        if (TRICL) {
                            const int rcode = fast_tri_chunk_test(ga[0], ga[1], ga[2], ga[3], ga[4], ga[5], gb[0], gb[1], gb[2], gb[3], gb[4], gb[5],
                                                                  fc->cell, rcut2_up);
                            need = (rcode & 256) != 0;
                            code = rcode & 255;
                        } else {
                            const float4 a0 = *reinterpret_cast<const float4 *>(fc->ax[0]), a1 = *reinterpret_cast<const float4 *>(fc->ax[1]),
                                         a2 = *reinterpret_cast<const float4 *>(fc->ax[2]);
                            const AxisF AX = {a0.x, a0.y, a0.z, a0.w}, AY = {a1.x, a1.y, a1.z, a1.w}, AZ = {a2.x, a2.y, a2.z, a2.w};
                            need = chunk_class_f32(ga, gb, AX, AY, AZ, rcut2_up, code);
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
                    const unsigned cidx = (unsigned)tb * GPT + (unsigned)(l & 7);
                    nbase = cidx * GS;
                    const double2 *jsrc = fc->rB + (size_t)(cidx * GREC + (unsigned)lane);
                    const unsigned dst = wp_a + (unsigned)FW_JST + stage * 1024u + (unsigned)lane * 16u;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(jsrc) : "memory");
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 512u), "l"(jsrc + 32) : "memory");
                    nvalid = true;
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
                // ---- B: the current chunk (committed one round ago)
                if (have) {
                    asm volatile("cp.async.wait_group 1;" ::: "memory");
                    const double2 *jst = reinterpret_cast<const double2 *>(wp + FW_JST + (stage ^ 1u) * 1024u);
                    const double2 jxy = jst[lane], jzw = jst[32 + lane];
                    const bool jpad = __double2hiint(jzw.y) < 0;
                    const unsigned jpos = cbase + (unsigned)lane;   // SORTED position of my j point: what the exact path reads
                    const unsigned jmeta = jpad ? FAST_PADMETA : (MULTICLS ? (jpos << 6) | (unsigned)__double2loint(jzw.y) : jpos);
                    bool mixed;
                    float jx, jy, jz;
                    bool skip = false;
                    if (TRICL) {
                        mixed = ccode == TRI_MIXED;
                        if (mixed) {
                            // no single image vector for this chunk pair: fp64 for every pair of it
                            uev += 32u;
                            uex += 1024u;
                            fast_exact_chunk<MULTICLS>(nb, p.edges2, p.nclsB, p.rcut2, p.inv_ddr, hist, cptab_s, lane, jxy.x, jxy.y, jzw.x, jzw.y,
                                                       cself, ex.rAg, cell);
                            skip = true;
                            jx = jy = jz = 0.f;
                        } else {
                            const int t3 = ((ccode & 3) + 3 * ((ccode >> 2) & 3) + 9 * ((ccode >> 4) & 3)) * 3;
                            jx = __double2float_rn(__dsub_rn(jxy.x, gs[t3]));
                            jy = __double2float_rn(__dsub_rn(jxy.y, gs[t3 + 1]));
                            jz = __double2float_rn(__dsub_rn(jzw.x, gs[t3 + 2]));
                        }
                    } else {
                        mixed = ((ccode & (ccode >> 1)) & 0x15) != 0;
                        // j relative to the group centre: subtraction of (g - S) in fp64, ONE rounding to fp32
                        if (ccode == 0 || mixed) {           // the common case (no image shift anywhere): fixed table slots
                            jx = __double2float_rn(__dsub_rn(jxy.x, gs[0]));
                            jy = __double2float_rn(__dsub_rn(jxy.y, gs[3]));
                            jz = __double2float_rn(__dsub_rn(jzw.x, gs[6]));
                        } else {
                            jx = __double2float_rn(__dsub_rn(jxy.x, gs[ccode & 3]));
                            jy = __double2float_rn(__dsub_rn(jxy.y, gs[3 + ((ccode >> 2) & 3)]));
                            jz = __double2float_rn(__dsub_rn(jzw.x, gs[6 + ((ccode >> 4) & 3)]));
                        }
                    }
                    if (jpad) {
                        jx = FAST_PAD;
                        jy = 0.f;
                        jz = 0.f;
                    }
                    if (skip) {
                    } else if (cself || mixed) {
                        // rare: the triangular self chunk / a chunk pair without a uniform image (small cells)
                        if (tail != head) {
                            uev += (unsigned)((tail - head + FU - 1) & ~(FU - 1));
                            fast_flush<MULTICLS, TRICL>(R, ex, ring, wp_a + (unsigned)FW_RING, head, tail, lane, qn, xq, uex);
                        }
                        head = 0;
                        tail = 0;
                        uev += fast_special<MULTICLS, TRICL>(p.f_smax, p.inv_ddr, R, ex, fc, ring, wp_a + (unsigned)FW_RING, jx, jy, jz, jmeta, cself, mixed, extx, exty,
                                                             extz, rc2t, e15m, hist_a, lane, qn, xq, uex);
                    } else {
                        const float bx = fmaxf(fabsf(jx) - extx, 0.f), by = fmaxf(fabsf(jy) - exty, 0.f), bz = fmaxf(fabsf(jz) - extz, 0.f);
                        const bool ok = __fmaf_rn(bz, bz, __fmaf_rn(by, by, bx * bx)) < rc2t && !jpad;
                        const unsigned m = __ballot_sync(0xffffffffu, ok);
                        if (ok) ring_put(ring, (tail + __popc(m & ((1u << lane) - 1u))) & (FRING - 1), jx, jy, jz, jmeta);
                        tail += __popc(m);
                        if (tail - head >= 32) {
                            __syncwarp();
                            uev += 32u;
                            fast_run<MULTICLS, TRICL, false, false>(R, ex, wp_a + (unsigned)FW_RING + (unsigned)(head & 32) * 16u, 32, 0.f, 0.f, 0.f,
                                                                    lane, qn, xq, uex);
                            __syncwarp();
                            head += 32;
                        }
                    }
                }
                if (!nvalid) break;
                have = true;
                ccode = ncode;
                cself = nself;
                cbase = nbase;
                stage ^= 1u;
            }
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            if (tail != head) {
                uev += (unsigned)((tail - head + FU - 1) & ~(FU - 1));
                fast_flush<MULTICLS, TRICL>(R, ex, ring, wp_a + (unsigned)FW_RING, head, tail, lane, qn, xq, uex);
            }
            if (qn > 0) {
                uex += (unsigned)qn;
                fast_settle<MULTICLS, TRICL>(nb, p.edges2, p.nclsB, hist, cptab_s, lane, qn, xq, ex.rAg, rB, cell);
                qn = 0;
            }
            // overflow guard of the uint32 shared histogram: the CTA counts the 32-pair steps it has evaluated since the
            // histogram was last re-based; the warp that crosses a multiple of the budget re-bases it (no barrier needed,
            // see flush_words).  Between two re-basings a word receives fewer than 2^30 + 8 units' worth of increments
            // (a unit is at most 32 x npadB pairs, npadB < 2^22 is checked on the host), i.e. it stays below 2^31.
            {
                unsigned old_ = 0;
                if (lane == 0) {
                    old_ = atomicAdd(evals_s, uev);
                    atomicAdd(&tot_s[0], (unsigned long long)uev);
                    if (uex) atomicAdd(&tot_s[1], (unsigned long long)uex);
                }
                old_ = __shfl_sync(0xffffffffu, old_, 0);
                if ((old_ + uev) / (FAST_FLUSH_EVALS / 32u) != old_ / (FAST_FLUSH_EVALS / 32u)) flush_words(frame, lane, 32);
            }
            q = __shfl_sync(0xffffffffu, qnext, 0);
        }

        if (__syncthreads_or(did ? 1 : 0)) {
            flush_words(frame, threadIdx.x, blockDim.x);
            if (threadIdx.x == 0) *evals_s = 0u;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (tot_s[0]) atomicAdd(&p.stats[2], tot_s[0] * (unsigned long long)GS);
        if (tot_s[1]) atomicAdd(&p.stats[3], tot_s[1]);
    }
}

} // namespace
