/*
 * mdprop_b200.h -- C ABI of libmdprop_b200.so: the B200 (sm_100a) implementation of the mdproptools
 * trajectory post-processing hot path.
 *
 * The reference (molmd/mdproptools v0.0.6) is pure Python; it has no FFI.  Its "native" layer is the
 * set of numba-jitted loops and numpy/FFT correlators listed below.  Each entry point here replaces
 * one of them; the Python package mdproptools_b200 binds these symbols with ctypes and keeps the
 * reference's public API on top (INTEGRATION.md shows the binding a maintainer of the reference would
 * add).  Citations are file:line relative to the reference root.
 *
 * Conventions
 *   - plain C types only; every pointer documented as DEVICE is a CUDA device pointer owned by the
 *     caller (the Python side uses torch tensors for that), HOST pointers are ordinary memory;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls enqueue work
 *     on it and return without synchronising unless stated;
 *   - return value 0 = success, negative = error; mdp_last_error() returns a thread-local message;
 *   - outputs documented "accumulate" are added to (caller zeroes), like the reference's kernels
 *     which receive zeroed arrays and add in place (rdf_cn.py:485-486, 633);
 *   - scratch memory lives in the context (grown on demand, reused between calls); one context per
 *     device per host thread.  There is NO CPU fallback anywhere in this library.
 */
#ifndef MDPROP_B200_H
#define MDPROP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDP_VERSION 100

typedef struct mdp_ctx mdp_ctx;

/* ---- context ------------------------------------------------------------------------------- */
int mdp_version(void);
const char *mdp_last_error(void);
int mdp_ctx_create(int device, mdp_ctx **out);
void mdp_ctx_destroy(mdp_ctx *ctx);
/* bytes of scratch currently held / upper bound the context may grow to (default 8 GiB); the pair engine and the FFT
 * correlation split their work (frames, channels) into batches that fit it */
int64_t mdp_ctx_scratch_bytes(mdp_ctx *ctx);
int mdp_ctx_set_scratch_limit(mdp_ctx *ctx, int64_t bytes);
/* counters: number of kernels this library launched since creation (bench.py's gpu_launches) */
int64_t mdp_ctx_launch_count(mdp_ctx *ctx);
/* optional kernel timing for benchmarks: when enabled, the library brackets its main kernels with CUDA events
 * on the launching stream.  tag 0 = pair kernel (k_pair), 1 = pair preparation (sort, boxes, work list),
 * 2 = streaming MSD kernel, 3 = correlation kernel, 4 = charge-flux kernel, 5 = windowed (all-origins) MSD kernel,
 * 6 = bitmask autocorrelation kernel, 7 = FFT all-origins MSD (the whole of mdp_cross_msd_fft), 8 = structure factor (the
 * whole of mdp_structure_factor: kernels k_sk_sort, k_sk_rho, k_sk_bins; and of mdp_sk_rho: k_sk_sort, k_sk_rho), 9 = binned
 * FFT correlation of complex series (the whole of mdp_isf_fft: kernels k_isf_*), 10 = grouped FFT autocorrelation (the
 * whole of mdp_group_acf_fft: kernels k_fft_*, k_msd_spec_acc), 11 = reorientation channels (the whole of mdp_orient_series:
 * kernel k_orient).  mdp_ctx_timing_read synchronises
 * on the recorded events, returns the summed milliseconds and the number of launches, and clears them. */
int mdp_ctx_timing(mdp_ctx *ctx, int enable);
int mdp_ctx_timing_read(mdp_ctx *ctx, int tag, double *ms_total, int64_t *count);
/* statistics of the last pair call: [0]=tile-pair items evaluated, [1]=nominal tile pairs,
 * [2]=pair distance evaluations actually executed (32 x chunk steps), device->host sync. */
int mdp_ctx_pair_stats(mdp_ctx *ctx, int64_t out[4]);

/* ---- binning ------------------------------------------------------------------------------- */
/*
 * Edge table of the reference's bin function  bin(rsq) = (int64)(sqrt(rsq) / ddr)
 * (rdf_cn.py:68 `np.sqrt(rsq)/ddr`, truncated at :85 `.astype(np.int64)`).
 * edges[k] (k = 0..nb) = smallest double rsq with bin(rsq) >= k, found by bisection on the bit
 * pattern with IEEE sqrt and divide, so that  bin(rsq) = #{k >= 1 : edges[k] <= rsq}  exactly.
 * HOST: edges[nb + 1].
 */
int mdp_bin_edges(double ddr, int nb, double *edges);

/* ---- pair kernels ---------------------------------------------------------------------------
 * Replace _calc_rsq + _remove_outliers + _rdf_loop / _cn_loop / _rdf_mol_loop / _cn_mol_loop
 * (rdf_cn.py:35-162).  Distances: d = a - b per axis, single-shift orthorhombic minimum image with
 * strict compares against l/2 (rdf_cn.py:50-55), rsq = (dx*dx + dy*dy) + dz*dz unfused fp64 (:56),
 * cutoff rsq < rcut2 strict (:66).  Results are integer counts, bit-exact.
 *
 * Point sets: SoA coordinates xyz = [nframes][3][n] doubles (DEVICE) with frame stride 3*n, in the
 * caller's row order (the reference's id order); cls = int32 class id per point in [0, ncls)
 * (DEVICE; cls_stride = n if it differs per frame, 0 if one array serves all frames).
 * box = HOST [nframes][3] box lengths as the reference passes them (lattice lengths or bound
 * extents, SURVEY appendix A.6).
 *
 * Set B == NULL  -> symmetric mode: unordered pairs i<j of set A, each counted ONCE in the
 *                   class-pair histogram (the x2 of rdf_cn.py:85-86 and the two role orders of
 *                   :89-96 are applied by mdp_hist_reduce weights);
 *                   hist rows = ncls_a*(ncls_a+1)/2, row(ci<=cj) = ci*ncls_a - ci*(ci-1)/2 + (cj-ci).
 * Set B != NULL  -> rectangular mode: every a in A against every b in B, no self exclusion
 *                   (rdf_cn.py:131-140); hist rows = ncls_a*ncls_b, row = ci*ncls_b + cj.
 *
 * Binning: edges = HOST [nbins+1] ascending rsq thresholds with edges[0] ignored (treated as 0);
 * bin(rsq) = #{k>=1 : edges[k] <= rsq}; pairs with bin >= nbins are dropped.  uniform_ddr > 0 tells
 * the kernel the table came from mdp_bin_edges(uniform_ddr, nbins) so it may locate the bin from an
 * fp32 estimate and correct it with the table; uniform_ddr = 0 -> the table is searched (use for the
 * per-relation cutoffs of the coordination-number calls, rdf_cn.py:112).
 *
 * hist_out: DEVICE uint64 [nframes][rows][nbins], accumulate.
 */
int mdp_pair_hist(mdp_ctx *ctx, int nframes,
                  int64_t n_a, const double *xyz_a, const int32_t *cls_a, int64_t cls_stride_a, int ncls_a,
                  int64_t n_b, const double *xyz_b, const int32_t *cls_b, int64_t cls_stride_b, int ncls_b,
                  const double *box, double rcut2, const double *edges, int nbins, double uniform_ddr,
                  uint64_t *hist_out, int flags, void *stream);
#define MDP_PAIR_NO_CULL 1     /* evaluate every tile pair (brute force, for A/B measurements) */
#define MDP_PAIR_NO_SORT 2     /* keep caller order inside tiles (no spatial sort; implies little culling) */
/* General triclinic minimum image (north-star extension: the reference has none and wraps tilted cells as if
 * they were orthogonal, SURVEY 7).  box = HOST [nframes][6] = {lx, ly, lz, xy, xz, yz} of the restricted
 * triclinic cell a=(lx,0,0), b=(xy,ly,0), c=(xz,yz,lz); the image is the sequential single shift z, y, x
 * (if |dz| > lz/2: dz -= s*lz, dy -= s*yz, dx -= s*xz; then y with xy; then x), each step an unfused fp64
 * subtraction in that order, everything else as above.  Nearest image whenever the cutoff is at most half
 * the smallest cell width and |xy|,|xz| <= lx/2, |yz| <= ly/2.  Definition and checker: oracle/oracle.c
 * pair_rsq_tri (parity unpinned by the reference). */
#define MDP_PAIR_TRICLINIC 4
/* Uniform-bin histograms are served by the fp32-filtered kernel (csrc/pair_fast.cuh: fp32 distance and bin, every pair
 * within the proven error bound of a bin edge re-evaluated by the reference's fp64 arithmetic; counts identical).  This
 * flag (or the environment variable MDP_PAIR_F64) selects the all-fp64 kernel instead, for A/B measurements and tests. */
#define MDP_PAIR_F64 16
/* mdp_pair_hist and mdp_pair_list return MDP_ERR_ARG for any other flag bit (8 selected a binning variant of the
 * all-fp64 kernel in earlier versions). */

/*
 * out[f][r][b] = sum_rows weights[r][row] * hist[f][row][b]     (all integer)
 * weights: HOST int32 [nout][rows].  For calc_atomic_rdf: row 0 of the output is g_full with weight 2
 * on every class pair (rdf_cn.py:85-86), relation (a,b) has weight 2 on row(a,a) if a==b else 1 on
 * row(a,b) (rdf_cn.py:89-96).  With cumulative != 0 the bins are prefix-summed first (coordination
 * counts: everything below each cutoff).  hist, out: DEVICE uint64; out is overwritten.
 */
int mdp_hist_reduce(mdp_ctx *ctx, int nframes, int rows, int nbins, const uint64_t *hist, int nout,
                    const int32_t *weights, int cumulative, uint64_t *out, void *stream);

/*
 * Neighbour list (replaces the cutoff searches of get_clusters cluster_analysis.py:150-161,
 * get_angle hydration_number.py:16-19 and ResidenceTime loop 1 residence_time.py:100-104):
 * every (a in A, b in B) with  rin2 < rsq <= rout2  (shell_mode 1, residence_time.py:102) or
 * rsq < rout2 (shell_mode 0, cluster_analysis.py:160), excluding a==b index pairs when
 * exclude_same_index != 0 (residence_time.py:103-104).  Output entries are (frame, ia, ib) in the
 * caller's row order, unordered within the list; list_out = DEVICE int32 [capacity][3];
 * rsq_out = DEVICE double[capacity] or NULL; count_out = DEVICE int64 (total found; if it exceeds
 * capacity only `capacity` entries were written -- call again with a bigger list).
 * flags: 0 or MDP_PAIR_TRICLINIC (box = [nframes][6]) / MDP_PAIR_NO_CULL / MDP_PAIR_NO_SORT.
 */
int mdp_pair_list(mdp_ctx *ctx, int nframes,
                  int64_t n_a, const double *xyz_a, int64_t n_b, const double *xyz_b,
                  const double *box, double rin2, double rout2, int shell_mode, int exclude_same_index,
                  int32_t *list_out, double *rsq_out, int64_t capacity, int64_t *count_out, int flags, void *stream);

/* ---- epilogues of the cutoff searches (csrc/epilogue.cu) -------------------------------------------
 * All take the neighbour list of mdp_pair_list (DEVICE int32 [m][3] = (frame, ia, ib), any order).
 *
 * mdp_list_group: the entries grouped by (frame, ia) -- segment s = frame * n_a + ia occupies slots
 * seg_off[s] .. seg_off[s+1] (DEVICE int64 [nframes*n_a + 1]) -- and sorted inside a segment by `key` (DEVICE uint32 [m],
 * or NULL for key = ib; ties by entry index).  key_out[slot] = key, perm_out[slot] = index of the entry (DEVICE, [m]).
 * This is the row order the reference's per-central-atom pandas code produces (hydration_number.py:69-73,
 * cluster_analysis.py:143-165). */
int mdp_list_group(mdp_ctx *ctx, int nframes, int64_t n_a, int64_t m, const int32_t *list, const uint32_t *key,
                   int64_t *seg_off, uint32_t *key_out, int64_t *perm_out, void *stream);
/* The distinct (ia, ib) pairs of a neighbour list as sorted keys ia * n_b + ib (residence_time.py:100-111 needs one
 * indicator series per ever-neighbour pair): keys_out = DEVICE int64 [capacity], count_out = DEVICE int64 (total found; only
 * `capacity` are written).  A bitmap over the n_a * n_b possible pairs + a popcount scan, no sort. */
int mdp_unique_pair_keys(mdp_ctx *ctx, int64_t m, const int32_t *list, int64_t n_a, int64_t n_b, int64_t *keys_out,
                         int64_t capacity, int64_t *count_out, void *stream);
/* get_angle (hydration_number.py:13-32) for every (frame, cation, water O) entry: cos between the minimum-image
 * displacement cation - O (rdf_cn.py:46-55 with the frame's box, HOST double [nframes][3]) and the bisector
 * (H1 + H2) - 2 O of raw coordinates (hydration_number.py:60-63), numpy's fp64 expression order.  cos_out = DEVICE
 * double [m] in (frame, cation, water) order; seg_off as in mdp_list_group; counts = DEVICE int32 [nframes][n_cat][2] =
 * (waters in range, waters with cos < threshold).  Coordinates: DEVICE double [nframes][3][n]. */
int mdp_hydration_count(mdp_ctx *ctx, int nframes, int64_t n_cat, const double *xyz_cat, int64_t n_wat, const double *xyz_o,
                        const double *xyz_h1, const double *xyz_h2, const double *box, int64_t m, const int32_t *list,
                        double threshold, double *cos_out, int64_t *seg_off, int32_t *counts, void *stream);
/* get_clusters' molecule completion and force filter (cluster_analysis.py:163-182): for every (frame, central atom) the
 * sorted, duplicate-free molecules owning an atom of the neighbour list (ib = atom row) whose
 * min(sum fx, sum fy, sum fz) * force_constant < max_force (sums over the molecule's atoms in atom order; force = DEVICE
 * double [nframes][3][n_atoms]; mol_seg_off = DEVICE int32 [n_mol+1]; mol_of_atom = DEVICE int32 [n_atoms]).
 * mol_out[seg_off[s] .. seg_off[s] + mol_count[s]) = those molecules (DEVICE uint32 [m], int32 [nframes*n_central]). */
int mdp_cluster_members(mdp_ctx *ctx, int nframes, int64_t n_central, int64_t n_atoms, const double *force, int64_t n_mol,
                        const int32_t *mol_seg_off, const int32_t *mol_of_atom, double force_constant, double max_force,
                        int64_t m, const int32_t *list, int64_t *seg_off, uint32_t *mol_out, int32_t *mol_count, void *stream);

/* The Python layer's default for small central sets (MDP_SHELL_GRID=0 selects mdp_pair_list): the entries mdp_pair_list returns (same arguments, orthogonal cell, no rsq
 * output), found through a cell grid over a SMALL set A (n_a <= 4096) held in shared memory while B is streamed once
 * (csrc/shell_grid.h).  Returns 0, or 1 when the grid does not apply (n_a too large, or the outer radius exceeds a third
 * of a box length in some frame): the caller then uses mdp_pair_list. */
int mdp_shell_search(mdp_ctx *ctx, int nframes, int64_t n_a, const double *xyz_a, int64_t n_b, const double *xyz_b,
                     const double *box, double rin2, double rout2, int shell_mode, int exclude_same_index,
                     int32_t *list_out, int64_t capacity, int64_t *count_out, void *stream);

/* ---- segmented (per-molecule) reductions ------------------------------------------------------
 * calc_com (com_mols.py:5-62) / _define_mol_cols (rdf_cn.py:218-241): for each segment s (molecule;
 * atoms seg_off[s]..seg_off[s+1]-1 in id order) out[c][s] = sum_a w[a]*attr[c][a] / sum_a w[a],
 * sequential fp64 accumulation in atom order, unfused.  attr = DEVICE [nframes][ncomp][n],
 * w = DEVICE [n] (masses), seg_off = DEVICE int32[nseg+1], out = DEVICE [nframes][ncomp][nseg].
 * wsum_out (DEVICE [nseg], may be NULL) receives sum_a w[a]; extra (DEVICE [n], may be NULL) is summed
 * unweighted into extra_out [nseg] (molecular charge, com_mols.py:43-46).
 */
int mdp_segment_com(mdp_ctx *ctx, int nframes, int ncomp, int64_t n, const double *attr, const double *w,
                    int64_t nseg, const int32_t *seg_off, double *out, double *wsum_out,
                    const double *extra, double *extra_out, void *stream);

/* ---- MSD (diffusion.py:207-238) ----------------------------------------------------------------
 * traj = DEVICE [nframes][3][n], ref = DEVICE [3][n] (the Time==0 frame, diffusion.py:213);
 * groups are contiguous row ranges: group_off = HOST int64[ngroups+1] (NULL = one group of all rows)
 * -- molecule types are contiguous in id order (com_mols.py:31-42).
 * sums_out = DEVICE [nframes][ngroups][4]: per-group SUMS of dx2, dy2, dz2 and (dx2+dy2)+dz2
 * (diffusion.py:214-215); the caller divides by the group sizes (groupby.mean, :218).
 * per_atom_out = DEVICE [nframes][4][n] or NULL (msd_all, :216).  scale multiplies coordinates
 * before differencing (the SI conversion of diffusion.py:201-203 happens before the subtraction).
 */
int mdp_msd_single_origin(mdp_ctx *ctx, int nframes, int64_t n, const double *traj, const double *ref,
                          double scale, const int64_t *group_off, int ngroups, double *sums_out,
                          double *per_atom_out, void *stream);
/* msd_int (diffusion.py:225-237): frames 0, stride, 2*stride, ...; per atom the MEAN over the nint-1
 * squared steps for dx2/dy2/dz2 and SUM/nint for msd (the n vs n-1 quirk of the reference).
 * out = DEVICE [4][n]. */
int mdp_msd_interval(mdp_ctx *ctx, int nframes, int64_t n, const double *traj, double scale, int stride,
                     double *out, void *stream);
/* Windowed MSD over all time origins (north-star extension, no reference implementation; defined by
 * oracle/oracle.c orc_msd_all_origins, 1e-10 relative):
 * sums_out = DEVICE [max_lag][ngroups][4] accumulate: scale^2 * sum over atoms of the group and over all
 * origins t0 with t0+lag < nframes of the squared displacement per axis, [3] = (x+y)+z; the caller divides
 * by count*(nframes-lag).  fp64 with FMA, fixed summation order (run-to-run deterministic). */
int mdp_msd_all_origins(mdp_ctx *ctx, int nframes, int64_t n, const double *traj, double scale,
                        const int64_t *group_off, int ngroups, int max_lag, double *sums_out, void *stream);

/* ---- Green-Kubo ---------------------------------------------------------------------------------
 * conductivity_loop (_conductivity.py:7-36): per frame, per molecule COM velocity (mass weighted,
 * sequential) times vel_scale, molecular charge (sum q) times q_scale, J[c][g][frame] = sum over
 * molecules of type g of q_mol * v_com,c.  vel = DEVICE [nframes][3][n]; mass,q = DEVICE [n];
 * seg_off = DEVICE int32 [nseg+1]; group_seg_off = HOST int64 [ngroups+1] (molecule types are contiguous
 * segment ranges); out = DEVICE [3][ngroups][out_stride] written at column frame0 + f. */
int mdp_charge_flux(mdp_ctx *ctx, int nframes, int64_t n, const double *vel, const double *mass,
                    const double *q, int64_t nseg, const int32_t *seg_off, const int64_t *group_seg_off,
                    int ngroups, double vel_scale, double q_scale, double *out, int64_t out_stride,
                    int64_t frame0, void *stream);
/* Conductivity.correlate (conductivity.py:97-114) / Viscosity.autocorrelate (viscosity.py:86-120):
 * out[c][tau] = (sum_{t < T-tau} a[c][t+tau] * b[c][t]) / (T - tau), direct fp64 sum (the reference
 * uses an FFT; agreement is to its round-off, ~1e-15 max|C|).  a,b,out = DEVICE [nchan][T];
 * nlags <= T lags are produced (out row stride = nlags). */
int mdp_xcorr_unbiased(mdp_ctx *ctx, int nchan, int64_t T, const double *a, const double *b, int64_t nlags,
                       double *out, void *stream);
/* The Python layer's default from 2048 steps on (MDP_XCORR_FFT=0 selects the direct sum): the same correlation through a
 * Stockham FFT in fp64, three radix-2 stages per pass (csrc/fft_corr.h) --
 * N log N instead of T^2/2, for the 10^6..10^7-step series of a viscosity run; agrees with mdp_xcorr_unbiased to the
 * round-off of an FFT, which is how the reference computes it: ~1e-15 of max|C| where T - tau is large, growing at the
 * last lags, where the absolute round-off of the lag sum is divided by T - tau.  Contract: 1e-10 of max_tau |C| at every
 * lag, measured to hold up to T = 10^7 with nlags = T (worst 9.3e-12, at lag T - 1).  Same arguments. */
int mdp_xcorr_fft(mdp_ctx *ctx, int nchan, int64_t T, const double *a, const double *b, int64_t nlags, double *out,
                  void *stream);
/* All-origins (cross) mean-square displacement of channel groups through the FFT of mdp_xcorr_fft (csrc/msd_fft.h, north-star
 * extension with no reference implementation; defined by the long-double direct sum of tests/native/cross_msd_direct.c):
 *   out[g][tau] = sum_{c in group g} (1/(T-tau)) sum_{t < T-tau} (a_c(t+tau) - a_c(t)) * (b_c(t+tau) - b_c(t)),  tau < nlags.
 * a, b = DEVICE [nchan][T]; b == NULL means b = a (the ordinary MSD summed over the group's channels); group_off = HOST int64
 * [ngroups+1], non-decreasing from 0 to nchan (contiguous channel groups, empty groups allowed, 1 <= ngroups <= 65535);
 * 1 <= nlags <= T; out = DEVICE [ngroups][nlags], overwritten.  Each channel's mean is subtracted first (the result does not
 * change; the cancellation of large offsets goes away).  O(nchan N log N) with N = 2^p >= T + nlags, p <= 30.  Agrees with
 * the direct long-double sum to 1e-10 of max_tau |out[g]| for T <= 10^5; the bound is absolute, so lags where out is small
 * next to its maximum (the first lags of a long diffusive series) are covered by it and nothing tighter.  Fixed summation
 * order, no atomics: run-to-run bit-identical, and the same bits under any scratch limit that admits the call.
 * MDP_ERR_ARG for bad sizes or group offsets, p > 30, or group accumulators (about ngroups * (4 N + 24 T) bytes) above the
 * context's scratch limit. */
int mdp_cross_msd_fft(mdp_ctx *ctx, int nchan, int64_t T, const double *a, const double *b, int ngroups, const int64_t *group_off,
                      int64_t nlags, double *out, void *stream);
/* Grouped all-origins autocorrelation through the same FFT pipeline (csrc/msd_fft.h: mdp_acf_epilogue; the velocity
 * autocorrelation of Diffusion.get_vacf; defined by the long-double direct sum of tests/vacf_oracle.py):
 *   out[g][tau] = sum_{c in group g} (1/(T-tau)) sum_{t < T-tau} a_c(t+tau) * a_c(t),   tau < nlags.
 * a = DEVICE [nchan][T], not centred (a mean, such as a velocity drift, is part of the result); group_off, nlags and out as
 * for mdp_cross_msd_fft (b = NULL): group_off = HOST int64 [ngroups+1], non-decreasing from 0 to nchan, empty groups
 * allowed (written as exactly 0), 1 <= ngroups <= 65535; 1 <= nlags <= T; out = DEVICE [ngroups][nlags], overwritten.  Two
 * channels of a group per forward transform, the spectra summed per group in the frequency domain, one inverse transform
 * per two groups: O(nchan N log N) with N = 2^p >= T + nlags, p <= 30, and no [nchan][nlags] intermediate.  Agrees with the
 * direct long-double sum to 1e-10 of max_tau |out[g]| (= out[g][0]) for T <= 10^5.  Fixed summation order, no atomics:
 * run-to-run bit-identical, and the same bits under any scratch limit that admits the call.  Scratch: group accumulators of
 * ngroups * (N/2 + 1) * 8 bytes plus the sub-batch work arrays.  MDP_ERR_ARG for every argument mdp_cross_msd_fft rejects
 * and for accumulators above the context's scratch limit. */
int mdp_group_acf_fft(mdp_ctx *ctx, int nchan, int64_t T, const double *a, int ngroups, const int64_t *group_off, int64_t nlags,
                      double *out, void *stream);
/* cumulative trapezoid along rows (conductivity.py:231 with leading zero, viscosity.py:151 without):
 * in = DEVICE [nrows][T]; out = DEVICE [nrows][T] if leading_zero else [nrows][T-1]; out = scale*integral. */
int mdp_cumtrapz(mdp_ctx *ctx, int nrows, int64_t T, const double *in, double dx, double scale,
                 int leading_zero, double *out, void *stream);

/* ---- static structure factor (extension: no reference implementation; defined by tests/sk_oracle.py) -------------------
 * Direct sum over reciprocal-lattice vectors of the restricted triclinic cell H = [a b c], a = (lx,0,0), b = (xy,ly,0),
 * c = (xz,yz,lz): cell = HOST double [6] = {lx, ly, lz, xy, xz, yz}, shared by every frame of the call (one call per run of
 * frames with the same cell).  For Miller triplets n (HOST int32 [nk][3], the caller's k-set, sorted by bin) and classes
 * c (cls = DEVICE int32 per atom in [0, ncls), cls_stride = n if it differs per frame, 0 if one array serves all frames,
 * NULL = every atom in class 0; atoms with a class outside [0, ncls) are left out):
 *   rho_c(n) = sum_{j in c} exp(2 pi i n.s_j),   s_j = H^-1 r_j   (xyz = DEVICE [nframes][3][n]; wrapped or unwrapped
 *              positions give the same result, n being integer)
 *   sums_out[f][row(a,b)][bin] = sum_{k = bin_off[bin]}^{bin_off[bin+1]-1} Re(rho_a(n_k) conj(rho_b(n_k)))
 * one row per unordered class pair a <= b, row(a,b) = a*ncls - a*(a-1)/2 + (b-a) (as mdp_pair_hist's symmetric mode);
 * bin_off = HOST int64 [nbins+1], non-decreasing from 0 to nk; sums_out = DEVICE double [nframes][ncls(ncls+1)/2][nbins],
 * overwritten.  nk = 0 and empty classes give zeros.
 * Accuracy contract (csrc/sk_phase.h, derived in DESIGN 4.5): the phase is the exact integer n.u mod 2^32 of 32-bit fixed-point
 * fractional coordinates, sin and cos are fp32, terms are summed in fp32 over at most 32 atoms and in fp64 beyond; for every
 * |h|, |k|, |l| <= 1024:  |rho_c(k)_device - rho_c(k)_exact| <= 1e-5 * N_c.
 * Fixed summation order, no atomics: run-to-run bit-identical, and the same bits under every scratch limit that admits the call.
 * MDP_ERR_ARG for negative sizes, n >= 2^31, ncls outside [1, 64], a non-positive or non-finite length, a non-finite tilt,
 * a Miller component beyond +-1024, or a bin_off that is not non-decreasing from 0 to nk. */
int mdp_structure_factor(mdp_ctx *ctx, int nframes, int64_t n, const double *xyz, const int32_t *cls, int64_t cls_stride,
                         int ncls, const double *cell, int64_t nk, const int32_t *miller, int nbins, const int64_t *bin_off,
                         double *sums_out, void *stream);
/* rho_c(n) itself, per k-vector and frame: the first half of mdp_structure_factor, with the same arguments up to miller, the
 * same checks, accuracy contract and frame sub-batches, and bit for bit the rho values that mdp_structure_factor bins.
 * rho_out = DEVICE complex fp64 (re, im) [ncls][nk][out_stride]; frame f of the call goes to column frame0 + f
 * (0 <= frame0, frame0 + nframes <= out_stride), so that successive calls fill one time series per (class, k) in place;
 * other columns are left alone.  MDP_ERR_ARG as for mdp_structure_factor, or for frames outside the series. */
int mdp_sk_rho(mdp_ctx *ctx, int nframes, int64_t n, const double *xyz, const int32_t *cls, int64_t cls_stride, int ncls,
               const double *cell, int64_t nk, const int32_t *miller, double *rho_out, int64_t out_stride, int64_t frame0,
               void *stream);
/* Binned, symmetrised all-origins correlation of complex series (csrc/isf_fft.h; the coherent intermediate scattering function
 * when rho holds mdp_sk_rho's series; defined by the long-double direct sum of tests/isf_oracle.py):
 *   out[p][bin][tau] = sum_{k = bin_off[bin]}^{bin_off[bin+1]-1} 1/(T-tau) sum_{t < T-tau}
 *                      1/2 Re( z_a(k,t+tau) z_b(k,t)* + z_b(k,t+tau) z_a(k,t)* ),   (a, b) = pairs[p],  tau < nlags.
 * rho = DEVICE complex fp64 (re, im) [nchan][nk][T], z_c(k,t) = rho[c][k][t], not centred; pairs = HOST int32 [npairs][2] of
 * channels in [0, nchan); bin_off = HOST int64 [nbins+1], non-decreasing from 0 to nk; 1 <= nlags <= T; out = DEVICE double
 * [npairs][nbins][nlags], overwritten.  Empty bins and nk = 0 give zeros.  One forward transform per (k, channel some pair
 * uses) of N = 2^p >= T + nlags points (p <= 30); the real, even spectrum of each (pair, bin) is summed over the bin's
 * k-vectors in k order and two pairs of the same bin share one inverse transform.
 * Agrees with the direct long-double sum to 1e-10 of max_tau |out[p][bin]| for T <= 10^5.  Fixed summation order, no atomics:
 * run-to-run bit-identical; the same bits under every scratch limit that admits the call; a bin's bits do not depend on
 * which other bins share the call; swapping the two channels of a pair gives the same bits.
 * MDP_ERR_ARG for bad sizes, a pair naming a channel outside [0, nchan), a bad bin_off, p > 30, or accumulators (about
 * npairs * nbins * (N/2 + 1) * 8 bytes) above the context's scratch limit. */
int mdp_isf_fft(mdp_ctx *ctx, int nchan, int64_t nk, int64_t T, const double *rho, int npairs, const int32_t *pairs, int nbins,
                const int64_t *bin_off, int64_t nlags, double *out, void *stream);

/* ---- reorientation (extension, no reference implementation; tests/reorient_oracle.py is the definition) --------------
 * Channels of molecule-fixed unit vectors (csrc/orient.h), one time series per (channel, vector):
 *   d_j = mic(r_j - r_i), d_k = mic(r_k - r_i) in the frame's restricted triclinic cell (rows a = (lx,0,0), b = (xy,ly,0),
 *   c = (xz,yz,lz); sequential LAMMPS reduction: d -= rint(d_z/lz) c, then rint(d_y/ly) b, then rint(d_x/lx) a);
 *   w = d_j (kind 0, bond), (d_j + d_k)/2 (kind 1, bisector), d_j x d_k (kind 2, normal);  u = w / |w|;
 *   rows 0-2: ux, uy, uz;  rows 3-7: (ux^2 - uy^2)/sqrt2, (2uz^2 - ux^2 - uy^2)/sqrt6, sqrt2 ux uy, sqrt2 ux uz, sqrt2 uy uz,
 * so that the sum of rows 0-2 of u(t).u(t') is P1(u.u') and 1.5 times the sum of rows 3-7 is P2(u.u'), exactly: the
 * all-origins autocorrelation of each row group (mdp_group_acf_fft) gives C1 and C2 with no per-lag Legendre evaluation.
 * xyz = DEVICE [nframes][3][n] positions (wrapped or unwrapped: the same vectors for molecules short next to half the cell);
 * cell = HOST [nframes][6] = (lx, ly, lz, xy, xz, yz) per frame; atoms = HOST int32 [nvec][3] rows of xyz (i, j, k; k is
 * ignored for a bond); out = DEVICE double [8][nvec][out_stride]: frame f of the call goes to column frame0 + f (0 <= frame0,
 * frame0 + nframes <= out_stride), so that successive calls fill one series in place; other columns are left alone.
 * fp64 throughout; with the library's unfused arithmetic the values are bit-identical to a host build of csrc/orient.h.
 * A zero-length or non-finite w gives NaN channels for that vector and frame.
 * MDP_ERR_ARG (checked on the host before anything is launched) for negative sizes, n >= 2^31, a kind outside [0, 3), an
 * atom index outside [0, n), a vector that repeats an atom, a non-positive or non-finite length, a non-finite tilt, or
 * frames outside the series. */
int mdp_orient_series(mdp_ctx *ctx, int nframes, int64_t n, const double *xyz, const double *cell, int kind, int64_t nvec,
                      const int32_t *atoms, double *out, int64_t out_stride, int64_t frame0, void *stream);

/* ---- residence time (residence_time.py:70-148) ---------------------------------------------------
 * Survival correlation from per-pair time bitmasks.  masks = DEVICE uint64 [npairs][nwords], bit t of
 * pair p set when the pair is inside the shell in frame t (built by mdp_pair_list + mdp_bitmask_fill).
 * cnt_out = DEVICE uint64 [T] accumulate: cnt[tau] = sum_p popcount(m_p & (m_p >> tau)). */
int mdp_bitmask_fill(mdp_ctx *ctx, int64_t nentries, const int32_t *list, int64_t n_b, const int64_t *pair_keys,
                     int64_t npairs, int nwords, uint64_t *masks, void *stream);
int mdp_bitmask_autocorr(mdp_ctx *ctx, int64_t npairs, int nwords, int64_t T, const uint64_t *masks,
                         uint64_t *cnt_out, void *stream);

/* The Python layer's default (MDP_SURVIVAL_RUNS=0 selects mdp_bitmask_autocorr): the same counts as mdp_bitmask_autocorr -- cnt_out accumulates, bit for bit
 * the same integers -- from the RUNS of each pair's bitmask: a pair with k runs costs 4*k(k+1)/2 integer updates of a
 * second-difference array instead of T^2/128 word operations (csrc/survival_runs.h).  T is limited by the shared-memory
 * array (about 25 000 frames). */
int mdp_survival_runs(mdp_ctx *ctx, int64_t npairs, int nwords, int64_t T, const uint64_t *masks, uint64_t *cnt_out,
                      void *stream);

/* ---- OLS through the origin (diffusion.py:323-329) -------------------------------------------------
 * out[c] = {sum t*t, sum t*y_c, sum y_c*y_c} over rows i0..i1-1; the host forms slope, bse, R2.
 * t = DEVICE [T], y = DEVICE [ncol][T], out = DEVICE [ncol][3]. */
int mdp_ols_sums(mdp_ctx *ctx, int ncol, int64_t T, const double *t, const double *y, int64_t i0, int64_t i1,
                 double *out, void *stream);

/* ---- number density along one axis (structural/number_density.py:30-154) ---------------------------
 * Per frame: {min, max} of coord over the atoms with key == surface_key (:77-83), then for every target key the histogram
 * of trunc(((x - min) - (max - min)) / bin_size) over atoms with x - min < dist (dist > 0, :88-99) or of
 * trunc((x - min) / bin_size) over atoms with x - min > dist (dist < 0, :100-110).  Negative indices wrap as numpy's do;
 * indices outside [-nbins, nbins) (an IndexError in the reference) are dropped.  target_keys is a HOST array.
 * coord, key = DEVICE [F][N]; counts_out = DEVICE uint64 [F][ntargets][nbins]; minmax_out = DEVICE [F][2] (NaN when a frame
 * has no surface atom, in which case its counts are zero). */
int mdp_axis_density(mdp_ctx *ctx, int nframes, int64_t n, const double *coord, const double *key, double surface_key,
                     int ntargets, const double *target_keys, double dist_from_interface, double bin_size, int nbins,
                     uint64_t *counts_out, double *minmax_out, void *stream);

/* ---- LAMMPS dump reader (replaces pymatgen parse_lammps_dumps at rdf_cn.py:176 etc.) ---------------
 * HOST-side, multi-threaded.  Parses one frame of dump text into SoA doubles scattered by id
 * (row id-1 <- the reference's sort_values("id"), rdf_cn.py:191-192).
 *   text,len      : the frame text starting at "ITEM: TIMESTEP"
 *   want          : array of nwant column names to extract
 *   out           : HOST [nwant][natoms] doubles (pinned memory recommended)
 *   header_out    : HOST double[16]: timestep, natoms, xlo,xhi,ylo,yhi,zlo,zhi (after the tilt
 *                   correction pymatgen applies), xy,xz,yz, triclinic flag, ncols, id_contiguous flag
 * mdp_dump_scan splits a buffer into frames (offsets of every "ITEM: TIMESTEP"). */
int64_t mdp_dump_scan(const char *text, int64_t len, int64_t *offsets, int64_t max_frames);
int mdp_dump_header(const char *text, int64_t len, double *header_out, char *columns_out, int columns_cap);
int mdp_dump_parse(const char *text, int64_t len, const char *const *want, int nwant, double *out,
                   int64_t out_stride, double *header_out, int nthreads);
/* A batch of frames in one call: frame f goes to out + f*frame_stride ([nwant][out_stride]) and headers_out + 16*f.
 * With many frames every worker thread parses whole frames (rows go straight to out[slot][id-1] while the ids are a
 * permutation of 1..natoms, else that frame takes mdp_dump_parse's ranking path); with fewer frames than half the
 * threads each frame is split over all threads as in mdp_dump_parse. */
int mdp_dump_parse_batch(int nframes, const char *const *texts, const int64_t *lens, const char *const *want, int nwant,
                         double *out, int64_t frame_stride, int64_t out_stride, double *headers_out, int nthreads);

/* The file pipeline's default with a GPU (io/pipeline.py; MDP_DEVICE_PARSE=0 selects the host parser above).
 * Device-side parse of the atom rows of nframes frames whose bytes are already in device memory: rows are placed by id
 * (out[f][slot][id-1]) with the exact fast path the host parser uses (dump_line.h).  begin/end = DEVICE int64 [nframes]:
 * byte offsets into text of the first row / one past the last row of each frame; longest = max(end - begin);
 * colsel = HOST int[ncols], output slot of file column c or -1.  seen = DEVICE uint32 [nframes][ceil(natoms/32)] scratch
 * and status = DEVICE uint64 [nframes][2] = {rows parsed, flags}, both zeroed by the call: a frame is valid iff rows ==
 * natoms and flags == 0; any other frame must be re-parsed with mdp_dump_parse (nothing is approximated on the device).
 * Uses no scratch of the context (safe next to other calls of the same context on another stream). */
int mdp_dump_parse_device(mdp_ctx *ctx, int nframes, const char *text, const int64_t *begin, const int64_t *end,
                          int64_t longest, int64_t natoms, int ncols, const int *colsel, int id_col, int nwant, double *out,
                          int64_t frame_stride, int64_t out_stride, uint32_t *seen, uint64_t *status, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MDPROP_B200_H */
