// orient.h -- the per-(vector, frame) body of the reorientation kernel (orient.cu): the minimum-image differences inside one
// molecule, the molecule-fixed vector of each kind, its direction u and the 8 real channels whose autocorrelations sum to the
// first- and second-rank Legendre correlations.  Host/device shared; exercised on the host by tests/native/orient_host.cpp.
// All fp64; the library builds with --fmad=false and the host emulation with -ffp-contract=off, rint, sqrt and division are
// correctly rounded on both sides, so host and device give the same bits.
//
// Cell: the restricted triclinic cell {lx, ly, lz, xy, xz, yz} with rows a = (lx,0,0), b = (xy,ly,0), c = (xz,yz,lz).  The
// minimum image reduces sequentially in LAMMPS order (Domain::minimum_image): d -= rint(d_z/lz) c, then d -= rint(d_y/ly) b,
// then d -= rint(d_x/lx) a.  That is the nearest image for vectors short next to half the cell, so wrapped and unwrapped
// positions give the same vectors.
//
// Channels of u (|u| = 1):  c0..c2 = ux, uy, uz                               sum_a c_a c'_a = u.u'     = P1(u.u')
//                           c3 = (ux^2 - uy^2) / sqrt 2,  c4 = (2 uz^2 - ux^2 - uy^2) / sqrt 6,
//                           c5 = sqrt 2 ux uy,  c6 = sqrt 2 ux uz,  c7 = sqrt 2 uy uz
// c3..c7 are an orthonormal basis of the traceless symmetric Q = u u^T - I/3, so sum_i c_i c'_i = Q:Q' = (u.u')^2 - 1/3 and
// P2(u.u') = 1.5 Q:Q' exactly (no constant term).  A zero-length or non-finite w gives NaN channels (0/0, inf/inf).
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#define MDP_HD __host__ __device__ __forceinline__
#else
#ifndef MDP_HD
#define MDP_HD inline
#endif
#endif

#define MDP_ORIENT_KINDS 3        // 0 = bond (i, j), 1 = bisector (i, j, k), 2 = normal (i, j, k)
#define MDP_ORIENT_CHANNELS 8

// d <- the minimum image of d in the cell
MDP_HD void mdp_orient_mic(const double *cell, double *d)
{
    double m = rint(d[2] / cell[2]);
    d[0] -= m * cell[4];
    d[1] -= m * cell[5];
    d[2] -= m * cell[2];
    m = rint(d[1] / cell[1]);
    d[0] -= m * cell[3];
    d[1] -= m * cell[1];
    m = rint(d[0] / cell[0]);
    d[0] -= m * cell[0];
}

// the 8 channels of one vector from the positions ri, rj, rk of its atoms (rk unused for a bond)
MDP_HD void mdp_orient_channels(const double *cell, int kind, const double *ri, const double *rj, const double *rk, double *ch)
{
    double dj[3] = {rj[0] - ri[0], rj[1] - ri[1], rj[2] - ri[2]};
    mdp_orient_mic(cell, dj);
    double w[3] = {dj[0], dj[1], dj[2]};
    if (kind != 0) {
        double dk[3] = {rk[0] - ri[0], rk[1] - ri[1], rk[2] - ri[2]};
        mdp_orient_mic(cell, dk);
        if (kind == 1) {
            w[0] = (dj[0] + dk[0]) * 0.5;
            w[1] = (dj[1] + dk[1]) * 0.5;
            w[2] = (dj[2] + dk[2]) * 0.5;
        } else {
            w[0] = dj[1] * dk[2] - dj[2] * dk[1];
            w[1] = dj[2] * dk[0] - dj[0] * dk[2];
            w[2] = dj[0] * dk[1] - dj[1] * dk[0];
        }
    }
    const double r = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
    const double x = w[0] / r, y = w[1] / r, z = w[2] / r;
    const double s2 = 1.41421356237309504880, r2 = 0.70710678118654752440, r6 = 0.40824829046386301637;
    const double xx = x * x, yy = y * y, zz = z * z;
    ch[0] = x;
    ch[1] = y;
    ch[2] = z;
    ch[3] = (xx - yy) * r2;
    ch[4] = (2.0 * zz - xx - yy) * r6;
    ch[5] = s2 * x * y;
    ch[6] = s2 * x * z;
    ch[7] = s2 * y * z;
}
