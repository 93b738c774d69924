// Host build of the reorientation kernel's body (mdproptools_b200/csrc/orient.h), laid out as mdp_orient_series writes it:
// out[8][nvec][out_stride], frame f at column frame0 + f, other columns untouched.  With -ffp-contract=off these are the
// device's bits.  TEST INFRASTRUCTURE ONLY.
#include <math.h>

#include "../../mdproptools_b200/csrc/orient.h"

extern "C" {

void emulate_orient_series(int nframes, long long n, const double *xyz, const double *cell, int kind, long long nvec,
                           const int *atoms, double *out, long long out_stride, long long frame0)
{
    for (int f = 0; f < nframes; ++f) {
        const double *x = xyz + (long long)f * 3 * n;
        for (long long v = 0; v < nvec; ++v) {
            const int ia = atoms[3 * v], ja = atoms[3 * v + 1], ka = kind ? atoms[3 * v + 2] : ia;
            double ri[3], rj[3], rk[3], ch[MDP_ORIENT_CHANNELS];
            for (int a = 0; a < 3; ++a) {
                ri[a] = x[a * n + ia];
                rj[a] = x[a * n + ja];
                rk[a] = x[a * n + ka];
            }
            mdp_orient_channels(cell + 6 * f, kind, ri, rj, rk, ch);
            for (int q = 0; q < MDP_ORIENT_CHANNELS; ++q) out[((long long)q * nvec + v) * out_stride + frame0 + f] = ch[q];
        }
    }
}

} // extern "C"
