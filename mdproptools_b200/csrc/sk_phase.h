// sk_phase.h -- the per-term body of the structure-factor kernel (sk.cu): fractional coordinates in 32-bit fixed point and
// the phase exp(2 pi i n.s) of one Miller triplet n at one atom.  Host/device shared; exercised on the host by
// tests/native/sk_phase_host.cpp.
//
// Cell: the restricted triclinic cell H = [a b c], a = (lx,0,0), b = (xy,ly,0), c = (xz,yz,lz).  s = H^-1 r in fp64, wrapped
// into [0,1) and stored as u = floor(frac(s) * 2^32) (a value of exactly 1.0 after rounding wraps to 0, which is the same
// point).  For an integer triplet the phase n.s mod 1 is then the exact integer p = h ux + k uy + l uz mod 2^32 (wrapping
// 32-bit multiply-adds, no range reduction, no precision lost at large |n|).  Its top 23 bits, rounded, are placed in the
// mantissa of a float in [1,2): f = that float - 1.5 in [-1/2, 1/2) exactly, so exp(2 pi i p/2^32) = -exp(2 pi i f); the
// kernel negates the fp64 class sums once at the end.  sin and cos of 2 pi f in fp32 (the device's __sincosf).
//
// Accuracy contract, per term and |n_i| <= MDP_SK_NLIM (DESIGN 4.5 derives it):
//   quantisation   sum |n_i| 2^-32 cycles                 <= 3 * 1024 * 2^-32 = 7.15e-7 cycles
//   rounding p to 23 bits                                 <= 2^-24 cycles                 = 5.96e-8 cycles
//   f * 2 pi in fp32 (constant and product rounding)      <= pi * 2^-23 rad               = 3.75e-7 rad
//   __sincosf on [-pi, pi] (CUDA Programming Guide)       <= 2^-21.41 per component  -> |d exp| <= 5.1e-7
//   fp32 sums of at most MDP_SK_CHUNK = 32 terms (|partial| <= j)  <= sqrt(2) 2^-24 (32 * 33 / 2 - 1) / 32 per term = 1.39e-6
// so |d exp| <= 2 pi (7.75e-7) + 3.75e-7 + 5.1e-7 + 1.39e-6 = 7.14e-6 per atom, and |rho_c(k)_device - rho_c(k)_exact| <=
// MDP_SK_EPS * N_c with MDP_SK_EPS = 1e-5 (the fp64 sums across chunks add about N_c^2 2^-53 / 64, below 1e-12 N_c for
// N_c <= 10^6).
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define MDP_HD __host__ __device__ __forceinline__
#else
#ifndef MDP_HD
#define MDP_HD inline
#endif
#endif

#define MDP_SK_NLIM 1024          // largest |h|, |k|, |l| the contract covers (k_max = 10 / A needs n <= 320 in a 200 A box)
#define MDP_SK_EPS 1e-5           // |rho_device - rho_exact| <= MDP_SK_EPS * N_c
#define MDP_SK_MAX_CLASSES 64     // classes per call
#define MDP_SK_CHUNK 32           // terms summed in fp32 before they enter the fp64 class sums

// fractional coordinates of r in the cell {lx, ly, lz, xy, xz, yz}: back substitution through the triangular H
MDP_HD void mdp_sk_frac(const double *cell, double x, double y, double z, double *s)
{
    const double sc = z / cell[2];
    const double sb = (y - sc * cell[5]) / cell[1];
    s[0] = (x - sb * cell[3] - sc * cell[4]) / cell[0];
    s[1] = sb;
    s[2] = sc;
}

// floor(frac(s) * 2^32) mod 2^32
MDP_HD uint32_t mdp_sk_fix(double s)
{
    const double w = (s - floor(s)) * 4294967296.0;              // in [0, 2^32]; exact scaling
    return (uint32_t)(unsigned long long)w;                      // 2^32 (s just below an integer) wraps to 0
}

// n.u + 2^8 mod 2^32 (the 2^8 rounds the 23-bit truncation below to nearest)
MDP_HD uint32_t mdp_sk_phase(int h, int k, int l, uint32_t ux, uint32_t uy, uint32_t uz)
{
    return (uint32_t)h * ux + 256u + (uint32_t)k * uy + (uint32_t)l * uz;
}

// f in [-1/2, 1/2) with f = p / 2^32 - 1/2 mod 1, to 2^-24
MDP_HD float mdp_sk_half_turn(uint32_t p)
{
    const uint32_t bits = 0x3f800000u | (p >> 9);
    float v;
#if defined(__CUDA_ARCH__)
    v = __uint_as_float(bits);
#else
    memcpy(&v, &bits, sizeof v);
#endif
    return v - 1.5f;
}

// the angle 2 pi f of one term, in [-pi, pi]
MDP_HD float mdp_sk_angle(uint32_t p)
{
    return mdp_sk_half_turn(p) * 6.28318530717958647692f;
}
