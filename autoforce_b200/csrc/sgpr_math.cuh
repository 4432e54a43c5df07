// Per-neighbour math of the SGPR descriptor: radial functions and solid harmonics
// r^l Y_lm with Cartesian gradients.  Host+device so that tests/ can compile the very
// same code with g++ and check it against the oracle without a GPU.
//
// Reference behaviour restated (never copied): theforce/descriptor/ylm.py:113-225
// (values + gradients, spherical-coordinate formulation there; here the same functions
// are evaluated as polynomials  Y_lm = Q_lm(z, r^2) (x+iy)^m, which has no division by
// sin(theta) and is smooth on the z axis), ylm.py:10-23 (environment-wide shear),
// descriptor/sesoap.py:172-184 + descriptor/cutoff.py:20-44 (radial part).
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define SGPR_HD __host__ __device__ __forceinline__
#else
#define SGPR_HD inline
#endif

namespace sgpr {

constexpr int kMaxL = 8;            // lmax <= 8
constexpr int kMaxNB = 12;          // nmax + 1 <= 12
constexpr double kTinyAngle = 1e-2; // ylm.py:10
constexpr int kMaxSpecies = 8;

// Coefficients of the Q_lm recursion (ylm.py:57-80), with sqrt(2 - delta_m0) folded
// into the diagonal seeds so that  p = sum_{components} c_a c_b  needs no m-weights
// (descriptor/sesoap.py:116-118,195-203: Yr = 2 tril - I, Yi = 2 triu(1)).
struct HarmCoef {
    double a[(kMaxL + 1) * (kMaxL + 1)];  // a[l*(kMaxL+1)+m], m <= l-1
    double b[(kMaxL + 1) * (kMaxL + 1)];  // b[l*(kMaxL+1)+m], m <= l-2
    double qmm[kMaxL + 1];                // Q_mm (with the sqrt(2) weight for m>0)
};

inline void fill_harm_coef(HarmCoef& hc) {
    const int W = kMaxL + 1;
    for (int i = 0; i < W * W; ++i) hc.a[i] = hc.b[i] = 0.0;
    const double pi = 3.14159265358979323846;
    double q = sqrt(1.0 / (4.0 * pi));  // Y00
    hc.qmm[0] = q;
    for (int l = 1; l <= kMaxL; ++l) {
        q *= -sqrt(1.0 + 1.0 / (2.0 * l));  // alp_dl
        hc.qmm[l] = q * sqrt(2.0);
    }
    for (int l = 1; l <= kMaxL; ++l)
        for (int m = 0; m <= l - 1; ++m) {
            hc.a[l * W + m] = sqrt((4.0 * l * l - 1.0) / ((double)l * l - (double)m * m));
            if (m <= l - 2)
                hc.b[l * W + m] = -sqrt((((double)l - 1.0) * ((double)l - 1.0) - (double)m * m) /
                                        (4.0 * ((double)l - 1.0) * ((double)l - 1.0) - 1.0));
        }
}

// index of the real component (l, m, part) in [0, (lmax+1)^2):
//   (l,0) -> l*l ; Re(l,m) -> l*l + 2m-1 ; Im(l,m) -> l*l + 2m
SGPR_HD int comp_index(int l, int m, int im) { return l * l + (m == 0 ? 0 : 2 * m - 1 + im); }

// Solid harmonics of the point (x,y,z) (already in the sheared frame if the shear
// applies).  Calls emit(idx, Y, dYdx, dYdy, dYdz) once per real component; gradients
// are w.r.t. the coordinates passed in.  LMAX is the compile-time bound, lmax the
// actual degree (lmax <= LMAX).
template <int LMAX, bool GRAD, class Emit>
SGPR_HD void solid_harmonics(const HarmCoef& hc, int lmax, double x, double y, double z, Emit&& emit) {
    const int W = kMaxL + 1;
    const double s = x * x + y * y + z * z;
    double Cm = 1.0, Sm = 0.0;     // Re, Im of (x+iy)^m
    double Cm1 = 0.0, Sm1 = 0.0;   // ... of (x+iy)^(m-1)
#pragma unroll
    for (int m = 0; m <= LMAX; ++m) {
        if (m <= lmax) {
            if (m > 0) {
                Cm1 = Cm; Sm1 = Sm;
                Cm = x * Cm1 - y * Sm1;
                Sm = y * Cm1 + x * Sm1;
            }
            // Q, dQ/dz, dQ/ds for l-1 and l-2 at this m
            double q1 = 0.0, q1z = 0.0, q1s = 0.0, q2 = 0.0, q2z = 0.0, q2s = 0.0;
#pragma unroll
            for (int l = m; l <= LMAX; ++l) {
                if (l <= lmax) {
                    double q, qz, qs;
                    if (l == m) {
                        q = hc.qmm[m]; qz = 0.0; qs = 0.0;
                    } else {
                        const double a = hc.a[l * W + m], b = hc.b[l * W + m];
                        q = a * (z * q1 + s * (b * q2));
                        if (GRAD) {
                            qz = a * (q1 + z * q1z + s * (b * q2z));
                            qs = a * (z * q1s + b * q2 + s * (b * q2s));
                        } else { qz = 0.0; qs = 0.0; }
                    }
                    q2 = q1; q2z = q1z; q2s = q1s;
                    q1 = q;  q1z = qz;  q1s = qs;
                    const int base = l * l;
                    if (m == 0) {
                        if (GRAD) emit(base, q, 2.0 * x * qs, 2.0 * y * qs, qz + 2.0 * z * qs);
                        else      emit(base, q, 0.0, 0.0, 0.0);
                    } else {
                        if (GRAD) {
                            const double qm = q * (double)m;
                            const double dz = qz + 2.0 * z * qs;
                            emit(base + 2 * m - 1, q * Cm, 2.0 * x * qs * Cm + qm * Cm1, 2.0 * y * qs * Cm - qm * Sm1, dz * Cm);
                            emit(base + 2 * m,     q * Sm, 2.0 * x * qs * Sm + qm * Sm1, 2.0 * y * qs * Sm + qm * Cm1, dz * Sm);
                        } else {
                            emit(base + 2 * m - 1, q * Cm, 0.0, 0.0, 0.0);
                            emit(base + 2 * m,     q * Sm, 0.0, 0.0, 0.0);
                        }
                    }
                }
            }
        }
    }
}

// ylm.py:16-18 : does this neighbour trigger the environment-wide shear?
SGPR_HD bool near_z_axis(double x, double y, double z) {
    const double tol = kTinyAngle * fabs(z);
    return (fabs(x) < tol) && (fabs(y) < tol);
}

// Radial part in scaled coordinates (d = |r|/u):  R(d) = cut(u d) exp(-d^2/2),
// cut(r) = (1 - r/rc)^2 [r < rc]   (cutoff.py:20-44, sesoap.py:176-183).
// Returns R and  Rp_over_d = R'(d)/d .
SGPR_HD void radial(double d, double u, double rc, double& R, double& Rp_over_d) {
    const double rt = u * d;
    const double step = (rt < rc) ? 1.0 : 0.0;
    const double w = 1.0 - rt / rc;
    const double ex = exp(-0.5 * d * d);
    const double cut = step * w * w;
    const double dcut = step * (-2.0 * w / rc);
    R = cut * ex;
    Rp_over_d = ((u * dcut) * ex) / d - cut * ex;
}

// Same functions for the hot kernels, division-free: d2 = d^2 and rd = 1/d are passed in, rc_inv = 1/rc.
// (1 - rt/rc is formed as 1 - rt * rc_inv: at most one ulp of rt/rc away.)
SGPR_HD void radial_fast(double d2, double d, double rd, double u, double rc, double rc_inv, double& R, double& Rp_over_d) {
    const double rt = u * d;
    const double step = (rt < rc) ? 1.0 : 0.0;
    const double w = 1.0 - rt * rc_inv;
    const double ex = exp(-0.5 * d2);
    const double cut = step * w * w;
    const double dcut = step * (-2.0 * w * rc_inv);
    R = cut * ex;
    Rp_over_d = ((u * dcut) * ex) * rd - cut * ex;
}

// a_{n,l} = 1 / ((2l+1) 2^(2n+l) n! (n+l)!)   (sesoap.py:119-128)
inline double anl(int n, int l) {
    double f1 = 1.0, f2 = 1.0;
    for (int k = 2; k <= n; ++k) f1 *= k;
    for (int k = 2; k <= n + l; ++k) f2 *= k;
    return 1.0 / ((2.0 * l + 1.0) * pow(2.0, 2 * n + l) * f1 * f2);
}

// Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11): counter-based, so the Langevin
// noise of (atom, step) is a pure function of the seed and needs no generator state in memory.  ctr is replaced by the
// output block.
SGPR_HD void philox4x32_10(uint32_t ctr[4], uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; ++r) {
        if (r > 0) {
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        const uint64_t p0 = (uint64_t)0xD2511F53u * ctr[0];
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * ctr[2];
        const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        const uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        const uint32_t c1 = ctr[1], c3 = ctr[3];
        ctr[0] = hi1 ^ c1 ^ k0;
        ctr[1] = lo1;
        ctr[2] = hi0 ^ c3 ^ k1;
        ctr[3] = lo0;
    }
}

// uniform in (0, 1) from the top 53 bits of a 64-bit word (never 0: the logarithm of Box-Muller stays finite)
SGPR_HD double philox_uniform(uint32_t lo, uint32_t hi) {
    const uint64_t x = ((uint64_t)hi << 32) | lo;
    return ((double)(x >> 11) + 0.5) * 1.1102230246251565404e-16;   // 2^-53
}

// Three standard normal deviates of the Langevin O step for one atom and step.  Key = seed; counter = {atom, call,
// step low word, step high word}; output words 0,1 and 2,3 of a block are two 64-bit words (low word first).  Box-Muller
// turns the two uniforms of call 0 into xi[0], xi[1]; the first normal of call 1 is xi[2].
SGPR_HD void langevin_normals(uint64_t seed, uint32_t atom, uint64_t step, double xi[3]) {
    const double two_pi = 6.283185307179586476925;
    for (uint32_t call = 0; call < 2; ++call) {
        uint32_t c[4] = {atom, call, (uint32_t)step, (uint32_t)(step >> 32)};
        philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
        const double u0 = philox_uniform(c[0], c[1]), u1 = philox_uniform(c[2], c[3]);
        const double rad = sqrt(-2.0 * log(u0));
        if (call == 0) {
            xi[0] = rad * cos(two_pi * u1);
            xi[1] = rad * sin(two_pi * u1);
        } else {
            xi[2] = rad * cos(two_pi * u1);
        }
    }
}

}  // namespace sgpr
