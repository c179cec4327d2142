/*
 * sag_detmath.h -- deterministic double-precision sin / cos / atan2 / log.
 *
 * Why: the parity bar of this repo is "GPU == oracle, bit for bit".  +, -, *, /, sqrt are correctly rounded
 * IEEE operations on both sides (nvcc -fmad=false, gcc -ffp-contract=off), but libm's and CUDA's
 * transcendental functions differ in the last ulp, and the point robot's stiff yaw servo plus box contacts
 * amplify an ulp into 1e-4 m within a thousand steps.  These routines are written with plain IEEE
 * operations in a fixed order, so the CUDA kernels and the CPU oracle get identical bits from them.
 *
 * The algorithms are the classic fdlibm ones (Cody-Waite reduction by pi/2 + minimax kernels; argument
 * range splitting for atan; 2^k(1+f) decomposition for log).  Accuracy against a long-double reference
 * (tests/test_detmath.py): sin / cos <= 1.5 ulp for |x| <= 20 and <= 3 ulp up to |x| = 7e4 away from their
 * zeros, where only an absolute bound holds (<= 5e-22 next to multiples of pi/2); atan2 <= 1.5 ulp; log
 * <= 0.9 ulp.  That is libm's class of accuracy, so neither side gains or loses fidelity to the reference,
 * which itself just calls numpy / MuJoCo's libm.
 *
 * Valid C99 and CUDA C++.  Used by oracle/sag_oracle.c and safe_adaptation_gym_b200/csrc/sag_core.cuh.
 */
#ifndef SAG_DETMATH_H
#define SAG_DETMATH_H
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define SAG_DM __host__ __device__ __forceinline__
#else
#define SAG_DM static inline
#endif

/* Horner steps use an explicit fused multiply-add: fma() is exactly specified by IEEE 754 (one rounding), so glibc's
 * fma and the GPU's DFMA give the same bits, and the polynomials cost half the instructions of separate mul + add
 * (the rest of the code base is compiled without contraction, see DESIGN.md 2). */
#define SAG_FMA(a, b, c) fma((a), (b), (c))

/* Polynomial coefficients.  On the device they live in constant memory so that DFMA/DMUL/DADD read them as constant-bank
 * operands (as 64-bit immediates every use costs two extra UMOV instructions: 10 % of the lidar kernel's instructions). */
#define SAG_DM_COEFFS                                                                                                     \
  { /* 0..5 sin S1..S6 */                                                                                                 \
    -1.66666666666666324348e-01, 8.33333333332248946124e-03, -1.98412698298579493134e-04, 2.75573137070700676789e-06,     \
    -2.50507602534068634195e-08, 1.58969099521155010221e-10,                                                              \
    /* 6..11 cos C1..C6 */                                                                                                \
    4.16666666666666019037e-02, -1.38888888888741095749e-03, 2.48015872894767294178e-05, -2.75573143513906633035e-07,     \
    2.08757232129817482790e-09, -1.13596475577881948265e-11,                                                              \
    /* 12..22 atan aT0..aT10 */                                                                                           \
    3.33333333333329318027e-01, -1.99999999998764832476e-01, 1.42857142725034663711e-01, -1.11111104054623557880e-01,     \
    9.09088713343650656196e-02, -7.69187620504482999495e-02, 6.66107313738753120669e-02, -5.83357013379057348645e-02,     \
    4.97687799461593236017e-02, -3.65315727442169155270e-02, 1.62858201153657823623e-02,                                  \
    /* 23..29 log Lg1..Lg7 */                                                                                             \
    6.666666666666735130e-01, 3.999999999940941908e-01, 2.857142874366239149e-01, 2.222219843214978396e-01,               \
    1.818357216161805012e-01, 1.531383769920937332e-01, 1.479819860511658591e-01                                          \
  }
#if defined(__CUDACC__)
static __constant__ double sag_dm_coeff_dev[30] = SAG_DM_COEFFS;
#endif
static const double sag_dm_coeff_host[30] = SAG_DM_COEFFS;
#if defined(__CUDA_ARCH__)
#define SAG_K(i) sag_dm_coeff_dev[i]
#else
#define SAG_K(i) sag_dm_coeff_host[i]
#endif

SAG_DM double sag_dm_from_bits(uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double((long long)b);
#else
  double d;
  memcpy(&d, &b, sizeof(d));
  return d;
#endif
}
SAG_DM uint64_t sag_dm_bits(double d) {
#if defined(__CUDA_ARCH__)
  return (uint64_t)__double_as_longlong(d);
#else
  uint64_t b;
  memcpy(&b, &d, sizeof(b));
  return b;
#endif
}

/* sin and cos of x, |x| < ~1e5 (yaw angles and sim time); beyond that accuracy degrades gracefully */
SAG_DM void sag_sincos(double x, double* sn, double* cs) {
  const double invpio2 = 6.36619772367581382433e-01;
  const double pio2_1 = 1.57079632673412561417e+00;  /* first 33 bits of pi/2 */
  const double pio2_1t = 6.07710050650619224932e-11; /* pi/2 - pio2_1 */
  double fk = x * invpio2;
  fk = fk >= 0.0 ? fk + 0.5 : fk - 0.5;
  long long k = (long long)fk; /* round to nearest, ties away from zero */
  double dk = (double)k;
  double r = (x - dk * pio2_1) - dk * pio2_1t;
  double z = r * r;
  /* kernel sin */
  const double S1 = SAG_K(0), S2 = SAG_K(1), S3 = SAG_K(2), S4 = SAG_K(3), S5 = SAG_K(4), S6 = SAG_K(5);
  double ps = SAG_FMA(z, SAG_FMA(z, SAG_FMA(z, SAG_FMA(z, S6, S5), S4), S3), S2);
  double ks = SAG_FMA(r * z, SAG_FMA(z, ps, S1), r);
  /* kernel cos */
  const double C1 = SAG_K(6), C2 = SAG_K(7), C3 = SAG_K(8), C4 = SAG_K(9), C5 = SAG_K(10), C6 = SAG_K(11);
  double pc = z * SAG_FMA(z, SAG_FMA(z, SAG_FMA(z, SAG_FMA(z, SAG_FMA(z, C6, C5), C4), C3), C2), C1);
  double hz = 0.5 * z;
  double w = 1.0 - hz;
  double kc = w + SAG_FMA(z, pc, (1.0 - w) - hz);
  int q = (int)(k & 3);
  double s = (q & 1) ? kc : ks;
  double c = (q & 1) ? ks : kc;
  if (q == 1 || q == 2) c = -c;
  if (q >= 2) s = -s;
  *sn = s;
  *cs = c;
}
SAG_DM double sag_sin(double x) { double s, c; sag_sincos(x, &s, &c); return s; }
SAG_DM double sag_cos(double x) { double s, c; sag_sincos(x, &s, &c); return c; }

/* atan(t), t >= 0.  fdlibm's four-way range reduction written without branches: the reduced argument is always one
 * division num / den (num = t, den = 1 in the lowest range -- exact), and the reconstruction hi - ((x*s - lo) - x) with
 * hi = lo = 0 equals x - x*s bit for bit (fma(x, s, -0) = x*s rounded once).  No divergence between the lanes of a warp. */
SAG_DM double sag_atan_pos(double t) {
  const int r1 = t >= 0.4375, r2 = t >= 0.6875, r3 = t >= 1.1875, r4 = t >= 2.4375;
  double num = r4 ? -1.0 : (r3 ? t - 1.5 : (r2 ? t - 1.0 : (r1 ? 2.0 * t - 1.0 : t)));
  double den = r4 ? t : (r3 ? 1.0 + 1.5 * t : (r2 ? t + 1.0 : (r1 ? 2.0 + t : 1.0)));
  double hi = r4 ? 1.57079632679489655800e+00 : (r3 ? 9.82793723247329054082e-01 : (r2 ? 7.85398163397448278999e-01 : (r1 ? 4.63647609000806093515e-01 : 0.0)));
  double lo = r4 ? 6.12323399573676603587e-17 : (r3 ? 1.39033110312309984516e-17 : (r2 ? 3.06161699786838301793e-17 : (r1 ? 2.26987774529616870924e-17 : 0.0)));
  double x = num / den;
  double z = x * x;
  double w = z * z;
  double s1 = z * SAG_FMA(w, SAG_FMA(w, SAG_FMA(w, SAG_FMA(w, SAG_FMA(w, SAG_K(22), SAG_K(20)), SAG_K(18)), SAG_K(16)), SAG_K(14)), SAG_K(12));
  double s2 = w * SAG_FMA(w, SAG_FMA(w, SAG_FMA(w, SAG_FMA(w, SAG_K(21), SAG_K(19)), SAG_K(17)), SAG_K(15)), SAG_K(13));
  return hi - (SAG_FMA(x, s1 + s2, -lo) - x);
}

/* atan2(y, x) in (-pi, pi]; atan2(0, 0) = 0 like numpy.angle */
SAG_DM double sag_atan2(double y, double x) {
  const double pi = 3.1415926535897931160e+00, pi_lo = 1.2246467991473531772e-16, pio2 = 1.57079632679489655800e+00;
  if (y == 0.0) return x >= 0.0 ? 0.0 : pi;
  if (x == 0.0) return y > 0.0 ? pio2 : -pio2;
  double ay = y < 0.0 ? -y : y, ax = x < 0.0 ? -x : x;
  double z = sag_atan_pos(ay / ax);
  if (x > 0.0) return y > 0.0 ? z : -z;
  return y > 0.0 ? pi - (z - pi_lo) : (z - pi_lo) - pi;
}

/* Lidar angle -> (bin, alias) for 16 bins (safe_adaptation_gym.py:210-216): with t = (atan2(ey, ex) mod 2 pi) / (2 pi / 16),
 * bin = floor(t) and alias = t - bin.  Instead of a full atan2 (two divisions, a four-way range reduction) the vector is
 * folded into the first half-bin -- |.| of both components, a swap about 45 deg, a reflection about 22.5 deg whose
 * tangent is (x - y) / (x + y) -- so that ONE division feeds the lowest-range atan polynomial (|r| <= tan(pi/8) < 0.4375,
 * no reduction), and the folds are undone on the integer bin index.  A fold turns t into c - t: the fraction becomes
 * 1 - a and the bin the one below.  On an exact bin edge this names the neighbouring bin with alias 1 instead of alias 0,
 * which yields the same three lidar contributions (s, 1*s, 0*s).  Agrees with the literal formula to a few ulp of t
 * (tests/test_detmath.py); the oracle keeps the literal one next to it (orc_lidar_literal). */
SAG_DM void sag_lidar_bin16(double ex, double ey, int* bin, double* alias) {
  const double tan_pi_8 = 4.1421356237309503e-01, eight_over_pi = 2.5464790894703255e+00;
  double ax = fabs(ex), ay = fabs(ey);
  const int s1 = ay > ax;
  double x = s1 ? ay : ax, y = s1 ? ax : ay;
  const int s2 = y > x * tan_pi_8;
  double num = s2 ? x - y : y, den = s2 ? x + y : x;
  double r = den > 0.0 ? num / den : 0.0; /* the zero vector has angle 0 like numpy.angle */
  double z = r * r;
  double w = z * z;
  double p1 = z * SAG_FMA(w, SAG_FMA(w, SAG_FMA(w, SAG_FMA(w, SAG_FMA(w, SAG_K(22), SAG_K(20)), SAG_K(18)), SAG_K(16)), SAG_K(14)), SAG_K(12));
  double p2 = w * SAG_FMA(w, SAG_FMA(w, SAG_FMA(w, SAG_FMA(w, SAG_K(21), SAG_K(19)), SAG_K(17)), SAG_K(15)), SAG_K(13));
  double a = (r - r * (p1 + p2)) * eight_over_pi; /* atan(r) in bins */
  int B = s2 ? 2 : 0, neg = s2;
  if (s1) { B = 4 - B; neg ^= 1; }
  if (ex < 0.0) { B = 8 - B; neg ^= 1; }
  if (ey < 0.0) { B = 16 - B; neg ^= 1; }
  *bin = neg ? B - 1 : B;
  *alias = neg ? 1.0 - a : a;
}

/* natural log of a positive normal double */
SAG_DM double sag_log(double x) {
  const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10;
  const double Lg1 = SAG_K(23), Lg2 = SAG_K(24), Lg3 = SAG_K(25), Lg4 = SAG_K(26), Lg5 = SAG_K(27), Lg6 = SAG_K(28), Lg7 = SAG_K(29);
  uint64_t b = sag_dm_bits(x);
  int32_t hx = (int32_t)(b >> 32);
  uint32_t lx = (uint32_t)b;
  int k = (hx >> 20) - 1023;
  hx &= 0x000fffff;
  int32_t i = (hx + 0x95f64) & 0x100000;
  uint64_t nb = ((uint64_t)(uint32_t)(hx | (i ^ 0x3ff00000)) << 32) | lx; /* normalise x or x/2 */
  k += i >> 20;
  double f = sag_dm_from_bits(nb) - 1.0;
  double dk = (double)k;
  double s = f / (2.0 + f);
  double z = s * s;
  double w = z * z;
  double t1 = w * SAG_FMA(w, SAG_FMA(w, Lg6, Lg4), Lg2);
  double t2 = z * SAG_FMA(w, SAG_FMA(w, SAG_FMA(w, Lg7, Lg5), Lg3), Lg1);
  double R = t2 + t1;
  double hfsq = 0.5 * f * f;
  return dk * ln2_hi - ((hfsq - (s * (hfsq + R) + dk * ln2_lo)) - f);
}

#endif
