/* ebw_math.h -- the per-dimension arithmetic of the extended Baum-Welch update (hmmh_mstep_ebw on the host, k_mstep_ebw
 * on the device).  One source for both compilers: on the device every operation is an explicitly rounded intrinsic, so
 * nvcc cannot contract a product and a sum into an FMA, and both sides round every operation the same way (the host
 * build has no FMA contraction either).  Plain C; included by hmm_host.c and mmi_kernels.cuh.
 *
 * Statistics of one Gaussian and dimension: S0 (occupancy), S1 = sum gamma x, S2c = sum gamma (x - mu)^2 about the
 * current mean mu; num = the label's (numerator) block, den = the posterior-weighted (denominator) block. */
#ifndef HMM_EBW_MATH_H
#define HMM_EBW_MATH_H

#if defined(__CUDA_ARCH__)
#define EBW_FN __device__ __forceinline__
#define EBW_ADD(a, b) __dadd_rn((a), (b))
#define EBW_SUB(a, b) __dsub_rn((a), (b))
#define EBW_MUL(a, b) __dmul_rn((a), (b))
#define EBW_DIV(a, b) __ddiv_rn((a), (b))
#define EBW_SQRT(a) __dsqrt_rn(a)
#else
#include <math.h>
#ifdef __CUDACC__
#define EBW_FN __host__ static inline
#else
#define EBW_FN static inline
#endif
#define EBW_ADD(a, b) ((a) + (b))
#define EBW_SUB(a, b) ((a) - (b))
#define EBW_MUL(a, b) ((a) * (b))
#define EBW_DIV(a, b) ((a) / (b))
#define EBW_SQRT(a) sqrt(a)
#endif

/* I-smoothing factor of the numerator's (S0, S1, Q): 1 + tau / S0_num, or 1 when the numerator has no occupancy */
EBW_FN double ebw_scale(double s0n, double tau) { return s0n > 0.0 ? EBW_ADD(1.0, EBW_DIV(tau, s0n)) : 1.0; }

/* Q = sum gamma x^2 = S2c + 2 mu S1 - mu^2 S0 */
EBW_FN double ebw_q(double s2c, double s1, double s0, double mu) {
  return EBW_SUB(EBW_ADD(s2c, EBW_MUL(EBW_MUL(2.0, mu), s1)), EBW_MUL(EBW_MUL(mu, mu), s0));
}

/* The largest real root of var D^2 + (dq + dg (var + mu^2) - 2 mu ds) D + (dq dg - ds^2): above it the new variance is
 * positive.  0 when no root is positive. */
EBW_FN double ebw_root(double dg, double ds, double dq, double mu, double var) {
  const double b = EBW_SUB(EBW_ADD(dq, EBW_MUL(dg, EBW_ADD(var, EBW_MUL(mu, mu)))), EBW_MUL(EBW_MUL(2.0, mu), ds));
  const double c = EBW_SUB(EBW_MUL(dq, dg), EBW_MUL(ds, ds));
  const double disc = EBW_SUB(EBW_MUL(b, b), EBW_MUL(EBW_MUL(4.0, var), c));
  if (!(disc >= 0.0)) return 0.0;
  const double r = EBW_DIV(EBW_ADD(-b, EBW_SQRT(disc)), EBW_MUL(2.0, var));
  return r > 0.0 ? r : 0.0;
}

/* The new mean and variance (variance about the NEW mean, floored) for the constant Dc, dg + Dc > 0 */
EBW_FN void ebw_update(double dg, double ds, double dq, double mu, double var, double Dc, double floor_, double *mu_new,
                       double *var_new) {
  const double den = EBW_ADD(dg, Dc);
  const double m = EBW_DIV(EBW_ADD(ds, EBW_MUL(Dc, mu)), den);
  double v = EBW_SUB(EBW_DIV(EBW_ADD(dq, EBW_MUL(Dc, EBW_ADD(var, EBW_MUL(mu, mu)))), den), EBW_MUL(m, m));
  if (v < floor_) v = floor_;
  *mu_new = m;
  *var_new = v;
}

#endif
