// mmi_kernels.cuh -- maximum mutual information training: the kernels that join the decode scores of every
// (utterance, word) cell to the posterior-weighted E-step (hmmcu_estep_mmi), and the extended Baum-Welch update of the
// means and variances (hmmcu_mstep_ebw).  The weighted E-step itself is k_fb_res / k_fb with their WEIGHTED flag.
#pragma once
#include "kernels.cuh"
#include "ebw_math.h"

namespace hmmk {

constexpr int kMmiWarps = 8;  // rows (utterances) per CTA of k_mmi_post, one warp each

// Word posteriors of utterance u, P(w|u) = exp(kappa S[u][w] - lse), lse = logsumexp_w' kappa S[u][w'] (double), and
// the hypotheses of the denominator: the label first, with its posterior however small, then at most H - 1 other words
// in descending order of posterior (lower word index first on a tie), each with P >= min_post.  Outputs, round-major
// so that the weights of one round are contiguous:
//   w[r * U + u]          weight of round r: r = 0 the label, r >= 1 the r-th other word (0 where there is none)
//   hyp[(r - 1) * U + u]  word of round r >= 1, -1 where there is none
//   term[u]               lse - kappa S[u][label]; NaN for an utterance that is left out (label -1, or a label score
//                         that is not finite: weight 0 and no other hypotheses)
// One warp per row; the row stays in L1 over the selection passes.
__global__ void __launch_bounds__(kMmiWarps * 32)
k_mmi_post(const double *__restrict__ S, const int32_t *__restrict__ label, int U, int V, double kappa, int H, double min_post,
           double *__restrict__ w, int32_t *__restrict__ hyp, double *__restrict__ term) {
  const int lane = threadIdx.x & 31;
  const int u = blockIdx.x * kMmiWarps + (threadIdx.x >> 5);
  if (u >= U) return;
  const double *s = S + (int64_t)u * V;
  const int lab = label[u];
  const double sl = lab >= 0 ? s[lab] : NAN;
  int r = 1;
  if (isfinite(sl)) {
    double m = -INFINITY;
    for (int k = lane; k < V; k += 32) m = fmax(m, kappa * s[k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    double z = 0.0;
    for (int k = lane; k < V; k += 32) {
      const double e = exp(kappa * s[k] - m);
      z += (e == e) ? e : 0.0;
    }
    const double lse = m + log(warp_sum(z));
    if (lane == 0) {
      w[u] = exp(kappa * sl - lse);
      term[u] = lse - kappa * sl;
    }
    // selection: the next hypothesis is the largest (a, -k) strictly after the previous one in that order
    double pa = INFINITY;
    int pk = -1;
    for (; r < H; r++) {
      double ba = -INFINITY;
      int bk = 0x7fffffff;
      for (int k = lane; k < V; k += 32) {
        if (k == lab) continue;
        const double a = kappa * s[k] - lse;
        if (!(a < pa || (a == pa && k > pk))) continue;  // (NaN never qualifies)
        if (a > ba || (a == ba && k < bk)) { ba = a; bk = k; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double oa = __shfl_xor_sync(0xffffffffu, ba, o);
        const int ok = __shfl_xor_sync(0xffffffffu, bk, o);
        if (oa > ba || (oa == ba && ok < bk)) { ba = oa; bk = ok; }
      }
      const double p = exp(ba);
      if (bk == 0x7fffffff || !(p >= min_post)) break;
      if (lane == 0) {
        w[(int64_t)r * U + u] = p;
        hyp[(int64_t)(r - 1) * U + u] = bk;
      }
      pa = ba;
      pk = bk;
    }
  } else if (lane == 0) {
    w[u] = 0.0;
    term[u] = NAN;
  }
  for (r += lane; r < H; r += 32) {
    w[(int64_t)r * U + u] = 0.0;
    hyp[(int64_t)(r - 1) * U + u] = -1;
  }
}

// The objective terms of the utterances of every word, in a fixed order: warp v sums term[] over the word's utterances
// (model_start / model_utts: the label map grouped by word, as set_train_map builds it), lane-strided, then by a
// butterfly.  obj[2 v] = sum of the terms, obj[2 v + 1] = the number of included utterances.
__global__ void k_mmi_tail(const double *__restrict__ term, const int32_t *__restrict__ model_start,
                           const int32_t *__restrict__ model_utts, int V, double *__restrict__ obj) {
  const int lane = threadIdx.x & 31;
  const int v = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (v >= V) return;
  double s = 0.0, n = 0.0;
  for (int k = model_start[v] + lane; k < model_start[v + 1]; k += 32) {
    const double t = term[model_utts[k]];
    if (t == t) { s += t; n += 1.0; }
  }
  s = warp_sum(s);
  n = warp_sum(n);
  if (lane == 0) { obj[2 * v] = s; obj[2 * v + 1] = n; }
}

// Extended Baum-Welch update of the means and variances (ebw_math.h): one warp per Gaussian, lanes over the dimensions;
// grid = (ceil(G / 8), V).  The per-dimension roots give D_min by a warp maximum; D = max(2 D_min, E S0_den); a
// Gaussian with dg + D <= 0 keeps its parameters.  Then inv_var = 1 / var and det = the product of the variances in
// index order, as k_mstep_apply forms them.  Mixture weights and transitions are not touched.
__global__ void __launch_bounds__(256)
k_mstep_ebw(const double *__restrict__ num_all, const double *__restrict__ den_all, int64_t ss, int N, int M, int D, double E,
            double tau, double floor_, double *__restrict__ muall, double *__restrict__ ivall, double *__restrict__ detall) {
  const int v = blockIdx.y, G = N * M, lane = threadIdx.x & 31;
  const int k = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (k >= G) return;
  const int64_t oS0 = (int64_t)N * N + 2 * N, oS1 = oS0 + G + (int64_t)k * D, oS2 = oS0 + G + (int64_t)G * D + (int64_t)k * D;
  const double *num = num_all + (int64_t)v * ss, *den = den_all + (int64_t)v * ss;
  double *mu = muall + ((int64_t)v * G + k) * D, *iv = ivall + ((int64_t)v * G + k) * D;
  const double s0n = num[oS0 + k], s0d = den[oS0 + k];
  const double sc = ebw_scale(s0n, tau);
  const double dg = __dsub_rn(__dmul_rn(s0n, sc), s0d);
  auto diffs = [&](int d, double m, double &ds, double &dq) {
    ds = __dsub_rn(__dmul_rn(num[oS1 + d], sc), den[oS1 + d]);
    dq = __dsub_rn(__dmul_rn(ebw_q(num[oS2 + d], num[oS1 + d], s0n, m), sc), ebw_q(den[oS2 + d], den[oS1 + d], s0d, m));
  };
  double dmin = 0.0;
  for (int d = lane; d < D; d += 32) {
    double ds, dq;
    const double m = mu[d];
    diffs(d, m, ds, dq);
    dmin = fmax(dmin, ebw_root(dg, ds, dq, m, __ddiv_rn(1.0, iv[d])));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dmin = fmax(dmin, __shfl_xor_sync(0xffffffffu, dmin, o));
  const double Dc = fmax(__dmul_rn(2.0, dmin), __dmul_rn(E, s0d));
  if (!(__dadd_rn(dg, Dc) > 0.0)) return;  // no occupancy in either block: unchanged
  double dt = 1.0;
  for (int d0 = 0; d0 < D; d0 += 32) {
    const int d = d0 + lane;
    double var = 1.0;
    if (d < D) {
      double ds, dq, mn;
      const double m = mu[d];
      diffs(d, m, ds, dq);
      ebw_update(dg, ds, dq, m, __ddiv_rn(1.0, iv[d]), Dc, floor_, &mn, &var);
      mu[d] = mn;
      iv[d] = __ddiv_rn(1.0, var);
    }
    const int nd = min(32, D - d0);
    for (int j = 0; j < nd; j++) dt = __dmul_rn(dt, __shfl_sync(0xffffffffu, var, j));  // product in index order
  }
  if (lane == 0) detall[(int64_t)v * G + k] = dt;
}

}  // namespace hmmk
