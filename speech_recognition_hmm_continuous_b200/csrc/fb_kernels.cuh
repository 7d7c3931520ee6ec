// fb_kernels.cuh -- scaled forward / backward for Baum-Welch training (calc_alpha, calc_beta,
// calc_transition_probab, calc_den_mix_coef, calc_probability; T-FS:1380-1664), latency-first.
//
// The recursion over time is a dependent chain; what bounds it is the latency of one step, not
// throughput.  So one THREAD owns one utterance and keeps the whole state vector in registers
// (no shuffles on the chain), the forward and the backward chains of an utterance run concurrently in
// two different warps, and each step rescales by an exact power of two taken from the largest exponent
// field of the step's components (integer instructions only; no division, no logarithm, no sum):
//   forward :  z_t = ((z_{t-1} A) o b~_t) 2^-e_t      b~_i(t) = exp(logb_i(t) - m_t), m_t = max_i logb_i(t)
//   backward:  w_t = (A (b~_{t+1} o w_{t+1})) 2^-e'_t  w_{T-1} = [0,..,0,1]   (final state only, T-FS:1484)
// Any positive per-frame scaling gives the same posteriors; the reference's c_t-scaled quantities
// are recovered exactly from per-frame normalisation:
//   alpha^_t(i) beta^_t(i) / c_t          = phi * z_t(i) w_t(i) / sum_j z_t(j) w_t(j)
//   alpha^_t(i) a_ij b_j(t+1) beta^_t+1(j) = phi * z_t(i) a_ij q_j / sum_kl z_t(k) a_kl q_l,  q = b~_{t+1} o w_{t+1}
// with phi = alpha^_{T-1}(N-1) (the reference's beta^ starts from the final state only, so its
// gammas sum to phi, not to 1), and
//   log P = sum_t m_t + ln2 sum_t e_t + log z_{T-1}(N-1)      (calc_probability, T-FS:1546-1549).
// The chain threads never touch global memory for their operands: the six other warps of the CTA stage
// the NEXT window of kFbWin frames of every utterance of the CTA into shared memory as b~ (double) while
// the chains consume the current one (two buffers) -- forward window from the start of the utterance,
// backward window from its end -- so a chain step is NS LDS.64, the banded matvec, the power-of-two
// scaling and two 16-byte stores of the scaled vector as the high words of its doubles (rows of 8 words, d32_pack).
// A second phase (one warp per utterance, lanes over frames) forms gamma, the transition sums and sum m_t.
#pragma once
#include "kernels.cuh"

namespace hmmk {

constexpr int kFbUtts = 8;        // utterances per CTA
constexpr int kFbThreads = 256;   // 8 warps: warp 0 = forward chains, warp 1 = backward chains, warps 2-7 stage; then all combine
constexpr int kFbWin = 64;        // frames per staged window
constexpr int kFbRow = 8;         // floats per row of the alpha / beta workspaces (NS <= 8)

// exp(y) for y <= 0 as a double: single-precision mantissa accuracy (the log-densities it is fed
// are single precision), double-precision range.  y < -700 -> 0.
__device__ __forceinline__ double exp_scaled(float y) {
  // Only ONE operation on the transcendental / conversion unit (ex2): the rounding of y log2(e) to an integer uses
  // the 1.5 * 2^23 trick on the FMA pipe, and the double is assembled from the float's bits with integer
  // instructions (a cvt.f64.f32 and a cvt.rni per value made the decode scorers wait on that unit).
  const float yc = fmaxf(y, -700.f);  // branch-free: the chain's five exponentials must overlap
  const float t = fmaf(yc, 1.4426950408889634f, 12582912.f);         // 1.5 * 2^23 + rint(yc log2 e)
  const float n = t - 12582912.f;
  const int ni = __float_as_int(t) - 0x4B400000;                      // the same integer
  float f = fmaf(yc, 1.4426950216293335f, -n);  // (float)log2(e)
  f = fmaf(yc, 1.9259629911e-8f, f);            // log2(e) - (float)log2(e)
  float p;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(p) : "f"(f));  // |f| <= 0.5: 2 ulp; p in [0.70, 1.42] is a normal float
  const unsigned pb = (unsigned)__float_as_int(p);
  const int hi = (int)(pb >> 3) + ((1023 - 127 + ni) << 20);          // exponent re-biased, 20 of the 23 mantissa bits
  const int lo = (int)(pb << 29);                                     // the other 3
  return (y < -700.f) ? 0.0 : __hiloint2double(hi, lo);
}

template <int NS>
__device__ __forceinline__ void load_lb(const float *__restrict__ p, float (&l)[NS]) {
#pragma unroll
  for (int i = 0; i < NS; i++) l[i] = __ldg(p + i);
}

__host__ __device__ inline size_t fb_smem_bytes(int NS) {
  return (size_t)2 * 2 * kFbUtts * (kFbWin * NS + 2) * sizeof(double);  // [buffer][direction][utterance][window]
}

// 2^-(E - 1023) for the largest exponent field E of the non-negative components v[]; 1 when that field is 0
// (all zero / denormal) or 0x7ff (inf / NaN).  e = E - 1023 (0 in the degenerate cases).
template <int NS>
__device__ __forceinline__ double pow2_scale_max(const double (&v)[NS], int &e) {
  int be = __double2hiint(v[0]) >> 20;
#pragma unroll
  for (int i = 1; i < NS; i++) be = max(be, __double2hiint(v[i]) >> 20);
  const bool ok = be > 0 && be < 0x7ff;
  e = ok ? be - 1023 : 0;
  return __hiloint2double(ok ? (2046 - be) << 20 : 0x3ff00000, 0);
}

// high word of a non-negative double, rounded to nearest: the full double range at 4 bytes per value (a float row
// would flush a state whose mass is below 2^-126 of the frame's largest, and the other chain can lift it back to
// order one: alpha^ beta^ of such a state is not small)
__device__ __forceinline__ uint32_t d32_pack(double v) {
  return (uint32_t)__double2hiint(v) + ((uint32_t)__double2loint(v) >> 31);
}
__device__ __forceinline__ double d32_unpack(uint32_t w) { return __hiloint2double((int)w, 0); }

template <int NS>
__device__ __forceinline__ void store_row(uint32_t *__restrict__ p, const double (&z)[NS]) {
  uint32_t f[kFbRow];
#pragma unroll
  for (int i = 0; i < kFbRow; i++) f[i] = (i < NS) ? d32_pack(z[i]) : 0u;
  *reinterpret_cast<uint4 *>(p) = make_uint4(f[0], f[1], f[2], f[3]);
  if (NS > 4) *reinterpret_cast<uint4 *>(p + 4) = make_uint4(f[4], f[5], f[6], f[7]);
}

// Outputs: gamma32[F][N] (the reference's alpha^ beta^ / c, T-FS:1709); per-model statistics head
// (num_trans, den_trans, den_mix, sum_logp, n_utt) by double atomics, one set per utterance;
// logp_utt[U] (0 for masked utterances).  alpha_ws / beta_ws: [F][kFbRow] workspaces of d32 words.
template <int NS, bool BANDED>
__global__ void __launch_bounds__(kFbThreads)
k_fb(const float *__restrict__ logb, const int64_t *__restrict__ off, const int32_t *__restrict__ u2m,
     const double *__restrict__ Aall, int U, uint32_t *__restrict__ alpha_ws, uint32_t *__restrict__ beta_ws,
     float *__restrict__ gamma, double *__restrict__ stats, int64_t stats_stride, int64_t off_sumlogp,
     double *__restrict__ logp_utt) {
  extern __shared__ __align__(16) uint8_t fb_smem[];
  constexpr int US = kFbWin * NS + 2;  // per-utterance stride, padded: the 8 chain lanes hit 8 different banks
  double *bf = reinterpret_cast<double *>(fb_smem);  // [2 buffers][2 directions][kFbUtts][US]  b~
  __shared__ double sA[kFbUtts][NS * NS];
  __shared__ double sphi[kFbUtts], slp[kFbUtts];
  __shared__ int64_t sbase[kFbUtts];
  __shared__ int sT[kFbUtts];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int u0 = blockIdx.x * kFbUtts;
  for (int idx = tid; idx < kFbUtts * NS * NS; idx += kFbThreads) {
    const int uu = idx / (NS * NS), k = idx - uu * NS * NS;
    const int u = u0 + uu;
    const int v = (u < U) ? u2m[u] : -1;
    sA[uu][k] = (v >= 0) ? Aall[(int64_t)v * NS * NS + k] : 0.0;
  }
  if (tid < kFbUtts) {
    const int u = u0 + tid;
    const bool live = u < U && u2m[u] >= 0;
    sbase[tid] = live ? off[u] : 0;
    sT[tid] = live ? (int)(off[u + 1] - off[u]) : 0;
  }
  __syncthreads();
  int Tmax = 0;
#pragma unroll
  for (int uu = 0; uu < kFbUtts; uu++) Tmax = max(Tmax, sT[uu]);

  // Staging of window w0 into buffer `buf` by `nthr` threads (index t0): item <-> (direction, utterance, frame).
  // Three items per pass so that their loads are in flight together.
  auto stage = [&](int w0, int buf, int t0, int nthr) {
    constexpr int NIT = 2 * kFbUtts * kFbWin, PASS = 3;
    double *dstb = bf + (size_t)buf * 2 * kFbUtts * US;
    for (int it0 = t0; it0 < NIT; it0 += PASS * nthr) {
      float l[PASS][NS];
      double *dst[PASS];
#pragma unroll
      for (int p = 0; p < PASS; p++) {
        const int it = it0 + p * nthr;
        dst[p] = nullptr;
        if (it < NIT) {
          const int dir = it / (kFbUtts * kFbWin), rem = it - dir * (kFbUtts * kFbWin);
          const int uu = rem / kFbWin, k = rem - uu * kFbWin;
          const int T = sT[uu];
          if (w0 + k < T) {
            const int t = dir == 0 ? w0 + k : T - 1 - (w0 + k);
            load_lb<NS>(logb + (sbase[uu] + t) * NS, l[p]);
            dst[p] = dstb + (size_t)(dir * kFbUtts + uu) * US + k * NS;
          }
        }
      }
#pragma unroll
      for (int p = 0; p < PASS; p++) {
        if (dst[p]) {
          float m = l[p][0];
#pragma unroll
          for (int i = 1; i < NS; i++) m = fmaxf(m, l[p][i]);
          const float ms = (m > kNegInf) ? m : 0.f;  // all states at -inf: every b~ is 0 (not NaN)
#pragma unroll
          for (int i = 0; i < NS; i++) dst[p][i] = exp_scaled(l[p][i] - ms);
        }
      }
    }
  };

  // ---------------- phase 1: the two chains of each utterance, one thread each ----------------
  const bool chain = warp < 2 && lane < kFbUtts && sT[lane & (kFbUtts - 1)] > 0;
  const int myT = chain ? sT[lane] : 0;
  const int64_t mybase = chain ? sbase[lane] : 0;
  double a[NS * NS];
#pragma unroll
  for (int k = 0; k < NS * NS; k++) a[k] = chain ? sA[lane][k] : 0.0;
  double z[NS];  // forward: z_t; backward: w_t
#pragma unroll
  for (int i = 0; i < NS; i++) z[i] = (warp == 1 && i == NS - 1) ? 1.0 : 0.0;
  int esum = 0;
  if (chain && warp == 1) store_row<NS>(beta_ws + (mybase + myT - 1) * kFbRow, z);  // final state only, T-FS:1484-1490
  stage(0, 0, tid, kFbThreads);
  __syncthreads();
  for (int w0 = 0, wi = 0; w0 < Tmax; w0 += kFbWin, wi++) {
    const double *bcur = bf + (size_t)(wi & 1) * 2 * kFbUtts * US;
    if (warp >= 2) {
      if (w0 + kFbWin < Tmax) stage(w0 + kFbWin, (wi + 1) & 1, tid - 64, kFbThreads - 64);
    } else if (chain && warp == 0) {  // forward: frames w0 .. w0+kFbWin-1
      const double *bw = bcur + (size_t)lane * US;
      const int kend = min(kFbWin, myT - w0);
      uint32_t *ap = alpha_ws + (mybase + w0) * kFbRow;
      for (int k = 0; k < kend; k++) {
        double b[NS], raw[NS];
#pragma unroll
        for (int i = 0; i < NS; i++) b[i] = bw[k * NS + i];
        if (w0 + k == 0) {
#pragma unroll
          for (int i = 0; i < NS; i++) raw[i] = (i == 0) ? b[0] : 0.0;  // pi = [1,0,..,0]  T-FS:232-234
        } else {
#pragma unroll
          for (int i = 0; i < NS; i++) {
            double aux;
            if (BANDED) {
              aux = z[i] * a[i * NS + i];
              if (i > 0) aux = fma(z[i - 1], a[(i - 1) * NS + i], aux);
            } else {
              aux = 0.0;
#pragma unroll
              for (int j = 0; j < NS; j++) aux = fma(z[j], a[j * NS + i], aux);
            }
            raw[i] = aux * b[i];
          }
        }
        int e;
        const double r = pow2_scale_max<NS>(raw, e);
#pragma unroll
        for (int i = 0; i < NS; i++) z[i] = raw[i] * r;
        store_row<NS>(ap + (size_t)k * kFbRow, z);
        esum += e;
      }
    } else if (chain && warp == 1) {  // backward: step j = w0 + k turns beta~_{T-1-j} into beta~_{T-2-j} with b~ of frame T-1-j
      const double *bw = bcur + (size_t)(kFbUtts + lane) * US;
      const int kend = min(kFbWin, myT - 1 - w0);
      for (int k = 0; k < kend; k++) {
        double q[NS], raw[NS];
#pragma unroll
        for (int j = 0; j < NS; j++) q[j] = bw[k * NS + j] * z[j];
#pragma unroll
        for (int i = 0; i < NS; i++) {
          double aux;
          if (BANDED) {
            aux = a[i * NS + i] * q[i];
            if (i + 1 < NS) aux = fma(a[i * NS + i + 1], q[i + 1], aux);
          } else {
            aux = 0.0;
#pragma unroll
            for (int j = 0; j < NS; j++) aux = fma(a[i * NS + j], q[j], aux);
          }
          raw[i] = aux;
        }
        int e;
        const double r = pow2_scale_max<NS>(raw, e);
#pragma unroll
        for (int i = 0; i < NS; i++) z[i] = raw[i] * r;
        store_row<NS>(beta_ws + (mybase + myT - 2 - (w0 + k)) * kFbRow, z);
      }
    }
    __syncthreads();  // window consumed, next one staged
  }
  if (chain && warp == 0) {
    double s = z[0];
#pragma unroll
    for (int i = 1; i < NS; i++) s += z[i];
    sphi[lane] = z[NS - 1] / s;                                       // alpha^_{T-1}(N-1)
    slp[lane] = 0.6931471805599453 * (double)esum + log(z[NS - 1]);  // + sum m_t, added in phase 2
  }
  __syncthreads();
  // ---------------- phase 2: one warp per utterance, lanes over frames ----------------
  for (int uu = warp; uu < kFbUtts; uu += kFbThreads / 32) {
    const int u = u0 + uu;
    if (u >= U) continue;
    const int v = u2m[u];
    if (v < 0) {  // masked utterance (its model has converged)
      if (lane == 0 && logp_utt) logp_utt[u] = 0.0;
      continue;
    }
    const int64_t base = off[u];
    const int T = (int)(off[u + 1] - base);
    const double *A = sA[uu];
    const double phi = sphi[uu];
    double acc_num[NS][2], acc_dt[NS], acc_dm[NS], acc_m = 0.0;
#pragma unroll
    for (int i = 0; i < NS; i++) { acc_num[i][0] = acc_num[i][1] = 0.0; acc_dt[i] = 0.0; acc_dm[i] = 0.0; }
    // the rows of frame t + 32 are fetched while frame t is being worked on (the loop is latency bound otherwise)
    struct Raw { uint4 a0, a1, b0, b1, c0, c1; float l0[NS], l1[NS]; };
    auto fetch = [&](int t, Raw &r) {
      const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
      r.a0 = r.a1 = r.b0 = r.b1 = r.c0 = r.c1 = z4;
#pragma unroll
      for (int i = 0; i < NS; i++) r.l0[i] = r.l1[i] = 0.f;
      if (t < T) {
        const uint4 *pa = reinterpret_cast<const uint4 *>(alpha_ws + (base + t) * kFbRow);
        const uint4 *pb = reinterpret_cast<const uint4 *>(beta_ws + (base + t) * kFbRow);
        r.a0 = pa[0]; r.b0 = pb[0];
        if (NS > 4) { r.a1 = pa[1]; r.b1 = pb[1]; }
        load_lb<NS>(logb + (base + t) * NS, r.l0);
        if (t < T - 1) {
          r.c0 = pb[2];  // beta row of frame t + 1 (rows are kFbRow = 8 words)
          if (NS > 4) r.c1 = pb[3];
          load_lb<NS>(logb + (base + t + 1) * NS, r.l1);
        }
      }
    };
    auto unpack = [](const uint4 &x0, const uint4 &x1, double (&o)[NS]) {
      const uint32_t f[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
      for (int i = 0; i < NS; i++) o[i] = d32_unpack(f[i]);
    };
    Raw cur, nxt;
    fetch(lane, cur);
    for (int t = lane; t < T; t += 32) {
      fetch(t + 32, nxt);
      double al[NS], be[NS], g[NS], G = 0.0;
      unpack(cur.a0, cur.a1, al);
      unpack(cur.b0, cur.b1, be);
      {
        float m = cur.l0[0];
#pragma unroll
        for (int i = 1; i < NS; i++) m = fmaxf(m, cur.l0[i]);
        acc_m += (double)m;  // sum_t m_t  (calc_probability); -inf when a frame has no density at all
      }
#pragma unroll
      for (int i = 0; i < NS; i++) {
        g[i] = al[i] * be[i];
        G += g[i];
      }
      const double sc = (G > 0.0) ? phi / G : 0.0;  // unreachable final state: no occupancy, as the reference
#pragma unroll
      for (int i = 0; i < NS; i++) {
        g[i] *= sc;  // alpha^ beta^ / c   T-FS:1617,1658,1709
        gamma[(base + t) * NS + i] = (float)g[i];
        acc_dm[i] += g[i];
      }
      if (t < T - 1) {
        float m = cur.l1[0];
#pragma unroll
        for (int i = 1; i < NS; i++) m = fmaxf(m, cur.l1[i]);
        double q[NS], b1[NS];
        unpack(cur.c0, cur.c1, b1);
#pragma unroll
        for (int j = 0; j < NS; j++) q[j] = exp_scaled(cur.l1[j] - ((m > kNegInf) ? m : 0.f)) * b1[j];
        double Z = 0.0;
#pragma unroll
        for (int i = 0; i < NS; i++) {
          double rb = 0.0;
#pragma unroll
          for (int j = 0; j < NS; j++) rb = fma(A[i * NS + j], q[j], rb);
          Z = fma(al[i], rb, Z);
        }
        const double zs = (Z > 0.0) ? phi / Z : 0.0;
#pragma unroll
        for (int i = 0; i < NS; i++) {
          acc_dt[i] += g[i];
          acc_num[i][0] += al[i] * A[i * NS + i] * q[i] * zs;                              // band j = i   T-FS:1611
          if (i + 1 < NS) acc_num[i][1] += al[i] * A[i * NS + i + 1] * q[i + 1] * zs;      // j = i + 1
        }
      }
      cur = nxt;
    }
    double *st = stats + (int64_t)v * stats_stride;
#pragma unroll
    for (int i = 0; i < NS; i++) {
      const double n0 = warp_sum(acc_num[i][0]), n1 = warp_sum(acc_num[i][1]);
      const double dt = warp_sum(acc_dt[i]), dm = warp_sum(acc_dm[i]);
      if (lane == 0) {
        atomicAdd(st + i * NS + i, n0);
        if (i + 1 < NS) atomicAdd(st + i * NS + i + 1, n1);
        atomicAdd(st + NS * NS + i, dt);
        atomicAdd(st + NS * NS + NS + i, dm);
      }
    }
    const double msum = warp_sum(acc_m);
    if (lane == 0) {
      const double lp = slp[uu] + msum;  // calc_probability T-FS:1546-1549
      atomicAdd(st + off_sumlogp, lp);
      atomicAdd(st + off_sumlogp + 1, 1.0);
      if (logp_utt) logp_utt[u] = lp;
    }
  }
}

}  // namespace hmmk
