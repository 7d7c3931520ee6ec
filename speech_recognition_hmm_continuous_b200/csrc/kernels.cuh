// kernels.cuh -- CUDA kernels (sm_100a) of the continuous-HMM hot path: feature / model packing,
// Gaussian-mixture emissions, scaled forward / backward with Baum-Welch accumulation, forward
// scoring, Viterbi, ranking.  Reference rows are those of SURVEY.md section 8a:
//   T-FS = train/source/hmm-fs/hmm_continuous_fs.c, R-FS = test/source/recognition-fs/...
//
// Numerical plan (DESIGN.md section 3): features and means are centred per dimension in double
// and stored in single precision; emissions are single-precision LOG densities; the recursions
// keep their state (alpha^, beta~, c~) in double and rescale every frame by the frame's largest
// log-density, which is algebraically the reference's 1/sum(alpha) scaling but cannot underflow;
// sufficient statistics are accumulated block-locally in single precision over bounded spans and
// flushed with double-precision atomics.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace hmmk {

constexpr float kNegInf = -INFINITY;
// log of the smallest positive double (4.94e-324): below this the reference's linear-domain
// densities are exactly 0 (SURVEY 0.2).
constexpr double kLogTrueMin = -744.4400719213812;

__host__ __device__ inline int round_up(int a, int b) { return (a + b - 1) / b * b; }

// Programmatic dependent launch (launch_pdl in hmmcu.cu).  pdl_wait() returns once the kernels this one depends on
// have completed and their writes are visible (at once after a plain launch); a kernel launched with launch_pdl calls
// it in every CTA before it reads anything an earlier kernel of its launch sequence wrote and before its first global
// write.  pdl_trigger() lets the next kernel of the stream be scheduled once every CTA of this one has called it or
// exited, so that its launch and prologue overlap this kernel's drain.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------
// centre: per-dimension mean of up to 4096 evenly strided frames (deterministic, one block).
// ------------------------------------------------------------------------------------------------
__global__ void k_center(const double *__restrict__ x, int64_t F, int D, int DP, double *__restrict__ ctr) {
  __shared__ double part[16][64];
  const int d = threadIdx.x & 63, grp = threadIdx.x >> 6;  // 1024 threads = 64 dims x 16 groups
  int64_t ns = F < 4096 ? F : 4096;
  int64_t stride = F / ns;
  for (int d0 = 0; d0 < DP; d0 += 64) {
    double s = 0.0;
    if (d0 + d < D)
      for (int64_t k = grp; k < ns; k += 16) s += x[(k * stride) * D + d0 + d];
    part[grp][d] = s;
    __syncthreads();
    if (grp == 0 && d0 + d < DP) {
      double t = 0.0;
      for (int g = 0; g < 16; g++) t += part[g][d];
      ctr[d0 + d] = (d0 + d < D) ? t / (double)ns : 0.0;
    }
    __syncthreads();
  }
}

// x64[F][D] -> x32[F][DP] = (float)(x - ctr); column D holds 1.0 (so that the first-order
// accumulator of that column is the occupancy S0), remaining pad columns 0.
// xabs[d] (float bits, zero-initialised) receives max |x - ctr| per dimension: the data radius that
// decides whether the expanded quadratic of the tensor-core emission path is accurate enough.
__global__ void k_pack_features(const double *__restrict__ x, const double *__restrict__ ctr, int64_t F, int D,
                                int DP, float *__restrict__ out, unsigned int *__restrict__ xabs) {
  __shared__ unsigned int smax[256];
  for (int i = threadIdx.x; i < DP; i += blockDim.x) smax[i] = 0u;
  __syncthreads();
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = F * DP;
  for (; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t f = idx / DP;
    int d = (int)(idx - f * DP);
    float v;
    if (d < D) {
      v = (float)(x[f * D + d] - ctr[d]);
      atomicMax(&smax[d], __float_as_uint(fabsf(v)));
    } else v = (d == D) ? 1.0f : 0.0f;
    out[idx] = v;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < D; i += blockDim.x) atomicMax(&xabs[i], smax[i]);
}

// Per Gaussian g (global index over V*N*M): mu32[g][DP] = mu - ctr, iv32[g][DP] = inverse variance
// (0 in the pad columns), k32[g] = log c - 0.5 (D log 2pi + log|det|)   [calc_gaus T-FS:1821-1836 in
// log form; c == 0 or det == 0 give -inf, i.e. density 0].
__global__ void k_pack_models(const double *__restrict__ mu, const double *__restrict__ iv,
                              const double *__restrict__ det, const double *__restrict__ c,
                              const double *__restrict__ ctr, int64_t VG, int D, int DP, float *__restrict__ mu32,
                              float *__restrict__ iv32, float *__restrict__ k32) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = VG * DP;
  for (; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t g = idx / DP;
    int d = (int)(idx - g * DP);
    if (d < D) {
      mu32[idx] = (float)(mu[g * D + d] - ctr[d]);
      iv32[idx] = (float)iv[g * D + d];
    } else {
      mu32[idx] = 0.f;
      iv32[idx] = 0.f;
    }
    if (d == 0) {
      double dt = det[g], cc = c[g];
      double k = -INFINITY;
      if (dt != 0.0 && cc > 0.0) k = log(cc) - 0.5 * ((double)D * 1.8378770664093453 + log(fabs(dt)));
      k32[g] = (float)k;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Emissions, CUDA-core version (calc_symbol_probab + calc_gaus, T-FS:1749-1841 / R-FS:860-947).
// One CTA = one tile of <= 64 frames against one model; Gaussians are processed in chunks of whole
// states (<= kGC Gaussians) staged in shared memory.
//   logb[(f - fbase) * ldb + colbase(v) + i] = log sum_m c_m N_m(x_f)
//   post[f * G + i*M + m] = c_m N_m / b_i   (training only)
// ------------------------------------------------------------------------------------------------
struct EmisTile {
  int64_t f0;  // first frame (global index)
  int nf;      // frames in the tile (<= 64)
  int v;       // model
};

constexpr int kEmisTF = 64;       // frames per tile
constexpr int kEmisThreads = 256;

// dynamic shared memory: par[GC][DP] float2 (mu, iv) | xs[DP][64] | lnt[GC][65] | lbs[SC][64]
__host__ __device__ inline size_t emis_smem_bytes(int GC, int SC, int DP) {
  return sizeof(float) * ((size_t)GC * DP * 2 + (size_t)DP * kEmisTF + (size_t)GC * (kEmisTF + 1) + (size_t)SC * kEmisTF) + 16;
}

template <bool POST>
__global__ void __launch_bounds__(kEmisThreads)
k_emis_simt(const EmisTile *__restrict__ tiles, const float *__restrict__ x32, const float *__restrict__ mu32,
            const float *__restrict__ iv32, const float *__restrict__ k32, int N, int M, int DP, int SC,
            float *__restrict__ logb, int64_t fbase, int64_t ldb, int decode, float *__restrict__ post) {
  extern __shared__ __align__(16) float smem[];
  const int G = N * M;
  const int GC = SC * M;
  float2 *par = reinterpret_cast<float2 *>(smem);
  float *xs = smem + (size_t)GC * DP * 2;
  float *lnt = xs + (size_t)DP * kEmisTF;
  float *lbs = lnt + (size_t)GC * (kEmisTF + 1);

  const EmisTile tile = tiles[blockIdx.x];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int fh = warp & 1, gq = warp >> 1;  // frame half, Gaussian-group phase
  const int fl = fh * 32 + lane;            // my frame inside the tile

  // stage x transposed: xs[d][f]
  for (int idx = tid; idx < kEmisTF * DP; idx += kEmisThreads) {
    int f = idx / DP, d = idx - f * DP;
    xs[d * kEmisTF + f] = (f < tile.nf) ? x32[(tile.f0 + f) * DP + d] : 0.f;
  }
  const int64_t gbase = (int64_t)tile.v * G;
  const int64_t col0 = decode ? (int64_t)tile.v * N : 0;

  for (int s0 = 0; s0 < N; s0 += SC) {
    const int sc = min(SC, N - s0);
    const int gc = sc * M;
    const int64_t g0 = gbase + (int64_t)s0 * M;
    __syncthreads();  // xs ready / previous chunk fully consumed
    for (int idx = tid; idx < gc * DP; idx += kEmisThreads)
      par[idx] = make_float2(mu32[g0 * DP + idx], iv32[g0 * DP + idx]);
    __syncthreads();
    // quadratic forms: 4 Gaussians per pass per thread
    for (int j = gq * 4; j < gc; j += 16) {
      float q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
      const int j1 = min(j + 1, gc - 1), j2 = min(j + 2, gc - 1), j3 = min(j + 3, gc - 1);
      const float2 *p0 = par + (size_t)j * DP, *p1 = par + (size_t)j1 * DP, *p2 = par + (size_t)j2 * DP,
                   *p3 = par + (size_t)j3 * DP;
#pragma unroll 4
      for (int d = 0; d < DP; d++) {
        const float xv = xs[d * kEmisTF + fl];
        float2 a = p0[d], b = p1[d], c = p2[d], e = p3[d];
        float t0 = xv - a.x, t1 = xv - b.x, t2 = xv - c.x, t3 = xv - e.x;
        q0 = fmaf(t0 * a.y, t0, q0);
        q1 = fmaf(t1 * b.y, t1, q1);
        q2 = fmaf(t2 * c.y, t2, q2);
        q3 = fmaf(t3 * e.y, t3, q3);
      }
      lnt[(size_t)j * (kEmisTF + 1) + fl] = fmaf(-0.5f, q0, k32[g0 + j]);
      if (j + 1 < gc) lnt[(size_t)(j + 1) * (kEmisTF + 1) + fl] = fmaf(-0.5f, q1, k32[g0 + j + 1]);
      if (j + 2 < gc) lnt[(size_t)(j + 2) * (kEmisTF + 1) + fl] = fmaf(-0.5f, q2, k32[g0 + j + 2]);
      if (j + 3 < gc) lnt[(size_t)(j + 3) * (kEmisTF + 1) + fl] = fmaf(-0.5f, q3, k32[g0 + j + 3]);
    }
    __syncthreads();
    // log-sum-exp over the mixtures of each state
    for (int idx = tid; idx < sc * kEmisTF; idx += kEmisThreads) {
      int s = idx / kEmisTF, f = idx - s * kEmisTF;
      const float *col = lnt + (size_t)(s * M) * (kEmisTF + 1) + f;
      float mx = kNegInf;
      for (int m = 0; m < M; m++) mx = fmaxf(mx, col[(size_t)m * (kEmisTF + 1)]);
      float lb = kNegInf;
      if (mx > kNegInf) {
        float sum = 0.f;
        for (int m = 0; m < M; m++) sum += __expf(col[(size_t)m * (kEmisTF + 1)] - mx);
        lb = mx + __logf(sum);
      }
      lbs[s * kEmisTF + f] = lb;
    }
    __syncthreads();
    for (int idx = tid; idx < tile.nf * sc; idx += kEmisThreads) {
      int f = idx / sc, s = idx - f * sc;
      logb[(tile.f0 + f - fbase) * ldb + col0 + s0 + s] = lbs[s * kEmisTF + f];
    }
    if (POST) {
      for (int idx = tid; idx < tile.nf * gc; idx += kEmisThreads) {
        int f = idx / gc, g = idx - f * gc;
        float lb = lbs[(g / M) * kEmisTF + f];
        float p = (lb > kNegInf) ? __expf(lnt[(size_t)g * (kEmisTF + 1) + f] - lb) : 0.f;
        post[(tile.f0 + f) * G + (int64_t)s0 * M + g] = p;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// warp helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------
// Mixture accumulators (calc_mix_param, T-FS:1691-1727), CUDA-core version.
// CTA (part p, model v, Gaussian chunk gcx) walks the utterances of model v assigned to part p.
// Thread (d, gg) owns column d of kAccGPT Gaussians g = k*NGG + gg of the chunk:
//   s1 += w x_d (centred x; column D is the constant 1 -> S0),  s2 += w (x_d - mu_old)^2
// with w = gamma_t(state(g)) * post_t(g).  Flushed by double atomics every <= kAccFlush frames.
// ------------------------------------------------------------------------------------------------
constexpr int kAccThreads = 256;
constexpr int kAccGPT = 8;     // Gaussians per thread
constexpr int kAccTF = 32;     // frames staged per step
constexpr int kAccFlush = 4096;

__global__ void __launch_bounds__(kAccThreads)
k_accum_simt(const float *__restrict__ x32, const float *__restrict__ gamma, const float *__restrict__ post,
             const float *__restrict__ mu32, const int64_t *__restrict__ off,
             const int32_t *__restrict__ model_utt_start, const int32_t *__restrict__ model_utts, int N, int M,
             int D, int DP, int nparts, double *__restrict__ stats, int64_t stats_stride, int64_t off_S0,
             int64_t off_S1, int64_t off_S2) {
  extern __shared__ __align__(16) float smem[];
  const int G = N * M;
  const int NGG = kAccThreads / DP;   // Gaussian groups
  const int GCH = NGG * kAccGPT;      // Gaussians per chunk
  float *xs = smem;                   // [kAccTF][DP]
  float *ws = smem + kAccTF * DP;     // [kAccTF][GCH]
  const int part = blockIdx.x, v = blockIdx.y, g0 = blockIdx.z * GCH;
  const int tid = threadIdx.x;
  const int d = tid % DP, gg = tid / DP;
  const bool active = gg < NGG;
  const int gcn = min(GCH, G - g0);

  float s1[kAccGPT], s2[kAccGPT], mu[kAccGPT];
#pragma unroll
  for (int k = 0; k < kAccGPT; k++) {
    s1[k] = 0.f; s2[k] = 0.f;
    int g = k * NGG + gg;
    mu[k] = (active && g < gcn) ? mu32[((int64_t)v * G + g0 + g) * DP + d] : 0.f;
  }
  double *st = stats + (int64_t)v * stats_stride;
  int since_flush = 0;

  auto flush = [&]() {
    if (active) {
#pragma unroll
      for (int k = 0; k < kAccGPT; k++) {
        int g = k * NGG + gg;
        if (g < gcn) {
          if (d < D) {
            atomicAdd(st + off_S1 + (int64_t)(g0 + g) * D + d, (double)s1[k]);
            atomicAdd(st + off_S2 + (int64_t)(g0 + g) * D + d, (double)s2[k]);
          } else if (d == D) {
            atomicAdd(st + off_S0 + g0 + g, (double)s1[k]);
          }
        }
        s1[k] = 0.f; s2[k] = 0.f;
      }
    }
  };

  const int ub = model_utt_start[v], ue = model_utt_start[v + 1];
  for (int ui = ub + part; ui < ue; ui += nparts) {
    const int u = model_utts[ui];
    const int64_t base = off[u];
    const int T = (int)(off[u + 1] - base);
    for (int t0 = 0; t0 < T; t0 += kAccTF) {
      const int nt = min(kAccTF, T - t0);
      __syncthreads();
      for (int idx = tid; idx < nt * DP; idx += kAccThreads) xs[idx] = x32[(base + t0) * DP + idx];
      for (int idx = tid; idx < nt * gcn; idx += kAccThreads) {
        int t = idx / gcn, g = idx - t * gcn;
        float gm = gamma[(base + t0 + t) * N + (g0 + g) / M];
        ws[t * GCH + g] = gm * post[(base + t0 + t) * G + g0 + g];
      }
      __syncthreads();
      if (active) {
        for (int t = 0; t < nt; t++) {
          const float xv = xs[t * DP + d];
          const float *wr = ws + t * GCH + gg;
#pragma unroll
          for (int k = 0; k < kAccGPT; k++) {
            const float w = wr[k * NGG];
            const float dif = xv - mu[k];
            s1[k] = fmaf(w, xv, s1[k]);
            s2[k] = fmaf(w * dif, dif, s2[k]);
          }
        }
      }
      since_flush += nt;
      if (since_flush >= kAccFlush) { flush(); since_flush = 0; }
    }
  }
  flush();
}

// S1 was accumulated on centred features: S1 += ctr * S0  (before any cross-rank reduction).
// mu != nullptr (tensor-core accumulators): the second-order slot holds the raw centred moment
// sum w x^2; turn it into the reference's sum w (x - mu_old)^2 (T-FS:1716-1719), in double:
//   sum w (x - m)^2 = sum w x^2 - 2 m sum w x + m^2 sum w,   m = mu_old - ctr.
__global__ void k_finalize_stats(double *__restrict__ stats, int64_t stats_stride, int V, int G, int D,
                                 int64_t off_S0, int64_t off_S1, int64_t off_S2, const double *__restrict__ ctr,
                                 const double *__restrict__ mu) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)V * G * D;
  if (idx >= total) return;
  int d = (int)(idx % D);
  int64_t vg = idx / D;
  int g = (int)(vg % G);
  int64_t v = vg / G;
  double *st = stats + v * stats_stride;
  const double s0 = st[off_S0 + g], s1 = st[off_S1 + (int64_t)g * D + d];
  if (mu) {
    const double m = mu[vg * D + d] - ctr[d];
    st[off_S2 + (int64_t)g * D + d] = st[off_S2 + (int64_t)g * D + d] - 2.0 * m * s1 + m * m * s0;
  }
  st[off_S1 + (int64_t)g * D + d] = s1 + ctr[d] * s0;
}

// ------------------------------------------------------------------------------------------------
// Forward score with the reference's linear-domain underflow emulated (the drop-in recogniser's
// path): one THREAD per (utterance, model) cell.  The fast scorers are in vit_kernels.cuh.
// ------------------------------------------------------------------------------------------------
constexpr int kScoreThreads = 128;

// forward score (calc_alpha + calc_probability, R-FS:739-836)
template <int NS>
__global__ void __launch_bounds__(kScoreThreads)
k_fwd_score(const float *__restrict__ logb, int64_t fbase, int64_t ldb, const int64_t *__restrict__ off, int u0,
            int V, const double *__restrict__ Aall, double *__restrict__ out, int emulate, int lay8) {
  // lay8: the interleaved layout k_emis_dec writes (dec_logb_index), ldb = number of state columns
  const int v = blockIdx.x * kScoreThreads + threadIdx.x;
  const int u = u0 + blockIdx.y;
  if (v >= V) return;
  const int64_t base = off[u];
  const int T = (int)(off[u + 1] - base);
  double A[NS * NS];
#pragma unroll
  for (int k = 0; k < NS * NS; k++) A[k] = Aall[(int64_t)v * NS * NS + k];
  double al[NS];
#pragma unroll
  for (int i = 0; i < NS; i++) al[i] = 0.0;
  double lp = 0.0;
  for (int t = 0; t < T; t++) {
    const int64_t f = base - fbase + t;
    const float *p = lay8 ? logb + ((f >> 3) * ldb + (int64_t)v * NS) * 8 + (f & 7) : logb + f * ldb + (int64_t)v * NS;
    const int ps = lay8 ? 8 : 1;
    float lbv[NS];
    float mt = kNegInf;
#pragma unroll
    for (int i = 0; i < NS; i++) {
      lbv[i] = p[i * ps];
      if (emulate && (double)lbv[i] < kLogTrueMin) lbv[i] = kNegInf;  // the reference's density is exactly 0
      mt = fmaxf(mt, lbv[i]);
    }
    double an[NS];
    double sum = 0.0;
#pragma unroll
    for (int i = 0; i < NS; i++) {
      double aux;
      if (t == 0) aux = (i == 0) ? 1.0 : 0.0;
      else {
        aux = 0.0;
#pragma unroll
        for (int j = 0; j < NS; j++) aux += al[j] * A[j * NS + i];
      }
      double b = (mt > kNegInf) ? exp((double)lbv[i] - (double)mt) : 0.0;
      an[i] = aux * b;
      if (emulate && an[i] > 0.0 && log(an[i]) + (double)mt < kLogTrueMin) an[i] = 0.0;  // product underflow
      sum += an[i];
    }
    const double cs = 1.0 / sum;
#pragma unroll
    for (int i = 0; i < NS; i++) al[i] = an[i] * cs;
    lp += (double)mt + log(sum);
  }
  out[(int64_t)u * V + v] = lp + log(al[NS - 1]);
}

// ------------------------------------------------------------------------------------------------
// Ranking (sorting_probab + label rule, R-FS:968-995 and 380-388) without sorting: a NaN never
// moves in the reference's bubble sort, every NaN-free run is sorted descending and stably on its
// own; only positions 0 and 1 of the result are consumed.
// ------------------------------------------------------------------------------------------------
__global__ void k_rank(const double *__restrict__ logp, int U, int V, double weight, int32_t *__restrict__ label,
                       int32_t *__restrict__ second) {
  int u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= U) return;
  const double *s = logp + (int64_t)u * V;
  auto val = [&](int k) { return 0.0 + weight * s[k]; };  // probab[k] += coef_model*logP, R-FS:366
  // run containing position 0: [0, e0)
  int first, sec;
  if (isnan(val(0))) {
    first = 0;
    // position 1: NaN stays; else max of run starting at 1
    if (V < 2) sec = 0;
    else if (isnan(val(1))) sec = 1;
    else {
      int best = 1;
      for (int k = 2; k < V && !isnan(val(k)); k++)
        if (val(k) > val(best)) best = k;
      sec = best;
    }
  } else {
    int best = 0, e0 = 1;
    for (; e0 < V && !isnan(val(e0)); e0++)
      if (val(e0) > val(best)) best = e0;
    first = best;
    if (V < 2) sec = 0;
    else if (e0 < 2) sec = 1;  // position 1 is a NaN
    else {
      int b2 = -1;
      for (int k = 0; k < e0; k++) {
        if (k == best) continue;
        if (b2 < 0 || val(k) > val(b2)) b2 = k;
      }
      sec = b2;
    }
  }
  label[u] = first;
  if (second) second[u] = sec;
}


// ------------------------------------------------------------------------------------------------
// M-step on the device (updating_transition_probab T-FS:1862-1889, updating_mix_param T-FS:1911-1955,
// changing_zero_coef T-FS:1338-1359, calc_det T-FS:1976-1991, inv_matrix T-FS:2012-2022) together with
// the per-word stopping rule of the trainer's main() (T-FS:326-358): one CTA per model, everything in
// double, the same operations in the same order as the host version hmmh_mstep().  Keeping it on the
// device removes the statistics download and the model upload from every EM iteration.
//   ctl[v] = sum_logp, ctl[V+v] = n_utt, ctl[2V+v] = 1 if model v was re-estimated, else 0.
// Like the reference, det / inverse are recomputed for EVERY mixture of a re-estimated model, also
// those of states with den_mix == 0 (whose stored inverse is thereby inverted again).
// ------------------------------------------------------------------------------------------------
// Step 1: the stopping rule, one thread per model.  upd[v] = 1 iff model v is re-estimated now.
__global__ void k_mstep_ctl(const double *__restrict__ stats, int64_t ss, int V, double threshold, double *__restrict__ em_old,
                            int *__restrict__ em_active, double *__restrict__ ctl, int *__restrict__ upd) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  pdl_trigger();
  if (v >= V) return;
  const double *st = stats + (int64_t)v * ss;
  const double probab = st[ss - 2], nutt = st[ss - 1];
  ctl[v] = probab;
  ctl[V + v] = nutt;
  int u = 0;
  if (em_active[v]) {
    const double variation = fabs((em_old[v] - probab) / em_old[v]);  // T-FS:326
    if (variation > threshold) { em_old[v] = probab; u = 1; }
    else em_active[v] = 0;
  }
  ctl[2 * V + v] = (double)u;
  upd[v] = u;
}

// Step 2: re-estimation.  grid = (1 + ceil(G / 8), V); block x = 0 does the transitions and the mixture
// weights of model y, block x >= 1 eight Gaussians, one warp each (lanes over the coefficients; the
// determinant is the product in index order, as calc_det forms it).
__global__ void __launch_bounds__(256)
k_mstep_apply(const double *__restrict__ stats, int64_t ss, int N, int M, int D, double floor_, const int *__restrict__ upd,
              double *__restrict__ Aall, double *__restrict__ call, double *__restrict__ muall, double *__restrict__ ivall,
              double *__restrict__ detall) {
  const int v = blockIdx.y, tid = threadIdx.x, G = N * M;
  pdl_wait();
  pdl_trigger();
  if (!upd[v]) return;
  const double *st = stats + (int64_t)v * ss;
  const double *num = st, *den = num + (int64_t)N * N, *denmix = den + N, *S0 = denmix + N;
  const double *S1 = S0 + G, *S2 = S1 + (int64_t)G * D;
  if (blockIdx.x == 0) {
    double *A = Aall + (int64_t)v * N * N, *c = call + (int64_t)v * G;
    for (int idx = tid; idx < N * N; idx += blockDim.x) {
      const int i = idx / N;
      if (den[i] != 0.0) A[idx] = num[idx] / den[i];
    }
    for (int i = tid; i < N; i += blockDim.x) {  // updating_mix_param's weights, then changing_zero_coef
      double *w = c + i * M;
      if (denmix[i] != 0.0)
        for (int k = 0; k < M; k++) w[k] = S0[i * M + k] / denmix[i];
      double s = 0.0;
      for (int k = 0; k < M; k++) {
        if (w[k] < floor_) w[k] = floor_;
        s += w[k];
      }
      for (int k = 0; k < M; k++) w[k] /= s;
    }
    return;
  }
  const int warp = tid >> 5, lane = tid & 31;
  const int k = (blockIdx.x - 1) * 8 + warp;
  if (k >= G) return;
  const int i = k / M;
  double *mu = muall + ((int64_t)v * G + k) * D, *iv = ivall + ((int64_t)v * G + k) * D;
  const bool fresh = denmix[i] != 0.0;
  const double s0 = S0[k];
  double dt = 1.0;
  for (int d0 = 0; d0 < D; d0 += 32) {
    const int d = d0 + lane;
    double var = 1.0;
    if (d < D) {
      if (fresh) {
        mu[d] = S1[(int64_t)k * D + d] / s0;
        var = S2[(int64_t)k * D + d] / s0;
        if (var < floor_) var = floor_;
      } else var = iv[d];  // not re-estimated: the stored inverse is inverted again, as the reference does
      iv[d] = 1.0 / var;
    }
    const int nd = min(32, D - d0);
    for (int j = 0; j < nd; j++) dt *= __shfl_sync(0xffffffffu, var, j);  // calc_det: product in index order
  }
  if (lane == 0) detall[(int64_t)v * G + k] = dt;
}

// Per-dimension extremes of the model set for the tensor-core accuracy guard: ext[d] = max iv_d,
// ext[DP + d] = max |mu_d - ctr_d| as the bit patterns of non-negative doubles (ordered like integers);
// NaN counts as +inf.  ext must be zeroed first.
__global__ void k_model_extremes(const double *__restrict__ mu, const double *__restrict__ iv, const double *__restrict__ ctr,
                                 int64_t VG, int D, int DP, unsigned long long *__restrict__ ext, const unsigned int *__restrict__ xabs,
                                 unsigned int *__restrict__ done, double *__restrict__ kappa_out) {
  const int d = threadIdx.x % DP, grp = threadIdx.x / DP, ngrp = blockDim.x / DP;
  if (d < D && grp < ngrp) {
    double ivm = 0.0, mum = 0.0;
    const double c0 = ctr[d];
    for (int64_t g = (int64_t)blockIdx.x * ngrp + grp; g < VG; g += (int64_t)gridDim.x * ngrp) {
      double a = iv[g * D + d], b = fabs(mu[g * D + d] - c0);
      if (!(a == a)) a = INFINITY;
      if (!(b == b)) b = INFINITY;
      ivm = fmax(ivm, a);
      mum = fmax(mum, b);
    }
    atomicMax(ext + d, (unsigned long long)__double_as_longlong(ivm));
    atomicMax(ext + DP + d, (unsigned long long)__double_as_longlong(mum));
  }
  // the last block to finish turns the extremes into kappa = sum_d 2 max(iv_d) r_d^2, r_d = largest centred |x| or
  // |mu| in dimension d: an upper bound on sum_k |Xaug_k W_k|; the 3xTF32 contraction carries ~1e-7 of it as error
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(done, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  // the finished extremes, one dimension per thread (the L2 copies: other blocks wrote them with atomics)
  __shared__ double part[8];
  double t = 0.0;
  for (int dd = threadIdx.x; dd < D; dd += blockDim.x) {
    const double ivm = __longlong_as_double((long long)__ldcg(ext + dd));
    double r = __longlong_as_double((long long)__ldcg(ext + DP + dd));
    if (xabs) r = fmax(r, (double)__uint_as_float(xabs[dd]));
    const double u = 2.0 * ivm * r * r;
    t += (u == u) ? u : INFINITY;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  if ((threadIdx.x & 31) == 0 && (threadIdx.x >> 5) < 8) part[threadIdx.x >> 5] = t;
  __syncthreads();
  if (threadIdx.x == 0) {
    double kappa = 0.0;
    for (int w = 0; w < min(8, (int)(blockDim.x + 31) / 32); w++) kappa += part[w];
    *kappa_out = kappa;
  }
}

}  // namespace hmmk
