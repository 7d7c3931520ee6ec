// vit_kernels.cuh -- decode recursions.
//
// (1) Viterbi with back-pointers in double precision (SURVEY row V1; the reference has no Viterbi, so
//     this follows its conventions: pi = [1,0,..], full A, termination in the final state, strict '>'
//     so that the lowest predecessor wins a tie).  State sequences must agree bit for bit with a
//     double-precision CPU restatement, so the emissions are recomputed here from the double masters
//     rather than taken from the single-precision tensor-core path.  Two kernels, split the way the
//     work parallelises:
//       k_logb64   log b_i(t) in double for every frame of every utterance against the utterance's
//                  model: one thread per frame with the frame in registers, the model's (mu, inverse
//                  variance) of one state at a time in shared memory (read as 16-byte broadcasts),
//                  online log-sum-exp over the mixtures.  Throughput bound (FP64 pipe).
//       k_viterbi  the delta recursion is a dependent chain: one THREAD per utterance with delta in
//                  registers, operands staged into shared memory one window at a time by the whole CTA
//                  (as in k_fb), back-pointers packed one byte per state into 64 bits per frame; then
//                  one warp per utterance walks them back, 32 frames per coalesced load.
// (2) The recogniser's cell scorers (calc_alpha + calc_probability, R-FS:739-836, for every
//     (utterance, model) cell; and the Viterbi score of every cell): one thread per cell, cells
//     flattened so that warps stay full for any vocabulary size, single-precision log-emissions
//     prefetched four frames ahead, the chain itself in double with the exact power-of-two scaling of
//     k_fb (no division, no logarithm inside the loop).
#pragma once
#include "fb_kernels.cuh"

namespace hmmk {

// ------------------------------------------------------------------------------------------------
// k_logb64
// ------------------------------------------------------------------------------------------------
constexpr int kLbGroup = 4;    // mixtures evaluated together
constexpr int kLbFrames = 64;  // frames (= threads) per CTA; same tiling as EmisTile (<= 64 frames of one utterance)

// smem: par[M][D] double2 (mu, iv) | lc[M] (log c, or -inf for a dead mixture) | hl[M] (0.5 log|det|)
__host__ __device__ inline size_t logb64_smem_bytes(int M, int D) { return sizeof(double) * ((size_t)2 * M * D + 2 * M) + 16; }

template <int DREG>  // DREG == D: frame held in registers, loops fully unrolled; DREG == 0: any D, frame re-read from global (L1)
__global__ void __launch_bounds__(kLbFrames)
k_logb64(const EmisTile *__restrict__ tiles, const double *__restrict__ x64, const double *__restrict__ call,
         const double *__restrict__ muall, const double *__restrict__ ivall, const double *__restrict__ detall, int N, int M,
         int D, double *__restrict__ logb64) {
  extern __shared__ __align__(16) double lsm[];
  double2 *par = reinterpret_cast<double2 *>(lsm);  // [M][D]
  double *slc = lsm + (size_t)2 * M * D, *shl = slc + M;
  const EmisTile tile = tiles[blockIdx.x];
  const int tid = threadIdx.x;
  const bool live = tid < tile.nf;
  const int64_t f = tile.f0 + (live ? tid : 0);
  const double *xr = x64 + f * D;
  const int G = N * M;
  const double lognorm = 0.5 * (double)D * 1.8378770664093453;
  double xreg[DREG > 0 ? DREG : 1];
  if (DREG > 0) {
#pragma unroll
    for (int d = 0; d < DREG; d++) xreg[d] = xr[d];
  }
  for (int i = 0; i < N; i++) {
    __syncthreads();
    const int64_t g0 = (int64_t)tile.v * G + (int64_t)i * M;
    for (int k = tid; k < M * D; k += kLbFrames) par[k] = make_double2(muall[g0 * D + k], ivall[g0 * D + k]);
    for (int m = tid; m < M; m += kLbFrames) {
      const double dt = detall[g0 + m], cc = call[g0 + m];
      // log(c) - 0.5 q - lognorm - 0.5 log|det| is summed below in this order (as the scalar restatement does)
      const bool ok = dt != 0.0 && cc > 0.0;
      slc[m] = ok ? log(cc) : -INFINITY;
      shl[m] = ok ? 0.5 * log(fabs(dt)) : 0.0;
    }
    __syncthreads();
    double mx = -INFINITY, acc = 0.0;
    // kLbGroup mixtures per pass: independent accumulation chains and independent exponentials keep the FP64 pipe
    // busy (one mixture at a time is a single dependent chain of ~40-instruction exp() calls)
    for (int m0 = 0; m0 < M; m0 += kLbGroup) {
      double q[kLbGroup];
      const double2 *pm[kLbGroup];
#pragma unroll
      for (int h = 0; h < kLbGroup; h++) {
        q[h] = 0.0;
        pm[h] = par + (size_t)min(m0 + h, M - 1) * D;
      }
      if (DREG > 0) {
#pragma unroll
        for (int d = 0; d < DREG; d++) {
#pragma unroll
          for (int h = 0; h < kLbGroup; h++) {
            const double2 p = pm[h][d];
            const double df = xreg[d] - p.x;
            q[h] += df * p.y * df;
          }
        }
      } else {
        for (int d = 0; d < D; d++) {
          const double xv = xr[d];
#pragma unroll
          for (int h = 0; h < kLbGroup; h++) {
            const double2 p = pm[h][d];
            const double df = xv - p.x;
            q[h] += df * p.y * df;
          }
        }
      }
      double ln[kLbGroup], gm = -INFINITY;
#pragma unroll
      for (int h = 0; h < kLbGroup; h++) {
        const bool ok = m0 + h < M && slc[min(m0 + h, M - 1)] > -INFINITY;
        ln[h] = ok ? slc[m0 + h] - 0.5 * q[h] - lognorm - shl[m0 + h] : -INFINITY;
        gm = fmax(gm, ln[h]);
      }
      if (gm > -INFINITY) {
        if (gm > mx) { acc *= exp(mx - gm); mx = gm; }  // exp(-inf) = 0 on the first group
        double sg = 0.0;
#pragma unroll
        for (int h = 0; h < kLbGroup; h++) sg += (ln[h] > -INFINITY) ? exp(ln[h] - mx) : 0.0;
        acc += sg;
      }
    }
    if (live) logb64[f * N + i] = (mx > -INFINITY) ? mx + log(acc) : -INFINITY;
  }
}

// ------------------------------------------------------------------------------------------------
// k_viterbi
// ------------------------------------------------------------------------------------------------
constexpr int kVitUtts = 8;
constexpr int kVitThreads = 256;
constexpr int kVitWin = 128;

__host__ __device__ inline size_t vit_smem_bytes(int NS) { return (size_t)kVitUtts * (kVitWin * NS + 2) * sizeof(double); }

template <int NS, bool BANDED>
__global__ void __launch_bounds__(kVitThreads)
k_viterbi(const double *__restrict__ logb64, const int64_t *__restrict__ off, const int32_t *__restrict__ u2m,
          const double *__restrict__ Aall, int U, unsigned long long *__restrict__ psi_ws, double *__restrict__ score,
          int32_t *__restrict__ path) {
  extern __shared__ __align__(16) uint8_t vsm[];
  constexpr int US = kVitWin * NS + 2;  // padded per-utterance stride (bank spread for the 8 chain lanes)
  double *lb = reinterpret_cast<double *>(vsm);  // [kVitUtts][US]
  __shared__ double sLA[kVitUtts][NS * NS];
  __shared__ int64_t sbase[kVitUtts];
  __shared__ int sT[kVitUtts];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int u0 = blockIdx.x * kVitUtts;
  for (int idx = tid; idx < kVitUtts * NS * NS; idx += kVitThreads) {
    const int uu = idx / (NS * NS), k = idx - uu * NS * NS;
    const int u = u0 + uu;
    sLA[uu][k] = (u < U) ? log(Aall[(int64_t)u2m[u] * NS * NS + k]) : 0.0;
  }
  if (tid < kVitUtts) {
    const int u = u0 + tid;
    sbase[tid] = (u < U) ? off[u] : 0;
    sT[tid] = (u < U) ? (int)(off[u + 1] - off[u]) : 0;
  }
  __syncthreads();
  int Tmax = 0;
#pragma unroll
  for (int uu = 0; uu < kVitUtts; uu++) Tmax = max(Tmax, sT[uu]);

  // ---------------- phase 1: delta recursion, one thread per utterance ----------------
  const bool chain = warp == 0 && lane < kVitUtts && sT[lane & (kVitUtts - 1)] > 0;
  const int myT = chain ? sT[lane] : 0;
  const int64_t mybase = chain ? sbase[lane] : 0;
  double la[NS * NS], dl[NS];
#pragma unroll
  for (int k = 0; k < NS * NS; k++) la[k] = chain ? sLA[lane][k] : 0.0;
#pragma unroll
  for (int i = 0; i < NS; i++) dl[i] = 0.0;
  for (int w0 = 0; w0 < Tmax; w0 += kVitWin) {
    __syncthreads();
    for (int it = tid; it < kVitUtts * kVitWin * NS; it += kVitThreads) {
      const int uu = it / (kVitWin * NS), rem = it - uu * (kVitWin * NS);
      const int k = rem / NS;
      if (w0 + k < sT[uu]) lb[(size_t)uu * US + rem] = logb64[(sbase[uu] + w0) * NS + rem];
    }
    __syncthreads();
    if (chain) {
      const double *bw = lb + (size_t)lane * US;
      const int kend = min(kVitWin, myT - w0);
      for (int k = 0; k < kend; k++) {
        double b[NS], dn[NS];
        unsigned long long ps = 0ull;
#pragma unroll
        for (int i = 0; i < NS; i++) b[i] = bw[k * NS + i];
        if (w0 + k == 0) {
#pragma unroll
          for (int i = 0; i < NS; i++) dn[i] = (i == 0 ? 0.0 : -INFINITY) + b[i];
        } else {
#pragma unroll
          for (int j = 0; j < NS; j++) {
            // Banded A (log a = -inf outside i in {j-1, j}): an out-of-band candidate is -inf (or NaN) and can
            // never win the strict '>' -- except that the scan STARTS from i = 0, whose candidate stands when
            // every other one is -inf as well.  So: start from i = 0 exactly as the full scan does, then only
            // the in-band predecessors need to be compared.
            double best = dl[0] + la[j];
            int arg = 0;
#pragma unroll
            for (int i = 1; i < NS; i++) {
              if (!BANDED || i == j || i + 1 == j) {
                const double cnd = dl[i] + la[i * NS + j];
                if (cnd > best) { best = cnd; arg = i; }  // strict: lowest index wins a tie
              }
            }
            dn[j] = best + b[j];
            ps |= (unsigned long long)arg << (8 * j);
          }
        }
#pragma unroll
        for (int i = 0; i < NS; i++) dl[i] = dn[i];
        psi_ws[mybase + w0 + k] = ps;
      }
    }
  }
  if (chain) score[u0 + lane] = dl[NS - 1];
  if (!path) return;
  __syncthreads();  // the chain thread's psi_ws stores are visible to the CTA's other warps after the barrier
  // ---------------- phase 2: back-trace from the final state, one warp per utterance ----------------
  for (int uu = warp; uu < kVitUtts; uu += kVitThreads / 32) {
    const int T = sT[uu];
    if (T == 0) continue;
    const int64_t base = sbase[uu];
    int sidx = NS - 1;
    const int clast = ((T - 1) / 32) * 32;
    for (int c0 = clast; c0 >= 0; c0 -= 32) {
      const int t = c0 + lane;
      const unsigned long long my_psi = (t < T) ? psi_ws[base + t] : 0ull;
      int my_state = 0;
      const int ns = min(32, T - c0);
      for (int s = ns - 1; s >= 0; s--) {
        if (lane == s) my_state = sidx;
        const unsigned long long ps = __shfl_sync(0xffffffffu, my_psi, s);
        sidx = (int)((ps >> (8 * sidx)) & 0xffull);
      }
      if (t < T) path[base + t] = my_state;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Cell scorers: thread <-> cell (utterance u0 + cell / V, model cell % V) of one utterance batch.
//   logb[(frame - fbase) * ldb + v * NS + i]   single-precision log b_i(t) of model v
// ------------------------------------------------------------------------------------------------
constexpr int kCellThreads = 128;
constexpr int kCellPF = 4;  // frames prefetched ahead of the chain

template <int NS>
__device__ __forceinline__ void cell_load(const float *__restrict__ p, float (&l)[NS]) {
#pragma unroll
  for (int i = 0; i < NS; i++) l[i] = __ldg(p + i);
}

// forward score: log P(O, q_T = N-1 | model)   (calc_alpha + calc_probability, R-FS:739-836), with the chain in SINGLE
// precision, in the LOG domain.  A double-precision linear chain issues ~140 instructions per (cell, frame) -- five
// software exponentials assembled into doubles, a scaling pass -- and was bound by instruction issue at half the HBM
// rate.  A single-precision chain in the linear domain is not an option: against a mismatched model a state's mass falls by
// e^-100 per frame relative to its neighbour's, and a state that is 2^-126 below the frame's maximum today can carry the
// best path tomorrow (measured: 2.5 % error in such a cell), where the reference's doubles still hold it.  So every state
// keeps its own magnitude: with lz_i = log2 of the scaled alpha (max_i lz_i = 0 after every frame),
//   lz'_i = log2(e) l_i + log2( sum_j 2^(lz_j + log2 a_ji) ),     m = max_i lz'_i,     lz_i <- lz'_i - m,
// and log P = ln2 (sum m_t + lz_{T-1}(N-1)), sum m_t in double.  The banded topology takes one ex2 and one lg2 per state
// (log-sum-exp of two terms), a full A takes N ex2 and one lg2.  "No mass" is the finite -1e30 instead of -inf, so that no
// difference of two infinities can arise.  Per (cell, frame), N = 5 banded: 9 transcendental-unit operations, ~60
// instructions, 4 N bytes of log-emissions.
// Error: a rounding of ~2^-17 (values of magnitude ~100) per step, the same size as that of the single-precision
// log-emissions it reads.
constexpr float kLzNone = -1e30f;
__device__ __forceinline__ float ex2_ftz(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2_ftz(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Walks the frames [brel, brel + T) of a cell through the interleaved layout k_emis_dec writes (dec_logb_index: blocks of 8
// frames, state-major inside a block): a (block, model) is N consecutive 32-byte sectors, read with 2 N 16-byte loads one
// block ahead of the chain; adjacent threads (models) read adjacent 32 N bytes.  first(l) is called for t = 0, step(l) for
// 0 < t < T, l = the N log-emissions of the frame.
template <int NS, class First, class Step>
__device__ __forceinline__ void cell_walk8(const float *__restrict__ logb8, int64_t S, int64_t brel, int T, int64_t col0, First first, Step step) {
  const int64_t fb0 = brel >> 3, fb1 = (brel + T - 1) >> 3;
  const float4 *p = reinterpret_cast<const float4 *>(logb8 + (fb0 * S + col0) * 8);
  const int64_t stride4 = S * 2;  // 16-byte words per block of 8 frames
  float4 nx[NS][2];
#pragma unroll
  for (int i = 0; i < NS; i++) { nx[i][0] = __ldg(p + 2 * i); nx[i][1] = __ldg(p + 2 * i + 1); }
  int tb = (int)(fb0 * 8 - brel);  // t of the block's first frame (<= 0 in the first block)
  for (int64_t fb = fb0; fb <= fb1; fb++, tb += 8) {
    float cur[8][NS];
#pragma unroll
    for (int i = 0; i < NS; i++) {
      cur[0][i] = nx[i][0].x; cur[1][i] = nx[i][0].y; cur[2][i] = nx[i][0].z; cur[3][i] = nx[i][0].w;
      cur[4][i] = nx[i][1].x; cur[5][i] = nx[i][1].y; cur[6][i] = nx[i][1].z; cur[7][i] = nx[i][1].w;
    }
    if (fb < fb1) {
      p += stride4;
#pragma unroll
      for (int i = 0; i < NS; i++) { nx[i][0] = __ldg(p + 2 * i); nx[i][1] = __ldg(p + 2 * i + 1); }
    }
    if (tb >= 1 && tb + 8 <= T) {  // a block in the interior of the utterance
#pragma unroll
      for (int k = 0; k < 8; k++) step(cur[k]);
    } else {
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int t = tb + k;
        if (t == 0) first(cur[k]);
        else if (t > 0 && t < T) step(cur[k]);
      }
    }
  }
}

template <int NS, bool BANDED, bool LAY8>
__global__ void __launch_bounds__(kCellThreads)
k_fwd_cells32(const float *__restrict__ logb, int64_t fbase, int64_t ldb, const int64_t *__restrict__ off, int u0, int nu,
              int V, const double *__restrict__ Aall, double *__restrict__ out) {
  const int64_t cell = (int64_t)blockIdx.x * kCellThreads + threadIdx.x;
  if (cell >= (int64_t)nu * V) return;
  const int u = u0 + (int)(cell / V), v = (int)(cell % V);
  const int64_t base = off[u];
  const int T = (int)(off[u + 1] - base);
  if (T <= 0) { out[(int64_t)u * V + v] = -INFINITY; return; }
  float la[NS * NS];  // log2 a_ij, "none" for a_ij = 0
#pragma unroll
  for (int k = 0; k < NS * NS; k++) {
    if (!BANDED || k % (NS + 1) == 0 || (k % NS > 0 && k % (NS + 1) == 1)) la[k] = fmaxf(lg2_ftz((float)Aall[(int64_t)v * NS * NS + k]), kLzNone);
    else la[k] = kLzNone;
  }
  float lz[NS];
  double msum = 0.0;  // sum of m_t (base-2 logarithms)
  constexpr float kL2E = 1.4426950408889634f;
  auto first = [&](const float (&l)[NS]) {  // pi = [1,0,..,0]
    const float m = l[0] * kL2E;            // -inf (density 0 in the entry state): the score is -inf, as log(0) in the reference
    msum = (double)m;
    lz[0] = 0.f;
#pragma unroll
    for (int i = 1; i < NS; i++) lz[i] = kLzNone;
  };
  auto step = [&](const float (&l)[NS]) {
    float nz[NS];
#pragma unroll
    for (int i = 0; i < NS; i++) {
      float lsum;  // log2 sum_j 2^(lz_j + la_ji)
      if (BANDED) {
        const float x = lz[i] + la[i * NS + i];
        if (i > 0) {
          const float y = lz[i - 1] + la[(i - 1) * NS + i];
          lsum = fmaxf(x, y) + lg2_ftz(1.f + ex2_ftz(-fabsf(x - y)));
        } else {
          lsum = x;
        }
      } else {
        float t[NS], mx;
#pragma unroll
        for (int j = 0; j < NS; j++) t[j] = lz[j] + la[j * NS + i];
        mx = t[0];
#pragma unroll
        for (int j = 1; j < NS; j++) mx = fmaxf(mx, t[j]);
        float sm = 0.f;
#pragma unroll
        for (int j = 0; j < NS; j++) sm += ex2_ftz(t[j] - mx);
        lsum = mx + lg2_ftz(sm);
      }
      nz[i] = fmaf(l[i], kL2E, lsum);
    }
    float m = nz[0];
#pragma unroll
    for (int i = 1; i < NS; i++) m = fmaxf(m, nz[i]);
#pragma unroll
    for (int i = 0; i < NS; i++) lz[i] = fmaxf(nz[i] - m, kLzNone);  // also turns -inf (density 0) and NaN (-inf - -inf) into "none"
    msum += (double)m;
  };
  if (LAY8) {
    cell_walk8<NS>(logb, ldb, base - fbase, T, (int64_t)v * NS, first, step);
    const double tot8 = msum + (double)lz[NS - 1];
    out[(int64_t)u * V + v] = (tot8 > -1e29) ? 0.6931471805599453 * tot8 : -INFINITY;
    return;
  }
  // log-emissions kCellPF frames ahead of the chain; the bulk of the frames runs without index clamps
  const float *p = logb + (base - fbase) * ldb + (int64_t)v * NS;
  float nxt[kCellPF][NS];
#pragma unroll
  for (int k = 0; k < kCellPF; k++) cell_load<NS>(p + (int64_t)min(k, T - 1) * ldb, nxt[k]);
  int t0 = 0;
  const float *pn = p + (int64_t)kCellPF * ldb;  // frame t0 + kCellPF
  for (; t0 + 2 * kCellPF <= T; t0 += kCellPF, pn += (int64_t)kCellPF * ldb) {
    float cur[kCellPF][NS];
#pragma unroll
    for (int k = 0; k < kCellPF; k++) {
#pragma unroll
      for (int i = 0; i < NS; i++) cur[k][i] = nxt[k][i];
    }
#pragma unroll
    for (int k = 0; k < kCellPF; k++) cell_load<NS>(pn + (int64_t)k * ldb, nxt[k]);
    if (t0 == 0) first(cur[0]); else step(cur[0]);
#pragma unroll
    for (int k = 1; k < kCellPF; k++) step(cur[k]);
  }
  for (; t0 < T; t0 += kCellPF) {
    float cur[kCellPF][NS];
#pragma unroll
    for (int k = 0; k < kCellPF; k++) {
#pragma unroll
      for (int i = 0; i < NS; i++) cur[k][i] = nxt[k][i];
    }
#pragma unroll
    for (int k = 0; k < kCellPF; k++) cell_load<NS>(p + (int64_t)min(t0 + kCellPF + k, T - 1) * ldb, nxt[k]);
#pragma unroll
    for (int k = 0; k < kCellPF; k++) {
      if (t0 + k < T) {
        if (t0 + k == 0) first(cur[k]); else step(cur[k]);
      }
    }
  }
  // a frame in which no state had mass left m = "none" (or -inf) in the sum
  const double tot = msum + (double)lz[NS - 1];
  out[(int64_t)u * V + v] = (tot > -1e29) ? 0.6931471805599453 * tot : -INFINITY;
}

// Viterbi score of every cell (V1; no reference code): delta in double, log domain.
template <int NS, bool BANDED>
__global__ void __launch_bounds__(kCellThreads)
k_vit_cells(const float *__restrict__ logb, int64_t fbase, int64_t ldb, const int64_t *__restrict__ off, int u0, int nu,
            int V, const double *__restrict__ Aall, double *__restrict__ out) {
  const int64_t cell = (int64_t)blockIdx.x * kCellThreads + threadIdx.x;
  if (cell >= (int64_t)nu * V) return;
  const int u = u0 + (int)(cell / V), v = (int)(cell % V);
  const int64_t base = off[u];
  const int T = (int)(off[u + 1] - base);
  double la[NS * NS];
#pragma unroll
  for (int k = 0; k < NS * NS; k++) la[k] = log(Aall[(int64_t)v * NS * NS + k]);
  double dl[NS];
#pragma unroll
  for (int i = 0; i < NS; i++) dl[i] = 0.0;
  const float *p = logb + (base - fbase) * ldb + (int64_t)v * NS;
  float nxt[kCellPF][NS];
#pragma unroll
  for (int k = 0; k < kCellPF; k++) cell_load<NS>(p + (int64_t)min(k, T - 1) * ldb, nxt[k]);
  for (int t0 = 0; t0 < T; t0 += kCellPF) {
    float cur[kCellPF][NS];
#pragma unroll
    for (int k = 0; k < kCellPF; k++) {
#pragma unroll
      for (int i = 0; i < NS; i++) cur[k][i] = nxt[k][i];
    }
#pragma unroll
    for (int k = 0; k < kCellPF; k++) cell_load<NS>(p + (int64_t)min(t0 + kCellPF + k, T - 1) * ldb, nxt[k]);
#pragma unroll
    for (int k = 0; k < kCellPF; k++) {
      if (t0 + k < T) {
        double dn[NS];
        if (t0 + k == 0) {
#pragma unroll
          for (int i = 0; i < NS; i++) dn[i] = (i == 0 ? 0.0 : -INFINITY) + (double)cur[k][i];
        } else {
#pragma unroll
          for (int j = 0; j < NS; j++) {
            double best = dl[0] + la[j];
#pragma unroll
            for (int i = 1; i < NS; i++) {
              if (!BANDED || i == j || i + 1 == j) {
                const double c = dl[i] + la[i * NS + j];
                if (c > best) best = c;
              }
            }
            dn[j] = best + (double)cur[k][j];
          }
        }
#pragma unroll
        for (int j = 0; j < NS; j++) dl[j] = dn[j];
      }
    }
  }
  out[(int64_t)u * V + v] = dl[NS - 1];
}

// k_vit_cells over the interleaved layout of k_emis_dec (cell_walk8)
template <int NS, bool BANDED>
__global__ void __launch_bounds__(kCellThreads)
k_vit_cells8(const float *__restrict__ logb8, int64_t fbase, int64_t S, const int64_t *__restrict__ off, int u0, int nu,
             int V, const double *__restrict__ Aall, double *__restrict__ out) {
  const int64_t cell = (int64_t)blockIdx.x * kCellThreads + threadIdx.x;
  if (cell >= (int64_t)nu * V) return;
  const int u = u0 + (int)(cell / V), v = (int)(cell % V);
  const int64_t base = off[u];
  const int T = (int)(off[u + 1] - base);
  if (T <= 0) { out[(int64_t)u * V + v] = 0.0; return; }  // as k_vit_cells: delta starts from 0 and no frame is applied
  double la[NS * NS];
#pragma unroll
  for (int k = 0; k < NS * NS; k++) la[k] = log(Aall[(int64_t)v * NS * NS + k]);
  double dl[NS];
#pragma unroll
  for (int i = 0; i < NS; i++) dl[i] = 0.0;
  auto first = [&](const float (&l)[NS]) {
#pragma unroll
    for (int i = 0; i < NS; i++) dl[i] = (i == 0 ? 0.0 : -INFINITY) + (double)l[i];
  };
  auto step = [&](const float (&l)[NS]) {
    double dn[NS];
#pragma unroll
    for (int j = 0; j < NS; j++) {
      double best = dl[0] + la[j];
#pragma unroll
      for (int i = 1; i < NS; i++) {
        if (!BANDED || i == j || i + 1 == j) {
          const double c = dl[i] + la[i * NS + j];
          if (c > best) best = c;
        }
      }
      dn[j] = best + (double)l[j];
    }
#pragma unroll
    for (int j = 0; j < NS; j++) dl[j] = dn[j];
  };
  cell_walk8<NS>(logb8, S, base - fbase, T, (int64_t)v * NS, first, step);
  out[(int64_t)u * V + v] = dl[NS - 1];
}

}  // namespace hmmk
