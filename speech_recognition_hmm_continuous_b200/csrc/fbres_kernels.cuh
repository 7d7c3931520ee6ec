// fbres_kernels.cuh -- scaled forward / backward for Baum-Welch training with every utterance RESIDENT in
// shared memory (calc_alpha, calc_beta, calc_transition_probab, calc_den_mix_coef, calc_probability;
// T-FS:1380-1664).  This is the default training recursion; k_fb (fb_kernels.cuh) remains for what does not
// fit here (very long utterances, a transition matrix outside the reference's DELTA = 1 band).
//
// HBM traffic is the minimum the interface allows: the log-emissions are read once (4 N bytes per frame, as
// coalesced 4-byte words) and the state posteriors written once (4 N bytes per frame, coalesced); alpha and beta
// never leave the SM.  Per utterance two arrays of T rows of N 32-bit words live in shared memory, frame-major:
//   F[t][i]      b~_i(t) = exp(logb_i(t) - m_t), m_t = max_i logb_i(t)   -- replaced by alpha~_t(i) as the forward chain passes
//   B[t][N-1-i]  the same b~_i(t), state order reversed                  -- replaced by q_t(i) as the backward chain passes
// Every chain reads and writes only its own array, in place (a step's operands and its result share an address), so
// the two chains of an utterance need no ordering between them; they run at the same time in two adjacent lanes of
// one warp and with ONE instruction stream -- the backward recursion is carried in q_t = b~_t o beta~_t, which obeys
// the forward recursion's form on the reversed state order:
//   forward :  alpha~_t(i)  = b~_t(i) (a_ii alpha~_{t-1}(i) + a_{i-1,i} alpha~_{t-1}(i-1)),   alpha~_0 = b~_0 o e_0
//   backward:  q_{t-1}(i)   = b~_{t-1}(i) (a_ii q_t(i) + a_{i,i+1} q_t(i+1)),                q_{T-1} = b~_{T-1} o e_{N-1}
// (final state only, T-FS:1484-1490; pi = [1,0,..], T-FS:232-234).  Every step rescales by an exact power of two
// (largest exponent field of the step's components, as in k_fb), so
//   log P = sum_t m_t + ln2 sum_t e_t + log alpha~_{T-1}(N-1)      (calc_probability, T-FS:1546-1549)
// and the reference's c_t-scaled quantities follow from per-frame normalisation with phi = alpha^_{T-1}(N-1):
//   xi_t(i,j)  = phi alpha~_t(i) a_ij q_{t+1}(j) / Z_t,   gamma_t(i) = sum_j xi_t(i,j),   Z_t = sum_ij (..)
//   gamma_{T-1} = phi e_{N-1}.
// Vectors are parked as the HIGH WORD of their double (11-bit exponent, 20-bit mantissa, rounded): the full
// double range at 4 bytes per value, read back into a double for free.  The 2^-21 rounding is below the noise of
// the single-precision log-emissions these values are made from (one ulp of a log-density of -80 is 7.6e-6).
//
// One persistent CTA per SM = four TEAMS of four warps; warp w belongs to team w >> 2 and the chain warp of team k is
// its warp with w & 3 == k: every team has a warp on each of the four sub-partitions of the SM (staging and the gamma
// phase use all four schedulers), and the four chain warps sit on four different sub-partitions, each with a
// double-precision pipe to itself.  A team takes
// a batch of utterances (as many as fit its quarter of the shared memory, longest first, from a global queue),
// stages them, runs the chains (two lanes per utterance), then forms gamma and the transition sums with all 128
// threads over frames, and writes gamma out through a small staging buffer.  Per-utterance sums go to a row of
// `ustats`; k_fb_reduce adds the rows of every model in a fixed order (bit-reproducible statistics).
// The batch counter is zeroed once when it is allocated; the last team to leave each launch zeroes it again.
#pragma once
#include "fb_kernels.cuh"

namespace hmmk {

constexpr int kResTeams = 4;
constexpr int kResTeamThreads = 128;
constexpr int kResThreads = kResTeams * kResTeamThreads;
constexpr int kResMaxUtts = 16;              // utterances per batch (two chain lanes each)
constexpr int kResSmemBytes = 227 * 1024;

struct ResBatch {
  int32_t first;  // index into the length-sorted utterance order
  int32_t count;
};

template <int NS>
struct ResTeamShared {
  double msum[kResMaxUtts];    // sum_t m_t
  double phi[kResMaxUtts], lp[kResMaxUtts];
  int64_t base[kResMaxUtts];
  int32_t T[kResMaxUtts], woff[kResMaxUtts], utt[kResMaxUtts], model[kResMaxUtts], pos[kResMaxUtts];
  int32_t next, pad_[3];
  uint32_t dummy[32 * (NS | 1)];  // rows the idle lanes of the chain warp walk in place
};

template <int NS> __host__ __device__ constexpr size_t res_fixed_bytes() { return (sizeof(ResTeamShared<NS>) + 15) / 16 * 16; }
// 32-bit words of F / B storage per team
template <int NS> __host__ __device__ constexpr int res_slot_words() {
  return (int)(((size_t)kResSmemBytes - kResTeams * res_fixed_bytes<NS>()) / 4 / kResTeams) & ~3;
}
inline int res_slot_words_rt(int N) {
  switch (N) {
    case 1: return res_slot_words<1>();
    case 2: return res_slot_words<2>();
    case 3: return res_slot_words<3>();
    case 4: return res_slot_words<4>();
    case 5: return res_slot_words<5>();
    case 6: return res_slot_words<6>();
    case 7: return res_slot_words<7>();
    case 8: return res_slot_words<8>();
    default: return 0;
  }
}
// row stride (words) of the frame-major arrays: odd, so that lanes over frames never share a bank
__host__ __device__ constexpr int res_row_stride(int NS) { return NS | 1; }
// words one utterance of T frames occupies
__host__ __device__ inline int64_t res_utt_words(int NS, int64_t T) { return 2 * (int64_t)res_row_stride(NS) * T; }
__host__ __device__ inline int res_stats_row(int NS) { return 4 * NS + 1; }  // [num a_ii | num a_i,i+1 | den_trans | den_mix | logP]

// One chain step.  The state y is carried UNSCALED by its own step's factor: the power of two r that normalises y is
// folded into the b~ of the step that consumes it, so the exponent arithmetic (integer pipe) runs beside the matrix-vector
// product instead of in front of it:      y' = (A-part of y) o (b~ r),   r = 2^-e,  e = largest exponent field of y.
// Any per-frame power of two drops out of gamma / xi; log P collects the e's (res_chain).
template <int NS>
__device__ __forceinline__ void res_step(const double (&bb)[NS], double (&y)[NS], const double (&cs)[NS], const double (&cn)[NS], int &esum) {
  double u[NS], c[NS];
#pragma unroll
  for (int i = 0; i < NS; i++) {
    double aux = y[i] * cs[i];
    if (i > 0) aux = fma(y[i - 1], cn[i], aux);
    u[i] = aux;
  }
  int e;
  const double r = pow2_scale_max<NS>(y, e);
#pragma unroll
  for (int i = 0; i < NS; i++) c[i] = bb[i] * r;
#pragma unroll
  for (int i = 0; i < NS; i++) y[i] = u[i] * c[i];
  esum += e;
}

// The two chains of every utterance of a batch: lanes 2j (forward) and 2j + 1 (backward) of one warp; the idle lanes
// walk in place on dummy rows, so that all 32 lanes share one control flow (per-lane bounds inside the loop cost a factor
// of two: scripts/ubench/chain_step.cu).  The utterances of a batch are sorted by length, so the common part [1, Tmin)
// is nearly everything; the ragged rest runs with per-lane bounds.  Every row is read (b~) and later written (the chain's
// vector) in place; a step's stores are issued one step late, inside the next step's arithmetic.
template <int NS>
__device__ __forceinline__ void res_chain(int lane, int count, const int32_t *Tarr, const int32_t *woff, const int32_t *model,
                                          const double *__restrict__ Aall, uint32_t *slot, uint32_t *dummy, double *phi, double *lp) {
  constexpr int RS = res_row_stride(NS);
  const int j = lane >> 1, dir = lane & 1;
  const bool act = j < count;
  const int T = act ? Tarr[j] : 0;
  int Tmax = T, Tmin = act ? T : 0x7fffffff;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Tmax = max(Tmax, __shfl_xor_sync(0xffffffffu, Tmax, o));
    Tmin = min(Tmin, __shfl_xor_sync(0xffffffffu, Tmin, o));
  }
  double cs[NS], cn[NS], y[NS];  // self / neighbour coefficients in this lane's state order
  {
    const double *A = Aall + (int64_t)(act ? model[j] : model[0]) * NS * NS;
#pragma unroll
    for (int i = 0; i < NS; i++) {
      const int js = dir ? NS - 1 - i : i;
      cs[i] = A[js * NS + js];
      if (dir) cn[i] = (js + 1 < NS) ? A[js * NS + js + 1] : 0.0;
      else cn[i] = (js > 0) ? A[(js - 1) * NS + js] : 0.0;
    }
  }
  // this lane's array, walked from its first frame: forward F[0..T), backward B[T-1..0]
  int step = act ? (dir ? -RS : RS) : 0;
  asm volatile("mov.b32 %0, %0;" : "+r"(step));  // keep it in a register (recomputing it from %tid costs an S2R per step)
  uint32_t *p = act ? slot + woff[j] + (dir ? RS * T + RS * (T - 1) : 0) : dummy + lane * RS;
  int esum = 0;
  double b0[NS], b1[NS];
  uint32_t w[NS];
  // first step: pi = e_0 (forward, T-FS:232-234) / final state only (backward, T-FS:1484-1490): y = b~ o e_0 in this lane's order
#pragma unroll
  for (int i = 0; i < NS; i++) y[i] = (i == 0) ? d32_unpack(p[0]) : 0.0;
#pragma unroll
  for (int i = 0; i < NS; i++) w[i] = d32_pack(y[i]);
  uint32_t *pw = p;  // the row the pending words w[] belong to
#pragma unroll
  for (int i = 0; i < NS; i++) b0[i] = d32_unpack(p[(T > 1 ? step : 0) + i]);
  int s = 1;
  for (; s + 2 < Tmin; s += 2) {  // steps s and s + 1; b~ of s + 1 and s + 2 are in flight meanwhile
#pragma unroll
    for (int i = 0; i < NS; i++) b1[i] = d32_unpack(p[2 * step + i]);
    res_step<NS>(b0, y, cs, cn, esum);
#pragma unroll
    for (int i = 0; i < NS; i++) pw[i] = w[i];
#pragma unroll
    for (int i = 0; i < NS; i++) w[i] = d32_pack(y[i]);
#pragma unroll
    for (int i = 0; i < NS; i++) b0[i] = d32_unpack(p[3 * step + i]);
    res_step<NS>(b1, y, cs, cn, esum);
#pragma unroll
    for (int i = 0; i < NS; i++) p[step + i] = w[i];
#pragma unroll
    for (int i = 0; i < NS; i++) w[i] = d32_pack(y[i]);
    p += 2 * step;
    pw = p;
  }
#pragma unroll
  for (int i = 0; i < NS; i++) pw[i] = w[i];
  // ragged rest: p is the row of step s - 1, b0 holds the b~ of step s (when s < T)
  for (; s < Tmax; s++) {
    if (s < T) {
      res_step<NS>(b0, y, cs, cn, esum);
#pragma unroll
      for (int i = 0; i < NS; i++) p[step + i] = d32_pack(y[i]);
      if (s + 1 < T) {
#pragma unroll
        for (int i = 0; i < NS; i++) b0[i] = d32_unpack(p[2 * step + i]);
      }
    }
    p += step;
  }
  if (act && dir == 0) {
    double sm = y[0];
#pragma unroll
    for (int i = 1; i < NS; i++) sm += y[i];
    phi[j] = y[NS - 1] / sm;                                          // alpha^_{T-1}(N-1)
    lp[j] = 0.6931471805599453 * (double)esum + log(y[NS - 1]);      // + sum m_t (k_fb_res)
  }
}

// WEIGHTED: utterance u's gamma rows and the transition and occupancy sums of its ustats row are multiplied by w[u]
// (the denominator of MMI training, hmmcu_estep_mmi); its log P is not.
template <int NS, bool WEIGHTED = false>
__global__ void __launch_bounds__(kResThreads, 1)
k_fb_res(const float *__restrict__ logb, const int64_t *__restrict__ off, const int32_t *__restrict__ u2m,
         const double *__restrict__ Aall, const int32_t *__restrict__ order, const int32_t *__restrict__ upos,
         const ResBatch *__restrict__ batches, int nbatches, int *__restrict__ counter, float *__restrict__ gamma,
         double *__restrict__ ustats, double *__restrict__ logp_utt, const double *__restrict__ w = nullptr) {
  extern __shared__ __align__(16) uint8_t res_smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int team = warp >> 2, role = warp & 3, tt = role * 32 + lane;  // tt: thread index within the team
  const bool chain_warp = role == team;
  constexpr size_t FX = res_fixed_bytes<NS>();
  constexpr int SW = res_slot_words<NS>();
  constexpr int K = 4 * NS + 1;
  constexpr int RS = res_row_stride(NS);
  ResTeamShared<NS> &S = *reinterpret_cast<ResTeamShared<NS> *>(res_smem + (size_t)team * FX);
  uint32_t *slot = reinterpret_cast<uint32_t *>(res_smem + kResTeams * FX) + (size_t)team * SW;
  auto team_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "n"(kResTeamThreads) : "memory"); };
  for (int i = tt; i < 32 * RS; i += kResTeamThreads) S.dummy[i] = 0x3fe00000u;  // 0.5
  pdl_wait();  // logb comes from the emission kernel just before
  if (tt == 0) S.next = atomicAdd(counter, 1);
  for (;;) {
    team_sync();
    const int b = S.next;
    if (b >= nbatches) {
      // Every team makes exactly one claim past the end, so the claim nbatches + teams - 1 is the last access to the
      // counter in this launch: that team leaves it at 0 for the next one.
      if (tt == 0 && b == nbatches + (int)gridDim.x * kResTeams - 1) atomicExch(counter, 0);
      pdl_trigger();
      break;
    }
    const ResBatch bd = batches[b];
    if (role == 0) {  // the batch's utterances: one lane each; word offsets by a prefix sum over the lanes
      int T = 0;
      if (lane < bd.count) {
        const int u = order[bd.first + lane];
        const int64_t f0 = off[u];
        T = (int)(off[u + 1] - f0);
        S.utt[lane] = u;
        S.pos[lane] = upos[u];
        S.model[lane] = u2m[u];
        S.base[lane] = f0;
        S.T[lane] = T;
      }
      int w = 2 * RS * T;
#pragma unroll
      for (int o = 1; o < kResMaxUtts; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += v;
      }
      if (lane < bd.count) S.woff[lane] = w - 2 * RS * T;
    }
    team_sync();
    // ---------------- staging, one warp per utterance: raw log-emissions into the rows of F by asynchronous 4-byte
    // copies (coalesced, all in flight at once), then b~ in place into F and reversed into B, and sum_t m_t ----------------
    for (int j = role; j < bd.count; j += 4) {
      const int T = S.T[j], n = T * NS;
      const uint32_t *src = reinterpret_cast<const uint32_t *>(logb) + S.base[j] * NS;
      uint32_t *F = slot + S.woff[j];
      for (int w = lane; w < n; w += 32) {
        const int t = w / NS, i = w - t * NS;
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(F + t * RS + i)), "l"(src + w) : "memory");
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncwarp();
    for (int j = role; j < bd.count; j += 4) {
      const int T = S.T[j];
      uint32_t *F = slot + S.woff[j];
      uint32_t *B = F + RS * T;
      double macc = 0.0;
#pragma unroll 2
      for (int t = lane; t < T; t += 32) {
        float l[NS];
#pragma unroll
        for (int i = 0; i < NS; i++) l[i] = __uint_as_float(F[t * RS + i]);
        float m = l[0];
#pragma unroll
        for (int i = 1; i < NS; i++) m = fmaxf(m, l[i]);
        macc += (double)m;                           // -inf when a frame has no density at all
        const float ms = (m > kNegInf) ? m : 0.f;    // all states at -inf: every b~ is 0 (not NaN)
#pragma unroll
        for (int i = 0; i < NS; i++) {
          const uint32_t w = d32_pack(exp_scaled(l[i] - ms));
          F[t * RS + i] = w;
          B[t * RS + NS - 1 - i] = w;
        }
      }
      macc = warp_sum(macc);
      if (lane == 0) S.msum[j] = macc;
    }
    team_sync();
    // ---------------- the chains; meanwhile the idle warps claim the team's next batch and pull it into L2 ----------------
    if (!chain_warp) {
      if (role == ((team + 1) & 3)) {
        int nb = 0;
        if (lane == 0) { nb = atomicAdd(counter, 1); S.next = nb; }
        nb = __shfl_sync(0xffffffffu, nb, 0);
        if (nb < nbatches) {
          const ResBatch nd = batches[nb];
          for (int j = 0; j < nd.count; j++) {
            const int u = order[nd.first + j];
            const char *q0 = reinterpret_cast<const char *>(logb + off[u] * NS);
            const char *q1 = reinterpret_cast<const char *>(logb + off[u + 1] * NS);
            for (const char *q = q0 + 128 * lane; q < q1; q += 128 * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(q));
          }
        }
      }
    } else {
      res_chain<NS>(lane, bd.count, S.T, S.woff, S.model, Aall, slot, S.dummy, S.phi, S.lp);
    }
    team_sync();
    // ---------------- gamma, transition and den sums: one warp per utterance, lanes over frames; gamma replaces alpha~
    // in its row of F and the rows leave as they lie ([frame][state], coalesced) ----------------
    for (int j = role; j < bd.count; j += 4) {
      const int T = S.T[j];
      uint32_t *F = slot + S.woff[j];          // alpha~_t(i)  at F[t RS + i]
      const uint32_t *B = F + RS * T;          // q_t(i)       at B[t RS + NS-1-i]
      const double *A = Aall + (int64_t)S.model[j] * NS * NS;
      double a0[NS], a1[NS];
#pragma unroll
      for (int i = 0; i < NS; i++) {
        a0[i] = A[i * NS + i];
        a1[i] = (i + 1 < NS) ? A[i * NS + i + 1] : 0.0;
      }
      double phi = S.phi[j];
      if constexpr (WEIGHTED) phi *= w[S.utt[j]];  // (enters sc below)
      double acc_n0[NS], acc_n1[NS], acc_dt[NS], acc_dm[NS];
#pragma unroll
      for (int i = 0; i < NS; i++) { acc_n0[i] = 0.0; acc_n1[i] = 0.0; acc_dt[i] = 0.0; acc_dm[i] = 0.0; }
#pragma unroll 2
      for (int t = lane; t < T; t += 32) {
        double al[NS], n0[NS], n1[NS], gu[NS], Z = 0.0;
#pragma unroll
        for (int i = 0; i < NS; i++) al[i] = d32_unpack(F[t * RS + i]);
        int ex;
        const double ra = pow2_scale_max<NS>(al, ex);  // the chains park their vectors unnormalised: bring them to [1, 2)
#pragma unroll
        for (int i = 0; i < NS; i++) al[i] *= ra;
        const bool inner = t + 1 < T;
        if (inner) {
          double q[NS];
#pragma unroll
          for (int i = 0; i < NS; i++) q[i] = d32_unpack(B[(t + 1) * RS + NS - 1 - i]);
          const double rq = pow2_scale_max<NS>(q, ex);
#pragma unroll
          for (int i = 0; i < NS; i++) q[i] *= rq;
#pragma unroll
          for (int i = 0; i < NS; i++) {
            n0[i] = al[i] * a0[i] * q[i];                                 // band j = i      T-FS:1611
            n1[i] = (i + 1 < NS) ? al[i] * a1[i] * q[i + 1] : 0.0;        // j = i + 1
            gu[i] = n0[i] + n1[i];
          }
        } else {  // last frame: beta^ is non-zero for the final state only (T-FS:1484-1490)
#pragma unroll
          for (int i = 0; i < NS; i++) { n0[i] = 0.0; n1[i] = 0.0; gu[i] = (i == NS - 1) ? al[i] : 0.0; }
        }
#pragma unroll
        for (int i = 0; i < NS; i++) Z += gu[i];
        const double sc = (Z > 0.0) ? phi * __drcp_rn(Z) : 0.0;  // unreachable final state: no occupancy, as the reference
#pragma unroll
        for (int i = 0; i < NS; i++) {
          const double g = gu[i] * sc;                 // alpha^ beta^ / c   T-FS:1617,1658,1709
          F[t * RS + i] = __float_as_uint((float)g);
          acc_dm[i] += g;
          if (inner) {
            acc_dt[i] += g;
            acc_n0[i] += n0[i] * sc;
            acc_n1[i] += n1[i] * sc;
          }
        }
      }
      __syncwarp();
      {
        uint32_t *dst = reinterpret_cast<uint32_t *>(gamma) + S.base[j] * NS;
        const int n = T * NS;
#pragma unroll 4
        for (int w = lane; w < n; w += 32) {
          const int t = w / NS, i = w - t * NS;
          dst[w] = F[t * RS + i];
        }
      }
      double *row = ustats + (int64_t)S.pos[j] * K;
#pragma unroll
      for (int i = 0; i < NS; i++) {
        const double v0 = warp_sum(acc_n0[i]), v1 = warp_sum(acc_n1[i]), v2 = warp_sum(acc_dt[i]), v3 = warp_sum(acc_dm[i]);
        if (lane == 0) {
          row[i] = v0;
          row[NS + i] = v1;
          row[2 * NS + i] = v2;
          row[3 * NS + i] = v3;
        }
      }
      if (lane == 0) {
        const double lp = S.lp[j] + S.msum[j];  // calc_probability T-FS:1546-1549
        row[4 * NS] = lp;
        if (logp_utt) logp_utt[S.utt[j]] = lp;
      }
    }
  }
}

// Per-model sums of the per-utterance rows, in a fixed order: thread (sub, k) adds rows sub, sub + nsub, .. of the
// model's block of rows (rows are stored in the model-grouped utterance order), then thread k adds the partial
// sums of the subsets in order.  Writes the head [num_trans | den_trans | den_mix] and the tail [sum_logP, n_utt]
// of the model's statistics (the statistics buffer was cleared before).
__global__ void __launch_bounds__(1024)
k_fb_reduce(const double *__restrict__ ustats, int NS, const int32_t *__restrict__ model_row_start, int V,
            double *__restrict__ stats, int64_t stats_stride, int64_t off_sumlogp) {
  __shared__ double part[1024];
  const int K = 4 * NS + 1;
  const int v = blockIdx.x, tid = threadIdx.x;
  if (v >= V) return;
  const int r0 = model_row_start[v], r1 = model_row_start[v + 1];
  const int nsub = (int)blockDim.x / K, sub = tid / K, k = tid - sub * K;
  double acc = 0.0;
  if (sub < nsub) {
#pragma unroll 4
    for (int r = r0 + sub; r < r1; r += nsub) acc += ustats[(int64_t)r * K + k];
  }
  part[tid] = acc;
  __syncthreads();
  if (tid < K) {
    double t = 0.0;
    for (int s = 0; s < nsub; s++) t += part[s * K + tid];
    double *st = stats + (int64_t)v * stats_stride;
    const int q = tid / NS, i = tid - q * NS;
    if (tid == 4 * NS) {
      st[off_sumlogp] = t;
      st[off_sumlogp + 1] = (double)(r1 - r0);
    } else if (q == 0) st[i * NS + i] = t;
    else if (q == 1) { if (i + 1 < NS) st[i * NS + i + 1] = t; }
    else if (q == 2) st[NS * NS + i] = t;
    else st[NS * NS + NS + i] = t;
  }
}

}  // namespace hmmk
