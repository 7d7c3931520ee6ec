// vtrain_kernels.cuh -- the alignment step of Viterbi (segmental k-means) training: the E-step's forward-backward
// replaced by the best state sequence of every utterance, with the outputs of k_fb_res / k_fb, so that the mixture
// accumulators, k_fb_reduce, the all-reduce and the M-step run unchanged:
//   gamma[F][N]   1 in the aligned state of each frame, 0 elsewhere (the accumulators then weight the frame's
//                 in-state mixture posteriors by it)
//   counts        num_trans[i][j] = #{t < T-1 : (s_t, s_t+1) = (i, j)}, den_trans[i] = #{t < T-1 : s_t = i},
//                 den_mix[i] = #{t < T : s_t = i}, and the Viterbi score in place of log P
//   logp_utt[U]   the Viterbi score (0 for a masked utterance)
//   path[F]       the alignment (-1 on the frames of a masked utterance)
// The delta recursion follows k_viterbi (pi = [1,0,..], log of the full A or its banded shortcut, strict '>' so that
// the lowest predecessor wins a tie, termination in state N-1) but reads the single-precision training log-emissions
// the E-step's emission kernel has just written, not a double-precision pass of its own.  An utterance with no path to
// the final state (score -inf, e.g. T < N with a banded A) gets neither occupancy nor counts; its score still enters
// sum_logp and n_utt, as log P = -inf does in the Baum-Welch E-step.
// Shape: one chain thread per utterance (delta in registers, log-emission windows staged into shared memory by the
// whole CTA, back-pointers packed one byte per state into 64 bits per frame), then one warp per utterance walks the
// back-pointers 32 frames at a time: lane t holds s_t, s_t+1 comes from lane t+1 by a shuffle, and every count is a
// ballot, so the sums need no atomics.  The counts leave either as the utterance's row of the per-utterance statistics
// (summed per model in a fixed order by k_fb_reduce; banded A) or, as k_fb does, by double atomics into the
// per-model statistics (integer-valued, so their order does not matter; sum_logp is the one non-integer sum).
#pragma once
#include "fb_kernels.cuh"

namespace hmmk {

constexpr int kVtUtts = 8;      // utterances per CTA: one chain lane each in warp 0, then one warp each
constexpr int kVtThreads = 256;
constexpr int kVtWin = 128;     // frames per staged window

// [kVtUtts][kVtWin * NS + 1] floats: an odd per-utterance stride, so the 8 chain lanes read 8 different banks
__host__ __device__ inline size_t vtrain_smem_bytes(int NS) { return (size_t)kVtUtts * (kVtWin * NS + 1) * sizeof(float); }

// ustats: rows [num a_ii | num a_i,i+1 | den_trans | den_mix | score] at row upos[u] (BANDED only), or NULL: atomics into
// stats[model][stats_stride] (num_trans, den_trans, den_mix at the head, sum_logp and n_utt at off_sumlogp).
template <int NS, bool BANDED>
__global__ void __launch_bounds__(kVtThreads)
k_vtrain(const float *__restrict__ logb, const int64_t *__restrict__ off, const int32_t *__restrict__ u2m,
         const double *__restrict__ Aall, int U, unsigned long long *__restrict__ psi_ws, int32_t *__restrict__ path,
         float *__restrict__ gamma, const int32_t *__restrict__ upos, double *__restrict__ ustats, double *__restrict__ stats,
         int64_t stats_stride, int64_t off_sumlogp, double *__restrict__ logp_utt) {
  extern __shared__ __align__(16) uint8_t vtsm[];
  constexpr int US = kVtWin * NS + 1;
  float *lb = reinterpret_cast<float *>(vtsm);  // [kVtUtts][US]
  __shared__ double sLA[kVtUtts][NS * NS];
  __shared__ double sScore[kVtUtts];
  __shared__ int64_t sbase[kVtUtts];
  __shared__ int sT[kVtUtts], sV[kVtUtts];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int u0 = blockIdx.x * kVtUtts;
  for (int idx = tid; idx < kVtUtts * NS * NS; idx += kVtThreads) {
    const int uu = idx / (NS * NS), k = idx - uu * NS * NS;
    const int u = u0 + uu;
    const int v = (u < U) ? u2m[u] : -1;
    sLA[uu][k] = (v >= 0) ? log(Aall[(int64_t)v * NS * NS + k]) : 0.0;
  }
  if (tid < kVtUtts) {
    const int u = u0 + tid;
    sV[tid] = (u < U) ? u2m[u] : -1;
    sbase[tid] = (u < U) ? off[u] : 0;
    sT[tid] = (u < U) ? (int)(off[u + 1] - off[u]) : 0;
    sScore[tid] = -INFINITY;  // no frame, no path
  }
  __syncthreads();
  int Tmax = 0;
#pragma unroll
  for (int uu = 0; uu < kVtUtts; uu++) Tmax = max(Tmax, sV[uu] >= 0 ? sT[uu] : 0);

  // ---------------- phase 1: delta recursion, one thread per live utterance (k_viterbi's) ----------------
  const int cl = lane & (kVtUtts - 1);
  const bool chain = warp == 0 && lane < kVtUtts && sV[cl] >= 0 && sT[cl] > 0;
  const int myT = chain ? sT[lane] : 0;
  const int64_t mybase = chain ? sbase[lane] : 0;
  double la[NS * NS], dl[NS];
#pragma unroll
  for (int k = 0; k < NS * NS; k++) la[k] = chain ? sLA[lane][k] : 0.0;
#pragma unroll
  for (int i = 0; i < NS; i++) dl[i] = 0.0;
  for (int w0 = 0; w0 < Tmax; w0 += kVtWin) {
    __syncthreads();
    for (int it = tid; it < kVtUtts * kVtWin * NS; it += kVtThreads) {
      const int uu = it / (kVtWin * NS), rem = it - uu * (kVtWin * NS);
      const int k = rem / NS;
      if (sV[uu] >= 0 && w0 + k < sT[uu]) lb[(size_t)uu * US + rem] = logb[(sbase[uu] + w0) * NS + rem];
    }
    __syncthreads();
    if (chain) {
      const float *bw = lb + (size_t)lane * US;
      const int kend = min(kVtWin, myT - w0);
      for (int k = 0; k < kend; k++) {
        double b[NS], dn[NS];
        unsigned long long ps = 0ull;
#pragma unroll
        for (int i = 0; i < NS; i++) b[i] = (double)bw[k * NS + i];
        if (w0 + k == 0) {
#pragma unroll
          for (int i = 0; i < NS; i++) dn[i] = (i == 0 ? 0.0 : -INFINITY) + b[i];
        } else {
#pragma unroll
          for (int j = 0; j < NS; j++) {
            // the banded shortcut of k_viterbi: the scan starts from i = 0 as the full one does, then only the in-band
            // predecessors can win the strict '>'
            double best = dl[0] + la[j];
            int arg = 0;
#pragma unroll
            for (int i = 1; i < NS; i++) {
              if (!BANDED || i == j || i + 1 == j) {
                const double cnd = dl[i] + la[i * NS + j];
                if (cnd > best) { best = cnd; arg = i; }
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
  if (chain) sScore[lane] = dl[NS - 1];
  __syncthreads();  // the chains' psi_ws stores and scores are visible to the CTA's other warps after the barrier

  // ---------------- phase 2: back-trace, gamma rows and counts, one warp per utterance ----------------
  for (int uu = warp; uu < kVtUtts; uu += kVtThreads / 32) {
    const int u = u0 + uu;
    if (u >= U) continue;
    const int T = sT[uu], v = sV[uu];
    const int64_t base = sbase[uu];
    if (v < 0) {  // masked utterance (its model has converged): not aligned
      for (int t = lane; t < T; t += 32) path[base + t] = -1;
      if (lane == 0) logp_utt[u] = 0.0;
      continue;
    }
    const double score = sScore[uu];
    const bool ok = score > -INFINITY;  // warp-uniform: some path reaches the final state
    int cn[NS * NS], cdt[NS], cdm[NS];  // warp-uniform counts (ballots)
#pragma unroll
    for (int k = 0; k < NS * NS; k++) cn[k] = 0;
#pragma unroll
    for (int i = 0; i < NS; i++) { cdt[i] = 0; cdm[i] = 0; }
    int sidx = NS - 1, later = 0;  // later: the state of the first frame of the chunk after this one
    for (int c0 = T > 0 ? ((T - 1) / 32) * 32 : -32; c0 >= 0; c0 -= 32) {
      const int t = c0 + lane;
      const unsigned long long my_psi = (t < T) ? psi_ws[base + t] : 0ull;
      int my_state = 0;
      const int ns = min(32, T - c0);
      for (int s = ns - 1; s >= 0; s--) {
        if (lane == s) my_state = sidx;
        const unsigned long long ps = __shfl_sync(0xffffffffu, my_psi, s);
        sidx = (int)((ps >> (8 * sidx)) & 0xffull);
      }
      int succ = __shfl_down_sync(0xffffffffu, my_state, 1);
      if (lane == 31) succ = later;
      later = __shfl_sync(0xffffffffu, my_state, 0);
      if (t < T) path[base + t] = my_state;
      // the chunk's gamma rows as consecutive words: word w is state w % NS of frame c0 + w / NS
#pragma unroll
      for (int w = lane; w < 32 * NS; w += 32) {
        const int f = w / NS, i = w - f * NS;
        const int sf = __shfl_sync(0xffffffffu, my_state, f);
        if (w < ns * NS) gamma[(base + c0) * NS + w] = (ok && sf == i) ? 1.f : 0.f;
      }
      if (ok) {
        const bool in = t < T, inner = t + 1 < T;
#pragma unroll
        for (int i = 0; i < NS; i++) {
          cdm[i] += __popc(__ballot_sync(0xffffffffu, in && my_state == i));
          cdt[i] += __popc(__ballot_sync(0xffffffffu, inner && my_state == i));
#pragma unroll
          for (int j = 0; j < NS; j++)
            if (!BANDED || j == i || j == i + 1) cn[i * NS + j] += __popc(__ballot_sync(0xffffffffu, inner && my_state == i && succ == j));
        }
      }
    }
    if (lane == 0) {
      logp_utt[u] = score;
      if (ustats) {
        double *row = ustats + (int64_t)upos[u] * (4 * NS + 1);
#pragma unroll
        for (int i = 0; i < NS; i++) {
          row[i] = (double)cn[i * NS + i];
          row[NS + i] = (i + 1 < NS) ? (double)cn[i * NS + i + 1] : 0.0;
          row[2 * NS + i] = (double)cdt[i];
          row[3 * NS + i] = (double)cdm[i];
        }
        row[4 * NS] = score;
      } else {
        double *st = stats + (int64_t)v * stats_stride;
#pragma unroll
        for (int k = 0; k < NS * NS; k++)
          if (cn[k]) atomicAdd(st + k, (double)cn[k]);
#pragma unroll
        for (int i = 0; i < NS; i++) {
          if (cdt[i]) atomicAdd(st + NS * NS + i, (double)cdt[i]);
          if (cdm[i]) atomicAdd(st + NS * NS + NS + i, (double)cdm[i]);
        }
        atomicAdd(st + off_sumlogp, score);
        atomicAdd(st + off_sumlogp + 1, 1.0);
      }
    }
  }
}

}  // namespace hmmk
