// tc_kernels.cuh -- tensor-core (tcgen05 / TMEM) kernels for sm_100a.
//
// Emissions as a dense contraction (north_star; calc_gaus / calc_symbol_probab, T-FS:1749-1841):
//   ln N_g(x_f) + ln c_g = kc[g] + sum_k Xaug[f][k] * W[g][k]
//   Xaug[f] = [ x_0..x_{DP-1} | x_0^2..x_{DP-1}^2 ]            (x centred, DP = padded D)
//   W[g]    = [ mu*iv         | -0.5*iv             ]            (pad columns 0)
//   kc[g]   = ln c - 0.5 (D ln 2pi + ln|det|) - 0.5 sum mu^2 iv  (added in the epilogue, exact fp32)
// computed with 3xTF32 (FP32-accurate split): every fp32 operand is split into hi = its top 11
// mantissa bits and lo = the exact remainder; D = Ah*Bh + Al*Bh + Ah*Bl accumulates in one TMEM
// tile through 3*KP/8 tcgen05.mma(kind::tf32, M=128, N=TN, K=8) instructions issued by one thread.
// The epilogue reads the accumulator back with tcgen05.ld and fuses the per-state log-sum-exp over
// the M mixtures (and, for training, the normalised per-mixture posteriors).
//
// Shared-memory operand layout (both operands K-major, SWIZZLE_NONE): one "slab" per K-step of 8
// values; inside a slab the 8-row x 16-byte core matrices are stored contiguously (128 B); the two
// K-chunks of a row group are 128 B apart (LBO), row groups 256 B apart (SBO):
//   byte(row, k) = (k/8)*slab + (row/8)*256 + ((k%8)/4)*128 + (row%8)*16 + (k%4)*4
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.cuh"

namespace hmmk {

constexpr int kTcRows = 128;       // frames per tile = UMMA M
constexpr int kTcThreads = 256;    // 8 warps
constexpr int kTcMaxTN = 192;      // Gaussians (columns) per tile, multiple of 16

struct TcTile {
  int32_t row0;    // TRAIN: index into frame_ids; DECODE: first frame of the tile relative to fbase
  int32_t nrows;   // valid rows (<= 128)
  int32_t img;     // first W image (TRAIN: the one image to use; DECODE: unused)
  int32_t state0;  // TRAIN: first state (within the model) covered by the image; DECODE: unused
  int32_t v;       // TRAIN: model; DECODE: unused
  int32_t pad;
};

__host__ __device__ inline int tc_slab_bytes(int rows) { return rows * 32; }
// bytes of one W image: hi and lo, KP/8 slabs each
__host__ __device__ inline size_t tc_image_bytes(int TN, int KP) { return (size_t)2 * (KP / 8) * tc_slab_bytes(TN); }
__host__ __device__ inline uint32_t tc_elem_off(int row, int k) {
  return (uint32_t)((row >> 3) * 256 + (((k & 7) >> 2) * 128) + ((row & 7) * 16) + ((k & 3) * 4));
}

// ---- raw PTX wrappers -------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  // SWIZZLE_NONE, K-major: LBO = 128 B (between the two K-chunks), SBO = 256 B (between 8-row groups)
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)(128 >> 4) << 16;
  d |= (uint64_t)(256 >> 4) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version 1 (Blackwell)
  return d;
}

__host__ __device__ inline uint32_t make_idesc_tf32(int M, int N) {
  // c_format F32 (1) @4, a_format TF32 (2) @7, b_format TF32 (2) @10, K-major A and B, N>>3 @17, M>>4 @24
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// One lane of a converged warp.  The MMA issue loops run under this predicate with warp-uniform operands
// (TMEM base re-broadcast with __shfl_sync) so that ptxas keeps descriptors in uniform registers; under
// `if (lane == 0)` it wrapped every tcgen05.mma in an ELECT / R2UR.BROADCAST waterfall loop (~120 cycles
// per issue, measured with scripts/debug_ws_timeline.py).
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred = 0, laneid = 0;
  asm volatile(
      "{\n\t"
      ".reg .b32 %%rx;\n\t"
      ".reg .pred %%px;\n\t"
      "elect.sync %%rx|%%px, %2;\n\t"
      "@%%px mov.s32 %1, 1;\n\t"
      "mov.s32 %0, %%rx;\n\t"
      "}\n"
      : "+r"(laneid), "+r"(pred)
      : "r"(0xFFFFFFFFu));
  return pred != 0;
}
__device__ __forceinline__ void tc_commit(uint64_t *mbar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(mbar)) : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t *mbar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(mbar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *mbar, uint32_t parity) {
  uint32_t done = 0;
  const uint32_t addr = smem_u32(mbar);
  while (!done) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// 8 consecutive accumulator columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float *v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; i++) v[i] = __uint_as_float(r[i]);
}

// v = hi + lo + r, |r| <= 2^-24 |v|: both parts rounded to nearest (cvt.rna), so the split is unbiased and
// the dropped lo*lo term of the 3xTF32 product is <= 2^-24 relative.
__device__ __forceinline__ float to_tf32_rn(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}
__device__ __forceinline__ void split_tf32(float v, float &hi, float &lo) {
  hi = to_tf32_rn(v);
  lo = to_tf32_rn(v - hi);
}

// ---- W image packer ----------------------------------------------------------------------------
// One image = TN Gaussian rows (whole states) x KP, hi slabs then lo slabs.  Image i covers global
// states [img_state0[i], img_state0[i] + img_nstates[i]); rows beyond are zero with kc = -inf.
__global__ void k_pack_w_tc(const double *__restrict__ mu, const double *__restrict__ iv, const double *__restrict__ det,
                            const double *__restrict__ c, const double *__restrict__ ctr, int M, int D, int DP, int TN,
                            const int32_t *__restrict__ img_state0, const int32_t *__restrict__ img_nstates,
                            float *__restrict__ images, float *__restrict__ kc) {
  const int img = blockIdx.x;
  const int KP = 2 * DP;
  const size_t img_floats = tc_image_bytes(TN, KP) / 4;
  float *hi = images + (size_t)img * img_floats;
  float *lo = hi + img_floats / 2;
  const int64_t g0 = (int64_t)img_state0[img] * M;
  const int ng = img_nstates[img] * M;
  for (int idx = threadIdx.x; idx < TN * KP; idx += blockDim.x) {
    const int n = idx / KP, k = idx - n * KP;
    const int part = k / DP, d = k - part * DP;
    float val = 0.f;
    if (n < ng && d < D) {
      const double m = mu[(g0 + n) * D + d] - ctr[d], w = iv[(g0 + n) * D + d];
      val = (float)(part == 0 ? m * w : -0.5 * w);
    }
    float h, l;
    split_tf32(val, h, l);
    const size_t o = (size_t)(k >> 3) * (tc_slab_bytes(TN) / 4) + tc_elem_off(n, k) / 4;
    hi[o] = h;
    lo[o] = l;
  }
  for (int n = threadIdx.x; n < TN; n += blockDim.x) {
    double k = -INFINITY;
    if (n < ng) {
      const double dt = det[g0 + n], cc = c[g0 + n];
      if (dt != 0.0 && cc > 0.0) {
        double q = 0.0;
        for (int d = 0; d < D; d++) {
          const double m = mu[(g0 + n) * D + d] - ctr[d];
          q += m * m * iv[(g0 + n) * D + d];
        }
        k = log(cc) - 0.5 * ((double)D * 1.8378770664093453 + log(fabs(dt))) - 0.5 * q;
      }
    }
    kc[(size_t)img * TN + n] = (float)k;
  }
}

// ---- emission GEMM ------------------------------------------------------------------------------
// dynamic smem: A_hi | A_lo (KP/8 slabs of 4 KB each) | B image (hi, lo) | kc[TN] | lbs[N<=8][128] (TRAIN)
__host__ __device__ inline size_t tc_emis_smem_bytes(int TN, int KP) {
  return (size_t)2 * (KP / 8) * tc_slab_bytes(kTcRows) + tc_image_bytes(TN, KP) + sizeof(float) * TN + sizeof(float) * 8 * kTcRows + 1024;
}

template <bool TRAIN>
__global__ void __launch_bounds__(kTcThreads, 1)
k_emis_tc(const TcTile *__restrict__ tiles, int ntiles, const int32_t *__restrict__ frame_ids, const float *__restrict__ x32,
          const float *__restrict__ images, const float *__restrict__ kcs, int nimages, int N, int M, int DP, int TN,
          float *__restrict__ logb, int64_t fbase, int64_t ldb, int S_total, int SCt, float *__restrict__ post) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ uint64_t mbar;
  __shared__ uint32_t tmem_base_s;
  const int KP = 2 * DP, NSLAB = KP / 8;
  const int aslab = tc_slab_bytes(kTcRows), bslab = tc_slab_bytes(TN);
  uint8_t *sm = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t *A_hi = sm, *A_lo = sm + (size_t)NSLAB * aslab;
  uint8_t *B_hi = A_lo + (size_t)NSLAB * aslab, *B_lo = B_hi + (size_t)NSLAB * bslab;
  float *kc = reinterpret_cast<float *>(B_lo + (size_t)NSLAB * bslab);
  float *lbs = kc + TN;  // [8][128]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int G = N * M;

  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < TN + 8) tmem_cols <<= 1;
  if (warp == 0) tmem_alloc(&tmem_base_s, tmem_cols);
  if (tid == 0) mbar_init(&mbar, 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = tmem_base_s;
  const uint32_t idesc = make_idesc_tf32(kTcRows, TN);
  uint32_t parity = 0;
  int cur_img = -1;

  // contiguous range of tiles per CTA (tiles are ordered by model, so W reloads are rare)
  const int per = (ntiles + gridDim.x - 1) / gridDim.x;
  const int t_begin = blockIdx.x * per, t_end = min(ntiles, t_begin + per);
  for (int ti = t_begin; ti < t_end; ti++) {
    const TcTile tile = tiles[ti];
    // ---- A tile: [x | x^2] of 128 frames, split hi / lo, straight into the UMMA layout ----
    {
      const int r = tid & 127, half = tid >> 7;  // half 0: x columns, half 1: x^2 columns
      int64_t f = -1;
      if (r < tile.nrows) f = TRAIN ? (int64_t)frame_ids[tile.row0 + r] : fbase + tile.row0 + r;
      const float4 *src = reinterpret_cast<const float4 *>(x32 + (f < 0 ? 0 : f) * DP);
      for (int q = 0; q < DP / 4; q++) {
        float4 xv = (f >= 0) ? src[q] : make_float4(0.f, 0.f, 0.f, 0.f);
        if (half) { xv.x *= xv.x; xv.y *= xv.y; xv.z *= xv.z; xv.w *= xv.w; }
        float4 h, l;
        split_tf32(xv.x, h.x, l.x); split_tf32(xv.y, h.y, l.y); split_tf32(xv.z, h.z, l.z); split_tf32(xv.w, h.w, l.w);
        const int k = half * DP + q * 4;
        const uint32_t o = (uint32_t)(k >> 3) * aslab + tc_elem_off(r, k);
        *reinterpret_cast<float4 *>(A_hi + o) = h;
        *reinterpret_cast<float4 *>(A_lo + o) = l;
      }
    }
    const int n_img = TRAIN ? 1 : nimages;
    for (int ii = 0; ii < n_img; ii++) {
      const int img = TRAIN ? tile.img : ii;
      if (img != cur_img) {  // ---- B image (pre-packed in global memory in the smem layout) ----
        const float4 *src = reinterpret_cast<const float4 *>(images + (size_t)img * (tc_image_bytes(TN, KP) / 4));
        float4 *dst = reinterpret_cast<float4 *>(B_hi);
        const int n16 = (int)(tc_image_bytes(TN, KP) / 16);
        for (int i = tid; i < n16; i += kTcThreads) dst[i] = src[i];
        for (int i = tid; i < TN; i += kTcThreads) kc[i] = kcs[(size_t)img * TN + i];
        cur_img = img;
      }
      fence_async_smem();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
      tc_fence_before();
      __syncthreads();
      if (warp == 0) {
        tc_fence_after();
        const uint32_t td = __shfl_sync(0xffffffffu, tmem_d, 0);
        if (elect_one_sync()) {
          const uint32_t a_hi = smem_u32(A_hi), a_lo = smem_u32(A_lo), b_hi = smem_u32(B_hi), b_lo = smem_u32(B_lo);
          uint32_t acc = 0;
          for (int p = 0; p < 3; p++) {  // Ah*Bh, Al*Bh, Ah*Bl
            const uint32_t a0 = (p == 1) ? a_lo : a_hi, b0 = (p == 2) ? b_lo : b_hi;
            for (int j = 0; j < NSLAB; j++) {
              tc_mma_tf32(td, make_smem_desc(a0 + j * aslab), make_smem_desc(b0 + j * bslab), idesc, acc);
              acc = 1;
            }
          }
          tc_commit(&mbar);
        }
        __syncwarp();
      }
      mbar_wait(&mbar, parity);
      parity ^= 1;
      tc_fence_after();

      // ---- epilogue: thread <-> (row = 32*(warp%4) + lane, column half = warp/4), whole states ----
      {
        const int row = 32 * (warp & 3) + lane;
        const int chalf = warp >> 2;
        const int st_img0 = TRAIN ? tile.state0 : img * SCt;                 // first state of the image (global for DECODE)
        const int st_lim = TRAIN ? N : S_total;
        const int nst = max(0, min(SCt, st_lim - st_img0));                  // states present in this image
        const int sh = (nst + 1) >> 1;
        const int s_beg = chalf ? sh : 0, s_end = chalf ? nst : sh;          // my states within the image
        const int c_beg = s_beg * M, c_end = s_end * M;
        const uint32_t trow = tmem_d + ((uint32_t)(32 * (warp & 3)) << 16);
        const bool live = row < tile.nrows;
        int64_t f = 0;
        if (live) f = TRAIN ? (int64_t)frame_ids[tile.row0 + row] : fbase + tile.row0 + row;
        float *lrow = TRAIN ? logb + f * N + st_img0 : logb + (f - fbase) * ldb + st_img0;
        // pass 1: log-sum-exp per state (online), columns walked in aligned chunks of 8
        {
          float mx = kNegInf, sum = 0.f;
          int mcount = 0, s = s_beg;
          for (int c0 = c_beg & ~7; c0 < c_end; c0 += 8) {
            float v[8];
            tmem_ld8(trow + c0, v);
#pragma unroll
            for (int j = 0; j < 8; j++) {
              const int col = c0 + j;
              if (col >= c_beg && col < c_end) {
                const float val = v[j] + kc[col];
                if (val > mx) { sum = sum * __expf(mx - val) + 1.f; mx = val; }
                else if (val > kNegInf) sum += __expf(val - mx);
                if (++mcount == M) {
                  const float lb = (mx > kNegInf) ? mx + __logf(sum) : kNegInf;
                  if (live) lrow[s] = lb;
                  if (TRAIN) lbs[(s - s_beg + chalf * 4) * kTcRows + row] = lb;
                  s++; mcount = 0; mx = kNegInf; sum = 0.f;
                }
              }
            }
          }
        }
        // pass 2 (training): normalised per-mixture posteriors  c_m N_m / b_i
        if (TRAIN && post != nullptr) {
          float *prow = post + f * G + (int64_t)st_img0 * M;
          int mcount = 0, s = s_beg;
          for (int c0 = c_beg & ~7; c0 < c_end; c0 += 8) {
            float v[8];
            tmem_ld8(trow + c0, v);
#pragma unroll
            for (int j = 0; j < 8; j++) {
              const int col = c0 + j;
              if (col >= c_beg && col < c_end) {
                const float lb = lbs[(s - s_beg + chalf * 4) * kTcRows + row];
                const float p = (lb > kNegInf) ? __expf(v[j] + kc[col] - lb) : 0.f;
                if (live) prow[col] = p;
                if (++mcount == M) { s++; mcount = 0; }
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncthreads();  // accumulator, kc and lbs are free again
    }
  }
  tc_fence_after();
  if (warp == 0) tmem_dealloc(tmem_d, tmem_cols);
}


// ================================================================================================
// Mixture accumulators on the tensor pipe (calc_mix_param, T-FS:1691-1727).
//
// Per tile of 128 frames of one model, per block of 128 Gaussians ("row block"):
//   GEMM1   L[g][f]  = sum_k W[g][k] Xaug[f][k]                (M = 128 Gaussians, N = 128 frames, K = KP)
//   weights w[g][f]  = gamma_f(state(g)) * exp(L + kc[g] - logb_f(state(g)))   = gamma * c_m N_m / b_i
//   GEMM2   S[g][k] += sum_f w[g][f] Xaug[f][k]                (M = 128 Gaussians, N = KP, K = 128 frames)
// The per-mixture posteriors are recomputed from the features instead of being read back from HBM:
// the kernel reads x (once), log b and gamma and writes nothing but the statistics.  Both GEMMs are
// 3xTF32 (FP32-accurate split, hi*hi + lo*hi + hi*lo) with the A operand in TENSOR MEMORY: W (hi, lo)
// is parked in TMEM for as long as the CTA stays on one (model, row block); GEMM1 leaves L in TMEM
// with one Gaussian per lane, the epilogue turns it into w in place (hi) and beside it (lo) with
// tcgen05.st, and GEMM2 consumes that directly.  Shared memory holds only the frame tile, twice:
// X (frames x columns, K-major for GEMM1) and XT (columns x frames, K-major for GEMM2) -- the
// MN-major operand form returned zeros for kind::tf32 on this part (scripts/tc_probe.cu).
// S accumulates in TMEM for at most kAccFlushTiles tiles, then moves to double-precision registers
// (the tensor pipe's FP32 accumulation truncates); registers are flushed with double atomics when the
// CTA's (model, row block) changes.
//   S[g][0..D-1] = sum w x (centred) -> S1,  S[g][D] = sum w -> S0 (x column D is the constant 1),
//   S[g][DP..DP+D-1] = sum w x^2 -> "raw" second moment; k_finalize_stats turns it into the
//   reference's sum w (x - mu_old)^2 in double.
//
// Shared-memory operand layouts (SWIZZLE_NONE K-major canonical form, 16-byte chunks of 4 values):
//   X  : byte(f, k) = (f%8)*16 + (k%4)*4 + (k/4)*128 + (f/8)*PX       PX = (KP/4)*128;   LBO 128, SBO PX
//   XT : byte(k, f) = (k%8)*16 + (f%4)*4 + (f/4)*128 + (k/8)*4096     (KP2 rows);        LBO 128, SBO 4096
// TMEM columns: [0,128) L / w_hi | [128,256) w_lo | [256, 256+KP2) S | [352, 352+2KP) W_hi, W_lo
// ================================================================================================
constexpr int kAccFlushTiles = 2;
constexpr int kAccTmW = 352;

__host__ __device__ inline int tc_kp2(int KP) { return (KP + 15) / 16 * 16; }
__host__ __device__ inline size_t tc_accT_image_bytes(int KP) { return (size_t)128 * 2 * KP * 4; }  // [128][Wh(KP) | Wl(KP)] row-major
__host__ __device__ inline size_t tc_acc_smem_bytes(int KP) {
  return (size_t)2 * 16 * (KP / 4) * 128 + (size_t)2 * (tc_kp2(KP) / 8) * 4096 + sizeof(float) * 128 * 8 + sizeof(int32_t) * 128 + 1024;
}
__host__ __device__ inline bool tc_acc_fits(int KP) { return KP <= 80 && tc_acc_smem_bytes(KP) <= 227 * 1024; }

__device__ __forceinline__ uint64_t make_smem_desc2(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
// A operand from tensor memory
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t *r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t *r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t *r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t *r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
               "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// kc2[g] = log2(e) (ln c - 0.5 (D ln 2pi + ln|det|) - 0.5 sum (mu - ctr)^2 iv), -inf for a Gaussian of density 0
// (c == 0 or det == 0): the additive constant of every Gaussian, one thread each, shared by all W packers.
__global__ void k_pack_kc(const double *__restrict__ mu, const double *__restrict__ iv, const double *__restrict__ det,
                          const double *__restrict__ c, const double *__restrict__ ctr, int64_t VG, int D, float *__restrict__ kc2) {
  // one warp per Gaussian, lanes over the dimensions (coalesced reads of mu / iv, shuffle reduction)
  const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  pdl_wait();
  pdl_trigger();
  if (g >= VG) return;
  double q = 0.0;
  for (int d = lane; d < D; d += 32) {
    const double m = mu[g * D + d] - ctr[d];
    q += m * m * iv[g * D + d];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  if (lane == 0) {
    double k = -INFINITY;
    const double dt = det[g], cc = c[g];
    if (dt != 0.0 && cc > 0.0) k = (log(cc) - 0.5 * ((double)D * 1.8378770664093453 + log(fabs(dt))) - 0.5 * q) * 1.4426950408889634;
    kc2[g] = (float)k;
  }
}

// W images for the accumulate kernel: image (v, rb) = Gaussians [rb*128, rb*128+128) of model v, row-major
// [128][Wh[KP] | Wl[KP]]; rows beyond G are zero with kc = -inf.  kcT is pre-multiplied by log2(e).
__global__ void k_pack_wT_tc(const double *__restrict__ mu, const double *__restrict__ iv, const float *__restrict__ kc2all,
                             const double *__restrict__ ctr, int G, int nRB, int D, int DP, float *__restrict__ images,
                             float *__restrict__ kcT) {
  const int img = blockIdx.y, v = img / nRB, rb = img - v * nRB;
  const int KP = 2 * DP;
  float *im = images + (size_t)img * (tc_accT_image_bytes(KP) / 4);
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 128 * KP; idx += gridDim.x * blockDim.x) {
    const int r = idx / KP, k = idx - r * KP;
    const int part = k / DP, d = k - part * DP;
    const int g = rb * 128 + r;
    float val = 0.f;
    if (g < G && d < D) {
      const int64_t gg = (int64_t)v * G + g;
      const double m = mu[gg * D + d] - ctr[d], w = iv[gg * D + d];
      val = (float)(part == 0 ? m * w : -0.5 * w);
    }
    float h, l;
    split_tf32(val, h, l);
    im[(size_t)r * 2 * KP + k] = h;
    im[(size_t)r * 2 * KP + KP + k] = l;
    if (k == 0) kcT[(size_t)img * 128 + r] = (g < G) ? kc2all[(int64_t)v * G + g] : kNegInf;
  }
}

// units: {row0 (index into frame_ids), nrows, img = v*nRB + rb, state0 unused, v, pad = rb}
__global__ void __launch_bounds__(kTcThreads, 1)
k_accum_tc(const TcTile *__restrict__ units, int nunits, const int32_t *__restrict__ frame_ids, const float *__restrict__ x32,
           const float *__restrict__ images, const float *__restrict__ kcT, const float *__restrict__ logb,
           const float *__restrict__ gamma, int N, int M, int G, int D, int DP, double *__restrict__ stats,
           int64_t stats_stride, int64_t off_S0, int64_t off_S1, int64_t off_S2) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ uint64_t mbar;
  __shared__ uint32_t tmem_base_s;
  const int KP = 2 * DP, KP2 = tc_kp2(KP), NSLAB = KP / 8;
  const uint32_t PX = (uint32_t)(KP / 4) * 128;
  uint8_t *sm = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t *Xh = sm, *Xl = sm + 16 * PX;
  uint8_t *XTh = Xl + 16 * PX, *XTl = XTh + (size_t)(KP2 / 8) * 4096;
  float *cfs = reinterpret_cast<float *>(XTl + (size_t)(KP2 / 8) * 4096);  // [128 frames][8]: log2(gamma) - logb*log2(e)
  int32_t *fid = reinterpret_cast<int32_t *>(cfs + 128 * 8);               // [128] frame index of each tile row, -1 = none
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (warp == 0) tmem_alloc(&tmem_base_s, 512);
  if (tid == 0) mbar_init(&mbar, 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem0 = tmem_base_s;
  const uint32_t tm_d1 = tmem0, tm_wl = tmem0 + 128, tm_d2 = tmem0 + 256, tm_w = tmem0 + kAccTmW;
  const uint32_t idesc1 = make_idesc_tf32(128, 128);
  const uint32_t idesc2 = make_idesc_tf32(128, KP2);
  uint32_t parity = 0;

  // this thread's share of the accumulator: Gaussian row `row`, 8-column groups [c8_beg, c8_end)
  const int row = 32 * (warp & 3) + lane;
  const int chalf = warp >> 2;
  const int nc8 = KP2 / 8;
  const int c8_beg = chalf ? (nc8 + 1) / 2 : 0, c8_end = chalf ? nc8 : (nc8 + 1) / 2;
  constexpr int kMaxC8 = 5;  // KP2 <= 80 (tc_acc_fits)
  double acc[kMaxC8 * 8];
#pragma unroll
  for (int i = 0; i < kMaxC8 * 8; i++) acc[i] = 0.0;

  const int per = (nunits + gridDim.x - 1) / gridDim.x;
  const int u_begin = blockIdx.x * per, u_end = min(nunits, u_begin + per);
  int cur_img = -1, cur_v = -1, cur_rb = 0, since_flush = 0;
  float kcr = kNegInf;
  const uint32_t trow = (uint32_t)(32 * (warp & 3)) << 16;

  auto drain_tmem = [&]() {  // S (TMEM, fp32) -> acc (registers, double)
#pragma unroll
    for (int q = 0; q < kMaxC8; q++) {
      const int c8 = c8_beg + q;
      if (c8 < c8_end) {
        float v[8];
        tmem_ld8(tm_d2 + trow + c8 * 8, v);
#pragma unroll
        for (int j = 0; j < 8; j++) acc[q * 8 + j] += (double)v[j];
      }
    }
  };
  auto flush_global = [&]() {  // acc -> statistics of (cur_v, cur_rb)
    const int g = cur_rb * 128 + row;
    double *st = stats + (int64_t)cur_v * stats_stride;
#pragma unroll
    for (int q = 0; q < kMaxC8; q++) {
      const int c8 = c8_beg + q;
#pragma unroll
      for (int j = 0; j < 8; j++) {
        if (c8 < c8_end && g < G) {
          const int k = c8 * 8 + j;
          const double a = acc[q * 8 + j];
          if (k < D) atomicAdd(st + off_S1 + (int64_t)g * D + k, a);
          else if (k == D) atomicAdd(st + off_S0 + g, a);
          else if (k >= DP && k < DP + D) atomicAdd(st + off_S2 + (int64_t)g * D + (k - DP), a);
        }
        acc[q * 8 + j] = 0.0;
      }
    }
  };

  for (int ui = u_begin; ui < u_end; ui++) {
    const TcTile unit = units[ui];
    if (unit.img != cur_img && cur_img >= 0) {  // (model, row block) changes: everything accumulated so far goes out
      if (since_flush > 0) { drain_tmem(); since_flush = 0; }
      flush_global();
    }
    // ---- frame ids and the per-frame, per-state weight exponent ----
    if (tid < 128) {
      const int f = (tid < unit.nrows) ? frame_ids[unit.row0 + tid] : -1;
      fid[tid] = f;
      for (int s = 0; s < 8; s++) {
        float cf = kNegInf;
        if (f >= 0 && s < N) {
          const float gm = __ldg(gamma + (int64_t)f * N + s), lb = __ldg(logb + (int64_t)f * N + s);
          if (gm > 0.f && lb > kNegInf) cf = __log2f(gm) - lb * 1.4426950408889634f;
        }
        cfs[tid * 8 + s] = cf;
      }
    }
    if (unit.img != cur_img) {  // W (hi | lo) of this row block -> TMEM, one Gaussian per lane
      const float *im = images + (size_t)unit.img * (tc_accT_image_bytes(KP) / 4) + (size_t)row * 2 * KP;
      const int nch = 2 * KP / 8;  // 8-column chunks
      for (int ch = chalf; ch < nch; ch += 2) {
        uint32_t r[8];
        const float4 a = __ldg(reinterpret_cast<const float4 *>(im + ch * 8)), b = __ldg(reinterpret_cast<const float4 *>(im + ch * 8 + 4));
        r[0] = __float_as_uint(a.x); r[1] = __float_as_uint(a.y); r[2] = __float_as_uint(a.z); r[3] = __float_as_uint(a.w);
        r[4] = __float_as_uint(b.x); r[5] = __float_as_uint(b.y); r[6] = __float_as_uint(b.z); r[7] = __float_as_uint(b.w);
        tmem_st8(tm_w + trow + ch * 8, r);
      }
      tmem_wait_st();
      cur_img = unit.img; cur_v = unit.v; cur_rb = unit.pad;
      kcr = (cur_rb * 128 + row < G) ? kcT[(size_t)unit.img * 128 + row] : kNegInf;
    }
    __syncthreads();  // fid
    // ---- X: [x | x^2] of 128 frames as rows, hi / lo ----
    {
      const int r = tid & 127, half = tid >> 7;
      const int f = fid[r];
      const float4 *src = reinterpret_cast<const float4 *>(x32 + (int64_t)(f < 0 ? 0 : f) * DP);
      const uint32_t rbase = (uint32_t)(r & 7) * 16 + (uint32_t)(r >> 3) * PX;
      for (int q = 0; q < DP / 4; q++) {
        float4 xv = (f >= 0) ? __ldg(src + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (half) { xv.x *= xv.x; xv.y *= xv.y; xv.z *= xv.z; xv.w *= xv.w; }
        float4 h, l;
        split_tf32(xv.x, h.x, l.x); split_tf32(xv.y, h.y, l.y); split_tf32(xv.z, h.z, l.z); split_tf32(xv.w, h.w, l.w);
        const uint32_t o = rbase + (uint32_t)(half * (DP / 4) + q) * 128;
        *reinterpret_cast<float4 *>(Xh + o) = h;
        *reinterpret_cast<float4 *>(Xl + o) = l;
      }
    }
    // ---- XT: the same tile with columns as rows (4 consecutive frames per 16-byte chunk) ----
    for (int it = tid; it < 32 * KP2; it += kTcThreads) {
      const int fg = it / KP2, n = it - fg * KP2;  // frames 4fg..4fg+3, Xaug column n
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (n < KP) {
        const int d = (n < DP) ? n : n - DP;
        const int f0 = fid[4 * fg], f1 = fid[4 * fg + 1], f2 = fid[4 * fg + 2], f3 = fid[4 * fg + 3];
        if (f0 >= 0) v.x = __ldg(x32 + (int64_t)f0 * DP + d);
        if (f1 >= 0) v.y = __ldg(x32 + (int64_t)f1 * DP + d);
        if (f2 >= 0) v.z = __ldg(x32 + (int64_t)f2 * DP + d);
        if (f3 >= 0) v.w = __ldg(x32 + (int64_t)f3 * DP + d);
        if (n >= DP) { v.x *= v.x; v.y *= v.y; v.z *= v.z; v.w *= v.w; }
      }
      float4 h, l;
      split_tf32(v.x, h.x, l.x); split_tf32(v.y, h.y, l.y); split_tf32(v.z, h.z, l.z); split_tf32(v.w, h.w, l.w);
      const uint32_t o = (uint32_t)(n & 7) * 16 + (uint32_t)fg * 128 + (uint32_t)(n >> 3) * 4096;
      *reinterpret_cast<float4 *>(XTh + o) = h;
      *reinterpret_cast<float4 *>(XTl + o) = l;
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    // ---- GEMM1: L[g][f] ----
    if (warp == 0) {
      tc_fence_after();
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem0, 0);
      if (elect_one_sync()) {
        const uint64_t xh = make_smem_desc2(smem_u32(Xh), 128, PX), xl = make_smem_desc2(smem_u32(Xl), 128, PX);
        uint32_t accf = 0;
        for (int p = 0; p < 3; p++) {  // Wh*Xh, Wl*Xh, Wh*Xl
          const uint32_t a0 = tb + kAccTmW + ((p == 1) ? KP : 0);
          const uint64_t b0 = (p == 2) ? xl : xh;
          for (int j = 0; j < NSLAB; j++) {
            tc_mma_tf32_ts(tb, a0 + j * 8, b0 + (uint64_t)(j * 16), idesc1, accf);  // +256 B per K-step
            accf = 1;
          }
        }
        tc_commit(&mbar);
      }
      __syncwarp();
    }
    mbar_wait(&mbar, parity);
    parity ^= 1;
    tc_fence_after();
    // ---- weights, in place: thread <-> (Gaussian row, 64 frames) ----
    {
      const int s = min((cur_rb * 128 + row) / M, 7);
      for (int c0 = chalf * 64; c0 < chalf * 64 + 64; c0 += 16) {
        uint32_t v[16], vl[16];
        tmem_ld16(tm_d1 + trow + c0, v);
#pragma unroll
        for (int j = 0; j < 16; j++) {
          const float y = fmaf(__uint_as_float(v[j]), 1.4426950408889634f, kcr + cfs[(c0 + j) * 8 + s]);
          float w;
          asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(w) : "f"(y));
          if (!(y > -150.f)) w = 0.f;  // -inf, NaN (inf - inf) and underflow
          float h, l;
          split_tf32(w, h, l);
          v[j] = __float_as_uint(h);
          vl[j] = __float_as_uint(l);
        }
        tmem_st16(tm_d1 + trow + c0, v);
        tmem_st16(tm_wl + trow + c0, vl);
      }
      tmem_wait_st();
    }
    tc_fence_before();
    __syncthreads();
    // ---- GEMM2: S[g][k] += sum_f w[g][f] Xaug[f][k] ----
    if (warp == 0) {
      tc_fence_after();
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem0, 0);
      if (elect_one_sync()) {
        const uint64_t xh = make_smem_desc2(smem_u32(XTh), 128, 4096), xl = make_smem_desc2(smem_u32(XTl), 128, 4096);
        uint32_t accf = since_flush > 0 ? 1u : 0u;
        for (int p = 0; p < 3; p++) {  // wh*Xh, wl*Xh, wh*Xl
          const uint32_t a0 = tb + ((p == 1) ? 128 : 0);
          const uint64_t b0 = (p == 2) ? xl : xh;
          for (int j = 0; j < 16; j++) {
            tc_mma_tf32_ts(tb + 256, a0 + j * 8, b0 + (uint64_t)(j * 16), idesc2, accf);
            accf = 1;
          }
        }
        tc_commit(&mbar);
      }
      __syncwarp();
    }
    mbar_wait(&mbar, parity);
    parity ^= 1;
    tc_fence_after();
    if (++since_flush >= kAccFlushTiles) { drain_tmem(); since_flush = 0; }
    tc_fence_before();
    __syncthreads();  // X, XT, cfs and the weight columns are free again
  }
  if (cur_img >= 0) {
    if (since_flush > 0) drain_tmem();
    flush_global();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 0) tmem_dealloc(tmem0, 512);
}

}  // namespace hmmk
