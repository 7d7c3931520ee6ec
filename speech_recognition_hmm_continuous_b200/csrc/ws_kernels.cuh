// ws_kernels.cuh -- warp-specialised, mbarrier-pipelined tcgen05 kernels for sm_100a.
//
// k_emis_ws: Gaussian-mixture emission log-likelihoods (calc_symbol_probab + calc_gaus, T-FS:1749-1841,
// R-FS:860-947) as a dense contraction on the tensor pipe with the per-state log-sum-exp fused into
// the epilogue.  One persistent CTA per SM, 17 warps in three roles that only meet at mbarriers:
//
//   warps 8-15 LOADERS   read 128 raw frames (fp32, centred; prefetched three levels ahead), form
//                        [x | x^2], split every value into TF32 hi + lo and write the A operand with
//                        tcgen05.st into TENSOR MEMORY (two warps per lane quarter, half a row per thread);
//                        (re)load the W image into shared memory when the unit's image changes
//   warp  16   MMA       one thread issues 3*KP/8 tcgen05.mma.kind::tf32 (hi*hi + lo*hi + hi*lo) per
//                        unit, A from TMEM, B = W from shared memory, into a TMEM accumulator stage,
//                        commits to free the operand stage and to publish the accumulator
//   warps 0-7  EPILOGUE  tcgen05.ld the accumulator (one frame per thread, two warps per lane quarter taking
//                        the 16-column groups of even / odd index), log-sum-exp over the M mixtures of each
//                        state (additive constants of the image from shared memory), store log b
//
// Why the frame operand lives in TMEM: with both operands in shared memory a K = 8 TF32 MMA of
// 128 x 80 reads (128 + 80) x 32 B = 6.6 KB for 40 cycles of math -- more than the 128 B/cycle the
// shared memory delivers; measured 120 cycles per MMA (scripts/debug_ws_timeline.py).  From TMEM the
// A operand costs no shared-memory bandwidth, the loaders need no generic->async proxy fence for it,
// and 160 KB of shared memory are freed.
//
// Two operand stages and two accumulator stages in TMEM keep the tensor pipe busy while the next
// frame tile is being expanded and the previous one reduced.  The additive constant kc[g] of every
// Gaussian is added in the epilogue in FP32 (round to nearest): folding it into the contraction was
// tried and rejected -- the tensor pipe's FP32 accumulation truncates, and a partial sum that starts
// at |kc| ~ 150 loses ~5e-5 of log-likelihood per frame, systematically (posteriors then sum to 1 - 5e-5).
// The epilogue forms log2(c_g N_g(x)) = fma(acc, log2 e, kc2[g]) with exactly the expression the
// accumulate kernel uses, so that the posteriors it recomputes are consistent with log b.
//
// Units are (W image, 128-frame tile) pairs ordered image-major, each CTA takes a contiguous range:
// training: explicit list (frames of one model gathered through frame_ids); decode: unit u = (u / ntiles,
// u % ntiles) over the contiguous frames of the current utterance batch.
//
// W image in shared memory (SWIZZLE_NONE, K-major, 16-byte chunks of 4 values), rows g, columns k:
//   byte(g, k) = (g%8)*16 + (k%4)*4 + (k/4)*128 + (g/8)*P,   P = (KP/4)*128;   LBO = 128, SBO = P,
//   K-step j starts at +256 j;  image = [hi: (TN/8) P][lo: (TN/8) P][kc2: TN floats].
// TMEM columns: operand stage a at 160 a: [x_hi (DP) | x2_hi (DP) | x_lo (DP) | x2_lo (DP)] (KP <= 80);
//               accumulator stage a at 320 + 96 a (TN <= 96); an image of one wide state (96 < TN <= 176) has a
//               single operand stage and its two accumulator stages at 160 + TN a.
#pragma once
#include <cuda_fp16.h>
#include "tc_kernels.cuh"

namespace hmmk {

constexpr int kWsEpiWarps = 8;    // epilogue warps (a multiple of 4: TMEM lane quarters; 12 measured slower: 80 registers per thread)
constexpr int kWsThreads = (kWsEpiWarps + 9) * 32;   // epilogue, 8 loaders, MMA issuer
constexpr int kWsMaxTN = 96;      // Gaussians (columns) per W image (two operand stages in tensor memory)
constexpr int kWsMaxTN1 = 176;    // ... of an image that holds one wide state (a single operand stage)
constexpr int kWsXch = 6;         // states per image when a state spans several 16-column chunks (M > 16)

// W image in global and shared memory: [hi: (TN/8) P][lo: (TN/8) P][kc2: TN floats]
__host__ __device__ inline size_t ws_image_bytes(int TN, int KP) { return (size_t)2 * (TN / 8) * (KP / 4) * 128 + (size_t)TN * 4; }
__host__ __device__ inline size_t ws_emis_smem_bytes(int TN, int KP) { return ws_image_bytes(TN, KP) + 1024 + 272; }

// Mixtures per state as laid out in the W image.  A 16-column chunk holds 16 / MP whole states (state boundaries never cut
// through a chunk; 16 % MP pad columns close it).  M <= 16: padded to a power of two -- except M = 3 and M = 5, where the
// padding would be a quarter / three eighths of every MMA: they are laid out as they are (five states of 3 and one pad
// column, three states of 5 and one pad column).  A chunk then holds an odd number of states, so a row-per-frame output
// needs 4-byte stores (k_emis_ws: measured 2x slower in the 1,000-word decode regime, every store its own sector); the
// decode kernel k_emis_dec writes an interleaved layout instead in which 4-byte stores of a warp fill whole lines.
// M > 16: padded to a multiple of 16 (a state spans M / 16 chunks).  Pad columns have W = 0 and kc = -inf (density 0).
__host__ __device__ inline int ws_pad_m(int M) {
  if (M > 16) return (M + 15) / 16 * 16;
  if (M == 3 || M == 5) return M;
  int p = 1;
  while (p < M) p <<= 1;
  return p;
}
// states per 16-column chunk (M <= 16), and the columns an image of `nstates` whole states occupies
__host__ __device__ inline int ws_states_per_chunk(int MPd) { return MPd <= 16 ? 16 / MPd : 1; }
__host__ __device__ inline int ws_image_cols(int MPd, int nstates) {
  if (MPd > 16) return nstates * MPd;
  const int spc = 16 / MPd;
  return (nstates + spc - 1) / spc * 16;
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// TF32 hi / lo split: hi = v rounded to nearest (ties away) to 11 significant bits with two integer
// instructions, lo = v - hi exactly (FP32); the tensor core ignores the low 13 mantissa bits of lo, which
// costs at most 2^-23 |v|, unbiased because lo has either sign.  (cvt.rna.tf32.f32 compiles to a longer
// NaN-safe sequence on sm_100a, and a rounded lo doubles the load on the ALU pipe, which is what bounds
// the loader and epilogue warps.)  The values here are finite.
__device__ __forceinline__ void split_tf32_fast(float v, float &hi, float &lo) {
  hi = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
  lo = v - hi;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, const float4 &v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&r)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}
// non-blocking poll (try_wait may suspend the thread for a long time when the phase is not complete)
__device__ __forceinline__ bool mbar_try(uint64_t *mbar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(done)
      : "r"(smem_u32(mbar)), "r"(parity)
      : "memory");
  return done != 0;
}

__device__ __forceinline__ void mbar_arrive(uint64_t *mbar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(mbar)) : "memory");
}

// Shared-window (32-bit address) forms: a generic pointer into dynamic shared memory costs a
// generic->shared conversion (three uniform instructions) at every use.
__device__ __forceinline__ void mbar_wait_a(uint32_t addr, uint32_t parity) {
  uint32_t done = 0;
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
__device__ __forceinline__ void mbar_arrive_a(uint32_t addr) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(addr) : "memory"); }
__device__ __forceinline__ void tc_commit_a(uint32_t addr) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ float4 lds_v4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ int lds_i32(uint32_t addr) {
  int v;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }

// W images for k_emis_ws: image i covers global states [img_state0[i], +img_nstates[i]), TN rows (whole
// states; rows beyond are zero), followed by kc2[TN] = log2(e) (ln c - 0.5 (D ln 2pi + ln|det|) - 0.5 sum mu^2 iv),
// -inf for a Gaussian with c == 0 or det == 0 (density 0 in the reference) and for the pad rows.
__global__ void k_pack_w_ws(const double *__restrict__ mu, const double *__restrict__ iv, const float *__restrict__ kc2all,
                            const double *__restrict__ ctr, int M, int MP, int D, int DP, int TN,
                            const int32_t *__restrict__ img_state0, const int32_t *__restrict__ img_nstates,
                            float *__restrict__ images) {
  const int img = blockIdx.y;
  const int KP = 2 * DP;
  pdl_wait();
  const uint32_t P = (uint32_t)(KP / 4) * 128;
  const size_t img_floats = ws_image_bytes(TN, KP) / 4;
  float *hi = images + (size_t)img * img_floats;
  float *lo = hi + (size_t)(TN / 8) * (P / 4);
  float *kc2 = lo + (size_t)(TN / 8) * (P / 4);
  const int64_t s0g = img_state0[img];
  const int nst = img_nstates[img];
  // image row n -> Gaussian index, or -1 for a pad row: chunk n / 16 holds states (n / 16) spc .. of MP columns each
  // (MP <= 16); a state of MP > 16 columns spans MP / 16 chunks
  auto gauss_of = [&](int n) -> int64_t {
    int st, m;
    if (MP > 16) { st = n / MP; m = n - st * MP; }
    else {
      const int spc = 16 / MP, c = n >> 4, w = n & 15;
      if (w >= spc * MP) return -1;
      st = c * spc + w / MP; m = w % MP;
    }
    return (st < nst && m < M) ? (s0g + st) * M + m : -1;
  };
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < TN * KP; idx += gridDim.x * blockDim.x) {
    const int n = idx / KP, k = idx - n * KP;
    const int part = k / DP, d = k - part * DP;
    const int64_t g = gauss_of(n);
    float val = 0.f;
    if (g >= 0 && d < D) {
      const double m = mu[g * D + d] - ctr[d], w = iv[g * D + d];
      val = (float)(part == 0 ? m * w : -0.5 * w);
    }
    float h, l;
    split_tf32(val, h, l);
    const size_t o = ((size_t)(n & 7) * 16 + (k & 3) * 4 + (size_t)(k >> 2) * 128 + (size_t)(n >> 3) * P) / 4;
    hi[o] = h;
    lo[o] = l;
    if (k == 0) kc2[n] = (g >= 0) ? kc2all[g] : kNegInf;
  }
}

// ---- half-precision operands (H16) of the emission kernels: the same contraction with kind::f16 MMAs (twice the TF32 rate) ----
// A TF32 operand keeps 11 significant bits, as a half does; hi + lo of a half split carry the same 22 bits as the 3xTF32
// split -- provided the halves stay inside the half's narrow exponent range.  Every dimension is therefore rescaled by powers
// of two (exact): x' = x / s1_d against W' = mu iv s1_d, and x''^2 = (x / s2_d)^2 against -iv s2_d^2 / 2, with s1_d, s2_d
// chosen so that the two factors of a term have the same magnitude (k_dec16_scales: both at most sqrt(kappa), the accuracy
// guard's bound, so nothing overflows; a lo part below the normal range costs at most 3e-8 times the other factor).
// W image: [hi: (TN/8) P16][lo: (TN/8) P16][kc2: TN floats], P16 = (KP/8) 128: K-major, 16-byte chunks of 8 halves.
__host__ __device__ inline size_t dec16_image_bytes(int TN, int KP) { return (size_t)2 * (TN / 8) * (KP / 8) * 128 + (size_t)TN * 4; }

// sc[0..DP) = 1/s1, [DP..2DP) = 1/s2, [2DP..3DP) = s1, [3DP..4DP) = s2^2   (powers of two; 1 for the pad dimensions)
__global__ void k_dec16_scales(const unsigned long long *__restrict__ ext, const unsigned int *__restrict__ xabs, int D, int DP, float *__restrict__ sc) {
  const int d = threadIdx.x;
  if (d >= DP) return;
  float s1 = 1.f, s2 = 1.f;
  bool dead = false;  // no frame leaves the centre in this dimension: both of its terms are exactly 0 (the constant kc holds the rest)
  if (d < D) {
    const double ivm = __longlong_as_double((long long)ext[d]), mum = __longlong_as_double((long long)ext[DP + d]);
    const double r = xabs ? (double)__uint_as_float(xabs[d]) : mum;
    const double wl = mum * ivm;                                  // largest |mu iv|
    dead = !(r > 0.0);
    if (r > 0.0 && wl > 0.0 && wl < INFINITY) s1 = exp2f(rintf(0.5f * log2f((float)(r / wl))));
    if (r > 0.0 && ivm > 0.0 && ivm < INFINITY) s2 = exp2f(rintf(0.25f * log2f((float)(2.0 * r * r / ivm))));
  }
  sc[d] = dead ? 0.f : 1.f / s1;
  sc[DP + d] = dead ? 0.f : 1.f / s2;
  sc[2 * DP + d] = dead ? 0.f : s1;
  sc[3 * DP + d] = dead ? 0.f : s2 * s2;
}

// two values at once: one packed conversion each way (the scalar conversions run on the quarter-rate unit, and an emission
// kernel that expands its frame tile per unit -- k_emis_ws -- was bound by them: C5 decode 21.0 -> 27.1 ms)
__device__ __forceinline__ void split_half2(float a, float b, uint32_t &hi, uint32_t &lo) {
  const __half2 h = __floats2half2_rn(a, b);  // low half = a, high half = b
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
  hi = *reinterpret_cast<const uint32_t *>(&h);
  lo = *reinterpret_cast<const uint32_t *>(&l);
}
__device__ __forceinline__ void split_half(float v, unsigned short &hi, unsigned short &lo) {
  const __half h = __float2half_rn(v);
  hi = __half_as_ushort(h);
  lo = __half_as_ushort(__float2half_rn(v - __half2float(h)));
}

// as k_pack_w_ws, for the half-precision images (column layout of the states, pad columns and kc2 are the same)
__global__ void k_pack_w_dec16(const double *__restrict__ mu, const double *__restrict__ iv, const float *__restrict__ kc2all,
                               const double *__restrict__ ctr, const float *__restrict__ sc, int M, int MP, int D, int DP, int TN,
                               const int32_t *__restrict__ img_state0, const int32_t *__restrict__ img_nstates,
                               unsigned char *__restrict__ images) {
  const int img = blockIdx.y;
  const int KP = 2 * DP;
  const uint32_t P = (uint32_t)(KP / 8) * 128;
  unsigned char *hi = images + (size_t)img * dec16_image_bytes(TN, KP);
  unsigned char *lo = hi + (size_t)(TN / 8) * P;
  float *kc2 = reinterpret_cast<float *>(lo + (size_t)(TN / 8) * P);
  const int64_t s0g = img_state0[img];
  const int nst = img_nstates[img];
  auto gauss_of = [&](int n) -> int64_t {
    int st, m;
    if (MP > 16) { st = n / MP; m = n - st * MP; }
    else {
      const int spc = 16 / MP, c = n >> 4, w = n & 15;
      if (w >= spc * MP) return -1;
      st = c * spc + w / MP; m = w % MP;
    }
    return (st < nst && m < M) ? (s0g + st) * M + m : -1;
  };
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < TN * KP; idx += gridDim.x * blockDim.x) {
    const int n = idx / KP, k = idx - n * KP;
    const int part = k / DP, d = k - part * DP;
    const int64_t g = gauss_of(n);
    float val = 0.f;
    if (g >= 0 && d < D) {
      const double m = mu[g * D + d] - ctr[d], w = iv[g * D + d];
      val = (float)(part == 0 ? m * w * (double)sc[2 * DP + d] : -0.5 * w * (double)sc[3 * DP + d]);
    }
    unsigned short h, l;
    split_half(val, h, l);
    const size_t o = (size_t)(n & 7) * 16 + (size_t)(k & 7) * 2 + (size_t)(k >> 3) * 128 + (size_t)(n >> 3) * P;
    *reinterpret_cast<unsigned short *>(hi + o) = h;
    *reinterpret_cast<unsigned short *>(lo + o) = l;
    if (k == 0) kc2[n] = (g >= 0) ? kc2all[g] : kNegInf;
  }
}

__device__ __forceinline__ uint32_t make_idesc_f16(int M, int N) {
  // c_format F32 (1) @4, a_format F16 (0) @7, b_format F16 (0) @10, K-major A and B, N>>3 @17, M>>4 @24
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void tc_mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// units == nullptr: decode, unit u = (image u / ntiles_dec, frames [128 (u % ntiles_dec), ...) of the batch, nframes_dec in all)
// MP: padded mixtures per state when <= 16 (1, 2, 4, 8, 16); 0 = a multiple of 16 given at run time (M)
// Warps: 0-7 epilogue (lane quarter w & 3; column groups of parity w >> 2), 8-15 loaders (lane quarter w & 3;
// chunks 0-2 / 3-4 of the doubled row), 16 MMA issuer.
// MR: mixtures of a state that are real (MR <= MP; the others are pad columns the log-sum-exp may skip), 0 = all MP
// H16: half-precision operands (images of k_pack_w_dec16, `scales` of k_dec16_scales; DP a multiple of 8)
template <bool TRAIN, int MP, int MR = 0, bool H16 = false>
__global__ void __launch_bounds__(kWsThreads, 1)
k_emis_ws(const TcTile *__restrict__ units, int nunits, int ntiles_dec, int nframes_dec, const int32_t *__restrict__ frame_ids,
          const float *__restrict__ x32, const float *__restrict__ images, int N, int M, int DP, int TN, float *__restrict__ logb,
          int64_t fbase, int64_t ldb, int S_total, int SCt, const float *__restrict__ scales = nullptr) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const int KP = 2 * DP, NSLAB = H16 ? KP / 16 : KP / 8;  // K per MMA: 16 halves / 8 TF32 (8 tensor-memory columns, 256 bytes of a W row group)
  const uint32_t P = H16 ? (uint32_t)(KP / 8) * 128 : (uint32_t)(KP / 4) * 128;
  const uint32_t w_bytes = 2 * (uint32_t)(TN / 8) * P, img_bytes = w_bytes + (uint32_t)TN * 4;
  const uint32_t Ws = (smem_u32(smem_raw) + 1023u) & ~1023u;  // [hi | lo], shared-window address
  __shared__ float ssc[2][40];  // H16: 1 / s1_d, 1 / s2_d
  if (H16) {
    for (int d = threadIdx.x; d < 80; d += kWsThreads) ssc[d / 40][d % 40] = (d % 40 < DP) ? scales[(d / 40) * DP + d % 40] : 1.f;
  }
  const uint32_t bars = Ws + w_bytes;
  const uint32_t full = bars, empty = bars + 16, dfull = bars + 32, dempty = bars + 48, tmem_slot = bars + 64;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    auto init = [](uint32_t addr, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(addr), "r"(count) : "memory"); };
    for (int s = 0; s < 2; s++) {
      init(full + 8 * s, 256);    // every loader thread arrives
      init(empty + 8 * s, 1);     // tcgen05.commit
      init(dfull + 8 * s, 1);     // tcgen05.commit
      init(dempty + 8 * s, kWsEpiWarps * 32);  // every epilogue thread arrives
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kWsEpiWarps + 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem0 = (uint32_t)lds_i32(tmem_slot);
  pdl_trigger();  // this CTA's work is a fixed unit range: nothing is left to claim
  // TMEM columns: AST operand stages of 160 [x_hi | x2_hi | x_lo | x2_lo], then two accumulator stages of ACS.
  // Images wider than 96 columns (one state of up to 176 mixtures) leave room for a single operand stage.
  const int AST = TN > 96 ? 1 : 2;
  const uint32_t ACS = TN > 96 ? (uint32_t)TN : 96u, acc0 = (uint32_t)AST * 160;
  __shared__ __align__(16) float skc[2][kWsMaxTN1];  // kc2 of the image the epilogue works on (two slots: image switches alternate)
  __shared__ float2 xch[2][4][32][kWsXch];  // partial (max, sum) of the odd chunks' warp, per unit parity / quarter / lane / state

  const int per = (nunits + gridDim.x - 1) / gridDim.x;
  const int u_begin = blockIdx.x * per, u_end = min(nunits, u_begin + per);
  auto get_unit = [&](int ui) -> TcTile {
    if (TRAIN) return units[ui];
    const int img = ui / ntiles_dec, t = ui - img * ntiles_dec;
    return TcTile{t * kTcRows, min(kTcRows, nframes_dec - t * kTcRows), img, img * SCt, 0, 0};
  };
  auto unit_at = [&](int ui) -> TcTile { return ui < u_end ? get_unit(ui) : TcTile{0, 0, -1, 0, 0, 0}; };

  if (warp >= kWsEpiWarps && warp < kWsEpiWarps + 8) {
    // =================================== LOADERS ===================================
    const int q = warp & 3, h = (warp - kWsEpiWarps) >> 2;
    const int r = 32 * q + lane;  // frame row of the tile = TMEM lane
    constexpr int kQ = H16 ? 6 : 5;  // float4 per thread: half a row (DP <= 40); halves go in groups of 8 dimensions: 24 + 16
    const int nq = DP / 4;
    const int j0 = h * kQ;        // this thread expands float4 [j0, j0 + kQ) of the row: x -> columns 4j.., x^2 -> columns DP + 4j..
    // Global loads run three levels ahead of the expansion so that no latency is exposed per unit:
    // unit descriptor (i+3) -> frame id (i+2) -> feature row (i+1), while unit i is split and stored.
    auto frame_of = [&](const TcTile &u) -> int64_t {
      if (r >= u.nrows) return -1;
      return TRAIN ? (int64_t)__ldg(frame_ids + u.row0 + r) : fbase + u.row0 + r;
    };
    auto load_row = [&](int64_t f, float4 (&xv)[kQ]) {
      const float4 *src = reinterpret_cast<const float4 *>(x32 + (f < 0 ? 0 : f) * DP) + j0;
#pragma unroll
      for (int j = 0; j < kQ; j++) xv[j] = (f >= 0 && j0 + j < nq) ? __ldg(src + j) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    const uint32_t xa0 = tmem0 + ((uint32_t)(32 * q) << 16);  // my lane
    int cur_img = -1;
    auto split4 = [](const float4 &v, uint32_t (&hi)[4], uint32_t (&lo)[4]) {
      float hh, ll;
      split_tf32_fast(v.x, hh, ll); hi[0] = __float_as_uint(hh); lo[0] = __float_as_uint(ll);
      split_tf32_fast(v.y, hh, ll); hi[1] = __float_as_uint(hh); lo[1] = __float_as_uint(ll);
      split_tf32_fast(v.z, hh, ll); hi[2] = __float_as_uint(hh); lo[2] = __float_as_uint(ll);
      split_tf32_fast(v.w, hh, ll); hi[3] = __float_as_uint(hh); lo[3] = __float_as_uint(ll);
    };
    auto expand = [&](int i, const TcTile &unit, const float4 (&xv)[kQ]) {
      const int s = i % AST, ku = i / AST;  // operand stage and its use count
      if (unit.img != cur_img) {
        // the tensor pipe may still be reading the old image: wait for the previous unit's MMAs
        if (i >= 1) mbar_wait_a(empty + 8 * ((i - 1) % AST), ((i - 1) / AST) & 1);
        const float4 *wsrc = reinterpret_cast<const float4 *>(images + (size_t)unit.img * (img_bytes / 4));
        for (int k = tid - kWsEpiWarps * 32; k < (int)(w_bytes / 16); k += 256) st_shared_v4(Ws + 16 * k, __ldg(wsrc + k));
        cur_img = unit.img;
      }
      mbar_wait_a(empty + 8 * s, (ku & 1) ^ 1);  // operand stage s is free (unit i-AST has been multiplied)
      tc_fence_after();
      // stage s: [x_hi (DP) | x2_hi (DP) | x_lo (DP) | x2_lo (DP)], 4 columns per store
      if (H16) {
        // stage s: [x' hi | x''^2 hi | x' lo | x''^2 lo], DP / 2 columns (two halves each) per block; 8 dimensions per store
        const uint32_t xs = xa0 + (uint32_t)s * 160;
        const int hb = DP / 2;
#pragma unroll
        for (int j = 0; j < kQ; j += 2) {
          if (j0 + j < nq) {
            const float v[8] = {xv[j].x, xv[j].y, xv[j].z, xv[j].w, xv[j + 1].x, xv[j + 1].y, xv[j + 1].z, xv[j + 1].w};
            uint32_t ah[4], al[4], qh[4], ql[4];
#pragma unroll
            for (int e = 0; e < 4; e++) {
              const int d0 = 4 * (j0 + j) + 2 * e;
              split_half2(v[2 * e] * ssc[0][d0], v[2 * e + 1] * ssc[0][d0 + 1], ah[e], al[e]);
              const float s0 = v[2 * e] * ssc[1][d0], s1 = v[2 * e + 1] * ssc[1][d0 + 1];
              split_half2(s0 * s0, s1 * s1, qh[e], ql[e]);
            }
            const uint32_t c0 = 2 * (j0 + j);
            tmem_st4(xs + c0, ah);
            tmem_st4(xs + hb + c0, qh);
            tmem_st4(xs + 2 * hb + c0, al);
            tmem_st4(xs + 3 * hb + c0, ql);
          }
        }
      } else {
      const uint32_t xa = xa0 + (uint32_t)s * 160 + 4 * j0;
#pragma unroll
      for (int j = 0; j < kQ; j++) {
        if (j0 + j < nq) {
          const float4 t = xv[j];
          uint32_t vh[4], vl[4];
          split4(t, vh, vl);
          tmem_st4(xa + 4 * j, vh);
          tmem_st4(xa + 80 + 4 * j, vl);
          split4(make_float4(t.x * t.x, t.y * t.y, t.z * t.z, t.w * t.w), vh, vl);
          tmem_st4(xa + DP + 4 * j, vh);
          tmem_st4(xa + 80 + DP + 4 * j, vl);
        }
      }
      }
      tmem_wait_st();
      tc_fence_before();
      fence_async_smem();  // the W image (generic-proxy writes) -> visible to the tensor core
      mbar_arrive_a(full + 8 * s);
    };
    TcTile d0 = unit_at(u_begin), d1 = unit_at(u_begin + 1), d2 = unit_at(u_begin + 2);
    int64_t f1 = frame_of(d1);
    float4 xa_[kQ], xb_[kQ];
    load_row(frame_of(d0), xa_);
    for (int ui = u_begin, i = 0; ui < u_end; ui += 2, i += 2) {  // two units per trip: the row buffers swap roles
      load_row(f1, xb_);                     // rows of unit i+1
      int64_t f2 = frame_of(d2);             // frame id of unit i+2
      TcTile d3 = unit_at(ui + 3);           // descriptor of unit i+3
      expand(i, d0, xa_);
      if (ui + 1 < u_end) {
        load_row(f2, xa_);                   // rows of unit i+2
        f1 = frame_of(d3);                   // frame id of unit i+3
        const TcTile d4 = unit_at(ui + 4);
        expand(i + 1, d1, xb_);
        d0 = d2; d1 = d3; d2 = d4;
      }
    }
  } else if (warp == kWsEpiWarps + 8) {
    // =================================== MMA ISSUER ===================================
    const uint32_t idesc = H16 ? make_idesc_f16(kTcRows, TN) : make_idesc_tf32(kTcRows, TN);
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem0, 0);
    for (int ui = u_begin, i = 0; ui < u_end; ui++, i++) {
      const int s = i & 1, sa = i % AST;
      const uint32_t ph = (i >> 1) & 1;
      mbar_wait_a(full + 8 * sa, (i / AST) & 1);  // operands landed
      mbar_wait_a(dempty + 8 * s, ph ^ 1);    // accumulator stage drained by the epilogue (unit i-2)
      tc_fence_after();
      if (elect_one_sync()) {
        const uint32_t xh = tb + (uint32_t)sa * 160, xl = xh + (H16 ? (uint32_t)DP : 80u);
        const uint64_t wh = make_smem_desc2(Ws, 128, P), wl = make_smem_desc2(Ws + (uint32_t)(TN / 8) * P, 128, P);
        const uint32_t d = tb + acc0 + (uint32_t)s * ACS;
        if (H16) {
          uint32_t acc = 0;
          for (int p = 0; p < 3; p++) {  // Xh*Wh, Xl*Wh, Xh*Wl
            const uint32_t a0 = (p == 1) ? xl : xh;
            const uint64_t b0 = (p == 2) ? wl : wh;
#pragma unroll 5
            for (int j = 0; j < NSLAB; j++) {
              tc_mma_f16_ts(d, a0 + j * 8, b0 + (uint64_t)(j * 16), idesc, acc);
              acc = 1;
            }
          }
        } else if (NSLAB == 10) {  // D = 39: fully unrolled
#pragma unroll
          for (int j = 0; j < 10; j++) tc_mma_tf32_ts(d, xh + j * 8, wh + (uint64_t)(j * 16), idesc, j > 0);  // Xh*Wh
#pragma unroll
          for (int j = 0; j < 10; j++) tc_mma_tf32_ts(d, xl + j * 8, wh + (uint64_t)(j * 16), idesc, 1);      // Xl*Wh
#pragma unroll
          for (int j = 0; j < 10; j++) tc_mma_tf32_ts(d, xh + j * 8, wl + (uint64_t)(j * 16), idesc, 1);      // Xh*Wl
        } else {
          uint32_t acc = 0;
          for (int p = 0; p < 3; p++) {  // Xh*Wh, Xl*Wh, Xh*Wl
            const uint32_t a0 = (p == 1) ? xl : xh;
            const uint64_t b0 = (p == 2) ? wl : wh;
            for (int j = 0; j < NSLAB; j++) {
              tc_mma_tf32_ts(d, a0 + j * 8, b0 + (uint64_t)(j * 16), idesc, acc);  // +256 B per K-step, in 16-byte units
              acc = 1;
            }
          }
        }
        tc_commit_a(empty + 8 * sa);  // operand stage (and, for the loaders' image switch, W) free when these MMAs retire
        tc_commit_a(dfull + 8 * s);   // accumulator ready
      }
      __syncwarp();
    }
  } else {
    // =================================== EPILOGUE (warps 0 .. kWsEpiWarps-1) ===================================
    constexpr int EH = kWsEpiWarps / 4;  // warps per TMEM lane quarter: column groups g with g % EH == h
    const int q = warp & 3, h = warp >> 2;
    const int row = 32 * q + lane;  // TMEM lane
    const uint32_t trow = (uint32_t)(32 * q) << 16;
    // unit descriptors two ahead and the frame id one ahead, so that no global-memory latency sits
    // between the accumulator becoming ready and its reduction
    auto frame_of = [&](const TcTile &u) -> int64_t {
      if (row >= u.nrows) return 0;
      return TRAIN ? (int64_t)__ldg(frame_ids + u.row0 + row) : fbase + u.row0 + row;
    };
    TcTile un0 = unit_at(u_begin), un1 = unit_at(u_begin + 1);
    int64_t fcur = frame_of(un0);
    const int mp = MP ? MP : M;               // M here is the padded count
    const int cpg = MP ? 1 : mp / 16;         // chunks per group: a chunk of 16/MP whole states, or one state of M/16 chunks
    const int spg = MP ? 16 / (MP ? MP : 16) : 1;  // states per group (16 % MP pad columns close a chunk)
    int epi_img = -1, nsw = 0;
    for (int ui = u_begin, i = 0; ui < u_end; ui++, i++) {
      const TcTile unit = un0;
      if (unit.img != epi_img) {
        // The additive constants of a new image go to shared memory once (global loads of them in every unit sat on
        // the critical path: the L1 lines do not survive the feature and image streams).  All eight epilogue warps
        // walk the units in the same order, so they meet here; two slots, so nobody overwrites what a slower warp
        // still reads.
        epi_img = unit.img;
        const float *kcg = images + (size_t)unit.img * (img_bytes / 4) + w_bytes / 4;
        for (int c = tid; c < TN; c += kWsEpiWarps * 32) skc[nsw & 1][c] = __ldg(kcg + c);
        asm volatile("bar.sync 9, %0;" ::"n"(kWsEpiWarps * 32) : "memory");
        nsw++;
      }
      const float *kcs = skc[(nsw - 1) & 1];
      const int64_t f = fcur;
      const int64_t fnext = frame_of(un1);
      const TcTile un2 = unit_at(ui + 2);
      const int s = i & 1;
      mbar_wait_a(dfull + 8 * s, (i >> 1) & 1);
      tc_fence_after();
      const int st_lim = TRAIN ? N : S_total;
      const int nst = max(0, min(SCt, st_lim - unit.state0));  // states present in this image
      const int ngroups = (nst + spg - 1) / spg;
      const bool live = row < unit.nrows;
      float *lrow = TRAIN ? logb + f * N + unit.state0 : logb + (f - fbase) * ldb + unit.state0;
      const uint32_t d = tmem0 + acc0 + (uint32_t)s * ACS + trow;
      const float4 *kc4 = reinterpret_cast<const float4 *>(kcs);  // warp-uniform addresses: broadcast loads
      constexpr int kMaxG = (kWsMaxTN / 16 + EH - 1) / EH;  // groups per warp when a group is one chunk
      if (MP) {
        // my groups: g = h, h + EH, ...; every accumulator chunk of mine in flight at once
        uint32_t v[kMaxG][16];
#pragma unroll
        for (int k = 0; k < kMaxG; k++)
          if (h + EH * k < ngroups) tmem_ld16_nowait(d + (h + EH * k) * 16, v[k]);
        tmem_wait_ld();
#pragma unroll
        for (int k = 0; k < kMaxG; k++) {
          const int c = h + EH * k;
          if (c < ngroups) {
            const float4 k0 = kc4[c * 4], k1 = kc4[c * 4 + 1], k2 = kc4[c * 4 + 2], k3 = kc4[c * 4 + 3];
            const float kc[16] = {k0.x, k0.y, k0.z, k0.w, k1.x, k1.y, k1.z, k1.w, k2.x, k2.y, k2.z, k2.w, k3.x, k3.y, k3.z, k3.w};
            float val[16];  // log2(c_g N_g(x)); -inf for a Gaussian of density 0 and for the pad columns
#pragma unroll
            for (int j = 0; j < 16; j++) val[j] = fmaf(__uint_as_float(v[k][j]), 1.4426950408889634f, kc[j]);
            constexpr int SPC = 16 / (MP ? MP : 16);  // whole states in this chunk, each reduced independently
            float lbv[SPC];
#pragma unroll
            for (int g = 0; g < SPC; g++) {
              constexpr int MU = MR ? MR : MP;  // columns MU .. MP-1 of a state are pad (density 0)
              float m = val[g * MP];
#pragma unroll
              for (int j = 1; j < MU; j++) m = fmaxf(m, val[g * MP + j]);
              const float ms = (m > kNegInf) ? m : 0.f;
              float sm_;
              // The largest term of the sum is 2^0 = 1: with up to three mixtures it is cheaper to order the values
              // (min / max on the ALU) than to send that term through the SFU as well -- the epilogue of the
              // small-mixture decode regime is bound by its MUFU operations (C4: M = 3, 4 -> 3 per state).
              if (MU == 1) {
                sm_ = 1.f;
              } else if (MU == 2) {
                sm_ = 1.f + ex2_approx(fminf(val[g * MP], val[g * MP + 1]) - ms);
              } else if (MU == 3) {
                const float a = val[g * MP], b = val[g * MP + 1], c3 = val[g * MP + 2];
                const float lo = fminf(fminf(a, b), c3), mid = fmaxf(fminf(a, b), fminf(fmaxf(a, b), c3));
                sm_ = 1.f + (ex2_approx(mid - ms) + ex2_approx(lo - ms));
              } else {
                sm_ = 0.f;
#pragma unroll
                for (int j = 0; j < MU; j++) sm_ += ex2_approx(val[g * MP + j] - ms);
              }
              lbv[g] = (m > kNegInf) ? (MU == 1 ? ms : ms + __log2f(sm_)) * 0.6931471805599453f : kNegInf;
            }
            // the chunk's states are contiguous in the output row: 16- / 8-byte stores when the row allows it (a lane
            // per frame makes every 4-byte store its own memory transaction)
            float *dst = lrow + c * SPC;
            if (live) {
              if (SPC % 4 == 0 && c * SPC + SPC <= nst && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
                for (int g = 0; g + 3 < SPC; g += 4) *reinterpret_cast<float4 *>(dst + g) = make_float4(lbv[g], lbv[g + 1], lbv[g + 2], lbv[g + 3]);
              } else if (SPC % 2 == 0 && c * SPC + SPC <= nst && (reinterpret_cast<uintptr_t>(dst) & 7) == 0) {
#pragma unroll
                for (int g = 0; g + 1 < SPC; g += 2) *reinterpret_cast<float2 *>(dst + g) = make_float2(lbv[g], lbv[g + 1]);
              } else {
#pragma unroll
                for (int g = 0; g < SPC; g++)
                  if (c * SPC + g < nst) dst[g] = lbv[g];
              }
            }
          }
        }
      } else {
        // One state spans cpg chunks.  The two warps of a lane quarter take the even / the odd chunks of every
        // state (online log-sum-exp over their own chunks); the odd warp hands its partial (max, sum) over
        // through shared memory and the even warp merges and stores.
        float pmx[kWsXch], psum[kWsXch];
        if (h < 2) {
#pragma unroll
        for (int sx = 0; sx < kWsXch; sx++) {
          pmx[sx] = kNegInf; psum[sx] = 0.f;
          if (sx < nst) {
            float mx = kNegInf, sum = 0.f;
            for (int cc = h; cc < cpg; cc += 2) {
              const int c = sx * cpg + cc;
              uint32_t v[16];
              tmem_ld16(d + c * 16, v);
              const float4 k0 = kc4[c * 4], k1 = kc4[c * 4 + 1], k2 = kc4[c * 4 + 2], k3 = kc4[c * 4 + 3];
              const float kc[16] = {k0.x, k0.y, k0.z, k0.w, k1.x, k1.y, k1.z, k1.w, k2.x, k2.y, k2.z, k2.w, k3.x, k3.y, k3.z, k3.w};
              float val[16];
#pragma unroll
              for (int j = 0; j < 16; j++) val[j] = fmaf(__uint_as_float(v[j]), 1.4426950408889634f, kc[j]);
              float m = val[0];
#pragma unroll
              for (int j = 1; j < 16; j++) m = fmaxf(m, val[j]);
              const float mn = fmaxf(mx, m);
              const float ms = (mn > kNegInf) ? mn : 0.f;
              float sm_ = 0.f;
#pragma unroll
              for (int j = 0; j < 16; j++) sm_ += ex2_approx(val[j] - ms);
              sum = fmaf(sum, ex2_approx(((mx > kNegInf) ? mx : ms) - ms), sm_);
              mx = mn;
            }
            pmx[sx] = mx; psum[sx] = sum;
          }
        }
        }
        if (h == 1) {
#pragma unroll
          for (int sx = 0; sx < kWsXch; sx++)
            if (sx < nst) xch[i & 1][q][lane][sx] = make_float2(pmx[sx], psum[sx]);
          // (bar.sync, not bar.arrive: this warp can be a whole unit ahead of its partner, and two arrivals of
          // the same warp would complete a barrier phase on their own)
          asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
        } else if (h == 0) {
          asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
#pragma unroll
          for (int sx = 0; sx < kWsXch; sx++) {
            if (sx < nst) {
              const float2 o = xch[i & 1][q][lane][sx];
              const float mn = fmaxf(pmx[sx], o.x);
              const float ms = (mn > kNegInf) ? mn : 0.f;
              const float sum = psum[sx] * ex2_approx(((pmx[sx] > kNegInf) ? pmx[sx] : ms) - ms) + o.y * ex2_approx(((o.x > kNegInf) ? o.x : ms) - ms);
              const float lb = (mn > kNegInf) ? (mn + __log2f(sum)) * 0.6931471805599453f : kNegInf;
              if (live) lrow[sx] = lb;
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive_a(dempty + 8 * s);
      un0 = un1; un1 = un2; fcur = fnext;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == kWsEpiWarps + 8) tmem_dealloc(tmem0, 512);
}


// ================================================================================================
// k_accum_ws: mixture accumulators (calc_mix_param, T-FS:1691-1727), warp-specialised and pipelined.
// Same mathematics as k_accum_tc (tc_kernels.cuh): per sub-tile of 32 frames of one model and block of
// 128 Gaussians
//   GEMM1  L[g][f]  = sum_k W[g][k] Xaug[f][k]           A = W (TMEM, parked per image), B = X  (smem)
//   w[g][f] = gamma_f(s(g)) exp(L + kc[g] - logb_f(s(g)))  epilogue, in place in TMEM (hi) + beside it (lo)
//   GEMM2  S[g][k] += sum_f w[g][f] Xaug[f][k]           A = w (TMEM), B = XT (smem)
// but the activities run concurrently on different warps and meet only at mbarriers (20 warps):
//   warps  8-12 X LOADERS   features three levels ahead in registers; X (frames x columns), TF32 hi / lo,
//                           and the per-frame weight exponents cfs
//   warps 13-17 XT LOADERS  the same tile transposed (columns x frames), TF32 hi / lo
//   warp  18    GEMM1 MMA   issues GEMM1 of the next unit as soon as its X tile (and the image's W) is there
//   warp  19    GEMM2 MMA   issues GEMM2 of the oldest unit as soon as its weights are there; two issuers
//                           because one warp's instruction stream serialised the whole pipeline
//   warps  0-7  EPILOGUE    L -> w with tcgen05.ld / tcgen05.st (warp w: TMEM lanes 32 (w%4).., frames
//                           16 (w/4)..); every kAccDrain sub-tiles S moves from TMEM (FP32, truncating
//                           accumulation) to FP32 in shared memory (round to nearest); when the CTA's (model,
//                           Gaussian block) changes, the partial sums go to the CTA's scratch slot (plain
//                           stores; k_finalize_slots adds the slots in a fixed order); loads the next image's
//                           W into TMEM
// Four shared-memory stages (X, XT, cfs) and four TMEM stages (L / w_hi, w_lo): with two, the GEMMs of one unit
// and the expansion / weight epilogue of the next alternated instead of overlapping (tensor pipe active < 30 %).
// TMEM columns: [0,128) L / w_hi x4 | [128,256) w_lo x4 | [256, 256+KP2) S | [352, 352+2KP) W_hi, W_lo
// Shared-memory layouts (SWIZZLE_NONE K-major, 16-byte chunks):
//   X  : byte(f, k) = (f%8)*16 + (k%4)*4 + (k/4)*128 + (f/8)*PX     PX = (KP/4)*128   (4 frame groups)
//   XT : byte(k, f) = (k%8)*16 + (f%4)*4 + (f/4)*128 + (k/8)*1024   (KP2/8 column groups)
// ================================================================================================
constexpr int kAccSub = 32;        // frames per sub-tile
constexpr int kAccStages = 4;      // sub-tiles in flight (shared-memory and TMEM stages)
constexpr int kAccDrain = 16;      // sub-tiles accumulated in TMEM before S moves out (512 frames)
constexpr int kAccLdWarps = 5;     // warps per loader role (X, XT)
constexpr int kAccG1Warp = 8 + 2 * kAccLdWarps;  // GEMM1 issuer; the GEMM2 issuer is the next warp
constexpr int kAccWsThreads = (kAccG1Warp + 2) * 32;  // 20 warps
constexpr int kAccSlots = 2;        // scratch slots per CTA for the partial sums of its first images
constexpr int kAccImgCap = 2048;   // unit -> image ids of this CTA's range cached in shared memory

// one stage: X hi | X lo (4 frame groups x PX) | XT hi | XT lo (KP2/8 column groups x 1024) | cfs[8][32]
__host__ __device__ inline size_t ws_acc_stage_bytes(int KP) {
  return (size_t)2 * (kAccSub / 8) * (KP / 4) * 128 + (size_t)2 * (tc_kp2(KP) / 8) * (kAccSub / 4) * 128 + kAccSub * 8 * 4;
}
// stages | barriers (256 B) | image ids | S accumulator [KP2][128] floats | 1 KB alignment slack
__host__ __device__ inline size_t ws_acc_smem_bytes(int KP) {
  return kAccStages * ws_acc_stage_bytes(KP) + 1024 + 256 + kAccImgCap * 4 + (size_t)tc_kp2(KP) * 128 * 4;
}

__global__ void __launch_bounds__(kAccWsThreads, 1)
k_accum_ws(const TcTile *__restrict__ units, int nunits, const int32_t *__restrict__ frame_ids, const float *__restrict__ x32,
           const float *__restrict__ images, const float *__restrict__ kcT, const float *__restrict__ logb,
           const float *__restrict__ gamma, int N, int M, int G, int D, int DP, double *__restrict__ stats,
           int64_t stats_stride, int64_t off_S0, int64_t off_S1, int64_t off_S2, float *__restrict__ scratch) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr int NST = kAccStages, SUB = kAccSub;
  const int KP = 2 * DP, KP2 = tc_kp2(KP), NSLAB = KP / 8, nq = DP / 4;
  const uint32_t PX = (uint32_t)(KP / 4) * 128;            // X: bytes per group of 8 frames
  constexpr uint32_t PT = (SUB / 4) * 128;                 // XT: bytes per group of 8 columns
  const uint32_t x_bytes = (SUB / 8) * PX, xt_bytes = (uint32_t)(KP2 / 8) * PT;
  const uint32_t cfs_off = 2 * x_bytes + 2 * xt_bytes;
  const uint32_t stage_bytes = cfs_off + SUB * 8 * 4;
  // everything in shared memory is addressed through the 32-bit shared window
  const uint32_t sm0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = sm0 + NST * stage_bytes;
  const uint32_t x_full = bars, x_free = bars + 8 * NST, d1_full = bars + 16 * NST, w_full = bars + 24 * NST, s_full = bars + 32 * NST,
                 s_free = s_full + 8, wimg_full = s_full + 16, tmem_slot = s_full + 24;
  const uint32_t simg = bars + 256;                        // int32 [kAccImgCap]
  const uint32_t sacc = simg + kAccImgCap * 4;             // float [KP2][128]: S per (column, Gaussian lane)
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int per = (nunits + gridDim.x - 1) / gridDim.x;
  const int u_begin = blockIdx.x * per, u_end = min(nunits, u_begin + per);
  const int n_my = max(0, u_end - u_begin);
  // The MMA issuers and the epilogue look at image boundaries several times per unit; the ids are staged once.
  for (int k = tid; k < min(n_my, kAccImgCap); k += kAccWsThreads)
    asm volatile("st.shared.s32 [%0], %1;" ::"r"(simg + 4 * k), "r"(__ldg(&units[u_begin + k].img)) : "memory");
  for (int k = tid; k < KP2 * 128; k += kAccWsThreads) sts_f32(sacc + 4 * k, 0.f);

  if (tid == 0) {
    auto init = [](uint32_t addr, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(addr), "r"(count) : "memory"); };
    for (int s = 0; s < NST; s++) {
      init(x_full + 8 * s, 2 * kAccLdWarps * 32);   // X and XT loaders
      init(x_free + 8 * s, 1);     // tcgen05.commit after GEMM2
      init(d1_full + 8 * s, 1);    // tcgen05.commit after GEMM1
      init(w_full + 8 * s, 256);   // epilogue threads
    }
    init(s_full, 1);
    init(s_free, 256);
    init(wimg_full, 256);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kAccG1Warp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem0 = (uint32_t)lds_i32(tmem_slot);

  auto img_at = [&](int ui) -> int {
    if (ui < u_begin || ui >= u_end) return -1;
    return (ui - u_begin < kAccImgCap) ? lds_i32(simg + 4 * (ui - u_begin)) : __ldg(&units[ui].img);
  };

  if (warp >= 8 && warp < 8 + kAccLdWarps) {
    // =================================== X LOADERS ===================================
    // thread <-> (frame row xr, column part): float4 [xq0, xq1) of the row, and the weight exponents of
    // states part, part + NPART of that frame.  Global loads run ahead of the expansion: unit descriptor
    // (i+3) -> frame id (i+2) -> operands (i+1), while unit i is split and stored.
    const int t = tid - 256;
    constexpr int NPART = kAccLdWarps * 32 / SUB;            // 5
    const int xr = t & (SUB - 1), part = t / SUB;
    const int qper = (nq + NPART - 1) / NPART;
    const int xq0 = min(nq, part * qper), xq1 = min(nq, xq0 + qper);  // float4 [xq0, xq1)
    constexpr int kXQ = (10 + NPART - 1) / NPART;            // DP <= 40
    constexpr int kCS = (8 + NPART - 1) / NPART;             // states per thread
    struct Pre { float4 x[kXQ]; float gm[kCS], lb[kCS]; };
    auto desc_at = [&](int ui) -> int2 { return ui < u_end ? __ldg(reinterpret_cast<const int2 *>(units + ui)) : make_int2(0, 0); };  // (row0, nrows)
    auto fid_of = [&](const int2 &u) -> int { return (xr < u.y) ? __ldg(frame_ids + u.x + xr) : -1; };
    auto load_pre = [&](int f, Pre &p) {
      const float4 *src = reinterpret_cast<const float4 *>(x32 + (int64_t)(f < 0 ? 0 : f) * DP);
#pragma unroll
      for (int j = 0; j < kXQ; j++) p.x[j] = (f >= 0 && xq0 + j < xq1) ? __ldg(src + xq0 + j) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int c = 0; c < kCS; c++) {
        const int st = part + c * NPART;
        const bool ok = f >= 0 && st < N;
        p.gm[c] = ok ? __ldg(gamma + (int64_t)f * N + st) : 0.f;
        p.lb[c] = ok ? __ldg(logb + (int64_t)f * N + st) : 0.f;
      }
    };
    const uint32_t rbase = (uint32_t)(xr & 7) * 16 + (uint32_t)(xr >> 3) * PX;
    auto expand = [&](int i, const Pre &cur) {
      const int s = i % NST;
      mbar_wait_a(x_free + 8 * s, ((i / NST) & 1) ^ 1);  // stage s: GEMM2 of unit i-NST has retired
      const uint32_t Xh = sm0 + (uint32_t)s * stage_bytes, Xl = Xh + x_bytes;
#pragma unroll
      for (int j = 0; j < kXQ; j++) {
        if (xq0 + j < xq1) {
          const float4 xx = cur.x[j];
          float4 h, l;
          split_tf32_fast(xx.x, h.x, l.x); split_tf32_fast(xx.y, h.y, l.y); split_tf32_fast(xx.z, h.z, l.z); split_tf32_fast(xx.w, h.w, l.w);
          uint32_t o = rbase + (uint32_t)(xq0 + j) * 128;
          st_shared_v4(Xh + o, h);
          st_shared_v4(Xl + o, l);
          split_tf32_fast(xx.x * xx.x, h.x, l.x); split_tf32_fast(xx.y * xx.y, h.y, l.y);
          split_tf32_fast(xx.z * xx.z, h.z, l.z); split_tf32_fast(xx.w * xx.w, h.w, l.w);
          o += (uint32_t)nq * 128;
          st_shared_v4(Xh + o, h);
          st_shared_v4(Xl + o, l);
        }
      }
      // weight exponent of frame xr per state: log2(gamma) - logb log2(e); -inf = no weight.  cfs[state][frame]
      const uint32_t cfs = Xh + cfs_off + 4 * xr;
#pragma unroll
      for (int c = 0; c < kCS; c++) {
        const int st = part + c * NPART;
        if (st < 8) {
          float cf = kNegInf;
          if (cur.gm[c] > 0.f && cur.lb[c] > kNegInf) cf = __log2f(cur.gm[c]) - cur.lb[c] * 1.4426950408889634f;
          sts_f32(cfs + st * SUB * 4, cf);
        }
      }
      fence_async_smem();
      mbar_arrive_a(x_full + 8 * s);
    };
    int2 d1 = desc_at(u_begin + 1), d2 = desc_at(u_begin + 2);
    int f1 = fid_of(d1);
    Pre pa, pb;
    load_pre(fid_of(desc_at(u_begin)), pa);
    for (int i = 0; i < n_my; i += 2) {  // two units per trip: the prefetch buffers swap roles instead of being copied
      load_pre(f1, pb);                                // operands of unit i+1
      int f2 = fid_of(d2);                             // frame id of unit i+2
      int2 d3 = desc_at(u_begin + i + 3);              // descriptor of unit i+3
      expand(i, pa);
      if (i + 1 < n_my) {
        load_pre(f2, pa);
        f1 = fid_of(d3);
        d2 = desc_at(u_begin + i + 4);
        expand(i + 1, pb);
      }
    }
  } else if (warp >= 8 + kAccLdWarps && warp < 8 + 2 * kAccLdWarps) {
    // =================================== XT LOADERS ===================================
    const int t = tid - (256 + kAccLdWarps * 32);
    constexpr int NFG = SUB / 4, NNL = kAccLdWarps * 32 / NFG;  // 8 frame groups of 4; 20 column lanes
    const int fg = t / NNL, nl = t % NNL;                       // frames 4fg..4fg+3, columns nl + NNL k
    constexpr int kTK = (40 + NNL - 1) / NNL;                   // DP <= 40
    struct Fids { int ft[4]; };
    auto desc_at = [&](int ui) -> int2 { return ui < u_end ? __ldg(reinterpret_cast<const int2 *>(units + ui)) : make_int2(0, 0); };
    auto fids_of = [&](const int2 &u) -> Fids {
      Fids f;
#pragma unroll
      for (int j = 0; j < 4; j++) f.ft[j] = (4 * fg + j < u.y) ? __ldg(frame_ids + u.x + 4 * fg + j) : -1;
      return f;
    };
    struct Pre { float xt[kTK][4]; };
    auto load_pre = [&](const Fids &f, Pre &p) {
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const float *src = x32 + (int64_t)(f.ft[j] < 0 ? 0 : f.ft[j]) * DP + nl;
#pragma unroll
        for (int k = 0; k < kTK; k++) p.xt[k][j] = (f.ft[j] >= 0 && nl + NNL * k < DP) ? __ldg(src + NNL * k) : 0.f;
      }
    };
    auto expand = [&](int i, const Pre &cur) {
      const int s = i % NST;
      mbar_wait_a(x_free + 8 * s, ((i / NST) & 1) ^ 1);
      const uint32_t XTh = sm0 + (uint32_t)s * stage_bytes + 2 * x_bytes, XTl = XTh + xt_bytes;
#pragma unroll
      for (int k = 0; k < kTK; k++) {  // rows n (x) and n + DP (x^2), 16-byte chunk = frames 4fg..4fg+3
        const int n = nl + NNL * k;
        if (n < DP) {
          float4 h, l;
          split_tf32_fast(cur.xt[k][0], h.x, l.x); split_tf32_fast(cur.xt[k][1], h.y, l.y);
          split_tf32_fast(cur.xt[k][2], h.z, l.z); split_tf32_fast(cur.xt[k][3], h.w, l.w);
          uint32_t o = (uint32_t)(n & 7) * 16 + (uint32_t)fg * 128 + (uint32_t)(n >> 3) * PT;
          st_shared_v4(XTh + o, h);
          st_shared_v4(XTl + o, l);
          split_tf32_fast(cur.xt[k][0] * cur.xt[k][0], h.x, l.x); split_tf32_fast(cur.xt[k][1] * cur.xt[k][1], h.y, l.y);
          split_tf32_fast(cur.xt[k][2] * cur.xt[k][2], h.z, l.z); split_tf32_fast(cur.xt[k][3] * cur.xt[k][3], h.w, l.w);
          const int n2 = n + DP;
          o = (uint32_t)(n2 & 7) * 16 + (uint32_t)fg * 128 + (uint32_t)(n2 >> 3) * PT;
          st_shared_v4(XTh + o, h);
          st_shared_v4(XTl + o, l);
        }
      }
      if (KP2 > KP && nl == 0) {  // pad rows of GEMM2's N
        for (int n = KP; n < KP2; n++) {
          const uint32_t o = (uint32_t)(n & 7) * 16 + (uint32_t)fg * 128 + (uint32_t)(n >> 3) * PT;
          st_shared_v4(XTh + o, make_float4(0.f, 0.f, 0.f, 0.f));
          st_shared_v4(XTl + o, make_float4(0.f, 0.f, 0.f, 0.f));
        }
      }
      fence_async_smem();
      mbar_arrive_a(x_full + 8 * s);
    };
    int2 d1 = desc_at(u_begin + 1), d2 = desc_at(u_begin + 2);
    Fids f1 = fids_of(d1);
    Pre pa, pb;
    load_pre(fids_of(desc_at(u_begin)), pa);
    for (int i = 0; i < n_my; i += 2) {
      load_pre(f1, pb);
      Fids f2 = fids_of(d2);
      int2 d3 = desc_at(u_begin + i + 3);
      expand(i, pa);
      if (i + 1 < n_my) {
        load_pre(f2, pa);
        f1 = fids_of(d3);
        d2 = desc_at(u_begin + i + 4);
        expand(i + 1, pb);
      }
    }
  } else if (warp == kAccG1Warp) {
    // =================================== GEMM1 ISSUER ===================================
    // GEMM1(i) needs x_full(i) -- which the loaders give only after GEMM2(i-NST) has retired, so the L / w
    // stage it overwrites is free -- and, for the first unit of an image, that image's W in tensor memory.
    // The two GEMMs are issued by two different warps: one warp's instruction stream (descriptor
    // arithmetic, barrier polls) was the serial bottleneck of the whole pipeline when it issued both.
    const uint32_t idesc1 = make_idesc_tf32(128, SUB);
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem0, 0);
    int nimg = 0, img_prev = -1;
    for (int i = 0; i < n_my; i++) {
      const int s = i % NST;
      const int img = img_at(u_begin + i);
      mbar_wait_a(x_full + 8 * s, (i / NST) & 1);
      if (img != img_prev) { mbar_wait_a(wimg_full, nimg & 1); nimg++; img_prev = img; }
      tc_fence_after();
      if (elect_one_sync()) {
        const uint32_t Xh = sm0 + (uint32_t)s * stage_bytes;
        const uint64_t bh = make_smem_desc2(Xh, 128, PX), bl = make_smem_desc2(Xh + x_bytes, 128, PX);
        const uint32_t d = tb + (uint32_t)s * SUB, wh = tb + kAccTmW, wl = wh + KP;
        if (NSLAB == 10) {  // D = 39: fully unrolled, addresses are immediates
#pragma unroll
          for (int j = 0; j < 10; j++) tc_mma_tf32_ts(d, wh + j * 8, bh + (uint64_t)(j * 16), idesc1, j > 0);  // Wh*Xh
#pragma unroll
          for (int j = 0; j < 10; j++) tc_mma_tf32_ts(d, wl + j * 8, bh + (uint64_t)(j * 16), idesc1, 1);      // Wl*Xh
#pragma unroll
          for (int j = 0; j < 10; j++) tc_mma_tf32_ts(d, wh + j * 8, bl + (uint64_t)(j * 16), idesc1, 1);      // Wh*Xl
        } else {
          uint32_t accf = 0;
          for (int p = 0; p < 3; p++) {
            const uint32_t a0 = (p == 1) ? wl : wh;
            const uint64_t b0 = (p == 2) ? bl : bh;
            for (int j = 0; j < NSLAB; j++) {
              tc_mma_tf32_ts(d, a0 + j * 8, b0 + (uint64_t)(j * 16), idesc1, accf);
              accf = 1;
            }
          }
        }
        tc_commit_a(d1_full + 8 * s);
      }
      __syncwarp();
    }
  } else if (warp == kAccG1Warp + 1) {
    // =================================== GEMM2 ISSUER ===================================
    // GEMM2(j) needs the weights of unit j (w_full) and, after a drain, S handed back by the epilogue.
    const uint32_t idesc2 = make_idesc_tf32(128, KP2);
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem0, 0);
    int cnt = 0, ndrain = 0;
    bool need_s_free = false;
    for (int j = 0; j < n_my; j++) {
      const int sj = j % NST;
      const bool last_of_img = img_at(u_begin + j + 1) != img_at(u_begin + j);  // also true for this CTA's last unit
      mbar_wait_a(w_full + 8 * sj, (j / NST) & 1);
      if (need_s_free) { mbar_wait_a(s_free, (ndrain - 1) & 1); need_s_free = false; }
      tc_fence_after();
      cnt++;
      const bool drain = last_of_img || cnt == kAccDrain;
      if (elect_one_sync()) {
        const uint32_t XTh = sm0 + (uint32_t)sj * stage_bytes + 2 * x_bytes;
        const uint64_t bh = make_smem_desc2(XTh, 128, PT), bl = make_smem_desc2(XTh + xt_bytes, 128, PT);
        const uint32_t wh = tb + (uint32_t)sj * SUB, wl = wh + 128, d = tb + 256;
#pragma unroll
        for (int k = 0; k < SUB / 8; k++) tc_mma_tf32_ts(d, wh + k * 8, bh + (uint64_t)(k * 16), idesc2, (cnt > 1 || k > 0) ? 1u : 0u);  // wh*Xh
#pragma unroll
        for (int k = 0; k < SUB / 8; k++) tc_mma_tf32_ts(d, wl + k * 8, bh + (uint64_t)(k * 16), idesc2, 1);                              // wl*Xh
#pragma unroll
        for (int k = 0; k < SUB / 8; k++) tc_mma_tf32_ts(d, wh + k * 8, bl + (uint64_t)(k * 16), idesc2, 1);                              // wh*Xl
        tc_commit_a(x_free + 8 * sj);
        if (drain) tc_commit_a(s_full);
      }
      __syncwarp();
      if (drain) { ndrain++; need_s_free = true; cnt = 0; }
    }
  } else {
    // =================================== EPILOGUE (warps 0-7) ===================================
    const int q = warp & 3, hb = warp >> 2;  // TMEM lane quarter; frame half (and column half of S)
    const int row = 32 * q + lane;
    const uint32_t trow = (uint32_t)(32 * q) << 16;
    constexpr int FH = SUB / 2;  // frames per thread and unit (16)
    static_assert(FH == 16, "one 16-column TMEM load per thread");
    const int nc8 = KP2 / 8;
    const int c8_beg = hb ? (nc8 + 1) / 2 : 0, c8_end = hb ? nc8 : (nc8 + 1) / 2;
    const uint32_t my_acc = sacc + 4 * row;  // + 512 per column
    int cnt = 0, ndrain = 0, nflush = 0;
    float kcr = kNegInf;
    int st = 0, cur_v = 0, cur_rb = 0;
    bool dead = false;  // every lane of this warp is a pad row of the current Gaussian block
    int img_prev = -1, img = img_at(u_begin), img_next = img_at(u_begin + 1);
    for (int i = 0; i < n_my; i++) {
      const int ui = u_begin + i, s = i % NST;
      const bool first = img != img_prev, last = img != img_next;
      if (first) {  // W (hi | lo) of this (model, Gaussian block) -> TMEM, one Gaussian per lane; halves split the columns
        const TcTile unit = units[ui];
        cur_v = unit.v; cur_rb = unit.pad;
        const float *im = images + (size_t)img * (tc_accT_image_bytes(KP) / 4) + (size_t)row * 2 * KP;
        for (int ch = hb; ch < 2 * KP / 16; ch += 2) {
          uint32_t r[16];
#pragma unroll
          for (int qq = 0; qq < 4; qq++) {
            const float4 a = __ldg(reinterpret_cast<const float4 *>(im + ch * 16 + qq * 4));
            r[qq * 4 + 0] = __float_as_uint(a.x); r[qq * 4 + 1] = __float_as_uint(a.y); r[qq * 4 + 2] = __float_as_uint(a.z); r[qq * 4 + 3] = __float_as_uint(a.w);
          }
          tmem_st16(tmem0 + kAccTmW + trow + ch * 16, r);
        }
        tmem_wait_st();
        tc_fence_before();
        mbar_arrive_a(wimg_full);
        const int g = cur_rb * 128 + row;
        kcr = (g < G) ? __ldg(kcT + (size_t)img * 128 + row) : kNegInf;
        st = min(g / M, 7);
        dead = cur_rb * 128 + 32 * q >= G;
      }
      mbar_wait_a(d1_full + 8 * s, (i / NST) & 1);
      if (!dead) {  // my FH frames: accumulator columns [FH hb, FH hb + FH) of stage s.  (The rows of a dead warp
                    // feed only pad rows of S, which are never read.)
        tc_fence_after();
        const int c0 = hb * FH;
        const uint32_t tl = tmem0 + (uint32_t)s * SUB + trow + c0;
        uint32_t v[16], vl[16];
        tmem_ld16_nowait(tl, v);
        const uint32_t cfs = sm0 + (uint32_t)s * stage_bytes + cfs_off + (uint32_t)(st * SUB + c0) * 4;
        const float4 e0 = lds_v4(cfs), e1 = lds_v4(cfs + 16), e2 = lds_v4(cfs + 32), e3 = lds_v4(cfs + 48);
        const float ce[16] = {e0.x, e0.y, e0.z, e0.w, e1.x, e1.y, e1.z, e1.w, e2.x, e2.y, e2.z, e2.w, e3.x, e3.y, e3.z, e3.w};
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; j++) {
          const float y = fmaf(__uint_as_float(v[j]), 1.4426950408889634f, kcr + ce[j]);
          const float w = ex2_approx(y);  // ex2(-inf) = +0 and underflow flushes to 0: no weight; y is never NaN
          float h, l;
          split_tf32_fast(w, h, l);
          v[j] = __float_as_uint(h);
          vl[j] = __float_as_uint(l);
        }
        tmem_st16(tl, v);
        tmem_st16(tl + 128, vl);
        tmem_wait_st();
        tc_fence_before();
      }
      mbar_arrive_a(w_full + 8 * s);
      cnt++;
      if (last || cnt == kAccDrain) {  // S: TMEM (FP32, truncating) -> shared memory (round to nearest)
        mbar_wait_a(s_full, ndrain & 1);
        tc_fence_after();
        for (int c = c8_beg; c < c8_end; c++) {
          float v[8];
          tmem_ld8(tmem0 + 256 + trow + c * 8, v);
#pragma unroll
          for (int j = 0; j < 8; j++) {
            const uint32_t a = my_acc + (uint32_t)(c * 8 + j) * 512;
            sts_f32(a, lds_f32(a) + v[j]);
          }
        }
        tc_fence_before();
        mbar_arrive_a(s_free);
        ndrain++; cnt = 0;
        if (last) {  // the CTA leaves this (model, Gaussian block)
          if (scratch && nflush < kAccSlots) {
            // partial sums of this CTA's first images go to its own scratch slots (plain coalesced stores);
            // k_finalize_slots adds the slots of every image in a fixed order.  Atomics from all CTAs at once
            // were a tail of several microseconds, and their order was not reproducible.
            // slot layout [row][KP2]: the finalising kernel reads rows; 16-byte stores here
            float *sl = scratch + ((size_t)(blockIdx.x * kAccSlots + nflush) * 128 + row) * KP2;
            for (int k = c8_beg * 8; k < c8_end * 8; k += 4) {
              const uint32_t a = my_acc + (uint32_t)k * 512;
              const float4 val = make_float4(lds_f32(a), lds_f32(a + 512), lds_f32(a + 1024), lds_f32(a + 1536));
              sts_f32(a, 0.f); sts_f32(a + 512, 0.f); sts_f32(a + 1024, 0.f); sts_f32(a + 1536, 0.f);
              *reinterpret_cast<float4 *>(sl + k) = val;
            }
          } else {  // a CTA that walks through many small images: double atomics, uncontended there
            const int g = cur_rb * 128 + row;
            double *stp = stats + (int64_t)cur_v * stats_stride;
            for (int k = c8_beg * 8; k < c8_end * 8; k++) {
              const uint32_t a = my_acc + (uint32_t)k * 512;
              const double val = (double)lds_f32(a);
              sts_f32(a, 0.f);
              if (g < G) {
                if (k < D) atomicAdd(stp + off_S1 + (int64_t)g * D + k, val);
                else if (k == D) atomicAdd(stp + off_S0 + g, val);
                else if (k >= DP && k < DP + D) atomicAdd(stp + off_S2 + (int64_t)g * D + (k - DP), val);
              }
            }
          }
          nflush++;
        }
      }
      img_prev = img; img = img_next; img_next = img_at(ui + 2);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == kAccG1Warp) tmem_dealloc(tmem0, 512);
}

// Adds the scratch slots of k_accum_ws to the statistics (in double, fixed order) and finishes them as
// k_finalize_stats does: S1 += ctr S0 (features were centred), S2 = sum w x^2 - 2 m sum w x + m^2 sum w with
// m = mu_old - ctr (the reference's sum w (x - mu_old)^2, T-FS:1716-1719).  One block = one Gaussian: thread
// (dimension d, part p) adds every fourth slot of the Gaussian's image, the four parts are combined in a fixed order
// through shared memory (so the result does not depend on scheduling), and S0 is read by everyone before one thread
// rewrites it.
constexpr int kFinParts = 4;
__global__ void __launch_bounds__(64 * kFinParts)
k_finalize_slots(double *__restrict__ stats, int64_t stats_stride, int G, int D, int DP, int KP2, int nRB, int64_t off_S0,
                 int64_t off_S1, int64_t off_S2, const double *__restrict__ ctr, const double *__restrict__ mu,
                 const float *__restrict__ scratch, const int32_t *__restrict__ slot_start, const int32_t *__restrict__ slot_ids,
                 const float *__restrict__ dsc = nullptr) {  // dsc: per-column factors of k_accum_h's scaled sums (powers of two)
  const int v = blockIdx.y, g = blockIdx.x, d = threadIdx.x & 63, part = threadIdx.x >> 6;
  const bool lived = d < D;
  double *st = stats + (int64_t)v * stats_stride;
  __shared__ double sp[kFinParts][3][64];
  const int img = v * nRB + (g >> 7), row = g & 127;
  const int k0 = slot_start[img], nk = slot_start[img + 1] - k0;  // (slot tables: uploaded with the training map)
  pdl_wait();
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  for (int k = part; k < nk; k += kFinParts) {
    const float *sl = scratch + ((size_t)slot_ids[k0 + k] * 128 + row) * KP2;
    s0 += (double)sl[D];
    if (lived) { s1 += (double)sl[d]; s2 += (double)sl[DP + d]; }
  }
  if (dsc) {
    s0 *= (double)dsc[D];
    if (lived) { s1 *= (double)dsc[d]; s2 *= (double)dsc[DP + d]; }
  }
  sp[part][0][d] = s0; sp[part][1][d] = s1; sp[part][2][d] = s2;
  // the statistics the atomic path may have left (CTAs that walked through many small images)
  const double b0 = st[off_S0 + g];
  const double b1 = lived ? st[off_S1 + (int64_t)g * D + d] : 0.0, b2 = lived ? st[off_S2 + (int64_t)g * D + d] : 0.0;
  __syncthreads();
  if (part != 0) return;
  s0 = b0; s1 = b1; s2 = b2;
#pragma unroll
  for (int p = 0; p < kFinParts; p++) { s0 += sp[p][0][d]; s1 += sp[p][1][d]; s2 += sp[p][2][d]; }
  if (lived) {
    const double m = mu[((int64_t)v * G + g) * D + d] - ctr[d];
    st[off_S2 + (int64_t)g * D + d] = s2 - 2.0 * m * s1 + m * m * s0;
    st[off_S1 + (int64_t)g * D + d] = s1 + ctr[d] * s0;
  }
  if (d == 0) st[off_S0 + g] = s0;
}

}  // namespace hmmk
