// acch_kernels.cuh -- k_accum_h: the mixture accumulators (calc_mix_param, T-FS:1691-1727) with HALF-PRECISION operands
// and frame tiles that are expanded ONCE per feature set instead of once per EM iteration.
//
// k_accum_ws (ws_kernels.cuh) spends 88 % of its time in the skeleton of its two loader roles: ten warps that re-read the
// fp32 frames every iteration, form [x | x^2], split every value into TF32 hi / lo and store the tile twice (X for GEMM1,
// its transpose XT for GEMM2, because TF32 operands must be K-major).  The features do not change between EM iterations, and
// half-precision operands may be MN-major (scripts/tc_probe_h.cu: exact on this part).  So
//   * k_pack_x16 writes, once per (features, training map), the expanded tile of every unit -- 64 frames x KP columns,
//     hi | lo halves, already in the shared-memory layout of the MMA operand -- and the kernel fetches a unit with ONE bulk
//     copy (cp.async.bulk, 20 KB, completing on the stage's mbarrier; UBLKCP in SASS).  No loader warps.
//   * the SAME tile is the B operand of both GEMMs (column blocks [q | x | Q], q and Q both x^2 under two scalings, see below):
//       GEMM1  L[g][f] = sum_k W[g][k] X[f][k]    B = [q | x] K-major  (N = frames,  K = columns; LBO 128, SBO PX)
//       GEMM2  S[g][k] += sum_f w[g][f] X[f][k]   B = [x | Q] MN-major (N = columns, K = frames;  LBO PX,  SBO 128)
//     byte(f, k) = (f/8) PX + (k/8) 128 + (f%8) 16 + (k%8) 2,  PX = (3 DP/8) 128
//   * kind::f16 MMAs (K = 16) run at twice the TF32 rate.
// Numerics: a half keeps the 11 significant bits of a TF32 operand, hi + lo of the split keep 22, and hi*hi + lo*hi + hi*lo in
// the FP32 accumulator is the 3xTF32 scheme -- provided the halves stay inside the half's exponent range (normal down to
// 2^-14, nothing below 2^-24).  The tiles must not depend on the models (they are packed once), so every dimension is scaled by
// powers of two taken from the DATA alone (k_acc16_scales, r_d = largest |x_d| about the centre):
//   x' = x / s1_d, max |x'| in [5.7, 11.3]; q = x^2 / s2_d likewise.  These face W' = mu iv s1_d and -iv s2_d / 2 in GEMM1, which
//     are then bounded by kappa / 8 (the accuracy guard's bound, <= 1250): the two factors of a term share its magnitude, and a
//     factor below 2^-3, whose lo half loses bits (absolute error 2^-25), costs <= 3e-8 times the other factor in a log-likelihood.
//   Q = x^2 / S2_d with max Q in [2^14.5, 2^15.5]: GEMM2 only, where no W' limits the scale.  The second-order sums enter the
//     variance as S2 - 2 m S1 + m^2 S0, so a frame close to the centre (x^2 far below r^2) must keep its relative precision: Q
//     keeps 22 bits down to |x| = r / 512 (q: r / 8; with q in GEMM2 a one-frame Gaussian near the centre of data with
//     r / sigma ~ 1000 missed the variance by 2e-4).
// The weights w <= 1 are scaled by 2^14 (exact; a weight down to 2^-17 keeps 22 bits) and the sums are scaled back in double by
// k_finalize_slots.  A weighted E-step (an MMI denominator round, whose weights carry the round's word posteriors, 1e-5 ..
// 1e-3 and below) adds wshift to that exponent, so that its largest weight comes to [2^13, 2^14) as well; wback = 2^-wshift
// undoes it in double (wshift 0, wback 1: unweighted E-steps are unchanged bit for bit).
//
// 13 warps: 0-7 epilogue (L -> w in place in tensor memory, drains of S, W images), 8-9 weight exponents (one thread per
// frame: log2 gamma - logb log2 e for every state), 10 bulk-copy producer, 11 GEMM1 issuer, 12 GEMM2 issuer.
// TMEM columns: [0, 256) four stages of L / w (64 frames: a thread of frame half hb reads L columns [32 hb, 32 hb + 32) and
// writes w_hi to [32 hb, +16), w_lo to [32 hb + 16, +16), two frames per column) | [256, 256 + KP) S | [352, 352 + KP) W hi, lo.
#pragma once

#include <cuda_fp16.h>

#include "dec_kernels.cuh"
#include "ws_kernels.cuh"

namespace hmmk {

constexpr int kAhSub = 64;      // frames per unit
constexpr int kAhStages = 4;    // units in flight (shared-memory and TMEM stages)
constexpr int kAhDrain = 8;     // units accumulated in TMEM before S moves out (512 frames)
constexpr int kAhCfWarps = kAhSub / 32;
constexpr int kAhProdWarp = 8 + kAhCfWarps;
constexpr int kAhG1Warp = kAhProdWarp + 1;
constexpr int kAhThreads = (kAhG1Warp + 2) * 32;  // 13 warps
constexpr int kAhTmS = 256, kAhTmW = 352;
constexpr float kAhWLog2 = 14.f;  // weights are scaled by 2^14

__host__ __device__ inline size_t ah_tile_bytes(int KP) { return (size_t)2 * (kAhSub / 8) * (3 * KP / 16) * 128; }  // hi | lo of [q | x | Q]
__host__ __device__ inline size_t ah_image_bytes(int KP) { return (size_t)128 * 2 * KP * 2; }  // [128][hi (KP halves) | lo (KP halves)]
__host__ __device__ inline size_t ah_stage_bytes(int KP) { return ah_tile_bytes(KP) + kAhSub * 8 * 4; }
// stages | 1 KB alignment slack | barriers (256 B) | image ids | S accumulator [KP][128] floats
__host__ __device__ inline size_t ah_smem_bytes(int KP) { return kAhStages * ah_stage_bytes(KP) + 1024 + 256 + kAccImgCap * 4 + (size_t)KP * 128 * 4; }

// sc[0, DP) = 1 / s2_d (q), [DP, 2DP) = 1 / s1_d (x), [2DP, 3DP) = 1 / S2_d (Q): the column blocks of a tile;
// [3DP, 4DP) = s2_d, [4DP, 5DP) = s1_d: the model side of GEMM1; [5DP, 7DP) = what a column of the scaled sums [S1 | S2] is
// multiplied by (k_finalize_slots).  All powers of two; 0 for a dimension in which no frame leaves the centre (its terms are
// exactly 0) and for the pad columns; column D of the x block is the constant 1 (its sum is the occupancy S0).
constexpr int kAhScN = 7;
__global__ void k_acc16_scales(const unsigned int *__restrict__ xabs, int D, int DP, float *__restrict__ sc) {
  const int d = threadIdx.x;
  if (d >= DP) return;
  float xs1 = 0.f, xs2 = 0.f, xs2b = 0.f, s1 = 0.f, s2 = 0.f, s2b = 0.f;
  if (d < D) {
    const float r = __uint_as_float(xabs[d]);
    if (r > 0.f && r < INFINITY) {
      const float e1 = rintf(log2f(r)) - 3.f, e2 = rintf(2.f * log2f(r)) - 3.f, e2b = e2 + 3.f - 15.f;
      s1 = exp2f(e1); xs1 = exp2f(-e1);
      s2 = exp2f(e2); xs2 = exp2f(-e2);
      s2b = exp2f(e2b); xs2b = exp2f(-e2b);
    }
  } else if (d == D) {
    xs1 = 1.f;
  }
  const float back = exp2f(-kAhWLog2);
  sc[d] = xs2; sc[DP + d] = xs1; sc[2 * DP + d] = xs2b;
  sc[3 * DP + d] = s2; sc[4 * DP + d] = s1;
  sc[5 * DP + d] = (d < D ? s1 : d == D ? 1.f : 0.f) * back;
  sc[6 * DP + d] = s2b * back;
}

// tiles[t] = (first row in frame_ids, rows) of unit tile t; one block per tile.  A thread takes (frame, 8 columns): eight
// consecutive threads write one 128-byte line of the tile.
__global__ void __launch_bounds__(256)
k_pack_x16(const int2 *__restrict__ tiles, const int32_t *__restrict__ frame_ids, const float *__restrict__ x32, const float *__restrict__ sc,
           int DP, unsigned char *__restrict__ x16) {
  const int KP = 2 * DP, NCHX = DP / 8, NCH = 3 * NCHX;
  const int2 tl = tiles[blockIdx.x];
  unsigned char *hi = x16 + (size_t)blockIdx.x * ah_tile_bytes(KP), *lo = hi + ah_tile_bytes(KP) / 2;
  for (int it = threadIdx.x; it < kAhSub * NCH; it += blockDim.x) {
    const int r = it & 7, c = (it >> 3) % NCH, fg = it / (8 * NCH), f = fg * 8 + r;
    uint4 h = make_uint4(0u, 0u, 0u, 0u), l = h;
    if (f < tl.y) {
      const int blk = c / NCHX, cc = c - blk * NCHX;  // 0: q, 1: x, 2: Q
      const float *src = x32 + (int64_t)__ldg(frame_ids + tl.x + f) * DP + cc * 8;
      const float *s = sc + blk * DP + cc * 8;
      const float4 a = __ldg(reinterpret_cast<const float4 *>(src)), b = __ldg(reinterpret_cast<const float4 *>(src + 4));
      float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
      for (int j = 0; j < 8; j++) v[j] = (blk != 1 ? v[j] * v[j] : v[j]) * s[j];
      split_half2(v[0], v[1], h.x, l.x); split_half2(v[2], v[3], h.y, l.y);
      split_half2(v[4], v[5], h.z, l.z); split_half2(v[6], v[7], h.w, l.w);
    }
    const size_t o = (size_t)fg * NCH * 128 + (size_t)c * 128 + (size_t)r * 16;
    *reinterpret_cast<uint4 *>(hi + o) = h;
    *reinterpret_cast<uint4 *>(lo + o) = l;
  }
}

// W images of the accumulate pass in halves: [img][128 Gaussians][hi (KP) | lo (KP)], columns [-iv s2 / 2 | mu iv s1] (the
// order of the tile's blocks q, x), scaled by the model-side factors of sc
__global__ void k_pack_wT_h(const double *__restrict__ mu, const double *__restrict__ iv, const float *__restrict__ kc2all,
                            const double *__restrict__ ctr, const float *__restrict__ sc, int G, int nRB, int D, int DP,
                            unsigned short *__restrict__ images, float *__restrict__ kcT) {
  const int img = blockIdx.y, v = img / nRB, rb = img - v * nRB;
  const int KP = 2 * DP;
  pdl_wait();
  unsigned short *im = images + (size_t)img * (ah_image_bytes(KP) / 2);
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 128 * KP; idx += gridDim.x * blockDim.x) {
    const int r = idx / KP, k = idx - r * KP;
    const int part = k / DP, d = k - part * DP;
    const int g = rb * 128 + r;
    float val = 0.f;
    if (g < G && d < D) {
      const int64_t gg = (int64_t)v * G + g;
      const double m = mu[gg * D + d] - ctr[d], w = iv[gg * D + d];
      val = (float)(part == 1 ? m * w * (double)sc[4 * DP + d] : -0.5 * w * (double)sc[3 * DP + d]);
    }
    unsigned short h, l;
    split_half(val, h, l);
    im[(size_t)r * 2 * KP + k] = h;
    im[(size_t)r * 2 * KP + KP + k] = l;
    if (k == 0) kcT[(size_t)img * 128 + r] = (g < G) ? kc2all[(int64_t)v * G + g] : kNegInf;
  }
}

__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst_smem, const void *src, uint32_t bytes, uint32_t mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem), "l"(src), "r"(bytes),
               "r"(mbar)
               : "memory");
}

// units: {row0 (index into frame_ids), nrows (<= 64), img = v nRB + rb, state0 = tile index in x16, v, pad = rb}
__global__ void __launch_bounds__(kAhThreads, 1)
k_accum_h(const TcTile *__restrict__ units, int nunits, const int32_t *__restrict__ frame_ids, const unsigned char *__restrict__ x16,
          const uint32_t *__restrict__ images, const float *__restrict__ kcT, const float *__restrict__ logb, const float *__restrict__ gamma,
          int N, int M, int G, int D, int DP, double *__restrict__ stats, int64_t stats_stride, int64_t off_S0, int64_t off_S1, int64_t off_S2,
          float *__restrict__ scratch, const float *__restrict__ dsc, float wshift, double wback) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr int NST = kAhStages, SUB = kAhSub;
  const int KP = 2 * DP, NK1 = KP / 16;
  const uint32_t PX = (uint32_t)(3 * DP / 8) * 128;       // bytes per group of 8 frames: blocks q, x, Q
  const uint32_t g2_off = (uint32_t)(DP / 8) * 128;       // GEMM2 reads the blocks x, Q
  const uint32_t x_bytes = (SUB / 8) * PX;                // one half (hi or lo) of a tile
  const uint32_t cfs_off = 2 * x_bytes;
  const uint32_t stage_bytes = cfs_off + SUB * 8 * 4;
  const uint32_t sm0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = sm0 + NST * stage_bytes;
  const uint32_t x_full = bars, x_free = bars + 8 * NST, d1_full = bars + 16 * NST, w_full = bars + 24 * NST, s_full = bars + 32 * NST,
                 s_free = s_full + 8, wimg_full = s_full + 16, tmem_slot = s_full + 24;
  const uint32_t simg = bars + 256;                       // int32 [kAccImgCap]
  const uint32_t sacc = simg + kAccImgCap * 4;            // float [KP][128]: S per (column, Gaussian lane)
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int per = (nunits + gridDim.x - 1) / gridDim.x;
  const int u_begin = blockIdx.x * per, u_end = min(nunits, u_begin + per);
  const int n_my = max(0, u_end - u_begin);
  for (int k = tid; k < min(n_my, kAccImgCap); k += kAhThreads)
    asm volatile("st.shared.s32 [%0], %1;" ::"r"(simg + 4 * k), "r"(__ldg(&units[u_begin + k].img)) : "memory");
  for (int k = tid; k < KP * 128; k += kAhThreads) sts_f32(sacc + 4 * k, 0.f);

  if (tid == 0) {
    auto init = [](uint32_t addr, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(addr), "r"(count) : "memory"); };
    for (int s = 0; s < NST; s++) {
      init(x_full + 8 * s, kAhCfWarps * 32 + 1);  // weight-exponent threads + the producer's expect_tx
      init(x_free + 8 * s, 1);                    // tcgen05.commit after GEMM2
      init(d1_full + 8 * s, 1);                   // tcgen05.commit after GEMM1
      init(w_full + 8 * s, 256);                  // epilogue threads
    }
    init(s_full, 1);
    init(s_free, 256);
    init(wimg_full, 256);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kAhG1Warp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem0 = (uint32_t)lds_i32(tmem_slot);
  // Above: only the unit table (uploaded with the training map) and this CTA's own shared and tensor memory.  Below:
  // gamma (k_fb_res), logb (k_emis_ws) and x16 (k_pack_x16) of this launch sequence, and the statistics.
  pdl_wait();
  pdl_trigger();  // this CTA's work is a fixed unit range: nothing is left to claim

  auto img_at = [&](int ui) -> int {
    if (ui < u_begin || ui >= u_end) return -1;
    return (ui - u_begin < kAccImgCap) ? lds_i32(simg + 4 * (ui - u_begin)) : __ldg(&units[ui].img);
  };

  if (warp >= 8 && warp < 8 + kAhCfWarps) {
    // =================================== WEIGHT EXPONENTS ===================================
    // thread <-> frame row xr of the unit: cf[state][xr] = log2 gamma - logb log2 e + 14 (-inf = no weight).  Global loads run
    // ahead of the hand-off: unit descriptor (i+3) -> frame id (i+2) -> gamma, logb (i+1), while unit i is stored.
    const int xr = tid - 256;
    struct Pre { float gm[8], lb[8]; };
    auto desc_at = [&](int ui) -> int2 { return ui < u_end ? __ldg(reinterpret_cast<const int2 *>(units + ui)) : make_int2(0, 0); };  // (row0, nrows)
    auto fid_of = [&](const int2 &u) -> int { return (xr < u.y) ? __ldg(frame_ids + u.x + xr) : -1; };
    auto load_pre = [&](int f, Pre &p) {
#pragma unroll
      for (int st = 0; st < 8; st++) {
        const bool ok = f >= 0 && st < N;
        p.gm[st] = ok ? __ldg(gamma + (int64_t)f * N + st) : 0.f;
        p.lb[st] = ok ? __ldg(logb + (int64_t)f * N + st) : 0.f;
      }
    };
    auto publish = [&](int i, const Pre &cur) {
      const int s = i % NST;
      mbar_wait_a(x_free + 8 * s, ((i / NST) & 1) ^ 1);  // stage s: GEMM2 of unit i-NST has retired
      const uint32_t cfs = sm0 + (uint32_t)s * stage_bytes + cfs_off + 4 * xr;
#pragma unroll
      for (int st = 0; st < 8; st++) {
        float cf = kNegInf;
        // (+ 14: the weights' scale 2^14.  cf is ~ +200 and rounded to 2^-16 as it is; added to kc in the epilogue the 14 would
        // cost another rounding of that size)
        if (cur.gm[st] > 0.f && cur.lb[st] > kNegInf) cf = fmaf(cur.lb[st], -1.4426950408889634f, __log2f(cur.gm[st]) + (kAhWLog2 + wshift));
        sts_f32(cfs + st * SUB * 4, cf);
      }
      mbar_arrive_a(x_full + 8 * s);
    };
    int2 d1 = desc_at(u_begin + 1), d2 = desc_at(u_begin + 2);
    int f1 = fid_of(d1);
    Pre pa, pb;
    load_pre(fid_of(desc_at(u_begin)), pa);
    for (int i = 0; i < n_my; i += 2) {  // two units per trip: the prefetch buffers swap roles instead of being copied
      load_pre(f1, pb);
      int f2 = fid_of(d2);
      int2 d3 = desc_at(u_begin + i + 3);
      publish(i, pa);
      if (i + 1 < n_my) {
        load_pre(f2, pa);
        f1 = fid_of(d3);
        d2 = desc_at(u_begin + i + 4);
        publish(i + 1, pb);
      }
    }
  } else if (warp == kAhProdWarp) {
    // =================================== PRODUCER ===================================
    if (lane == 0) {
      const uint32_t tile_bytes = 2 * x_bytes;
      int tnext = n_my > 0 ? __ldg(&units[u_begin].state0) : 0;
      for (int i = 0; i < n_my; i++) {
        const int s = i % NST, tcur = tnext;
        if (i + 1 < n_my) tnext = __ldg(&units[u_begin + i + 1].state0);
        mbar_wait_a(x_free + 8 * s, ((i / NST) & 1) ^ 1);
        mbar_expect_tx_a(x_full + 8 * s, tile_bytes);
        bulk_copy_g2s(sm0 + (uint32_t)s * stage_bytes, x16 + (size_t)tcur * tile_bytes, tile_bytes, x_full + 8 * s);
      }
    }
  } else if (warp == kAhG1Warp) {
    // =================================== GEMM1 ISSUER ===================================
    const uint32_t idesc1 = make_idesc_f16(128, SUB);
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
        const uint32_t d = tb + (uint32_t)s * SUB, wh = tb + kAhTmW, wl = wh + DP;
        if (NK1 == 5) {  // D = 39: fully unrolled, addresses are immediates
#pragma unroll
          for (int j = 0; j < 5; j++) tc_mma_f16_ts(d, wh + j * 8, bh + (uint64_t)(j * 16), idesc1, j > 0);  // Wh*Xh
#pragma unroll
          for (int j = 0; j < 5; j++) tc_mma_f16_ts(d, wl + j * 8, bh + (uint64_t)(j * 16), idesc1, 1);      // Wl*Xh
#pragma unroll
          for (int j = 0; j < 5; j++) tc_mma_f16_ts(d, wh + j * 8, bl + (uint64_t)(j * 16), idesc1, 1);      // Wh*Xl
        } else {
          uint32_t accf = 0;
          for (int p = 0; p < 3; p++) {
            const uint32_t a0 = (p == 1) ? wl : wh;
            const uint64_t b0 = (p == 2) ? bl : bh;
            for (int j = 0; j < NK1; j++) {
              tc_mma_f16_ts(d, a0 + j * 8, b0 + (uint64_t)(j * 16), idesc1, accf);
              accf = 1;
            }
          }
        }
        tc_commit_a(d1_full + 8 * s);
      }
      __syncwarp();
    }
  } else if (warp == kAhG1Warp + 1) {
    // =================================== GEMM2 ISSUER ===================================
    const uint32_t idesc2 = make_idesc_f16(128, KP) | (1u << 16);  // B is MN-major: the tile as [frames][columns]
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem0, 0);
    const uint64_t kstep = (uint64_t)((2 * PX) >> 4);  // 16 frames = two groups of 8
    int cnt = 0, ndrain = 0;
    bool need_s_free = false;
    for (int j = 0; j < n_my; j++) {
      const int sj = j % NST;
      const bool last_of_img = img_at(u_begin + j + 1) != img_at(u_begin + j);  // also true for this CTA's last unit
      mbar_wait_a(w_full + 8 * sj, (j / NST) & 1);
      if (need_s_free) { mbar_wait_a(s_free, (ndrain - 1) & 1); need_s_free = false; }
      tc_fence_after();
      cnt++;
      const bool drain = last_of_img || cnt == kAhDrain;
      if (elect_one_sync()) {
        const uint32_t Xh = sm0 + (uint32_t)sj * stage_bytes;
        const uint64_t bh = make_smem_desc2(Xh + g2_off, PX, 128), bl = make_smem_desc2(Xh + x_bytes + g2_off, PX, 128);
        const uint32_t w0 = tb + (uint32_t)sj * SUB, d = tb + kAhTmS;
#pragma unroll
        for (int k = 0; k < SUB / 16; k++)
          tc_mma_f16_ts(d, w0 + 32 * (k >> 1) + 8 * (k & 1), bh + kstep * k, idesc2, (cnt > 1 || k > 0) ? 1u : 0u);  // wh*Xh
#pragma unroll
        for (int k = 0; k < SUB / 16; k++) tc_mma_f16_ts(d, w0 + 32 * (k >> 1) + 8 * (k & 1) + 16, bh + kstep * k, idesc2, 1);  // wl*Xh
#pragma unroll
        for (int k = 0; k < SUB / 16; k++) tc_mma_f16_ts(d, w0 + 32 * (k >> 1) + 8 * (k & 1), bl + kstep * k, idesc2, 1);       // wh*Xl
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
    const int nc8 = KP / 8;
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
      if (first) {  // W of this (model, Gaussian block) -> TMEM, one Gaussian per lane: hb = 0 the hi halves, hb = 1 the lo halves
        const TcTile unit = units[ui];
        cur_v = unit.v; cur_rb = unit.pad;
        const uint32_t *im = images + (size_t)img * (ah_image_bytes(KP) / 4) + (size_t)row * KP + hb * DP;
        for (int ch = 0; ch < DP / 8; ch++) {
          const uint4 a = __ldg(reinterpret_cast<const uint4 *>(im + ch * 8)), b = __ldg(reinterpret_cast<const uint4 *>(im + ch * 8 + 4));
          const uint32_t r[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
          tmem_st8(tmem0 + kAhTmW + trow + hb * DP + ch * 8, r);
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
      if (!dead) {  // my 32 frames: accumulator columns [32 hb, 32 hb + 32) of stage s
        tc_fence_after();
        const uint32_t tl = tmem0 + (uint32_t)s * SUB + trow + 32 * hb;
        uint32_t v0[16], v1[16], wh[16], wl[16];
        tmem_ld16_nowait(tl, v0);
        tmem_ld16_nowait(tl + 16, v1);
        const uint32_t cfs = sm0 + (uint32_t)s * stage_bytes + cfs_off + (uint32_t)(st * SUB + 32 * hb) * 4;
        float ce[32];
#pragma unroll
        for (int j = 0; j < 8; j++) {
          const float4 e = lds_v4(cfs + 16 * j);
          ce[4 * j] = e.x; ce[4 * j + 1] = e.y; ce[4 * j + 2] = e.z; ce[4 * j + 3] = e.w;
        }
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; j += 2) {  // ex2(-inf) = +0 and underflow flushes to 0: no weight; the exponent is never NaN
          const float a = ex2_approx(fmaf(__uint_as_float(v0[j]), 1.4426950408889634f, kcr + ce[j]));
          const float b = ex2_approx(fmaf(__uint_as_float(v0[j + 1]), 1.4426950408889634f, kcr + ce[j + 1]));
          split_half2(a, b, wh[j >> 1], wl[j >> 1]);
        }
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          const float a = ex2_approx(fmaf(__uint_as_float(v1[j]), 1.4426950408889634f, kcr + ce[16 + j]));
          const float b = ex2_approx(fmaf(__uint_as_float(v1[j + 1]), 1.4426950408889634f, kcr + ce[16 + j + 1]));
          split_half2(a, b, wh[8 + (j >> 1)], wl[8 + (j >> 1)]);
        }
        tmem_st16(tl, wh);
        tmem_st16(tl + 16, wl);
        tmem_wait_st();
        tc_fence_before();
      }
      mbar_arrive_a(w_full + 8 * s);
      cnt++;
      if (last || cnt == kAhDrain) {  // S: TMEM (FP32, truncating) -> shared memory (round to nearest)
        mbar_wait_a(s_full, ndrain & 1);
        tc_fence_after();
        for (int c = c8_beg; c < c8_end; c++) {
          float v[8];
          tmem_ld8(tmem0 + kAhTmS + trow + c * 8, v);
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
          if (scratch && nflush < kAccSlots) {  // slot layout [row][KP], as k_accum_ws (k_finalize_slots scales the sums back)
            float *sl = scratch + ((size_t)(blockIdx.x * kAccSlots + nflush) * 128 + row) * KP;
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
              const double val = (double)lds_f32(a) * ((double)__ldg(dsc + k) * wback);
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
  if (warp == kAhG1Warp) tmem_dealloc(tmem0, 512);
}

}  // namespace hmmk
