// dec_kernels.cuh -- k_emis_dec: the emission contraction of the DECODE regime (every frame of an utterance batch
// against every model of the vocabulary; calc_symbol_probab + calc_gaus, R-FS:860-947, inside the recogniser's loops
// R-FS:341-369) for mixtures of up to 16 Gaussians per state.
//
// k_emis_ws (ws_kernels.cuh) walks (image, frame tile) pairs image-major: the W image stays in shared memory and every
// unit re-expands its 128 frames ([x | x^2], TF32 hi / lo) into tensor memory -- with a 1,000-word vocabulary that is 200
// expansions of the same frames, a quarter of all instructions of a kernel that is bound by instruction issue.  Here the
// loops are swapped: a CTA expands a frame tile ONCE into tensor memory and keeps it there while ALL W images stream
// past it.  A W image is 60 KB; one per 1,440 tensor-pipe cycles and SM would be ~12 TB/s of L2 reads, so the CTAs work
// in CLUSTERS of two: every CTA fetches half of the image with a bulk-tensor-engine copy that is MULTICAST into the
// shared memory of both (cp.async.bulk ... .multicast::cluster), each CTA's `full` barrier counting the bytes of both
// halves.  A stage is refilled only when the MMAs of both CTAs have released it (tcgen05.commit multicast to the
// `empty` barriers of the cluster).  Pairs, not clusters of four: pairs fill all 148 SMs of a B200, while 37 clusters of
// four do not all fit its GPCs at once (DESIGN.md, "Measured and dropped").
//
// Warps (18): 0-11 epilogue (TMEM lane quarter w & 3, 16-column groups g with g % 3 == w >> 2: log-sum-exp over the
// mixtures of every state, additive constants from shared memory, stores log b), 12-15 frame expanders (one frame row per
// thread, once per round), 16 MMA issuer (also copies the image's constants out of the W stage before it is released),
// 17 producer (one lane issues the multicast copies).
// Rounds: round r of CTA b is frame tile r * gridDim + b; every CTA of a cluster runs the same number of rounds and every
// round runs all images (a CTA without a tile in the last round still fetches and releases its half).
// TMEM columns: [0, 160) the frame tile [x_hi | x2_hi | x_lo | x2_lo] (DP <= 40), then THREE accumulator stages of 96
// columns (TN <= 96): the log-sum-exp epilogue of a unit takes longer than its MMAs, and with two stages the tensor pipe
// waited for it (period = (MMA + epilogue) / 2; measured 54 % pipe activity, the same as k_emis_ws).  W image layout and
// the MMA descriptors are k_emis_ws's.
#pragma once
#include "ws_kernels.cuh"

namespace hmmk {

constexpr int kDecCluster = 2;     // CTAs per cluster (half of every image per CTA)
constexpr int kDecEpiWarps = 12;
constexpr int kDecThreads = (kDecEpiWarps + 6) * 32;  // + 4 expanders, MMA issuer, producer
constexpr int kDecStages = 3;                         // W images in flight per CTA
constexpr int kDecAcc = 3;                            // accumulator stages in tensor memory
// half-precision operands: an image is half as large and its MMAs take half as long, so twice the stages cover the same
// refill latency; the frame tile takes 80 tensor-memory columns instead of 160, which leaves room for a fourth accumulator
constexpr int kDecStages16 = 6;
constexpr int kDecAcc16 = 4;

// Output layout of k_emis_dec ("interleaved"): blocks of 8 frames, state-major inside a block,
//   logb[((f / 8) * S + s) * 8 + f % 8]        f = frame of the batch, s = state column (model * N + state), S = ldb
// A thread of the epilogue owns a frame row, so its store of one state is 4 bytes; in the row-per-frame layout every such
// store is a sector of its own (32 sectors per warp instruction), here 8 lanes share a sector and a warp instruction writes
// four full sectors.  The cell scorers read a (block, model) as N consecutive sectors with 16-byte loads.
__host__ __device__ inline int64_t dec_logb_index(int64_t f, int64_t s, int64_t S) { return ((f >> 3) * S + s) * 8 + (f & 7); }
__host__ __device__ inline size_t dec_logb_floats(int64_t nframes, int64_t S) { return (size_t)((nframes + 7) / 8) * 8 * (size_t)S; }

__host__ __device__ inline size_t dec_emis_smem_bytes(int TN, int KP, bool h16 = false) {
  return (h16 ? kDecStages16 * ((size_t)2 * (TN / 8) * (KP / 8) * 128 + (size_t)TN * 4) : kDecStages * ws_image_bytes(TN, KP)) + 1024 + 512;
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx_a(uint32_t addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(addr), "r"(bytes) : "memory");
}
// global -> shared memory of every CTA in `mask` (same offset in each), completing `bytes` on the barrier at the same
// offset in each of them
__device__ __forceinline__ void bulk_copy_multicast(uint32_t dst_smem, const void *src, uint32_t bytes, uint32_t mbar, uint16_t mask) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(mbar), "h"(mask)
               : "memory");
}
// arrive (once) on the barrier at this offset in every CTA of `mask` when all MMAs issued so far by this thread have retired
__device__ __forceinline__ void tc_commit_multicast(uint32_t mbar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(mbar), "h"(mask) : "memory");
}

// MP: padded mixtures per state (1, 2, 3, 4, 5, 8, 16); MR: real mixtures of a state (0 = all MP);
// H16: half-precision operands (images of k_pack_w_dec16, `scales` of k_dec16_scales)
template <int MP, int MR, bool H16>
__global__ void __launch_bounds__(kDecThreads, 1)
k_emis_dec(int ntiles, int nframes, int nimg, const float *__restrict__ x32, const float *__restrict__ images, int DP, int TN,
           float *__restrict__ logb, int64_t fbase, int64_t ldb, int S_total, int SCt, const float *__restrict__ scales) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr int NST = H16 ? kDecStages16 : kDecStages;
  const int KP = 2 * DP;
  const uint32_t P = H16 ? (uint32_t)(KP / 8) * 128 : (uint32_t)(KP / 4) * 128;
  const uint32_t w_bytes = 2 * (uint32_t)(TN / 8) * P, img_bytes = w_bytes + (uint32_t)TN * 4;
  const uint32_t Ws = (smem_u32(smem_raw) + 1023u) & ~1023u;  // NST stages of img_bytes (multiples of 64)
  const uint32_t bars = (Ws + NST * img_bytes + 15u) & ~15u;
  constexpr int NA = H16 ? kDecAcc16 : kDecAcc;
  const uint32_t full = bars, empty = bars + 8 * NST, dfull = bars + 16 * NST, dempty = dfull + 8 * NA, kfull = dfull + 16 * NA, xfull = dfull + 24 * NA,
                 xempty = xfull + 8, tmem_slot = xfull + 16;
  __shared__ __align__(16) float skc[kDecAcc16][kWsMaxTN];  // additive constants of the image an accumulator stage belongs to
  __shared__ float ssc[2][40];                             // H16: 1 / s1_d, 1 / s2_d
  if (H16) {
    for (int d = threadIdx.x; d < 80; d += kDecThreads) ssc[d / 40][d % 40] = (d % 40 < DP) ? scales[(d / 40) * DP + d % 40] : 1.f;
  }
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t crank = cluster_ctarank();
  constexpr uint16_t kMask = (1u << kDecCluster) - 1;

  if (tid == 0) {
    auto init = [](uint32_t addr, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(addr), "r"(count) : "memory"); };
    for (int s = 0; s < NST; s++) {
      init(full + 8 * s, 1);             // this CTA's producer (arrive.expect_tx); the bytes come from both CTAs
      init(empty + 8 * s, kDecCluster);  // tcgen05.commit of every CTA of the cluster
    }
    for (int a = 0; a < NA; a++) {
      init(dfull + 8 * a, 1);                   // tcgen05.commit
      init(dempty + 8 * a, kDecEpiWarps * 32);  // every epilogue thread
      init(kfull + 8 * a, 32);                  // the MMA warp's lanes (constants copied)
    }
    init(xfull, 128);   // every expander thread
    init(xempty, 1);    // tcgen05.commit after the last image of a round
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kDecEpiWarps + 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // every CTA's barriers exist before anybody's copies or commits reach them
  tc_fence_after();
  const uint32_t tmem0 = (uint32_t)lds_i32(tmem_slot);
  constexpr uint32_t acc0 = H16 ? 96 : 160, ACS = 96;  // the frame tile: 2 DP (<= 80) columns of halves, 4 DP (<= 160) of TF32

  const int G = gridDim.x;
  const int nrounds = (ntiles + G - 1) / G;
  auto tile_of = [&](int r) { return r * G + (int)blockIdx.x; };
  auto rows_of = [&](int r) { const int t = tile_of(r); return t < ntiles ? min(kTcRows, nframes - t * kTcRows) : 0; };

  if (warp == kDecEpiWarps + 5) {
    // =================================== PRODUCER ===================================
    const uint32_t qbytes = img_bytes / kDecCluster;  // a multiple of 16 (img_bytes is a multiple of 64)
    if (lane == 0) {
      int n = 0;
      for (int r = 0; r < nrounds; r++) {
        for (int j = 0; j < nimg; j++, n++) {
          const int s = n % NST;
          mbar_wait_a(empty + 8 * s, ((n / NST) & 1) ^ 1);  // both CTAs have multiplied what the stage held
          mbar_expect_tx_a(full + 8 * s, img_bytes);
          bulk_copy_multicast(Ws + (uint32_t)s * img_bytes + crank * qbytes,
                              reinterpret_cast<const char *>(images) + (size_t)j * img_bytes + (size_t)crank * qbytes, qbytes, full + 8 * s, kMask);
        }
      }
    }
  } else if (warp == kDecEpiWarps + 4) {
    // =================================== MMA ISSUER ===================================
    const uint32_t idesc = H16 ? make_idesc_f16(kTcRows, TN) : make_idesc_tf32(kTcRows, TN);
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem0, 0);
    const int NSLAB = H16 ? KP / 16 : KP / 8;  // K per MMA: 16 halves / 8 TF32 = 8 tensor-memory columns and 256 bytes of a W row group either way
    int n = 0, nu = 0;  // W stage uses; accumulator stage uses (only rounds with a tile)
    for (int r = 0; r < nrounds; r++) {
      const bool have = rows_of(r) > 0;
      if (have) {
        mbar_wait_a(xfull, r & 1);  // the round's frames are in tensor memory
        tc_fence_after();
      }
      for (int j = 0; j < nimg; j++, n++) {
        const int s = n % NST;
        mbar_wait_a(full + 8 * s, (n / NST) & 1);  // the image (both halves) has landed
        if (have) {
          const int a = nu % NA;
          mbar_wait_a(dempty + 8 * a, ((nu / NA) & 1) ^ 1);  // accumulator stage (and its constants) drained by the epilogue
          // the additive constants leave the stage before it is released
          const uint32_t kc_src = Ws + (uint32_t)s * img_bytes + w_bytes;
          for (int c = lane; c < TN; c += 32) skc[a][c] = lds_f32(kc_src + 4 * c);
          mbar_arrive_a(kfull + 8 * a);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint32_t xh = tb, xl = xh + (H16 ? (uint32_t)DP : 80u);
            const uint32_t wbase = Ws + (uint32_t)s * img_bytes;
            const uint64_t wh = make_smem_desc2(wbase, 128, P), wl = make_smem_desc2(wbase + (uint32_t)(TN / 8) * P, 128, P);
            const uint32_t d = tb + acc0 + (uint32_t)a * ACS;
            uint32_t acc = 0;
            for (int p = 0; p < 3; p++) {  // Xh*Wh, Xl*Wh, Xh*Wl
              const uint32_t a0 = (p == 1) ? xl : xh;
              const uint64_t b0 = (p == 2) ? wl : wh;
#pragma unroll 10
              for (int k = 0; k < NSLAB; k++) {
                if (H16) tc_mma_f16_ts(d, a0 + k * 8, b0 + (uint64_t)(k * 16), idesc, acc);
                else tc_mma_tf32_ts(d, a0 + k * 8, b0 + (uint64_t)(k * 16), idesc, acc);
                acc = 1;
              }
            }
            tc_commit_multicast(empty + 8 * s, kMask);  // stage s may be refilled once both CTAs say so
            tc_commit_a(dfull + 8 * a);
            if (j == nimg - 1) tc_commit_a(xempty);  // the frame tile may be replaced
          }
          __syncwarp();
          nu++;
        } else {
          // no tile in this round: nothing reads the stage here, release it straight away
          __syncwarp();
          if (elect_one_sync()) tc_commit_multicast(empty + 8 * s, kMask);
          __syncwarp();
        }
      }
    }
  } else if (warp >= kDecEpiWarps) {
    // =================================== FRAME EXPANDERS (warps 12-15) ===================================
    const int q = warp & 3;
    const int row = 32 * q + lane;  // frame row of the tile = TMEM lane
    const int nq = DP / 4;
    const uint32_t xa0 = tmem0 + ((uint32_t)(32 * q) << 16);
    auto split4 = [](const float4 &v, uint32_t (&hi)[4], uint32_t (&lo)[4]) {
      float hh, ll;
      split_tf32_fast(v.x, hh, ll); hi[0] = __float_as_uint(hh); lo[0] = __float_as_uint(ll);
      split_tf32_fast(v.y, hh, ll); hi[1] = __float_as_uint(hh); lo[1] = __float_as_uint(ll);
      split_tf32_fast(v.z, hh, ll); hi[2] = __float_as_uint(hh); lo[2] = __float_as_uint(ll);
      split_tf32_fast(v.w, hh, ll); hi[3] = __float_as_uint(hh); lo[3] = __float_as_uint(ll);
    };
    for (int r = 0; r < nrounds; r++) {
      const int nrows = rows_of(r);
      if (nrows == 0) continue;
      const int64_t f = fbase + (int64_t)tile_of(r) * kTcRows + row;
      float4 xv[10];
      const float4 *src = reinterpret_cast<const float4 *>(x32 + f * DP);
#pragma unroll
      for (int j = 0; j < 10; j++) xv[j] = (row < nrows && j < nq) ? __ldg(src + j) : make_float4(0.f, 0.f, 0.f, 0.f);
      mbar_wait_a(xempty, (r & 1) ^ 1);  // the MMAs of the previous round have retired (the rows are already in registers)
      tc_fence_after();
      const uint32_t xa = xa0;
      if (H16) {
        // columns: [x' hi | x''^2 hi | x' lo | x''^2 lo], DP / 2 columns (two halves each) per block; 8 dimensions per store
        const int hb = DP / 2;
#pragma unroll
        for (int j = 0; j < 10; j += 2) {
          if (j < nq) {
            const float v[8] = {xv[j].x, xv[j].y, xv[j].z, xv[j].w, xv[j + 1].x, xv[j + 1].y, xv[j + 1].z, xv[j + 1].w};
            uint32_t ah[4], al[4], qh[4], ql[4];
#pragma unroll
            for (int e = 0; e < 4; e++) {
              const int d0 = 4 * j + 2 * e;
              split_half2(v[2 * e] * ssc[0][d0], v[2 * e + 1] * ssc[0][d0 + 1], ah[e], al[e]);
              const float s0 = v[2 * e] * ssc[1][d0], s1 = v[2 * e + 1] * ssc[1][d0 + 1];
              split_half2(s0 * s0, s1 * s1, qh[e], ql[e]);
            }
            tmem_st4(xa + 2 * j, ah);
            tmem_st4(xa + hb + 2 * j, qh);
            tmem_st4(xa + 2 * hb + 2 * j, al);
            tmem_st4(xa + 3 * hb + 2 * j, ql);
          }
        }
      } else {
#pragma unroll
      for (int j = 0; j < 10; j++) {
        if (j < nq) {
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
      mbar_arrive_a(xfull);
    }
  } else {
    // =================================== EPILOGUE (warps 0-11) ===================================
    constexpr int EH = kDecEpiWarps / 4;  // warps per TMEM lane quarter: column groups g with g % EH == h
    const int q = warp & 3, h = warp >> 2;
    const int row = 32 * q + lane;
    const uint32_t trow = (uint32_t)(32 * q) << 16;
    constexpr int SPC = 16 / MP;                      // whole states per 16-column chunk
    constexpr int kMaxG = (kWsMaxTN / 16 + EH - 1) / EH;
    int nu = 0;
    for (int r = 0; r < nrounds; r++) {
      const int nrows = rows_of(r);
      if (nrows == 0) continue;
      const bool live = row < nrows;
      // interleaved output (see dec_logb_index): frame row -> block of 8 frames, 8 consecutive lanes fill one 32-byte sector
      float *lrow0 = logb + ((int64_t)tile_of(r) * (kTcRows / 8) + (row >> 3)) * ldb * 8 + (row & 7);
      for (int j = 0; j < nimg; j++, nu++) {
        const int a = nu % NA;
        const int state0 = j * SCt;
        const int nst = max(0, min(SCt, S_total - state0));  // states present in this image
        const int ngroups = (nst + SPC - 1) / SPC;
        mbar_wait_a(kfull + 8 * a, (nu / NA) & 1);
        mbar_wait_a(dfull + 8 * a, (nu / NA) & 1);
        tc_fence_after();
        const uint32_t d = tmem0 + acc0 + (uint32_t)a * ACS + trow;
        const float4 *kc4 = reinterpret_cast<const float4 *>(skc[a]);  // warp-uniform addresses: broadcast loads
        float *lrow = lrow0 + (int64_t)state0 * 8;
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
            for (int jj = 0; jj < 16; jj++) val[jj] = fmaf(__uint_as_float(v[k][jj]), 1.4426950408889634f, kc[jj]);
            float lbv[SPC];
#pragma unroll
            for (int g = 0; g < SPC; g++) {
              constexpr int MU = MR ? MR : MP;  // columns MU .. MP-1 of a state are pad (density 0)
              if (MU == 1) {
                lbv[g] = val[g * MP] * 0.6931471805599453f;  // -inf stays -inf
              } else {
                // log-sum-exp with ONE guard instruction: the reference point is max(m, -1e30), finite, so a state whose
                // mixtures are all dead (-inf) gives sum = 0 and lg2(0) = -inf on its own -- no select before, none after
                // (k_emis_ws orders the values to save an ex2; here the epilogue is bound by instruction issue, not by the
                // transcendental unit: 16 instead of 23 instructions per state of three mixtures)
                float m = val[g * MP];
#pragma unroll
                for (int jj = 1; jj < MU; jj++) m = fmaxf(m, val[g * MP + jj]);
                const float ms = fmaxf(m, -1e30f);
                float sm_ = ex2_approx(val[g * MP] - ms);
#pragma unroll
                for (int jj = 1; jj < MU; jj++) sm_ += ex2_approx(val[g * MP + jj] - ms);
                float lg;
                asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(sm_));
                lbv[g] = (ms + lg) * 0.6931471805599453f;
              }
            }
            float *dst = lrow + c * SPC * 8;
            if (live) {
#pragma unroll
              for (int g = 0; g < SPC; g++)
                if (c * SPC + g < nst) dst[g * 8] = lbv[g];
            }
          }
        }
        tc_fence_before();
        mbar_arrive_a(dempty + 8 * a);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // nobody leaves while a peer may still write into its shared memory or signal its barriers
  tc_fence_after();
  if (warp == kDecEpiWarps + 4) tmem_dealloc(tmem0, 512);
}

}  // namespace hmmk
