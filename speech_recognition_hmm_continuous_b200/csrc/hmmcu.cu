// hmmcu.cu -- the C ABI of include/hmm_cuda.h over the kernels in kernels.cuh.
// One context = one device + one stream; all work is enqueued on that stream and the entry
// points that return host data synchronise it.  There is no CPU fallback anywhere in this file.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "hmm_cuda.h"
#include "kernels.cuh"
#include "fb_kernels.cuh"
#include "fbres_kernels.cuh"
#include "tc_kernels.cuh"
#include "ws_kernels.cuh"
#include "dec_kernels.cuh"
#include "acch_kernels.cuh"
#include "vit_kernels.cuh"
#include "vtrain_kernels.cuh"
#include "init_kernels.cuh"

using namespace hmmk;

namespace {

char g_create_err[512] = "";
std::atomic<uint64_t> g_alloc_epoch{0};  // bumped whenever a device buffer moves (any context, any host thread): cached CUDA graphs hold raw pointers

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    g_alloc_epoch++;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) { cudaFree(p); g_alloc_epoch++; }
    p = nullptr;
    cap = 0;
  }
  template <typename T> T *as() { return reinterpret_cast<T *>(p); }
};

struct Timer {
  cudaEvent_t a = nullptr, b = nullptr;
  bool used = false;
  // every begin / end pair since the last reset (a call that works in batches, hmmcu_forward_scores): "<name>_total"
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pairs;
  size_t npairs = 0;
  bool collect = false;
};

// A launch sequence captured once and replayed: the EM iteration is a dozen short kernels, and launching
// them one by one costs more host time than they run.
struct GraphSlot {
  cudaGraphExec_t exec = nullptr;
  uint64_t key = 0;
  int seen = 0;
  int64_t nlaunch = 0;
  bool bad = false;
};

}  // namespace

struct hmmcu_ctx {
  int dev = 0;
  cudaStream_t st = nullptr;
  // multi-stream models (hmmcu_link_streams): the further feature streams of this (primary) context, and on a linked
  // context its primary.  Linked contexts run on the primary's CUDA stream; st_own is the stream to destroy.
  cudaStream_t st_own = nullptr;
  std::vector<hmmcu_ctx *> linked;
  hmmcu_ctx *primary = nullptr;
  DevBuf logb_joint;  // sum over the streams of the log-emissions [F][N] (training)
  // feature upload pipeline: chunk copies on their own stream, packed on `st` as they land
  cudaStream_t st_copy = nullptr;
  // side branches of the M-step launch sequence (the accuracy-guard scan and one of the two W packers run beside the
  // main chain; fork / join by events, inside the captured graph as well)
  cudaStream_t st_aux[2] = {};
  cudaEvent_t ev_fork[2] = {}, ev_join[2] = {};
  static constexpr int kUpChunks = 16;
  int up_chunks = 4;         // "upload_chunks" option
  cudaEvent_t ev_chunk[kUpChunks] = {};
  cudaEvent_t ev_idle = nullptr;
  bool stream_open = false;  // between hmmcu_features_begin and _end
  bool mstep_fork = true;    // "mstep_fork" option: side streams inside the M-step launch sequence
  void *stage_h[4] = {};     // pinned staging buffers of the ingest pipeline (hmmcu_staging), kept for the context's life
  size_t stage_cap[4] = {};
  int64_t stream_frames = 0;
  int stream_next = 0;
  double *ctr_h = nullptr;  // pinned [256]
  char err[512] = "";
  int64_t launches = 0;
  int sm_count = 148;
  bool timing = false;
  int use_graph = 1;          // replay the E-step / M-step launch sequences as CUDA graphs ("graphs" option)
  uint64_t cfg_epoch = 0;     // bumped by everything that changes what those sequences launch
  GraphSlot g_estep, g_estep_vit, g_mstep;  // g_estep_vit: the E-step with the Viterbi alignment (hmmcu_estep_viterbi)
  int train_path = 0;         // emission / accumulate path of the last E-step: 0 CUDA cores, 1 k_emis_tc, 2 warp-specialised
  std::map<std::string, Timer> timers;

  // features
  int U = 0, D = 0, DP = 0, Tmax = 0;
  int64_t F = 0;
  bool have_features = false;
  DevBuf x64_own;            // when uploaded from the host
  const double *d_x64 = nullptr;
  DevBuf x32, ctr, off_d, xabs_d;
  std::vector<int64_t> off;
  double kappa = 0.0;          // bound on the summed magnitude of the expanded quadratic's terms
  bool kappa_stale = true;     // features or models changed since kappa was last read back
  // device-resident EM control (hmmcu_em_reset / hmmcu_mstep)
  DevBuf em_old, em_active, ctl_d, ext_d, upd_d;
  double *ctl_h = nullptr;     // pinned: [3V + 1] sum_logp, n_utt, updated, kappa
  size_t ctl_cap = 0;

  // models
  int V = 0, N = 0, M = 0, G = 0, Dm = 0;
  bool have_models = false, pack_dirty = true;
  bool banded = false;  // every A is upper-bidiagonal (the left-to-right DELTA=1 topology of T-FS:774-795)
  DevBuf A, c, mu, iv, det, mu32, iv32, k32, kc2;
  bool kc_dirty = true, simt_dirty = true;

  // training map
  std::vector<int32_t> u2m;
  DevBuf u2m_d, mus_d, mu_d, tiles_d;
  DevBuf vit_map, vit_tiles;
  std::vector<int32_t> vit_u2m;
  int64_t n_vit_tiles = 0;
  uint64_t feat_epoch = 1, vit_epoch = 0;  // feat_epoch: bumped when the utterance geometry changes
  int32_t *path_h = nullptr;   // pinned staging for hmmcu_viterbi's path
  size_t path_h_cap = 0;
  DevBuf in_lst, in_off, in_vk, in_cent, in_sum, in_dist, in_cnt, in_idx, in_dd, in_ord;  // initial-model builder  // utt2model, model_utt_start, model_utts, emission tiles
  int64_t n_train_tiles = 0;
  int max_utts_per_model = 0;

  // tensor-core emission path (tc_kernels.cuh)
  int use_tc = 1;
  bool last_tc = false;   // whether the most recent emission launch used the tensor-core kernel
  struct TcSet {
    DevBuf images, kc, s0, ns;
    std::vector<int32_t> s0_h, ns_h;  // what the device tables hold
    int TN = 0, SCt = 0, nimg = 0;
    DevBuf images16, scales16;  // half-precision images of k_emis_dec (decode set only)
    bool dirty = true;
  } tc_train, tc_dec, ws_train, ws_dec;
  int use_ws = 1;  // warp-specialised pipelined emission kernel (0 = the single-buffered k_emis_tc)
  DevBuf tc_tiles_train, frame_ids_d, tc_tiles_dec, ws_tiles_train;
  int64_t n_tc_tiles_train = 0, n_ws_tiles_train = 0;
  // tensor-core accumulate kernel: W images per (model, block of 128 Gaussians) and its work units
  DevBuf acc_images, acc_kc, acc_units, acc_units64, acc_scratch, acc_slot_start, acc_slot_ids;
  int64_t n_acc_units64 = 0;
  int use_ws_acc = 1;  // warp-specialised accumulate kernel (0 = k_accum_tc)
  // k_accum_h (acch_kernels.cuh): half-precision operands, the expanded frame tiles of all units packed once per feature set
  int use_h_acc = 1;
  DevBuf acc_images16, acc_sc, acc_unitsH, acc_slot_start_h, acc_slot_ids_h, x16, x16_tiles;
  int64_t n_acc_unitsH = 0, n_x16_tiles = 0;
  uint64_t x_version = 1, map_version = 1, x16_x = 0, x16_map = 0;  // what x16 was packed from
  int use_dec_emis = 1;  // decode emissions with the frames resident in tensor memory and the W images multicast over a cluster (k_emis_dec)
  int dec_f16 = 1;       // decode emission kernels with half-precision operands (kind::f16 MMAs at twice the TF32 rate)
  int dec_budget_kb = 0; // log-emission budget of a decode batch in KiB (0 = 6 GiB or a third of the free memory); tests
  bool last_acc_h = false;  // the last accumulate launch was k_accum_h
  bool last_dec16 = false;  // the last decode emission launch (k_emis_dec / k_emis_ws<false>) used half-precision operands
  int dec_grid = 0;      // CTAs of k_emis_dec (whole clusters that fit the device at once), 0 = not asked yet
  int use_res_fb = 1;  // shared-memory-resident forward-backward (k_fb_res) whenever the utterances fit and A is banded
  DevBuf res_order, res_upos, res_batches, res_counter, ustats;
  // peer all-reduce over NVLink (hmmcu_peer_*): my receive area of tagged words [2 slot sets][world][stats_n] x 16 B;
  // the areas of all ranks as mapped here; the iteration counter lives on the device
  DevBuf peer_area, peer_ptrs_d, peer_seq_d;
  std::vector<void *> peer_ptrs;        // [world], entry `rank` = my own area
  std::vector<void *> peer_opened;      // IPC mappings to close
  int peer_rank = -1, peer_world = 0;
  int64_t peer_n = 0;                   // doubles per slot the area was sized for
  int64_t n_res_batches = 0;
  int res_batch_max = 0;  // the most utterances in one of those batches
  int n_live = 0;         // utterances of the training map that belong to a model (the others are masked)
  bool res_fits = false;  // every utterance of the training map fits one team's shared memory
  bool acc_dirty = true;
  int64_t n_acc_units = 0;

  // workspaces
  DevBuf logb, logb64, post, gamma, alpha_ws, beta_ws, stats, logp_utt_d, score_d, psi_ws, path_d, tiles_dec, rank_in, rank_out;
  int64_t stats_n = 0;
};

// k_fb_res takes the forward-backward of the current training map (otherwise k_fb does)
static bool res_fb_on(const hmmcu_ctx *ctx) { return ctx->use_res_fb && ctx->banded && ctx->res_fits && ctx->n_res_batches > 0; }
// CTAs of its launch: one per SM at most, none without a batch
static int res_grid(const hmmcu_ctx *ctx) { return (int)std::min<int64_t>(ctx->n_res_batches, ctx->sm_count); }

static int fail(hmmcu_ctx *c, int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(c ? c->err : g_create_err, 512, fmt, ap);
  va_end(ap);
  return code;
}

#define CK(call)                                                                                    \
  do {                                                                                              \
    cudaError_t e_ = (call);                                                                        \
    if (e_ != cudaSuccess)                                                                          \
      return fail(ctx, e_ == cudaErrorMemoryAllocation ? HMMCU_ENOMEM : HMMCU_ECUDA, "%s failed: %s (%s:%d)", #call, \
                  cudaGetErrorString(e_), __FILE__, __LINE__);                                      \
  } while (0)

#define LAUNCH_CHECK()                                                                              \
  do {                                                                                              \
    ctx->launches++;                                                                                \
    cudaError_t e_ = cudaGetLastError();                                                            \
    if (e_ != cudaSuccess)                                                                          \
      return fail(ctx, HMMCU_ECUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

// A launch with programmatic dependent launch: the kernel may be scheduled as soon as every CTA of the previous kernel
// of the stream has called pdl_trigger() or exited, and its CTAs run up to pdl_wait() (kernels.cuh) meanwhile.  Only
// for kernels that call pdl_wait() in every CTA before they touch what an earlier kernel wrote.  Under stream capture
// the edge from the previous kernel node becomes a programmatic edge of the graph.
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = &attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

static void t_begin(hmmcu_ctx *ctx, const char *name) {
  if (!ctx->timing) return;
  Timer &t = ctx->timers[name];
  if (t.collect) {
    if (t.npairs == t.pairs.size()) {
      std::pair<cudaEvent_t, cudaEvent_t> pr;
      cudaEventCreate(&pr.first);
      cudaEventCreate(&pr.second);
      t.pairs.push_back(pr);
    }
    cudaEventRecord(t.pairs[t.npairs].first, ctx->st);
    return;
  }
  if (!t.a) {
    cudaEventCreate(&t.a);
    cudaEventCreate(&t.b);
  }
  cudaEventRecord(t.a, ctx->st);
}
static void t_end(hmmcu_ctx *ctx, const char *name) {
  if (!ctx->timing) return;
  Timer &t = ctx->timers[name];
  if (t.collect) {
    cudaEventRecord(t.pairs[t.npairs++].second, ctx->st);
    t.used = true;
    return;
  }
  cudaEventRecord(t.b, ctx->st);
  t.used = true;
}
// back to one begin / end pair per call
static void t_single(hmmcu_ctx *ctx, const char *name) {
  if (!ctx->timing) return;
  ctx->timers[name].collect = false;
}
// start collecting every begin / end pair of `name` (until the next call of this)
static void t_collect(hmmcu_ctx *ctx, const char *name) {
  if (!ctx->timing) return;
  Timer &t = ctx->timers[name];
  t.collect = true;
  t.npairs = 0;
}


// enqueue() issues a fixed launch sequence on ctx->st.  The first two calls under a key run it directly (lazy
// allocations and function attributes settle), the third captures it, later ones replay the graph.
template <typename F>
static int run_graphed(hmmcu_ctx *ctx, GraphSlot &gs, uint64_t key, F &&enqueue) {
  // (per-kernel timing records events between the kernels; events recorded by graph nodes cannot be timed)
  if (!ctx->use_graph || ctx->timing || gs.bad) return enqueue();
  key = key * 0x9E3779B97F4A7C15ull + g_alloc_epoch.load() * 1000003ull + ctx->cfg_epoch;
  if (gs.key != key) {
    if (gs.exec) cudaGraphExecDestroy(gs.exec);
    gs.exec = nullptr;
    gs.key = key;
    gs.seen = 0;
  }
  if (gs.exec) {
    CK(cudaGraphLaunch(gs.exec, ctx->st));
    ctx->launches += gs.nlaunch;
    return HMMCU_OK;
  }
  if (++gs.seen < 3) return enqueue();
  const int64_t l0 = ctx->launches;
  if (cudaStreamBeginCapture(ctx->st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
    cudaGetLastError();
    gs.bad = true;
    return enqueue();
  }
  const int rc = enqueue();
  cudaGraph_t g = nullptr;
  cudaError_t e = cudaStreamEndCapture(ctx->st, &g);
  if (rc == HMMCU_OK && e == cudaSuccess && g) e = cudaGraphInstantiate(&gs.exec, g, 0);
  if (g) cudaGraphDestroy(g);
  if (rc != HMMCU_OK || e != cudaSuccess || !gs.exec) {  // not capturable here: run it the plain way from now on
    cudaGetLastError();
    gs.exec = nullptr;
    gs.bad = true;
    ctx->launches = l0;
    return rc != HMMCU_OK ? rc : enqueue();
  }
  gs.nlaunch = ctx->launches - l0;
  CK(cudaGraphLaunch(gs.exec, ctx->st));
  return HMMCU_OK;
}

int hmmcu_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int hmmcu_create(int device, hmmcu_ctx **out) {
  if (!out) return fail(nullptr, HMMCU_EINVAL, "hmmcu_create: out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(nullptr, HMMCU_ENODEV, "no CUDA device (%s); this library has no CPU path",
                e == cudaSuccess ? "count is 0" : cudaGetErrorString(e));
  if (device < 0 || device >= n) return fail(nullptr, HMMCU_EINVAL, "device %d out of range (%d present)", device, n);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
    return fail(nullptr, HMMCU_ECUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, HMMCU_ENODEV, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major,
                prop.minor);
  hmmcu_ctx *ctx = new hmmcu_ctx();
  ctx->dev = device;
  ctx->sm_count = prop.multiProcessorCount;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&ctx->st, cudaStreamNonBlocking)) != cudaSuccess) {
    fail(nullptr, HMMCU_ECUDA, "stream creation: %s", cudaGetErrorString(e));
    delete ctx;
    return HMMCU_ECUDA;
  }
  ctx->st_own = ctx->st;
  bool ok = cudaStreamCreateWithFlags(&ctx->st_copy, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&ctx->ev_idle, cudaEventDisableTiming) == cudaSuccess &&
            cudaMallocHost((void **)&ctx->ctr_h, sizeof(double) * 256) == cudaSuccess;
  for (int k = 0; ok && k < hmmcu_ctx::kUpChunks; k++) ok = cudaEventCreateWithFlags(&ctx->ev_chunk[k], cudaEventDisableTiming) == cudaSuccess;
  for (int k = 0; ok && k < 2; k++)
    ok = cudaStreamCreateWithFlags(&ctx->st_aux[k], cudaStreamNonBlocking) == cudaSuccess &&
         cudaEventCreateWithFlags(&ctx->ev_fork[k], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&ctx->ev_join[k], cudaEventDisableTiming) == cudaSuccess;
  if (!ok) {
    fail(nullptr, HMMCU_ECUDA, "upload pipeline creation: %s", cudaGetErrorString(cudaGetLastError()));
    hmmcu_destroy(ctx);
    return HMMCU_ECUDA;
  }
  *out = ctx;
  return HMMCU_OK;
}

static void unlink_streams(hmmcu_ctx *ctx) {
  if (ctx->primary) {  // a linked context leaves its primary
    auto &l = ctx->primary->linked;
    l.erase(std::remove(l.begin(), l.end(), ctx), l.end());
    cudaStreamSynchronize(ctx->st);
    ctx->st = ctx->st_own;
    ctx->primary = nullptr;
  }
  for (hmmcu_ctx *q : ctx->linked) {  // a primary releases its streams
    cudaStreamSynchronize(ctx->st);
    q->st = q->st_own;
    q->primary = nullptr;
  }
  ctx->linked.clear();
}

void hmmcu_destroy(hmmcu_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->dev);
  cudaStreamSynchronize(ctx->st);
  unlink_streams(ctx);
  for (void *p : ctx->peer_opened) cudaIpcCloseMemHandle(p);
  ctx->peer_area.release(); ctx->peer_ptrs_d.release(); ctx->peer_seq_d.release();
  ctx->logb_joint.release();
  DevBuf *bufs[] = {&ctx->x64_own, &ctx->x32, &ctx->ctr, &ctx->off_d, &ctx->A, &ctx->c, &ctx->mu, &ctx->iv, &ctx->det,
                    &ctx->mu32, &ctx->iv32, &ctx->k32, &ctx->kc2, &ctx->u2m_d, &ctx->mus_d, &ctx->mu_d, &ctx->tiles_d, &ctx->logb,
                    &ctx->post, &ctx->gamma, &ctx->alpha_ws, &ctx->stats, &ctx->logp_utt_d, &ctx->score_d,
                    &ctx->psi_ws, &ctx->path_d, &ctx->tiles_dec, &ctx->rank_in, &ctx->rank_out, &ctx->tc_train.images, &ctx->tc_train.kc, &ctx->tc_train.s0,
                    &ctx->tc_train.ns, &ctx->xabs_d, &ctx->tc_dec.images, &ctx->tc_dec.kc, &ctx->tc_dec.s0, &ctx->tc_dec.ns, &ctx->tc_tiles_train,
                    &ctx->frame_ids_d, &ctx->tc_tiles_dec, &ctx->acc_images, &ctx->acc_kc, &ctx->acc_units, &ctx->beta_ws, &ctx->em_old, &ctx->em_active, &ctx->ctl_d, &ctx->ext_d, &ctx->upd_d, &ctx->ws_train.images, &ctx->ws_train.s0, &ctx->ws_train.ns,
                    &ctx->ws_dec.images, &ctx->ws_dec.images16, &ctx->ws_dec.scales16, &ctx->ws_dec.s0, &ctx->ws_dec.ns, &ctx->ws_tiles_train, &ctx->acc_units64, &ctx->logb64, &ctx->acc_scratch, &ctx->acc_slot_start, &ctx->acc_slot_ids, &ctx->in_lst, &ctx->in_off, &ctx->in_vk, &ctx->in_cent,
                    &ctx->in_sum, &ctx->in_dist, &ctx->in_cnt, &ctx->in_idx, &ctx->in_dd, &ctx->in_ord, &ctx->vit_map, &ctx->vit_tiles,
                    &ctx->res_order, &ctx->res_upos, &ctx->res_batches, &ctx->res_counter, &ctx->ustats,
                    &ctx->acc_images16, &ctx->acc_sc, &ctx->acc_unitsH, &ctx->acc_slot_start_h, &ctx->acc_slot_ids_h, &ctx->x16, &ctx->x16_tiles};
  for (DevBuf *b : bufs) b->release();
  for (auto &kv : ctx->timers) {
    if (kv.second.a) cudaEventDestroy(kv.second.a);
    if (kv.second.b) cudaEventDestroy(kv.second.b);
    for (auto &pr : kv.second.pairs) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
  }
  if (ctx->g_estep.exec) cudaGraphExecDestroy(ctx->g_estep.exec);
  if (ctx->g_estep_vit.exec) cudaGraphExecDestroy(ctx->g_estep_vit.exec);
  if (ctx->g_mstep.exec) cudaGraphExecDestroy(ctx->g_mstep.exec);
  if (ctx->ctl_h) cudaFreeHost(ctx->ctl_h);
  if (ctx->ctr_h) cudaFreeHost(ctx->ctr_h);
  if (ctx->path_h) cudaFreeHost(ctx->path_h);
  for (cudaEvent_t e : ctx->ev_chunk)
    if (e) cudaEventDestroy(e);
  if (ctx->ev_idle) cudaEventDestroy(ctx->ev_idle);
  for (void *p : ctx->stage_h)
    if (p) cudaFreeHost(p);
  if (ctx->st_copy) cudaStreamDestroy(ctx->st_copy);
  for (int k = 0; k < 2; k++) {
    if (ctx->ev_fork[k]) cudaEventDestroy(ctx->ev_fork[k]);
    if (ctx->ev_join[k]) cudaEventDestroy(ctx->ev_join[k]);
    if (ctx->st_aux[k]) cudaStreamDestroy(ctx->st_aux[k]);
  }
  cudaStreamDestroy(ctx->st_own);
  delete ctx;
}

const char *hmmcu_last_error(const hmmcu_ctx *ctx) { return ctx ? ctx->err : g_create_err; }
void *hmmcu_stream(hmmcu_ctx *ctx) { return ctx ? (void *)ctx->st : nullptr; }
int hmmcu_synchronize(hmmcu_ctx *ctx) {
  CK(cudaSetDevice(ctx->dev));
  CK(cudaStreamSynchronize(ctx->st));
  return HMMCU_OK;
}
int hmmcu_host_alloc(void **p, uint64_t bytes) { return cudaMallocHost(p, bytes) == cudaSuccess ? HMMCU_OK : HMMCU_ENOMEM; }
void hmmcu_host_free(void *p) {
  if (p) cudaFreeHost(p);
}
int64_t hmmcu_launch_count(const hmmcu_ctx *ctx) { return ctx ? ctx->launches : 0; }
void hmmcu_enable_timing(hmmcu_ctx *ctx, int on) { ctx->timing = on != 0; ctx->cfg_epoch++; }
double hmmcu_last_kernel_ms(const hmmcu_ctx *ctx, const char *name) {
  if (strcmp(name, "kappa") == 0) return ctx->kappa;            // accuracy-guard value of the current pack
  if (strcmp(name, "tc_active") == 0) return ctx->last_tc ? 1.0 : 0.0;
  if (strcmp(name, "dec_f16_active") == 0) return ctx->last_dec16 ? 1.0 : 0.0;
  if (strcmp(name, "acc_h_active") == 0) return ctx->last_acc_h ? 1.0 : 0.0;
  if (strcmp(name, "dec_grid") == 0) return (double)ctx->dec_grid;                // CTAs of the last k_emis_dec launch configuration
  // the k_fb_res batches of the current training map: how many, the most utterances in one, the teams that claim them
  if (strcmp(name, "res_batches") == 0) return res_fb_on(ctx) ? (double)ctx->n_res_batches : 0.0;
  if (strcmp(name, "res_batch_max") == 0) return res_fb_on(ctx) ? (double)ctx->res_batch_max : 0.0;
  if (strcmp(name, "res_teams") == 0) return res_fb_on(ctx) ? (double)(kResTeams * res_grid(ctx)) : 0.0;
  {  // "<name>_total": the sum over the batches of the last hmmcu_forward_scores / hmmcu_viterbi_scores call
    const size_t ln = strlen(name);
    if (ln > 6 && strcmp(name + ln - 6, "_total") == 0) {
      auto itt = ctx->timers.find(std::string(name, ln - 6));
      if (itt == ctx->timers.end() || !itt->second.used) return -1.0;
      const Timer &t = itt->second;
      if (!t.collect) return hmmcu_last_kernel_ms(ctx, std::string(name, ln - 6).c_str());
      double tot = 0.0;
      for (size_t k = 0; k < t.npairs; k++) {
        float ms1 = 0.f;
        if (cudaEventSynchronize(t.pairs[k].second) != cudaSuccess || cudaEventElapsedTime(&ms1, t.pairs[k].first, t.pairs[k].second) != cudaSuccess) {
          cudaGetLastError();
          return -1.0;
        }
        tot += ms1;
      }
      return tot;
    }
  }
  auto it = ctx->timers.find(name);
  if (it == ctx->timers.end() || !it->second.used) return -1.0;
  if (it->second.collect) {  // the last pair
    const Timer &t = it->second;
    float ms1 = 0.f;
    if (t.npairs == 0 || cudaEventSynchronize(t.pairs[t.npairs - 1].second) != cudaSuccess ||
        cudaEventElapsedTime(&ms1, t.pairs[t.npairs - 1].first, t.pairs[t.npairs - 1].second) != cudaSuccess) {
      cudaGetLastError();
      return -1.0;
    }
    return (double)ms1;
  }
  float ms = 0.f;
  if (cudaEventSynchronize(it->second.b) != cudaSuccess || cudaEventElapsedTime(&ms, it->second.a, it->second.b) != cudaSuccess) {
    cudaGetLastError();
    return -1.0;
  }
  return (double)ms;
}
int hmmcu_set_option(hmmcu_ctx *ctx, const char *key, int value) {
  if (!ctx || !key) return HMMCU_EINVAL;
  ctx->cfg_epoch++;
  if (strcmp(key, "graphs") == 0) { ctx->use_graph = value; return HMMCU_OK; }
  if (strcmp(key, "mstep_fork") == 0) { ctx->mstep_fork = value != 0; return HMMCU_OK; }
  if (strcmp(key, "upload_chunks") == 0) { ctx->up_chunks = std::max(1, std::min(value, hmmcu_ctx::kUpChunks)); return HMMCU_OK; }
  if (strcmp(key, "tc_emis") == 0) { ctx->use_tc = value; return HMMCU_OK; }
  if (strcmp(key, "ws_emis") == 0) { ctx->use_ws = value; return HMMCU_OK; }
  if (strcmp(key, "ws_acc") == 0) { ctx->use_ws_acc = value; ctx->acc_dirty = true; return HMMCU_OK; }
  if (strcmp(key, "h_acc") == 0) { ctx->use_h_acc = value; ctx->acc_dirty = true; return HMMCU_OK; }
  if (strcmp(key, "res_fb") == 0) { ctx->use_res_fb = value; return HMMCU_OK; }
  if (strcmp(key, "dec_f16") == 0) { ctx->dec_f16 = value; ctx->ws_dec.dirty = true; return HMMCU_OK; }
  if (strcmp(key, "dec_budget_kb") == 0) { ctx->dec_budget_kb = value; return HMMCU_OK; }
  if (strcmp(key, "dec_emis") == 0) { ctx->use_dec_emis = value; return HMMCU_OK; }
  return fail(ctx, HMMCU_EINVAL, "unknown option %s", key);
}
int64_t hmmcu_stats_size(int N, int M, int D) {
  return (int64_t)N * N + 2 * N + (int64_t)N * M + 2 * (int64_t)N * M * D + 2;
}

// --------------------------------------------------------------------------- feature streams ----
// Multi-stream models (param_number > 1, T-FS:1406-1409 / R-FS:341-364): b_i(t) is the PRODUCT of the per-stream
// mixture densities.  Every stream lives in its own context (own features, own mixtures, the same A, the same
// utterance geometry); linking makes `primary` add the log-emissions of the others before its recursions, and makes
// the others accumulate their mixture statistics with the primary's state posteriors.  n = 0 unlinks.
int hmmcu_link_streams(hmmcu_ctx *primary, hmmcu_ctx *const *others, int n) {
  if (!primary || n < 0 || (n > 0 && !others)) return HMMCU_EINVAL;
  if (primary->primary) return fail(primary, HMMCU_EINVAL, "link_streams: this context is itself linked to another");
  hmmcu_ctx *ctx = primary;  // for CK
  CK(cudaSetDevice(primary->dev));
  unlink_streams(primary);
  for (int k = 0; k < n; k++) {
    hmmcu_ctx *q = others[k];
    if (!q || q == primary || q->primary || !q->linked.empty() || q->dev != primary->dev) {
      unlink_streams(primary);
      return fail(primary, HMMCU_EINVAL, "link_streams: stream %d must be another, unlinked context on the same device", k + 1);
    }
    CK(cudaStreamSynchronize(q->st));
    q->st = primary->st;
    q->primary = primary;
    primary->linked.push_back(q);
  }
  return HMMCU_OK;
}

// the linked contexts must describe the same utterances and the same model topology as their primary
static int check_linked(hmmcu_ctx *ctx) {
  for (hmmcu_ctx *q : ctx->linked) {
    if (!q->have_features || !q->have_models) return fail(ctx, HMMCU_EINVAL, "a linked stream has no features or models");
    if (q->U != ctx->U || q->off != ctx->off) return fail(ctx, HMMCU_EINVAL, "linked streams differ in their utterance lengths");
    if (q->V != ctx->V || q->N != ctx->N) return fail(ctx, HMMCU_EINVAL, "linked streams differ in words or states (V=%d/%d, N=%d/%d)", ctx->V, q->V, ctx->N, q->N);
  }
  return HMMCU_OK;
}

// flush_a / flush_b: the operand is ONE stream's log-density and the reference's linear-domain density underflows to exactly 0
// below DBL_TRUE_MIN (it flushes every stream's symbol_probab on its own before multiplying them, R-FS:341-367)
__global__ void k_add_logb(float *__restrict__ out, const float *__restrict__ a, const float *__restrict__ b, int64_t n, int flush_a = 0,
                           int flush_b = 0) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float x = a[i], y = b[i];
    if (flush_a && (double)x < kLogTrueMin) x = kNegInf;
    if (flush_b && (double)y < kLogTrueMin) y = kNegInf;
    out[i] = x + y;
  }
}
// the per-word statistics every stream shares: [num_trans N*N, den_trans N, den_mix N] at the head, [sum_logP, n_utt] at the tail
__global__ void k_copy_shared_stats(double *__restrict__ dst, int64_t ss_dst, const double *__restrict__ src, int64_t ss_src, int V, int head) {
  const int v = blockIdx.x;
  if (v >= V) return;
  for (int k = threadIdx.x; k < head + 2; k += blockDim.x) {
    if (k < head) dst[v * ss_dst + k] = src[v * ss_src + k];
    else dst[v * ss_dst + ss_dst - 2 + (k - head)] = src[v * ss_src + ss_src - 2 + (k - head)];
  }
}

// ---------------------------------------------------------------------------------- features ----
// geometry of a new feature set: validation, offsets, buffers (shared by the one-shot and the streaming upload)
static int features_geometry(hmmcu_ctx *ctx, const int64_t *frame_off, int U, int D) {
  const int DP = round_up(D + 1, 4);
  if (DP > 256) return fail(ctx, HMMCU_EINVAL, "set_features: D=%d too large (max 251)", D);
  if (frame_off[0] != 0) return fail(ctx, HMMCU_EINVAL, "set_features: frame_off[0] must be 0");
  int Tmax = 0;
  for (int u = 0; u < U; u++) {
    int64_t T = frame_off[u + 1] - frame_off[u];
    if (T < 1 || T > (1 << 30)) return fail(ctx, HMMCU_EINVAL, "set_features: utterance %d has %lld frames", u, (long long)T);
    Tmax = std::max(Tmax, (int)T);
  }
  CK(cudaSetDevice(ctx->dev));
  const int64_t F = U > 0 ? frame_off[U] : 0;
  // frame ids are 32-bit on the device (frame_ids, tile rows): 2^31 frames would be 172 GB of doubles at D = 10 already
  if (F > (int64_t)INT32_MAX - 4096) return fail(ctx, HMMCU_EINVAL, "set_features: %lld frames in one feature set (max 2^31 - 4096 per context)", (long long)F);
  // same utterance geometry as before (the trainer re-reading its feature files every iteration,
  // T-FS:272-321): the training map built from it stays valid
  const bool same_geometry = ctx->have_features && ctx->U == U && ctx->D == D && (int)ctx->off.size() == U + 1 &&
                             memcmp(ctx->off.data(), frame_off, sizeof(int64_t) * (U + 1)) == 0;
  ctx->U = U; ctx->D = D; ctx->DP = DP; ctx->F = F; ctx->Tmax = Tmax;
  if (!same_geometry) {
    ctx->off.assign(frame_off, frame_off + U + 1);
    ctx->u2m.clear();
    ctx->cfg_epoch++;
    ctx->feat_epoch++;
  }
  ctx->pack_dirty = true;  // the centre may move
  ctx->kappa_stale = true;
  ctx->have_features = true;
  ctx->x_version++;
  ctx->stream_open = false;
  if (F == 0) return HMMCU_OK;
  CK(ctx->off_d.ensure(sizeof(int64_t) * (U + 1)));
  if (!same_geometry) CK(cudaMemcpyAsync(ctx->off_d.p, ctx->off.data(), sizeof(int64_t) * (U + 1), cudaMemcpyHostToDevice, ctx->st));
  CK(ctx->x32.ensure(sizeof(float) * F * DP));
  CK(ctx->ctr.ensure(sizeof(double) * DP));
  CK(ctx->xabs_d.ensure(sizeof(unsigned int) * DP));
  return HMMCU_OK;
}

static int pack_range(hmmcu_ctx *ctx, int64_t f0, int64_t f1) {
  const int D = ctx->D, DP = ctx->DP;
  const int64_t total = (f1 - f0) * DP;
  const int blocks = (int)std::min<int64_t>((total + 255) / 256, (int64_t)ctx->sm_count * 16);
  k_pack_features<<<blocks, 256, 0, ctx->st>>>(ctx->d_x64 + f0 * D, ctx->ctr.as<double>(), f1 - f0, D, DP, ctx->x32.as<float>() + f0 * DP,
                                              ctx->xabs_d.as<unsigned int>());
  LAUNCH_CHECK();
  return HMMCU_OK;
}

// centre + packed fp32 rows from fp64 features already in device memory
static int pack_from_device(hmmcu_ctx *ctx) {
  t_begin(ctx, "pack");
  k_center<<<1, 1024, 0, ctx->st>>>(ctx->d_x64, ctx->F, ctx->D, ctx->DP, ctx->ctr.as<double>());
  LAUNCH_CHECK();
  CK(cudaMemsetAsync(ctx->xabs_d.p, 0, sizeof(unsigned int) * ctx->DP, ctx->st));
  int rc = pack_range(ctx, 0, ctx->F);
  if (rc) return rc;
  t_end(ctx, "pack");
  return HMMCU_OK;
}

static int set_features_common(hmmcu_ctx *ctx, const double *x_host, const double *x_dev, const int64_t *frame_off,
                               int U, int D) {
  if (!ctx) return HMMCU_EINVAL;
  if (U < 0 || D < 1 || !frame_off || (U > 0 && !x_host && !x_dev)) return fail(ctx, HMMCU_EINVAL, "set_features: bad arguments");
  int rc0 = features_geometry(ctx, frame_off, U, D);
  if (rc0) return rc0;
  const int DP = ctx->DP;
  const int64_t F = ctx->F;
  if (F == 0) return HMMCU_OK;
  if (x_host) {
    // Upload pipeline: the copy engine streams the frames in chunks on its own stream while the host
    // forms the centre from the same strided sample k_center takes (same summation order), and `st`
    // packs every chunk as soon as it has landed.  The copy and the packing overlap; only the last
    // chunk's packing is exposed.
    CK(ctx->x64_own.ensure(sizeof(double) * F * D));
    ctx->d_x64 = ctx->x64_own.as<double>();
    CK(cudaEventRecord(ctx->ev_idle, ctx->st));            // earlier kernels may still read the old features
    CK(cudaStreamWaitEvent(ctx->st_copy, ctx->ev_idle, 0));
    // A few chunks of halving size (1/2, 1/4, ..): every chunk boundary costs the copy engine a few microseconds
    // (measured: 16 equal chunks are 60 us slower end to end than 2-4), and only the last chunk's packing is exposed.
    const int nch = (int)std::max<int64_t>(1, std::min<int64_t>(ctx->up_chunks, F / 4096));
    int64_t cb[hmmcu_ctx::kUpChunks + 1];
    cb[0] = 0;
    for (int k = 1; k < nch; k++) cb[k] = cb[k - 1] + (F - cb[k - 1]) / 2;
    cb[nch] = F;
    for (int k = 0; k < nch; k++) {
      const int64_t f0 = cb[k], f1 = cb[k + 1];
      if (f1 > f0) CK(cudaMemcpyAsync(ctx->x64_own.as<double>() + f0 * D, x_host + f0 * D, sizeof(double) * (f1 - f0) * D, cudaMemcpyHostToDevice, ctx->st_copy));
      CK(cudaEventRecord(ctx->ev_chunk[k], ctx->st_copy));
    }
    {  // the centre, on the host, while the copy engine runs (k_center's sample and order: 16 interleaved partial sums)
      const int64_t ns = F < 4096 ? F : 4096, stride = F / ns;
      for (int d = 0; d < DP; d++) {
        double t = 0.0;
        if (d < D) {
          double part[16];
          for (int g = 0; g < 16; g++) {
            double sacc = 0.0;
            for (int64_t k = g; k < ns; k += 16) sacc += x_host[(k * stride) * D + d];
            part[g] = sacc;
          }
          for (int g = 0; g < 16; g++) t += part[g];
          t /= (double)ns;
        }
        ctx->ctr_h[d] = t;
      }
      CK(cudaMemcpyAsync(ctx->ctr.p, ctx->ctr_h, sizeof(double) * DP, cudaMemcpyHostToDevice, ctx->st));
      CK(cudaEventRecord(ctx->ev_idle, ctx->st));  // ctr_h is free again once this has run
    }
    CK(cudaMemsetAsync(ctx->xabs_d.p, 0, sizeof(unsigned int) * DP, ctx->st));
    t_begin(ctx, "pack");
    for (int k = 0; k < nch; k++) {
      const int64_t f0 = cb[k], f1 = cb[k + 1];
      CK(cudaStreamWaitEvent(ctx->st, ctx->ev_chunk[k], 0));
      if (f1 > f0) {
        int rc = pack_range(ctx, f0, f1);
        if (rc) return rc;
      }
    }
    t_end(ctx, "pack");
    // the caller's host buffer may be reused as soon as we return
    CK(cudaStreamSynchronize(ctx->st_copy));
    CK(cudaEventSynchronize(ctx->ev_idle));
  } else {
    ctx->d_x64 = x_dev;
    return pack_from_device(ctx);
  }
  return HMMCU_OK;
}

// Streaming upload for the ingest pipeline (SURVEY 8f-2): the caller announces the geometry, then hands over
// frame ranges in any order from (ideally pinned) staging buffers as its readers fill them; every range is copied
// asynchronously on the copy stream and the ticket tells when the staging buffer may be refilled.  _end forms the
// centre and the packed rows on the device exactly as hmmcu_set_features_device does, so the context ends up in
// the same state as after hmmcu_set_features on the concatenated buffer.
// Pinned staging buffer `slot` (0..3) of at least `bytes`, owned by the context and reused across ingests: pinning
// costs ~0.3 ms per MiB, more than reading the same bytes from the page cache.
void *hmmcu_staging(hmmcu_ctx *ctx, int slot, uint64_t bytes) {
  if (!ctx || slot < 0 || slot >= 4) return nullptr;
  if (ctx->stage_cap[slot] >= bytes) return ctx->stage_h[slot];
  if (cudaSetDevice(ctx->dev) != cudaSuccess) return nullptr;
  if (ctx->stage_h[slot]) { cudaStreamSynchronize(ctx->st_copy); cudaFreeHost(ctx->stage_h[slot]); }
  ctx->stage_h[slot] = nullptr;
  ctx->stage_cap[slot] = 0;
  // a quarter of headroom: the jobs of a job file differ by a few per cent in size, and re-pinning three buffers costs 11-12 ms
  // (measured), as much as the rest of a small job
  bytes += bytes / 4;
  if (cudaHostAlloc(&ctx->stage_h[slot], bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  ctx->stage_cap[slot] = bytes;
  return ctx->stage_h[slot];
}

int hmmcu_features_begin(hmmcu_ctx *ctx, const int64_t *frame_off, int U, int D) {
  if (!ctx) return HMMCU_EINVAL;
  if (U < 1 || D < 1 || !frame_off) return fail(ctx, HMMCU_EINVAL, "features_begin: bad arguments");
  if (ctx->stream_open) CK(cudaStreamSynchronize(ctx->st_copy));  // an abandoned ingest: its copies may still be reading the staging buffers
  int rc = features_geometry(ctx, frame_off, U, D);
  if (rc) return rc;
  ctx->have_features = false;  // until _end
  CK(ctx->x64_own.ensure(sizeof(double) * ctx->F * D));
  ctx->d_x64 = ctx->x64_own.as<double>();
  CK(cudaEventRecord(ctx->ev_idle, ctx->st));  // earlier kernels may still read the old features
  CK(cudaStreamWaitEvent(ctx->st_copy, ctx->ev_idle, 0));
  ctx->stream_open = true;
  ctx->stream_frames = 0;
  ctx->stream_next = 0;
  return HMMCU_OK;
}

int hmmcu_features_append(hmmcu_ctx *ctx, const double *x, int64_t first_frame, int64_t n_frames, int *ticket) {
  if (!ctx) return HMMCU_EINVAL;
  if (!ctx->stream_open) return fail(ctx, HMMCU_EINVAL, "features_append: no hmmcu_features_begin");
  if (!x || first_frame < 0 || n_frames < 1 || first_frame + n_frames > ctx->F) return fail(ctx, HMMCU_EINVAL, "features_append: bad frame range");
  CK(cudaSetDevice(ctx->dev));
  const int slot = ctx->stream_next;
  ctx->stream_next = (slot + 1) % hmmcu_ctx::kUpChunks;
  CK(cudaMemcpyAsync(ctx->x64_own.as<double>() + first_frame * ctx->D, x, sizeof(double) * n_frames * ctx->D, cudaMemcpyHostToDevice, ctx->st_copy));
  CK(cudaEventRecord(ctx->ev_chunk[slot], ctx->st_copy));
  ctx->stream_frames += n_frames;
  if (ticket) *ticket = slot;
  return HMMCU_OK;
}

int hmmcu_features_wait(hmmcu_ctx *ctx, int ticket) {
  if (!ctx) return HMMCU_EINVAL;
  if (ticket < 0 || ticket >= hmmcu_ctx::kUpChunks) return fail(ctx, HMMCU_EINVAL, "features_wait: bad ticket");
  CK(cudaEventSynchronize(ctx->ev_chunk[ticket]));
  return HMMCU_OK;
}

int hmmcu_features_end(hmmcu_ctx *ctx) {
  if (!ctx) return HMMCU_EINVAL;
  if (!ctx->stream_open) return fail(ctx, HMMCU_EINVAL, "features_end: no hmmcu_features_begin");
  if (ctx->stream_frames != ctx->F) return fail(ctx, HMMCU_EINVAL, "features_end: %lld of %lld frames appended", (long long)ctx->stream_frames, (long long)ctx->F);
  CK(cudaSetDevice(ctx->dev));
  ctx->stream_open = false;
  CK(cudaEventRecord(ctx->ev_idle, ctx->st_copy));
  CK(cudaStreamWaitEvent(ctx->st, ctx->ev_idle, 0));
  ctx->have_features = true;
  return pack_from_device(ctx);
}

int hmmcu_set_features(hmmcu_ctx *ctx, const double *x, const int64_t *frame_off, int U, int D) {
  return set_features_common(ctx, x, nullptr, frame_off, U, D);
}
int hmmcu_set_features_device(hmmcu_ctx *ctx, const double *x_dev, const int64_t *frame_off, int U, int D) {
  return set_features_common(ctx, nullptr, x_dev, frame_off, U, D);
}

// ------------------------------------------------------------------------------------ models ----
int hmmcu_set_models(hmmcu_ctx *ctx, int V, int N, int M, int D, const double *A, const double *c, const double *mu,
                     const double *inv_var, const double *det) {
  if (!ctx) return HMMCU_EINVAL;
  if (V < 1 || N < 1 || M < 1 || D < 1 || !A || !c || !mu || !inv_var || !det) return fail(ctx, HMMCU_EINVAL, "set_models: bad arguments");
  if (N > 8) return fail(ctx, HMMCU_EINVAL, "set_models: N=%d states not supported yet (max 8)", N);
  CK(cudaSetDevice(ctx->dev));
  const int64_t G = (int64_t)N * M, VG = V * G;
  CK(ctx->A.ensure(sizeof(double) * V * N * N));
  CK(ctx->c.ensure(sizeof(double) * VG));
  CK(ctx->mu.ensure(sizeof(double) * VG * D));
  CK(ctx->iv.ensure(sizeof(double) * VG * D));
  CK(ctx->det.ensure(sizeof(double) * VG));
  CK(cudaMemcpyAsync(ctx->A.p, A, sizeof(double) * V * N * N, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemcpyAsync(ctx->c.p, c, sizeof(double) * VG, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemcpyAsync(ctx->mu.p, mu, sizeof(double) * VG * D, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemcpyAsync(ctx->iv.p, inv_var, sizeof(double) * VG * D, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemcpyAsync(ctx->det.p, det, sizeof(double) * VG, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaStreamSynchronize(ctx->st));
  ctx->banded = true;
  for (int64_t k = 0; k < (int64_t)V * N * N && ctx->banded; k++) {
    const int i = (int)((k / N) % N), j = (int)(k % N);
    if ((j < i || j > i + 1) && A[k] != 0.0) ctx->banded = false;
  }
  if (V != ctx->V || N != ctx->N || M != ctx->M) ctx->u2m.clear();
  ctx->V = V; ctx->N = N; ctx->M = M; ctx->G = (int)G;
  ctx->Dm = D;
  ctx->have_models = true;
  ctx->pack_dirty = true;
  ctx->kappa_stale = true;
  ctx->cfg_epoch++;
  return HMMCU_OK;
}

// ------------------------------------------------------------- initial models on the device ----
// creating_initial_model (T-FS:732-1317) for V words at once from the context's features: utterance u belongs
// to word utt2model[u] (-1 = not used).  The models are left in the context exactly as hmmcu_set_models would
// leave them (read them back with hmmcu_get_models).  Bit-identical to hmmh_init_model(), see init_kernels.cuh.
int hmmcu_init_models(hmmcu_ctx *ctx, const int32_t *utt2model, int V, int N, int M) {
  if (!ctx) return HMMCU_EINVAL;
  if (!ctx->have_features || ctx->U < 1 || !ctx->d_x64) return fail(ctx, HMMCU_EINVAL, "init_models: set the features first");
  if (!utt2model || V < 1 || N < 1 || N > 8 || M < 1 || M > 255) return fail(ctx, HMMCU_EINVAL, "init_models: bad arguments (N <= 8, M <= 255)");
  const int D = ctx->D, U = ctx->U;
  if (D > 64) return fail(ctx, HMMCU_EINVAL, "init_models: D=%d not supported on the device (max 64); use hmmh_init_model", D);
  CK(cudaSetDevice(ctx->dev));
  const int VN = V * N;
  // the frames of every (word, state) in the reference's order: utterance by utterance, uniform segments (T-FS:1005-1013)
  std::vector<int32_t> cntv((size_t)VN + 1, 0);
  for (int u = 0; u < U; u++) {
    const int v = utt2model[u];
    if (v < -1 || v >= V) return fail(ctx, HMMCU_EINVAL, "utt2model[%d]=%d out of range", u, v);
    if (v < 0) continue;
    const int T = (int)(ctx->off[u + 1] - ctx->off[u]), q = T / N, r = T % N;
    for (int k = 0; k < N; k++) cntv[(size_t)v * N + k + 1] += q + (k < r ? 1 : 0);
  }
  for (int i = 0; i < VN; i++) cntv[i + 1] += cntv[i];
  const int64_t E = cntv[VN];
  if (E == 0) return fail(ctx, HMMCU_EINVAL, "init_models: no frames");
  std::vector<int32_t> lst((size_t)E), vk((size_t)E), fill(cntv.begin(), cntv.end() - 1);
  for (int u = 0; u < U; u++) {
    const int v = utt2model[u];
    if (v < 0) continue;
    const int64_t f0 = ctx->off[u];
    const int T = (int)(ctx->off[u + 1] - f0), q = T / N, r = T % N;
    int t = 0;
    for (int k = 0; k < N; k++) {
      const int len = q + (k < r ? 1 : 0);
      int32_t &w = fill[(size_t)v * N + k];
      for (int j = 0; j < len; j++, t++) { lst[w] = (int32_t)(f0 + t); vk[w] = v * N + k; w++; }
    }
  }
  const size_t GD = (size_t)VN * M * D, G = (size_t)VN * M;
  CK(ctx->in_lst.ensure(sizeof(int32_t) * E));
  CK(ctx->in_vk.ensure(sizeof(int32_t) * E));
  CK(ctx->in_off.ensure(sizeof(int32_t) * (VN + 1)));
  CK(ctx->in_cent.ensure(sizeof(double) * GD));
  CK(ctx->in_sum.ensure(sizeof(double) * GD));
  CK(ctx->in_dist.ensure(sizeof(double) * G));
  CK(ctx->in_cnt.ensure(sizeof(double) * G));
  CK(ctx->in_idx.ensure((size_t)E));
  CK(ctx->in_dd.ensure(sizeof(double) * E));
  CK(ctx->in_ord.ensure(sizeof(int) * G));
  CK(ctx->A.ensure(sizeof(double) * VN * N));
  CK(ctx->c.ensure(sizeof(double) * G));
  CK(ctx->mu.ensure(sizeof(double) * GD));
  CK(ctx->iv.ensure(sizeof(double) * GD));
  CK(ctx->det.ensure(sizeof(double) * G));
  CK(cudaMemcpyAsync(ctx->in_lst.p, lst.data(), sizeof(int32_t) * E, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemcpyAsync(ctx->in_vk.p, vk.data(), sizeof(int32_t) * E, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemcpyAsync(ctx->in_off.p, cntv.data(), sizeof(int32_t) * (VN + 1), cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemsetAsync(ctx->in_cent.p, 0, sizeof(double) * GD, ctx->st));
  CK(cudaMemsetAsync(ctx->in_dist.p, 0, sizeof(double) * G, ctx->st));
  const double *x = ctx->d_x64;
  auto classify = [&](int have) -> int {
    if (D == 39)
      k_init_classify<39><<<(unsigned)((E + 127) / 128), 128, 0, ctx->st>>>(x, ctx->in_lst.as<int32_t>(), ctx->in_vk.as<int32_t>(), E, ctx->in_cent.as<double>(), M, D,
                                                                           have, ctx->in_idx.as<uint8_t>(), ctx->in_dd.as<double>());
    else
      k_init_classify<0><<<(unsigned)((E + 255) / 256), 256, 0, ctx->st>>>(x, ctx->in_lst.as<int32_t>(), ctx->in_vk.as<int32_t>(), E, ctx->in_cent.as<double>(), M, D,
                                                                          have, ctx->in_idx.as<uint8_t>(), ctx->in_dd.as<double>());
    LAUNCH_CHECK();
    return HMMCU_OK;
  };
  auto accumulate = [&](int have, int mode, bool all) -> int {
    const int warps = VN * have;
    k_init_accumulate<<<(warps * 32 + 127) / 128, 128, 0, ctx->st>>>(x, ctx->in_lst.as<int32_t>(), ctx->in_off.as<int32_t>(), ctx->in_idx.as<uint8_t>(),
                                                                    ctx->in_dd.as<double>(), ctx->in_cent.as<double>(), VN, M, D, have, mode, all,
                                                                    ctx->in_sum.as<double>(), ctx->in_dist.as<double>(), ctx->in_cnt.as<double>());
    LAUNCH_CHECK();
    return HMMCU_OK;
  };
  auto update = [&](int have, int have_next) -> int {
    k_init_update<<<(VN * 32 + 127) / 128, 128, 0, ctx->st>>>(ctx->in_cent.as<double>(), ctx->in_sum.as<double>(), ctx->in_dist.as<double>(), ctx->in_cnt.as<double>(),
                                                     VN, M, D, have, have_next, ctx->in_ord.as<int>());
    LAUNCH_CHECK();
    return HMMCU_OK;
  };
  auto split_to = [&](int have) { return have >= M ? have : (2 * have < M ? 2 * have : M); };
  int rc;
  t_begin(ctx, "init");
  // one centroid per state (T-FS:996-1030), then the first split
  if ((rc = accumulate(1, 0, true)) != HMMCU_OK) return rc;
  int have = split_to(1);
  if ((rc = update(1, have)) != HMMCU_OK) return rc;
  while (have > 1) {  // three k-means passes per level (T-FS:1034-1094); the last one also splits for the next level
    for (int pass = 0; pass < 3; pass++) {
      if ((rc = classify(have)) != HMMCU_OK) return rc;
      if ((rc = accumulate(have, 0, false)) != HMMCU_OK) return rc;
      const int nxt = (pass == 2) ? split_to(have) : have;
      if ((rc = update(have, nxt)) != HMMCU_OK) return rc;
      if (pass == 2) {
        if (nxt == have) have = 0;  // M reached: done
        else have = nxt;
      }
    }
  }
  // variances and weights (init_mix_param, T-FS:864-932)
  if ((rc = classify(M)) != HMMCU_OK) return rc;
  if ((rc = accumulate(M, 1, M == 1)) != HMMCU_OK) return rc;
  k_init_finish<<<(VN + 63) / 64, 64, 0, ctx->st>>>(ctx->in_cent.as<double>(), ctx->in_sum.as<double>(), ctx->in_cnt.as<double>(), ctx->in_off.as<int32_t>(), V, N,
                                                   M, D, ctx->A.as<double>(), ctx->c.as<double>(), ctx->mu.as<double>(), ctx->iv.as<double>(),
                                                   ctx->det.as<double>());
  LAUNCH_CHECK();
  t_end(ctx, "init");
  CK(cudaStreamSynchronize(ctx->st));  // the host vectors above were copied asynchronously
  if (V != ctx->V || N != ctx->N || M != ctx->M) ctx->u2m.clear();
  ctx->V = V; ctx->N = N; ctx->M = M; ctx->G = N * M;
  ctx->Dm = D;
  ctx->banded = true;  // the DELTA = 1 band
  ctx->have_models = true;
  ctx->pack_dirty = true;
  ctx->kappa_stale = true;
  ctx->cfg_epoch++;
  return HMMCU_OK;
}

// model extremes -> ext_d, kappa -> kappa_out (device); no synchronisation
static int launch_kappa(hmmcu_ctx *ctx, double *kappa_out) {
  const int D = ctx->Dm, DP = round_up(D + 1, 4);
  const int64_t VG = (int64_t)ctx->V * ctx->G;
  CK(ctx->ext_d.ensure(sizeof(unsigned long long) * (2 * DP + 1)));  // extremes + the finished-block counter
  CK(cudaMemsetAsync(ctx->ext_d.p, 0, sizeof(unsigned long long) * (2 * DP + 1), ctx->st));
  const int ngrp = std::max(1, 256 / DP);
  const int blocks = (int)std::min<int64_t>((VG + ngrp - 1) / ngrp, (int64_t)ctx->sm_count * 4);
  k_model_extremes<<<blocks, 256, 0, ctx->st>>>(ctx->mu.as<double>(), ctx->iv.as<double>(), ctx->ctr.as<double>(), VG, D, DP,
                                               ctx->ext_d.as<unsigned long long>(), ctx->F > 0 ? ctx->xabs_d.as<unsigned int>() : nullptr,
                                               reinterpret_cast<unsigned int *>(ctx->ext_d.as<unsigned long long>() + 2 * DP), kappa_out);
  LAUNCH_CHECK();
  return HMMCU_OK;
}

static int ensure_ctl(hmmcu_ctx *ctx) {
  const size_t n = 3 * (size_t)ctx->V + 1;
  CK(ctx->ctl_d.ensure(sizeof(double) * n));
  if (n > ctx->ctl_cap) {
    if (ctx->ctl_h) cudaFreeHost(ctx->ctl_h);
    ctx->ctl_h = nullptr;
    CK(cudaMallocHost((void **)&ctx->ctl_h, sizeof(double) * n));
    ctx->ctl_cap = n;
    g_alloc_epoch++;
  }
  return HMMCU_OK;
}

static int ensure_packed(hmmcu_ctx *ctx) {
  if (!ctx->have_features || !ctx->have_models) return fail(ctx, HMMCU_EINVAL, "features and models must both be set first");
  if (ctx->Dm != ctx->D) return fail(ctx, HMMCU_EINVAL, "models have D=%d but features have D=%d", ctx->Dm, ctx->D);
  if (!ctx->pack_dirty) return HMMCU_OK;
  CK(ctx->ctr.ensure(sizeof(double) * ctx->DP));
  if (ctx->F == 0) CK(cudaMemsetAsync(ctx->ctr.p, 0, sizeof(double) * ctx->DP, ctx->st));
  ctx->pack_dirty = false;
  ctx->simt_dirty = true;  // the packed forms below are rebuilt on first use
  ctx->kc_dirty = true;
  ctx->tc_train.dirty = true;
  ctx->tc_dec.dirty = true;
  ctx->ws_train.dirty = true;
  ctx->ws_dec.dirty = true;
  ctx->acc_dirty = true;
  if (ctx->kappa_stale) {  // after set_features / set_models; hmmcu_mstep refreshes it with its own read-back
    int rc = ensure_ctl(ctx);
    if (rc) return rc;
    if ((rc = launch_kappa(ctx, ctx->ctl_d.as<double>() + 3 * ctx->V)) != HMMCU_OK) return rc;
    CK(cudaMemcpyAsync(ctx->ctl_h + 3 * ctx->V, ctx->ctl_d.as<double>() + 3 * ctx->V, sizeof(double), cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    ctx->kappa = ctx->ctl_h[3 * ctx->V];
    ctx->kappa_stale = false;
  }
  return HMMCU_OK;
}

// CUDA-core kernels' parameter arrays (mu32, iv32, k32), built only when that path runs
static int ensure_simt_pack(hmmcu_ctx *ctx) {
  if (!ctx->simt_dirty) return HMMCU_OK;
  const int64_t VG = (int64_t)ctx->V * ctx->G;
  CK(ctx->mu32.ensure(sizeof(float) * VG * ctx->DP));
  CK(ctx->iv32.ensure(sizeof(float) * VG * ctx->DP));
  CK(ctx->k32.ensure(sizeof(float) * VG));
  int64_t total = VG * ctx->DP;
  int blocks = (int)std::min<int64_t>((total + 255) / 256, (int64_t)ctx->sm_count * 16);
  t_begin(ctx, "pack");
  k_pack_models<<<blocks, 256, 0, ctx->st>>>(ctx->mu.as<double>(), ctx->iv.as<double>(), ctx->det.as<double>(),
                                            ctx->c.as<double>(), ctx->ctr.as<double>(), VG, ctx->D, ctx->DP,
                                            ctx->mu32.as<float>(), ctx->iv32.as<float>(), ctx->k32.as<float>());
  LAUNCH_CHECK();
  t_end(ctx, "pack");
  ctx->simt_dirty = false;
  return HMMCU_OK;
}

// additive constants of all Gaussians (log2 units), shared by the tensor-core W packers
static int launch_pack_kc(hmmcu_ctx *ctx) {
  const int64_t VG = (int64_t)ctx->V * ctx->G;
  CK(launch_pdl(k_pack_kc, (unsigned)((VG * 32 + 255) / 256), 256, 0, ctx->st, ctx->mu.as<double>(), ctx->iv.as<double>(),
                ctx->det.as<double>(), ctx->c.as<double>(), ctx->ctr.as<double>(), VG, ctx->D, ctx->kc2.as<float>()));
  LAUNCH_CHECK();
  return HMMCU_OK;
}
static int ensure_kc(hmmcu_ctx *ctx) {
  if (!ctx->kc_dirty) return HMMCU_OK;
  const int64_t VG = (int64_t)ctx->V * ctx->G;
  CK(ctx->kc2.ensure(sizeof(float) * VG));
  int rc = launch_pack_kc(ctx);
  if (rc) return rc;
  ctx->kc_dirty = false;
  return HMMCU_OK;
}

// ---- tensor-core path: W images ------------------------------------------------------------------
// use_tc: 0 = never, 1 = when the accuracy guard allows it (default), 2 = always (testing)
constexpr double kTcKappaMax = 1.0e4;
static bool tc_supported(const hmmcu_ctx *ctx) {
  if (!ctx->use_tc || ctx->M > kTcMaxTN || ctx->N > 8) return false;
  if (ctx->use_tc == 1 && !(ctx->kappa <= kTcKappaMax)) return false;
  const int SCt = std::max(1, kTcMaxTN / ctx->M);
  const int TN = round_up(std::min(SCt, ctx->V * ctx->N) * ctx->M, 16);
  if (!tc_acc_fits(2 * ctx->DP)) return false;
  return tc_emis_smem_bytes(TN, 2 * ctx->DP) <= 227 * 1024;
}

// k_accum_h instead of k_accum_ws: a matter of shapes and options only (the packed forms follow it)
static bool h_acc_on(const hmmcu_ctx *ctx) {
  return ctx->use_ws_acc && ctx->use_h_acc && ctx->DP % 8 == 0 && ctx->DP <= 40 && ctx->N <= 8 && ctx->xabs_d.p != nullptr && ctx->F > 0;
}

static int launch_pack_acc(hmmcu_ctx *ctx) {
  const int KP = 2 * ctx->DP, nRB = (ctx->G + 127) / 128, nimg = ctx->V * nRB;
  if (h_acc_on(ctx)) {
    CK(launch_pdl(k_pack_wT_h, dim3((128 * KP + 255) / 256, nimg), 256, 0, ctx->st, ctx->mu.as<double>(), ctx->iv.as<double>(),
                  ctx->kc2.as<float>(), ctx->ctr.as<double>(), ctx->acc_sc.as<float>(), ctx->G, nRB, ctx->D, ctx->DP,
                  ctx->acc_images16.as<unsigned short>(), ctx->acc_kc.as<float>()));
    LAUNCH_CHECK();
    return HMMCU_OK;
  }
  k_pack_wT_tc<<<dim3((128 * KP + 255) / 256, nimg), 256, 0, ctx->st>>>(ctx->mu.as<double>(), ctx->iv.as<double>(), ctx->kc2.as<float>(),
                                                                        ctx->ctr.as<double>(), ctx->G, nRB, ctx->D, ctx->DP,
                                                                        ctx->acc_images.as<float>(), ctx->acc_kc.as<float>());
  LAUNCH_CHECK();
  return HMMCU_OK;
}

static int ensure_acc_images(hmmcu_ctx *ctx) {
  if (!ctx->acc_dirty) return HMMCU_OK;
  const int KP = 2 * ctx->DP, nRB = (ctx->G + 127) / 128, nimg = ctx->V * nRB;
  if (h_acc_on(ctx)) {
    CK(ctx->acc_images16.ensure(ah_image_bytes(KP) * nimg));
    CK(ctx->acc_sc.ensure(sizeof(float) * kAhScN * ctx->DP));
  } else {
    CK(ctx->acc_images.ensure(tc_accT_image_bytes(KP) * nimg));
  }
  CK(ctx->acc_kc.ensure(sizeof(float) * 128 * (size_t)nimg));
  int rc = ensure_kc(ctx);
  if (rc) return rc;
  t_begin(ctx, "pack");
  if ((rc = launch_pack_acc(ctx)) != HMMCU_OK) return rc;
  t_end(ctx, "pack");
  ctx->acc_dirty = false;
  return HMMCU_OK;
}

// mode 0: training images (per model, CT column tiles each); mode 1: decode images (all states concatenated)
static int ensure_tc_images(hmmcu_ctx *ctx, int mode) {
  hmmcu_ctx::TcSet &ts = mode == 0 ? ctx->tc_train : ctx->tc_dec;
  if (!ts.dirty) return HMMCU_OK;
  const int N = ctx->N, M = ctx->M, V = ctx->V;
  const int SCmax = std::max(1, kTcMaxTN / M);
  std::vector<int32_t> s0, ns;
  if (mode == 0) {
    ts.SCt = std::min(SCmax, N);
    for (int v = 0; v < V; v++)
      for (int s = 0; s < N; s += ts.SCt) { s0.push_back(v * N + s); ns.push_back(std::min(ts.SCt, N - s)); }
  } else {
    const int S = V * N;
    ts.SCt = std::min(SCmax, S);
    for (int s = 0; s < S; s += ts.SCt) { s0.push_back(s); ns.push_back(std::min(ts.SCt, S - s)); }
  }
  ts.TN = round_up(ts.SCt * M, 16);
  ts.nimg = (int)s0.size();
  const int KP = 2 * ctx->DP;
  CK(ts.images.ensure(tc_image_bytes(ts.TN, KP) * ts.nimg));
  CK(ts.kc.ensure(sizeof(float) * (size_t)ts.TN * ts.nimg));
  CK(ts.s0.ensure(sizeof(int32_t) * ts.nimg));
  CK(ts.ns.ensure(sizeof(int32_t) * ts.nimg));
  CK(cudaMemcpyAsync(ts.s0.p, s0.data(), sizeof(int32_t) * ts.nimg, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemcpyAsync(ts.ns.p, ns.data(), sizeof(int32_t) * ts.nimg, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaStreamSynchronize(ctx->st));  // s0 / ns are stack vectors
  t_begin(ctx, "pack");
  k_pack_w_tc<<<ts.nimg, 256, 0, ctx->st>>>(ctx->mu.as<double>(), ctx->iv.as<double>(), ctx->det.as<double>(), ctx->c.as<double>(),
                                           ctx->ctr.as<double>(), M, ctx->D, ctx->DP, ts.TN, ts.s0.as<int32_t>(), ts.ns.as<int32_t>(),
                                           ts.images.as<float>(), ts.kc.as<float>());
  LAUNCH_CHECK();
  t_end(ctx, "pack");
  ts.dirty = false;
  return HMMCU_OK;
}

// ---- warp-specialised emission kernel: images and launch ----------------------------------------
// image geometry of the warp-specialised emission kernel: whole states per image (SCt) and its columns (TN)
static void ws_geometry(const hmmcu_ctx *ctx, int nstates_avail, int &SCt, int &TN) {
  const int MPd = ws_pad_m(ctx->M);
  if (MPd <= 16) SCt = std::min((kWsMaxTN / 16) * ws_states_per_chunk(MPd), nstates_avail);
  else if (MPd <= kWsMaxTN) SCt = std::min(std::min(kWsMaxTN / MPd, kWsXch), nstates_avail);
  else SCt = 1;  // one wide state per image
  TN = round_up(ws_image_cols(MPd, SCt), 16);
}
static bool ws_supported(const hmmcu_ctx *ctx) {
  const int MPd = ws_pad_m(ctx->M);
  if (!ctx->use_ws || MPd > kWsMaxTN1 || ctx->DP > 40) return false;
  int SCt, TN;
  ws_geometry(ctx, ctx->V * ctx->N, SCt, TN);
  return ws_emis_smem_bytes(TN, 2 * ctx->DP) <= 227 * 1024;
}

// half-precision decode images: the padded feature row must be whole groups of 8 (K = 16 halves per MMA), DP <= 40, M <= 16
static bool f16_possible(const hmmcu_ctx *ctx) {
  // (kappa bounds the scaled operands by ~2 sqrt(kappa): far inside the half's range while the accuracy guard holds)
  return ctx->DP % 8 == 0 && ctx->DP <= 40 && ctx->ext_d.p != nullptr && ctx->kappa <= kTcKappaMax;
}
static bool dec16_wanted(const hmmcu_ctx *ctx) { return ctx->dec_f16 && f16_possible(ctx); }      // decode set: k_emis_dec, k_emis_ws<false>
// The training emission kernel keeps its 3xTF32 operands: it is bound by the instruction issue of its loaders and its
// epilogue, not by the MMAs (measured with half-precision operands: no gain), and its images are re-packed inside the
// M-step's captured graph.
static bool train16_wanted(const hmmcu_ctx *) { return false; }

static int launch_pack_ws(hmmcu_ctx *ctx, hmmcu_ctx::TcSet &ts) {
  const int KP = 2 * ctx->DP;
  CK(launch_pdl(k_pack_w_ws, dim3((ts.TN * KP + 255) / 256, ts.nimg), 256, 0, ctx->st, ctx->mu.as<double>(), ctx->iv.as<double>(),
                ctx->kc2.as<float>(), ctx->ctr.as<double>(), ctx->M, ws_pad_m(ctx->M), ctx->D, ctx->DP, ts.TN, ts.s0.as<int32_t>(),
                ts.ns.as<int32_t>(), ts.images.as<float>()));
  LAUNCH_CHECK();
  return HMMCU_OK;
}

static int ensure_ws_images(hmmcu_ctx *ctx, int mode) {
  hmmcu_ctx::TcSet &ts = mode == 0 ? ctx->ws_train : ctx->ws_dec;
  if (!ts.dirty) return HMMCU_OK;
  const int N = ctx->N, V = ctx->V;
  std::vector<int32_t> s0, ns;
  int TN;
  if (mode == 0) {
    ws_geometry(ctx, N, ts.SCt, TN);
    for (int v = 0; v < V; v++)
      for (int s = 0; s < N; s += ts.SCt) { s0.push_back(v * N + s); ns.push_back(std::min(ts.SCt, N - s)); }
  } else {
    const int S = V * N;
    ws_geometry(ctx, S, ts.SCt, TN);
    for (int s = 0; s < S; s += ts.SCt) { s0.push_back(s); ns.push_back(std::min(ts.SCt, S - s)); }
  }
  const int KP = 2 * ctx->DP;
  if (TN != ts.TN || s0 != ts.s0_h || ns != ts.ns_h) {  // geometry changed: (re)upload the image table
    ts.TN = TN;
    ts.s0_h = s0;
    ts.ns_h = ns;
    ts.nimg = (int)s0.size();
    CK(ts.s0.ensure(sizeof(int32_t) * ts.nimg));
    CK(ts.ns.ensure(sizeof(int32_t) * ts.nimg));
    CK(cudaMemcpyAsync(ts.s0.p, s0.data(), sizeof(int32_t) * ts.nimg, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(ts.ns.p, ns.data(), sizeof(int32_t) * ts.nimg, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));  // s0 / ns are stack vectors
  }
  CK(ts.images.ensure(ws_image_bytes(ts.TN, KP) * ts.nimg));  // not only on a new geometry: the feature width may have changed
  {
    int rc = ensure_kc(ctx);
    if (rc) return rc;
  }
  t_begin(ctx, "pack");
  {
    int rc = launch_pack_ws(ctx, ts);
    if (rc) return rc;
  }
  if (mode == 1 ? dec16_wanted(ctx) : train16_wanted(ctx)) {  // half-precision images: scales from the extremes the accuracy guard collected
    CK(ts.images16.ensure(dec16_image_bytes(ts.TN, KP) * ts.nimg));
    CK(ts.scales16.ensure(sizeof(float) * 4 * ctx->DP));
    k_dec16_scales<<<1, 64, 0, ctx->st>>>(ctx->ext_d.as<unsigned long long>(), ctx->F > 0 ? ctx->xabs_d.as<unsigned int>() : nullptr, ctx->D, ctx->DP,
                                         ts.scales16.as<float>());
    LAUNCH_CHECK();
    k_pack_w_dec16<<<dim3((ts.TN * KP + 255) / 256, ts.nimg), 256, 0, ctx->st>>>(ctx->mu.as<double>(), ctx->iv.as<double>(), ctx->kc2.as<float>(),
                                                                              ctx->ctr.as<double>(), ts.scales16.as<float>(), ctx->M, ws_pad_m(ctx->M), ctx->D,
                                                                              ctx->DP, ts.TN, ts.s0.as<int32_t>(), ts.ns.as<int32_t>(),
                                                                              ts.images16.as<unsigned char>());
    LAUNCH_CHECK();
  }
  t_end(ctx, "pack");
  ts.dirty = false;
  return HMMCU_OK;
}

// TRAIN: units = explicit list (nunits); decode: nunits = nimg * ntiles over nframes contiguous frames from fbase
template <bool TRAIN>
static int launch_emis_ws(hmmcu_ctx *ctx, const TcTile *units_dev, int64_t nunits, int ntiles_dec, int nframes_dec, float *logb,
                          int64_t fbase, int64_t ldb) {
  ctx->last_tc = true;
  if (nunits == 0) return HMMCU_OK;
  if (nunits > 0x7fffffff) return fail(ctx, HMMCU_EINVAL, "emission units overflow");
  hmmcu_ctx::TcSet &ts = TRAIN ? ctx->ws_train : ctx->ws_dec;
  const size_t smem = ws_emis_smem_bytes(ts.TN, 2 * ctx->DP);
  const int grid = (int)std::min<int64_t>(nunits, ctx->sm_count);
  const int MPd = ws_pad_m(ctx->M);
  const bool h16 = (TRAIN ? train16_wanted(ctx) : dec16_wanted(ctx)) && ts.images16.p != nullptr;
  if (!TRAIN) ctx->last_dec16 = h16;
#define WS_LAUNCH4(MPT, MRT, HT)                                                                                             \
  do {                                                                                                                       \
    CK(cudaFuncSetAttribute(k_emis_ws<TRAIN, MPT, MRT, HT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));        \
    k_emis_ws<TRAIN, MPT, MRT, HT><<<grid, kWsThreads, smem, ctx->st>>>(units_dev, (int)nunits, ntiles_dec, nframes_dec,     \
                                                               ctx->frame_ids_d.as<int32_t>(), ctx->x32.as<float>(),         \
                                                               HT ? ts.images16.as<float>() : ts.images.as<float>(), ctx->N, \
                                                               MPd, ctx->DP, ts.TN, logb, fbase, ldb, ctx->V * ctx->N,       \
                                                               ts.SCt, ts.scales16.as<float>());                             \
  } while (0)
#define WS_LAUNCH(MPT)                              \
  do {                                              \
    if (h16) WS_LAUNCH4(MPT, 0, true);              \
    else WS_LAUNCH4(MPT, 0, false);                 \
  } while (0)
  switch (MPd) {
    case 1: WS_LAUNCH(1); break;
    case 2: WS_LAUNCH(2); break;
    case 3: WS_LAUNCH(3); break;
    case 4: WS_LAUNCH(4); break;
    case 5: WS_LAUNCH(5); break;
    case 8: WS_LAUNCH(8); break;
    case 16: WS_LAUNCH(16); break;
    default: WS_LAUNCH(0); break;
  }
#undef WS_LAUNCH4
#undef WS_LAUNCH
  LAUNCH_CHECK();
  return HMMCU_OK;
}

template <bool TRAIN>
static int launch_emis_tc(hmmcu_ctx *ctx, const TcTile *tiles_dev, int ntiles, float *logb, int64_t fbase, int64_t ldb, float *post) {
  ctx->last_tc = true;
  if (ntiles == 0) return HMMCU_OK;
  hmmcu_ctx::TcSet &ts = TRAIN ? ctx->tc_train : ctx->tc_dec;
  const size_t smem = tc_emis_smem_bytes(ts.TN, 2 * ctx->DP);
  CK(cudaFuncSetAttribute(k_emis_tc<TRAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = std::min(ntiles, ctx->sm_count);
  k_emis_tc<TRAIN><<<grid, kTcThreads, smem, ctx->st>>>(tiles_dev, ntiles, ctx->frame_ids_d.as<int32_t>(), ctx->x32.as<float>(),
                                                        ts.images.as<float>(), ts.kc.as<float>(), ts.nimg, ctx->N, ctx->M, ctx->DP,
                                                        ts.TN, logb, fbase, ldb, ctx->V * ctx->N, ts.SCt, post);
  LAUNCH_CHECK();
  return HMMCU_OK;
}


// decode emissions, frames resident in tensor memory, W images multicast over clusters of two CTAs (dec_kernels.cuh)
template <int MP, int MR, bool H16>
static int launch_emis_dec_c(hmmcu_ctx *ctx, int ntiles, int nframes, float *logb, int64_t fbase, int64_t ldb) {
  hmmcu_ctx::TcSet &ts = ctx->ws_dec;
  const size_t smem = dec_emis_smem_bytes(ts.TN, 2 * ctx->DP, H16);
  auto kern = k_emis_dec<MP, MR, H16>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kDecCluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(kDecThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = ctx->st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (ctx->dec_grid == 0) {  // whole clusters that are resident together: one CTA per SM, two SMs of one GPC per cluster
    cfg.gridDim = dim3((ctx->sm_count / kDecCluster) * kDecCluster);
    int ncl = 0;
    if (cudaOccupancyMaxActiveClusters(&ncl, kern, &cfg) != cudaSuccess || ncl < 1) {
      cudaGetLastError();
      ctx->dec_grid = -1;
    } else {
      ctx->dec_grid = std::min(ncl, ctx->sm_count / kDecCluster) * kDecCluster;
    }
  }
  if (ctx->dec_grid < 0) return HMMCU_EINVAL;
  const int want = ((ntiles + kDecCluster - 1) / kDecCluster) * kDecCluster;
  cfg.gridDim = dim3(std::min(ctx->dec_grid, want));
  const float *x32 = ctx->x32.as<float>(), *img = H16 ? ts.images16.as<float>() : ts.images.as<float>(), *scales = ts.scales16.as<float>();
  int nimg = ts.nimg, DP = ctx->DP, TN = ts.TN, S_total = ctx->V * ctx->N, SCt = ts.SCt;
  CK(cudaLaunchKernelEx(&cfg, kern, ntiles, nframes, nimg, x32, img, DP, TN, logb, fbase, ldb, S_total, SCt, scales));
  ctx->last_dec16 = H16;
  ctx->launches++;
  ctx->last_tc = true;
  return HMMCU_OK;
}
template <int MP, int MR>
static int launch_emis_dec_t(hmmcu_ctx *ctx, int ntiles, int nframes, float *logb, int64_t fbase, int64_t ldb) {
  if (dec16_wanted(ctx) && ws_pad_m(ctx->M) <= 16 && ctx->ws_dec.images16.p)
    return launch_emis_dec_c<MP, MR, true>(ctx, ntiles, nframes, logb, fbase, ldb);
  return launch_emis_dec_c<MP, MR, false>(ctx, ntiles, nframes, logb, fbase, ldb);
}
static int launch_emis_dec(hmmcu_ctx *ctx, int ntiles, int nframes, float *logb, int64_t fbase, int64_t ldb) {
  switch (ws_pad_m(ctx->M)) {
    case 1: return launch_emis_dec_t<1, 0>(ctx, ntiles, nframes, logb, fbase, ldb);
    case 2: return launch_emis_dec_t<2, 0>(ctx, ntiles, nframes, logb, fbase, ldb);
    case 3: return launch_emis_dec_t<3, 0>(ctx, ntiles, nframes, logb, fbase, ldb);
    case 4: return launch_emis_dec_t<4, 0>(ctx, ntiles, nframes, logb, fbase, ldb);
    case 5: return launch_emis_dec_t<5, 0>(ctx, ntiles, nframes, logb, fbase, ldb);
    case 8: return launch_emis_dec_t<8, 0>(ctx, ntiles, nframes, logb, fbase, ldb);
    case 16: return launch_emis_dec_t<16, 0>(ctx, ntiles, nframes, logb, fbase, ldb);
    default: return HMMCU_EINVAL;
  }
}
static bool dec_supported(const hmmcu_ctx *ctx) {
  return ctx->use_dec_emis && ws_pad_m(ctx->M) <= 16 && ctx->DP <= 40 && ctx->dec_grid >= 0 && ctx->sm_count >= kDecCluster;
}

// --------------------------------------------------------------------------------- emissions ----
static int emis_chunk_states(const hmmcu_ctx *ctx) { return std::max(1, std::min(ctx->N, 128 / ctx->M)); }

template <bool POST>
static int launch_emis(hmmcu_ctx *ctx, const EmisTile *tiles_dev, int64_t ntiles, float *logb, int64_t fbase, int64_t ldb,
                       int decode, float *post) {
  ctx->last_tc = false;
  if (ntiles == 0) return HMMCU_OK;
  {
    int rc = ensure_simt_pack(ctx);
    if (rc) return rc;
  }
  const int SC = emis_chunk_states(ctx);
  const size_t smem = emis_smem_bytes(SC * ctx->M, SC, ctx->DP);
  if (smem > 227 * 1024) return fail(ctx, HMMCU_EINVAL, "M=%d mixtures x D=%d does not fit the emission kernel's shared memory", ctx->M, ctx->D);
  CK(cudaFuncSetAttribute(k_emis_simt<POST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_emis_simt<POST><<<(unsigned)ntiles, kEmisThreads, smem, ctx->st>>>(tiles_dev, ctx->x32.as<float>(), ctx->mu32.as<float>(),
                                                                       ctx->iv32.as<float>(), ctx->k32.as<float>(), ctx->N,
                                                                       ctx->M, ctx->DP, SC, logb, fbase, ldb, decode, post);
  LAUNCH_CHECK();
  return HMMCU_OK;
}

int hmmcu_emissions(hmmcu_ctx *ctx, int u, int v, double *logb, double *post) {
  if (!ctx) return HMMCU_EINVAL;
  CK(cudaSetDevice(ctx->dev));
  int rc = ensure_packed(ctx);
  if (rc) return rc;
  if (u < 0 || u >= ctx->U || v < 0 || v >= ctx->V || !logb) return fail(ctx, HMMCU_EINVAL, "emissions: bad arguments");
  const int64_t f0 = ctx->off[u];
  const int T = (int)(ctx->off[u + 1] - f0);
  std::vector<EmisTile> tiles;
  for (int t = 0; t < T; t += kEmisTF) tiles.push_back({f0 + t, std::min(kEmisTF, T - t), v});
  DevBuf tl, lb, ps;
  CK(tl.ensure(sizeof(EmisTile) * tiles.size()));
  CK(lb.ensure(sizeof(float) * T * ctx->N));
  CK(ps.ensure(sizeof(float) * (size_t)T * ctx->G));
  CK(cudaMemcpyAsync(tl.p, tiles.data(), sizeof(EmisTile) * tiles.size(), cudaMemcpyHostToDevice, ctx->st));
  // post is indexed by global frame: offset the pointer so that frame f0 lands at ps[0]
  if (tc_supported(ctx)) {
    if ((rc = ensure_tc_images(ctx, 0)) != HMMCU_OK) return rc;
    std::vector<int32_t> ids(T);
    for (int t = 0; t < T; t++) ids[t] = (int32_t)(f0 + t);
    std::vector<TcTile> tt;
    const int CT = (ctx->N + ctx->tc_train.SCt - 1) / ctx->tc_train.SCt;
    for (int ct = 0; ct < CT; ct++)
      for (int t = 0; t < T; t += kTcRows) tt.push_back({t, std::min(kTcRows, T - t), v * CT + ct, ct * ctx->tc_train.SCt, v, 0});
    DevBuf tl2;
    CK(tl2.ensure(sizeof(TcTile) * tt.size()));
    CK(ctx->frame_ids_d.ensure(sizeof(int32_t) * T));
    CK(cudaMemcpyAsync(tl2.p, tt.data(), sizeof(TcTile) * tt.size(), cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(ctx->frame_ids_d.p, ids.data(), sizeof(int32_t) * T, cudaMemcpyHostToDevice, ctx->st));
    ctx->u2m.clear();  // frame_ids_d was overwritten: the training map must be rebuilt
    rc = launch_emis_tc<true>(ctx, tl2.as<TcTile>(), (int)tt.size(), lb.as<float>() - f0 * ctx->N, 0, ctx->N, ps.as<float>() - f0 * ctx->G);
    if (rc) return rc;
    CK(cudaStreamSynchronize(ctx->st));
    tl2.release();
  } else {
    rc = launch_emis<true>(ctx, tl.as<EmisTile>(), (int64_t)tiles.size(), lb.as<float>(), f0, ctx->N, 0,
                           ps.as<float>() - f0 * ctx->G);
    if (rc) return rc;
  }
  std::vector<float> hl((size_t)T * ctx->N), hp((size_t)T * ctx->G);
  CK(cudaMemcpyAsync(hl.data(), lb.p, sizeof(float) * hl.size(), cudaMemcpyDeviceToHost, ctx->st));
  CK(cudaMemcpyAsync(hp.data(), ps.p, sizeof(float) * hp.size(), cudaMemcpyDeviceToHost, ctx->st));
  CK(cudaStreamSynchronize(ctx->st));
  for (size_t k = 0; k < hl.size(); k++) logb[k] = (double)hl[k];
  if (post)
    for (size_t k = 0; k < hp.size(); k++) post[k] = (double)hp[k];
  tl.release(); lb.release(); ps.release();
  return HMMCU_OK;
}

// ----------------------------------------------------------------------- decode (all cells) ----
template <int NS> struct ScoreLaunch {
  static void fwd(hmmcu_ctx *ctx, const float *logb, int64_t fbase, int64_t ldb, int u0, int nu, double *out, int emulate, bool lay8) {
    if (emulate) {  // the reference's linear-domain underflow, cell by cell (slow path, drop-in recogniser)
      dim3 grid((ctx->V + kScoreThreads - 1) / kScoreThreads, nu);
      k_fwd_score<NS><<<grid, kScoreThreads, 0, ctx->st>>>(logb, fbase, ldb, ctx->off_d.as<int64_t>(), u0, ctx->V,
                                                           ctx->A.as<double>(), out, emulate, lay8 ? 1 : 0);
      return;
    }
    const unsigned grid = (unsigned)(((int64_t)nu * ctx->V + kCellThreads - 1) / kCellThreads);
    // the single-precision log-domain chain (sum of the frame maxima in double)
#define FWD32(B, L) k_fwd_cells32<NS, B, L><<<grid, kCellThreads, 0, ctx->st>>>(logb, fbase, ldb, ctx->off_d.as<int64_t>(), u0, nu, ctx->V, ctx->A.as<double>(), out)
    if (ctx->banded) { if (lay8) FWD32(true, true); else FWD32(true, false); }
    else { if (lay8) FWD32(false, true); else FWD32(false, false); }
#undef FWD32
  }
  static void vit(hmmcu_ctx *ctx, const float *logb, int64_t fbase, int64_t ldb, int u0, int nu, double *out, bool lay8) {
    const unsigned grid = (unsigned)(((int64_t)nu * ctx->V + kCellThreads - 1) / kCellThreads);
    if (lay8) {
      if (ctx->banded)
        k_vit_cells8<NS, true><<<grid, kCellThreads, 0, ctx->st>>>(logb, fbase, ldb, ctx->off_d.as<int64_t>(), u0, nu, ctx->V,
                                                                   ctx->A.as<double>(), out);
      else
        k_vit_cells8<NS, false><<<grid, kCellThreads, 0, ctx->st>>>(logb, fbase, ldb, ctx->off_d.as<int64_t>(), u0, nu, ctx->V,
                                                                    ctx->A.as<double>(), out);
      return;
    }
    if (ctx->banded)
      k_vit_cells<NS, true><<<grid, kCellThreads, 0, ctx->st>>>(logb, fbase, ldb, ctx->off_d.as<int64_t>(), u0, nu, ctx->V,
                                                                ctx->A.as<double>(), out);
    else
      k_vit_cells<NS, false><<<grid, kCellThreads, 0, ctx->st>>>(logb, fbase, ldb, ctx->off_d.as<int64_t>(), u0, nu, ctx->V,
                                                                 ctx->A.as<double>(), out);
  }
  static cudaError_t path(hmmcu_ctx *ctx, const double *logb64, const int32_t *map, double *score, int32_t *path) {
    const size_t smem = vit_smem_bytes(NS);
    const int grid = (ctx->U + kVitUtts - 1) / kVitUtts;
    cudaError_t e;
    if (ctx->banded) {
      if ((e = cudaFuncSetAttribute(k_viterbi<NS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
      k_viterbi<NS, true><<<grid, kVitThreads, smem, ctx->st>>>(logb64, ctx->off_d.as<int64_t>(), map, ctx->A.as<double>(), ctx->U,
                                                                ctx->psi_ws.as<unsigned long long>(), score, path);
    } else {
      if ((e = cudaFuncSetAttribute(k_viterbi<NS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
      k_viterbi<NS, false><<<grid, kVitThreads, smem, ctx->st>>>(logb64, ctx->off_d.as<int64_t>(), map, ctx->A.as<double>(), ctx->U,
                                                                 ctx->psi_ws.as<unsigned long long>(), score, path);
    }
    return cudaSuccess;
  }
};

#define DISPATCH_N(n, stmt)                       \
  switch (n) {                                    \
    case 1: { constexpr int NS = 1; stmt; } break; \
    case 2: { constexpr int NS = 2; stmt; } break; \
    case 3: { constexpr int NS = 3; stmt; } break; \
    case 4: { constexpr int NS = 4; stmt; } break; \
    case 5: { constexpr int NS = 5; stmt; } break; \
    case 6: { constexpr int NS = 6; stmt; } break; \
    case 7: { constexpr int NS = 7; stmt; } break; \
    case 8: { constexpr int NS = 8; stmt; } break; \
    default: return fail(ctx, HMMCU_EINVAL, "N=%d states not supported", n); \
  }

// mode 0: forward score, 1: Viterbi score
// log-emissions of frames [fb0, fb1) against all V models of context c into c->logb ([frames][V*N])
// lay8: in = the caller can read k_emis_dec's interleaved layout (dec_logb_index); out = the layout that was written
static int decode_emissions(hmmcu_ctx *ctx, int64_t fb0, int64_t fb1, bool *lay8) {
  const int64_t S = (int64_t)ctx->V * ctx->N;
  int rc;
  const bool want8 = lay8 && *lay8;
  if (lay8) *lay8 = false;
  CK(ctx->logb.ensure(sizeof(float) * dec_logb_floats(fb1 - fb0, S)));
  if (tc_supported(ctx) && ws_supported(ctx)) {
    if ((rc = ensure_ws_images(ctx, 1)) != HMMCU_OK) return rc;
    const int nfr = (int)(fb1 - fb0), ntl = (nfr + kTcRows - 1) / kTcRows;
    t_begin(ctx, "emis");
    rc = HMMCU_EINVAL;
    if (want8 && dec_supported(ctx) && ctx->ws_dec.TN <= kWsMaxTN) {
      rc = launch_emis_dec(ctx, ntl, nfr, ctx->logb.as<float>(), fb0, S);
      if (rc == HMMCU_OK) *lay8 = true;
    }
    if (rc != HMMCU_OK) rc = launch_emis_ws<false>(ctx, nullptr, (int64_t)ctx->ws_dec.nimg * ntl, ntl, nfr, ctx->logb.as<float>(), fb0, S);
    if (rc) return rc;
    t_end(ctx, "emis");
  } else if (tc_supported(ctx)) {
    if ((rc = ensure_tc_images(ctx, 1)) != HMMCU_OK) return rc;
    std::vector<TcTile> tt;
    for (int64_t f = fb0; f < fb1; f += kTcRows) tt.push_back({(int32_t)(f - fb0), (int)std::min<int64_t>(kTcRows, fb1 - f), 0, 0, 0, 0});
    CK(ctx->tc_tiles_dec.ensure(sizeof(TcTile) * tt.size()));
    CK(cudaMemcpyAsync(ctx->tc_tiles_dec.p, tt.data(), sizeof(TcTile) * tt.size(), cudaMemcpyHostToDevice, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    t_begin(ctx, "emis");
    rc = launch_emis_tc<false>(ctx, ctx->tc_tiles_dec.as<TcTile>(), (int)tt.size(), ctx->logb.as<float>(), fb0, S, nullptr);
    if (rc) return rc;
    t_end(ctx, "emis");
  } else {
    std::vector<EmisTile> tiles;
    for (int64_t f = fb0; f < fb1; f += kEmisTF)
      for (int v = 0; v < ctx->V; v++) tiles.push_back({f, (int)std::min<int64_t>(kEmisTF, fb1 - f), v});
    CK(ctx->tiles_dec.ensure(sizeof(EmisTile) * tiles.size()));
    CK(cudaMemcpyAsync(ctx->tiles_dec.p, tiles.data(), sizeof(EmisTile) * tiles.size(), cudaMemcpyHostToDevice, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));  // `tiles` goes out of scope
    t_begin(ctx, "emis");
    rc = launch_emis<false>(ctx, ctx->tiles_dec.as<EmisTile>(), (int64_t)tiles.size(), ctx->logb.as<float>(), fb0, S, 1, nullptr);
    if (rc) return rc;
    t_end(ctx, "emis");
  }
  return HMMCU_OK;
}

// mode 0: forward score, 1: Viterbi score
static int score_all(hmmcu_ctx *ctx, double *out_host, int mode, int emulate) {
  if (!ctx || !out_host) return HMMCU_EINVAL;
  if (ctx->primary) return fail(ctx, HMMCU_EINVAL, "scores: this context is a linked stream; call its primary");
  CK(cudaSetDevice(ctx->dev));
  int rc = ensure_packed(ctx);
  if (rc) return rc;
  if ((rc = check_linked(ctx)) != HMMCU_OK) return rc;
  for (hmmcu_ctx *q : ctx->linked)
    if ((rc = ensure_packed(q)) != HMMCU_OK) return fail(ctx, rc, "linked stream: %s", q->err);
  if (ctx->U == 0) return HMMCU_OK;
  const int64_t S = (int64_t)ctx->V * ctx->N;
  CK(ctx->score_d.ensure(sizeof(double) * (size_t)ctx->U * ctx->V));
  t_collect(ctx, "emis");
  t_collect(ctx, mode == 0 ? "score" : "viterbi");
  // utterance batches so that the log-emission buffer stays under ~6 GiB (a third of the free memory when that is less):
  // large batches keep the tail of k_emis_dec's rounds small (every CTA walks all images once per frame tile it holds)
  int64_t budget_bytes = 6144ll << 20;
  if (ctx->dec_budget_kb > 0) budget_bytes = (int64_t)ctx->dec_budget_kb << 10;  // tests: many small batches
  else if ((int64_t)(sizeof(float) * dec_logb_floats(ctx->off[ctx->U] - ctx->off[0], S)) > std::max<int64_t>((int64_t)ctx->logb.cap, 256ll << 20)) {
    // (only a call that needs a larger buffer than the context already holds asks the driver: cudaMemGetInfo costs
    // 0.2-0.5 ms, as much as a whole small decode)
    size_t mem_free = 0, mem_total = 0;
    if (cudaMemGetInfo(&mem_free, &mem_total) == cudaSuccess) budget_bytes = std::min<int64_t>(budget_bytes, (int64_t)((mem_free + ctx->logb.cap) / 3));
    else cudaGetLastError();
    budget_bytes = std::max<int64_t>(budget_bytes, 256ll << 20);
  }
  const int64_t budget_frames = std::max<int64_t>(ctx->Tmax, budget_bytes / (4 * S));
  // the scores of a batch go back to the host (copy stream) while the next batch is computed
  // (a call that fits one batch copies on the context's stream: no events, no second stream)
  const bool one_batch = ctx->off[ctx->U] - ctx->off[0] <= budget_frames;
  cudaEvent_t ev_done[2] = {nullptr, nullptr};
  for (int k = 0; k < 2 && !one_batch; k++) CK(cudaEventCreateWithFlags(&ev_done[k], cudaEventDisableTiming));
  struct EvGuard { cudaEvent_t *e; ~EvGuard() { for (int k = 0; k < 2; k++) if (e[k]) cudaEventDestroy(e[k]); } } ev_guard{ev_done};
  int pend_u0 = -1, pend_u1 = -1, nbatch = 0;
  auto copy_back = [&](int a, int b, cudaEvent_t ev) -> cudaError_t {
    cudaError_t e = cudaStreamWaitEvent(ctx->st_copy, ev, 0);
    if (e != cudaSuccess) return e;
    return cudaMemcpyAsync(out_host + (size_t)a * ctx->V, ctx->score_d.as<double>() + (size_t)a * ctx->V, sizeof(double) * (size_t)(b - a) * ctx->V,
                           cudaMemcpyDeviceToHost, ctx->st_copy);
  };
  int u0 = 0;
  while (u0 < ctx->U) {
    int u1 = u0;
    while (u1 < ctx->U && ctx->off[u1 + 1] - ctx->off[u0] <= budget_frames) u1++;
    if (u1 == u0) u1 = u0 + 1;
    const int64_t fb0 = ctx->off[u0], fb1 = ctx->off[u1];
    // the interleaved layout of k_emis_dec is read by k_fwd_cells32, k_vit_cells8 and k_fwd_score; with several feature
    // streams every stream has to write it (their log-emissions are added element by element)
    auto can8 = [](const hmmcu_ctx *c) { return tc_supported(c) && ws_supported(c) && dec_supported(c); };
    bool all8 = can8(ctx);
    for (hmmcu_ctx *q : ctx->linked) all8 = all8 && can8(q);
    bool lay8 = all8;
    if ((rc = decode_emissions(ctx, fb0, fb1, &lay8)) != HMMCU_OK) return rc;
    for (hmmcu_ctx *q : ctx->linked) {  // multi-stream models: the product of the streams' densities (R-FS:341-364)
      bool l8 = all8;
      if ((rc = decode_emissions(q, fb0, fb1, &l8)) != HMMCU_OK) return fail(ctx, rc, "linked stream: %s", q->err);
      if (l8 != lay8) return fail(ctx, HMMCU_ECUDA, "linked stream: the streams' log-emissions differ in layout");
      const int64_t n = (int64_t)dec_logb_floats(fb1 - fb0, S);  // whole blocks of 8 frames (>= the frames either layout holds)
      const int fl = (mode == 0 && emulate) ? 1 : 0;  // underflow emulation: per stream, before the product
      k_add_logb<<<(int)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8), 256, 0, ctx->st>>>(ctx->logb.as<float>(), ctx->logb.as<float>(),
                                                                                                     q->logb.as<float>(), n, fl && q == ctx->linked[0], fl);
      LAUNCH_CHECK();
    }
    t_begin(ctx, mode == 0 ? "score" : "viterbi");
    if (mode == 0) {
      DISPATCH_N(ctx->N, ScoreLaunch<NS>::fwd(ctx, ctx->logb.as<float>(), fb0, S, u0, u1 - u0, ctx->score_d.as<double>(), emulate, lay8));
    } else {
      DISPATCH_N(ctx->N, ScoreLaunch<NS>::vit(ctx, ctx->logb.as<float>(), fb0, S, u0, u1 - u0, ctx->score_d.as<double>(), lay8));
    }
    LAUNCH_CHECK();
    t_end(ctx, mode == 0 ? "score" : "viterbi");
    if (!one_batch) {
      CK(cudaEventRecord(ev_done[nbatch & 1], ctx->st));
      if (pend_u0 >= 0) CK(copy_back(pend_u0, pend_u1, ev_done[(nbatch - 1) & 1]));  // blocks this thread for pageable memory; the device works on
      pend_u0 = u0; pend_u1 = u1;
    }
    nbatch++;
    u0 = u1;
  }
  if (one_batch) {
    CK(cudaMemcpyAsync(out_host, ctx->score_d.p, sizeof(double) * (size_t)ctx->U * ctx->V, cudaMemcpyDeviceToHost, ctx->st));
  } else {
    if (pend_u0 >= 0) CK(copy_back(pend_u0, pend_u1, ev_done[(nbatch - 1) & 1]));
    CK(cudaStreamSynchronize(ctx->st_copy));
  }
  CK(cudaStreamSynchronize(ctx->st));
  return HMMCU_OK;
}

int hmmcu_forward_scores(hmmcu_ctx *ctx, double *logp, int emulate_underflow) { return score_all(ctx, logp, 0, emulate_underflow); }
int hmmcu_viterbi_scores(hmmcu_ctx *ctx, double *score) { return score_all(ctx, score, 1, 0); }

int hmmcu_rank(hmmcu_ctx *ctx, const double *logp, int U, int V, double weight, int32_t *label, int32_t *second) {
  if (!ctx || !logp || !label || U < 0 || V < 1) return fail(ctx, HMMCU_EINVAL, "rank: bad arguments");
  if (U == 0) return HMMCU_OK;
  CK(cudaSetDevice(ctx->dev));
  CK(ctx->rank_in.ensure(sizeof(double) * (size_t)U * V));
  CK(ctx->rank_out.ensure(sizeof(int32_t) * 2 * (size_t)U));
  CK(cudaMemcpyAsync(ctx->rank_in.p, logp, sizeof(double) * (size_t)U * V, cudaMemcpyHostToDevice, ctx->st));
  k_rank<<<(U + 127) / 128, 128, 0, ctx->st>>>(ctx->rank_in.as<double>(), U, V, weight, ctx->rank_out.as<int32_t>(),
                                               ctx->rank_out.as<int32_t>() + U);
  LAUNCH_CHECK();
  CK(cudaMemcpyAsync(label, ctx->rank_out.p, sizeof(int32_t) * U, cudaMemcpyDeviceToHost, ctx->st));
  if (second) CK(cudaMemcpyAsync(second, ctx->rank_out.as<int32_t>() + U, sizeof(int32_t) * U, cudaMemcpyDeviceToHost, ctx->st));
  CK(cudaStreamSynchronize(ctx->st));
  return HMMCU_OK;
}

// ------------------------------------------------------------------------------------ E-step ----
static int set_train_map(hmmcu_ctx *ctx, const int32_t *utt2model) {
  const int U = ctx->U, V = ctx->V;
  if ((int)ctx->u2m.size() == U && memcmp(ctx->u2m.data(), utt2model, sizeof(int32_t) * U) == 0) return HMMCU_OK;
  for (int u = 0; u < U; u++)
    if (utt2model[u] < -1 || utt2model[u] >= V) return fail(ctx, HMMCU_EINVAL, "utt2model[%d]=%d out of range", u, utt2model[u]);
  std::vector<int32_t> start(V + 1, 0), utts(U);
  for (int u = 0; u < U; u++)
    if (utt2model[u] >= 0) start[utt2model[u] + 1]++;  // -1 = utterance masked out of this E-step
  ctx->max_utts_per_model = 0;
  for (int v = 0; v < V; v++) {
    ctx->max_utts_per_model = std::max(ctx->max_utts_per_model, start[v + 1]);
    start[v + 1] += start[v];
  }
  std::vector<int32_t> fill(start.begin(), start.end() - 1);
  for (int u = 0; u < U; u++)
    if (utt2model[u] >= 0) utts[fill[utt2model[u]]++] = u;
  std::vector<EmisTile> tiles;
  for (int u = 0; u < U; u++) {
    if (utt2model[u] < 0) continue;
    const int64_t f0 = ctx->off[u];
    const int T = (int)(ctx->off[u + 1] - f0);
    for (int t = 0; t < T; t += kEmisTF) tiles.push_back({f0 + t, std::min(kEmisTF, T - t), utt2model[u]});
  }
  ctx->n_train_tiles = (int64_t)tiles.size();
  {  // tensor-core tiles: the frames of each model, concatenated, in rows of 128
    std::vector<int32_t> ids;
    ids.reserve((size_t)ctx->F);
    std::vector<TcTile> tt;
    const int SCt = std::min(std::max(1, kTcMaxTN / ctx->M), ctx->N);
    const int CT = (ctx->N + SCt - 1) / SCt;
    for (int v = 0; v < V; v++) {
      const int32_t r0 = (int32_t)ids.size();
      for (int k = start[v]; k < start[v + 1]; k++) {
        const int u = utts[k];
        for (int64_t f = ctx->off[u]; f < ctx->off[u + 1]; f++) ids.push_back((int32_t)f);
      }
      const int32_t r1 = (int32_t)ids.size();
      for (int ct = 0; ct < CT; ct++)
        for (int32_t r = r0; r < r1; r += kTcRows) tt.push_back({r, std::min<int32_t>(kTcRows, r1 - r), v * CT + ct, ct * SCt, v, 0});
    }
    ctx->n_tc_tiles_train = (int64_t)tt.size();
    {  // the same tiles under the warp-specialised kernel's image geometry
      std::vector<TcTile> wt;
      int SCw, TNw;
      ws_geometry(ctx, ctx->N, SCw, TNw);
      const int CTw = (ctx->N + SCw - 1) / SCw;
      int32_t r0w = 0;
      for (int v = 0; v < V; v++) {
        int32_t nfr = 0;
        for (int k = start[v]; k < start[v + 1]; k++) nfr += (int32_t)(ctx->off[utts[k] + 1] - ctx->off[utts[k]]);
        for (int ct = 0; ct < CTw; ct++)
          for (int32_t r = 0; r < nfr; r += kTcRows) wt.push_back({r0w + r, std::min<int32_t>(kTcRows, nfr - r), v * CTw + ct, ct * SCw, v, 0});
        r0w += nfr;
      }
      ctx->n_ws_tiles_train = (int64_t)wt.size();
      CK(ctx->ws_tiles_train.ensure(sizeof(TcTile) * std::max<size_t>(wt.size(), 1)));
      CK(cudaMemcpyAsync(ctx->ws_tiles_train.p, wt.data(), sizeof(TcTile) * wt.size(), cudaMemcpyHostToDevice, ctx->st));
      CK(cudaStreamSynchronize(ctx->st));
    }
    {  // accumulate-kernel units, ordered (model, row block, tile)
      std::vector<TcTile> au;
      const int nRB = (ctx->G + 127) / 128;
      int32_t r0 = 0;
      for (int v = 0; v < V; v++) {
        int32_t nfr = 0;
        for (int k = start[v]; k < start[v + 1]; k++) nfr += (int32_t)(ctx->off[utts[k] + 1] - ctx->off[utts[k]]);
        for (int rb = 0; rb < nRB; rb++)
          for (int32_t r = 0; r < nfr; r += kTcRows) au.push_back({r0 + r, std::min<int32_t>(kTcRows, nfr - r), v * nRB + rb, 0, v, rb});
        r0 += nfr;
      }
      ctx->n_acc_units = (int64_t)au.size();
      CK(ctx->acc_units.ensure(sizeof(TcTile) * std::max<size_t>(au.size(), 1)));
      CK(cudaMemcpyAsync(ctx->acc_units.p, au.data(), sizeof(TcTile) * au.size(), cudaMemcpyHostToDevice, ctx->st));
      CK(cudaStreamSynchronize(ctx->st));
      // the same units in sub-tiles of kAccSub frames for the warp-specialised kernel
      std::vector<TcTile> a64;
      r0 = 0;
      for (int v = 0; v < V; v++) {
        int32_t nfr = 0;
        for (int k = start[v]; k < start[v + 1]; k++) nfr += (int32_t)(ctx->off[utts[k] + 1] - ctx->off[utts[k]]);
        for (int rb = 0; rb < nRB; rb++)
          for (int32_t r = 0; r < nfr; r += kAccSub) a64.push_back({r0 + r, std::min<int32_t>(kAccSub, nfr - r), v * nRB + rb, 0, v, rb});
        r0 += nfr;
      }
      ctx->n_acc_units64 = (int64_t)a64.size();
      CK(ctx->acc_units64.ensure(sizeof(TcTile) * std::max<size_t>(a64.size(), 1)));
      CK(cudaMemcpyAsync(ctx->acc_units64.p, a64.data(), sizeof(TcTile) * a64.size(), cudaMemcpyHostToDevice, ctx->st));
      {  // scratch slots of k_accum_ws: CTA c covers units [c per, (c+1) per) and writes the partial sums of
         // its j-th distinct image (j < kAccSlots) into slot c kAccSlots + j; per image, the slots to add up
        const int64_t nun = (int64_t)a64.size();
        const int grid = (int)std::min<int64_t>(nun, ctx->sm_count);
        const int nimg = V * nRB;
        std::vector<std::vector<int32_t>> lists(nimg);
        if (grid > 0) {
          const int64_t per = (nun + grid - 1) / grid;
          for (int c = 0; c < grid; c++) {
            int j = -1, prev = -1;
            for (int64_t k = c * per; k < std::min(nun, (c + 1) * per); k++) {
              if (a64[k].img != prev) { prev = a64[k].img; j++; if (j < kAccSlots) lists[prev].push_back(c * kAccSlots + j); }
            }
          }
        }
        std::vector<int32_t> sstart(nimg + 1, 0), sids;
        for (int i = 0; i < nimg; i++) { sids.insert(sids.end(), lists[i].begin(), lists[i].end()); sstart[i + 1] = (int32_t)sids.size(); }
        CK(ctx->acc_slot_start.ensure(sizeof(int32_t) * sstart.size()));
        CK(ctx->acc_slot_ids.ensure(sizeof(int32_t) * std::max<size_t>(sids.size(), 1)));
        CK(cudaMemcpyAsync(ctx->acc_slot_start.p, sstart.data(), sizeof(int32_t) * sstart.size(), cudaMemcpyHostToDevice, ctx->st));
        CK(cudaMemcpyAsync(ctx->acc_slot_ids.p, sids.data(), sizeof(int32_t) * sids.size(), cudaMemcpyHostToDevice, ctx->st));
        CK(ctx->acc_scratch.ensure(sizeof(float) * (size_t)std::max(grid, 1) * kAccSlots * tc_kp2(2 * ctx->DP) * 128));
      }
      {  // k_accum_h: units of kAhSub frames; state0 = the unit's tile in x16 (the row blocks of a model share its tiles);
         // the same slot scheme over this kernel's CTA ranges
        std::vector<TcTile> ah;
        std::vector<int2> tl;
        r0 = 0;
        for (int v = 0; v < V; v++) {
          int32_t nfr = 0;
          for (int k = start[v]; k < start[v + 1]; k++) nfr += (int32_t)(ctx->off[utts[k] + 1] - ctx->off[utts[k]]);
          const int32_t t0 = (int32_t)tl.size();
          for (int32_t r = 0; r < nfr; r += kAhSub) tl.push_back(make_int2(r0 + r, std::min<int32_t>(kAhSub, nfr - r)));
          for (int rb = 0; rb < nRB; rb++)
            for (int32_t r = 0; r < nfr; r += kAhSub) ah.push_back({r0 + r, std::min<int32_t>(kAhSub, nfr - r), v * nRB + rb, t0 + r / kAhSub, v, rb});
          r0 += nfr;
        }
        ctx->n_acc_unitsH = (int64_t)ah.size();
        ctx->n_x16_tiles = (int64_t)tl.size();
        CK(ctx->acc_unitsH.ensure(sizeof(TcTile) * std::max<size_t>(ah.size(), 1)));
        CK(ctx->x16_tiles.ensure(sizeof(int2) * std::max<size_t>(tl.size(), 1)));
        CK(cudaMemcpyAsync(ctx->acc_unitsH.p, ah.data(), sizeof(TcTile) * ah.size(), cudaMemcpyHostToDevice, ctx->st));
        CK(cudaMemcpyAsync(ctx->x16_tiles.p, tl.data(), sizeof(int2) * tl.size(), cudaMemcpyHostToDevice, ctx->st));
        const int64_t nun = (int64_t)ah.size();
        const int grid = (int)std::min<int64_t>(nun, ctx->sm_count);
        const int nimg = V * nRB;
        std::vector<std::vector<int32_t>> lists(nimg);
        if (grid > 0) {
          const int64_t per = (nun + grid - 1) / grid;
          for (int c = 0; c < grid; c++) {
            int j = -1, prev = -1;
            for (int64_t k = c * per; k < std::min(nun, (c + 1) * per); k++) {
              if (ah[k].img != prev) { prev = ah[k].img; j++; if (j < kAccSlots) lists[prev].push_back(c * kAccSlots + j); }
            }
          }
        }
        std::vector<int32_t> sstart(nimg + 1, 0), sids;
        for (int i = 0; i < nimg; i++) { sids.insert(sids.end(), lists[i].begin(), lists[i].end()); sstart[i + 1] = (int32_t)sids.size(); }
        CK(ctx->acc_slot_start_h.ensure(sizeof(int32_t) * sstart.size()));
        CK(ctx->acc_slot_ids_h.ensure(sizeof(int32_t) * std::max<size_t>(sids.size(), 1)));
        CK(cudaMemcpyAsync(ctx->acc_slot_start_h.p, sstart.data(), sizeof(int32_t) * sstart.size(), cudaMemcpyHostToDevice, ctx->st));
        CK(cudaMemcpyAsync(ctx->acc_slot_ids_h.p, sids.data(), sizeof(int32_t) * sids.size(), cudaMemcpyHostToDevice, ctx->st));
        CK(cudaStreamSynchronize(ctx->st));
      }
      CK(cudaStreamSynchronize(ctx->st));
    }
    CK(ctx->frame_ids_d.ensure(sizeof(int32_t) * std::max<size_t>(ids.size(), 1)));
    CK(ctx->tc_tiles_train.ensure(sizeof(TcTile) * std::max<size_t>(tt.size(), 1)));
    CK(cudaMemcpyAsync(ctx->frame_ids_d.p, ids.data(), sizeof(int32_t) * ids.size(), cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(ctx->tc_tiles_train.p, tt.data(), sizeof(TcTile) * tt.size(), cudaMemcpyHostToDevice, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
  }
  CK(ctx->u2m_d.ensure(sizeof(int32_t) * std::max(U, 1)));
  CK(ctx->mus_d.ensure(sizeof(int32_t) * (V + 1)));
  CK(ctx->mu_d.ensure(sizeof(int32_t) * std::max(U, 1)));
  CK(ctx->tiles_d.ensure(sizeof(EmisTile) * std::max<size_t>(tiles.size(), 1)));
  CK(cudaMemcpyAsync(ctx->u2m_d.p, utt2model, sizeof(int32_t) * U, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemcpyAsync(ctx->mus_d.p, start.data(), sizeof(int32_t) * (V + 1), cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemcpyAsync(ctx->mu_d.p, utts.data(), sizeof(int32_t) * U, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemcpyAsync(ctx->tiles_d.p, tiles.data(), sizeof(EmisTile) * tiles.size(), cudaMemcpyHostToDevice, ctx->st));
  {  // k_fb_res: the live utterances longest first, cut into batches that fit one team's shared memory and hold at most
     // ceil(live / teams) utterances, so that a small corpus still reaches every team of the grid (a batch's time is its
     // longest chain plus staging and the gamma phase over all its frames); the row of every utterance in the
     // per-utterance statistics (= its position in the model-grouped list)
    const int nlive = start[V];
    ctx->n_live = nlive;
    const int teams = kResTeams * std::max(ctx->sm_count, 1);
    const int per_batch = std::max(1, std::min(kResMaxUtts, (nlive + teams - 1) / teams));
    std::vector<int32_t> order(utts.begin(), utts.begin() + nlive), upos(std::max(U, 1), 0);
    for (int k = 0; k < nlive; k++) upos[utts[k]] = k;
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return ctx->off[a + 1] - ctx->off[a] > ctx->off[b + 1] - ctx->off[b]; });
    const int64_t cap = res_slot_words_rt(ctx->N);
    std::vector<ResBatch> rb;
    ctx->res_fits = cap > 0;
    ctx->res_batch_max = 0;
    for (int k = 0; k < nlive && ctx->res_fits;) {
      int64_t used = 0;
      int n = 0;
      while (k + n < nlive && n < per_batch) {
        const int64_t w = res_utt_words(ctx->N, ctx->off[order[k + n] + 1] - ctx->off[order[k + n]]);
        if (used + w > cap) break;
        used += w;
        n++;
      }
      if (n == 0) { ctx->res_fits = false; break; }  // an utterance longer than a team's shared memory: k_fb takes the E-step
      rb.push_back({k, n});
      ctx->res_batch_max = std::max(ctx->res_batch_max, n);
      k += n;
    }
    ctx->n_res_batches = ctx->res_fits ? (int64_t)rb.size() : 0;
    CK(ctx->res_order.ensure(sizeof(int32_t) * std::max(nlive, 1)));
    CK(ctx->res_upos.ensure(sizeof(int32_t) * std::max(U, 1)));
    CK(ctx->res_batches.ensure(sizeof(ResBatch) * std::max<size_t>(rb.size(), 1)));
    if (!ctx->res_counter.p) {  // k_fb_res leaves it at 0 after every launch
      CK(ctx->res_counter.ensure(sizeof(int)));
      CK(cudaMemsetAsync(ctx->res_counter.p, 0, sizeof(int), ctx->st));
    }
    CK(ctx->ustats.ensure(sizeof(double) * (size_t)std::max(nlive, 1) * res_stats_row(std::min(ctx->N, 8))));
    CK(cudaMemcpyAsync(ctx->res_order.p, order.data(), sizeof(int32_t) * nlive, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(ctx->res_upos.p, upos.data(), sizeof(int32_t) * U, cudaMemcpyHostToDevice, ctx->st));
    if (!rb.empty()) CK(cudaMemcpyAsync(ctx->res_batches.p, rb.data(), sizeof(ResBatch) * rb.size(), cudaMemcpyHostToDevice, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
  }
  CK(cudaStreamSynchronize(ctx->st));
  ctx->u2m.assign(utt2model, utt2model + U);
  ctx->cfg_epoch++;
  ctx->map_version++;
  return HMMCU_OK;
}

// The expanded half-precision frame tiles of k_accum_h: packed when the features or the training map have changed
// (not per EM iteration -- the models do not enter), with the data-only scales of k_acc16_scales.
// Preparation (allocations, the scales): need_pack tells the launch sequence to pack the tiles (launch_pack_x16), which it
// does beside the emission and forward-backward kernels -- only the accumulate kernel reads them.
static int prepare_x16(hmmcu_ctx *ctx, bool &need_pack) {
  need_pack = !(ctx->x16_x == ctx->x_version && ctx->x16_map == ctx->map_version);
  if (!need_pack) return HMMCU_OK;
  CK(ctx->acc_sc.ensure(sizeof(float) * kAhScN * ctx->DP));
  CK(ctx->x16.ensure(ah_tile_bytes(2 * ctx->DP) * (size_t)std::max<int64_t>(ctx->n_x16_tiles, 1)));
  if (ctx->x16_x != ctx->x_version) {  // the scales follow the data's radius; the W images follow the scales
    k_acc16_scales<<<1, 64, 0, ctx->st>>>(ctx->xabs_d.as<unsigned int>(), ctx->D, ctx->DP, ctx->acc_sc.as<float>());
    LAUNCH_CHECK();
    ctx->acc_dirty = true;
  }
  return HMMCU_OK;
}
static int launch_pack_x16(hmmcu_ctx *ctx, cudaStream_t st) {
  if (ctx->n_x16_tiles > 0) {
    k_pack_x16<<<(unsigned)ctx->n_x16_tiles, 256, 0, st>>>(ctx->x16_tiles.as<int2>(), ctx->frame_ids_d.as<int32_t>(), ctx->x32.as<float>(),
                                                          ctx->acc_sc.as<float>(), ctx->DP, ctx->x16.as<unsigned char>());
    LAUNCH_CHECK();
  }
  return HMMCU_OK;
}

// phases: 1 = clear the statistics + emissions, 2 = forward-backward, 4 = mixture accumulators.  fb_logb / acc_gamma
// replace the context's own log-emissions in the recursions / its own state posteriors in the accumulators
// (multi-stream models); with all phases and no replacement this is the plain single-stream E-step.  align: phase 2 is
// the Viterbi alignment (k_vtrain) instead of forward-backward; it writes the same gamma and statistics, and its path.
static int estep_core(hmmcu_ctx *ctx, const int32_t *utt2model, int phases, const float *fb_logb, const float *acc_gamma,
                      bool align = false) {
  CK(cudaSetDevice(ctx->dev));
  int rc = ensure_packed(ctx);
  if (rc) return rc;
  if (ctx->U > 0 && !utt2model) return fail(ctx, HMMCU_EINVAL, "estep: utt2model is NULL");
  const int N = ctx->N, M = ctx->M, D = ctx->D, DP = ctx->DP, G = ctx->G, V = ctx->V, U = ctx->U;
  const int64_t ss = hmmcu_stats_size(N, M, D);
  const int64_t off_S0 = (int64_t)N * N + 2 * N, off_S1 = off_S0 + G, off_S2 = off_S1 + (int64_t)G * D,
                off_lp = off_S2 + (int64_t)G * D;
  ctx->stats_n = ss * V;
  CK(ctx->stats.ensure(sizeof(double) * ctx->stats_n));
  // ---- preparation (host work, allocations, packed model forms): everything the launch sequence needs ----
  const bool use_tc = U > 0 && tc_supported(ctx);
  const bool ws_emis = use_tc && ws_supported(ctx);
  const bool ws_acc = use_tc && ctx->use_ws_acc && DP <= 40 && ws_acc_smem_bytes(2 * DP) <= 227 * 1024;
  const bool h_acc = ws_acc && h_acc_on(ctx);
  bool pack16 = false;
  if (U > 0) {
    rc = set_train_map(ctx, utt2model);
    if (rc) return rc;
    const int64_t F = ctx->F;
    CK(ctx->logb.ensure(sizeof(float) * F * N));
    if (!use_tc) CK(ctx->post.ensure(sizeof(float) * F * G));
    CK(ctx->gamma.ensure(sizeof(float) * F * N));
    if (align) {
      CK(ctx->psi_ws.ensure(sizeof(unsigned long long) * F));
      CK(ctx->path_d.ensure(sizeof(int32_t) * F));
    } else if (!res_fb_on(ctx)) {  // k_fb_res keeps alpha / beta on the SM
      CK(ctx->alpha_ws.ensure(sizeof(uint32_t) * F * kFbRow));
      CK(ctx->beta_ws.ensure(sizeof(uint32_t) * F * kFbRow));
    }
    CK(ctx->logp_utt_d.ensure(sizeof(double) * U));
    if (ws_emis) {
      if ((rc = ensure_ws_images(ctx, 0)) != HMMCU_OK) return rc;
    } else if (use_tc) {
      if ((rc = ensure_tc_images(ctx, 0)) != HMMCU_OK) return rc;
    }
    if (use_tc) {
      if (h_acc && (phases & 4) && (rc = prepare_x16(ctx, pack16)) != HMMCU_OK) return rc;
      if ((rc = ensure_acc_images(ctx)) != HMMCU_OK) return rc;
    } else {
      if ((rc = ensure_simt_pack(ctx)) != HMMCU_OK) return rc;
    }
  }
  ctx->train_path = ws_emis ? 2 : use_tc ? 1 : 0;
  t_single(ctx, "emis");
  // ---- the launch sequence: statistics cleared, emissions, forward-backward, accumulators ----
  const float *lb_fb = fb_logb ? fb_logb : ctx->logb.as<float>();
  const float *gm_acc = acc_gamma ? acc_gamma : ctx->gamma.as<float>();
  const bool res_fb = res_fb_on(ctx);
  auto enqueue = [&]() -> int {
    if (phases & 1) CK(cudaMemsetAsync(ctx->stats.p, 0, sizeof(double) * ctx->stats_n, ctx->st));
    if (U == 0) return HMMCU_OK;
    // masked utterances report 0 (k_fb_res writes the live ones only); cleared here, so that no memset node sits between the
    // emission kernel and k_fb_res
    if ((phases & 2) && res_fb && !align && ctx->n_live < U) CK(cudaMemsetAsync(ctx->logp_utt_d.p, 0, sizeof(double) * U, ctx->st));
    int rc2;
    bool fb_forked = false;
    const bool pack_forked = pack16 && !ctx->timing && (phases & 3) && ctx->mstep_fork;
    if (pack_forked) {  // the half-precision frame tiles, beside the emission and forward-backward kernels
      CK(cudaEventRecord(ctx->ev_fork[1], ctx->st));
      CK(cudaStreamWaitEvent(ctx->st_aux[1], ctx->ev_fork[1], 0));
      if ((rc2 = launch_pack_x16(ctx, ctx->st_aux[1])) != HMMCU_OK) return rc2;
      CK(cudaEventRecord(ctx->ev_join[1], ctx->st_aux[1]));
    }
    // 1. emissions (+ per-mixture posteriors on the CUDA-core path)
    if (phases & 1) {
    t_begin(ctx, "emis");
    if (ws_emis) rc2 = launch_emis_ws<true>(ctx, ctx->ws_tiles_train.as<TcTile>(), ctx->n_ws_tiles_train, 0, 0, ctx->logb.as<float>(), 0, N);
    else if (use_tc) rc2 = launch_emis_tc<true>(ctx, ctx->tc_tiles_train.as<TcTile>(), (int)ctx->n_tc_tiles_train, ctx->logb.as<float>(), 0, N, nullptr);
    else rc2 = launch_emis<true>(ctx, ctx->tiles_d.as<EmisTile>(), ctx->n_train_tiles, ctx->logb.as<float>(), 0, N, 0, ctx->post.as<float>());
    if (rc2) return rc2;
    t_end(ctx, "emis");
    }
    // 2. forward / backward, gamma, transition statistics, log-probabilities
    if (phases & 2) {
    const char *tname = align ? "align" : "fwdbwd";
    t_begin(ctx, tname);
    {
        if (align) {
        // the Viterbi alignment: per-utterance rows for k_fb_reduce below, or atomics into the statistics (vtrain_kernels.cuh)
        const int blocks = (U + kVtUtts - 1) / kVtUtts;
        const size_t vsm = vtrain_smem_bytes(N);
        double *rows = res_fb ? ctx->ustats.as<double>() : nullptr;
        if (ctx->banded) {
          DISPATCH_N(N, (k_vtrain<NS, true><<<blocks, kVtThreads, vsm, ctx->st>>>(
                            lb_fb, ctx->off_d.as<int64_t>(), ctx->u2m_d.as<int32_t>(), ctx->A.as<double>(), U,
                            ctx->psi_ws.as<unsigned long long>(), ctx->path_d.as<int32_t>(), ctx->gamma.as<float>(),
                            ctx->res_upos.as<int32_t>(), rows, ctx->stats.as<double>(), ss, off_lp, ctx->logp_utt_d.as<double>())));
        } else {
          DISPATCH_N(N, (k_vtrain<NS, false><<<blocks, kVtThreads, vsm, ctx->st>>>(
                            lb_fb, ctx->off_d.as<int64_t>(), ctx->u2m_d.as<int32_t>(), ctx->A.as<double>(), U,
                            ctx->psi_ws.as<unsigned long long>(), ctx->path_d.as<int32_t>(), ctx->gamma.as<float>(),
                            ctx->res_upos.as<int32_t>(), nullptr, ctx->stats.as<double>(), ss, off_lp, ctx->logp_utt_d.as<double>())));
        }
        LAUNCH_CHECK();
        } else if (res_fb) {
        // every utterance resident in shared memory: log-emissions read once, gamma written once (fbres_kernels.cuh)
        const int grid = res_grid(ctx);
        DISPATCH_N(N, CK(cudaFuncSetAttribute(k_fb_res<NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, kResSmemBytes));
                   CK(launch_pdl(k_fb_res<NS>, grid, kResThreads, kResSmemBytes, ctx->st, lb_fb, ctx->off_d.as<int64_t>(),
                                 ctx->u2m_d.as<int32_t>(), ctx->A.as<double>(), ctx->res_order.as<int32_t>(), ctx->res_upos.as<int32_t>(),
                                 ctx->res_batches.as<ResBatch>(), (int)ctx->n_res_batches, ctx->res_counter.as<int>(),
                                 ctx->gamma.as<float>(), ctx->ustats.as<double>(), ctx->logp_utt_d.as<double>())));
        LAUNCH_CHECK();
        }
        if (res_fb) {
        // the per-model sums of the transition statistics feed nothing before the M-step: beside the accumulate kernel
        fb_forked = !ctx->timing && (phases & 4) && ctx->mstep_fork;
        if (fb_forked) {
          CK(cudaEventRecord(ctx->ev_fork[0], ctx->st));
          CK(cudaStreamWaitEvent(ctx->st_aux[0], ctx->ev_fork[0], 0));
        }
        k_fb_reduce<<<V, 1024, 0, fb_forked ? ctx->st_aux[0] : ctx->st>>>(ctx->ustats.as<double>(), N, ctx->mus_d.as<int32_t>(), V, ctx->stats.as<double>(), ss,
                                                                        off_lp);
        LAUNCH_CHECK();
        if (fb_forked) CK(cudaEventRecord(ctx->ev_join[0], ctx->st_aux[0]));
      } else if (!align) {
      const int blocks = (U + kFbUtts - 1) / kFbUtts;
      const size_t fsm = fb_smem_bytes(N);
      if (ctx->banded) {
        DISPATCH_N(N, (cudaFuncSetAttribute(k_fb<NS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsm), k_fb<NS, true><<<blocks, kFbThreads, fsm, ctx->st>>>(
                          lb_fb, ctx->off_d.as<int64_t>(), ctx->u2m_d.as<int32_t>(), ctx->A.as<double>(), U,
                          ctx->alpha_ws.as<uint32_t>(), ctx->beta_ws.as<uint32_t>(), ctx->gamma.as<float>(), ctx->stats.as<double>(),
                          ss, off_lp, ctx->logp_utt_d.as<double>())));
      } else {
        DISPATCH_N(N, (cudaFuncSetAttribute(k_fb<NS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsm), k_fb<NS, false><<<blocks, kFbThreads, fsm, ctx->st>>>(
                          lb_fb, ctx->off_d.as<int64_t>(), ctx->u2m_d.as<int32_t>(), ctx->A.as<double>(), U,
                          ctx->alpha_ws.as<uint32_t>(), ctx->beta_ws.as<uint32_t>(), ctx->gamma.as<float>(), ctx->stats.as<double>(),
                          ss, off_lp, ctx->logp_utt_d.as<double>())));
      }
      LAUNCH_CHECK();
      }
    }
    t_end(ctx, tname);
    }
    // 3. mixture accumulators
    if (!(phases & 4)) {
      if (fb_forked) CK(cudaStreamWaitEvent(ctx->st, ctx->ev_join[0], 0));
      return HMMCU_OK;
    }
    if (pack_forked) CK(cudaStreamWaitEvent(ctx->st, ctx->ev_join[1], 0));
    else if (pack16) {
      t_begin(ctx, "pack_x16");
      if ((rc2 = launch_pack_x16(ctx, ctx->st)) != HMMCU_OK) return rc2;
      t_end(ctx, "pack_x16");
    }
    t_begin(ctx, "accum");
    if (h_acc) {
      const size_t smem = ah_smem_bytes(2 * DP);
      const int grid = (int)std::min<int64_t>(ctx->n_acc_unitsH, ctx->sm_count);
      const float *dsc = ctx->acc_sc.as<float>() + 5 * DP;
      if (grid > 0) {
        CK(cudaFuncSetAttribute(k_accum_h, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK(launch_pdl(k_accum_h, grid, kAhThreads, smem, ctx->st, ctx->acc_unitsH.as<TcTile>(), (int)ctx->n_acc_unitsH,
                      ctx->frame_ids_d.as<int32_t>(), ctx->x16.as<unsigned char>(), ctx->acc_images16.as<uint32_t>(), ctx->acc_kc.as<float>(),
                      ctx->logb.as<float>(), gm_acc, N, M, G, D, DP, ctx->stats.as<double>(), ss, off_S0, off_S1, off_S2,
                      ctx->acc_scratch.as<float>(), dsc));
        LAUNCH_CHECK();
      }
      CK(launch_pdl(k_finalize_slots, dim3(G, V), 64 * kFinParts, 0, ctx->st, ctx->stats.as<double>(), ss, G, D, DP, 2 * DP, (G + 127) / 128,
                    off_S0, off_S1, off_S2, ctx->ctr.as<double>(), ctx->mu.as<double>(), ctx->acc_scratch.as<float>(),
                    ctx->acc_slot_start_h.as<int32_t>(), ctx->acc_slot_ids_h.as<int32_t>(), dsc));
      LAUNCH_CHECK();
    } else if (ws_acc) {
      const size_t smem = ws_acc_smem_bytes(2 * DP);
      const int grid = (int)std::min<int64_t>(ctx->n_acc_units64, ctx->sm_count);
      if (grid > 0) {
        CK(cudaFuncSetAttribute(k_accum_ws, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_accum_ws<<<grid, kAccWsThreads, smem, ctx->st>>>(ctx->acc_units64.as<TcTile>(), (int)ctx->n_acc_units64, ctx->frame_ids_d.as<int32_t>(),
                                                           ctx->x32.as<float>(), ctx->acc_images.as<float>(), ctx->acc_kc.as<float>(),
                                                           ctx->logb.as<float>(), gm_acc, N, M, G, D, DP,
                                                           ctx->stats.as<double>(), ss, off_S0, off_S1, off_S2, ctx->acc_scratch.as<float>());
        LAUNCH_CHECK();
      }
      k_finalize_slots<<<dim3(G, V), 64 * kFinParts, 0, ctx->st>>>(ctx->stats.as<double>(), ss, G, D, DP, tc_kp2(2 * DP), (G + 127) / 128, off_S0,
                                                                  off_S1, off_S2, ctx->ctr.as<double>(), ctx->mu.as<double>(),
                                                                  ctx->acc_scratch.as<float>(), ctx->acc_slot_start.as<int32_t>(),
                                                                  ctx->acc_slot_ids.as<int32_t>());
      LAUNCH_CHECK();
    } else if (use_tc) {
      const size_t smem = tc_acc_smem_bytes(2 * DP);
      CK(cudaFuncSetAttribute(k_accum_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      const int grid = (int)std::min<int64_t>(ctx->n_acc_units, ctx->sm_count);
      if (grid > 0) {
        k_accum_tc<<<grid, kTcThreads, smem, ctx->st>>>(ctx->acc_units.as<TcTile>(), (int)ctx->n_acc_units, ctx->frame_ids_d.as<int32_t>(),
                                                        ctx->x32.as<float>(), ctx->acc_images.as<float>(), ctx->acc_kc.as<float>(),
                                                        ctx->logb.as<float>(), gm_acc, N, M, G, D, DP,
                                                        ctx->stats.as<double>(), ss, off_S0, off_S1, off_S2);
        LAUNCH_CHECK();
      }
      const int64_t total = (int64_t)V * G * D;
      k_finalize_stats<<<(unsigned)((total + 255) / 256), 256, 0, ctx->st>>>(ctx->stats.as<double>(), ss, V, G, D, off_S0, off_S1,
                                                                            off_S2, ctx->ctr.as<double>(), ctx->mu.as<double>());
      LAUNCH_CHECK();
    } else {
      const int NGG = kAccThreads / DP, GCH = NGG * kAccGPT;
      const int nz = (G + GCH - 1) / GCH;
      int nparts = std::max(1, (2 * ctx->sm_count + V * nz - 1) / (V * nz));
      nparts = std::min(nparts, std::max(1, ctx->max_utts_per_model));
      const size_t smem = sizeof(float) * (size_t)kAccTF * (DP + GCH);
      dim3 grid(nparts, V, nz);
      k_accum_simt<<<grid, kAccThreads, smem, ctx->st>>>(ctx->x32.as<float>(), gm_acc, ctx->post.as<float>(),
                                                         ctx->mu32.as<float>(), ctx->off_d.as<int64_t>(),
                                                         ctx->mus_d.as<int32_t>(), ctx->mu_d.as<int32_t>(), N, M, D, DP, nparts,
                                                         ctx->stats.as<double>(), ss, off_S0, off_S1, off_S2);
      LAUNCH_CHECK();
      const int64_t total = (int64_t)V * G * D;
      k_finalize_stats<<<(unsigned)((total + 255) / 256), 256, 0, ctx->st>>>(ctx->stats.as<double>(), ss, V, G, D, off_S0, off_S1,
                                                                            off_S2, ctx->ctr.as<double>(), nullptr);
      LAUNCH_CHECK();
    }
    t_end(ctx, "accum");
    if (fb_forked) CK(cudaStreamWaitEvent(ctx->st, ctx->ev_join[0], 0));
    return HMMCU_OK;
  };
  const uint64_t key = 1u | ((ctx->use_res_fb && ctx->banded && ctx->res_fits) ? (1u << 8) : 0u) | (use_tc ? 2u : 0u) | (ws_emis ? 4u : 0u) | (ws_acc ? 8u : 0u) | (h_acc ? 32u : 0u) | (pack16 ? 64u : 0u) | (ctx->banded ? 16u : 0u) | (align ? (1u << 9) : 0u);
  ctx->last_tc = use_tc;
  if (phases & 4) ctx->last_acc_h = h_acc;
  // (pieces of a multi-stream E-step: plain launches)
  const int rcq = (phases != 7 || fb_logb || acc_gamma) ? enqueue() : run_graphed(ctx, align ? ctx->g_estep_vit : ctx->g_estep, key, enqueue);
  if (rcq == HMMCU_OK && pack16) { ctx->x16_x = ctx->x_version; ctx->x16_map = ctx->map_version; }
  return rcq;
}

// the host copies of an E-step's results (each may be NULL); path[F] is written by the Viterbi alignment only
static int estep_download(hmmcu_ctx *ctx, double *stats, double *logp_utt, int32_t *path) {
  const int U = ctx->U;
  if (logp_utt && U > 0) CK(cudaMemcpyAsync(logp_utt, ctx->logp_utt_d.p, sizeof(double) * U, cudaMemcpyDeviceToHost, ctx->st));
  if (stats) CK(cudaMemcpyAsync(stats, ctx->stats.p, sizeof(double) * ctx->stats_n, cudaMemcpyDeviceToHost, ctx->st));
  if (path && U > 0 && ctx->F > 0) CK(cudaMemcpyAsync(path, ctx->path_d.p, sizeof(int32_t) * ctx->F, cudaMemcpyDeviceToHost, ctx->st));
  if (stats || logp_utt || path) CK(cudaStreamSynchronize(ctx->st));
  return HMMCU_OK;
}

int hmmcu_estep(hmmcu_ctx *ctx, const int32_t *utt2model, double *stats, double *logp_utt) {
  if (!ctx) return HMMCU_EINVAL;
  if (ctx->primary) return fail(ctx, HMMCU_EINVAL, "estep: this context is a linked stream; call its primary");
  int rc;
  const int U = ctx->U;
  if (ctx->linked.empty()) {
    if ((rc = estep_core(ctx, utt2model, 7, nullptr, nullptr)) != HMMCU_OK) return rc;
  } else {
    // multi-stream: per-stream emissions, their sum, ONE pair of recursions, per-stream accumulators
    if ((rc = check_linked(ctx)) != HMMCU_OK) return rc;
    if ((rc = estep_core(ctx, utt2model, 1, nullptr, nullptr)) != HMMCU_OK) return rc;
    for (hmmcu_ctx *q : ctx->linked)
      if ((rc = estep_core(q, utt2model, 1, nullptr, nullptr)) != HMMCU_OK) return fail(ctx, rc, "linked stream: %s", q->err);
    const int64_t n = ctx->F * ctx->N;
    if (U > 0 && n > 0) {
      CK(ctx->logb_joint.ensure(sizeof(float) * n));
      const float *acc = ctx->logb.as<float>();
      const int blocks = (int)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8);
      for (hmmcu_ctx *q : ctx->linked) {
        k_add_logb<<<blocks, 256, 0, ctx->st>>>(ctx->logb_joint.as<float>(), acc, q->logb.as<float>(), n);
        LAUNCH_CHECK();
        acc = ctx->logb_joint.as<float>();
      }
    }
    if ((rc = estep_core(ctx, utt2model, 6, ctx->logb_joint.as<float>(), nullptr)) != HMMCU_OK) return rc;
    for (hmmcu_ctx *q : ctx->linked) {
      if ((rc = estep_core(q, utt2model, 4, nullptr, ctx->gamma.as<float>())) != HMMCU_OK) return fail(ctx, rc, "linked stream: %s", q->err);
      k_copy_shared_stats<<<ctx->V, 64, 0, ctx->st>>>(q->stats.as<double>(), q->stats_n / q->V, ctx->stats.as<double>(), ctx->stats_n / ctx->V, ctx->V,
                                                      ctx->N * ctx->N + 2 * ctx->N);
      LAUNCH_CHECK();
    }
  }
  return estep_download(ctx, stats, logp_utt, nullptr);
}

int hmmcu_estep_viterbi(hmmcu_ctx *ctx, const int32_t *utt2model, double *stats, double *logp_utt, int32_t *path) {
  if (!ctx) return HMMCU_EINVAL;
  if (ctx->primary) return fail(ctx, HMMCU_EINVAL, "estep_viterbi: this context is a linked stream; call its primary");
  if (!ctx->linked.empty()) return fail(ctx, HMMCU_EINVAL, "estep_viterbi: Viterbi training of multi-stream (linked) models is not supported");
  const int rc = estep_core(ctx, utt2model, 7, nullptr, nullptr, true);
  if (rc != HMMCU_OK) return rc;
  return estep_download(ctx, stats, logp_utt, path);
}

// ------------------------------------------------------------------------- device-resident EM ----
int hmmcu_em_reset(hmmcu_ctx *ctx) {
  if (!ctx || !ctx->have_models) return fail(ctx, HMMCU_EINVAL, "em_reset: set the models first");
  CK(cudaSetDevice(ctx->dev));
  const int V = ctx->V;
  CK(ctx->em_old.ensure(sizeof(double) * V));
  CK(ctx->em_active.ensure(sizeof(int) * V));
  std::vector<double> one(V, 1.0);  // old_probab starts at 1.0, T-FS:228
  std::vector<int> act(V, 1);
  CK(cudaMemcpyAsync(ctx->em_old.p, one.data(), sizeof(double) * V, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaMemcpyAsync(ctx->em_active.p, act.data(), sizeof(int) * V, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaStreamSynchronize(ctx->st));
  return HMMCU_OK;
}

int hmmcu_mstep(hmmcu_ctx *ctx, double threshold, double *sum_logp, double *n_utt, int32_t *updated) {
  if (!ctx || !ctx->have_models || ctx->stats_n != hmmcu_stats_size(ctx->N, ctx->M, ctx->Dm) * ctx->V || !ctx->em_old.p)
    return fail(ctx, HMMCU_EINVAL, "mstep: needs hmmcu_em_reset and an E-step on the current model set");
  CK(cudaSetDevice(ctx->dev));
  const int V = ctx->V;
  int rc = ensure_ctl(ctx);
  if (rc) return rc;
  const int64_t ssz = hmmcu_stats_size(ctx->N, ctx->M, ctx->Dm);
  CK(ctx->upd_d.ensure(sizeof(int) * V));
  {
    const int DP = round_up(ctx->Dm + 1, 4);
    CK(ctx->ext_d.ensure(sizeof(unsigned long long) * (2 * DP + 1)));
  }
  // The warp-specialised tensor-core path will want its packed model forms again right after this M-step: they
  // are rebuilt here, inside the same launch sequence, instead of lazily by the next E-step.
  const bool repack = ctx->train_path == 2 && !ctx->pack_dirty && !ctx->ws_train.dirty && !ctx->acc_dirty && !ctx->kc_dirty &&
                      ctx->have_features && ctx->Dm == ctx->D;
  auto enqueue = [&]() -> int {
    t_begin(ctx, "mstep");
    k_mstep_ctl<<<(V + 127) / 128, 128, 0, ctx->st>>>(ctx->stats.as<double>(), ssz, V, threshold, ctx->em_old.as<double>(),
                                                      ctx->em_active.as<int>(), ctx->ctl_d.as<double>(), ctx->upd_d.as<int>());
    LAUNCH_CHECK();
    CK(launch_pdl(k_mstep_apply, dim3(1 + (ctx->G + 7) / 8, V), 256, 0, ctx->st, ctx->stats.as<double>(), ssz, ctx->N, ctx->M, ctx->Dm,
                  1.0e-5 /* FINITE_PROBAB, T-FS:39 */, ctx->upd_d.as<int>(), ctx->A.as<double>(), ctx->c.as<double>(),
                  ctx->mu.as<double>(), ctx->iv.as<double>(), ctx->det.as<double>()));
    LAUNCH_CHECK();
    int rc2;
    // The accuracy-guard scan and the second W packer do not feed the main chain (new parameters -> kc -> emission
    // images): they run on side streams, joined before the control block is read back.  With the per-kernel timers
    // on everything stays on one stream, so that the timers keep their meaning.
    const bool fork = !ctx->timing && ctx->mstep_fork;
    auto on_stream = [&](cudaStream_t side, auto launch) -> int {
      cudaStream_t keep = ctx->st;
      ctx->st = side;
      const int r = launch();
      ctx->st = keep;
      return r;
    };
    if (fork) {
      CK(cudaEventRecord(ctx->ev_fork[0], ctx->st));
      CK(cudaStreamWaitEvent(ctx->st_aux[0], ctx->ev_fork[0], 0));
      if ((rc2 = on_stream(ctx->st_aux[0], [&] { return launch_kappa(ctx, ctx->ctl_d.as<double>() + 3 * V); })) != HMMCU_OK) return rc2;
      CK(cudaEventRecord(ctx->ev_join[0], ctx->st_aux[0]));
    } else {
      if ((rc2 = launch_kappa(ctx, ctx->ctl_d.as<double>() + 3 * V)) != HMMCU_OK) return rc2;
    }
    t_end(ctx, "mstep");
    if (repack) {
      t_begin(ctx, "pack");
      if ((rc2 = launch_pack_kc(ctx)) != HMMCU_OK) return rc2;
      if (fork) {
        CK(cudaEventRecord(ctx->ev_fork[1], ctx->st));
        CK(cudaStreamWaitEvent(ctx->st_aux[1], ctx->ev_fork[1], 0));
        if ((rc2 = on_stream(ctx->st_aux[1], [&] { return launch_pack_acc(ctx); })) != HMMCU_OK) return rc2;
        CK(cudaEventRecord(ctx->ev_join[1], ctx->st_aux[1]));
      }
      if ((rc2 = launch_pack_ws(ctx, ctx->ws_train)) != HMMCU_OK) return rc2;
      if (fork) CK(cudaStreamWaitEvent(ctx->st, ctx->ev_join[1], 0));
      else if ((rc2 = launch_pack_acc(ctx)) != HMMCU_OK) return rc2;
      t_end(ctx, "pack");
    }
    if (fork) CK(cudaStreamWaitEvent(ctx->st, ctx->ev_join[0], 0));
    CK(cudaMemcpyAsync(ctx->ctl_h, ctx->ctl_d.p, sizeof(double) * (3 * (size_t)V + 1), cudaMemcpyDeviceToHost, ctx->st));
    return HMMCU_OK;
  };
  uint64_t tbits;
  memcpy(&tbits, &threshold, sizeof(tbits));
  if ((rc = run_graphed(ctx, ctx->g_mstep, (tbits * 31u) ^ (repack ? 2u : 0u) ^ (ctx->mstep_fork ? 4u : 0u), enqueue)) != HMMCU_OK) return rc;
  CK(cudaStreamSynchronize(ctx->st));
  for (int v = 0; v < V; v++) {
    if (sum_logp) sum_logp[v] = ctx->ctl_h[v];
    if (n_utt) n_utt[v] = ctx->ctl_h[V + v];
    if (updated) updated[v] = ctx->ctl_h[2 * V + v] != 0.0;
  }
  ctx->kappa = ctx->ctl_h[3 * V];
  ctx->kappa_stale = false;
  if (repack) {  // the forms of the training path are current; every other packed form is stale
    ctx->simt_dirty = true;
    ctx->tc_train.dirty = true;
    ctx->tc_dec.dirty = true;
    ctx->ws_dec.dirty = true;
  } else {
    ctx->pack_dirty = true;
  }
  return HMMCU_OK;
}

int hmmcu_get_models(hmmcu_ctx *ctx, double *A, double *c, double *mu, double *inv_var, double *det) {
  if (!ctx || !ctx->have_models) return fail(ctx, HMMCU_EINVAL, "get_models: no models");
  CK(cudaSetDevice(ctx->dev));
  const int64_t V = ctx->V, N = ctx->N, G = ctx->G, D = ctx->Dm;
  if (A) CK(cudaMemcpyAsync(A, ctx->A.p, sizeof(double) * V * N * N, cudaMemcpyDeviceToHost, ctx->st));
  if (c) CK(cudaMemcpyAsync(c, ctx->c.p, sizeof(double) * V * G, cudaMemcpyDeviceToHost, ctx->st));
  if (mu) CK(cudaMemcpyAsync(mu, ctx->mu.p, sizeof(double) * V * G * D, cudaMemcpyDeviceToHost, ctx->st));
  if (inv_var) CK(cudaMemcpyAsync(inv_var, ctx->iv.p, sizeof(double) * V * G * D, cudaMemcpyDeviceToHost, ctx->st));
  if (det) CK(cudaMemcpyAsync(det, ctx->det.p, sizeof(double) * V * G, cudaMemcpyDeviceToHost, ctx->st));
  CK(cudaStreamSynchronize(ctx->st));
  return HMMCU_OK;
}

double *hmmcu_stats_device(hmmcu_ctx *ctx, int64_t *n_doubles) {
  if (!ctx) return nullptr;
  if (n_doubles) *n_doubles = ctx->stats_n;
  return ctx->stats.as<double>();
}

int hmmcu_stats_download(hmmcu_ctx *ctx, double *stats) {
  if (!ctx || !stats) return HMMCU_EINVAL;
  CK(cudaSetDevice(ctx->dev));
  CK(cudaMemcpyAsync(stats, ctx->stats.p, sizeof(double) * ctx->stats_n, cudaMemcpyDeviceToHost, ctx->st));
  CK(cudaStreamSynchronize(ctx->st));
  return HMMCU_OK;
}


// ------------------------------------------------------- peer all-reduce over NVLink (no library) ----
// Area of a rank: tagged words [2 slot sets][world][n] x 16 B.  Iteration `seq` (1, 2, ..) uses slot set seq & 1.
// Every double travels as two 8-byte words {low half, seq} {high half, seq} written with one 16-byte volatile store ("LL"
// stores, the scheme of the collective libraries' low-latency protocol); an aligned 8-byte word is written atomically, so a
// word whose tag equals this iteration's seq carries this iteration's data, and the receiver simply polls the words it is
// about to add: no fence, no flags, nothing to reset (the area starts zeroed and seq starts at 1).  A thread pushes its
// elements to every peer and then adds the peers' elements in rank order as they land.  Twice the NVLink bytes of plain
// doubles (1 MB per peer at C2), but no block depends on another block, and no fence: faster than the fenced forms with
// flags at 2, 4 and 8 GPUs (DESIGN.md section 6).
constexpr int kPeerBlocks = 128;
__device__ __forceinline__ void st_ll(void *p, uint32_t lo, uint32_t hi, uint32_t tag) {
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(lo), "r"(tag), "r"(hi), "r"(tag) : "memory");
}
__device__ __forceinline__ bool ld_ll(const void *p, uint32_t tag, double &v) {
  uint32_t lo, t0, hi, t1;
  asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo), "=r"(t0), "=r"(hi), "=r"(t1) : "l"(p) : "memory");
  v = __hiloint2double((int)hi, (int)lo);
  return t0 == tag && t1 == tag;
}
__global__ void __launch_bounds__(256)
k_peer_allreduce_ll(double *__restrict__ stats, int64_t n, void *const *__restrict__ areas, int rank, int world,
                    unsigned long long *__restrict__ seq_p, unsigned int *__restrict__ done, int *__restrict__ err) {
  const unsigned long long seq = *seq_p + 1;
  const int set = (int)(seq & 1);
  const uint32_t tag = (uint32_t)seq;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = tid; i < n; i += nth) {
    const double v = stats[i];
    const uint32_t lo = (uint32_t)__double2loint(v), hi = (uint32_t)__double2hiint(v);
    for (int q = 0; q < world; q++) {
      if (q == rank) continue;
      st_ll(reinterpret_cast<char *>(areas[q]) + (((int64_t)set * world + rank) * n + i) * 16, lo, hi, tag);
    }
  }
  const char *mine = reinterpret_cast<const char *>(areas[rank]) + (int64_t)set * world * n * 16;
  long long t0 = 0;
  for (int64_t i = tid; i < n; i += nth) {
    double sacc = 0.0;
    for (int q = 0; q < world; q++) {
      if (q == rank) { sacc += stats[i]; continue; }
      const char *p = mine + ((int64_t)q * n + i) * 16;
      double v;
      unsigned int spins = 0;
      while (!ld_ll(p, tag, v)) {
        if ((++spins & 1023u) == 0) {  // bounded: ~20 s, then *err = 1
          long long t1;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
          if (t0 == 0) t0 = t1;
          if (t1 - t0 > 20000000000ll) { *err = 1; v = 0.0; break; }
        }
      }
      sacc += v;
    }
    stats[i] = sacc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int prev = atomicAdd(&done[world], 1u);
    if (prev == gridDim.x - 1) {  // every block has read the counter by now
      done[world] = 0;
      *seq_p = seq;
    }
  }
}

static int64_t peer_slot_doubles(const hmmcu_ctx *ctx) { return hmmcu_stats_size(ctx->N, ctx->M, ctx->Dm) * ctx->V; }
static size_t peer_area_bytes(int64_t n, int world) { return (size_t)16 * 2 * (size_t)world * (size_t)n; }

static void peer_close(hmmcu_ctx *ctx) {
  for (void *p : ctx->peer_opened) cudaIpcCloseMemHandle(p);
  ctx->peer_opened.clear();
  ctx->peer_ptrs.clear();
  ctx->peer_rank = -1;
  ctx->peer_world = 0;
}

int hmmcu_peer_export(hmmcu_ctx *ctx, int world, void *handle_out) {
  if (!ctx || world < 1 || world > 64) return fail(ctx, HMMCU_EINVAL, "peer_export: bad arguments");
  if (!ctx->have_models) return fail(ctx, HMMCU_EINVAL, "peer_export: set the models first");
  CK(cudaSetDevice(ctx->dev));
  CK(cudaStreamSynchronize(ctx->st));
  peer_close(ctx);
  const int64_t n = peer_slot_doubles(ctx);
  ctx->peer_area.release();  // a fresh allocation: the handle names the allocation, not a sub-range
  CK(ctx->peer_area.ensure(peer_area_bytes(n, world)));
  CK(cudaMemsetAsync(ctx->peer_area.p, 0, peer_area_bytes(n, world), ctx->st));
  CK(ctx->peer_seq_d.ensure(sizeof(unsigned long long) + sizeof(unsigned int) * 80 + sizeof(int)));  // seq | done[80] (done[world]: blocks finished) | err
  CK(cudaMemsetAsync(ctx->peer_seq_d.p, 0, sizeof(unsigned long long) + sizeof(unsigned int) * 80 + sizeof(int), ctx->st));
  CK(cudaStreamSynchronize(ctx->st));
  ctx->peer_n = n;
  ctx->peer_world = world;
  if (handle_out) {
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, ctx->peer_area.p));
    static_assert(sizeof(cudaIpcMemHandle_t) == HMMCU_IPC_HANDLE_BYTES, "IPC handle size");
    memcpy(handle_out, &h, sizeof(h));
  }
  return HMMCU_OK;
}

void *hmmcu_peer_area(hmmcu_ctx *ctx) { return ctx ? ctx->peer_area.p : nullptr; }

int hmmcu_peer_import_pointers(hmmcu_ctx *ctx, int rank, int world, void *const *areas) {
  if (!ctx || !areas || world != ctx->peer_world || rank < 0 || rank >= world || !ctx->peer_area.p)
    return fail(ctx, HMMCU_EINVAL, "peer_import: call hmmcu_peer_export with the same world size first");
  CK(cudaSetDevice(ctx->dev));
  ctx->peer_ptrs.assign(areas, areas + world);
  ctx->peer_ptrs[rank] = ctx->peer_area.p;
  ctx->peer_rank = rank;
  CK(ctx->peer_ptrs_d.ensure(sizeof(void *) * world));
  CK(cudaMemcpyAsync(ctx->peer_ptrs_d.p, ctx->peer_ptrs.data(), sizeof(void *) * world, cudaMemcpyHostToDevice, ctx->st));
  CK(cudaStreamSynchronize(ctx->st));
  return HMMCU_OK;
}

int hmmcu_peer_import(hmmcu_ctx *ctx, int rank, int world, const void *handles) {
  if (!ctx || !handles || world != ctx->peer_world || rank < 0 || rank >= world || !ctx->peer_area.p)
    return fail(ctx, HMMCU_EINVAL, "peer_import: call hmmcu_peer_export with the same world size first");
  CK(cudaSetDevice(ctx->dev));
  std::vector<void *> areas(world, nullptr);
  for (int q = 0; q < world; q++) {
    if (q == rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char *)handles + (size_t)q * HMMCU_IPC_HANDLE_BYTES, sizeof(h));
    void *p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      cudaGetLastError();
      peer_close(ctx);
      return fail(ctx, HMMCU_ECUDA, "peer_import: cudaIpcOpenMemHandle(rank %d): %s", q, cudaGetErrorString(e));
    }
    ctx->peer_opened.push_back(p);
    areas[q] = p;
  }
  return hmmcu_peer_import_pointers(ctx, rank, world, areas.data());
}

static int peer_ready(hmmcu_ctx *ctx, const char *what) {
  if (!ctx) return HMMCU_EINVAL;
  if (ctx->peer_rank < 0 || ctx->peer_world < 1) return fail(ctx, HMMCU_EINVAL, "%s: no peers (hmmcu_peer_export / _import)", what);
  if (ctx->stats_n != ctx->peer_n) return fail(ctx, HMMCU_EINVAL, "%s: the statistics changed size since hmmcu_peer_export (%lld vs %lld doubles)", what,
                                                (long long)ctx->stats_n, (long long)ctx->peer_n);
  return HMMCU_OK;
}

int hmmcu_peer_allreduce(hmmcu_ctx *ctx) {
  int rc = peer_ready(ctx, "peer_allreduce");
  if (rc) return rc;
  CK(cudaSetDevice(ctx->dev));
  if (ctx->peer_world == 1) return HMMCU_OK;
  unsigned long long *seq = ctx->peer_seq_d.as<unsigned long long>();
  unsigned int *done = reinterpret_cast<unsigned int *>(seq + 1);
  int *err = reinterpret_cast<int *>(done + 80);
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(kPeerBlocks, ctx->sm_count), (ctx->peer_n + 255) / 256));
  t_begin(ctx, "allreduce");
  k_peer_allreduce_ll<<<blocks, 256, 0, ctx->st>>>(ctx->stats.as<double>(), ctx->peer_n, ctx->peer_ptrs_d.as<void *>(), ctx->peer_rank,
                                                   ctx->peer_world, seq, done, err);
  LAUNCH_CHECK();
  t_end(ctx, "allreduce");
  return HMMCU_OK;
}

int hmmcu_peer_error(hmmcu_ctx *ctx) {
  if (!ctx || !ctx->peer_seq_d.p) return 0;
  int e = 0;
  if (cudaSetDevice(ctx->dev) != cudaSuccess || cudaStreamSynchronize(ctx->st) != cudaSuccess) return 1;
  const char *p = (const char *)ctx->peer_seq_d.p + sizeof(unsigned long long) + sizeof(unsigned int) * 80;
  if (cudaMemcpy(&e, p, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
  return e != 0;
}

// ----------------------------------------------------------------------------------- Viterbi ----
__global__ void k_add_f64(double *__restrict__ acc, const double *__restrict__ b, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) acc[i] += b[i];
}

// double-precision log-emissions of every utterance against its own model into ctx->logb64 ([F][N])
static int viterbi_logb64(hmmcu_ctx *ctx, const int32_t *utt2model) {
  const int U = ctx->U;
  if (ctx->Dm != ctx->D) return fail(ctx, HMMCU_EINVAL, "models have D=%d but features have D=%d", ctx->Dm, ctx->D);
  const size_t lsm = logb64_smem_bytes(ctx->M, ctx->D);
  if (lsm > 227 * 1024) return fail(ctx, HMMCU_EINVAL, "M=%d mixtures x D=%d does not fit the double-precision emission kernel", ctx->M, ctx->D);
  // tiles and the utterance -> model map only change with the utterance geometry or utt2model: kept between calls
  if (ctx->vit_epoch != ctx->feat_epoch || (int)ctx->vit_u2m.size() != U || memcmp(ctx->vit_u2m.data(), utt2model, sizeof(int32_t) * U) != 0) {
    std::vector<EmisTile> tiles;
    for (int u = 0; u < U; u++) {
      const int64_t f0 = ctx->off[u];
      const int T = (int)(ctx->off[u + 1] - f0);
      for (int t = 0; t < T; t += kLbFrames) tiles.push_back({f0 + t, std::min(kLbFrames, T - t), utt2model[u]});
    }
    CK(ctx->vit_map.ensure(sizeof(int32_t) * U));
    CK(cudaMemcpyAsync(ctx->vit_map.p, utt2model, sizeof(int32_t) * U, cudaMemcpyHostToDevice, ctx->st));
    CK(ctx->vit_tiles.ensure(sizeof(EmisTile) * tiles.size()));
    CK(cudaMemcpyAsync(ctx->vit_tiles.p, tiles.data(), sizeof(EmisTile) * tiles.size(), cudaMemcpyHostToDevice, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    ctx->n_vit_tiles = (int64_t)tiles.size();
    ctx->vit_u2m.assign(utt2model, utt2model + U);
    ctx->vit_epoch = ctx->feat_epoch;
  }
  CK(ctx->logb64.ensure(sizeof(double) * (size_t)ctx->F * ctx->N));
  t_begin(ctx, "logb64");
  if (ctx->D == 39) {  // the MFCC + delta + delta-delta layout every config uses
    CK(cudaFuncSetAttribute(k_logb64<39>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsm));
    k_logb64<39><<<(unsigned)ctx->n_vit_tiles, kLbFrames, lsm, ctx->st>>>(ctx->vit_tiles.as<EmisTile>(), ctx->d_x64, ctx->c.as<double>(),
                                                                     ctx->mu.as<double>(), ctx->iv.as<double>(), ctx->det.as<double>(),
                                                                     ctx->N, ctx->M, ctx->D, ctx->logb64.as<double>());
  } else {
    CK(cudaFuncSetAttribute(k_logb64<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsm));
    k_logb64<0><<<(unsigned)ctx->n_vit_tiles, kLbFrames, lsm, ctx->st>>>(ctx->vit_tiles.as<EmisTile>(), ctx->d_x64, ctx->c.as<double>(),
                                                                    ctx->mu.as<double>(), ctx->iv.as<double>(), ctx->det.as<double>(),
                                                                    ctx->N, ctx->M, ctx->D, ctx->logb64.as<double>());
  }
  LAUNCH_CHECK();
  t_end(ctx, "logb64");
  return HMMCU_OK;
}

int hmmcu_viterbi(hmmcu_ctx *ctx, const int32_t *utt2model, double *score, int32_t *path) {
  if (!ctx) return HMMCU_EINVAL;
  if (ctx->primary) return fail(ctx, HMMCU_EINVAL, "viterbi: this context is a linked stream; call its primary");
  CK(cudaSetDevice(ctx->dev));
  if (!ctx->have_features || !ctx->have_models) return fail(ctx, HMMCU_EINVAL, "features and models must both be set first");
  if (ctx->U == 0) return HMMCU_OK;
  if (!utt2model || !score) return fail(ctx, HMMCU_EINVAL, "viterbi: bad arguments");
  const int U = ctx->U;
  for (int u = 0; u < U; u++)
    if (utt2model[u] < 0 || utt2model[u] >= ctx->V) return fail(ctx, HMMCU_EINVAL, "utt2model[%d]=%d out of range", u, utt2model[u]);
  int rc = check_linked(ctx);
  if (rc) return rc;
  if ((rc = viterbi_logb64(ctx, utt2model)) != HMMCU_OK) return rc;
  for (hmmcu_ctx *q : ctx->linked) {  // multi-stream models: log b = sum over the streams
    if ((rc = viterbi_logb64(q, utt2model)) != HMMCU_OK) return fail(ctx, rc, "linked stream: %s", q->err);
    const int64_t n = ctx->F * ctx->N;
    k_add_f64<<<(int)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8), 256, 0, ctx->st>>>(ctx->logb64.as<double>(), q->logb64.as<double>(), n);
    LAUNCH_CHECK();
  }
  t_single(ctx, "viterbi");
  CK(ctx->psi_ws.ensure(sizeof(unsigned long long) * ctx->F));
  CK(ctx->path_d.ensure(sizeof(int32_t) * ctx->F));
  CK(ctx->logp_utt_d.ensure(sizeof(double) * U));
  t_begin(ctx, "viterbi");
  DISPATCH_N(ctx->N, CK(ScoreLaunch<NS>::path(ctx, ctx->logb64.as<double>(), ctx->vit_map.as<int32_t>(), ctx->logp_utt_d.as<double>(),
                                               path ? ctx->path_d.as<int32_t>() : nullptr)));
  LAUNCH_CHECK();
  t_end(ctx, "viterbi");
  CK(cudaMemcpyAsync(score, ctx->logp_utt_d.p, sizeof(double) * U, cudaMemcpyDeviceToHost, ctx->st));
  if (path) {  // through pinned staging: a copy into pageable memory is staged by the driver in small pieces
    if ((size_t)ctx->F > ctx->path_h_cap) {
      if (ctx->path_h) cudaFreeHost(ctx->path_h);
      ctx->path_h = nullptr;
      ctx->path_h_cap = 0;
      CK(cudaMallocHost((void **)&ctx->path_h, sizeof(int32_t) * (size_t)ctx->F));
      ctx->path_h_cap = (size_t)ctx->F;
    }
    CK(cudaMemcpyAsync(ctx->path_h, ctx->path_d.p, sizeof(int32_t) * ctx->F, cudaMemcpyDeviceToHost, ctx->st));
  }
  CK(cudaStreamSynchronize(ctx->st));
  if (path) memcpy(path, ctx->path_h, sizeof(int32_t) * (size_t)ctx->F);
  return HMMCU_OK;
}

