/*
 * hmm_host.c -- host side of the drop-in path, plain C: the reference's file formats, the initial
 * model builder, the M-step and the EM control loop.  All device work goes through the C ABI in
 * include/hmm_cuda.h; nothing here computes emissions, alpha/beta or accumulators on the CPU.
 *
 * T-FS = /root/reference/train/source/hmm-fs/hmm_continuous_fs.c
 * R-FS = /root/reference/test/source/recognition-fs/recognition_continuous_fs.c
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "hmm_cuda.h"
#include "em_loop.h"

#define HM_THRESHOLD 1.0e-3 /* T-FS:37 */
#define HM_DELTA 1          /* T-FS:38 */
#define HM_FLOOR 1.0e-5     /* T-FS:39 */

/* ------------------------------------------------------------------ model container -------- */
int hmmh_model_alloc(hmmh_model *m, int N, int M, int D) {
  if (!m || N < 1 || M < 1 || D < 1) return HMMCU_EINVAL;
  size_t g = (size_t)N * M;
  m->N = N; m->M = M; m->D = D;
  m->A = (double *)calloc((size_t)N * N, sizeof(double));
  m->c = (double *)calloc(g, sizeof(double));
  m->mu = (double *)calloc(g * D, sizeof(double));
  m->inv_var = (double *)calloc(g * D, sizeof(double));
  m->det = (double *)calloc(g, sizeof(double));
  if (!m->A || !m->c || !m->mu || !m->inv_var || !m->det) { hmmh_model_free(m); return HMMCU_ENOMEM; }
  return HMMCU_OK;
}

void hmmh_model_free(hmmh_model *m) {
  if (!m) return;
  free(m->A); free(m->c); free(m->mu); free(m->inv_var); free(m->det);
  m->A = m->c = m->mu = m->inv_var = m->det = NULL;
}

/* ------------------------------------------------------------------ feature files ---------- */
/* int32 D then T x D doubles; T is whatever is left in the file (T-FS:527-581). A trailing
 * partial frame is dropped, as the reference's fread loop consumes it without using it fully. */
int hmmh_read_features(const char *path, double **x, int *T, int *D) {
  FILE *f = fopen(path, "rb");
  if (!f) return HMMCU_EIO;
  int d = 0;
  if (fread(&d, sizeof(int), 1, f) != 1 || d < 1 || d > 4096) { fclose(f); return HMMCU_EIO; }
  fseek(f, 0, SEEK_END);
  long bytes = ftell(f) - (long)sizeof(int);
  fseek(f, sizeof(int), SEEK_SET);
  long frames = bytes / ((long)sizeof(double) * d);
  double *buf = (double *)malloc(sizeof(double) * (size_t)(frames > 0 ? frames : 1) * d);
  if (!buf) { fclose(f); return HMMCU_ENOMEM; }
  if (frames > 0 && fread(buf, sizeof(double) * d, (size_t)frames, f) != (size_t)frames) { free(buf); fclose(f); return HMMCU_EIO; }
  fclose(f);
  *x = buf; *T = (int)frames; *D = d;
  return HMMCU_OK;
}

int hmmh_write_features(const char *path, const double *x, int T, int D) {
  FILE *f = fopen(path, "wb");
  if (!f) return HMMCU_EIO;
  int ok = fwrite(&D, sizeof(int), 1, f) == 1 && fwrite(x, sizeof(double) * D, (size_t)T, f) == (size_t)T;
  fclose(f);
  return ok ? HMMCU_OK : HMMCU_EIO;
}

/* ------------------------------------------------------------------ .hmm files -------------- */
/* size_t len | word[len] | int N | int P | int M[P] | int D[P] | A rows | per state: c[M], then per
 * mixture mean[D], det, inv_var[D]   (writer T-FS:2058-2144, reader T-FS:612-712 / R-FS:612-712). */
static int rd(FILE *f, void *p, size_t n) { return fread(p, 1, n, f) == n; }

/* P >= 1 feature streams in one file: N, P, M[P], D[P], A, then stream by stream the states' mixtures.  Stream p comes
 * back as streams[p] (own M and D, the shared A and word copied into each). */
int hmmh_read_model_streams(const char *path, hmmh_model *streams, int max_streams, int *P_out, int len_bytes) {
  if (!path || !streams || max_streams < 1 || !P_out) return HMMCU_EINVAL;
  FILE *f = fopen(path, "rb");
  if (!f) return HMMCU_EIO;
  unsigned char head[8];
  if (!rd(f, head, 8)) { fclose(f); return HMMCU_EIO; }
  unsigned long long len8 = 0; unsigned int len4 = 0;
  memcpy(&len8, head, 8); memcpy(&len4, head, 4);
  if (len_bytes == 0) len_bytes = (len8 < 64) ? 8 : 4; /* a 4-byte header followed by text never reads as a small u64 */
  size_t len = len_bytes == 8 ? (size_t)len8 : (size_t)len4;
  char word[64];
  if (len >= sizeof(word)) { fclose(f); return HMMCU_EIO; }
  fseek(f, len_bytes, SEEK_SET);
  memset(word, 0, sizeof(word));
  int N, P, M[HMMH_MAX_STREAMS], D[HMMH_MAX_STREAMS];
  if (!rd(f, word, len) || !rd(f, &N, 4) || !rd(f, &P, 4)) { fclose(f); return HMMCU_EIO; }
  if (P < 1 || P > HMMH_MAX_STREAMS || P > max_streams || N < 1 || N > HMMH_MAX_FILE_STATES) { fclose(f); return HMMCU_EINVAL; }
  if (!rd(f, M, 4 * (size_t)P) || !rd(f, D, 4 * (size_t)P)) { fclose(f); return HMMCU_EIO; }
  for (int p = 0; p < P; p++)
    if (M[p] < 1 || D[p] < 1 || M[p] > 4096 || D[p] > 4096) { fclose(f); return HMMCU_EIO; }
  int rc = HMMCU_OK, got = 0;
  for (; got < P && rc == HMMCU_OK; got++) {
    rc = hmmh_model_alloc(&streams[got], N, M[got], D[got]);
    if (rc == HMMCU_OK) memcpy(streams[got].word, word, sizeof(word));
  }
  int ok = rc == HMMCU_OK && rd(f, streams[0].A, sizeof(double) * N * N);
  for (int p = 0; ok && p < P; p++) {
    hmmh_model *m = &streams[p];
    if (p > 0) memcpy(m->A, streams[0].A, sizeof(double) * N * N);
    for (int i = 0; ok && i < N; i++) {
      ok = rd(f, m->c + (size_t)i * m->M, sizeof(double) * m->M);
      for (int j = 0; ok && j < m->M; j++) {
        size_t k = (size_t)i * m->M + j;
        ok = rd(f, m->mu + k * m->D, sizeof(double) * m->D) && rd(f, m->det + k, sizeof(double)) &&
             rd(f, m->inv_var + k * m->D, sizeof(double) * m->D);
      }
    }
  }
  fclose(f);
  if (!ok) {
    for (int p = 0; p < got; p++) hmmh_model_free(&streams[p]);
    return rc != HMMCU_OK ? rc : HMMCU_EIO;
  }
  *P_out = P;
  return HMMCU_OK;
}

int hmmh_read_model(const char *path, hmmh_model *m, int len_bytes) {
  int P = 0;
  return hmmh_read_model_streams(path, m, 1, &P, len_bytes); /* a multi-stream file gives HMMCU_EINVAL here */
}

int hmmh_write_model_streams(const char *path, const hmmh_model *streams, int P) {
  if (!path || !streams || P < 1 || P > HMMH_MAX_STREAMS) return HMMCU_EINVAL;
  FILE *f = fopen(path, "wb");
  if (!f) return HMMCU_EIO;
  const hmmh_model *m0 = &streams[0];
  size_t len = strlen(m0->word);
  int ok = fwrite(&len, sizeof(size_t), 1, f) == 1 && fwrite(m0->word, 1, len, f) == len &&
           fwrite(&m0->N, sizeof(int), 1, f) == 1 && fwrite(&P, sizeof(int), 1, f) == 1;
  for (int p = 0; ok && p < P; p++) ok = fwrite(&streams[p].M, sizeof(int), 1, f) == 1;
  for (int p = 0; ok && p < P; p++) ok = fwrite(&streams[p].D, sizeof(int), 1, f) == 1;
  ok = ok && fwrite(m0->A, sizeof(double), (size_t)m0->N * m0->N, f) == (size_t)m0->N * m0->N;
  for (int p = 0; ok && p < P; p++) {
    const hmmh_model *m = &streams[p];
    if (m->N != m0->N) ok = 0;
    for (int i = 0; ok && i < m->N; i++) {
      ok = fwrite(m->c + (size_t)i * m->M, sizeof(double), m->M, f) == (size_t)m->M;
      for (int j = 0; ok && j < m->M; j++) {
        size_t k = (size_t)i * m->M + j;
        ok = fwrite(m->mu + k * m->D, sizeof(double), m->D, f) == (size_t)m->D && fwrite(m->det + k, sizeof(double), 1, f) == 1 &&
             fwrite(m->inv_var + k * m->D, sizeof(double), m->D, f) == (size_t)m->D;
      }
    }
  }
  fclose(f);
  return ok ? HMMCU_OK : HMMCU_EIO;
}

int hmmh_write_model(const char *path, const hmmh_model *m) { return hmmh_write_model_streams(path, m, 1); }

/* ------------------------------------------------------------------ small helpers ----------- */
/* changing_zero_coef T-FS:1338-1359 */
static void floor_and_renormalise(double *w, int n) {
  double s = 0.0;
  for (int k = 0; k < n; k++) {
    if (w[k] < HM_FLOOR) w[k] = HM_FLOOR;
    s += w[k];
  }
  for (int k = 0; k < n; k++) w[k] /= s;
}

/* variance vector -> (det, inverse) in place: calc_det T-FS:1976-1991, inv_matrix T-FS:2012-2022 */
static double det_then_invert(double *v, int D) {
  double det = 1.0;
  for (int d = 0; d < D; d++) det *= v[d];
  for (int d = 0; d < D; d++) v[d] = 1.0 / v[d];
  return det;
}

/* descending order of keys[0..n), adjacent swaps on strict '<' only (T-FS:1289-1317) */
static void order_desc(const double *keys, int *idx, int n) {
  for (int i = 0; i < n; i++) idx[i] = i;
  for (int again = 1; again;) {
    again = 0;
    for (int i = 0; i + 1 < n; i++)
      if (keys[idx[i]] < keys[idx[i + 1]]) {
        int t = idx[i]; idx[i] = idx[i + 1]; idx[i + 1] = t;
        again = 1;
      }
  }
}

/* ------------------------------------------------------------------ M-step ------------------ */
/* stats layout: num_trans[N][N] den_trans[N] den_mix[N] S0[N][M] S1[N][M][D] S2c[N][M][D] sum_logp n_utt
 * updating_transition_probab T-FS:1862-1889, updating_mix_param T-FS:1911-1955, then determinant and
 * inverse of EVERY mixture as main() does (T-FS:339-346) -- also for states with den_mix == 0, whose
 * inv_var is therefore inverted a second time, as in the reference. */
int hmmh_mstep(hmmh_model *m, const double *stats) {
  if (!m || !stats) return HMMCU_EINVAL;
  const int N = m->N, M = m->M, D = m->D;
  const double *num = stats, *den = num + (size_t)N * N, *denmix = den + N, *S0 = denmix + N;
  const double *S1 = S0 + (size_t)N * M, *S2 = S1 + (size_t)N * M * D;
  for (int i = 0; i < N; i++) {
    if (den[i] == 0.0) continue;
    for (int j = 0; j < N; j++) m->A[i * N + j] = num[i * N + j] / den[i];
  }
  for (int i = 0; i < N; i++) {
    if (denmix[i] == 0.0) continue;
    for (int j = 0; j < M; j++) {
      size_t k = (size_t)i * M + j;
      m->c[k] = S0[k] / denmix[i];
      for (int d = 0; d < D; d++) {
        m->mu[k * D + d] = S1[k * D + d] / S0[k];
        double var = S2[k * D + d] / S0[k];
        if (var < HM_FLOOR) var = HM_FLOOR;
        m->inv_var[k * D + d] = var;
      }
    }
  }
  for (int i = 0; i < N; i++) floor_and_renormalise(m->c + (size_t)i * M, M);
  for (size_t k = 0; k < (size_t)N * M; k++) m->det[k] = det_then_invert(m->inv_var + k * D, D);
  return HMMCU_OK;
}

/* ------------------------------------------------------------------ initial model ----------- */
/* creating_initial_model T-FS:732-1317.  Segment k of an utterance of T frames is [seg[k], seg[k+1]):
 * T/N frames each, the first T%N segments one longer (T-FS:1005-1013). */
typedef struct {
  int N, M, D, U;
  const double *x;
  const int64_t *off;
} init_job;

static void segment_bounds(int T, int N, int *seg) {
  int q = T / N, r = T % N;
  seg[0] = 0;
  for (int k = 0; k < N; k++) seg[k + 1] = seg[k] + q + (k < r ? 1 : 0);
}

/* nearest of nmix centroids by squared Euclidean distance; the first minimum wins; *which is left
 * alone when nothing beats 1e20 (classifying, T-FS:1179-1215) */
static double nearest_centroid(const double *x, const double *cent, int nmix, int D, int *which) {
  double best = 1.0e20;
  for (int i = 0; i < nmix; i++) {
    double dist = 0.0;
    for (int d = 0; d < D; d++) {
      double a = cent[(size_t)i * D + d] - x[d];
      dist += a * a;
    }
    if (dist < best) { best = dist; *which = i; }
  }
  return best;
}

int hmmh_init_model(hmmh_model *m, const double *x, const int64_t *frame_off, int U) {
  if (!m || !x || !frame_off || U < 1) return HMMCU_EINVAL;
  const int N = m->N, M = m->M, D = m->D;
  const size_t NM = (size_t)N * M;
  /* transitions: uniform over the allowed band i..i+DELTA (T-FS:774-795) */
  for (int i = 0; i < N; i++)
    for (int j = 0; j < N; j++) {
      double a = 0;
      if (j >= i && j <= i + HM_DELTA) a = (HM_DELTA + 1 > N - i) ? 1.0 / (double)(N - i) : 1.0 / (double)(HM_DELTA + 1);
      m->A[i * N + j] = a;
    }
  double *cent = (double *)calloc(NM * D, sizeof(double));
  double *sum = (double *)calloc(NM * D, sizeof(double));
  double *dist = (double *)calloc(NM, sizeof(double));
  int *cnt = (int *)calloc(NM, sizeof(int));
  int *seg = (int *)malloc(sizeof(int) * (N + 1));
  int *ord = (int *)malloc(sizeof(int) * (M > 0 ? M : 1));
  int *dur = (int *)calloc((size_t)N, sizeof(int));
  if (!cent || !sum || !dist || !cnt || !seg || !ord || !dur) {
    free(cent); free(sum); free(dist); free(cnt); free(seg); free(ord); free(dur);
    return HMMCU_ENOMEM;
  }
  int which = 0;

  /* one centroid per state: the mean of its segment over all utterances (T-FS:996-1030) */
  for (int u = 0; u < U; u++) {
    int T = (int)(frame_off[u + 1] - frame_off[u]);
    const double *xu = x + (size_t)frame_off[u] * D;
    segment_bounds(T, N, seg);
    for (int k = 0; k < N; k++)
      for (int t = seg[k]; t < seg[k + 1]; t++) {
        for (int d = 0; d < D; d++) cent[(size_t)k * M * D + d] += xu[(size_t)t * D + d];
        cnt[(size_t)k * M]++;
      }
  }
  for (int k = 0; k < N; k++)
    for (int d = 0; d < D; d++) cent[(size_t)k * M * D + d] /= (double)cnt[(size_t)k * M];

  int have = 1;
  while (have < M) {
    /* split (T-FS:1120-1158): double while 2*have < M, else split the M-have most distorted cells */
    int next = have;
    for (int k = 0; k < N; k++) {
      double *ck = cent + (size_t)k * M * D;
      if (2 * have < M) {
        for (int j = 0; j < have; j++) {
          for (int d = 0; d < D; d++) ck[(size_t)(have + j) * D + d] = ck[(size_t)j * D + d] * (1.005);
          for (int d = 0; d < D; d++) ck[(size_t)j * D + d] = ck[(size_t)j * D + d] * (0.995);
        }
        next = 2 * have;
      } else {
        order_desc(dist + (size_t)k * M, ord, have);
        for (int j = 0; j < M - have; j++) {
          int src = ord[j];
          for (int d = 0; d < D; d++) ck[(size_t)(have + j) * D + d] = ck[(size_t)src * D + d] * (1.005);
          for (int d = 0; d < D; d++) ck[(size_t)src * D + d] = ck[(size_t)src * D + d] * (0.995);
        }
        next = M;
      }
    }
    have = next;
    /* three k-means passes (T-FS:1043-1090) */
    for (int pass = 0; pass < 3; pass++) {
      for (int k = 0; k < N; k++)
        for (int j = 0; j < have; j++) {
          cnt[(size_t)k * M + j] = 0;
          dist[(size_t)k * M + j] = 0.0;
          for (int d = 0; d < D; d++) sum[((size_t)k * M + j) * D + d] = 0.0;
        }
      for (int u = 0; u < U; u++) {
        int T = (int)(frame_off[u + 1] - frame_off[u]);
        const double *xu = x + (size_t)frame_off[u] * D;
        segment_bounds(T, N, seg);
        for (int k = 0; k < N; k++)
          for (int t = seg[k]; t < seg[k + 1]; t++) {
            /* T-FS:1076 credits the distortion to the cell chosen by THIS call (gcc evaluates the call
             * before the lvalue); pinned against the compiled reference in the tests */
            double dd = nearest_centroid(xu + (size_t)t * D, cent + (size_t)k * M * D, have, D, &which);
            dist[(size_t)k * M + which] += dd;
            cnt[(size_t)k * M + which]++;
            for (int d = 0; d < D; d++) sum[((size_t)k * M + which) * D + d] += xu[(size_t)t * D + d];
          }
      }
      /* new centroids; an empty cell is refilled from the most distorted ones (T-FS:1236-1269) */
      for (int k = 0; k < N; k++) {
        double *ck = cent + (size_t)k * M * D;
        for (int j = 0; j < have; j++)
          for (int d = 0; d < D; d++) ck[(size_t)j * D + d] = sum[((size_t)k * M + j) * D + d] / (double)cnt[(size_t)k * M + j];
        order_desc(dist + (size_t)k * M, ord, have);
        int nxt = 0;
        for (int j = 0; j < have; j++)
          if (cnt[(size_t)k * M + j] == 0) {
            int src = ord[nxt++];
            for (int d = 0; d < D; d++) ck[(size_t)j * D + d] = ck[(size_t)src * D + d] * (1.005);
            for (int d = 0; d < D; d++) ck[(size_t)src * D + d] = ck[(size_t)src * D + d] * (0.995);
          }
      }
    }
  }

  /* variances and weights from one more classification pass (T-FS:864-932) */
  for (size_t k = 0; k < NM; k++) m->c[k] = 0.0;
  for (size_t k = 0; k < NM * D; k++) m->inv_var[k] = 0.0;
  for (int u = 0; u < U; u++) {
    int T = (int)(frame_off[u + 1] - frame_off[u]);
    const double *xu = x + (size_t)frame_off[u] * D;
    segment_bounds(T, N, seg);
    for (int k = 0; k < N; k++) {
      for (int t = seg[k]; t < seg[k + 1]; t++) {
        nearest_centroid(xu + (size_t)t * D, cent + (size_t)k * M * D, M, D, &which);
        size_t g = (size_t)k * M + which;
        for (int d = 0; d < D; d++) {
          double a = xu[(size_t)t * D + d] - cent[g * D + d];
          m->inv_var[g * D + d] += a * a;
        }
        m->c[g]++;
      }
      dur[k] += seg[k + 1] - seg[k];
    }
  }
  for (size_t g = 0; g < NM; g++) {
    for (int d = 0; d < D; d++) {
      m->inv_var[g * D + d] /= m->c[g];
      if (m->inv_var[g * D + d] < HM_FLOOR) m->inv_var[g * D + d] = HM_FLOOR;
    }
    m->det[g] = det_then_invert(m->inv_var + g * D, D);
    for (int d = 0; d < D; d++) m->mu[g * D + d] = cent[g * D + d];
  }
  for (int i = 0; i < N; i++) {
    double s = 0.0;
    for (int j = 0; j < M; j++) {
      m->c[(size_t)i * M + j] /= (double)dur[i];
      s += m->c[(size_t)i * M + j];
    }
    if (s > 1.001 || s < 0.999) printf("error on computing  initial output symbol probabilities: sum = %f \n", s);
  }
  for (int i = 0; i < N; i++) floor_and_renormalise(m->c + (size_t)i * M, M);
  free(cent); free(sum); free(dist); free(cnt); free(seg); free(ord); free(dur);
  return HMMCU_OK;
}

/* ------------------------------------------------------------------ EM control loop --------- */
static int upload_models(hmmcu_ctx *ctx, const hmmh_model *models, int V) {
  const int N = models[0].N, M = models[0].M, D = models[0].D;
  const size_t g = (size_t)N * M;
  double *A = (double *)malloc(sizeof(double) * V * N * N), *c = (double *)malloc(sizeof(double) * V * g);
  double *mu = (double *)malloc(sizeof(double) * V * g * D), *iv = (double *)malloc(sizeof(double) * V * g * D);
  double *det = (double *)malloc(sizeof(double) * V * g);
  if (!A || !c || !mu || !iv || !det) { free(A); free(c); free(mu); free(iv); free(det); return HMMCU_ENOMEM; }
  for (int v = 0; v < V; v++) {
    if (models[v].N != N || models[v].M != M || models[v].D != D) { free(A); free(c); free(mu); free(iv); free(det); return HMMCU_EINVAL; }
    memcpy(A + (size_t)v * N * N, models[v].A, sizeof(double) * N * N);
    memcpy(c + v * g, models[v].c, sizeof(double) * g);
    memcpy(mu + v * g * D, models[v].mu, sizeof(double) * g * D);
    memcpy(iv + v * g * D, models[v].inv_var, sizeof(double) * g * D);
    memcpy(det + v * g, models[v].det, sizeof(double) * g);
  }
  int rc = hmmcu_set_models(ctx, V, N, M, D, A, c, mu, iv, det);
  free(A); free(c); free(mu); free(iv); free(det);
  return rc;
}

int hmmh_upload_models(hmmcu_ctx *ctx, const hmmh_model *models, int V) { return upload_models(ctx, models, V); }

/* T-FS:238-361 for V words at once and P feature streams (models[p * V + v] = stream p of word v; ctxs[p] holds
 * stream p's features; ctxs[1..] are linked to ctxs[0] here).  Every word keeps the reference's own stopping rule; a
 * word that has converged drops out of the following E-steps (its utterances are masked with -1).  estep(ctx, map)
 * leaves the statistics of the current models on the device: Baum-Welch (hmmh_train*) or Viterbi (hmmh_train_viterbi). */
int hmmh_em_loop(hmmcu_ctx *const *ctxs, int P, hmmh_model *models, int V, const int32_t *utt2model, int U, double *mean_logp,
                 int *iterations, int max_iter, hmmh_allreduce_fn allreduce, void *user, hmmh_estep_fn estep) {
  if (!ctxs || P < 1 || P > HMMH_MAX_STREAMS || !models || V < 1 || (U > 0 && !utt2model)) return HMMCU_EINVAL;
  hmmcu_ctx *ctx = ctxs[0];
  double *probab = (double *)malloc(sizeof(double) * V), *nutt = (double *)malloc(sizeof(double) * V);
  double *probab_q = (double *)malloc(sizeof(double) * V), *nutt_q = (double *)malloc(sizeof(double) * V);
  int32_t *updated = (int32_t *)malloc(sizeof(int32_t) * V), *updated_q = (int32_t *)malloc(sizeof(int32_t) * V);
  char *active = (char *)malloc(V);
  int32_t *map = (int32_t *)malloc(sizeof(int32_t) * (U > 0 ? U : 1));
  if (!probab || !nutt || !probab_q || !nutt_q || !updated || !updated_q || !active || !map) {
    free(probab); free(nutt); free(probab_q); free(nutt_q); free(updated); free(updated_q); free(active); free(map);
    return HMMCU_ENOMEM;
  }
  for (int v = 0; v < V; v++) { active[v] = 1; if (iterations) iterations[v] = 0; if (mean_logp) mean_logp[v] = 0.0; }
  /* the model sets go up once; the E-step, the all-reduce and the M-step then stay on the device */
  int rc = HMMCU_OK;
  for (int p = 0; p < P && rc == HMMCU_OK; p++) {
    rc = upload_models(ctxs[p], models + (size_t)p * V, V);
    if (rc == HMMCU_OK) rc = hmmcu_em_reset(ctxs[p]);
  }
  if (rc == HMMCU_OK && P > 1) rc = hmmcu_link_streams(ctx, ctxs + 1, P - 1);
  int n_active = V, it = 0, remap = 1;
  while (rc == HMMCU_OK && n_active > 0 && (max_iter <= 0 || it < max_iter)) {
    it++;
    if (remap) {
      for (int u = 0; u < U; u++) map[u] = active[utt2model[u]] ? utt2model[u] : -1;
      remap = 0;
    }
    if ((rc = estep(ctx, map)) != HMMCU_OK) break;
    for (int p = 0; allreduce && p < P && rc == HMMCU_OK; p++) {
      int64_t n = 0;
      double *dev = hmmcu_stats_device(ctxs[p], &n);
      rc = allreduce(user, dev, n, hmmcu_stream(ctxs[p]));
    }
    if (rc != HMMCU_OK) break;
    if ((rc = hmmcu_mstep(ctx, HM_THRESHOLD, probab, nutt, updated)) != HMMCU_OK) break;
    for (int p = 1; p < P && rc == HMMCU_OK; p++) rc = hmmcu_mstep(ctxs[p], HM_THRESHOLD, probab_q, nutt_q, updated_q);
    if (rc != HMMCU_OK) break;
    for (int v = 0; v < V; v++) {
      if (!active[v]) continue;
      if (iterations) iterations[v] = it;
      if (mean_logp) mean_logp[v] = probab[v] / nutt[v];
      if (!updated[v]) { active[v] = 0; n_active--; remap = 1; }
    }
  }
  for (int p = 0; p < P && rc == HMMCU_OK; p++) {  /* bring the trained parameters back into the caller's structs */
    hmmh_model *mp = models + (size_t)p * V;
    const int N = mp[0].N, M = mp[0].M, D = mp[0].D;
    const size_t g = (size_t)N * M;
    double *A = (double *)malloc(sizeof(double) * V * N * N), *c = (double *)malloc(sizeof(double) * V * g);
    double *mu = (double *)malloc(sizeof(double) * V * g * D), *iv = (double *)malloc(sizeof(double) * V * g * D);
    double *det = (double *)malloc(sizeof(double) * V * g);
    if (!A || !c || !mu || !iv || !det) rc = HMMCU_ENOMEM;
    else if ((rc = hmmcu_get_models(ctxs[p], A, c, mu, iv, det)) == HMMCU_OK) {
      for (int v = 0; v < V; v++) {
        memcpy(mp[v].A, A + (size_t)v * N * N, sizeof(double) * N * N);
        memcpy(mp[v].c, c + v * g, sizeof(double) * g);
        memcpy(mp[v].mu, mu + v * g * D, sizeof(double) * g * D);
        memcpy(mp[v].inv_var, iv + v * g * D, sizeof(double) * g * D);
        memcpy(mp[v].det, det + v * g, sizeof(double) * g);
      }
    }
    free(A); free(c); free(mu); free(iv); free(det);
  }
  if (P > 1) hmmcu_link_streams(ctx, NULL, 0);
  free(probab); free(nutt); free(probab_q); free(nutt_q); free(updated); free(updated_q); free(active); free(map);
  return rc;
}

static int estep_baum_welch(hmmcu_ctx *ctx, const int32_t *map) { return hmmcu_estep(ctx, map, NULL, NULL); }

int hmmh_train_streams(hmmcu_ctx *const *ctxs, int P, hmmh_model *models, int V, const int32_t *utt2model, int U, double *mean_logp,
                       int *iterations, int max_iter, hmmh_allreduce_fn allreduce, void *user) {
  return hmmh_em_loop(ctxs, P, models, V, utt2model, U, mean_logp, iterations, max_iter, allreduce, user, estep_baum_welch);
}

int hmmh_train(hmmcu_ctx *ctx, hmmh_model *models, int V, const int32_t *utt2model, int U, double *mean_logp,
               int *iterations, int max_iter, hmmh_allreduce_fn allreduce, void *user) {
  if (!ctx) return HMMCU_EINVAL;
  return hmmh_train_streams(&ctx, 1, models, V, utt2model, U, mean_logp, iterations, max_iter, allreduce, user);
}
