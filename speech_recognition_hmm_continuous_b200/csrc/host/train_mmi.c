/* train_mmi.c -- hmmh_train_mmi: maximum mutual information training, the MMI E-step and the extended Baum-Welch
 * M-step for a fixed number of iterations.  Not hmmh_em_loop: its per-word stopping rule has no counterpart here. */
#include "hmm_cuda.h"
#include "em_loop.h"

int hmmh_train_mmi(hmmcu_ctx *ctx, hmmh_model *models, int V, const int32_t *label, int U, double kappa, int max_hyp,
                   double E, double tau, int iterations, double *objective, hmmh_allreduce_fn allreduce, void *user) {
  if (!ctx || !models || V < 1 || (U > 0 && !label) || iterations < 0) return HMMCU_EINVAL;
  int rc = hmmh_upload_models(ctx, models, V);
  for (int k = 0; k < iterations && rc == HMMCU_OK; k++) {
    if ((rc = hmmcu_estep_mmi(ctx, label, kappa, max_hyp, NULL)) != HMMCU_OK) break;
    if (allreduce) {
      int64_t n = 0;
      double *dev = hmmcu_stats_device(ctx, &n);
      if ((rc = allreduce(user, dev, n, hmmcu_stream(ctx))) != HMMCU_OK) break;
    }
    double F = 0.0, n_utt = 0.0;
    if ((rc = hmmcu_mmi_objective(ctx, &F, &n_utt)) != HMMCU_OK) break;
    if (objective) objective[k] = F / n_utt;
    rc = hmmcu_mstep_ebw(ctx, E, tau);
  }
  if (rc == HMMCU_OK) rc = hmmh_download_models(ctx, models, V);
  return rc;
}
