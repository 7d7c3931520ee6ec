/* train_viterbi.c -- hmmh_train_viterbi: the EM loop of hmm_host.c with the Viterbi alignment as its E-step.  Kept out
 * of hmm_host.c, which is also linked on its own against stand-ins for the device entry points it calls. */
#include "hmm_cuda.h"
#include "em_loop.h"

static int estep_viterbi(hmmcu_ctx *ctx, const int32_t *map) { return hmmcu_estep_viterbi(ctx, map, NULL, NULL, NULL); }

int hmmh_train_viterbi(hmmcu_ctx *ctx, hmmh_model *models, int V, const int32_t *utt2model, int U, double *mean_logp,
                       int *iterations, int max_iter, hmmh_allreduce_fn allreduce, void *user) {
  if (!ctx) return HMMCU_EINVAL;
  return hmmh_em_loop(&ctx, 1, models, V, utt2model, U, mean_logp, iterations, max_iter, allreduce, user, estep_viterbi);
}
