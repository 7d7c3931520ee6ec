/* em_loop.h -- the EM control loop shared by hmmh_train, hmmh_train_streams and hmmh_train_viterbi (library-internal,
 * not exported from libhmmcu.so). */
#ifndef HMM_EM_LOOP_H
#define HMM_EM_LOOP_H

#include "hmm_cuda.h"

/* One E-step of the current models over the utterance map (-1 = masked), statistics left on the device. */
typedef int (*hmmh_estep_fn)(hmmcu_ctx *ctx, const int32_t *map);

__attribute__((visibility("hidden")))
int hmmh_em_loop(hmmcu_ctx *const *ctxs, int P, hmmh_model *models, int V, const int32_t *utt2model, int U, double *mean_logp,
                 int *iterations, int max_iter, hmmh_allreduce_fn allreduce, void *user, hmmh_estep_fn estep);

#endif
