/* ofb_train.h -- C ABI of the Q-learning update path in libofb.so (sm_100a).
 *
 * Replaces, for the bi-head pointer model, the Keras calls on the far side of the forward
 * (paths under /root/reference/ofighters; SURVEY.md 8(f) rank 1):
 *   Trainer.replay's targets      agents/qlearnIA_V2.py:237-280   -> ofb_trainer_td_targets
 *   model.fit(x, y, epochs=1, batch_size=B)          :281-286    -> ofb_trainer_fit
 *        = one optimiser step on  mse(output1) + mse(output2)  with BatchNormalization in
 *          training mode (batch statistics, moving averages updated) and Adam(lr)   :188,308
 * and, for prioritized replay (ofb_replay.h), the sample-weighted fit (ofb_trainer_fit_weighted) and the TD errors that
 * set the priorities (ofb_trainer_td_errors); for a target network with Double DQN, targets whose pointer and action are
 * chosen by the online predictions and scored by the target network's (ofb_trainer_td_targets_double; the reference has
 * neither, both are opt-in departures).
 *   model weights (save / load_model)                :70,298      -> ofb_trainer_get_weights
 *
 * Conventions are those of ofb.h: int return codes, ofb_last_error(), caller-owned device buffers,
 * asynchronous on `stream`, no CPU fallback.  The handle owns the fp32 master weights, Adam's
 * moments and the activation workspace for max_batch samples (sized at create time; nothing is
 * allocated by fit).
 *
 * Weights travel as ONE flat fp32 array in Keras layer order with Keras layouts -- the order of
 * ofighters_b200.policy.WEIGHT_SPEC: conv1/kernel [3,3,2,8], conv1/bias, norm1/gamma, beta, mean,
 * var, conv2 ... conv4, dense1/kernel [5008,100], bias, dense2, output1, updense1, upconv1/kernel,
 * bias, upnorm1/gamma, beta, mean, var, ... upconv4/kernel [3,3,8,1], bias  (571 730 values).
 *
 * Arithmetic: fp32 throughout (Keras' default dtype), sums over a batch accumulated in fp64.
 * Keras defaults that matter: BatchNormalization momentum 0.99, epsilon 1e-3, batch variance is the
 * biased one; Adam beta1 0.9, beta2 0.999, epsilon 1e-7, update
 *   lr_t = lr * sqrt(1 - beta2^t) / (1 - beta1^t);  p -= lr_t * m / (sqrt(v) + epsilon).
 * Keras / TensorFlow are un-pinned and absent: PARITY UNPINNED, the checker is the torch-autograd
 * restatement oracle/policy_train_torch.py.
 */
#ifndef OFB_TRAIN_H
#define OFB_TRAIN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OFB_TRAIN_N_PARAMS 571730

typedef struct ofb_trainer ofb_trainer;

typedef struct ofb_train_config {
    float lr;              /* Adam(lr=0.0001)                     qlearnIA_V2.py:304,308 */
    float beta1, beta2, adam_eps;
    float bn_momentum, bn_eps;
    int32_t bn_unbiased_moving_var;   /* 0 = Keras (biased), 1 = TF fused kernels (n / (n - 1)) */
    int32_t max_batch;     /* samples per fit the workspace is sized for (reference: batch_size = 8) */
    int32_t reserved[8];
} ofb_train_config;

void ofb_train_default_config(ofb_train_config *cfg);

int ofb_trainer_create(const float *weights_flat_host, int64_t n_params, const ofb_train_config *cfg, int device,
                       ofb_trainer **out);
int ofb_trainer_destroy(ofb_trainer *t);

/* model.fit on one batch (one Adam step).
 *   maps_bits_dev   uint32 [B, 2, 5000]    the samples' images (bit y*400+x; ch0 ship_map, ch1 laser_map)
 *   vec_dev         float  [B, 8]
 *   target_act_dev  float  [B, 2]          y for output1
 *   target_ptr_dev  float  [B, 400, 400]   y for output2
 *   loss_dev        float  [3]             (total, mse(output1), mse(output2)) of the batch BEFORE the update,
 *                                          i.e. history['loss'][0]; may be NULL */
int ofb_trainer_fit(ofb_trainer *t, const uint32_t *maps_bits_dev, const float *vec_dev, const float *target_act_dev,
                    const float *target_ptr_dev, int batch, float *loss_dev, void *stream);

/* model.fit(..., sample_weight=w) (prioritized replay's importance weights): one Adam step on
 *   sum over the two heads of (1/B) sum_b w_b * mse_b,   mse_b = sample b's mean squared error over that head's elements,
 * which is tf.keras' sample_weight under SUM_OVER_BATCH_SIZE; with w = 1 it is ofb_trainer_fit's loss.  loss_dev receives
 * the weighted losses (what history['loss'] reports when sample_weight is given).  BatchNormalization keeps unweighted
 * batch statistics, as Keras does.  sample_weight_dev float [B], every w_b >= 0.  Standalone Keras 2.2 divided instead by
 * the fraction of non-zero weights, so the two forms differ only when some w_b = 0. */
int ofb_trainer_fit_weighted(ofb_trainer *t, const uint32_t *maps_bits_dev, const float *vec_dev, const float *target_act_dev,
                             const float *target_ptr_dev, const float *sample_weight_dev, int batch, float *loss_dev,
                             void *stream);

/* Training-mode forward only (the predictions fit() differentiates): act [B,2], ptr [B,400,400], either may be NULL. */
int ofb_trainer_forward(ofb_trainer *t, const uint32_t *maps_bits_dev, const float *vec_dev, int batch, float *act_dev,
                        float *ptr_dev, void *stream);

/* Trainer.replay's targets (agents/qlearnIA_V2.py:262-280) from predictions on obs and next_obs:
 *   target[b]      = act_obs[b];      target[b][iaction[b]]            = r[b] + gamma * max(act_next[b]) * !done[b]
 *   ptr_target[b]  = ptr_obs[b];      ptr_target[b][px[b]][py[b]]      = r[b] + gamma * max(ptr_next[b]) * !done[b]
 * (the reference indexes the [row, col] map with the (x, y) pointer tuple -- reproduced).  act_* float [B,2], ptr_* float
 * [B,400,400], iaction int32 [B], pointer int32 [B,2] = (x, y), reward float [B], done uint8 [B].  target_act_dev may alias
 * act_obs_dev and target_ptr_dev may alias ptr_obs_dev. */
int ofb_trainer_td_targets(const float *act_obs_dev, const float *ptr_obs_dev, const float *act_next_dev,
                           const float *ptr_next_dev, const int32_t *iaction_dev, const int32_t *pointer_dev,
                           const float *reward_dev, const uint8_t *done_dev, float gamma, int batch,
                           float *target_act_dev, float *target_ptr_dev, void *stream);

/* Signed TD errors (prioritized replay's priorities) at the entries ofb_trainer_td_targets overwrites, same arguments:
 *   td_act[b] = target[b][iaction[b]] - act_obs[b][iaction[b]],   td_ptr[b] = ptr_target[b][px][py] - ptr_obs[b][px][py]
 * with each target computed by ofb_trainer_td_targets' own fp32 expression, so td equals t_target - prediction exactly.
 * Call it before ofb_trainer_td_targets overwrites act_obs / ptr_obs in place.  td_* float [B]. */
int ofb_trainer_td_errors(const float *act_obs_dev, const float *ptr_obs_dev, const float *act_next_dev,
                          const float *ptr_next_dev, const int32_t *iaction_dev, const int32_t *pointer_dev,
                          const float *reward_dev, const uint8_t *done_dev, float gamma, int batch, float *td_act_dev,
                          float *td_ptr_dev, void *stream);

/* ofb_trainer_td_targets / ofb_trainer_td_errors with a discount per sample in place of gamma (n-step returns,
 * ofb_replay_gather_nstep): the overwritten entries become  r[b] + (discount[b] * max) * !done[b],  in the same rounding
 * order, so discount[b] = gamma gives the scalar forms' results bit for bit.  discount_dev float [B]. */
int ofb_trainer_td_targets_discounted(const float *act_obs_dev, const float *ptr_obs_dev, const float *act_next_dev,
                                      const float *ptr_next_dev, const int32_t *iaction_dev, const int32_t *pointer_dev,
                                      const float *reward_dev, const uint8_t *done_dev, const float *discount_dev, int batch,
                                      float *target_act_dev, float *target_ptr_dev, void *stream);
int ofb_trainer_td_errors_discounted(const float *act_obs_dev, const float *ptr_obs_dev, const float *act_next_dev,
                                     const float *ptr_next_dev, const int32_t *iaction_dev, const int32_t *pointer_dev,
                                     const float *reward_dev, const uint8_t *done_dev, const float *discount_dev, int batch,
                                     float *td_act_dev, float *td_ptr_dev, void *stream);

/* Double DQN targets (van Hasselt, Guez & Silver 2016) for a target network: the online network's predictions on next_obs
 * SELECT, the target network's EVALUATE, in one pass over the maps.  Other arguments as ofb_trainer_td_targets_discounted;
 * discount_dev [B] replaces gamma when it is not NULL.
 *   act head:      a* = (act_next_online[b][1] > act_next_online[b][0]) ? 1 : 0        (ties to 0, the decode's rule)
 *                  target[b][iaction[b]]   = r + (g * act_next_target[b][a*]) * keep
 *   pointer head:  p* = the first flat index (row-major [400][400], as stored) at which ptr_next_online[b] attains its
 *                  maximum in fmaxf semantics, so a NaN is never selected; p* = 0 when the map holds no non-NaN value.
 *                  ptr_target[b][px][py]   = r + (g * ptr_next_target[b][p*]) * keep        (the [x][y] entry, as today)
 * with g = discount ? discount[b] : gamma, keep = done[b] ? 0 : 1 and the same fp32 roundings as ofb_trainer_td_targets
 * (no fma).  The rest of target_* is a copy of the obs predictions; target_act_dev may alias act_obs_dev and target_ptr_dev
 * may alias ptr_obs_dev (in place).  td_act_dev / td_ptr_dev (float [B], both or neither NULL) receive target - prediction,
 * the prediction read before an in-place overwrite, so the prioritized path needs this one pass instead of
 * ofb_trainer_td_errors + ofb_trainer_td_targets.  ptr_obs_dev, ptr_next_online_dev and target_ptr_dev must be 16-byte
 * aligned.  With target maps equal to the online maps the results equal ofb_trainer_td_targets[_discounted] and
 * ofb_trainer_td_errors[_discounted] bit for bit, for maps without NaN and without a +0 / -0 tie at the maximum.
 * Deterministic, allocates nothing. */
int ofb_trainer_td_targets_double(const float *act_obs_dev, const float *ptr_obs_dev, const float *act_next_online_dev,
                                  const float *ptr_next_online_dev, const float *act_next_target_dev,
                                  const float *ptr_next_target_dev, const int32_t *iaction_dev, const int32_t *pointer_dev,
                                  const float *reward_dev, const uint8_t *done_dev, float gamma, const float *discount_dev, int batch,
                                  float *target_act_dev, float *target_ptr_dev, float *td_act_dev, float *td_ptr_dev, void *stream);

/* ---- Data-parallel fit (synchronised BatchNormalization over W ranks).
 * Each rank holds a replica of the model and a shard of one global batch.  A sharded fit equals the fit of the concatenated
 * batch: every sum over the batch is accumulated locally into an exchange buffer and summed over the ranks by a caller-supplied
 * reducer before the kernel that consumes it, and the global sample count replaces B in every normalisation.  Adam then runs
 * on every rank on identical reduced gradients, so the replicas stay identical without a weight broadcast.
 *
 * Exchange buffers (caller-owned device memory, so that a framework can hand them straight to its collectives):
 *   stats_dev  double [OFB_TRAIN_STATS_LEN]
 *     [OFB_TRAIN_STATS_FWD + 16 l, +16)   forward BN sums of BN layer l = 0..6 (norm1..norm4, upnorm1..upnorm3):
 *                                         sum y in channels 0..7, sum y^2 in 8..15 (unused channels stay 0)
 *     [OFB_TRAIN_STATS_LOSS, +2)          the two loss accumulators: sum of (weighted) squared errors of output1, output2
 *     [OFB_TRAIN_STATS_BWD + 16 l, +16)   backward BN sums of layer l: sum dz in 0..7, sum dz * xhat in 8..15
 *   grads_dev  float [OFB_TRAIN_N_PARAMS]   the gradients, flat in the weights' order (get_grads reads them)
 * Reduce stages, in the order a sharded fit calls the reducer (16 calls per fit):
 *   OFB_STAGE_FWD_BN + l   for l = 0, 1, ..., 6   (the trunk norm1..norm4, then the pointer head upnorm1..upnorm3)
 *   OFB_STAGE_LOSS
 *   OFB_STAGE_BWD_BN + l   for l = 6, 5, ..., 0   (the backward walks the pointer head first, then the trunk)
 *   OFB_STAGE_GRADS
 * A reducer call must sum its slice over the ranks in `stream` order (the result in place on every rank) before any later
 * work on `stream` runs; every rank must see the same sums, bit for bit, for the replicas to stay identical. */
#define OFB_TRAIN_N_BN 7
#define OFB_TRAIN_STATS_FWD 0
#define OFB_TRAIN_STATS_LOSS 112
#define OFB_TRAIN_STATS_BWD 114
#define OFB_TRAIN_STATS_LEN 226
enum {
    OFB_STAGE_FWD_BN = 0,       /* + layer, 0..6 */
    OFB_STAGE_LOSS = 7,
    OFB_STAGE_BWD_BN = 8,       /* + layer, 8..14 */
    OFB_STAGE_GRADS = 15
};

/* Use stats_dev / grads_dev (layouts above, both non-NULL, on the trainer's device, valid while set) instead of the handle's
 * own sums, loss accumulators and gradients; both NULL restores the handle's own buffers.  Every entry point then reads and
 * writes the caller's buffers; with the handle's own buffers every entry point launches exactly what it launched before. */
int ofb_trainer_set_exchange(ofb_trainer *t, double *stats_dev, float *grads_dev);

/* Reduce hook: fn(ctx, stage, stream) sums stage's slice of the exchange buffers over the ranks and returns 0, or non-zero
 * to abort the fit.  fn == NULL removes it.  Only ofb_trainer_fit_shard calls it; ofb_trainer_fit / _weighted / _forward
 * stay local.  A reducer needs exchange buffers. */
typedef int (*ofb_reduce_fn)(void *ctx, int stage, void *stream);
int ofb_trainer_set_reducer(ofb_trainer *t, ofb_reduce_fn fn, void *ctx);

/* One Adam step on a global batch of batch_global samples, of which this rank holds batch_local (1 <= batch_local <=
 * max_batch, batch_local <= batch_global; batch_global != batch_local needs a reducer).  Arguments as ofb_trainer_fit;
 * sample_weight_dev float [batch_local] may be NULL (unweighted) or the local samples' weights (ofb_trainer_fit_weighted).
 * batch_global replaces B in the BN statistics (mean, variance, the n / (n - 1) of bn_unbiased_moving_var), in the BN
 * backward, in the 2 / n of the losses' gradients and in the reported losses.  Each BN layer's gamma / beta gradients are
 * written from the LOCAL backward sums, before the BWD_BN reduce, so that the GRADS reduce counts each rank's share once.
 * loss_dev receives the global batch's losses on every rank.  With W = 1 and no reducer this is ofb_trainer_fit[_weighted]
 * (same kernels, same arguments).  If the reducer fails the call returns OFB_E_STATE and the trainer's state is undefined:
 * the moving statistics, the gradients or the exchange buffers may already have changed. */
int ofb_trainer_fit_shard(ofb_trainer *t, const uint32_t *maps_bits_dev, const float *vec_dev, const float *target_act_dev,
                          const float *target_ptr_dev, const float *sample_weight_dev, int batch_local, int batch_global,
                          float *loss_dev, void *stream);

/* Flat copies to HOST (synchronise `stream` first): current weights / gradients of the last fit (the exchange gradients
 * when exchange buffers are set: after a sharded fit, the reduced ones). */
int ofb_trainer_get_weights(ofb_trainer *t, float *weights_flat_host, void *stream);
int ofb_trainer_get_grads(ofb_trainer *t, float *grads_flat_host, void *stream);
int64_t ofb_trainer_steps(const ofb_trainer *t);   /* optimiser steps taken (Adam's t) */

#ifdef __cplusplus
}
#endif
#endif /* OFB_TRAIN_H */
