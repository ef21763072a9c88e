/* ofb_replay.h -- C ABI of the device-resident replay memory in libofb.so (sm_100a).
 *
 * The reference keeps Trainer.memory as a deque of (obs, iaction, ipointer, reward, next_obs, done) with every observation
 * a pair of 400x400 maps (agents/qlearnIA_V2.py:237-238).  At batch scale the maps are far too large to keep: 40 000 B per
 * arena and frame in OFB_MAP_BITS format.  This memory keeps arena STATE SNAPSHOTS instead -- the header, the ship records
 * and the live prefix of the laser list of ofb_common.cuh's arena block, about 1 KB at the default workload -- and
 * rasterises only the transitions that are sampled, with the raster code of the frame kernel, so the gathered maps are
 * bit-identical to those the frame wrote.
 *
 * A transition of tracked arena a and policy ship p is (obs_t, a_t, r_{t+1}, obs_{t+1}, done_{t+1}) from two consecutive
 * snapshots of the arena (QlearnIA.play's rules, agents/qlearnIA_V2.py:372-401):
 *   - it exists only if the ship was alive at t and both snapshots belong to the same episode (the header's episode
 *     counter, which every ofb_reset of the arena increments -- masked resets included);
 *   - reward = the ship's pending reward at t+1 (obs_vec[0] of the next observation), done = the ship is dead at t+1;
 *     so a death yields exactly one transition, with done = 1.
 *
 * Conventions are those of ofb.h.  The handle owns the ring of `depth` frame slots (64-bit addressed: depth x count x
 * ofb_state_stride bytes) and its per-transition fields, all allocated at create time; push, index and gather allocate
 * nothing and never synchronise the host.  A ring of depth D holds the transitions of the last D-1 pushed frames: the
 * newest slot has no successor yet (D - n frames for an n-step memory, ofb_replay_set_n_step).
 *
 * Opt-in prioritized replay (ofb_replay_enable_priorities) adds a sampling mass per transition, a device sampler that
 * draws in proportion to it over the same candidates as ofb_replay_index, and the update of the masses from TD errors.
 *
 * Tensor formats (P = policy ships of the memory, in the order of ship_index_host)
 *   iaction  int32 [N, P]          played action index of every policy ship of the handle's N arenas (PolicyB200.act)
 *   xy       int32 [N, P, 2]       played pointer (x, y)
 *   ids      int32 [M]             transition ids from ofb_replay_index (opaque; valid until the next push)
 *   gather outputs, per sampled transition b: maps_* uint32 [B, 2, W*H/32] (OFB_MAP_BITS), vec_* float [B, 8] (ofb_obs_vec's
 *   head of the ship), iaction int32 [B], pointer int32 [B, 2] = (x, y), reward float [B], done uint8 [B] -- the formats of
 *   ofb_trainer_td_targets and ofb_trainer_fit (ofb_train.h).
 */
#ifndef OFB_REPLAY_H
#define OFB_REPLAY_H

#include <stdint.h>
#include "ofb.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ofb_replay ofb_replay;

/* Track arenas [first, first + count) of handle h and their policy ships ship_index_host[P] (host, distinct, < n_ships), with
 * a ring of depth >= 2 frames.  depth * count * P must stay below 2^31. */
int ofb_replay_create(const ofb_arenas *h, int64_t first, int64_t count, const int32_t *ship_index_host, int32_t n_policy,
                      int32_t depth, ofb_replay **out);
int ofb_replay_destroy(ofb_replay *r);
/* device bytes the handle owns (ring + per-transition fields + index scratch) */
int64_t ofb_replay_device_bytes(const ofb_replay *r);
/* frames pushed since create (host counter) */
int64_t ofb_replay_pushes(const ofb_replay *r);

/* Snapshot the tracked arenas' current state into the next slot, with the PLAYED (iaction, xy) of their policy ships, and
 * complete the previous slot's transitions (valid flag, reward, done).  Call it after the actions of the frame were
 * chosen and before the frame is stepped, so the snapshot is the observation the action was chosen on.  h must be the
 * handle the memory was created on. */
int ofb_replay_push(ofb_replay *r, const ofb_arenas *h, const int32_t *iaction_dev, const int32_t *xy_dev, void *stream);

/* Compact the ids of the valid transitions into ids_dev (capacity (depth - 1) * count * P) in age order: oldest frame first,
 * then arena, then ship.  count_dev (int32 [1]) receives their number. */
int ofb_replay_index(ofb_replay *r, int32_t *ids_dev, int32_t *count_dev, void *stream);

/* Rasterise both snapshots of each of the `batch` transitions ids_dev[0..batch) and write their fields (any output may be
 * NULL to skip it). */
int ofb_replay_gather(const ofb_replay *r, const int32_t *ids_dev, int32_t batch, uint32_t *maps_obs_dev, float *vec_obs_dev,
                      uint32_t *maps_next_dev, float *vec_next_dev, int32_t *iaction_dev, int32_t *pointer_dev,
                      float *reward_dev, uint8_t *done_dev, void *stream);

/* ---- N-step returns (Sutton 1988; Hessel et al. 2018).
 * An n-step memory keeps the same one-step fields per frame t -- valid1[t] (alive at t, same episode at t and t+1),
 * r[t] (the pending reward at t+1), done1[t] (dead at t+1) -- and builds the target R + gamma^k max Q(s_{t+k}) when it gathers.
 * Transition (t, a, p) exists iff valid1[t] and t <= T - n (T = the newest frame), so a ring of depth D holds the transitions of
 * the frames [T - D + 1, T - n].  Its window of k frames walks j = 0, 1, ...:
 *   - done1[t+j]:          k = j + 1, done = 1 (a death: no bootstrap);
 *   - else j + 1 = n:      k = n, done = 0;
 *   - else !valid1[t+j+1]: k = j + 1, done = 0 (the episode ends after frame t+j+1 through a restart, full or masked: a
 *                          time-limit truncation, so the target bootstraps from s_{t+j+1}, the episode's last observation).
 * Gathered: obs = s_t, next = s_{t+k}, the action of frame t, steps = k, the return R and discount = gamma^k, in fp32 without
 * fma: R = r[t+k-1], then R = r[t+j] + gamma * R for j = k-2 .. 0; discount = k - 1 products starting from gamma.  With
 * priorities, frame T - n gets the largest mass at the push of T, the push that makes it a candidate.
 * For n = 1 every rule above is the one-step memory's. */

/* Make the memory's transitions n-step, 1 <= n <= depth - 1 (default 1).  Only before the first push; in either order with
 * ofb_replay_enable_priorities. */
int ofb_replay_set_n_step(ofb_replay *r, int32_t n);

/* ofb_replay_gather for n-step transitions, with the discount gamma: maps / vec / iaction / pointer as there (next = s_{t+k}),
 * return_out float [B] = R, done_out uint8 [B], discount_out float [B] = gamma^k, steps_out int32 [B] = k; any output may be
 * NULL.  The targets are ofb_trainer_td_targets_discounted's.  On a one-step memory it equals ofb_replay_gather with
 * discount = gamma and steps = 1; ofb_replay_gather refuses an n-step memory (its reward, done and next are one-step). */
int ofb_replay_gather_nstep(const ofb_replay *r, const int32_t *ids_dev, int32_t batch, float gamma, uint32_t *maps_obs_dev,
                            float *vec_obs_dev, uint32_t *maps_next_dev, float *vec_next_dev, int32_t *iaction_dev,
                            int32_t *pointer_dev, float *return_dev, uint8_t *done_dev, float *discount_dev, int32_t *steps_dev,
                            void *stream);

/* ---- Prioritized replay (Schaul et al. 2016, proportional variant).
 * Every transition id carries a sampling mass; a transition is drawn with probability mass / (sum of the valid masses).
 * The mass is (|td_act| + |td_ptr| + eps)^alpha, the TD errors of ofb_trainer_td_errors (both heads regress on the same
 * return r + gamma * max).  A transition gets the largest mass set so far (initially 1) when it becomes a candidate, so a new
 * transition is likely drawn at least once. */
typedef struct ofb_replay_prio_config {
    float alpha;          /* >= 0; 0 = uniform */
    float eps;            /* >= 0, added to |td| so that a zero error keeps a chance */
    uint64_t seed;        /* key of the sampler's Philox stream */
    int32_t reserved[8];
} ofb_replay_prio_config;

/* Allocate the masses (fp32 [depth * count * P], indexed by transition id), the device maximum mass and the sampler's tile
 * scratch.  Allowed once, before the first push; nothing allocates afterwards.  ofb_replay_device_bytes counts them. */
int ofb_replay_enable_priorities(ofb_replay *r, const ofb_replay_prio_config *cfg);

/* Draw `batch` transitions in proportion to their masses, stratified: draw b falls in [b, b+1) / batch of the total mass,
 * with U_b from Philox keyed by (seed, samples drawn so far, b) -- a run is reproducible.  No host synchronisation, no
 * allocation.  ids_out int32 [batch] (age order is non-decreasing in b), weight_out float [batch] = the importance weight
 * (mass_b / mass_min)^(-beta) <= 1 with mass_min the smallest non-zero valid mass, which equals Schaul's
 * (N P(i))^(-beta) / max_j w_j over the whole memory.  n_valid_out int32 [1] = number of valid transitions of non-zero mass
 * (all valid ones when eps > 0); when it is 0 the ids and weights are left undefined.  Ids stay valid until the next push.
 * Cost: one pass over the valid flags and masses of all candidates, then one tile of 2048 candidates per draw. */
int ofb_replay_sample_prioritized(ofb_replay *r, int32_t batch, float beta, int32_t *ids_out, float *weight_out,
                                  int32_t *n_valid_out, void *stream);

/* mass[ids[b]] = (|td_act[b]| + |td_ptr[b]| + eps)^alpha and raise the maximum mass.  ids int32 [batch] (ids out of
 * [0, depth * count * P) are skipped), td_* float [batch].  Duplicate ids must carry identical errors (they do when they come
 * from one forward), so the result is deterministic. */
int ofb_replay_update_priorities(ofb_replay *r, const int32_t *ids_dev, const float *td_act_dev, const float *td_ptr_dev,
                                 int32_t batch, void *stream);

/* Copy to device buffers, any of which may be NULL: the masses (float [depth * count * P]), the maximum mass (float [1]) and
 * the fp64 total mass the last ofb_replay_sample_prioritized drew from (double [1]). */
int ofb_replay_read_priorities(const ofb_replay *r, float *mass_dev, float *max_mass_dev, double *last_total_dev, void *stream);

/* ---- Prioritized replay sharded over W ranks (one memory per rank, one global batch).
 * Each rank draws its share of the batch from its own memory in proportion to its masses, so transition i of rank r is drawn
 * with P(i) = m_i / (W M_r) (M_r = the rank's total mass).  Schaul's weights over the union of the memories are then
 *   w_i = (P(i) / min_j P(j))^(-beta) = ((m_i / M_r) / g)^(-beta),   g = min over ranks of m_min,r / M_r,
 * i.e. the local weight (m_i / m_min,r)^(-beta) of ofb_replay_sample_prioritized times the rank's factor
 * ((m_min,r / M_r) / g)^(-beta) <= 1.  Both calls below run on the device without a host synchronisation. */

/* out_dev double [2] = (total mass M_r, smallest non-zero mass m_min,r) of the last ofb_replay_sample_prioritized (undefined
 * when it found no drawable transition). */
int ofb_replay_sample_stats(const ofb_replay *r, double *out_dev, void *stream);

/* weight_dev[b] *= ((local_stats[1] / local_stats[0]) / global_ratio[0])^(-beta) for b < batch, the factor in fp64 and the
 * product rounded once to fp32.  local_stats_dev double [2] from ofb_replay_sample_stats, global_ratio_dev double [1] = g (the
 * minimum over the ranks of local_stats[1] / local_stats[0]).  Leaves the weights unchanged when a total or g is not > 0. */
int ofb_replay_rescale_weights(float *weight_dev, int32_t batch, float beta, const double *local_stats_dev,
                               const double *global_ratio_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* OFB_REPLAY_H */
