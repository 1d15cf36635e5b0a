/*
 * uavsim.h -- C ABI of libuavsim.so, the B200 (sm_100a) batched UAV/target tracking simulator.
 *
 * The reference (tjuDavidWang/MARL-UAVs-Targets-Tracking) is pure Python and has no FFI layer; its
 * boundary for this path is the `Environment` object (src/environment.py:12-164).  Each entry point
 * below names the reference interface it stands in for.  A reference-side binding (ctypes) is shown
 * in INTEGRATION.md; the shipped one is marl_uavs_targets_tracking_b200/_cabi.py.
 *
 * Conventions
 *   - plain C types only; all array arguments are raw pointers + the sizes fixed at create time.
 *   - "device pointer" = memory of the CUDA device given to uavsim_create (PyTorch owns it in the
 *     shipped host code; the library owns only the handle and a few KB of scratch).
 *   - arrays are environment-major structure-of-arrays: [E,n] / [E,m] / [E,n,12] / [4,E,n].
 *   - every call returns 0 on success, a positive cudaError_t, or a negative UAVSIM_ERR_* code;
 *     uavsim_last_error() gives a message.  There is no CPU fallback: without a CUDA device every
 *     compute call fails.
 *   - a handle is not thread-safe; use one handle per GPU / rank.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 */
#ifndef UAVSIM_H
#define UAVSIM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UAVSIM_ABI_VERSION 1
#define UAVSIM_OBS_DIM 12   /* src/environment.py:29 state_dim = (4+1)+4+(2+1) */
#define UAVSIM_MAX_UAV 128  /* neighbour sets are kept as 2 x 64-bit words per UAV */

enum {
  UAVSIM_ERR_ARG = -1,         /* bad argument / NULL pointer */
  UAVSIM_ERR_UNBOUND = -2,     /* uavsim_bind not called or a needed buffer is NULL */
  UAVSIM_ERR_UNSUPPORTED = -3, /* size outside what the kernels support */
  UAVSIM_ERR_NO_PMI = -4       /* mode PMI without uavsim_set_pmi_weights */
};

/* reward modes: which branch of UAV.calculate_cooperative_reward (src/agent/uav.py:312-322) runs */
enum {
  UAVSIM_MODE_SELF = 0, /* MAAC:   cooperative = 0 -> raw reward (src/main.py:75-76)                    */
  UAVSIM_MODE_MEAN = 1, /* MAAC-G: pmi is None -> neighbour mean (src/agent/uav.py:293-310)             */
  UAVSIM_MODE_PMI = 2   /* MAAC-R: PMI-softmax weighted neighbour rewards (src/agent/uav.py:262-291)    */
};

/* Scenario constants = the config keys Environment.reset/step read (src/environment.py:97-107,
 * :207-224), already converted as the reference does (h_max fields are pi / yaml value). */
typedef struct UavSimParams {
  int32_t n_uav;      /* config['environment']['n_uav']      */
  int32_t m_targets;  /* config['environment']['m_targets']  */
  int32_t na;         /* config['environment']['na']         */
  int32_t num_steps;  /* episode length for the `done` flag (src/main.py:128 --num_steps), 0 = never */
  double x_max, y_max;
  double dt, uav_v_max, uav_h_max, dc, dp;
  double tgt_v_max, tgt_h_max;
  double alpha, beta, gamma;
} UavSimParams;

/* Device buffers the kernels read and write.  Required unless marked optional (may be NULL). */
typedef struct UavSimBuffers {
  /* state, updated in place by uavsim_step: UAV.x/.y/.h/.a (src/agent/uav.py:25-35), TARGET.x/.y/.h */
  double *ux, *uy, *uh;  /* [E,n] */
  int32_t *ua;           /* [E,n] last action index */
  double *tx, *ty, *th;  /* [E,m] */
  /* step input: the `actions` argument of Environment.step (src/environment.py:120) */
  int32_t *actions;      /* [E,n] in {0..na-1} */
  /* step outputs = the triple Environment.step returns (src/environment.py:157-164) */
  float *obs;            /* [E,n,12] next_states (UAV.get_local_state, src/agent/uav.py:156-197) */
  float *rew4;           /* [4,E,n]: 'rewards', 'target_tracking_reward', 'boundary_punishment',
                                     'duplicate_tracking_punishment' */
  int32_t *covered;      /* [E] covered_targets (src/environment.py:246-253) */
  int32_t *tracker_cnt;  /* optional [E,m]: UAVs strictly within dp of each target */
  int32_t *done;         /* optional [E]: 1 when the step counter reaches num_steps */
  /* scratch for UAVSIM_MODE_PMI (optional otherwise) */
  double *raw;           /* [E,n] weighted raw reward (UAV.raw_reward, src/environment.py:219) */
  uint64_t *nbr_bits;    /* [E,n,2] neighbour set d<=dp as bit masks */
  /* optional integer masks for parity tests (uint8 0/1); all five or none */
  uint8_t *obs_mask;     /* [E,n,m] d(u,t) <= dp at observe time (src/agent/uav.py:111) */
  uint8_t *comm_mask;    /* [E,n,n] d(u,v) <= dc, v moved iff v<u (src/agent/uav.py:135) */
  uint8_t *nbr_mask;     /* [E,n,n] d(u,v) <= dp, all moved (src/agent/uav.py:305) */
  uint8_t *dup_mask;     /* [E,n,n] d(u,v) <= 2dp (src/agent/uav.py:225) */
  uint8_t *cover_mask;   /* [E,n,m] d(u,t) <  dp (src/environment.py:250) */
} UavSimBuffers;

/* PMINetwork in eval mode with BatchNorm folded into the Linear layers (src/models/PMINet.py:41-62).
 * Host pointers; the library copies them to the device. */
typedef struct UavSimPmiWeights {
  int32_t hidden;    /* H: 32, 64, 128 or 256 */
  int32_t _pad;
  const float *w0;   /* [3H,5]: rows 0..H-1 fc_comm (5 inputs), H..2H-1 fc_obs (4, padded), 2H..3H-1
                        fc_boundary_state (3, padded); padding entries must be 0 */
  const float *b0;   /* [3H] */
  const float *w1;   /* [H,3H] fc1 */
  const float *b1;   /* [H] */
  const float *w2;   /* [H] fc2 */
  float b2;
  float _pad2;
} UavSimPmiWeights;

typedef struct uavsim uavsim_t;

int uavsim_abi_version(void);
const char *uavsim_last_error(void);

/* Environment.__init__ (src/environment.py:13-43).  env_id_offset = global id of this handle's first
 * environment (rank sharding: rank r of R passes r*E/R) -- it only keys the counter-based RNG, so
 * results do not depend on how environments are split over GPUs. */
int uavsim_create(const UavSimParams *params, int64_t n_envs, int64_t env_id_offset, int device, uavsim_t **out);
int uavsim_destroy(uavsim_t *h);
int uavsim_bind(uavsim_t *h, const UavSimBuffers *buffers);

/* Environment.reset (src/environment.py:45-107): UAVs on the line x_i = i*x_max/(n+1), y = y_max/2,
 * heading U(-pi,pi), last action U{0..na-1}; targets U(0,x_max) x U(0,y_max), heading U(-pi,pi).
 * Draws come from Philox4x32-10 keyed (seed; entity, stream, global env id).  Also writes the
 * pre-step observation and clears the step counter and episode statistics. */
int uavsim_reset(uavsim_t *h, uint64_t seed, void *stream);

/* Replay path: after the caller has written a recorded reset into the bound state buffers, build the
 * pre-step observation (empty lists -> -1 blocks, src/agent/uav.py:170-186) and clear counters. */
int uavsim_begin_episode(uavsim_t *h, void *stream);

/* Random policy: actions[e,i] ~ U{0..na-1} from Philox keyed (seed; i, global env id, step). */
int uavsim_random_actions(uavsim_t *h, uint64_t seed, int64_t step, void *stream);

/* Environment.step (src/environment.py:120-164) for all E environments, device buffers. */
int uavsim_step(uavsim_t *h, int mode, double cooperative, void *stream);

/* nsteps x (uavsim_random_actions(seed, first_step + k); uavsim_step) queued on `stream` without returning to the
 * caller in between: the random-policy rollout of BASELINE configs[1].  Outputs hold the last step's values. */
int uavsim_run_random_policy(uavsim_t *h, int mode, double cooperative, uint64_t seed, int64_t first_step,
                             int64_t nsteps, void *stream);

/* Same, host buffers (pinned for real overlap): copies h_actions [E,n] in, steps, copies obs [E,n,12],
 * rew4 [4,E,n], covered [E] out, pipelined over `chunks` env ranges.  Blocks until the outputs are in
 * host memory.  Any output pointer may be NULL (skipped). */
int uavsim_step_host(uavsim_t *h, int mode, double cooperative, const int32_t *h_actions, float *h_obs,
                     float *h_rew4, int32_t *h_covered, int chunks, void *stream);

/* The same step queued without waiting: returns once the copies and kernels are enqueued and hands back a ticket;
 * uavsim_step_host_wait(ticket) blocks until that step's outputs are in its host buffers.  A caller that already
 * holds the next actions (a random or scripted policy, an action sequence under evaluation) may queue step t+1 --
 * with OTHER host output buffers -- before waiting for step t: the download of step t then overlaps the upload and
 * the kernels of step t+1 (chunk by chunk; the library orders the device-side reuse of the action and output
 * arrays itself).  At most two steps should be in flight; every other entry point of the handle must only be
 * called after the last ticket has been waited for.  (src/train.py:142-196 is closed-loop -- the next action
 * depends on this observation -- and uses uavsim_step_host.) */
int uavsim_step_host_async(uavsim_t *h, int mode, double cooperative, const int32_t *h_actions, float *h_obs,
                           float *h_rew4, int32_t *h_covered, int chunks, void *stream, int64_t *ticket);
int uavsim_step_host_wait(uavsim_t *h, int64_t ticket);

/* alpha/beta/gamma are re-read from config on every Environment.step (src/environment.py:219-220);
 * this updates them without recreating the handle. */
int uavsim_set_reward_weights(uavsim_t *h, double alpha, double beta, double gamma);

/* pmi argument of Environment.step / PMINetwork.inference (src/models/PMINet.py:64-72). */
int uavsim_set_pmi_weights(uavsim_t *h, const UavSimPmiWeights *w, void *stream);

/* Which kernel runs Environment.step: 0 = automatic (n_uav, m_targets <= 16 and a batch of at most ~2.5 waves: the
 * two-warp kernel of csrc/step_small_kernel.cuh; 64 x 64 swarms with 16-byte aligned buffers: the per-UAV fast kernel of
 * csrc/step_fast_kernel.cuh; the generic kernel otherwise), 1 = always the generic kernel, 2 = the per-UAV fast kernel,
 * 3 = the all-pairs tile kernel of csrc/step_tile_kernel.cuh, 4 = the small-swarm kernel (2-4: an error if the kernel
 * cannot serve the shape / the bound buffers).  All kernels decide every integer output identically; the switch exists
 * for tests and A/B timing. */
int uavsim_set_step_path(uavsim_t *h, int path);

/* Which kernel evaluates the PMI MLP: 0 = automatic (tensor cores when hidden is 64 or 128, the neighbour lists fit and
 * the fc1 weights fit fp16 after the per-unit rebalancing of uavsim_set_pmi_weights), 1 = fp32 CUDA cores, 2 = tcgen05
 * tensor cores with split fp16 hi + lo operands (error if unsupported, also when weights uploaded later do not fit). */
int uavsim_set_pmi_path(uavsim_t *h, int path);

/* Episode statistics accumulated by uavsim_step since the last reset (src/train.py:181-192):
 * out[0..3] = sums of rewards / tracking / boundary / duplicate over env-steps and UAVs,
 * out[4] = sum of covered_targets over env-steps, out[5] = max covered_targets,
 * out[6] = env-steps accumulated, out[7] = pair rows the tensor-core PMI kernel evaluated with inputs beyond the range its
 * fp16 activations hold for the uploaded weights (their logits saturate; 0 in any run the tensor path serves exactly,
 * DESIGN.md section 3.2; the CUDA-core kernel has no such limit and never counts).  Synchronises `stream`.  Every kernel
 * accumulates the reward sums as integer counts of 2^-22 of the float32 values it writes to rew4, one per (environment,
 * UAV, step) -- exact in any order, so the totals are bit-reproducible although CTAs draw their environments from a
 * counter, and do not depend on which kernel served a step; resolution 2.4e-7 per value. */
int uavsim_episode_stats(uavsim_t *h, double out[8], void *stream);

/* number of kernels this handle has launched (bench.py reports it as gpu_launches) */
int64_t uavsim_launch_count(const uavsim_t *h);
int64_t uavsim_step_count(const uavsim_t *h);

/* ------------------------------------------------------------------------------------------------
 * Prioritized replay on the device -- PrioritizedReplayBuffer (src/train.py:73-139).
 * The ring (states [C,D] f32, actions [C] i32, rewards [C] f32, next_states [C,D] f32, priorities [C] f32)
 * lives in device memory owned by the handle; inputs and outputs are caller-owned DEVICE pointers.
 * ------------------------------------------------------------------------------------------------ */
typedef struct uavsim_replay uavsim_replay_t;

/* PrioritizedReplayBuffer.__init__(capacity, alpha) (src/train.py:74-79) */
int uavsim_replay_create(int64_t capacity, int state_dim, double alpha, int device, uavsim_replay_t **out);
int uavsim_replay_destroy(uavsim_replay_t *h);

/* add(transition_dict) (src/train.py:81-98): `count` transitions, each stored with the current maximum
 * priority (1.0 while the buffer is empty); a batch longer than the capacity keeps its last `capacity` rows. */
int uavsim_replay_add(uavsim_replay_t *h, const float *states, const int32_t *actions, const float *rewards,
                      const float *next_states, int64_t count, void *stream);

/* sample(batch_size, beta) (src/train.py:100-132): *n_out = min(batch, size) draws with replacement,
 * P(i) = priority_i^alpha / sum, by inverse CDF like numpy.random.choice(p=...); weights (size*P(i))^-beta / max.
 * `uniforms` = n_out doubles in [0,1) on the device, or NULL to draw them from Philox4x32-10 keyed
 * (seed; sample index, counter). */
int uavsim_replay_sample(uavsim_replay_t *h, int64_t batch, double beta, const double *uniforms, uint64_t seed,
                         uint64_t counter, float *o_states, int32_t *o_actions, float *o_rewards, float *o_next_states,
                         int64_t *o_indices, float *o_weights, int64_t *n_out, void *stream);

/* update_priorities(indices, priorities) (src/train.py:134-136): sequential assignment, the last write to a
 * repeated index wins.  Precondition, not checked here (that would synchronise the stream): every priority is finite
 * and non-negative (-0.0 counts as zero).  A NaN, infinite or negative priority makes later samples undefined. */
int uavsim_replay_update_priorities(uavsim_replay_t *h, const int64_t *indices, const float *priorities,
                                    int64_t count, void *stream);

/* size() (src/train.py:138-139), ring write position, kernels launched so far */
int64_t uavsim_replay_size(const uavsim_replay_t *h);
int64_t uavsim_replay_pos(const uavsim_replay_t *h);
int64_t uavsim_replay_launch_count(const uavsim_replay_t *h);

/* Checkpoint / inspection: copy slots [0, size) of the ring, all `capacity` priorities and the probabilities of
 * the last sample call into HOST buffers (any may be NULL).  Synchronises `stream`. */
int uavsim_replay_export(uavsim_replay_t *h, float *states, int32_t *actions, float *rewards, float *next_states,
                         float *priorities, float *probabilities, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Fused policy step of the batched rollout: probs = softmax(fc2(relu(fc1(obs)))) (FnnPolicyNet,
 * src/models/actor_critic.py:85-99) and one categorical draw per row (ActorCritic.take_action,
 * src/models/actor_critic.py:138-148) in one launch.  All pointers are DEVICE pointers, weights in torch layout.
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t state_dim; /* 12 */
  int32_t hidden;    /* <= 512 */
  int32_t n_actions; /* 2 .. 16 */
  int32_t _pad;
  const float *w1;   /* fc1.weight [hidden, state_dim] */
  const float *b1;   /* fc1.bias   [hidden] */
  const float *w2;   /* fc2.weight [n_actions, hidden] */
  const float *b2;   /* fc2.bias   [n_actions] */
} UavSimPolicyWeights;

/* actions[r] ~ Categorical(probs[r, :]) with the uniform Philox4x32-10 (seed; r, counter); probs [rows, n_actions] may be
 * NULL.  obs [rows, 12] float32 (e.g. the environment's observation buffer), 16-byte aligned: the kernel reads rows with
 * 16-byte loads, and a misaligned obs is refused with UAVSIM_ERR_ARG. */
int uavsim_policy_sample(const float *obs, int64_t rows, const UavSimPolicyWeights *w, uint64_t seed, uint64_t counter,
                         int32_t *actions, float *probs, int device, void *stream);

/* Greedy twin of uavsim_policy_sample, the deterministic action rule of evaluation: actions[r] = the smallest index among
 * the maximal probabilities of row r as the kernel computes them, i.e. torch.argmax of the probs output (NULL allowed).
 * Same argument checks; no random draw. */
int uavsim_policy_greedy(const float *obs, int64_t rows, const UavSimPolicyWeights *w, int32_t *actions, float *probs,
                         int device, void *stream);

/* Device trajectory buffers of uavsim_run_policy (T = nsteps); any field may be NULL: that output then goes to the
 * bound buffer, overwritten step by step.  obs must be 16-byte aligned, like the bound observation buffer. */
typedef struct UavSimTrajectory {
  float *obs;        /* [T+1,E,n,12]: slot 0 <- the bound observation before the first step, slot k+1 <- step k */
  int32_t *actions;  /* [T,E,n]     : the actions drawn for step k */
  float *rew4;       /* [T,4,E,n]   : the four reward planes of step k */
  int32_t *covered;  /* [T,E]       : covered targets after step k */
} UavSimTrajectory;

/* Learned-policy rollout of a whole episode without returning to the caller between steps (src/train.py:160-176 for
 * all environments at once): for k = 0 .. nsteps-1
 *     uavsim_policy_sample(obs_k, E*n, w, seed, first_counter + k, actions_k, NULL, device, stream);
 *     uavsim_step(h, mode, cooperative, stream);
 * where obs_k / actions_k (and the step's obs / rew4 / covered outputs) are the trajectory slots of step k, or the bound
 * buffers where a field of `traj` is NULL (traj may be NULL: everything in place).  The result is bit-identical to that
 * loop in every output -- observations, actions, reward planes, covered counts, done, the state, the step counter and
 * uavsim_episode_stats -- because the same kernels run on the same data: the step kernel is chosen as uavsim_step chooses
 * it.  The policy launches and the small-swarm step kernel use programmatic dependent launch, so each grid is scheduled
 * while its predecessor drains (the policy kernel stages its weights meanwhile).  After the last step the last slot of
 * every given field is copied into the bound buffer, so the bound obs / actions / rew4 / covered hold what stepping one
 * step at a time leaves there, and the next uavsim_step continues the episode.  The bound pointers are restored on
 * every exit.  Every argument is checked before anything is queued: on an error nothing is enqueued and the step
 * counter does not move (n_actions must equal the handle's na; with uavsim_set_step_path 2 or 3 every trajectory slot
 * must be 16-byte aligned, i.e. E*n % 4 == 0 when actions are recorded, else UAVSIM_ERR_UNSUPPORTED).  The policy
 * launches count in uavsim_launch_count. */
int uavsim_run_policy(uavsim_t *h, int mode, double cooperative, const UavSimPolicyWeights *w, uint64_t seed,
                      uint64_t first_counter, int64_t nsteps, const UavSimTrajectory *traj, void *stream);

/* Evaluation of a policy over many episodes in one call (the reference's `--phase evaluate`, src/train.py evaluate, for
 * all environments at once), in place on the bound buffers: for k = 0 .. n_episodes-1
 *     uavsim_reset(h, reset_seeds[k], stream);
 *     nsteps x (policy launch -> bound actions; uavsim_step; per-environment accumulation)
 * greedy = 0: step t of episode k draws as uavsim_policy_sample with counter first_counter + k*nsteps + t, i.e. each
 * episode is uavsim_run_policy(h, mode, cooperative, w, seed, first_counter + k*nsteps, nsteps, NULL, stream);
 * greedy = 1: uavsim_policy_greedy (seed and first_counter unused).  reset_seeds: HOST array [n_episodes].
 * env_stats: DEVICE float64 [n_episodes, E, 6], 8-byte aligned: per environment the sums over UAVs and steps of the four
 * reward planes (rewards, target_tracking, boundary, duplicate; as the statistics hold them: counts of 2^-22 of the fp32
 * values), the covered-target sum and the covered-target maximum over steps.  These are the integers the episode
 * statistics add up, so for every episode the sum of its rows over environments equals uavsim_episode_stats out[0..4]
 * and their maximum out[5], bit for bit, whichever step kernel ran.
 * The result is bit-identical to the loop above in the bound obs / actions / rew4 / covered, done, the state, the step
 * counter and uavsim_episode_stats (which hold the last episode).  uavsim_launch_count counts the loop's launches plus
 * nsteps + 1 per episode (the accumulation and the row output).  Every argument is checked before anything is queued
 * (negative counts, NULL reset_seeds / env_stats when n_episodes > 0, a misaligned env_stats, greedy not 0 / 1, the
 * weights, n_actions != na, the PMI path): on an error nothing is enqueued and the step counter does not move.
 * n_episodes = 0 queues nothing.  The handle keeps an [E,6] int64 accumulator, allocated on the first call. */
int uavsim_evaluate_policy(uavsim_t *h, int mode, double cooperative, const UavSimPolicyWeights *w, int greedy,
                           uint64_t seed, uint64_t first_counter, const uint64_t *reset_seeds, int64_t n_episodes,
                           int64_t nsteps, double *env_stats, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* UAVSIM_H */
