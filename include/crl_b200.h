/*
 * crl_b200.h -- C ABI of the B200-native batched simulator for competitive-rl's
 * vectorised env-stepping path.
 *
 * The reference (ucla-rlcourse/competitive-rl) is pure Python and has no FFI; the
 * boundary it exposes for this path is the vec-env protocol returned by
 *   make_envs(env_id, seed, log_dir, num_envs, asynchronous, resized_dim, frame_stack,
 *             action_repeat)                       competitive_rl/make_envs.py:67-118
 *   VecEnv.reset / step_async / step_wait / seed   competitive_rl/utils/base_vec_env.py:63-252
 * implemented by DummyVecEnv (utils/dummy_vec_env.py:27-75) and SubprocVecEnv
 * (utils/subproc_vec_env.py:81-129).  Each entry point below names the reference
 * interface it replaces.  INTEGRATION.md shows the ctypes binding a maintainer of
 * the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / CUDA types in the signatures
 *     (`stream` is a cudaStream_t passed as void*, NULL = legacy default stream);
 *   - every call returns 0 on success or a negative CRL_E_* code; crl_last_error()
 *     returns a thread-local message; no exceptions cross the ABI;
 *   - calls are stream-ordered and never synchronise the host unless stated;
 *   - `*_dev` pointers are device memory owned by the CALLER (e.g. torch tensors);
 *     `*_host` pointers are host memory; a handle is not thread-safe.
 *   - there is NO CPU fallback: without a CUDA device every call fails.
 */
#ifndef CRL_B200_H
#define CRL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRL_OK 0
#define CRL_E_INVALID (-1)   /* bad argument / unsupported configuration */
#define CRL_E_CUDA (-2)      /* a CUDA runtime call failed (message has the detail) */
#define CRL_E_STATE (-3)     /* call order violated (e.g. step before atlas/reset) */
#define CRL_E_SERVES (-4)    /* injected serve table exhausted */

#define CRL_ABI_VERSION 2
#define CRL_PONG_ATLAS_BYTES (22 * 22 * 34 * 160 * 3)
#define CRL_PONG_STATE_DOUBLES 10

typedef struct crl_pong crl_pong; /* opaque handle: one shard of envs on one GPU */

typedef struct crl_pong_config {
    int32_t num_envs;       /* envs in this shard (make_envs num_envs) */
    int32_t n_agents;       /* 1 = "cPong-v0" (built-in right bat), 2 = "cPongDouble-v0" */
    int32_t resized_dim;    /* make_envs resized_dim: 84 or 42 */
    int32_t frame_stack;    /* make_envs frame_stack; 0 = None (one channel) */
    int32_t max_num_rounds; /* gym registry kwarg, pong/register.py:13-22 (21) */
    int32_t device;         /* CUDA device ordinal */
    int32_t stack_mode;     /* 0 = every step writes the full (C, dim, dim) stack per agent, like FrameStack._get_ob
                               (utils/atari_wrappers.py:257-259).  1 = double-write ring: the observation buffers are
                               uint8 [num_envs][2*C][dim][dim] rings OWNED BY THE CALLER ACROSS STEPS (same pointers every
                               call); a step stores the newest frame at slots k and k + C, k = crl_pong_ring_phase(), and
                               the observation is the view of slots k+1 .. k+C (oldest -> newest): 2 frames written
                               instead of C.  Needs frame_stack >= 2. */
    int32_t zero_on_done;   /* 1 = FrameStackTensor semantics (utils/utils.py:145-173): after a done the history is all
                               zeros and only the newest frame is the reset observation, instead of FrameStack.reset's
                               C copies (utils/atari_wrappers.py:246-250) */
    uint64_t seed;          /* serve RNG seed (Philox); ignored once serves are injected */
    int64_t first_env;      /* global index of env 0 of this shard: RNG streams are keyed by
                               global env index, so results do not depend on the sharding */
} crl_pong_config;

int crl_abi_version(void);
const char* crl_last_error(void);

/* Construct the shard == running the num_envs thunks of make_env_a2c_atari
 * (utils/atari_wrappers.py:40-53): every PongGame constructor consumes two serves
 * (pong/base_pong_env.py:211, 312). */
int crl_pong_create(const crl_pong_config* cfg, crl_pong** out);
int crl_pong_destroy(crl_pong* h);

/* Scoreboard atlas: rows 0..33 of the 210x160x3 frame for every score pair,
 * uint8 [22][22][34][160][3] (what Scoreboard.draw, pong/base_pong_env.py:474-487,
 * leaves on the surface).  Builds the preprocessed-scoreboard tables on the device.
 * Must be called once before reset/step.  Synchronises the stream. */
int crl_pong_load_atlas(crl_pong* h, const uint8_t* strips_host, size_t bytes, void* stream);

/* Validation mode: replace the serve RNG by a table, serves_host[num_envs][k][2] =
 * (vx, vy) of the k-th serve each env consumes since construction (the reference
 * draws them from stdlib `random`, pong/base_pong_env.py:314-320).  Re-runs the
 * constructors so serves 0 and 1 come from the table.  Synchronises. */
int crl_pong_inject_serves(crl_pong* h, const double* serves_host, int32_t k, void* stream);

/* VecEnv.seed(seed) (base_vec_env.py:163-176): the reference Pong envs ignore seeds
 * (pong/base_pong_env.py:38-39); here it re-keys the serve RNG for FUTURE serves. */
int crl_pong_seed(crl_pong* h, uint64_t seed);

/* VecEnv.reset(): obs{0,1}_dev receive uint8 [num_envs][C][dim][dim] per agent
 * (obs1_dev is ignored for n_agents == 1).  stack_mode 1: [num_envs][2*C][dim][dim] rings, see crl_pong_config. */
int crl_pong_reset(crl_pong* h, uint8_t* obs0_dev, uint8_t* obs1_dev, void* stream);

/* VecEnv.step(actions) == step_async + step_wait with auto-reset on done.
 *   actions_dev      int32 [num_envs][2] (Double; 0/1/2 or 999 = built-in rule-based bat,
 *                    pong/base_pong_env.py:116-134) or int32 [num_envs] (single)
 *   rew_dev          float32 [num_envs][2]  np.sign of the frameskip reward sum (ClipRewardEnv)
 *   done_dev         uint8   [num_envs]
 *   num_steps_dev    int32   [num_envs]     info["num_steps"]
 *   real_reward_dev  float32 [num_envs][2]  info["real_reward"]
 * Observations of envs that finished are already those of the auto-reset. */
int crl_pong_step(crl_pong* h, const int32_t* actions_dev, uint8_t* obs0_dev, uint8_t* obs1_dev, float* rew_dev,
                  uint8_t* done_dev, int32_t* num_steps_dev, float* real_reward_dev, void* stream);

/* The two halves of crl_pong_step, for callers that want to overlap or time them:
 * game core only (one thread per env), then the fused rasteriser+preprocessing. */
int crl_pong_step_state(crl_pong* h, const int32_t* actions_dev, float* rew_dev, uint8_t* done_dev,
                        int32_t* num_steps_dev, float* real_reward_dev, void* stream);
int crl_pong_render_obs(crl_pong* h, uint8_t* obs0_dev, uint8_t* obs1_dev, void* stream);
/* float32 observations, as a STOCK gym install produces them (SURVEY.md F7): gym's Box without a dtype is float32
 * (pong/base_pong_env.py:22-24), MaxAndSkipEnv pools float32 frames (utils/atari_wrappers.py:106-115) and cv2 takes its
 * float paths, so an observation pixel is the UNROUNDED fp32 area sum -- except in frames that reset() returned, which
 * bypass MaxAndSkipEnv un-pooled as uint8 (:162-163) and enter the stack as rounded integers.  Use instead of
 * crl_pong_render_obs after crl_pong_step_state / crl_pong_reset_state: obs{0,1}_dev are float32
 * [num_envs][C][dim][dim]; terminal != 0 renders info["terminal_observation"] of the envs flagged in only_done_dev
 * (may be NULL = all) instead of the current observation.  One thread per pixel (not a tuned path), stack_mode 0 only. */
int crl_pong_render_obs_f32(crl_pong* h, int32_t terminal, const uint8_t* only_done_dev, float* obs0_dev, float* obs1_dev,
                            void* stream);
/* VecEnv.reset() without rendering (for callers that render with crl_pong_render_obs_f32) */
int crl_pong_reset_state(crl_pong* h, void* stream);
/* stack_mode 1: slot k the last step wrote the newest frame to (and to k + C); the observation is slots k+1 .. k+C.
 * Advanced by crl_pong_step / crl_pong_step_state, 0 after crl_pong_reset.  No device work, no synchronisation. */
int crl_pong_ring_phase(crl_pong* h);
/* same output through the one-thread-per-pixel reference rasteriser (cross-check) */
int crl_pong_render_obs_generic(crl_pong* h, uint8_t* obs0_dev, uint8_t* obs1_dev, void* stream);

/* Observation buffers whose contents the library may trust (stack_mode 0).  Registers `count` buffer sets: set i is
 * obs0_devs_host[i] and, for cPongDouble, obs1_devs_host[i] (may be NULL for cPong), each of crl_pong_render_obs's size.
 * The library remembers which frames a set holds after every render into it; at 84x84 a later crl_pong_render_obs (or
 * step / reset / step_host) into the same set stores only the 16-byte chunks whose frames changed.
 * The caller must therefore not write into a registered buffer, or must call crl_pong_forget_obs afterwards; the
 * library's own other writers (render_obs_generic, render_obs_f32, terminal_obs, load_atlas) do so themselves.
 * count = 0 unregisters every set.  Synchronises the stream.  Environment: CRL_PONG_FULL_OBS=1 at crl_pong_create makes
 * every render store whole stacks (A/B runs). */
#define CRL_PONG_MAX_OBS_SETS 16
int crl_pong_set_obs_buffers(crl_pong* h, uint8_t* const* obs0_devs_host, uint8_t* const* obs1_devs_host, int32_t count,
                             void* stream);
/* the registered sets' contents are unknown (the caller wrote into them): the next render into each stores it whole */
int crl_pong_forget_obs(crl_pong* h);

/* info["terminal_observation"] of the LAST step: writes, for every env whose
 * done_dev[i] != 0, the stacked observation the episode ended with into
 * term{0,1}_dev[i] (same layout as obs); other envs' slots are left untouched. */
int crl_pong_terminal_obs(crl_pong* h, const uint8_t* done_dev, uint8_t* term0_dev, uint8_t* term1_dev, void* stream);

/* Host-buffer form of step (what a numpy caller of the reference's VecEnv.step sees):
 * copies actions host->device, steps, copies rew/done/num_steps/real_reward back and,
 * when obs*_host are non-NULL, the observations too.  Synchronises the stream.
 * The small results leave on an internal side stream as soon as the game-core kernel has
 * produced them, i.e. behind the rasteriser; the side stream is joined before the call returns.
 * Host buffers should be pinned for full PCIe bandwidth.  obs*_dev are still required
 * (device staging owned by the caller). */
int crl_pong_step_host(crl_pong* h, const int32_t* actions_host, uint8_t* obs0_dev, uint8_t* obs1_dev,
                       uint8_t* obs0_host, uint8_t* obs1_host, float* rew_host, uint8_t* done_host,
                       int32_t* num_steps_host, float* real_reward_host, void* stream);

/* Game state, float64 [num_envs][10]: ball_x, ball_y, vx, vy, left_y, right_y,
 * score_left, score_right, num_rounds, num_steps (PongGame fields).
 *
 * crl_pong_set_state writes the game state only: Bat._current_move, the serve counter, the
 * MaxAndSkip buffers and the FrameStack history keep what they held.  Integer fields take the
 * C (int) truncation, vx / vy are stored as given.  The set_state domain, per row:
 *   ball_x in [0, 156], ball_y in [0, 190], left_y and right_y in [0, 255],
 *   vx and vy finite with |v| <= 64, score_left and score_right in [0, 21],
 *   num_rounds in [0, max_num_rounds - 1], num_steps in [0, 10000],
 *   every integer field integral.
 * The check runs on the device: a row outside the domain is not applied (that env keeps its
 * state) and the next crl_pong_check returns CRL_E_INVALID ("state outside the set_state domain").
 * A point scored after set_state can still take a score from 21 to 22 (when rounds remain):
 * the scoreboard atlas has no strip for such a score, and, as the reference's renderer leaves
 * them without a strip, frames showing it have plain white rows 0..33, no text. */
int crl_pong_get_state(crl_pong* h, double* state_dev, void* stream);
int crl_pong_set_state(crl_pong* h, const double* state_dev, void* stream);

/* VecEnv.get_images()/render (base_vec_env.py:189-216): raw 210x160x3 uint8 frame of
 * env `env` as agent 0 sees it, and (rgb1_dev may be NULL) agent 1's mirrored copy. */
int crl_pong_render_raw(crl_pong* h, int32_t env, uint8_t* rgb0_dev, uint8_t* rgb1_dev, void* stream);

/* Synthetic rollout driver: uniform actions in {0,1,2}, Philox keyed by (seed, step). */
int crl_pong_random_actions(int32_t* actions_dev, int32_t n_values, uint64_t seed, uint64_t step, void* stream);

/* Episode statistics accumulated on the device since construction (for the optional
 * end-of-run gather across GPUs; the reference tallies these on the host in
 * pong/evaluate.py:53-88 and utils/utils.py:23-60).  stats_host[8] (uint64):
 * [0] finished episodes, [1] sum of episode lengths in env-steps, [2] episodes won by the
 * left agent, [3] by the right agent, [4] draws, [5] sum over episodes of
 * (score_left - score_right + 64), [6..7] reserved.  Synchronises the stream. */
int crl_pong_get_stats(crl_pong* h, uint64_t* stats_host, void* stream);

/* Number of kernel launches this library has issued from this process (bench.py's
 * gpu_launches), and the deferred error check (synchronises): CRL_E_SERVES after a
 * serve-table overrun, CRL_E_INVALID after a step saw an action outside {0, 1, 2}
 * (cPongDouble: or 999) -- the reference asserts / raises IndexError there
 * (pong/base_pong_env.py:42, :124, :134); the device step plays it as 1 (stay) -- and
 * CRL_E_INVALID after crl_pong_set_state refused a row outside the set_state domain.  The flags
 * are cleared once reported; when several are set, the message names each of them and the code is
 * the first one's in this order: set_state domain, action, serve table. */
uint64_t crl_launch_count(void);
int crl_pong_check(crl_pong* h, void* stream);

/* Observation buffers.  crl_obs_alloc allocates `bytes` of device memory on `device` for the observations the
 * rasterisers write (crl_pong_*: obs0_dev / obs1_dev, and the rings of stack_mode 1).  Where the device supports generic
 * memory compression (CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED) the memory is a compressible mapping
 * (cuMemCreate with CU_MEM_ALLOCATION_COMP_GENERIC, size rounded up to the allocation granularity): Pong frames are
 * mostly constant runs, which the memory system then moves to and from DRAM in fewer bytes.  Contents and addressing
 * are those of any device memory.  *compressed is 1 when the driver granted compressible memory, 0 when the buffer is
 * an ordinary allocation (no support, or the request was refused).  crl_obs_free synchronises the device, then
 * releases a buffer crl_obs_alloc returned (NULL: no-op). */
int crl_obs_alloc(int32_t device, size_t bytes, void** ptr, int32_t* compressed);
int crl_obs_free(void* ptr);

/* ======================================================================================
 * cPongTournament-v0 per-env opponents
 * The reference's TournamentEnvWrapper (pong/competitive_pong_env.py:9-53) lets ONE built-in opponent play every env of
 * the batch.  A crl_pong_opp handle lets every env of a 42x42 cPongDouble shard play its own opponent, drawn from a
 * pool, in one kernel launch per step (crl_pong_opp_act), with no host synchronisation.
 *
 *   Pool        1..16 entries; an entry is CRL_PONG_OPP_RULE_BASED, CRL_PONG_OPP_RANDOM, or one of 8 network slots
 *               holding a LightActorCritic (utils/network.py:73-93: 4x42x42 -> conv 4x4/2 (16) -> conv 2x2/2 (16) ->
 *               1600 -> 3 logits).  ActorCritic networks are not supported.
 *   Assignment  int32 opponent id per env (an index into the pool): given explicitly, or drawn with the pool's weights
 *               from Philox keyed by (seed, global env index first_env + i, the env's count of finished episodes), so
 *               draws do not depend on the sharding.
 *   Stack       uint8 [num_envs][4][42][42] per handle, oldest -> newest, zero at creation.  Every act pushes agent 1's
 *               observation of the previous step, whatever the env's opponent is; done does not clear it (the
 *               reference's policy_serving.Policy stack is never cleared either).
 *   Action      written into column 1 of the caller's int32 [num_envs][2] step buffer (column 0 is the learner's):
 *               RULE_BASED 999; RANDOM a Philox-uniform draw from {0, 1, 2} keyed by (seed, global env index, act
 *               count); a network the argmax (ties: lowest index) of its actor logits over stack / 255 in fp32.
 *   Episodes    act receives the previous step's reward and done.  Agent 0's clipped rewards are summed per env; an env
 *               that finished credits the episode to the pool entry it played (agent 0 wins when the sum is > 0,
 *               draws at 0, loses below: pong/evaluate.py:53-88) and, with resample != 0, draws a new id.
 *
 * League mode (crl_pong_opp_set_pairs, crl_pong_opp_act_pairs, crl_pong_opp_get_pair_stats): both agents of every env
 * are played from the pool, so one launch per step evaluates every pairing of the pool in one batch.
 *   Pool        as above (crl_pong_opp_load_net, crl_pong_opp_set_pool); the pool's weights are not used.
 *   Pairings    pairs[P][2] = (pool index of seat 0, pool index of seat 1), 1 <= P <= CRL_PONG_OPP_MAX_PAIRS; repeated
 *               pairings and self-pairings (a, a) are allowed.  The env of global index g = first_env + i plays pairing
 *               g mod P (the non-negative remainder) for the whole run: nothing is redrawn, so the assignment does not
 *               depend on the sharding.
 *   Stacks      two uint8 [4][42][42] stacks per env, oldest -> newest.  Seat 0 is fed agent 0's observation, seat 1
 *               agent 1's (already mirrored by the env, so a network plays either seat as it was trained).  Both are
 *               zeroed by crl_pong_opp_set_pairs; done does not clear them, restart(clear_stacks != 0) does.
 *   Actions     every act_pairs writes both columns of the int32 [num_envs][2] step buffer: RULE_BASED 999 (the step
 *               accepts it for either bat); RANDOM a Philox-uniform draw from {0, 1, 2} keyed by (seed, global env
 *               index, act count), seat 1 on the stream of crl_pong_opp_act's RANDOM and seat 0 on a stream of its own;
 *               a network the argmax (ties: lowest index) of its fp32 actor logits over its seat's stack / 255, computed
 *               exactly as crl_pong_opp_act computes them.
 *   Episodes    agent 0's (seat 0's) clipped rewards are summed per env; an env that finished credits the episode to its
 *               pairing: [episodes, wins, draws, losses] of seat 0 (> 0, == 0, < 0).  As with crl_pong_opp_act, an
 *               episode is credited by the act_pairs call that follows the step that ended it.
 *   Modes       crl_pong_opp_act returns CRL_E_STATE in league mode and crl_pong_opp_act_pairs outside it.
 *               crl_pong_opp_set_pool leaves league mode: it zeroes the per-env reward sums and agent 1's stacks (the act
 *               count runs on), and crl_pong_opp_assign must follow it as always.  League mode does not change the
 *               opponent ids, the episode counts of the draws or the per-entry statistics of crl_pong_opp_get_stats.
 *
 * Learner mode (crl_pong_opp_load_learner, crl_pong_opp_act_learner): per-env opponents as above in seat 1, and in seat 0
 * a LightActorCritic learner whose network runs in the same launch, returning what a PPO rollout stores for the step.
 *   Learner     its own weights (crl_pong_opp_load_learner: the whole image, critic included), not one of the 8 slots,
 *               so a pool keeps all of them.  Every env runs it, whatever its opponent.
 *   Seat 1      exactly as crl_pong_opp_act: bookkeeping, redraws, pool actions, agent 1's stack, the act count, the
 *               per-entry statistics.  Only the opponents' logits are not returned.
 *   Ring        a uint8 [4][42][42] stack per env of agent 0's observations, oldest -> newest, with FrameStackTensor's
 *               semantics (utils/utils.py:145-173): every act_learner pushes agent 0's observation of the previous step,
 *               and when that step's done is set the env's ring is zeroed first, so that only the newest slot is
 *               non-zero.  All rings are zeroed on entering learner mode (the first act_learner after create,
 *               crl_pong_opp_set_pool or crl_pong_opp_set_pairs) and by every crl_pong_opp_restart in learner mode,
 *               whatever clear_stacks (a VecEnv reset starts every episode afresh).  They take num_envs * 7056 bytes,
 *               allocated by the first act_learner (shared with league mode's seat-0 stacks).
 *   Network     conv1 / conv2 / actor exactly as for a pool network (fp32 over stack / 255), and critic_linear
 *               (1600 -> 1) as one more sum of the same kind.
 *   Action      sample != 0: u = r32 * 2^-32 from Philox keyed by (seed, global env index, act count) with tag 4, a
 *               stream of its own, so it does not depend on the sharding or the batch; with m = max(l) and
 *               e_k = expf(l_k - m), s = (e_0 + e_1) + e_2, c_0 = e_0 / s and c_1 = c_0 + e_1 / s in fp32, the action
 *               is 0 if u < c_0, 1 if u < c_1, else 2 (u and c_k compared exactly).  sample == 0: the argmax of the
 *               logits, ties to the lowest index.
 *   Outputs     the action in column 0 of the step buffer; log pi(action) = l_a - (m + logf(s)) and the value; the
 *               logits if asked; the stack the learner acted on (the ring after the push, oldest -> newest).
 *   Modes       crl_pong_opp_act returns CRL_E_STATE in learner mode, so the two cannot be mixed: a frame of agent 0
 *               would be missing from the rings.  crl_pong_opp_set_pool and crl_pong_opp_set_pairs leave learner mode;
 *               crl_pong_opp_act_learner returns CRL_E_STATE in league mode, before crl_pong_opp_load_learner and before
 *               crl_pong_opp_assign.  Reloading the learner's weights does not leave learner mode.
 *
 * Self-play mode (crl_pong_opp_set_selfplay, crl_pong_opp_act_selfplay): league mode in which any seat of a pairing may
 * be the learner of learner mode, so one launch per step plays the current policy against itself, frozen snapshots and
 * built-in opponents, and returns what a PPO rollout stores for every learner seat.
 *   Pairings    pairs[P][2], 1 <= P <= CRL_PONG_OPP_MAX_PAIRS; each seat is a pool index or CRL_PONG_OPP_LEARNER.  Env
 *               g = first_env + i plays pairing g mod P for the whole run, as in league mode.  A pairing without a
 *               learner seat is allowed; its envs play exactly as in league mode.
 *   Learner     a learner seat runs the learner's image (crl_pong_opp_load_learner), computed as in learner mode: conv1 /
 *               conv2 / actor / critic in fp32 over stack / 255.  sample != 0: u = r32 * 2^-32 from Philox keyed by
 *               (seed, global env index, act count), tag 4 (learner mode's stream) in seat 0 and tag 5 in seat 1, and
 *               learner mode's inverse-CDF rule; sample == 0: the argmax of the logits, ties to the lowest index.
 *   Pool seats  as in league mode: RULE_BASED 999, RANDOM a draw from tag 3 in seat 0 and tag 1 in seat 1, a network the
 *               argmax of its logits.
 *   Rings       the two stacks of league mode, seat 0's fed agent 0's observations and seat 1's agent 1's: every act
 *               pushes the agent's observation of the previous step.  A learner seat's ring has FrameStackTensor's
 *               zeroing (when the previous step's done is set, the other three slots are zeroed first); a pool seat's is
 *               never cleared on done.  crl_pong_opp_set_selfplay zeroes both rings of every env.  crl_pong_opp_restart
 *               zeroes every learner seat's ring (before the next act's push), whatever clear_stacks; pool seats follow
 *               league mode's rule (zeroed by clear_stacks != 0 only).
 *   Episodes    credited per pairing from seat 0's side, as in league mode (crl_pong_opp_get_pair_stats).
 *   Outputs     both columns of the step buffer; for each learner seat log pi(action) and the value (0 and 0 for a pool
 *               seat); each seat's logits, learner or pool network (0 for RULE_BASED and RANDOM); for each learner seat
 *               the stack it acted on, oldest first (a pool seat's rows of stack_out are not written).
 *   Modes       crl_pong_opp_set_selfplay needs a pool (CRL_E_STATE otherwise), validates every seat and then enters
 *               self-play mode, allocating seat 0's stacks on first use as crl_pong_opp_set_pairs does.
 *               crl_pong_opp_act_selfplay returns CRL_E_STATE outside self-play mode and before crl_pong_opp_load_learner.
 *               In self-play mode crl_pong_opp_act, crl_pong_opp_act_pairs and crl_pong_opp_act_learner return
 *               CRL_E_STATE.  crl_pong_opp_set_pool and crl_pong_opp_set_pairs leave self-play mode; reloading the
 *               learner does not.  crl_pong_opp_set_pairs refuses CRL_PONG_OPP_LEARNER.
 * ====================================================================================== */
#define CRL_PONG_OPP_MAX_POOL 16
#define CRL_PONG_OPP_SLOTS 8
#define CRL_PONG_OPP_RULE_BASED (-1)   /* pool entry kinds; 0 .. CRL_PONG_OPP_SLOTS-1 = network slot */
#define CRL_PONG_OPP_RANDOM (-2)
#define CRL_PONG_OPP_MAX_PAIRS 256    /* pairings of league mode */
#define CRL_PONG_OPP_LEARNER (-3)     /* a learner seat of a self-play pairing */
/* LightActorCritic parameters in state-dict order, each row-major: conv1.weight [16][4][4][4], conv1.bias [16],
 * conv2.weight [16][16][2][2], conv2.bias [16], critic_linear.weight [1][1600], critic_linear.bias [1],
 * actor_linear.weight [3][1600], actor_linear.bias [3] (the critic is evaluated for the learner only) */
#define CRL_PONG_OPP_NET_FLOATS 8484

typedef struct crl_pong_opp crl_pong_opp; /* opaque handle: the opponents of one shard of envs on one GPU */

/* seed keys the draws and RANDOM's actions; first_env is the global index of env 0 of the shard */
int crl_pong_opp_create(int32_t num_envs, int32_t device, uint64_t seed, int64_t first_env, crl_pong_opp** out);
int crl_pong_opp_destroy(crl_pong_opp* h);
/* re-keys future draws and RANDOM actions; no device work */
int crl_pong_opp_seed(crl_pong_opp* h, uint64_t seed);
/* network slot <- params_host[CRL_PONG_OPP_NET_FLOATS] (finite).  Synchronises the stream. */
int crl_pong_opp_load_net(crl_pong_opp* h, int32_t slot, const float* params_host, size_t count, void* stream);
/* pool <- kinds_host[pool_size] (RULE_BASED, RANDOM or a loaded slot) with draw weights weights_host[pool_size] (>= 0,
 * not all 0; NULL = uniform).  Zeroes the per-entry statistics; crl_pong_opp_assign must follow before the next act. */
int crl_pong_opp_set_pool(crl_pong_opp* h, const int32_t* kinds_host, const double* weights_host, int32_t pool_size,
                          void* stream);
/* every env's opponent id <- ids_host[num_envs] (validated; synchronises), or drawn from the pool (ids_host NULL) */
int crl_pong_opp_assign(crl_pong_opp* h, const int32_t* ids_host, void* stream);
/* restarts the per-env reward sums (VecEnv.reset); clear_stacks != 0 also zeroes every frame stack */
int crl_pong_opp_restart(crl_pong_opp* h, int32_t clear_stacks, void* stream);
/* One step's opponents, before crl_pong_step:
 *   obs1_dev     uint8 [num_envs][42][42] agent 1's observation of the previous step (frame_stack None), 4-byte aligned
 *   rew_dev      float32 [num_envs][2] and done_dev uint8 [num_envs] of the previous step, or both NULL for the first
 *                act after a reset (no episode bookkeeping)
 *   resample     != 0: envs whose previous step ended an episode draw a new opponent id before acting
 *   actions_dev  int32 [num_envs][2]: column 1 receives the opponents' actions, column 0 is not touched
 *   logits_dev   float32 [num_envs][3] or NULL: the network envs' actor logits (0 for the other kinds) */
int crl_pong_opp_act(crl_pong_opp* h, const uint8_t* obs1_dev, const float* rew_dev, const uint8_t* done_dev, int32_t resample,
                     int32_t* actions_dev, float* logits_dev, void* stream);
/* ids_dev int32 [num_envs] <- every env's current opponent id */
int crl_pong_opp_get_ids(crl_pong_opp* h, int32_t* ids_dev, void* stream);
/* stats_host uint64 [16][4]: per pool entry, episodes finished against it, agent 0's wins, draws, losses (since the
 * last crl_pong_opp_set_pool).  Synchronises the stream. */
int crl_pong_opp_get_stats(crl_pong_opp* h, uint64_t* stats_host, void* stream);
/* Enters (or re-enters) league mode: pairs_host int32 [num_pairs][2] pool indices (seat 0, seat 1), every one validated
 * against the current pool (CRL_E_STATE without a pool).  Zeroes the pairing statistics, the per-env reward sums and
 * both stacks of every env, and restarts the ring.  Seat 0's stacks (num_envs * 7056 bytes) are allocated by the first
 * call, so a handle that never enters league mode does not pay for them. */
int crl_pong_opp_set_pairs(crl_pong_opp* h, const int32_t* pairs_host, int32_t num_pairs, void* stream);
/* One league step, before crl_pong_step:
 *   obs0_dev, obs1_dev  uint8 [num_envs][42][42] agent 0's and agent 1's observations of the previous step, 4-byte aligned
 *   rew_dev, done_dev   as crl_pong_opp_act (both NULL for the first act after a reset)
 *   actions_dev         int32 [num_envs][2]: both columns receive the seats' actions
 *   logits_dev          float32 [num_envs][2][3] or NULL: each network seat's actor logits (0 for the other kinds) */
int crl_pong_opp_act_pairs(crl_pong_opp* h, const uint8_t* obs0_dev, const uint8_t* obs1_dev, const float* rew_dev,
                           const uint8_t* done_dev, int32_t* actions_dev, float* logits_dev, void* stream);
/* stats_host uint64 [num_pairs][4]: per pairing, episodes finished, seat 0's wins, draws, losses (since the last
 * crl_pong_opp_set_pairs).  1 <= num_pairs <= CRL_PONG_OPP_MAX_PAIRS; rows past the league's P read 0.  Synchronises
 * the stream. */
int crl_pong_opp_get_pair_stats(crl_pong_opp* h, uint64_t* stats_host, int32_t num_pairs, void* stream);
/* learner <- params_host[CRL_PONG_OPP_NET_FLOATS] (finite), the whole image (pack_light_actor_critic order), critic
 * included; checked as crl_pong_opp_load_net.  Synchronises the stream: call it once per update, not per step. */
int crl_pong_opp_load_learner(crl_pong_opp* h, const float* params_host, size_t count, void* stream);
/* One learner-mode step, before crl_pong_step (enters learner mode, see above):
 *   obs0_dev, obs1_dev  uint8 [num_envs][42][42] agent 0's and agent 1's observations of the previous step, 4-byte aligned
 *   rew_dev, done_dev   as crl_pong_opp_act (both NULL for the first act after a reset)
 *   resample            as crl_pong_opp_act
 *   sample              != 0: sample the learner's action from its softmax; 0: the argmax
 *   actions_dev         int32 [num_envs][2]: column 0 the learner's action, column 1 the opponent's
 *   logp_value_dev      float32 [num_envs][2]: log pi(action), value
 *   logits_dev          float32 [num_envs][3] or NULL: the learner's logits
 *   stack_out_dev       uint8 [num_envs][4][42][42], 4-byte aligned: the stack the learner acted on, oldest first */
int crl_pong_opp_act_learner(crl_pong_opp* h, const uint8_t* obs0_dev, const uint8_t* obs1_dev, const float* rew_dev,
                             const uint8_t* done_dev, int32_t resample, int32_t sample, int32_t* actions_dev,
                             float* logp_value_dev, float* logits_dev, uint8_t* stack_out_dev, void* stream);
/* Enters (or re-enters) self-play mode: pairs_host int32 [num_pairs][2], each seat a pool index or CRL_PONG_OPP_LEARNER,
 * every one validated (CRL_E_STATE without a pool).  Zeroes the pairing statistics, the per-env reward sums and both
 * stacks of every env, and restarts the ring, as crl_pong_opp_set_pairs does. */
int crl_pong_opp_set_selfplay(crl_pong_opp* h, const int32_t* pairs_host, int32_t num_pairs, void* stream);
/* One self-play step, before crl_pong_step (see above):
 *   obs0_dev, obs1_dev  uint8 [num_envs][42][42] agent 0's and agent 1's observations of the previous step, 4-byte aligned
 *   rew_dev, done_dev   as crl_pong_opp_act (both NULL for the first act after a reset)
 *   sample              != 0: sample the learner seats' actions from their softmax; 0: the argmax
 *   actions_dev         int32 [num_envs][2]: both columns
 *   logp_value_dev      float32 [num_envs][2][2]: per seat log pi(action), value (0, 0 for a pool seat)
 *   logits_dev          float32 [num_envs][2][3] or NULL: each seat's logits (0 for RULE_BASED and RANDOM)
 *   stack_out_dev       uint8 [num_envs][2][4][42][42], 4-byte aligned: each learner seat's stack, oldest first */
int crl_pong_opp_act_selfplay(crl_pong_opp* h, const uint8_t* obs0_dev, const uint8_t* obs1_dev, const float* rew_dev,
                              const uint8_t* done_dev, int32_t sample, int32_t* actions_dev, float* logp_value_dev,
                              float* logits_dev, uint8_t* stack_out_dev, void* stream);

/* ======================================================================================
 * cCarRacing-v0 / cCarRacingDouble-v0
 * Replaces the env stack built by make_car_racing / make_car_racing_double
 * (car_racing/register.py:29-53): gym.make(id) [TimeLimit(1000)] -> FrameStack |
 * MultipleFrameStack + FlattenMultiAgentObservation -> WrapPyTorch, stepped by a vec-env.
 * ====================================================================================== */
#define CRL_CAR_DRAWS 24          /* np_random.uniform draws of one _create_track attempt */
#define CRL_CAR_STATE_DOUBLES 24
#define CRL_CAR_GLYPH_BYTES (11 * 8 * 4 + 11)

typedef struct crl_car crl_car;

typedef struct crl_car_config {
    int32_t num_envs;
    int32_t num_players;        /* 1 = "cCarRacing-v0", 2 = "cCarRacingDouble-v0" */
    int32_t frame_stack;        /* make_envs frame_stack; 0 = None */
    int32_t action_repeat;      /* CarRacing(action_repeat=...), 0/None = 1 */
    int32_t max_episode_steps;  /* gym registry TimeLimit (car_racing/register.py:14,21): 1000; 0 = off */
    int32_t device;
    int32_t done_mode;          /* two cars: 0 = env done when ANY car is (FlattenMultiAgentObservation.step,
                                   utils/atari_wrappers.py:323-331, the make_envs path); 1 = when car 0 is
                                   (make_competitive_car_racing returns d[0], make_competitive_car_racing.py:29-33) */
    int32_t stack_mode;         /* 0 = every step writes the whole (players * C, 96, 96) observation (FrameStack._get_ob /
                                   FlattenMultiAgentObservation, utils/atari_wrappers.py:257-259, 333-334).  1 = double-write
                                   ring: obs_dev is uint8 [num_envs][players][2*C][96][96], owned by the caller ACROSS
                                   steps (same pointer every call); a step stores each player's new frame at slots k and
                                   k + C, k = crl_car_ring_phase(), and the player's stack is the view of slots
                                   k+1 .. k+C (oldest -> newest).  Needs frame_stack >= 2.  term_obs_dev rows stay plain
                                   [players * C][96][96] stacks. */
    uint64_t seed;              /* track / birth-place RNG (Philox) */
    int64_t first_env;          /* global index of env 0 of this shard */
} crl_car_config;

int crl_car_create(const crl_car_config* cfg, crl_car** out);
int crl_car_destroy(crl_car* h);

/* HUD glyphs: the reward text "%05.0f" is drawn into every observation with COMIC.TTF 5 px,
 * non-antialiased (car_racing_multi_players.py:225-229, 669).  uint8 [11][8][4] bitmaps of
 * "0123456789-" followed by [11] advances.  Optional: without it no text is drawn. */
int crl_car_load_glyphs(crl_car* h, const uint8_t* glyphs_host, size_t bytes, void* stream);

/* Validation mode: draws_host[num_envs][k_draws][24] = the np_random.uniform values of the k-th
 * _create_track attempt of each env (car_racing_multi_players.py:268-270), birth_host
 * [num_envs][k_birth][num_players] = the shuffled birth_place_indices of the k-th reset
 * (:508-509; may be NULL).  Synchronises. */
int crl_car_inject_tracks(crl_car* h, const double* draws_host, int32_t k_draws, const int32_t* birth_host,
                          int32_t k_birth, void* stream);

/* VecEnv.reset(): obs_dev uint8 [num_envs][num_players * C][96][96]. */
/* CarRacing.reset(use_local_track=<json>) (car_racing_multi_players.py:376-381): replay recorded tracks instead of
 * generating them.  pts_host: float64 [n_tracks][CRL_CAR_MAX_TRACK][3] = (beta, x, y) of every track point (the JSON
 * rows are [alpha, beta, x, y]; alpha is not used downstream), counts_host: int32 [n_tracks] points per track.  From the
 * next reset on, env i (global index) uses track i % n_tracks at every reset.  n_tracks = 0 returns to generated tracks. */
int crl_car_load_tracks(crl_car* h, const double* pts_host, const int32_t* counts_host, int32_t n_tracks, void* stream);
int crl_car_reset(crl_car* h, uint8_t* obs_dev, void* stream);

/* VecEnv.seed(seed) (base_vec_env.py:163-176 -> CarRacing.seed, car_racing_multi_players.py:248-250): re-keys the
 * track / birth-place RNG for the tracks generated from now on (env i uses the stream of its global index).  Tracks
 * generated ahead of time under the old seed are dropped.  Synchronises. */
int crl_car_seed(crl_car* h, uint64_t seed, void* stream);

/* VecEnv.step with auto-reset.
 *   actions_dev     float32 [num_envs][num_players][2]  (steer, gas/brake), clipped like process_action
 *   rew_dev         float32 [num_envs][num_players]     per-car step reward (the Double wrapper returns [:, 0])
 *   done_dev        uint8   [num_envs]                  any car done, or TimeLimit
 *   num_steps_dev   int32   [num_envs]                  info["num_steps"]
 *   truncated_dev   uint8   [num_envs]                  bit 1: the gym TimeLimit fired on this step (the key
 *                                                       info["TimeLimit.truncated"] exists), bit 0: its value -- `not done`
 *                                                       with one car; always False with two, whose `done` is a (truthy) dict
 *   term_obs_dev    may be NULL; else same layout as obs: rows of finished envs receive
 *                   info["terminal_observation"]. */
int crl_car_step(crl_car* h, const float* actions_dev, uint8_t* obs_dev, float* rew_dev, uint8_t* done_dev,
                 int32_t* num_steps_dev, uint8_t* truncated_dev, uint8_t* term_obs_dev, void* stream);

/* Pre-age the envs: TimeLimit._elapsed_steps of every env (gym TimeLimit, car_racing/register.py:14,21), int32
 * [num_envs] on the device.  A rollout whose envs were all reset together truncates them all on the same step; a
 * long-running trainer sees them spread out, which is what this reproduces for measurements and tests. */
int crl_car_set_elapsed(crl_car* h, const int32_t* elapsed_dev, void* stream);

/* Host-buffer form of crl_car_step (what a numpy caller of the reference's VecEnv.step sees): copies the actions
 * host->device, steps, copies rew / done / num_steps / truncated back and, when obs_host is non-NULL, the observation
 * too.  obs_dev (and term_obs_dev, may be NULL) are device staging owned by the caller.  Synchronises the stream. */
int crl_car_step_host(crl_car* h, const float* actions_host, uint8_t* obs_dev, uint8_t* obs_host, float* rew_host,
                      uint8_t* done_host, int32_t* num_steps_host, uint8_t* truncated_host, uint8_t* term_obs_dev,
                      void* stream);

/* the two halves of crl_car_step: game core (no rendering, no auto-reset), then
 * render + auto-reset + render of the reset envs */
int crl_car_step_state(crl_car* h, const float* actions_dev, float* rew_dev, uint8_t* done_dev,
                       int32_t* num_steps_dev, uint8_t* truncated_dev, void* stream);
int crl_car_render_obs(crl_car* h, uint8_t* obs_dev, uint8_t* term_obs_dev, void* stream);

/* float64 [num_envs * num_players][24]: hull x, y, angle, vx, vy, w; per wheel: joint angle,
 * omega, gas, #tiles touched; reward; tiles visited. */
int crl_car_get_state(crl_car* h, double* state_dev, void* stream);
/* Debug / tests: put every car into the state described by float64 [num_envs * num_players][24] (layout of
 * crl_car_get_state; used: hull pose and velocity, wheel joint angles, omega, gas, reward).  Wheels are placed on their
 * joint anchors moving rigidly with the hull; joint impulses, car-car contacts and wheel tile sets are cleared. */
int crl_car_set_state(crl_car* h, const double* state_dev, void* stream);
/* Debug / tests: render every player's view of the CURRENT state as one more frame of the stack (what a step's rendering
 * does, without the game core and without the auto-reset passes), e.g. after crl_car_set_state. */
int crl_car_render_state(crl_car* h, uint8_t* obs_dev, void* stream);
/* stack_mode 1: slot k the last step wrote the new frames to (and to k + C).  0 after crl_car_reset. */
int crl_car_ring_phase(crl_car* h);
/* stack_mode 0 without moving frames (FrameStack, utils/atari_wrappers.py:222-259, as it is: a fully materialised
 * [players * C][96][96] stack per env).  Register `count` >= frame_stack + 1 (<= 16) observation buffers of the usual
 * layout; from then on crl_car_reset accepts any of them and the k-th crl_car_step / crl_car_render_obs /
 * crl_car_render_state after it must be given the next one in rotation (CRL_E_INVALID otherwise).  Each new frame is
 * written straight into the frame_stack buffers it will appear in (channel C-1 of the current one, C-2 of the next,
 * ...), so the C-1 frames that stay are never copied and no internal ring is kept: the bytes a step writes are the
 * observation bytes, and it reads none.  What a call returned stays intact for count - frame_stack further calls.
 * count = 0 returns to the plain mode (caller-chosen buffer per call, internal ring + stack-shift kernel). */
int crl_car_set_obs_rotation(crl_car* h, uint8_t* const* obs_devs_host, int32_t count, void* stream);
/* number of tiles of env `env`'s current track, and (if non-NULL) its track points float64 [n][3] beta, x, y */
int crl_car_get_track(crl_car* h, int32_t env, int32_t* n_out, double* pts_host, int32_t max_points, void* stream);

int crl_car_random_actions(float* actions_dev, int32_t n_values, uint64_t seed, uint64_t step, void* stream);
/* [0] episodes [1] sum of episode lengths [2] sum of tiles visited (car 0) [3] auto-resets that found no track
 * generated ahead and built it inside the step [4] car fixture polygons taller than their 8-row span table (cut; impossible for rigid fixtures at obs_scale)
 * [5] launches of the ahead-of-time track generator so far */
int crl_car_get_stats(crl_car* h, uint64_t* stats_host, void* stream);
/* car-car contacts of cCarRacingDouble (what box2d-py's b2World::Step resolves between the fixtures of the two
 * cars, car_dynamics.py:63-68,94-96): int32 [num_envs] touching fixture pairs per env after the last step, and the
 * number of contacts dropped so far because an env had more than 8 touching pairs at once (either may be NULL). */
int crl_car_get_contacts(crl_car* h, int32_t* counts_host, int32_t* overflow_host, void* stream);
int crl_car_check(crl_car* h, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CRL_B200_H */
