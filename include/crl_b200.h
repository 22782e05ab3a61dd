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
 * score_left, score_right, num_rounds, num_steps (PongGame fields). */
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
 * (pong/base_pong_env.py:42, :124, :134); the device step plays it as 1 (stay). */
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
