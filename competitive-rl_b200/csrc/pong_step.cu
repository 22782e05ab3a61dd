// pong_step.cu -- the Pong game core: one thread per environment, state in registers.
//
// Replaces (paths relative to /root/reference/competitive_rl/):
//   PongGame.step / _reset_round / reset_game        pong/base_pong_env.py:213-257
//   Ball.move / _bounce / reset / *_out_of_arena     pong/base_pong_env.py:314-381
//   Bat.move, AutoBat.move, auto_action              pong/base_pong_env.py:412-471
//   Pong{Single,Double}PlayerEnv._step / _reset      pong/base_pong_env.py:41-51, 113-147
//   MaxAndSkipEnv.step (frameskip 4, reward sum)     utils/atari_wrappers.py:118-160
//   ClipRewardEnv.step / reset                       utils/atari_wrappers.py:166-181
//   FrameStack deque bookkeeping                     utils/atari_wrappers.py:246-255
//   DummyVecEnv.step_wait auto-reset                 utils/dummy_vec_env.py:51-63
//
// The kernel does not draw anything: it records WHAT each buffered frame shows
// (RenderState, 8 bytes) and the rasteriser (pong_raster.cu) turns the frame
// specs of the FrameStack deque into uint8 observations.
//
// Arithmetic: positions are ints (pygame.Rect stores ints and truncates toward
// zero on store), ball velocity is fp64 exactly as the Python floats of the
// reference.  All fp64 ops use explicit round-to-nearest intrinsics so nothing is
// contracted into an FMA (an FMA changes the last bit of y_on_bat).
#include "pong_common.cuh"

namespace crl {

struct Game {
    int ball_x, ball_y;
    double vx, vy;
    int left_y, right_y;
    int score_left, score_right, num_rounds, num_steps;
    int serve_count;
};

// Ball.reset, pong/base_pong_env.py:314-320.  Validation mode: the k-th draw triple
// (uniform, choice, choice) is replaced by serves[env][k] = (vx, vy).  Otherwise
// Philox4x32-10 keyed by (seed, global env index) with the serve ordinal as counter.
__device__ __forceinline__ void ball_reset(const PongDev& p, int e, Game& g) {
    g.ball_x = BALL_X0;
    g.ball_y = BALL_Y0;
    if (p.serves != nullptr) {
        int k = g.serve_count;
        if (k >= p.serves_k) {
            atomicOr(p.serve_overrun, 1);
            k = p.serves_k - 1;
        }
        const double2 s = reinterpret_cast<const double2*>(p.serves)[(size_t)e * p.serves_k + k];
        g.vx = s.x;
        g.vy = s.y;
    } else {
        uint64_t gi = (uint64_t)(p.first_env + e);
        uint32_t r[4];
        philox4x32_10((uint32_t)g.serve_count, 0u, (uint32_t)gi, (uint32_t)(gi >> 32), (uint32_t)p.seed,
                      (uint32_t)(p.seed >> 32), r);
        // random.uniform(a, b) = a + (b - a) * random(), 53-bit random()
        double u = (double)((((uint64_t)r[0] >> 5) << 26) | ((uint64_t)r[1] >> 6)) * (1.0 / 9007199254740992.0);
        const double lo = __dmul_rn((double)SPEED, 0.3), hi = (double)SPEED;
        double vy0 = __dadd_rn(lo, __dmul_rn(__dadd_rn(hi, -lo), u));
        g.vx = (r[2] & 0x80000000u) ? (double)SPEED : -(double)SPEED;
        g.vy = (r[3] & 0x80000000u) ? vy0 : -vy0;
    }
    g.serve_count += 1;
}

// auto_action, pong/base_pong_env.py:457-471
__device__ __forceinline__ int auto_action(double ball_speed_x, int rect_cy, int ball_cy) {
    int d = 0;
    if (ball_speed_x < 0) {
        if (rect_cy < ARENA_CENTERY) d = 1;
        else if (rect_cy > ARENA_CENTERY) d = -1;
    } else if (ball_speed_x > 0) {
        d = (rect_cy < ball_cy) ? 1 : -1;
    }
    return d;
}

// Bat.move, pong/base_pong_env.py:412-418; returns Bat._current_move
__device__ __forceinline__ int bat_move(int& y, int direction) {
    int mv = direction * SPEED;
    y += mv;
    if (y + BAT_H > ARENA_BOTTOM) y += ARENA_BOTTOM - (y + BAT_H);
    else if (y < ARENA_TOP) y += ARENA_TOP - y;
    return mv;
}

// Ball.move + _bounce, pong/base_pong_env.py:325-361, 375-381.  (int) is cvt.rzi:
// the truncation toward zero of pygame's Rect attribute store.
__device__ __forceinline__ void ball_move(Game& g, int left_move, int right_move) {
    const int prev_left = g.ball_x, prev_right = g.ball_x + BALL_SIZE;
    const int rb_left = RIGHT_BAT_X, lb_right = LEFT_BAT_X + BAT_W;
    const double by = (double)g.ball_y;
    const double y_on_right = __dadd_rn(__dmul_rn(__ddiv_rn((double)(rb_left - prev_right), g.vx), g.vy), by);
    const double y_on_left = __dadd_rn(__dmul_rn(__ddiv_rn((double)(lb_right - prev_left), g.vx), g.vy), by);
    g.ball_x = (int)__dadd_rn((double)g.ball_x, g.vx);
    g.ball_y = (int)__dadd_rn(by, g.vy);
    if (g.vy < 0 && g.ball_y <= ARENA_TOP) {
        g.vy = -g.vy;
        g.ball_y = ARENA_TOP;
    } else if (g.vy > 0 && g.ball_y + BALL_SIZE >= ARENA_BOTTOM) {
        g.vy = -g.vy;
        g.ball_y = ARENA_BOTTOM - BALL_SIZE;
    } else if (g.vx < 0 && g.ball_x <= lb_right && __dadd_rn(y_on_left, (double)BALL_SIZE) >= (double)g.left_y &&
               y_on_left <= (double)(g.left_y + BAT_H) && prev_left > lb_right) {
        g.vx = -g.vx;
        g.vy = __dadd_rn(g.vy, __dmul_rn((double)left_move, 0.7));
        g.ball_x = lb_right;
        g.ball_y = (int)y_on_left;
    } else if (g.vx > 0 && g.ball_x + BALL_SIZE >= rb_left &&
               __dadd_rn(y_on_right, (double)BALL_SIZE) >= (double)g.right_y &&
               y_on_right <= (double)(g.right_y + BAT_H) && prev_right < rb_left) {
        g.vx = -g.vx;
        g.vy = __dadd_rn(g.vy, __dmul_rn((double)right_move, 0.7));
        g.ball_x = rb_left - BALL_SIZE;
        g.ball_y = (int)y_on_right;
    }
}

// PongGame._reset_round (:247-250) followed by both Bat.reset (:420-422)
__device__ __forceinline__ void reset_round(const PongDev& p, int e, Game& g) {
    ball_reset(p, e, g);
    g.num_rounds += 1;
    g.num_steps = 0;
    g.left_y = BAT_Y0;
    g.right_y = BAT_Y0;
}

// PongGame.reset_game, pong/base_pong_env.py:252-257
__device__ __forceinline__ void reset_game(const PongDev& p, int e, Game& g) {
    g.score_left = g.score_right = 0;
    reset_round(p, e, g);
    g.num_rounds = 0;
}

// One game frame: env._step action decode (:113-142 / :41-46) + PongGame.step (:213-245).
__device__ __forceinline__ bool game_frame(const PongDev& p, int e, Game& g, int a_left, int a_right, int& r0, int& r1) {
    int left_dir, right_dir;
    const int ball_cy = g.ball_y + (BALL_SIZE >> 1);
    if (p.n_agents == 2) {
        right_dir = (a_right == CHEAT_CODES) ? auto_action(g.vx, g.right_y + (BAT_H >> 1), ball_cy) : a_right - 1;
        left_dir = (a_left == CHEAT_CODES) ? auto_action(-g.vx, g.left_y + (BAT_H >> 1), ball_cy) : a_left - 1;
    } else {
        left_dir = a_left - 1;                                              // BAT_DIRECTIONS[a]
        right_dir = auto_action(g.vx, g.right_y + (BAT_H >> 1), ball_cy);   // AutoBat.move :445-454
    }
    g.num_steps += 1;
    const int lm = bat_move(g.left_y, left_dir);
    const int rm = bat_move(g.right_y, right_dir);
    ball_move(g, lm, rm);
    r0 = r1 = 0;
    if (g.ball_x < 0) {
        g.score_right += 1;
        r0 = -1; r1 = 1;
        reset_round(p, e, g);
    } else if (g.ball_x + BALL_SIZE > SCREEN_W) {
        g.score_left += 1;
        r0 = 1; r1 = -1;
        reset_round(p, e, g);
    } else if (g.num_steps > MAX_STEP_PER_ROUND) {
        reset_round(p, e, g);
    }
    return g.num_rounds >= p.max_rounds;
}

__device__ __forceinline__ Game load_game(const PongDev& p, int e) {
    Game g;
    const int32_t b = p.ball[e], t = p.bats[e], s = p.score[e];
    g.ball_x = (int)(int16_t)(b & 0xffff);
    g.ball_y = (int)(int16_t)(b >> 16);
    g.vx = p.vx[e];
    g.vy = p.vy[e];
    g.left_y = t & 0xffff;
    g.right_y = (t >> 16) & 0xffff;
    g.score_left = s & 0xff;
    g.score_right = (s >> 8) & 0xff;
    g.num_rounds = (s >> 16) & 0xffff;
    g.num_steps = p.num_steps[e];
    g.serve_count = p.serve_count[e];
    return g;
}

__device__ __forceinline__ void store_game(const PongDev& p, int e, const Game& g) {
    p.ball[e] = (int32_t)((uint32_t)(g.ball_x & 0xffff) | ((uint32_t)(g.ball_y & 0xffff) << 16));
    p.vx[e] = g.vx;
    p.vy[e] = g.vy;
    p.bats[e] = g.left_y | (g.right_y << 16);
    p.score[e] = g.score_left | (g.score_right << 8) | (g.num_rounds << 16);
    p.num_steps[e] = g.num_steps;
    p.serve_count[e] = g.serve_count;
}

__device__ __forceinline__ RenderState snapshot(const Game& g) {
    return make_render_state(g.ball_x, g.ball_y, g.left_y, g.right_y, g.score_left, g.score_right);
}

// env.reset() through the wrapper stack: reset_game, ClipRewardEnv._steps = 0, and the
// FrameStack deque filled with n copies of the RAW (un-pooled) reset frame
// (utils/atari_wrappers.py:246-250, :162-163).  MaxAndSkip's buffers are NOT cleared.
__device__ __forceinline__ void env_reset(const PongDev& p, int e, Game& g) {
    reset_game(p, e, g);
    p.clip_steps[e] = 0;
    const RenderState rs = snapshot(g);
    const FrameSpec spec = make_uint4(rs.x, rs.y | (1u << 17), rs.x, rs.y | (1u << 17));   // bit 17: reset()'s un-pooled frame
    // FrameStackTensor.update (utils/utils.py:159-170): `obs *= mask` zeroes the history of a finished env before the
    // reset observation is appended; valid bit 0 = the all-zero frame
    const FrameSpec old = p.zero_on_done ? make_uint4(0u, 0u, 0u, 0u) : spec;
    for (int k = 0; k + 1 < p.c; ++k) p.hist[(size_t)k * p.n + e] = old;
    p.hist[(size_t)(p.c - 1) * p.n + e] = spec;
}

// PongGame.__init__: Ball.__init__ -> reset() (:312) then reset_game() (:211): two serves.
__global__ void pong_construct_kernel(PongDev p) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.n) return;
    Game g;
    g.serve_count = 0;
    g.score_left = g.score_right = g.num_rounds = g.num_steps = 0;
    g.left_y = g.right_y = BAT_Y0;
    ball_reset(p, e, g);
    reset_game(p, e, g);
    store_game(p, e, g);
    p.clip_steps[e] = 0;
    p.skipbuf[e] = make_uint2(0u, 0u);                   // np.zeros buffers, atari_wrappers.py:106-115
    p.skipbuf[(size_t)p.n + e] = make_uint2(0u, 0u);
    for (int k = 0; k < p.c; ++k) {
        p.hist[(size_t)k * p.n + e] = make_uint4(0u, 0u, 0u, 0u);
        p.term_hist[(size_t)k * p.n + e] = make_uint4(0u, 0u, 0u, 0u);
    }
}

__global__ void pong_reset_kernel(PongDev p) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.n) return;
    Game g = load_game(p, e);
    env_reset(p, e, g);
    store_game(p, e, g);
}

__global__ void __launch_bounds__(128)
pong_step_kernel(PongDev p, const int32_t* __restrict__ actions, float* __restrict__ rew, uint8_t* __restrict__ done_out,
                 int32_t* __restrict__ num_steps_out, float* __restrict__ real_reward) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.n) return;
    Game g = load_game(p, e);
    int a_left, a_right = 1;
    if (p.n_agents == 2) {
        const int2 a = reinterpret_cast<const int2*>(actions)[e];
        a_left = a.x;
        a_right = a.y;
    } else {
        a_left = actions[e];
    }
    // The reference rejects anything else (assert action_space.contains, :42; BAT_DIRECTIONS[a], :124/:134).  A device
    // kernel cannot raise: the step treats the action as "stay" and crl_pong_check reports it.
    const bool ok_left = (unsigned)a_left <= 2u || (p.n_agents == 2 && a_left == CHEAT_CODES);
    const bool ok_right = (unsigned)a_right <= 2u || (p.n_agents == 2 && a_right == CHEAT_CODES);
    if (!ok_left || !ok_right) {
        atomicOr(p.serve_overrun, 2);
        if (!ok_left) a_left = 1;
        if (!ok_right) a_right = 1;
    }
    RenderState buf0 = p.skipbuf[e], buf1 = p.skipbuf[(size_t)p.n + e];
    int total0 = 0, total1 = 0;
    bool done = false;
#pragma unroll 1
    for (int i = 0; i < 4; ++i) {   // MaxAndSkipEnv.step, skip = 4
        int r0, r1;
        done = game_frame(p, e, g, a_left, a_right, r0, r1);
        if (i == 2) buf0 = snapshot(g);
        if (i == 3) buf1 = snapshot(g);
        total0 += r0;
        total1 += r1;
        if (done) break;            // buffers keep stale frames on an early done
    }
    p.skipbuf[e] = buf0;
    p.skipbuf[(size_t)p.n + e] = buf1;
    // FrameStack.step: deque.append(max of the two buffered frames)
    const FrameSpec spec = make_uint4(buf0.x, buf0.y, buf1.x, buf1.y);
    FrameSpec h[MAX_STACK];
#pragma unroll
    for (int k = 0; k < MAX_STACK; ++k)
        if (k + 1 < p.c) h[k] = p.hist[(size_t)(k + 1) * p.n + e];
#pragma unroll
    for (int k = 0; k < MAX_STACK; ++k)
        if (k + 1 < p.c) p.hist[(size_t)k * p.n + e] = h[k];
    p.hist[(size_t)(p.c - 1) * p.n + e] = spec;
    // ClipRewardEnv.step: _steps += 1; real_reward; np.sign
    const int steps = p.clip_steps[e] + 1;
    p.clip_steps[e] = steps;
    num_steps_out[e] = steps;
    reinterpret_cast<float2*>(real_reward)[e] = make_float2((float)total0, (float)total1);
    reinterpret_cast<float2*>(rew)[e] =
        make_float2((float)((total0 > 0) - (total0 < 0)), (float)((total1 > 0) - (total1 < 0)));
    done_out[e] = done ? 1 : 0;
    p.last_done[e] = done ? 1 : 0;
    if (done) {   // vec-env auto-reset: keep the terminal deque, then env.reset()
        atomicAdd(&p.stats[0], 1ull);
        atomicAdd(&p.stats[1], (unsigned long long)steps);
        atomicAdd(&p.stats[g.score_left > g.score_right ? 2 : (g.score_left < g.score_right ? 3 : 4)], 1ull);
        atomicAdd(&p.stats[5], (unsigned long long)(g.score_left - g.score_right + 64));
#pragma unroll
        for (int k = 0; k < MAX_STACK; ++k)
            if (k + 1 < p.c) p.term_hist[(size_t)k * p.n + e] = h[k];
        p.term_hist[(size_t)(p.c - 1) * p.n + e] = spec;
        env_reset(p, e, g);
    }
    store_game(p, e, g);
}

// state[n][10] = ball_x, ball_y, vx, vy, left_y, right_y, score_l, score_r, rounds, steps
__global__ void pong_get_state_kernel(PongDev p, double* state) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.n) return;
    const Game g = load_game(p, e);
    double* s = state + (size_t)e * 10;
    s[0] = g.ball_x; s[1] = g.ball_y; s[2] = g.vx; s[3] = g.vy; s[4] = g.left_y; s[5] = g.right_y;
    s[6] = g.score_left; s[7] = g.score_right; s[8] = g.num_rounds; s[9] = g.num_steps;
}

// v is an integer in [lo, hi] (false for NaN)
__device__ __forceinline__ bool int_in(double v, double lo, double hi) { return v >= lo && v <= hi && v == trunc(v); }

// The set_state domain (include/crl_b200.h): every field fits the packed state and the 8-bit render-state coordinates,
// and every score has an atlas strip.  A row outside it is not applied; crl_pong_check reports it (flag bit 4).
__device__ __forceinline__ bool state_in_domain(const double* s, int max_rounds) {
    return int_in(s[0], 0.0, (double)(SCREEN_W - BALL_SIZE)) && int_in(s[1], 0.0, (double)(ARENA_BOTTOM - BALL_SIZE)) &&
           fabs(s[2]) <= 64.0 && fabs(s[3]) <= 64.0 && int_in(s[4], 0.0, 255.0) && int_in(s[5], 0.0, 255.0) &&
           int_in(s[6], 0.0, (double)(ATLAS_SCORES - 1)) && int_in(s[7], 0.0, (double)(ATLAS_SCORES - 1)) &&
           int_in(s[8], 0.0, (double)(max_rounds - 1)) && int_in(s[9], 0.0, (double)MAX_STEP_PER_ROUND);
}

__global__ void pong_set_state_kernel(PongDev p, const double* state) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.n) return;
    const double* s = state + (size_t)e * 10;
    if (!state_in_domain(s, p.max_rounds)) {
        atomicOr(p.serve_overrun, 4);
        return;
    }
    Game g = load_game(p, e);
    g.ball_x = (int)s[0]; g.ball_y = (int)s[1]; g.vx = s[2]; g.vy = s[3]; g.left_y = (int)s[4]; g.right_y = (int)s[5];
    g.score_left = (int)s[6]; g.score_right = (int)s[7]; g.num_rounds = (int)s[8]; g.num_steps = (int)s[9];
    store_game(p, e, g);
}

// Synthetic rollout driver: uniform actions in {0,1,2}, Philox keyed by (seed, step).
__global__ void pong_random_actions_kernel(int32_t* actions, int n_values, uint64_t seed, uint64_t step) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;   // one thread per 4 values
    if (i * 4 >= n_values) return;
    uint32_t r[4];
    philox4x32_10((uint32_t)i, 0u, (uint32_t)step, (uint32_t)(step >> 32), (uint32_t)seed, (uint32_t)(seed >> 32), r);
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (i * 4 + k < n_values) actions[i * 4 + k] = (int32_t)(((uint64_t)r[k] * 3u) >> 32);
}

static inline int blocks_for(int n, int t) { return (n + t - 1) / t; }

cudaError_t launch_pong_construct(const PongDev& p, cudaStream_t s) {
    pong_construct_kernel<<<blocks_for(p.n, 128), 128, 0, s>>>(p);
    return cudaGetLastError();
}
cudaError_t launch_pong_reset(const PongDev& p, cudaStream_t s) {
    pong_reset_kernel<<<blocks_for(p.n, 128), 128, 0, s>>>(p);
    return cudaGetLastError();
}
cudaError_t launch_pong_step(const PongDev& p, const int32_t* actions, float* rew, uint8_t* done, int32_t* num_steps,
                             float* real_reward, cudaStream_t s) {
    pong_step_kernel<<<blocks_for(p.n, 128), 128, 0, s>>>(p, actions, rew, done, num_steps, real_reward);
    return cudaGetLastError();
}
cudaError_t launch_pong_get_state(const PongDev& p, double* state, cudaStream_t s) {
    pong_get_state_kernel<<<blocks_for(p.n, 128), 128, 0, s>>>(p, state);
    return cudaGetLastError();
}
cudaError_t launch_pong_set_state(const PongDev& p, const double* state, cudaStream_t s) {
    pong_set_state_kernel<<<blocks_for(p.n, 128), 128, 0, s>>>(p, state);
    return cudaGetLastError();
}
cudaError_t launch_pong_random_actions(int32_t* actions, int n_values, uint64_t seed, uint64_t step, cudaStream_t s) {
    pong_random_actions_kernel<<<blocks_for((n_values + 3) / 4, 128), 128, 0, s>>>(actions, n_values, seed, step);
    return cudaGetLastError();
}

}  // namespace crl
