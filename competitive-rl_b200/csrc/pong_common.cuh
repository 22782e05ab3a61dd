// pong_common.cuh -- device-side data layout shared by the Pong kernels (sm_100a).
//
// Reference path being replaced (paths relative to /root/reference/competitive_rl/):
//   pong/base_pong_env.py      game core + 210x160x3 renderer
//   utils/atari_wrappers.py    MaxAndSkipEnv / WarpFrame / ClipRewardEnv / FrameStack / WrapPyTorch
//   utils/dummy_vec_env.py     batch loop + auto-reset
//
// HBM layout: every per-env quantity is a structure-of-arrays column of N
// elements, so one-thread-per-env kernels read and write fully coalesced.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace crl {

// ---- geometry: PongGame.__init__, pong/base_pong_env.py:158-211 with the env ctor
// arguments of :27-36 (window 160x210, ball_speed = bat_speed = 4) ----
constexpr int SCREEN_W = 160;
constexpr int SCREEN_H = 210;
constexpr int ARENA_TOP = 34;
constexpr int ARENA_BOTTOM = 194;  // Rect(0, 34, 160, 160): height = window WIDTH (:275-276)
constexpr int ARENA_CENTERY = 114;
constexpr int BALL_SIZE = 4;
constexpr int BALL_X0 = 78;
constexpr int BALL_Y0 = 112;
constexpr int BAT_W = 5;
constexpr int BAT_H = 15;
constexpr int BAT_Y0 = 107;
constexpr int LEFT_BAT_X = 16;
constexpr int RIGHT_BAT_X = 139;
constexpr int SPEED = 4;
constexpr int MAX_STEP_PER_ROUND = 10000;
constexpr int CHEAT_CODES = 999;   // pong/base_pong_env.py:9
constexpr int MIRROR_ROW = 25;     // new_flip[25:] = new_flip[25:, ::-1], :153-154
constexpr int ATLAS_ROWS = 34;     // frame rows above the arena
constexpr int ATLAS_SCORES = 22;
constexpr int MAX_TAPS = 5;        // 160->42: <=5 horizontal taps, 210->42: 5 vertical taps
constexpr int MAX_DIM = 84;
constexpr int MAX_STACK = 8;

// What one rendered game frame depends on: 8 bytes.
//   x: ball_x | ball_y<<8 | left_y<<16 | right_y<<24
//   y: score_left | score_right<<8 | valid<<16   (valid=0: the np.zeros MaxAndSkip buffer)
//      | raw<<17 (the frame reset() returned: it bypasses MaxAndSkipEnv's buffers; only the float32 mode cares)
typedef uint2 RenderState;

// One preprocessed observation frame = max of two rendered frames (MaxAndSkipEnv
// slots 0/1, utils/atari_wrappers.py:136-156) = 16 bytes: (A.x, A.y, B.x, B.y).
typedef uint4 FrameSpec;

__host__ __device__ inline RenderState make_render_state(int bx, int by, int ly, int ry, int sl, int sr) {
    RenderState r;
    r.x = (uint32_t)(bx & 255) | ((uint32_t)(by & 255) << 8) | ((uint32_t)(ly & 255) << 16) | ((uint32_t)(ry & 255) << 24);
    r.y = (uint32_t)(sl & 255) | ((uint32_t)(sr & 255) << 8) | (1u << 16);
    return r;
}

// cv2 INTER_AREA tap tables (OpenCV computeResizeAreaTab; SURVEY.md A.2). Taps of one
// destination index are contiguous source indices src0 .. src0+n-1.
struct AreaTabs {
    int dim;
    int text_rows;                 // dst rows touching src rows < ARENA_TOP
    uint8_t x_src0[MAX_DIM], x_n[MAX_DIM];
    uint8_t y_src0[MAX_DIM], y_n[MAX_DIM];
    float x_a[MAX_DIM][MAX_TAPS];  // alpha (fp32, as cv2 stores them)
    float x_pa[MAX_DIM][MAX_TAPS]; // fl(255 * alpha): one white source pixel's contribution
    float y_b[MAX_DIM][MAX_TAPS];
    uint8_t x_first[SCREEN_W], x_last[SCREEN_W];  // first/last dst column whose taps include src col
    uint8_t y_first[SCREEN_H], y_last[SCREEN_H];
};

// Device-resident state of one vectorised Pong env (all pointers are device memory).
struct PongDev {
    int n;              // envs on this device
    int n_agents;       // 1 = cPong-v0 (AutoBat on the right), 2 = cPongDouble-v0
    int dim;            // resized_dim
    int c;              // frames per observation (frame_stack or 1)
    int max_rounds;
    // stack_mode 1: the observation buffers are double-write rings [n][2c][dim][dim]: the newest frame goes to slots
    // ring_phase and ring_phase + c, the observation is the strided view of slots ring_phase + 1 .. ring_phase + c
    // (oldest -> newest), so a step writes 2 frames per agent instead of c.  Slot j holds hist[(j - ring_phase - 1) mod c].
    int ring;
    int ring_phase;     // slot the newest frame was written to by the current step (host-tracked, advanced per step)
    int fill_all;       // 1 after reset(): every env's ring is rewritten completely by the next render
    int zero_on_done;   // FrameStackTensor semantics (utils/utils.py:145-173): a reset clears the history to zero frames
                        // instead of filling it with copies of the reset frame (FrameStack.reset)
    int64_t first_env;  // global index of env 0 (RNG streams are keyed by global index)
    uint64_t seed;
    // --- game state (PongGame fields) ---
    int32_t* ball;       // x | y<<16
    double* vx;
    double* vy;
    int32_t* bats;       // left_y | right_y<<16
    int32_t* score;      // score_left | score_right<<8 | num_rounds<<16
    int32_t* num_steps;  // PongGame._num_steps
    int32_t* clip_steps; // ClipRewardEnv._steps
    int32_t* serve_count;
    uint8_t* last_done;     // [n] done flag of the last step (ring mode: these envs' rings are rewritten completely)
    RenderState* skipbuf;   // [2][n]  MaxAndSkipEnv._obs_buffer as render states
    FrameSpec* hist;        // [c][n]  FrameStack deque, slot 0 = oldest
    FrameSpec* term_hist;   // [c][n]  deque at the terminal step (for terminal_observation)
    // --- validation mode: injected serves ---
    const double* serves;   // [n][K][2] (vx, vy) or nullptr
    int serves_k;
    int32_t* serve_overrun; // device flag
    // episode statistics, accumulated on done: [0] episodes, [1] sum of episode lengths (env-steps),
    // [2] left wins, [3] right wins, [4] draws, [5] sum of (score_left - score_right) + 64*episodes
    unsigned long long* stats;
    // next (env, agent) stack the rasteriser's warps take (zeroed before every launch): the GPU as a whole sweeps the
    // observation buffers front to back, which the DRAM write path sustains ~16 % better than a static grid stride
    unsigned long long* work_counter;
    // --- renderer data ---
    const AreaTabs* tabs;
    const uint8_t* atlas;      // [22][22][34][160][3] RGB
    const uint8_t* text_tab;   // [22*22*3][2 agents][text_stride] preprocessed rows above the arena
    const uint8_t* tmpl;       // [dim*dim (+pad)] rect-free frame (score 0:0)
    int text_stride;           // bytes per text_tab entry (multiple of 16)
    int text_w0, text_w1;      // 32-bit words [w0, w1) of an entry that differ between entries or from tmpl (host scan after the tables
                               // are built; until then the whole entry): all the 42x42 quad kernel copies on a score change
    const void* fast_tabs;     // FastTabs<dim> image for the hot kernel (nullptr: dim not specialised)
    int fast_ok;               // atlas rows sharing a dst row with the arena are pure white
    int raster_grid[3];        // persistent grids of the hot kernels on this handle's device: [0] 84x84, [1] 42x42 one frame
                               // per warp, [2] 42x42 four frames per warp
    int quad_ok;               // the 42x42 geometry the four-frames-per-warp kernel relies on holds
};

// ---- Philox4x32-10 (counter-based; streams keyed by seed and global env index) ----
__host__ __device__ inline void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4]) {
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// host-side launchers (defined in the .cu files)
cudaError_t launch_pong_construct(const PongDev& p, cudaStream_t s);
cudaError_t launch_pong_reset(const PongDev& p, cudaStream_t s);
cudaError_t launch_pong_step(const PongDev& p, const int32_t* actions, float* rew, uint8_t* done, int32_t* num_steps,
                             float* real_reward, cudaStream_t s);
cudaError_t launch_pong_get_state(const PongDev& p, double* state, cudaStream_t s);
cudaError_t launch_pong_set_state(const PongDev& p, const double* state, cudaStream_t s);
cudaError_t launch_pong_random_actions(int32_t* actions, int n_values, uint64_t seed, uint64_t step, cudaStream_t s);

cudaError_t launch_pong_build_tables(const PongDev& p, uint8_t* text_tab, uint8_t* tmpl, cudaStream_t s);
// shown != nullptr: incremental 84x84 stack render (pong_raster_incremental_ok must hold): obs* hold the frames shown
// ([agent][c][n]) describes; afterwards shown = hist
cudaError_t launch_pong_raster(const PongDev& p, const FrameSpec* hist, uint8_t* obs0, uint8_t* obs1, FrameSpec* shown,
                               cudaStream_t s);
bool pong_raster_incremental_ok(const PongDev& p, const void* obs0, const void* obs1);
// ring = 1: obs* are 2c-slot rings, rewritten completely (terminal observations are always plain stacks: ring = 0)
cudaError_t launch_pong_raster_generic(const PongDev& p, const FrameSpec* hist, const uint8_t* only_done, int ring,
                                       uint8_t* obs0, uint8_t* obs1, cudaStream_t s);
cudaError_t launch_pong_raster_f32(const PongDev& p, const FrameSpec* hist, const uint8_t* only_done, float* obs0, float* obs1,
                                   cudaStream_t s);
cudaError_t pong_raster_init(int grid_out[3]);
bool pong_quad_ok(const AreaTabs& a);
size_t pong_fast_tabs_bytes(int dim);
bool pong_fast_tabs_fill(const AreaTabs& a, int text_stride, void* host_buf);   // false: geometry not supported
cudaError_t launch_pong_build_bat_lut(int dim, void* fast_tabs_dev, cudaStream_t s);
cudaError_t launch_pong_raw_frame(const PongDev& p, int env, uint8_t* rgb0, uint8_t* rgb1, cudaStream_t s);

}  // namespace crl
