// pong_raster.cu -- frame rasteriser fused with the atari_wrappers preprocessing.
//
// Replaces, in ONE kernel and without ever materialising a 210x160x3 frame
// (paths relative to /root/reference/competitive_rl/):
//   _get_screen_img / _get_screen_img_double_player   pong/base_pong_env.py:66-74, 149-155
//   Arena.draw, Ball.draw, Bat.draw, Scoreboard.draw   pong/base_pong_env.py:278-280, 322-323, 406-410, 480-487
//   MaxAndSkipEnv max over the two buffered frames     utils/atari_wrappers.py:153-156
//   WarpFrame: cv2.cvtColor(RGB2GRAY) + cv2.resize(INTER_AREA)   utils/atari_wrappers.py:215-219
//   FrameStack._get_ob + WrapPyTorch (CHW, oldest first)         utils/atari_wrappers.py:257-259, 35-37
//
// Arithmetic restated from cv2 4.13 (SURVEY.md A.1/A.2, pinned in tests/test_oracle_cv2.py):
//   gray  = (R*9798 + G*19235 + B*3735 + 16384) >> 15
//   area  = per source row: buf = sum_t fl(fl(S)*alpha_t) (ascending sx, un-fused);
//           rows: sum = fl(beta_0*buf_0), then sum = fl(sum + fl(beta_k*buf_k));
//           dst = saturate_u8(rint_half_even(sum)).   __fmul_rn/__fadd_rn keep it un-fused.
//
// Structure exploited: a Pong frame is white border + black arena + <=3 white
// rectangles + the scoreboard text above the arena.  So the preprocessed frame is
//   * rows above the arena: a function of the score pair(s) only -> looked up from a
//     table built once per atlas (pong_build_tables_kernel),
//   * everything else: a constant template, except the few destination pixels whose
//     3x3 (5x5 at 42x42) source footprint touches a rectangle -> evaluated exactly.
// Each warp stages one frame in shared memory (template fill, pixel patches), then
// streams it out with coalesced 16-byte stores.
#include "pong_raster_dev.cuh"

namespace crl {

// ---------------------------------------------------------------------------------
// Table builder: text_tab[(pair*3+kind)*2+agent][text_stride] and tmpl[dim*dim (+pad)].
// kind 0: both frames show `pair`; 1: the other frame shows (l+1, r); 2: (l, r+1).
__global__ void pong_build_tables_kernel(PongDev p, uint8_t* text_tab, uint8_t* tmpl, int tmpl_bytes) {
    const int dd = p.dim * p.dim;
    const int entries = ATLAS_SCORES * ATLAS_SCORES * 3 * 2;
    const long long total = (long long)entries * p.text_stride + tmpl_bytes;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        FrameCtx c;
#pragma unroll
        for (int k = 0; k < 6; ++k) c.rect[k] = 0u;
        c.any_valid = true;
        c.blank = false;
        int pix;
        uint8_t* dst;
        if (i < (long long)entries * p.text_stride) {
            const int entry = (int)(i / p.text_stride);
            pix = (int)(i % p.text_stride);
            const int agent = entry & 1, kind = (entry >> 1) % 3, pair = (entry >> 1) / 3;
            int l = pair / ATLAS_SCORES, r = pair % ATLAS_SCORES;
            c.pairA = pair;
            if (kind == 1 && l + 1 < ATLAS_SCORES) l += 1;
            if (kind == 2 && r + 1 < ATLAS_SCORES) r += 1;
            c.pairB = l * ATLAS_SCORES + r;
            c.mirror = agent != 0;
            dst = text_tab + i;
        } else {
            pix = (int)(i - (long long)entries * p.text_stride);
            c.pairA = c.pairB = 0;
            c.mirror = false;
            dst = tmpl + pix;
        }
        *dst = (pix < dd) ? eval_pixel(p.tabs, c, p.atlas, pix / p.dim, pix % p.dim) : (uint8_t)0;
    }
}

// ---------------------------------------------------------------------------------
// Reference rasteriser: one thread per destination pixel, no tables, no shortcuts.
// Used for terminal observations (rare) and as the in-library cross-check of the
// fast kernel (tests/test_gpu_pong_parity.py).
__global__ void pong_raster_generic_kernel(PongDev p, const FrameSpec* __restrict__ hist,
                                           const uint8_t* __restrict__ only_done, int ring, uint8_t* obs0, uint8_t* obs1) {
    const int dd = p.dim * p.dim;
    // ring: every slot j of the 2c-slot ring is rewritten with the frame it must hold, hist[(j - ring_phase - 1) mod c]
    const int slots = ring ? 2 * p.c : p.c;
    const long long total = (long long)p.n * p.n_agents * slots * dd;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int pix = (int)(i % dd);
        long long f = i / dd;
        const int pos = (int)(f % slots);
        f /= slots;
        const int env = (int)(f % p.n), agent = (int)(f / p.n);
        if (only_done != nullptr && !only_done[env]) continue;
        const int slot = ring ? ((pos - p.ring_phase - 1) % p.c + p.c) % p.c : pos;
        const FrameCtx c = make_ctx(hist[(size_t)slot * p.n + env], agent);
        uint8_t* out = (agent ? obs1 : obs0) + ((size_t)env * slots + pos) * dd;
        out[pix] = c.any_valid ? eval_pixel(p.tabs, c, p.atlas, pix / p.dim, pix % p.dim) : (uint8_t)0;
    }
}

// ---------------------------------------------------------------------------------
// float32 observations, as a stock gym install produces them (SURVEY.md F7): Box without a dtype is float32
// (pong/base_pong_env.py:22-24), so MaxAndSkipEnv pools float32 frames (utils/atari_wrappers.py:106-115) and WarpFrame's
// cv2 calls take their float paths: the observation is the UNROUNDED fp32 area sum.  The exception are frames that come
// from reset(): MaxAndSkipEnv.reset passes the raw uint8 array through un-pooled (:162-163), so those go through the
// uint8 path and enter the float32 stack as rounded integers (frame spec bit 17).  One thread per destination pixel.
__global__ void pong_raster_f32_kernel(PongDev p, const FrameSpec* __restrict__ hist, const uint8_t* __restrict__ only_done,
                                       float* obs0, float* obs1) {
    const int dd = p.dim * p.dim;
    const long long total = (long long)p.n * p.n_agents * p.c * dd;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int pix = (int)(i % dd);
        long long f = i / dd;
        const int slot = (int)(f % p.c);
        f /= p.c;
        const int env = (int)(f % p.n), agent = (int)(f / p.n);
        if (only_done != nullptr && !only_done[env]) continue;
        const FrameSpec spec = hist[(size_t)slot * p.n + env];
        const FrameCtx c = make_ctx(spec, agent);
        float v = 0.f;
        if (c.any_valid) {
            if ((spec.y >> 17) & 1u) v = (float)eval_pixel(p.tabs, c, p.atlas, pix / p.dim, pix % p.dim);
            else v = eval_pixel_sum<true>(p.tabs, c, p.atlas, pix / p.dim, pix % p.dim);
        }
        ((agent ? obs1 : obs0) + ((size_t)env * p.c + slot) * dd)[pix] = v;
    }
}

// ---------------------------------------------------------------------------------
// Raw 210x160x3 export of one env's CURRENT game state (VecEnv.render / get_images,
// utils/base_vec_env.py:189-216).  Not on the step path.
__global__ void pong_raw_frame_kernel(PongDev p, int env, uint8_t* rgb0, uint8_t* rgb1) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= SCREEN_W * SCREEN_H) return;
    const int y = i / SCREEN_W, x = i % SCREEN_W;
    const int32_t b = p.ball[env], t = p.bats[env], s = p.score[env];
    const int bx = (int16_t)(b & 0xffff), by = (int16_t)(b >> 16), ly = t & 0xffff, ry = (t >> 16) & 0xffff;
    const int pair = (s & 0xff) * ATLAS_SCORES + ((s >> 8) & 0xff);
    uint8_t r, g, bl;
    if (y < ATLAS_ROWS && !scores_in_atlas((uint32_t)s, (uint32_t)s)) {
        r = g = bl = 255;   // a score past 21: no text
    } else if (y < ATLAS_ROWS) {
        const uint8_t* a = p.atlas + ((size_t)(pair * ATLAS_ROWS + y) * SCREEN_W + x) * 3;
        r = a[0]; g = a[1]; bl = a[2];
    } else if (y >= ARENA_BOTTOM) {
        r = g = bl = 255;
    } else {
        const bool w = (x >= bx && x < bx + BALL_SIZE && y >= by && y < by + BALL_SIZE) ||
                       (x >= LEFT_BAT_X && x < LEFT_BAT_X + BAT_W && y >= ly && y < ly + BAT_H) ||
                       (x >= RIGHT_BAT_X && x < RIGHT_BAT_X + BAT_W && y >= ry && y < ry + BAT_H);
        r = g = bl = w ? 255 : 0;
    }
    uint8_t* o0 = rgb0 + (size_t)i * 3;
    o0[0] = r; o0[1] = g; o0[2] = bl;
    if (rgb1 != nullptr) {
        const int xm = (y >= MIRROR_ROW) ? SCREEN_W - 1 - x : x;
        uint8_t* o1 = rgb1 + ((size_t)y * SCREEN_W + xm) * 3;
        o1[0] = r; o1[1] = g; o1[2] = bl;
    }
}

// ---------------------------------------------------------------------------------
static inline int frame_smem_bytes(const PongDev& p) { return ((p.dim * p.dim + 15) / 16) * 16; }

cudaError_t launch_pong_build_tables(const PongDev& p, uint8_t* text_tab, uint8_t* tmpl, cudaStream_t s) {
    pong_build_tables_kernel<<<148 * 8, 256, 0, s>>>(p, text_tab, tmpl, frame_smem_bytes(p));
    return cudaGetLastError();
}

cudaError_t launch_pong_raster_generic(const PongDev& p, const FrameSpec* hist, const uint8_t* only_done, int ring,
                                       uint8_t* obs0, uint8_t* obs1, cudaStream_t s) {
    pong_raster_generic_kernel<<<148 * 16, 256, 0, s>>>(p, hist, only_done, ring, obs0, obs1);
    return cudaGetLastError();
}

cudaError_t launch_pong_raster_f32(const PongDev& p, const FrameSpec* hist, const uint8_t* only_done, float* obs0, float* obs1,
                                   cudaStream_t s) {
    pong_raster_f32_kernel<<<148 * 16, 256, 0, s>>>(p, hist, only_done, obs0, obs1);
    return cudaGetLastError();
}

cudaError_t launch_pong_raw_frame(const PongDev& p, int env, uint8_t* rgb0, uint8_t* rgb1, cudaStream_t s) {
    pong_raw_frame_kernel<<<(SCREEN_W * SCREEN_H + 255) / 256, 256, 0, s>>>(p, env, rgb0, rgb1);
    return cudaGetLastError();
}

}  // namespace crl
