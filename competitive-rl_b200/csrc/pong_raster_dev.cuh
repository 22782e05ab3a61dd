// pong_raster_dev.cuh -- device helpers shared by the rasteriser kernels: the analytic
// description of a max-pooled Pong frame and the exact per-pixel evaluator.
#pragma once
#include "pong_common.cuh"

namespace crl {

// ---------------------------------------------------------------------------------
// Per-frame context: what the two max-pooled rendered frames contain, in the
// viewing agent's coordinates (agent 1 sees rows >= 25 mirrored in x).
struct FrameCtx {
    uint32_t rect[6];   // x0 | x1<<8 | y0<<16 | y1<<24 (arena-clipped; 0 = empty)
    int pairA, pairB;   // atlas score-pair index l*22+r of the two frames
    bool blank;         // a frame's score pair is outside the atlas: the rows above the arena are white (no text)
    bool mirror;
    bool any_valid;
};

__device__ __forceinline__ uint32_t pack_rect(int x0, int x1, int y0, int y1, bool mirror) {
    x0 = max(x0, 0); x1 = min(x1, SCREEN_W);
    y0 = max(y0, ARENA_TOP); y1 = min(y1, ARENA_BOTTOM);   // white-on-white outside the arena
    if (x1 <= x0 || y1 <= y0) return 0u;
    if (mirror) { const int t = SCREEN_W - x1; x1 = SCREEN_W - x0; x0 = t; }
    return (uint32_t)x0 | ((uint32_t)x1 << 8) | ((uint32_t)y0 << 16) | ((uint32_t)y1 << 24);
}

__device__ __forceinline__ FrameCtx make_ctx(const FrameSpec f, const int agent) {
    FrameCtx c;
    uint32_t ax = f.x, ay = f.y, bx = f.z, by = f.w;
    const bool va = (ay >> 16) & 1u, vb = (by >> 16) & 1u;
    c.any_valid = va || vb;
    c.mirror = agent != 0;
    if (!va) { ax = bx; ay = by; }      // max(0-frame, X) = X
    if (!vb) { bx = ax; by = ay; }
    c.blank = !scores_in_atlas(ay, by);
    c.pairA = c.blank ? 0 : (int)(ay & 255u) * ATLAS_SCORES + (int)((ay >> 8) & 255u);
    c.pairB = c.blank ? 0 : (int)(by & 255u) * ATLAS_SCORES + (int)((by >> 8) & 255u);
    {
        const int x = ax & 255u, y = (ax >> 8) & 255u, l = (ax >> 16) & 255u, r = (ax >> 24) & 255u;
        c.rect[0] = pack_rect(x, x + BALL_SIZE, y, y + BALL_SIZE, c.mirror);
        c.rect[1] = pack_rect(LEFT_BAT_X, LEFT_BAT_X + BAT_W, l, l + BAT_H, c.mirror);
        c.rect[2] = pack_rect(RIGHT_BAT_X, RIGHT_BAT_X + BAT_W, r, r + BAT_H, c.mirror);
    }
    if (ax == bx) {
        c.rect[3] = c.rect[4] = c.rect[5] = 0u;
    } else {
        const int x = bx & 255u, y = (bx >> 8) & 255u, l = (bx >> 16) & 255u, r = (bx >> 24) & 255u;
        c.rect[3] = pack_rect(x, x + BALL_SIZE, y, y + BALL_SIZE, c.mirror);
        c.rect[4] = pack_rect(LEFT_BAT_X, LEFT_BAT_X + BAT_W, l, l + BAT_H, c.mirror);
        c.rect[5] = pack_rect(RIGHT_BAT_X, RIGHT_BAT_X + BAT_W, r, r + BAT_H, c.mirror);
    }
    return c;
}

// bit t set <=> lo <= s0 + t < hi, for t in [0, n)
__device__ __forceinline__ uint32_t span_bits(int lo, int hi, int s0, int n) {
    const int a = max(lo - s0, 0), b = min(hi - s0, n);
    return (b > a) ? (((1u << b) - 1u) & ~((1u << a) - 1u)) : 0u;
}

// gray value of the max-pooled source pixel in the rows above the arena
__device__ __forceinline__ int text_gray(const FrameCtx& c, const uint8_t* __restrict__ atlas, int sy, int sx) {
    if (c.blank) return 255;   // max(white, X) = white; gray(255, 255, 255) = 255
    const int ax = (c.mirror && sy >= MIRROR_ROW) ? (SCREEN_W - 1 - sx) : sx;
    const uint8_t* pa = atlas + ((size_t)(c.pairA * ATLAS_ROWS + sy) * SCREEN_W + ax) * 3;
    const uint8_t* pb = atlas + ((size_t)(c.pairB * ATLAS_ROWS + sy) * SCREEN_W + ax) * 3;
    const int r = max((int)pa[0], (int)pb[0]), g = max((int)pa[1], (int)pb[1]), b = max((int)pa[2], (int)pb[2]);
    return (r * 9798 + g * 19235 + b * 3735 + 16384) >> 15;   // cv2 RGB2GRAY, 15-bit fixed point
}

// the same pixel as cv2.cvtColor(float32 RGB -> GRAY) computes it (stock gym: float32 observation buffers, SURVEY.md F7):
// fma(B, 0.114f, fma(R, 0.299f, G * 0.587f)) in fp32 -- pinned against cv2 4.13 on random and Pong-like images
// (tests/test_oracle_cv2.py); pure white gives exactly 255.0f, so only the antialiased text pixels differ from text_gray
__device__ __forceinline__ float text_gray_f32(const FrameCtx& c, const uint8_t* __restrict__ atlas, int sy, int sx) {
    if (c.blank) return 255.f;
    const int ax = (c.mirror && sy >= MIRROR_ROW) ? (SCREEN_W - 1 - sx) : sx;
    const uint8_t* pa = atlas + ((size_t)(c.pairA * ATLAS_ROWS + sy) * SCREEN_W + ax) * 3;
    const uint8_t* pb = atlas + ((size_t)(c.pairB * ATLAS_ROWS + sy) * SCREEN_W + ax) * 3;
    const float r = (float)max((int)pa[0], (int)pb[0]), g = (float)max((int)pa[1], (int)pb[1]), b = (float)max((int)pa[2], (int)pb[2]);
    return __fmaf_rn(b, 0.114f, __fmaf_rn(r, 0.299f, __fmul_rn(g, 0.587f)));
}

// Value of destination pixel (dy, dx) before rounding: cv2's INTER_AREA float sequence evaluated on the
// analytically-described source frame.  FLOAT_GRAY: the gray conversion of the float32 path (see text_gray_f32).
template <bool FLOAT_GRAY>
__device__ __forceinline__ float eval_pixel_sum(const AreaTabs* __restrict__ T, const FrameCtx& c,
                                                const uint8_t* __restrict__ atlas, int dy, int dx) {
    const int sx0 = T->x_src0[dx], nx = T->x_n[dx];
    const int sy0 = T->y_src0[dy], ny = T->y_n[dy];
    uint32_t hp[6], vp[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const uint32_t r = c.rect[k];
        hp[k] = span_bits(r & 255u, (r >> 8) & 255u, sx0, nx);
        vp[k] = span_bits((r >> 16) & 255u, r >> 24, sy0, ny);
    }
    float sum = 0.f;
#pragma unroll 1
    for (int ty = 0; ty < ny; ++ty) {
        const int sy = sy0 + ty;
        float buf = 0.f;
        if (sy < ARENA_TOP) {
            for (int tx = 0; tx < nx; ++tx) {
                const float gv = FLOAT_GRAY ? text_gray_f32(c, atlas, sy, sx0 + tx) : (float)text_gray(c, atlas, sy, sx0 + tx);
                buf = __fadd_rn(buf, __fmul_rn(gv, T->x_a[dx][tx]));
            }
        } else {
            uint32_t pat = 0u;
            if (sy >= ARENA_BOTTOM) {
                pat = 0xffffffffu;
            } else {
#pragma unroll
                for (int k = 0; k < 6; ++k) pat |= ((vp[k] >> ty) & 1u) ? hp[k] : 0u;
            }
#pragma unroll
            for (int tx = 0; tx < MAX_TAPS; ++tx)
                if (tx < nx && ((pat >> tx) & 1u)) buf = __fadd_rn(buf, T->x_pa[dx][tx]);
        }
        const float term = __fmul_rn(T->y_b[dy][ty], buf);
        sum = (ty == 0) ? term : __fadd_rn(sum, term);
    }
    return sum;
}

// uint8 observation: saturate_cast<uchar>(cvRound(sum)), round half to even
__device__ __forceinline__ uint8_t eval_pixel(const AreaTabs* __restrict__ T, const FrameCtx& c,
                                              const uint8_t* __restrict__ atlas, int dy, int dx) {
    const int v = __float2int_rn(eval_pixel_sum<false>(T, c, atlas, dy, dx));
    return (uint8_t)min(max(v, 0), 255);
}

}  // namespace crl
