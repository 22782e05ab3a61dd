// pong_raster_fast.cu -- the hot kernel: frame rasteriser fused with max-pool, gray,
// INTER_AREA resize, FrameStack and CHW layout, one warp per (env, agent) observation stack.
//
// Replaces (paths relative to /root/reference/competitive_rl/): the renderer
// pong/base_pong_env.py:66-74,149-155,278-280,322-323,406-410,480-487; MaxAndSkipEnv's max
// utils/atari_wrappers.py:153-156; WarpFrame :215-219; FrameStack._get_ob :257-259;
// WrapPyTorch :35-37.  Arithmetic: see pong_raster.cu's header (cv2 4.13 restated).
//
// Shape of the work (84x84): a preprocessed frame is 7 056 bytes of which ~100 depend on
// the ball and bats; the rest is the scoreboard rows (table lookup by score pair) and a
// constant template.  Each warp keeps the TEMPLATE resident in its shared-memory frame
// buffer and, per frame,
//   A. computes in registers what differs from the template:
//        - bat columns: a bat always covers the same source columns, so a destination row of
//          the 4-column bat strip is a pure function of (row, which of its vertical taps are
//          inside a bat) -> one 32-bit LUT word per row, one lane per row;
//        - ball: the <=4x4 destination pixels of each of the two pooled ball positions are
//          evaluated exactly (cv2's un-fused fp32 order), one pixel per lane, taking nearby
//          bats into account;
//        - the scoreboard rows for this frame's score pair(s) (only when they changed);
//   B. waits until the TMA engine has finished READING the previous frame out of the buffer,
//      restores the bytes that frame had patched, writes this frame's patches,
//   C. hands the buffer to the TMA engine: one cp.async.bulk shared->global of 7 056 bytes
//      (fence.proxy.async first), so the drain costs one instruction and overlaps step A of
//      the next frame.
// HBM traffic = the observation bytes, written once; ~100 B/env of state are read.  Into buffers whose contents the
// library tracks (crl_pong_set_obs_buffers), the incremental instantiation stores only the 16-byte chunks a frame can
// have changed since the buffer's last render (INC below).
// The grid is persistent: SMs x resident CTAs, warps stride over the stacks.
#include <type_traits>

#include "pong_raster_dev.cuh"

namespace crl {

template <int TAPS> struct alignas(16) TapEnt;
template <> struct alignas(16) TapEnt<3> { uint32_t meta; float w[3]; };
template <> struct alignas(16) TapEnt<5> { uint32_t meta; float w[5]; uint32_t pad[2]; };
// meta: src0 | tapmask<<8 | (y only) mask of taps lying in the white border rows <<16

#ifndef CRL_FAST84_CTAS
#define CRL_FAST84_CTAS 3    // resident CTAs per SM of the 84x84 kernel: see pong_raster_init
#endif
// CTAS: resident CTAs per SM the kernel is compiled for (__launch_bounds__) and launched with
template <int DIM> struct FastCfg;
template <> struct FastCfg<84> { static constexpr int TAPS = 3, VEC = 16, CTAS = CRL_FAST84_CTAS; };
template <> struct FastCfg<42> { static constexpr int TAPS = 5, VEC = 4, CTAS = 3; };

constexpr int FAST_WARPS = 8;
constexpr int FIRST_PAD = 224;   // y_first/y_last padded to a multiple of 16 bytes
constexpr int BAT_ROWS = 8;      // destination rows one bat can touch (checked on the host)

template <int DIM> struct alignas(16) FastTabs {
    TapEnt<FastCfg<DIM>::TAPS> xe[DIM], ye[DIM];
    uint32_t bat_lut[2][DIM][1 << FastCfg<DIM>::TAPS];   // [view side][dst row][vertical tap bits] -> 4 pixels
    float xlut[DIM][1 << FastCfg<DIM>::TAPS];            // [dst column][white horizontal taps] -> cv2's row sum (eval_from_pat's buf)
    uint8_t x_first[SCREEN_W], x_last[SCREEN_W], y_first[FIRST_PAD], y_last[FIRST_PAD];
    uint32_t bat_c0[2], pad[2];                           // first of the 4 destination columns per side
};

template <int VEC> struct VecT;
template <> struct VecT<16> { typedef uint4 type; };
template <> struct VecT<4> { typedef uint32_t type; };

__device__ __forceinline__ void st_stream(uint4* ptr, const uint4 v) {
    asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(ptr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}
__device__ __forceinline__ void st_stream(uint32_t* ptr, const uint32_t v) {
    asm volatile("st.global.cs.u32 [%0], %1;" ::"l"(ptr), "r"(v) : "memory");
}

// ---- TMA bulk store (shared::cta -> global), bulk_group completion ----
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s), "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// bits of v (<= 5) moved to positions 0, 6, 12, 18, 24
__device__ __forceinline__ uint32_t spread6(uint32_t v) { return (v * 0x108421u) & 0x1041041u; }

// mask8 = extent mask << 8 of a rect starting at r0; returns which of the taps starting at s0 it covers
__device__ __forceinline__ uint32_t tap_bits(uint32_t mask8, int r0, int s0) {
    const int sh = min(max(8 - (r0 - s0), 0), 31);
    return mask8 >> sh;
}

// cv2 INTER_AREA float sequence for one destination pixel given, per vertical tap t (6-bit
// field t of `pat`), which horizontal taps are white.  X.w = fl(255*alpha), Y.w = beta.
template <int TAPS>
__device__ __forceinline__ uint32_t eval_from_pat(const TapEnt<TAPS>& X, const TapEnt<TAPS>& Y, uint32_t pat) {
    float sum = 0.f;
#pragma unroll
    for (int t = 0; t < TAPS; ++t) {
        const uint32_t pr = pat >> (6 * t);
        float buf = (pr & 1u) ? X.w[0] : 0.f;               // 0 + w == w exactly; absent taps add +0
#pragma unroll
        for (int u = 1; u < TAPS; ++u) buf = __fadd_rn(buf, ((pr >> u) & 1u) ? X.w[u] : 0.f);
        const float term = __fmul_rn(Y.w[t], buf);           // padded taps have weight 0
        sum = (t == 0) ? term : __fadd_rn(sum, term);
    }
    const int v = __float2int_rn(sum);                       // cvRound: half to even
    return (uint32_t)min(max(v, 0), 255);
}

// eval_from_pat with the horizontal sums looked up: xl = T->xlut[dx] holds, for every subset of white horizontal taps, the
// float the sequential additions of eval_from_pat arrive at (built with the same __fadd_rn chain, so bit-identical).
template <int TAPS>
__device__ __forceinline__ uint32_t eval_from_pat_lut(const float* __restrict__ xl, const TapEnt<TAPS>& Y, uint32_t pat) {
    float sum = 0.f;
#pragma unroll
    for (int t = 0; t < TAPS; ++t) {
        const float term = __fmul_rn(Y.w[t], xl[(pat >> (6 * t)) & ((1u << TAPS) - 1u)]);
        sum = (t == 0) ? term : __fadd_rn(sum, term);
    }
    const int v = __float2int_rn(sum);
    return (uint32_t)min(max(v, 0), 255);
}

template <int DIM>
__global__ void pong_build_xlut_kernel(FastTabs<DIM>* T) {
    constexpr int TAPS = FastCfg<DIM>::TAPS, NP = 1 << TAPS;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= DIM * NP) return;
    const int bits = i % NP, dx = i / NP;
    const TapEnt<TAPS> X = T->xe[dx];
    float buf = (bits & 1) ? X.w[0] : 0.f;
    for (int u = 1; u < TAPS; ++u) buf = __fadd_rn(buf, ((bits >> u) & 1) ? X.w[u] : 0.f);
    T->xlut[dx][bits] = buf;
}

// One 4-pixel LUT word per (view side, destination row, vertical tap bits).
template <int DIM>
__global__ void pong_build_bat_lut_kernel(FastTabs<DIM>* T) {
    constexpr int TAPS = FastCfg<DIM>::TAPS, NP = 1 << TAPS;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * DIM * NP) return;
    const int vp = i % NP, dy = (i / NP) % DIM, side = i / (NP * DIM);
    const TapEnt<TAPS> Y = T->ye[dy];
    const uint32_t ymask = (Y.meta >> 8) & 255u;
    uint32_t word = 0u;
    for (int j = 0; j < 4; ++j) {
        const int dx = (int)T->bat_c0[side] + j;
        uint32_t v = 0u;
        if (dx < DIM) {
            const TapEnt<TAPS> X = T->xe[dx];
            const uint32_t xmask = (X.meta >> 8) & 255u;
            const uint32_t hb = tap_bits(((1u << BAT_W) - 1u) << 8, side ? RIGHT_BAT_X : LEFT_BAT_X, X.meta & 255u) & xmask;
            const uint32_t pat = xmask * spread6((Y.meta >> 16) & 255u) | hb * spread6((uint32_t)vp & ymask);
            v = eval_from_pat<TAPS>(X, Y, pat);
        }
        word |= v << (8 * j);
    }
    T->bat_lut[side][dy][vp] = word;
}

// Scoreboard rows for a score combination that is not in text_tab (the two pooled frames differ by
// more than one point, or a score is past 21 (blank: white rows, no text); only reachable through
// crl_pong_set_state): exact evaluation straight from the atlas.  Arena taps count as black here; pixels that
// also see a rectangle are overwritten by the bat/ball patches, which (fast_ok) treat the atlas rows they share
// a destination row with as white.  Reached from game states only with blank: two different in-atlas pairs need a
// history frame pooling buffers more than one point apart, which exists only in terminal observations (generic kernel).
__device__ __forceinline__ uint8_t eval_text_pixel(const AreaTabs* __restrict__ T, const uint8_t* __restrict__ atlas,
                                                   int pairA, int pairB, bool blank, bool mirror, int dy, int dx) {
    const int sx0 = T->x_src0[dx], nx = T->x_n[dx], sy0 = T->y_src0[dy], ny = T->y_n[dy];
    float sum = 0.f;
    for (int ty = 0; ty < ny; ++ty) {
        const int sy = sy0 + ty;
        float buf = 0.f;
        for (int tx = 0; tx < nx; ++tx) {
            int g = 0;
            if (sy < ARENA_TOP && blank) {
                g = 255;
            } else if (sy < ARENA_TOP) {
                const int sx = sx0 + tx;
                const int ax = (mirror && sy >= MIRROR_ROW) ? (SCREEN_W - 1 - sx) : sx;
                const uint8_t* pa = atlas + ((size_t)(pairA * ATLAS_ROWS + sy) * SCREEN_W + ax) * 3;
                const uint8_t* pb = atlas + ((size_t)(pairB * ATLAS_ROWS + sy) * SCREEN_W + ax) * 3;
                g = (max((int)pa[0], (int)pb[0]) * 9798 + max((int)pa[1], (int)pb[1]) * 19235 +
                     max((int)pa[2], (int)pb[2]) * 3735 + 16384) >> 15;
            }
            buf = __fadd_rn(buf, __fmul_rn((float)g, T->x_a[dx][tx]));
        }
        const float term = __fmul_rn(T->y_b[dy][ty], buf);
        sum = (ty == 0) ? term : __fadd_rn(sum, term);
    }
    return (uint8_t)min(max(__float2int_rn(sum), 0), 255);
}

// ---- incremental stacks (INC): what a frame buffer already holds decides what is stored ----
// (env, agent) stacks per work ticket of the incremental kernel: its stacks store ~1/20 of the bytes, so one atomic per
// stack would make the counter a bottleneck
#ifndef CRL_INC_TICKET
#define CRL_INC_TICKET 4
#endif

__device__ __forceinline__ uint32_t spec_diff(const FrameSpec& a, const FrameSpec& b) {
    const uint32_t nr = ~(1u << 17);   // the raw bit only matters to the float32 mode
    return (a.x ^ b.x) | ((a.y ^ b.y) & nr) | (a.z ^ b.z) | ((a.w ^ b.w) & nr);
}

// scoreboard entry of a frame (the kernel's text_id), -2 when its score combination is outside text_tab (also: a score
// past the atlas); any_valid = 0: the all-zero frame
__device__ __forceinline__ int frame_text_id(FrameSpec f, int agent, bool& any_valid) {
    const bool va = (f.y >> 16) & 1u, vb = (f.w >> 16) & 1u;
    any_valid = va || vb;
    if (!va) f.y = f.w;
    if (!vb) f.w = f.y;
    if (!scores_in_atlas(f.y, f.w)) return -2;
    const int pairA = (int)(f.y & 255u) * ATLAS_SCORES + (int)((f.y >> 8) & 255u);
    const int pairB = (int)(f.w & 255u) * ATLAS_SCORES + (int)((f.w >> 8) & 255u);
    int base = pairA, kind = 0;
    if (pairA != pairB) {
        const int d = pairB - pairA;
        if (d == ATLAS_SCORES) kind = 1;
        else if (d == 1 && (pairA % ATLAS_SCORES) != ATLAS_SCORES - 1) kind = 2;
        else if (d == -ATLAS_SCORES) { base = pairB; kind = 1; }
        else if (d == -1 && (pairB % ATLAS_SCORES) != ATLAS_SCORES - 1) { base = pairB; kind = 2; }
        else return -2;
    }
    return (base * 3 + kind) * 2 + agent;
}

// Byte offsets of the bat word and the ball pixel this lane patches for frame f (-1: none): the offset arithmetic of phases
// A2 / A3 of pong_raster_fast_kernel, without the pixel values.  For a frame that has valid render states.
template <int DIM>
__device__ __forceinline__ void frame_patch_offsets(const FastTabs<DIM>* T, FrameSpec f, int agent, int lane, int& bat_off,
                                                    int& ball_off) {
    const int cL = (int)T->bat_c0[0], cR = (int)T->bat_c0[1];
    const int b_side = lane >> 4, b_which = (lane >> 3) & 1, b_row = lane & 7;
    const int p_which = lane >> 4, p_col = lane & 3, p_row = (lane >> 2) & 3;
    if (!((f.y >> 16) & 1u)) { f.x = f.z; f.y = f.w; }
    if (!((f.w >> 16) & 1u)) { f.z = f.x; f.w = f.y; }
    const bool same = (f.x == f.z);
    const int lyA = (f.x >> 16) & 255u, ryA = f.x >> 24, lyB = (f.z >> 16) & 255u, ryB = f.z >> 24;
    const int vlA = agent ? ryA : lyA, vrA = agent ? lyA : ryA;
    const int vlB = agent ? ryB : lyB, vrB = agent ? lyB : ryB;
    bat_off = -1;
    {
        const int y0 = b_which ? (b_side ? vrB : vlB) : (b_side ? vrA : vlA);
        const int c0 = max(y0, ARENA_TOP), c1 = min(y0 + BAT_H, ARENA_BOTTOM);
        if (c1 > c0 && !(b_which && same)) {
            const int dy = (int)T->y_first[c0] + b_row;
            if (dy <= (int)T->y_last[c1 - 1]) bat_off = dy * DIM + (b_side ? cR : cL);
        }
    }
    ball_off = -1;
    {
        const FrameSpec& g = f;
        const uint32_t bx = p_which ? g.z : g.x;
        int x0 = bx & 255u, x1 = min(x0 + BALL_SIZE, SCREEN_W);
        int y0 = (bx >> 8) & 255u, y1 = min(y0 + BALL_SIZE, ARENA_BOTTOM);
        y0 = max(y0, ARENA_TOP);
        if (agent) { const int t = SCREEN_W - x1; x1 = SCREEN_W - x0; x0 = t; }
        if (x1 > x0 && y1 > y0 && !(p_which && same)) {
            const int dx = (int)T->x_first[x0] + p_col, dy = (int)T->y_first[y0] + p_row;
            if (dx <= (int)T->x_last[x1 - 1] && dy <= (int)T->y_last[y1 - 1]) ball_off = dy * DIM + dx;
        }
    }
}

// RING: the ring observation mode (crl_pong_config::stack_mode 1).  A template parameter, so that the plain-stack
// instantiation carries none of the ring's run-time branches and state in its hot loop.
// INC (plain stacks only): the output buffers hold the frames `shown` ([agent][c][n] FrameSpecs) describes; a frame is
// stored only where it can differ from the one it replaces.  A frame equals the template outside its patches (bat
// words, ball pixels) and its scoreboard words [text_w0, text_w1), so the chunks touched by the old frame's patches,
// the new frame's patches and, when the scoreboard entries differ, the scoreboard words cover every changed byte.
// Frames whose specs are equal (ignoring the raw bit) are not stored at all; the all-zero frame and scoreboards outside
// text_tab are stored whole.  Afterwards `shown` holds hist.
template <int DIM, bool RING, bool INC>
__global__ void __launch_bounds__(FAST_WARPS * 32, FastCfg<DIM>::CTAS)
pong_raster_fast_kernel(PongDev p, const FrameSpec* __restrict__ hist, uint8_t* __restrict__ obs0,
                        uint8_t* __restrict__ obs1, const FastTabs<DIM>* __restrict__ gtabs, FrameSpec* __restrict__ shown) {
    constexpr int TAPS = FastCfg<DIM>::TAPS, VEC = FastCfg<DIM>::VEC;
    constexpr int DD = DIM * DIM, FB = ((DD + 15) / 16) * 16, NCH = DD / VEC;
#ifndef CRL_RASTER_TMA
#define CRL_RASTER_TMA 0
#endif
    constexpr bool USE_TMA = (DD % 16 == 0) && (CRL_RASTER_TMA != 0) && !INC;
    constexpr int TEXT_ITERS = 3;   // text_stride <= 96 vectors (checked on the host)
    typedef typename VecT<VEC>::type V;
    typedef FastTabs<DIM> Tabs;
    static_assert(DD % VEC == 0, "frame must be a whole number of store vectors");
    static_assert(!INC || (!RING && VEC == 16), "incremental stacks: 16-byte chunks, plain stacks");

    extern __shared__ uint4 smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(smem_raw);
    const Tabs* T = reinterpret_cast<const Tabs*>(smem);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t* sm8 = smem + sizeof(Tabs) + (size_t)warp * FB;
    V* sm = reinterpret_cast<V*>(sm8);

    // ---- CTA prologue: tables into shared memory, template into every warp's frame buffer ----
    {
        const uint4* src = reinterpret_cast<const uint4*>(gtabs);
        uint4* dst = reinterpret_cast<uint4*>(smem);
        for (int i = threadIdx.x; i < (int)(sizeof(Tabs) / 16); i += blockDim.x) dst[i] = src[i];
        const uint4* tm = reinterpret_cast<const uint4*>(p.tmpl);
        uint4* f = reinterpret_cast<uint4*>(sm8);
        for (int i = lane; i < FB / 16; i += 32) f[i] = tm[i];
    }
    __syncthreads();

    const int text_chunks = p.text_stride / VEC;
    const int cL = (int)T->bat_c0[0], cR = (int)T->bat_c0[1];
    // lane roles
    const int b_side = lane >> 4, b_which = (lane >> 3) & 1, b_row = lane & 7;   // bat strip rows
    const int p_which = lane >> 4, p_col = lane & 3, p_row = (lane >> 2) & 3;    // ball pixels
    // what the previous frame left patched in the buffer (restored before the next write)
    int prev_bat_off = -1, prev_ball_off = -1;
    uint32_t prev_bat_rest = 0u, prev_ball_old = 0u;
    int cur_text = -1;          // text_tab entry whose rows are in the buffer (-1: template's)
    bool pending = false;       // a bulk store may still be reading the buffer
    FrameSpec prev_spec = make_uint4(0u, 0u, 0u, 0u);   // INC: the frame whose patches prev_bat_off / prev_ball_off are
    bool prev_known = false;

    // Stacks are handed out by a global counter, not by a static grid stride: all resident warps then write within one
    // compact window of the observation buffers that advances front to back, like the CTA dispatcher of a non-persistent
    // launch would make them.  Measured with the drain alone (tools/probes/raster_store_probe.cu): 6.8 TB/s against
    // 5.8-5.9 TB/s for the static stride.
    // A ticket covers ~4 frames (one stack of 4, or 4 stacks of 1): one atomic per 28 KB written; one per 7 KB frame
    // makes the counter itself the bottleneck (2.7 TB/s in the probe).
    const long long n_stacks = (long long)p.n * p.n_agents;
    // frames a stack writes: c (plain stack), or the newest frame twice (ring; all 2c slots only after a reset)
    const int per_ticket = INC ? CRL_INC_TICKET : max(1, 4 / (RING ? 2 : p.c));
    const int out_slots = RING ? 2 * p.c : p.c;
    long long s = 0, s_end = 0;
    for (;;) {
        if (s >= s_end) {
            unsigned long long ticket = 0ull;
            if (lane == 0) ticket = atomicAdd(p.work_counter, (unsigned long long)per_ticket);
            s = (long long)__shfl_sync(0xffffffffu, ticket, 0);
            s_end = min(s + per_ticket, n_stacks);
            if (s >= n_stacks) break;
        }
        const long long s_cur = s++;
        const int env = (int)(s_cur / p.n_agents), agent = (int)(s_cur % p.n_agents);
        uint8_t* out_stack = (agent ? obs1 : obs0) + (size_t)env * out_slots * DD;
        FrameSpec my_spec = make_uint4(0u, 0u, 0u, 0u), my_shown = make_uint4(0u, 0u, 0u, 0u);
        FrameSpec* shown_at = INC ? shown + ((size_t)agent * p.c + lane) * p.n + env : nullptr;
        if (lane < p.c) {
            my_spec = hist[(size_t)lane * p.n + env];
            if (INC) my_shown = *shown_at;
        }
        // ring: only the newest frame is new, unless the env was just reset (its whole history changed)
        const int first_slot = (RING && !p.fill_all && !p.last_done[env]) ? p.c - 1 : 0;

        for (int slot = first_slot; slot < p.c; ++slot) {
            FrameSpec f;
            f.x = __shfl_sync(0xffffffffu, my_spec.x, slot);
            f.y = __shfl_sync(0xffffffffu, my_spec.y, slot);
            f.z = __shfl_sync(0xffffffffu, my_spec.z, slot);
            f.w = __shfl_sync(0xffffffffu, my_spec.w, slot);
            const FrameSpec f_raw = f;
            FrameSpec o = f;   // INC: what the buffer's slot holds
            if (INC) {
                o.x = __shfl_sync(0xffffffffu, my_shown.x, slot);
                o.y = __shfl_sync(0xffffffffu, my_shown.y, slot);
                o.z = __shfl_sync(0xffffffffu, my_shown.z, slot);
                o.w = __shfl_sync(0xffffffffu, my_shown.w, slot);
                if (spec_diff(f, o) == 0u) continue;   // the slot already holds this frame
            }
            // plain stack: frame `slot` goes to channel `slot`.  Ring: to slot ring_phase + 1 + slot and to its double
            // c slots before or after it, whichever exists (the newest frame: ring_phase + c and ring_phase)
            uint8_t* out8 = out_stack + (size_t)slot * DD;
            uint8_t* out8b = nullptr;
            if (RING) {
                const int pos = p.ring_phase + 1 + slot;
                out8 = out_stack + (size_t)pos * DD;
                out8b = out_stack + (size_t)(pos >= p.c ? pos - p.c : pos + p.c) * DD;
            }

            // ---- frame context (warp-uniform) ----
            const bool va = (f.y >> 16) & 1u, vb = (f.w >> 16) & 1u;
            if (!va) { f.x = f.z; f.y = f.w; }
            if (!vb) { f.z = f.x; f.w = f.y; }
            const int pairA = (int)(f.y & 255u) * ATLAS_SCORES + (int)((f.y >> 8) & 255u);
            const int pairB = (int)(f.w & 255u) * ATLAS_SCORES + (int)((f.w >> 8) & 255u);
            int base = pairA, kind = 0;
            const bool blank = !scores_in_atlas(f.y, f.w);   // a score past 21: no text, never a table index
            bool text_ok = !blank;
            if (text_ok && pairA != pairB) {   // one point scored between the two pooled frames
                const int d = pairB - pairA;
                if (d == ATLAS_SCORES) kind = 1;
                else if (d == 1 && (pairA % ATLAS_SCORES) != ATLAS_SCORES - 1) kind = 2;
                // d < 0 and |d| not in {1, 22} are not reached from game states: a history frame pools sub-steps 2 and 3 of
                // one step (a done replaces the whole history), so frame B never shows fewer points, nor two more, than A
                else if (d == -ATLAS_SCORES) { base = pairB; kind = 1; }
                else if (d == -1 && (pairB % ATLAS_SCORES) != ATLAS_SCORES - 1) { base = pairB; kind = 2; }
                else text_ok = false;
            }

            if (!(va || vb)) {
                // both MaxAndSkip buffers still np.zeros (a done on the very first sub-steps after
                // construction; not reachable in play): the frame is all zeros.  The staged buffer is untouched.
                V z;
                memset(&z, 0, sizeof z);
                V* out = reinterpret_cast<V*>(out8);
                for (int k = lane; k < NCH; k += 32) st_stream(out + k, z);
                if (RING) {
                    V* outb = reinterpret_cast<V*>(out8b);
                    for (int k = lane; k < NCH; k += 32) st_stream(outb + k, z);
                }
                continue;
            }

            // ======== A. everything that differs from the template, in registers ========
            const bool same = (f.x == f.z);
            // view coordinates: agent 1 sees the arena mirrored in x, so the view-left bat strip
            // shows the game's right bat
            const int lyA = (f.x >> 16) & 255u, ryA = f.x >> 24, lyB = (f.z >> 16) & 255u, ryB = f.z >> 24;
            const int vlA = agent ? ryA : lyA, vrA = agent ? lyA : ryA;
            const int vlB = agent ? ryB : lyB, vrB = agent ? lyB : ryB;

            // ---- A1. scoreboard rows (only when the buffer holds another score pair's) ----
            const int text_id = text_ok ? (base * 3 + kind) * 2 + agent : -2;
            const bool reload_text = text_id != cur_text || !text_ok;
            const uint8_t* __restrict__ te8 = p.text_tab + (size_t)text_id * p.text_stride;
            if (reload_text && text_ok && lane * 128 < p.text_stride)   // pull the entry's lines L2 -> L1 now, copy in phase B
                asm volatile("prefetch.global.L1 [%0];" ::"l"(te8 + lane * 128));

            // ---- A2. bat strips: lane = (view side, frame A|B, row); one LUT word per row ----
            int bat_off = -1;
            uint32_t bat_val = 0u, bat_rest = 0u;
            {
                const int yA = b_side ? vrA : vlA, yB = b_side ? vrB : vlB;
                const int y0 = b_which ? yB : yA;
                const int c0 = max(y0, ARENA_TOP), c1 = min(y0 + BAT_H, ARENA_BOTTOM);   // white on white outside
                if (c1 > c0 && !(b_which && same)) {
                    const int dy = (int)T->y_first[c0] + b_row;
                    if (dy <= (int)T->y_last[c1 - 1]) {
                        const uint32_t meta = T->ye[dy].meta;
                        const int sy0 = meta & 255u;
                        const int a0 = max(yA, ARENA_TOP), a1 = min(yA + BAT_H, ARENA_BOTTOM);
                        const int b0 = max(yB, ARENA_TOP), b1 = min(yB + BAT_H, ARENA_BOTTOM);
                        uint32_t vbits = 0u;
                        if (a1 > a0) vbits |= tap_bits(((1u << (a1 - a0)) - 1u) << 8, a0, sy0);
                        if (b1 > b0) vbits |= tap_bits(((1u << (b1 - b0)) - 1u) << 8, b0, sy0);
                        vbits &= (meta >> 8) & 255u;
                        bat_val = T->bat_lut[b_side][dy][vbits];
                        bat_rest = T->bat_lut[b_side][dy][0];
                        bat_off = dy * DIM + (b_side ? cR : cL);
                    }
                }
            }

            // ---- A3. ball pixels: lane = (frame A|B, 4x4 window position), exact evaluation ----
            int ball_off = -1;
            uint32_t ball_val = 0u;
            {
                // both balls in view coordinates, clipped to the arena rows (white on white outside)
                int ax0 = f.x & 255u, ax1 = min(ax0 + BALL_SIZE, SCREEN_W);
                int ay0 = (f.x >> 8) & 255u, ay1 = min(ay0 + BALL_SIZE, ARENA_BOTTOM);
                ay0 = max(ay0, ARENA_TOP);
                int bx0 = f.z & 255u, bx1 = min(bx0 + BALL_SIZE, SCREEN_W);
                int by0 = (f.z >> 8) & 255u, by1 = min(by0 + BALL_SIZE, ARENA_BOTTOM);
                by0 = max(by0, ARENA_TOP);
                if (agent) {
                    int t = SCREEN_W - ax1; ax1 = SCREEN_W - ax0; ax0 = t;
                    t = SCREEN_W - bx1; bx1 = SCREEN_W - bx0; bx0 = t;
                }
                const bool ea = ax1 > ax0 && ay1 > ay0, eb = bx1 > bx0 && by1 > by0 && !same;
                const int mx0 = p_which ? bx0 : ax0, mx1 = p_which ? bx1 : ax1;
                const int my0 = p_which ? by0 : ay0, my1 = p_which ? by1 : ay1;
                if (p_which ? eb : ea) {
                    const int dx = (int)T->x_first[mx0] + p_col, dy = (int)T->y_first[my0] + p_row;
                    if (dx <= (int)T->x_last[mx1 - 1] && dy <= (int)T->y_last[my1 - 1]) {
                        const TapEnt<TAPS> X = T->xe[dx], Y = T->ye[dy];
                        const int sx0 = X.meta & 255u, sy0 = Y.meta & 255u;
                        const uint32_t xmask = (X.meta >> 8) & 255u, ymask = (Y.meta >> 8) & 255u;
                        uint32_t pat = xmask * spread6((Y.meta >> 16) & 255u);   // border rows: all white
                        if (ea)
                            pat |= (tap_bits(((1u << (ax1 - ax0)) - 1u) << 8, ax0, sx0) & xmask) *
                                   spread6(tap_bits(((1u << (ay1 - ay0)) - 1u) << 8, ay0, sy0) & ymask);
                        if (eb)
                            pat |= (tap_bits(((1u << (bx1 - bx0)) - 1u) << 8, bx0, sx0) & xmask) *
                                   spread6(tap_bits(((1u << (by1 - by0)) - 1u) << 8, by0, sy0) & ymask);
                        // a bat strip under this pixel: both frames' bats of that side
                        const bool nl = (unsigned)(dx - cL) < 4u, nr = (unsigned)(dx - cR) < 4u;
                        if (nl || nr) {
                            const int yA = nr ? vrA : vlA, yB = nr ? vrB : vlB;
                            const int a0 = max(yA, ARENA_TOP), a1 = min(yA + BAT_H, ARENA_BOTTOM);
                            const int b0 = max(yB, ARENA_TOP), b1 = min(yB + BAT_H, ARENA_BOTTOM);
                            uint32_t vbits = 0u;
                            if (a1 > a0) vbits |= tap_bits(((1u << (a1 - a0)) - 1u) << 8, a0, sy0);
                            if (b1 > b0) vbits |= tap_bits(((1u << (b1 - b0)) - 1u) << 8, b0, sy0);
                            const uint32_t hb = tap_bits(((1u << BAT_W) - 1u) << 8, nr ? RIGHT_BAT_X : LEFT_BAT_X, sx0);
                            pat |= (hb & xmask) * spread6(vbits & ymask);
                        }
                        ball_val = eval_from_pat_lut<TAPS>(T->xlut[dx], Y, pat);
                        ball_off = dy * DIM + dx;
                    }
                }
            }

            // ---- A4 (INC). what to store: the whole frame, or the chunks under both frames' patches and, when the
            //      scoreboard entries differ, the chunks [ta, tb) of the scoreboard words ----
            bool whole = true;
            int ta = 0, tb = 0, old_bat = -1, old_ball = -1;
            if (INC) {
                bool old_valid;
                const int old_text = frame_text_id(o, agent, old_valid);
                whole = !old_valid || old_text == -2 || !text_ok;
                if (!whole && old_text != text_id) { ta = p.text_w0 * 4 >> 4; tb = min((p.text_w1 * 4 + 15) >> 4, NCH); }
                if (!whole) {
                    if (prev_known && spec_diff(o, prev_spec) == 0u) { old_bat = prev_bat_off; old_ball = prev_ball_off; }
                    else frame_patch_offsets<DIM>(T, o, agent, lane, old_bat, old_ball);
                }
            }

            // ======== B. the buffer: wait for the previous drain, restore, patch ========
            if (pending) {
                if (lane == 0) bulk_wait_read();
                __syncwarp();
            }
            if (prev_bat_off >= 0) {
                if (DIM % 4 == 0) {
                    *reinterpret_cast<uint32_t*>(sm8 + prev_bat_off) = prev_bat_rest;
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) sm8[prev_bat_off + j] = (uint8_t)(prev_bat_rest >> (8 * j));
                }
            }
            __syncwarp();
            if (prev_ball_off >= 0) sm8[prev_ball_off] = (uint8_t)prev_ball_old;   // after the bats: a ball pixel may lie on a strip
            __syncwarp();
            if (reload_text) {
                if (text_ok) {
                    const V* __restrict__ te = reinterpret_cast<const V*>(te8);
#pragma unroll
                    for (int j = 0; j < TEXT_ITERS; ++j)
                        if (lane + 32 * j < text_chunks) sm[lane + 32 * j] = te[lane + 32 * j];
                } else {   // score combination outside the table: exact rows straight from the atlas
                    const int n_text = p.tabs->text_rows * DIM;
                    for (int i = lane; i < n_text; i += 32)
                        sm8[i] = eval_text_pixel(p.tabs, p.atlas, pairA, pairB, blank, agent != 0, i / DIM, i % DIM);
                }
                cur_text = text_id;
                __syncwarp();
            }
            uint32_t ball_old = 0u;
            if (ball_off >= 0) ball_old = sm8[ball_off];      // template / scoreboard value under the ball
            __syncwarp();
            if (bat_off >= 0) {
                if (DIM % 4 == 0) {
                    *reinterpret_cast<uint32_t*>(sm8 + bat_off) = bat_val;
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) sm8[bat_off + j] = (uint8_t)(bat_val >> (8 * j));
                }
            }
            __syncwarp();
            if (ball_off >= 0) sm8[ball_off] = (uint8_t)ball_val;   // overrides the strip LUT where the ball is near
            prev_bat_off = bat_off; prev_bat_rest = bat_rest;
            prev_ball_off = ball_off; prev_ball_old = ball_old;
            prev_spec = f_raw; prev_known = true;

            // ======== C. drain ========
#ifdef CRL_RASTER_NO_DRAIN
            // measurement build: everything but the stores (the kernel's compute floor); the output is left unwritten
            continue;
#endif
            if (INC && !whole) {
                // Every lane stores the chunk under each of its patch offsets.  Lanes that hit the same chunk in one
                // instruction store the same 16 bytes and coalesce; a chunk stored by two instructions gets the same bytes
                // twice.  (A shared-memory bitmap that deduplicated the chunks first cost more in atomics than it saved.)
                __syncwarp();
                V* out = reinterpret_cast<V*>(out8);
                for (int u = ta + lane; u < tb; u += 32) st_stream(out + u, sm[u]);
                const int offs[4] = {old_bat, old_ball, bat_off, ball_off};
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (offs[k] >= 0) st_stream(out + (offs[k] >> 4), sm[offs[k] >> 4]);
                __syncwarp();
            } else if (USE_TMA) {
                fence_proxy_async_smem();    // generic-proxy writes -> visible to the async proxy
                __syncwarp();
                if (lane == 0) {
                    bulk_store(out8, sm8, DD);
                    if (RING) bulk_store(out8b, sm8, DD);
                }
                pending = true;
            } else {
                __syncwarp();
                V* out = reinterpret_cast<V*>(out8);
                if (!RING) {
#pragma unroll
                    for (int j = 0; j < (NCH + 31) / 32; ++j)
                        if ((j + 1) * 32 <= NCH || lane + 32 * j < NCH) st_stream(out + lane + 32 * j, sm[lane + 32 * j]);
                } else {
                    V* outb = reinterpret_cast<V*>(out8b);
#pragma unroll
                    for (int j = 0; j < (NCH + 31) / 32; ++j)
                        if ((j + 1) * 32 <= NCH || lane + 32 * j < NCH) {
                            const V v = sm[lane + 32 * j];
                            st_stream(out + lane + 32 * j, v);
                            st_stream(outb + lane + 32 * j, v);
                        }
                }
                __syncwarp();
            }
        }
        if (INC && lane < p.c) *shown_at = my_spec;
        prev_known = false;   // patch offsets depend on the agent too
    }
    if (USE_TMA && lane == 0) bulk_wait_all();   // the buffer must outlive the last drain
}

// ---------------------------------------------------------------------------------
// 42x42 (the make_envs default, what every built-in agent consumes): FOUR frames per warp.
//
// A 42x42 frame is 1 764 bytes, a quarter of the 84x84 one, but what has to be computed per frame (two bat strips, two
// pooled ball positions, the scoreboard rows) is the same, so the one-frame-per-warp kernel above is bound by
// instruction issue at 42x42 (518 warp-instructions per 1 764 bytes, 0.52 of the HBM roofline).  Here a warp owns a QUAD
// of four frames that are adjacent in the output (with frame_stack 4: the stack of one (env, agent); with frame_stack
// None: four consecutive envs) = 7 056 bytes = 441 16-byte vectors.  Lane group g = lane >> 3 works on frame g, so every
// instruction of the patch phase serves four frames at once: per side the (frame A | frame B, row) items of the bat strips
// (a bat touches <= 4 destination rows and exactly two destination columns -> one 16-bit store), per pooled ball the
// <= 3 x 2 destination pixels.  The quad is then drained as one flat run of 16-byte st.global.cs (1 764 is not a multiple
// of 16, 7 056 is), instead of 4-byte stores.  Arithmetic is the kernel's above, so the results are bit-identical.
// Quads containing an unusual frame (both pool buffers zero, score combination outside text_tab or past the atlas) are evaluated exactly,
// pixel by pixel, like pong_raster_generic_kernel does.
// the tables of FastTabs the quad kernel keeps in shared memory (the bat LUT narrowed to the two columns a bat touches)
template <int DIM> struct alignas(16) QuadTabs {
    TapEnt<FastCfg<DIM>::TAPS> xe[DIM], ye[DIM];
    float xlut[DIM][1 << FastCfg<DIM>::TAPS];
    uint16_t bat2[2][DIM][1 << FastCfg<DIM>::TAPS];
    uint8_t x_first[SCREEN_W], x_last[SCREEN_W], y_first[FIRST_PAD], y_last[FIRST_PAD];
    uint32_t bat_c0[2], pad[2];
};

#ifndef CRL_QUAD_CTAS
#define CRL_QUAD_CTAS 2      // measured: 3 CTAs per SM (80 registers, 108 B of spills) 0.236 ms per step, 2 CTAs 0.2 ms
#endif
#ifndef CRL_QUAD_WARPS
#define CRL_QUAD_WARPS 10      // measured per 65 536-env step: 8 warps x 2 CTAs 0.202 ms, 10 x 2 (96 registers) 0.191 ms, 11 x 2 and 8 x 3 (80 registers, spills) 0.23 ms
#endif
constexpr int QUAD_WARPS = CRL_QUAD_WARPS;
template <int DIM>
__global__ void __launch_bounds__(QUAD_WARPS * 32, CRL_QUAD_CTAS)
pong_raster_quad_kernel(PongDev p, const FrameSpec* __restrict__ hist, uint8_t* __restrict__ obs0,
                        uint8_t* __restrict__ obs1, const FastTabs<DIM>* __restrict__ gtabs) {
    constexpr int TAPS = FastCfg<DIM>::TAPS, NP = 1 << TAPS;
    constexpr int DD = DIM * DIM, QB = 4 * DD, NV = QB / 16, DW = DD / 4;
    constexpr int TEXT_WORDS_MAX = 96 * DD / (42 * 42);      // pong_fast_tabs_fill refuses longer scoreboard entries (96 * 4 bytes at 42 x 42)
    typedef QuadTabs<DIM> Tabs;
    static_assert(QB % 16 == 0 && DD % 4 == 0, "a quad must be a whole number of 16-byte vectors");

    extern __shared__ uint4 smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(smem_raw);
    Tabs* Tw = reinterpret_cast<Tabs*>(smem);
    const Tabs* T = Tw;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 3, sub = lane & 7;                 // frame of the quad, lane within its group
    uint8_t* smq = smem + sizeof(Tabs) + (size_t)warp * QB;  // the warp's quad buffer (16-byte aligned)
    uint8_t* sm8 = smq + g * DD;                             // this group's frame
    const uint32_t* tm32 = reinterpret_cast<const uint32_t*>(p.tmpl);

    auto load_templates = [&]() {
        uint32_t* q32 = reinterpret_cast<uint32_t*>(smq);
        for (int i = lane; i < DW; i += 32) {
            const uint32_t v = tm32[i];
            q32[i] = v; q32[DW + i] = v; q32[2 * DW + i] = v; q32[3 * DW + i] = v;
        }
    };
    {   // CTA prologue: tables into shared memory, the template into every frame of every warp's quad buffer
        const int tid = threadIdx.x, nt = blockDim.x;
        for (int i = tid; i < DIM; i += nt) { Tw->xe[i] = gtabs->xe[i]; Tw->ye[i] = gtabs->ye[i]; }
        for (int i = tid; i < DIM * NP; i += nt) (&Tw->xlut[0][0])[i] = (&gtabs->xlut[0][0])[i];
        for (int i = tid; i < 2 * DIM * NP; i += nt) (&Tw->bat2[0][0][0])[i] = (uint16_t)(&gtabs->bat_lut[0][0][0])[i];
        for (int i = tid; i < SCREEN_W; i += nt) { Tw->x_first[i] = gtabs->x_first[i]; Tw->x_last[i] = gtabs->x_last[i]; }
        for (int i = tid; i < FIRST_PAD; i += nt) { Tw->y_first[i] = gtabs->y_first[i]; Tw->y_last[i] = gtabs->y_last[i]; }
        if (tid < 2) Tw->bat_c0[tid] = gtabs->bat_c0[tid];
        load_templates();
    }
    __syncthreads();

    // the words of a scoreboard entry that can differ from what a frame buffer holds (PongDev::text_w0 / text_w1: the rows
    // with the score digits), clipped to what the copy loops below are sized for
    const int text_w0 = p.text_w0, text_nw = min(p.text_w1, min(p.text_stride / 4, TEXT_WORDS_MAX)) - p.text_w0;
    const int cL = (int)T->bat_c0[0], cR = (int)T->bat_c0[1];
    const int b_which = sub >> 2, b_row = sub & 3;           // bat items of one side: (frame A | B, row)
    const int p_col = sub & 3, p_row = sub >> 2;             // ball pixels of one pooled frame: 4 x 2 window
    // what the previous quad left patched in this group's frame (restored before the next patches)
    int bat_off[2] = {-1, -1}, ball_off[2] = {-1, -1};
    uint32_t bat_rest[2] = {0u, 0u}, ball_old[2] = {0u, 0u};
    int cur_text = -1;

    // 32-bit work indices (the host launches this kernel only when they fit)
    const unsigned c = (unsigned)p.c, n_env = (unsigned)p.n;
    const unsigned frames_per_agent = n_env * c;
    const unsigned quads_per_agent = (frames_per_agent + 3u) / 4u;
    const unsigned n_quads = quads_per_agent * (unsigned)p.n_agents;
    const bool two = p.n_agents == 2;
    constexpr unsigned PER_TICKET = 4;                       // one atomic per 28 KB written (see the kernel above)
    // With few warps per SM (the quad buffers fill the shared memory) little hides a dependent global load: the next
    // ticket is drawn while the current one is worked on, and the frame specs of a ticket's quads are pulled into L1
    // (one prefetch per lane) as soon as the ticket is known.
    auto frame_of = [&](unsigned F, unsigned& env, unsigned& slot) {
        if (c == 4u) { env = F >> 2; slot = F & 3u; }
        else if (c == 1u) { env = F; slot = 0u; }
        else { env = F / c; slot = F - env * c; }
    };
    unsigned next_ticket = 0u;
    if (lane == 0) next_ticket = (unsigned)atomicAdd(p.work_counter, (unsigned long long)PER_TICKET);
    unsigned s = 0u, s_end = 0u;
    for (;;) {
        if (s >= s_end) {
            s = __shfl_sync(0xffffffffu, next_ticket, 0);
            if (s >= n_quads) break;
            s_end = min(s + PER_TICKET, n_quads);
            if (sub < PER_TICKET && s + sub < n_quads) {     // lane (g, sub): frame g of quad s + sub
                const unsigned F_ = (two ? (s + sub) >> 1 : s + sub) * 4u + g;
                if (F_ < frames_per_agent) {
                    unsigned e_, sl_;
                    frame_of(F_, e_, sl_);
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(hist + (size_t)sl_ * n_env + e_));
                }
            }
            if (lane == 0) next_ticket = (unsigned)atomicAdd(p.work_counter, (unsigned long long)PER_TICKET);   // used a ticket later
        }
        const unsigned id = s++;
        // agents interleaved, so that both observation buffers are written front to back in step
        const int agent = two ? (int)(id & 1u) : 0;
        const unsigned q = two ? (id >> 1) : id;
        const unsigned F = q * 4u + g;
        const bool valid = F < frames_per_agent;
        unsigned env = 0u, slot = 0u;
        if (valid) frame_of(F, env, slot);
        uint8_t* out_quad = (agent ? obs1 : obs0) + (size_t)q * QB;
        FrameSpec f = make_uint4(0u, 0u, 0u, 0u);
        if (valid) f = hist[(size_t)slot * n_env + env];
        const FrameSpec f_raw = f;

        // ---- frame context (uniform within the lane group) ----
        const bool va = (f.y >> 16) & 1u, vb = (f.w >> 16) & 1u;
        if (!va) { f.x = f.z; f.y = f.w; }
        if (!vb) { f.z = f.x; f.w = f.y; }
        const int pairA = (int)(f.y & 255u) * ATLAS_SCORES + (int)((f.y >> 8) & 255u);
        const int pairB = (int)(f.w & 255u) * ATLAS_SCORES + (int)((f.w >> 8) & 255u);
        int base = pairA, kind = 0;
        bool text_ok = scores_in_atlas(f.y, f.w);            // a score past 21: the exact path draws no text
        if (text_ok && pairA != pairB) {   // one point scored between the two pooled frames
            const int d = pairB - pairA;
            if (d == ATLAS_SCORES) kind = 1;
            else if (d == 1 && (pairA % ATLAS_SCORES) != ATLAS_SCORES - 1) kind = 2;
            else if (d == -ATLAS_SCORES) { base = pairB; kind = 1; }   // d < 0: not reached from game states (see above)
            else if (d == -1 && (pairB % ATLAS_SCORES) != ATLAS_SCORES - 1) { base = pairB; kind = 2; }
            else text_ok = false;
        }
        const bool unusual = valid && (!(va || vb) || !text_ok);
        if (__any_sync(0xffffffffu, unusual)) {
            // ======== exact path: every pixel of the four frames from the atlas and the frame specs ========
            __syncwarp();
            for (int j = 0; j < 4; ++j) {
                FrameSpec fj;
                fj.x = __shfl_sync(0xffffffffu, f_raw.x, 8 * j); fj.y = __shfl_sync(0xffffffffu, f_raw.y, 8 * j);
                fj.z = __shfl_sync(0xffffffffu, f_raw.z, 8 * j); fj.w = __shfl_sync(0xffffffffu, f_raw.w, 8 * j);
                const FrameCtx cx = make_ctx(fj, agent);
                for (int pix = lane; pix < DD; pix += 32)
                    smq[j * DD + pix] = cx.any_valid ? eval_pixel(p.tabs, cx, p.atlas, pix / DIM, pix % DIM) : (uint8_t)0;
            }
            __syncwarp();
            const int n_valid = (int)min(4u, frames_per_agent - q * 4u);
            const uint32_t* q32 = reinterpret_cast<const uint32_t*>(smq);
            uint32_t* o32 = reinterpret_cast<uint32_t*>(out_quad);
            for (int i = lane; i < n_valid * DW; i += 32) st_stream(o32 + i, q32[i]);
            __syncwarp();
            load_templates();                                 // back to the resident-template state
            cur_text = -1;
            bat_off[0] = bat_off[1] = ball_off[0] = ball_off[1] = -1;
            __syncwarp();
            continue;
        }

        const bool same = (f.x == f.z);
        const int lyA = (f.x >> 16) & 255u, ryA = f.x >> 24, lyB = (f.z >> 16) & 255u, ryB = f.z >> 24;
        const int vlA = agent ? ryA : lyA, vrA = agent ? lyA : ryA;   // view coordinates (agent 1: mirrored in x)
        const int vlB = agent ? ryB : lyB, vrB = agent ? lyB : ryB;

        // the scoreboard rows this frame needs: pull the table entry (L2-resident, 304 bytes) into L1 now, copy it below
        const int text_id = (base * 3 + kind) * 2 + agent;
        const bool reload_text = valid && text_id != cur_text;
        const uint32_t* __restrict__ te = reinterpret_cast<const uint32_t*>(p.text_tab + (size_t)text_id * p.text_stride);
        if (reload_text && sub * 128 < p.text_stride)
            asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const uint8_t*>(te) + sub * 128));

        // ======== restore what the previous quad patched ========
#pragma unroll
        for (int r = 0; r < 2; ++r)
            if (bat_off[r] >= 0) *reinterpret_cast<uint16_t*>(sm8 + bat_off[r]) = (uint16_t)bat_rest[r];
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 2; ++r)
            if (ball_off[r] >= 0) sm8[ball_off[r]] = (uint8_t)ball_old[r];   // after the bats: a ball pixel may lie on a strip
        __syncwarp();

        // vertical tap masks of the two pooled bats per view side (arena-clipped, as tap_bits wants them)
        const int la0 = max(vlA, ARENA_TOP), la1 = min(vlA + BAT_H, ARENA_BOTTOM), lb0 = max(vlB, ARENA_TOP), lb1 = min(vlB + BAT_H, ARENA_BOTTOM);
        const int ra0 = max(vrA, ARENA_TOP), ra1 = min(vrA + BAT_H, ARENA_BOTTOM), rb0 = max(vrB, ARENA_TOP), rb1 = min(vrB + BAT_H, ARENA_BOTTOM);
        auto bat_vbits = [&](bool right, int sy0) -> uint32_t {
            const int a0 = right ? ra0 : la0, a1 = right ? ra1 : la1, b0 = right ? rb0 : lb0, b1 = right ? rb1 : lb1;
            uint32_t vbits = 0u;
            if (a1 > a0) vbits |= tap_bits(((1u << (a1 - a0)) - 1u) << 8, a0, sy0);
            if (b1 > b0) vbits |= tap_bits(((1u << (b1 - b0)) - 1u) << 8, b0, sy0);
            return vbits;
        };

        // ======== ball pixels: round r = pooled frame r, lane = pixel of its 4 x 2 window; exact evaluation (values only:
        //          nothing here touches the frame buffer, so the scoreboard prefetch above has time to land) ========
        uint32_t ball_val[2] = {0u, 0u};
        {
            int ax0 = f.x & 255u, ax1 = min(ax0 + BALL_SIZE, SCREEN_W);
            int ay0 = (f.x >> 8) & 255u, ay1 = min(ay0 + BALL_SIZE, ARENA_BOTTOM);
            ay0 = max(ay0, ARENA_TOP);
            int bx0 = f.z & 255u, bx1 = min(bx0 + BALL_SIZE, SCREEN_W);
            int by0 = (f.z >> 8) & 255u, by1 = min(by0 + BALL_SIZE, ARENA_BOTTOM);
            by0 = max(by0, ARENA_TOP);
            if (agent) {
                int t = SCREEN_W - ax1; ax1 = SCREEN_W - ax0; ax0 = t;
                t = SCREEN_W - bx1; bx1 = SCREEN_W - bx0; bx0 = t;
            }
            const bool ea = valid && ax1 > ax0 && ay1 > ay0, eb = valid && bx1 > bx0 && by1 > by0 && !same;
            const uint32_t axm = ((1u << (ax1 - ax0)) - 1u) << 8, aym = ((1u << (ay1 - ay0)) - 1u) << 8;
            const uint32_t bxm = ((1u << (bx1 - bx0)) - 1u) << 8, bym = ((1u << (by1 - by0)) - 1u) << 8;
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                ball_off[r] = -1;
                const int mx0 = r ? bx0 : ax0, mx1 = r ? bx1 : ax1, my0 = r ? by0 : ay0, my1 = r ? by1 : ay1;
                if (r ? eb : ea) {
                    const int dx = (int)T->x_first[mx0] + p_col, dy = (int)T->y_first[my0] + p_row;
                    if (dx <= (int)T->x_last[mx1 - 1] && dy <= (int)T->y_last[my1 - 1]) {
                        const uint32_t xmeta = T->xe[dx].meta;
                        const TapEnt<TAPS> Y = T->ye[dy];
                        const int sx0 = xmeta & 255u, sy0 = Y.meta & 255u;
                        const uint32_t xmask = (xmeta >> 8) & 255u, ymask = (Y.meta >> 8) & 255u;
                        uint32_t pat = xmask * spread6((Y.meta >> 16) & 255u);   // border rows: all white
                        if (ea) pat |= (tap_bits(axm, ax0, sx0) & xmask) * spread6(tap_bits(aym, ay0, sy0) & ymask);
                        if (eb) pat |= (tap_bits(bxm, bx0, sx0) & xmask) * spread6(tap_bits(bym, by0, sy0) & ymask);
                        const bool nl = (unsigned)(dx - cL) < 4u, nr = (unsigned)(dx - cR) < 4u;
                        if (nl || nr) {                                   // a bat strip under this pixel: both frames' bats
                            const uint32_t hb = tap_bits(((1u << BAT_W) - 1u) << 8, nr ? RIGHT_BAT_X : LEFT_BAT_X, sx0);
                            pat |= (hb & xmask) * spread6(bat_vbits(nr, sy0) & ymask);
                        }
                        ball_val[r] = eval_from_pat_lut<TAPS>(T->xlut[dx], Y, pat);
                        ball_off[r] = dy * DIM + dx;
                    }
                }
            }
        }

        // ======== scoreboard rows of this frame's score pair(s), when the buffer holds another pair's ========
        if (__any_sync(0xffffffffu, reload_text)) {
            // The four frames of a quad are the four stack slots of one env (frame_stack 4): one score pair in about half the
            // quads; then the entry is fetched once by the whole warp (2-3 words per lane instead of 6-12 per lane of every group)
            // and stored into the four frame buffers.
            // All loads of an entry are issued before its first store (fixed trip counts, no branch between them): one
            // round trip to L1 / L2 per reload instead of one per chunk of a copy loop.
            const int id0 = __shfl_sync(0xffffffffu, text_id, 0);
            if (text_nw <= 0) {                              // every entry equals the template
                if (reload_text) cur_text = text_id;
            } else if (__all_sync(0xffffffffu, valid && text_id == id0)) {
                uint32_t* q32 = reinterpret_cast<uint32_t*>(smq);
                auto copy_warp = [&](auto KC) {
                    constexpr int K = decltype(KC)::value;
                    uint32_t w[K];
                    int wi[K];
#pragma unroll
                    for (int k = 0; k < K; ++k) {
                        wi[k] = text_w0 + min(lane + 32 * k, text_nw - 1);   // past the end: the last word again (same value, same place)
                        w[k] = te[wi[k]];
                    }
#pragma unroll
                    for (int k = 0; k < K; ++k) {
                        q32[wi[k]] = w[k]; q32[DW + wi[k]] = w[k]; q32[2 * DW + wi[k]] = w[k]; q32[3 * DW + wi[k]] = w[k];
                    }
                };
                if (text_nw <= 64) copy_warp(std::integral_constant<int, 2>{});
                else copy_warp(std::integral_constant<int, (TEXT_WORDS_MAX + 31) / 32>{});
                cur_text = text_id;
            } else if (reload_text) {
                uint32_t* d32 = reinterpret_cast<uint32_t*>(sm8);
                auto copy_group = [&](auto KC) {
                    constexpr int K = decltype(KC)::value;
                    uint32_t w[K];
#pragma unroll
                    for (int k = 0; k < K; ++k) w[k] = te[text_w0 + min(sub + 8 * k, text_nw - 1)];
#pragma unroll
                    for (int k = 0; k < K; ++k)
                        if (sub + 8 * k < text_nw) d32[text_w0 + sub + 8 * k] = w[k];
                };
                if (text_nw <= 48) copy_group(std::integral_constant<int, 6>{});
                else copy_group(std::integral_constant<int, (TEXT_WORDS_MAX + 7) / 8>{});
                cur_text = text_id;
            }
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 2; ++r)
            if (ball_off[r] >= 0) ball_old[r] = sm8[ball_off[r]];     // template / scoreboard value under the ball
        __syncwarp();

        // ======== bat strips: round r = view side r, lane = (frame A | B, row); one LUT entry (two pixels) per row ========
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            bat_off[r] = -1;
            const int y0 = b_which ? (r ? vrB : vlB) : (r ? vrA : vlA);
            const int c0 = max(y0, ARENA_TOP), c1 = min(y0 + BAT_H, ARENA_BOTTOM);   // white on white outside
            if (valid && c1 > c0 && !(b_which && same)) {
                const int dy = (int)T->y_first[c0] + b_row;
                if (dy <= (int)T->y_last[c1 - 1]) {
                    const uint32_t meta = T->ye[dy].meta;
                    const uint32_t vbits = bat_vbits(r != 0, meta & 255u) & ((meta >> 8) & 255u);
                    bat_off[r] = dy * DIM + (r ? cR : cL);
                    bat_rest[r] = T->bat2[r][dy][0];
                    *reinterpret_cast<uint16_t*>(sm8 + bat_off[r]) = T->bat2[r][dy][vbits];
                }
            }
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 2; ++r)
            if (ball_off[r] >= 0) sm8[ball_off[r]] = (uint8_t)ball_val[r];   // overrides the strip LUT where the ball is near
        __syncwarp();

        // ======== drain: the quad as one run of 16-byte streaming stores ========
        if (q * 4u + 4u <= frames_per_agent) {
            const uint4* q128 = reinterpret_cast<const uint4*>(smq);
            uint4* out = reinterpret_cast<uint4*>(out_quad);
#pragma unroll
            for (int j = 0; j < (NV + 31) / 32; ++j)
                if ((j + 1) * 32 <= NV || lane + 32 * j < NV) st_stream(out + lane + 32 * j, q128[lane + 32 * j]);
        } else {                                             // the last, partial quad of a buffer
            const int n_valid = (int)(frames_per_agent - q * 4u);
            const uint32_t* q32 = reinterpret_cast<const uint32_t*>(smq);
            uint32_t* o32 = reinterpret_cast<uint32_t*>(out_quad);
            for (int i = lane; i < n_valid * DW; i += 32) st_stream(o32 + i, q32[i]);
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------
// host side
template <int DIM>
static bool fill_fast_tabs(const AreaTabs& a, FastTabs<DIM>* t) {
    constexpr int TAPS = FastCfg<DIM>::TAPS;
    memset(t, 0, sizeof *t);
    for (int i = 0; i < DIM; ++i) {
        if (a.x_n[i] > TAPS || a.y_n[i] > TAPS) return false;
        t->xe[i].meta = (uint32_t)a.x_src0[i] | (((1u << a.x_n[i]) - 1u) << 8);
        uint32_t white = 0u;
        for (int k = 0; k < a.y_n[i]; ++k) {
            const int sy = a.y_src0[i] + k;
            if (sy < ARENA_TOP || sy >= ARENA_BOTTOM) white |= 1u << k;
        }
        t->ye[i].meta = (uint32_t)a.y_src0[i] | (((1u << a.y_n[i]) - 1u) << 8) | (white << 16);
        for (int k = 0; k < TAPS; ++k) {
            t->xe[i].w[k] = k < a.x_n[i] ? a.x_pa[i][k] : 0.f;
            t->ye[i].w[k] = k < a.y_n[i] ? a.y_b[i][k] : 0.f;
        }
    }
    memcpy(t->x_first, a.x_first, SCREEN_W);
    memcpy(t->x_last, a.x_last, SCREEN_W);
    memcpy(t->y_first, a.y_first, SCREEN_H);
    memcpy(t->y_last, a.y_last, SCREEN_H);
    // geometry the lane mapping relies on
    for (int side = 0; side < 2; ++side) {   // bat strip: 4 destination columns starting at a multiple of 4
        const int x0 = side ? RIGHT_BAT_X : LEFT_BAT_X;
        const int c0 = (a.x_first[x0] / 4) * 4;
        if (a.x_last[x0 + BAT_W - 1] > c0 + 3 || c0 + 3 >= DIM) return false;
        t->bat_c0[side] = (uint32_t)c0;
    }
    for (int y = ARENA_TOP; y + 1 <= ARENA_BOTTOM; ++y) {   // a (clipped) bat touches <= BAT_ROWS rows
        const int y1 = y + BAT_H < ARENA_BOTTOM ? y + BAT_H : ARENA_BOTTOM;
        if (a.y_last[y1 - 1] - a.y_first[y] + 1 > BAT_ROWS) return false;
    }
    for (int x = 0; x < SCREEN_W; ++x) {                    // a ball touches <= 4x4 destination pixels
        const int x1 = x + BALL_SIZE < SCREEN_W ? x + BALL_SIZE : SCREEN_W;
        if (a.x_last[x1 - 1] - a.x_first[x] + 1 > 4) return false;
    }
    for (int y = ARENA_TOP; y < ARENA_BOTTOM; ++y) {
        const int y1 = y + BALL_SIZE < ARENA_BOTTOM ? y + BALL_SIZE : ARENA_BOTTOM;
        if (a.y_last[y1 - 1] - a.y_first[y] + 1 > 4) return false;
    }
    return true;
}

// geometry the four-frames-per-warp kernel relies on: a bat touches at most 4 destination rows and only the first two
// columns of its strip, whose byte offset is even in every row (16-bit store); a ball touches at most 3 x 2 pixels
template <int DIM>
static bool quad_geometry_ok(const AreaTabs& a) {
    if (DIM % 2) return false;
    for (int side = 0; side < 2; ++side) {
        const int x0 = side ? RIGHT_BAT_X : LEFT_BAT_X;
        const int c0 = (a.x_first[x0] / 4) * 4;
        if (a.x_first[x0] != c0 || a.x_last[x0 + BAT_W - 1] > c0 + 1) return false;
    }
    for (int y = ARENA_TOP; y + 1 <= ARENA_BOTTOM; ++y) {
        const int y1 = y + BAT_H < ARENA_BOTTOM ? y + BAT_H : ARENA_BOTTOM;
        if (a.y_last[y1 - 1] - a.y_first[y] + 1 > 4) return false;
    }
    for (int x = 0; x < SCREEN_W; ++x) {
        const int x1 = x + BALL_SIZE < SCREEN_W ? x + BALL_SIZE : SCREEN_W;
        if (a.x_last[x1 - 1] - a.x_first[x] + 1 > 4) return false;
    }
    for (int y = ARENA_TOP; y < ARENA_BOTTOM; ++y) {
        const int y1 = y + BALL_SIZE < ARENA_BOTTOM ? y + BALL_SIZE : ARENA_BOTTOM;
        if (a.y_last[y1 - 1] - a.y_first[y] + 1 > 2) return false;
    }
    return true;
}

bool pong_quad_ok(const AreaTabs& a) { return a.dim == 42 && quad_geometry_ok<42>(a); }

template <int DIM>
static size_t quad_smem_bytes() {
    return sizeof(QuadTabs<DIM>) + (size_t)QUAD_WARPS * 4 * DIM * DIM;
}

template <int DIM>
static size_t fast_smem_bytes() {
    constexpr int FB = ((DIM * DIM + 15) / 16) * 16;
    return sizeof(FastTabs<DIM>) + (size_t)FAST_WARPS * FB;
}

size_t pong_fast_tabs_bytes(int dim) {
    return dim == 84 ? sizeof(FastTabs<84>) : dim == 42 ? sizeof(FastTabs<42>) : 0;
}

bool pong_fast_tabs_fill(const AreaTabs& a, int text_stride, void* host_buf) {
    if (a.dim == 84) return text_stride <= 96 * 16 && fill_fast_tabs<84>(a, reinterpret_cast<FastTabs<84>*>(host_buf));
    if (a.dim == 42) return text_stride <= 96 * 4 && fill_fast_tabs<42>(a, reinterpret_cast<FastTabs<42>*>(host_buf));
    return false;
}

cudaError_t launch_pong_build_bat_lut(int dim, void* fast_tabs_dev, cudaStream_t s) {
    if (dim == 84) {
        pong_build_bat_lut_kernel<84><<<(2 * 84 * 8 + 127) / 128, 128, 0, s>>>(reinterpret_cast<FastTabs<84>*>(fast_tabs_dev));
        pong_build_xlut_kernel<84><<<(84 * 8 + 127) / 128, 128, 0, s>>>(reinterpret_cast<FastTabs<84>*>(fast_tabs_dev));
    } else if (dim == 42) {
        pong_build_bat_lut_kernel<42><<<(2 * 42 * 32 + 127) / 128, 128, 0, s>>>(reinterpret_cast<FastTabs<42>*>(fast_tabs_dev));
        pong_build_xlut_kernel<42><<<(42 * 32 + 127) / 128, 128, 0, s>>>(reinterpret_cast<FastTabs<42>*>(fast_tabs_dev));
    }
    return cudaGetLastError();
}

// per device (called at handle creation): opt in to the dynamic shared memory size and size the persistent grid
cudaError_t pong_raster_init(int g_grid[3]) {
    cudaError_t e;
    int dev = 0, sms = 0, nb = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    // the instantiations of a size (plain stack, ring; 84x84 also incremental) share the shared-memory size and the
    // register budget (__launch_bounds__), so one occupancy query per size sizes the grid for all of them
    const void* fast[2][2] = {{(const void*)pong_raster_fast_kernel<84, false, false>, (const void*)pong_raster_fast_kernel<84, true, false>},
                              {(const void*)pong_raster_fast_kernel<42, false, false>, (const void*)pong_raster_fast_kernel<42, true, false>}};
    const int smem[2] = {(int)fast_smem_bytes<84>(), (int)fast_smem_bytes<42>()};
    for (int d = 0; d < 2; ++d)
        for (int r = 0; r < 2; ++r)
            if ((e = cudaFuncSetAttribute(fast[d][r], cudaFuncAttributeMaxDynamicSharedMemorySize, smem[d])) != cudaSuccess) return e;
    e = cudaFuncSetAttribute(pong_raster_fast_kernel<84, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem[0]);
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, pong_raster_fast_kernel<84, false, false>, FAST_WARPS * 32, smem[0]);
    if (e != cudaSuccess) return e;
    // 84x84: FastCfg<84>::CTAS per SM.  With uncompressed observation buffers the DRAM write path preferred fewer
    // concurrent write streams (2 CTAs: 0.523 ms per launch, 3: 0.535 ms).  With compressible buffers DRAM is no longer
    // the limit and the kernel gains from the warps that hide its own latency: 3 CTAs 0.4886 ms against 0.4963 ms with 2
    // (B200, 65 536 envs, stack mode; the ring instantiation spills 8 bytes at 3 and lost 2 %, 192.5 against 196.2 M
    // env-steps/s, less than the headline gains)
    g_grid[0] = sms * max(min(nb, FastCfg<84>::CTAS), 1);
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, pong_raster_fast_kernel<42, false, false>, FAST_WARPS * 32, smem[1]);
    if (e != cudaSuccess) return e;
    g_grid[1] = sms * max(nb, 1);
    e = cudaFuncSetAttribute(pong_raster_quad_kernel<42>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)quad_smem_bytes<42>());
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, pong_raster_quad_kernel<42>, QUAD_WARPS * 32, quad_smem_bytes<42>());
    if (e != cudaSuccess) return e;
    g_grid[2] = sms * max(nb, 1);
    return cudaSuccess;
}

static bool fast_path(const PongDev& p, const void* obs0, const void* obs1) {
    const bool aligned = ((uintptr_t)obs0 % 16 == 0) && ((uintptr_t)obs1 % 16 == 0);
    return p.fast_tabs != nullptr && p.fast_ok && aligned && (p.dim == 84 || p.dim == 42);
}

bool pong_raster_incremental_ok(const PongDev& p, const void* obs0, const void* obs1) {
    return fast_path(p, obs0, obs1) && p.dim == 84 && !p.ring;
}

cudaError_t launch_pong_raster(const PongDev& p, const FrameSpec* hist, uint8_t* obs0, uint8_t* obs1, FrameSpec* shown,
                               cudaStream_t s) {
    const long long n_stacks = (long long)p.n * p.n_agents;
    if (n_stacks == 0) return cudaSuccess;
    if (shown && !pong_raster_incremental_ok(p, obs0, obs1)) return cudaErrorInvalidValue;
    if (!fast_path(p, obs0, obs1)) return launch_pong_raster_generic(p, hist, nullptr, p.ring, obs0, obs1, s);
    const long long want = (n_stacks + FAST_WARPS - 1) / FAST_WARPS;
    cudaError_t me = cudaMemsetAsync(p.work_counter, 0, sizeof(unsigned long long), s);
    if (me != cudaSuccess) return me;
    if (p.dim == 84) {
        const unsigned grid = (unsigned)min((long long)p.raster_grid[0], want);
        const FastTabs<84>* tabs = reinterpret_cast<const FastTabs<84>*>(p.fast_tabs);
        if (shown) {
            pong_raster_fast_kernel<84, false, true><<<grid, FAST_WARPS * 32, fast_smem_bytes<84>(), s>>>(p, hist, obs0, obs1, tabs, shown);
        } else if (p.ring) {
            pong_raster_fast_kernel<84, true, false><<<grid, FAST_WARPS * 32, fast_smem_bytes<84>(), s>>>(p, hist, obs0, obs1, tabs, nullptr);
        } else {
            pong_raster_fast_kernel<84, false, false><<<grid, FAST_WARPS * 32, fast_smem_bytes<84>(), s>>>(p, hist, obs0, obs1, tabs, nullptr);
        }
    } else if (p.quad_ok && !p.ring && (long long)p.n * p.c * p.n_agents < (1LL << 31)) {
        const long long quads = (((long long)p.n * p.c + 3) / 4) * p.n_agents;
        const unsigned grid = (unsigned)min((long long)p.raster_grid[2], (quads + 4 * QUAD_WARPS - 1) / (4 * QUAD_WARPS));
        pong_raster_quad_kernel<42><<<grid, QUAD_WARPS * 32, quad_smem_bytes<42>(), s>>>(
            p, hist, obs0, obs1, reinterpret_cast<const FastTabs<42>*>(p.fast_tabs));
    } else {
        const unsigned grid = (unsigned)min((long long)p.raster_grid[1], want);
        const FastTabs<42>* tabs = reinterpret_cast<const FastTabs<42>*>(p.fast_tabs);
        if (p.ring) pong_raster_fast_kernel<42, true, false><<<grid, FAST_WARPS * 32, fast_smem_bytes<42>(), s>>>(p, hist, obs0, obs1, tabs, nullptr);
        else pong_raster_fast_kernel<42, false, false><<<grid, FAST_WARPS * 32, fast_smem_bytes<42>(), s>>>(p, hist, obs0, obs1, tabs, nullptr);
    }
    return cudaGetLastError();
}

}  // namespace crl
