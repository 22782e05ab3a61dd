// pong_opponent.cu -- per-env built-in opponents of cPongTournament-v0 (include/crl_b200.h, crl_pong_opp_*).
//
// Replaces, for a batch in which every env plays its own opponent, what TournamentEnvWrapper + policy_serving.Policy
// (competitive_rl/pong/competitive_pong_env.py:9-53, utils/policy_serving.py:10-66) do for one opponent per batch.
// One launch of pong_opp_act_kernel per wrapper step, no host synchronisation:
//   1. episode bookkeeping of the step before: agent 0's clipped reward is summed per env; an env that finished credits
//      the episode to its opponent (win / draw / loss of agent 0, as pong/evaluate.py:53-88 classifies) and, with
//      resample, draws its next opponent from the pool;
//   2. frame stack: agent 1's newest 42x42 frame goes into the env's uint8 4-frame ring (whatever its opponent is);
//   3. action into column 1 of the int32 (N, 2) step buffer: 999 for RULE_BASED, a Philox draw from {0, 1, 2} for
//      RANDOM, or the greedy action of a LightActorCritic network (utils/network.py:73-93) over stack / 255 in fp32.
// The networks run on the SIMT fp32 pipe with explicit __fmaf_rn (the library is compiled with -fmad=false).  Each CTA
// owns a contiguous range of envs; it sorts them by network slot in shared memory and then runs every slot present
// with that slot's weights staged once in shared memory, one env at a time over all its threads.
//
// League mode (crl_pong_opp_set_pairs / crl_pong_opp_act_pairs) is the same kernel instantiated for two seats: env g
// plays pairing g mod P, both seats act from their own stack (seat 0 from agent 0's frames, seat 1 from agent 1's),
// and a finished episode is credited to the pairing.  The per-env thread files one work item per network seat, so a
// slot's weights are still staged once per 64-env chunk whichever seats use it.
//
// Learner mode (crl_pong_opp_load_learner / crl_pong_opp_act_learner) is the one-seat kernel with LEARNER set: seat 1
// is played exactly as above, and seat 0 is a LightActorCritic learner with its own weights (actor and critic) staged
// like a ninth slot, run for every env of the chunk after the pool's slots.  It acts on a FrameStackTensor ring of agent
// 0's frames (zeroed on done), samples its action from the softmax of its logits (or takes the argmax) and writes what
// a PPO rollout stores: the action, its log-probability, the value and the stack it acted on.
//
// Self-play mode (crl_pong_opp_set_selfplay / crl_pong_opp_act_selfplay) is the two-seat kernel with LEARNER set: league
// mode in which a pairing's seat may be the learner instead of a pool entry.  The per-env thread files learner seats in a
// ninth work list, so the learner's image is still staged once per 64-env chunk, and the learner acts on that seat's own
// ring with learner mode's zeroing and sampling (seat 1 draws from a Philox stream of its own).
#include <string.h>

#include <cmath>
#include <vector>

#include "../../include/crl_b200.h"
#include "crl_host.h"
#include "pong_common.cuh"

using namespace crl;

namespace crl {
namespace opp {

constexpr int DIM = 42;
constexpr int FRAME = DIM * DIM;             // 1764 bytes, 441 words
constexpr int FRAME_WORDS = FRAME / 4;
constexpr int STACK = 4;
constexpr int H1 = 20;                       // conv1 4x4 / 2: 42 -> 20
constexpr int H2 = 10;                       // conv2 2x2 / 2: 20 -> 10
constexpr int C1 = 16, C2 = 16;
constexpr int FEATS = C2 * H2 * H2;          // 1600
constexpr int THREADS = 224;                 // 7 warps: conv1 = 200 items of 2 positions x 16 channels
constexpr int SUB = 64;                      // envs a CTA sorts by slot at a time

// A slot's weights in shared memory (floats), transposed at load time so that a thread's 16 output channels of one
// tap are 16 consecutive floats (four broadcast 128-bit loads):
//   W1[64][16]  tap (ci*16 + kh*4 + kw), channel    conv1
//   B1[16]
//   W2[64][16]  tap (ci*4 + kh*2 + kw), channel     conv2
//   B2[16]
//   WA[3][1600] feature (c*100 + y*10 + x)           actor_linear (the flatten order of (16, 10, 10))
//   BA[4]       3 used
constexpr int OFF_W1 = 0, OFF_B1 = OFF_W1 + 64 * C1, OFF_W2 = OFF_B1 + C1, OFF_B2 = OFF_W2 + 64 * C2,
              OFF_WA = OFF_B2 + C2, OFF_BA = OFF_WA + 3 * FEATS, NET_DEV = OFF_BA + 4;
static_assert(NET_DEV % 4 == 0, "slot image is copied as float4");
// the state-dict order of CRL_PONG_OPP_NET_FLOATS (LightActorCritic: conv1.weight, conv1.bias, conv2.weight, conv2.bias,
// critic_linear.weight, critic_linear.bias, actor_linear.weight, actor_linear.bias)
constexpr int SD_W1 = 0, SD_B1 = SD_W1 + C1 * STACK * 16, SD_W2 = SD_B1 + C1, SD_B2 = SD_W2 + C2 * C1 * 4,
              SD_WC = SD_B2 + C2, SD_BC = SD_WC + FEATS, SD_WA = SD_BC + 1, SD_BA = SD_WA + 3 * FEATS, SD_END = SD_BA + 3;
static_assert(SD_END == CRL_PONG_OPP_NET_FLOATS, "flat layout of the header");
// the learner's image: a slot image followed by critic_linear
//   WC[1600]    feature (c*100 + y*10 + x)
//   BC[4]       1 used
constexpr int OFF_WC = NET_DEV, OFF_BC = OFF_WC + FEATS, NET_LRN = OFF_BC + 4;
static_assert(NET_LRN % 4 == 0, "learner image is copied as float4");

// shared memory of the act kernel (floats unless noted); h2 reuses the input stack, which conv1 is done with.  The
// learner kernel stages the larger learner image and reduces 4 sums (3 logits, the value) per warp.
template <bool LEARNER>
struct Smem {
    static constexpr int W = 0, X = W + (LEARNER ? NET_LRN : NET_DEV), HID = X + STACK * FRAME, LUT = HID + C1 * H1 * H1,
                         RS = LEARNER ? 4 : 3, RED = LUT + 256, FLOATS = RED + 8 * RS;
};
// + the work list uint8 [slot][SEATS * SUB] and its counts int [16]; self-play (SEATS == 2, LEARNER) adds a ninth list,
// the learner's, and a byte per env of the chunk: bit `seat` set = zero that seat's ring before the push
template <int SEATS, bool LEARNER>
__host__ __device__ constexpr int work_lists() { return CRL_PONG_OPP_SLOTS + (SEATS == 2 && LEARNER ? 1 : 0); }
template <int SEATS, bool LEARNER = false>
constexpr size_t smem_bytes() {
    return Smem<LEARNER>::FLOATS * sizeof(float) + work_lists<SEATS, LEARNER>() * SUB * SEATS + 16 * sizeof(int) +
           (SEATS == 2 && LEARNER ? SUB : 0);
}
constexpr size_t SMEM_BYTES = smem_bytes<1>();
static_assert(SUB <= 64, "a league work item is (env in chunk) | seat << 6");

constexpr int KIND_RULE = CRL_PONG_OPP_RULE_BASED;   // CRL_PONG_OPP_RANDOM is the other negative kind
constexpr uint8_t PAIR_LEARNER = 255;                 // a learner seat (CRL_PONG_OPP_LEARNER) in the uint8 pairing table
static_assert(CRL_PONG_OPP_MAX_POOL < PAIR_LEARNER, "pool indices and the learner sentinel are distinct");

struct OppArgs {
    int n;
    int pool_size;
    int phase;                // ring slot the newest frame goes to this step; the stack is slots phase+1 .. phase (oldest -> newest)
    int resample;
    int64_t first_env;
    uint64_t seed;
    uint64_t step;            // RANDOM's counter: act calls since the handle was created
    int8_t kind[CRL_PONG_OPP_MAX_POOL];      // CRL_PONG_OPP_RULE_BASED, CRL_PONG_OPP_RANDOM or a network slot
    uint64_t cum[CRL_PONG_OPP_MAX_POOL];     // draw: entry k is the first with r32 < cum[k]
    const uint8_t* obs1;      // [n][1764] agent 1's observation of the previous step
    const float* rew;         // [n][2] or nullptr (no bookkeeping this step)
    const uint8_t* done;      // [n]
    int32_t* actions;         // [n][2], column 1 written
    float* logits;            // [n][3] or nullptr
    int32_t* ids;             // [n]
    uint8_t* stack;           // [n][4][1764]
    float* ret;               // [n] agent 0's summed clipped reward of the episode in progress
    uint32_t* episodes;       // [n] episodes finished since the handle was created (the draw counter)
    unsigned long long* stats;   // [16][4] (league: [P][4]) episodes, wins, draws, losses of agent 0
    const float* nets;        // [8][NET_DEV]
    // league mode only (SEATS == 2); the fields above keep their offsets in the parameter block
    int num_pairs;
    uint8_t pairs[CRL_PONG_OPP_MAX_PAIRS][2];   // pool index of seat 0, seat 1
    const uint8_t* obs0;      // [n][1764] agent 0's observation of the previous step
    uint8_t* stack0;          // [n][4][1764] seat 0's stacks; `stack` holds seat 1's
    // learner mode only (SEATS == 1, LEARNER): obs0 and stack0 above are agent 0's frames and the learner's ring
    int sample;               // != 0: sample the action from the softmax, else the argmax
    const float* learner;     // [NET_LRN]
    float* logp_value;        // [n][2] (self-play: [n][2][2])
    float* learner_logits;    // [n][3] or nullptr
    uint8_t* stack_out;       // [n][4][1764] the stack the learner acted on, oldest -> newest (self-play: [n][2][4][1764])
    // self-play mode only (SEATS == 2, LEARNER): pairs[p][seat] == PAIR_LEARNER is a learner seat, whose logits go to
    // `logits` [n][2][3] like a pool network's
    int clear_rings;          // != 0: every learner seat's ring is zeroed before this act's push (a restart)
};

// Philox streams: (global env, tag) x counter, keyed by the seed.  tag 1 = RANDOM's actions (seat 1), tag 2 = opponent
// draws, tag 3 = RANDOM's actions in seat 0 (league mode), tag 4 = the learner's sampled actions (learner mode, and seat 0
// in self-play mode), tag 5 = the learner's sampled actions in seat 1 (self-play mode).
__device__ __forceinline__ uint32_t opp_rand(uint64_t seed, int64_t g, uint32_t tag, uint64_t ctr) {
    uint32_t r[4];
    philox4x32_10((uint32_t)g, (uint32_t)((uint64_t)g >> 32) ^ (tag << 24), (uint32_t)ctr, (uint32_t)(ctr >> 32),
                  (uint32_t)seed, (uint32_t)(seed >> 32), r);
    return r[0];
}

__device__ __forceinline__ int opp_draw(const OppArgs& a, int64_t g, uint32_t episode) {
    const uint64_t r = opp_rand(a.seed, g, 2u, episode);
    int k = 0;
    while (k < a.pool_size - 1 && r >= a.cum[k]) ++k;
    return k;
}

// The learner's outputs from its fp32 logits l and value v (thread 0): the action (a draw u = r32 * 2^-32 from the tag 4
// stream, or tag 5 for seat 1 in self-play, the first k with u < c_k of the cumulative softmax, or the argmax),
// log pi(action) and the value.  SEATS == 1: seat 0 of learner mode; SEATS == 2: `seat` of self-play mode.
template <int SEATS>
__device__ __forceinline__ void learner_out(const OppArgs& a, int i, int seat, const float (&l)[3], float v) {
    const float mx = fmaxf(fmaxf(l[0], l[1]), l[2]);
    const float e0 = expf(l[0] - mx), e1 = expf(l[1] - mx), e2 = expf(l[2] - mx);
    const float s = (e0 + e1) + e2;
    int act = 0;
    if (a.sample) {
        const float c0 = e0 / s, c1 = c0 + e1 / s;   // action 2 takes the rest, whatever c_2 rounds to
        const uint32_t tag = SEATS == 1 || seat == 0 ? 4u : 5u;
        const double u = (double)opp_rand(a.seed, a.first_env + i, tag, a.step) * 0x1p-32;   // exact, and so is the compare
        act = u < (double)c0 ? 0 : u < (double)c1 ? 1 : 2;
    } else {
        float best = l[0];                     // argmax, ties to the lowest index
        if (l[1] > best) { act = 1; best = l[1]; }
        if (l[2] > best) act = 2;
    }
    const float la = act == 0 ? l[0] : act == 1 ? l[1] : l[2];
    const int o = SEATS == 1 ? i : 2 * i + seat;   // the (env, seat) row
    a.logp_value[2 * o] = la - (mx + logf(s));   // log softmax: l_a - logsumexp(l)
    a.logp_value[2 * o + 1] = v;
    a.actions[SEATS == 1 ? 2 * i : o] = act;
    float* const lgs = SEATS == 1 ? a.learner_logits : a.logits;
    if (lgs) {
        float* lg = lgs + 3 * o;
        lg[0] = l[0]; lg[1] = l[1]; lg[2] = l[2];
    }
}

// SEATS == 1: column 1 of the step buffer (the per-env opponents); SEATS == 2: both columns (league mode).
// LEARNER, SEATS == 1: column 0 too, from the learner's network (learner mode).
// LEARNER, SEATS == 2: a seat of any pairing may be the learner's (self-play mode).
template <int SEATS, bool LEARNER>
__global__ void __launch_bounds__(THREADS, 2) pong_opp_act_kernel(const OppArgs a) {
    using L = Smem<LEARNER>;
    constexpr bool SELF = SEATS == 2 && LEARNER;
    constexpr int NS = CRL_PONG_OPP_SLOTS + (LEARNER ? 1 : 0);   // the learner is slot CRL_PONG_OPP_SLOTS
    constexpr int NL = work_lists<SEATS, LEARNER>();
    extern __shared__ __align__(16) float sm[];
    float* const w = sm + L::W;
    float* const xs = sm + L::X;
    float* const h1 = sm + L::HID;
    float* const h2 = xs;
    float* const lut = sm + L::LUT;
    float* const red = sm + L::RED;
    uint8_t* const list = (uint8_t*)(sm + L::FLOATS);                     // [slot][SEATS * SUB]
    int* const cnt = (int*)(list + NL * SUB * SEATS);                   // [slot]
    uint8_t* const zero = (uint8_t*)(cnt + 16);                          // self-play: [SUB] rings to zero, bit per seat
    const int tid = threadIdx.x;

    for (int b = tid; b < 256; b += THREADS) lut[b] = (float)b / 255.0f;
    const int r0 = (int)((int64_t)a.n * blockIdx.x / gridDim.x), r1 = (int)((int64_t)a.n * (blockIdx.x + 1) / gridDim.x);
    for (int e0 = r0; e0 < r1; e0 += SUB) {
        const int ne = min(SUB, r1 - e0);
        if (tid < NL) cnt[tid] = 0;
        __syncthreads();
        // ---- per env: bookkeeping of the step before, redraw, actions of the non-network kinds, sort by slot
        if (SEATS == 1 && tid < ne) {
            const int i = e0 + tid;
            const int64_t g = a.first_env + i;
            int id = a.ids[i];
            if (a.rew) {
                float r = a.ret[i] + a.rew[2 * i];
                if (a.done[i]) {
                    unsigned long long* st = a.stats + 4 * id;
                    atomicAdd(st, 1ull);
                    atomicAdd(st + (r > 0.f ? 1 : r == 0.f ? 2 : 3), 1ull);
                    r = 0.f;
                    const uint32_t ep = a.episodes[i] + 1u;
                    a.episodes[i] = ep;
                    if (a.resample) {
                        id = opp_draw(a, g, ep);
                        a.ids[i] = id;
                    }
                }
                a.ret[i] = r;
            }
            const int kind = a.kind[id];
            if (kind >= 0) {
                list[kind * SUB + atomicAdd(&cnt[kind], 1)] = (uint8_t)tid;
            } else {
                a.actions[2 * i + 1] = kind == KIND_RULE ? CHEAT_CODES
                                                         : (int32_t)(((uint64_t)opp_rand(a.seed, g, 1u, a.step) * 3u) >> 32);
                if (a.logits) a.logits[3 * i] = a.logits[3 * i + 1] = a.logits[3 * i + 2] = 0.f;
            }
        }
        if (SEATS == 2 && tid < ne) {   // league: the env's pairing is fixed by its global index
            const int i = e0 + tid;
            const int64_t g = a.first_env + i;
            int64_t pr = g % a.num_pairs;
            if (pr < 0) pr += a.num_pairs;
            const int p = (int)pr;
            if (a.rew) {
                float r = a.ret[i] + a.rew[2 * i];
                if (a.done[i]) {
                    unsigned long long* st = a.stats + 4 * p;
                    atomicAdd(st, 1ull);
                    atomicAdd(st + (r > 0.f ? 1 : r == 0.f ? 2 : 3), 1ull);
                    r = 0.f;
                }
                a.ret[i] = r;
            }
            int zm = 0;
#pragma unroll
            for (int seat = 0; seat < 2; ++seat) {
                if (SELF && a.pairs[p][seat] == PAIR_LEARNER) {   // before kind[] is indexed
                    list[CRL_PONG_OPP_SLOTS * 2 * SUB + atomicAdd(&cnt[CRL_PONG_OPP_SLOTS], 1)] = (uint8_t)(tid | seat << 6);
                    if (a.clear_rings || (a.done && a.done[i])) zm |= 1 << seat;
                    continue;
                }
                if (SELF) a.logp_value[4 * i + 2 * seat] = a.logp_value[4 * i + 2 * seat + 1] = 0.f;
                const int kind = a.kind[a.pairs[p][seat]];
                if (kind >= 0) {
                    list[kind * 2 * SUB + atomicAdd(&cnt[kind], 1)] = (uint8_t)(tid | seat << 6);
                } else {
                    a.actions[2 * i + seat] =
                        kind == KIND_RULE ? CHEAT_CODES
                                          : (int32_t)(((uint64_t)opp_rand(a.seed, g, seat ? 1u : 3u, a.step) * 3u) >> 32);
                    if (a.logits) {
                        float* lg = a.logits + 6 * i + 3 * seat;
                        lg[0] = lg[1] = lg[2] = 0.f;
                    }
                }
            }
            if (SELF) zero[tid] = (uint8_t)zm;
        }
        if (SELF) __syncthreads();   // the push below reads `zero`
        // ---- the newest frame into ring slot `phase` of every env of the range (league: of both seats' stacks;
        //      learner: of both, and an env whose previous step ended has its learner ring zeroed first; self-play: of
        //      both, and a learner seat's ring is zeroed first after a done or a restart)
#pragma unroll
        for (int seat = SEATS == 2 || LEARNER ? 0 : 1; seat < 2; ++seat) {
            const uint32_t* src = (const uint32_t*)((seat ? a.obs1 : a.obs0) + (size_t)e0 * FRAME);
            uint32_t* dst = (uint32_t*)((seat ? a.stack : a.stack0) + (size_t)e0 * STACK * FRAME + (size_t)a.phase * FRAME);
            for (int k = tid; k < ne * FRAME_WORDS; k += THREADS) {
                const int e = k / FRAME_WORDS, j = k - e * FRAME_WORDS;
                dst[(size_t)e * STACK * FRAME_WORDS + j] = src[k];
                if (LEARNER && (SELF ? (zero[e] >> seat & 1) != 0 : seat == 0 && a.done && a.done[e0 + e])) {
                    uint32_t* ring = (uint32_t*)((seat ? a.stack : a.stack0) + (size_t)(e0 + e) * STACK * FRAME);
#pragma unroll
                    for (int d = 1; d < STACK; ++d) ring[((a.phase + d) & 3) * FRAME_WORDS + j] = 0u;
                }
            }
        }
        __syncthreads();
        // ---- networks, slot by slot (learner mode: then the learner, for every env of the range)
        for (int s = 0; s < NS; ++s) {
            const bool lrn = LEARNER && s == CRL_PONG_OPP_SLOTS;
            const int m = lrn && !SELF ? ne : cnt[s];
            if (m == 0) continue;
            if (lrn) {
                const float4* src = (const float4*)a.learner;
                for (int k = tid; k < NET_LRN / 4; k += THREADS) ((float4*)w)[k] = src[k];
            } else {
                const float4* src = (const float4*)(a.nets + (size_t)s * NET_DEV);
                for (int k = tid; k < NET_DEV / 4; k += THREADS) ((float4*)w)[k] = src[k];
            }
            for (int q = 0; q < m; ++q) {
                const int item = lrn && !SELF ? q : list[s * SEATS * SUB + q];
                const int i = e0 + (SEATS == 1 ? item : item & (SUB - 1));
                const int seat = lrn && !SELF ? 0 : SEATS == 1 ? 1 : item >> 6;
                {   // stack / 255 -> xs[ci][42][42], ci 0 = oldest (the learner's bytes also go to stack_out)
                    const uint32_t* src = (const uint32_t*)(((SEATS == 1 && !LEARNER) || seat ? a.stack : a.stack0) + (size_t)i * STACK * FRAME);
                    for (int k = tid; k < STACK * FRAME_WORDS; k += THREADS) {
                        const int ci = k / FRAME_WORDS, j = k - ci * FRAME_WORDS;
                        const uint32_t v = src[((a.phase + 1 + ci) & 3) * FRAME_WORDS + j];
                        if (lrn) ((uint32_t*)a.stack_out)[(size_t)(SELF ? 2 * i + seat : i) * STACK * FRAME_WORDS + k] = v;
                        float4 f;
                        f.x = lut[v & 255]; f.y = lut[(v >> 8) & 255]; f.z = lut[(v >> 16) & 255]; f.w = lut[v >> 24];
                        *(float4*)&xs[ci * FRAME + 4 * j] = f;
                    }
                }
                __syncthreads();
                if (tid < H1 * H1 / 2) {   // conv1 + relu: positions (oy, ox) and (oy, ox + 10), all 16 channels
                    const int oy = tid / 10, ox = tid - oy * 10;
                    float acc0[C1], acc1[C1];
#pragma unroll
                    for (int c = 0; c < C1; ++c) acc0[c] = acc1[c] = w[OFF_B1 + c];
#pragma unroll 1
                    for (int ci = 0; ci < STACK; ++ci)
#pragma unroll
                        for (int kh = 0; kh < 4; ++kh)
#pragma unroll
                            for (int kw = 0; kw < 4; ++kw) {
                                const float* xp = xs + ci * FRAME + (2 * oy + kh) * DIM + 2 * ox + kw;
                                const float x0 = xp[0], x1 = xp[20];
                                const float4* wp = (const float4*)(w + OFF_W1 + (ci * 16 + kh * 4 + kw) * C1);
#pragma unroll
                                for (int c4 = 0; c4 < C1 / 4; ++c4) {
                                    const float4 wv = wp[c4];
                                    acc0[4 * c4 + 0] = __fmaf_rn(wv.x, x0, acc0[4 * c4 + 0]);
                                    acc0[4 * c4 + 1] = __fmaf_rn(wv.y, x0, acc0[4 * c4 + 1]);
                                    acc0[4 * c4 + 2] = __fmaf_rn(wv.z, x0, acc0[4 * c4 + 2]);
                                    acc0[4 * c4 + 3] = __fmaf_rn(wv.w, x0, acc0[4 * c4 + 3]);
                                    acc1[4 * c4 + 0] = __fmaf_rn(wv.x, x1, acc1[4 * c4 + 0]);
                                    acc1[4 * c4 + 1] = __fmaf_rn(wv.y, x1, acc1[4 * c4 + 1]);
                                    acc1[4 * c4 + 2] = __fmaf_rn(wv.z, x1, acc1[4 * c4 + 2]);
                                    acc1[4 * c4 + 3] = __fmaf_rn(wv.w, x1, acc1[4 * c4 + 3]);
                                }
                            }
#pragma unroll
                    for (int c = 0; c < C1; ++c) {
                        h1[c * H1 * H1 + oy * H1 + ox] = fmaxf(acc0[c], 0.f);
                        h1[c * H1 * H1 + oy * H1 + ox + 10] = fmaxf(acc1[c], 0.f);
                    }
                }
                __syncthreads();
                if (tid < 2 * H2 * H2) {   // conv2 + relu: one position, 8 channels
                    const int half = tid / (H2 * H2), p = tid - half * H2 * H2, oy = p / H2, ox = p - oy * H2;
                    float acc[8];
#pragma unroll
                    for (int c = 0; c < 8; ++c) acc[c] = w[OFF_B2 + half * 8 + c];
#pragma unroll 4
                    for (int ci = 0; ci < C1; ++ci)
#pragma unroll
                        for (int kh = 0; kh < 2; ++kh)
#pragma unroll
                            for (int kw = 0; kw < 2; ++kw) {
                                const float x = h1[ci * H1 * H1 + (2 * oy + kh) * H1 + 2 * ox + kw];
                                const float4* wp = (const float4*)(w + OFF_W2 + (ci * 4 + kh * 2 + kw) * C2 + half * 8);
                                const float4 u = wp[0], v = wp[1];
                                acc[0] = __fmaf_rn(u.x, x, acc[0]); acc[1] = __fmaf_rn(u.y, x, acc[1]);
                                acc[2] = __fmaf_rn(u.z, x, acc[2]); acc[3] = __fmaf_rn(u.w, x, acc[3]);
                                acc[4] = __fmaf_rn(v.x, x, acc[4]); acc[5] = __fmaf_rn(v.y, x, acc[5]);
                                acc[6] = __fmaf_rn(v.z, x, acc[6]); acc[7] = __fmaf_rn(v.w, x, acc[7]);
                            }
#pragma unroll
                    for (int c = 0; c < 8; ++c) h2[(half * 8 + c) * H2 * H2 + p] = fmaxf(acc[c], 0.f);
                }
                __syncthreads();
                {   // actor_linear (learner: and critic_linear): strided partial sums, warp tree, then 7 warp sums in order
                    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
                    for (int f = tid; f < FEATS; f += THREADS) {
                        const float x = h2[f];
                        s0 = __fmaf_rn(w[OFF_WA + f], x, s0);
                        s1 = __fmaf_rn(w[OFF_WA + FEATS + f], x, s1);
                        s2 = __fmaf_rn(w[OFF_WA + 2 * FEATS + f], x, s2);
                        if (lrn) s3 = __fmaf_rn(w[OFF_WC + f], x, s3);
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
                        if (lrn) s3 += __shfl_xor_sync(0xffffffffu, s3, o);
                    }
                    if ((tid & 31) == 0) {
                        red[L::RS * (tid >> 5)] = s0; red[L::RS * (tid >> 5) + 1] = s1; red[L::RS * (tid >> 5) + 2] = s2;
                        if (lrn) red[L::RS * (tid >> 5) + 3] = s3;
                    }
                }
                __syncthreads();
                if (tid == 0) {
                    float l[3];
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        float v = 0.f;
                        for (int wi = 0; wi < THREADS / 32; ++wi) v += red[L::RS * wi + k];
                        l[k] = v + w[OFF_BA + k];
                    }
                    if (lrn) {
                        float v = 0.f;
                        for (int wi = 0; wi < THREADS / 32; ++wi) v += red[L::RS * wi + 3];
                        learner_out<SEATS>(a, i, seat, l, v + w[OFF_BC]);
                        continue;      // the rest of this block is a pool network's; thread 0 joins the next barrier
                    }
                    int act = 0;                       // argmax, ties to the lowest index
                    float best = l[0];
                    if (l[1] > best) { act = 1; best = l[1]; }
                    if (l[2] > best) act = 2;
                    a.actions[2 * i + seat] = act;
                    if (a.logits) {
                        float* lg = a.logits + (SEATS == 1 ? 3 * i : 6 * i + 3 * seat);
                        lg[0] = l[0]; lg[1] = l[1]; lg[2] = l[2];
                    }
                }
            }
            __syncthreads();   // thread 0 is done with this slot's bias before the next slot's weights arrive
        }
    }
}

// explicit assignment (ids already validated on the host) or a draw from the pool for every env
__global__ void pong_opp_draw_kernel(const OppArgs a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.n) a.ids[i] = opp_draw(a, a.first_env + i, a.episodes[i]);
}

}  // namespace opp
}  // namespace crl

using namespace crl::opp;

struct crl_pong_opp {
    int n = 0, device = 0, grid = 0, grid_league = 0, grid_learner = 0, grid_selfplay = 0;
    uint64_t seed = 0;
    int64_t first_env = 0;
    uint64_t steps = 0;
    int phase = 0;
    int pool_size = 0;
    bool assigned = false;
    bool loaded[CRL_PONG_OPP_SLOTS] = {};
    int8_t kind[CRL_PONG_OPP_MAX_POOL] = {};
    uint64_t cum[CRL_PONG_OPP_MAX_POOL] = {};
    DeviceAllocs allocs;
    float* nets = nullptr;
    int32_t* ids = nullptr;
    uint8_t* stack = nullptr;
    float* ret = nullptr;
    uint32_t* episodes = nullptr;
    unsigned long long* stats = nullptr;
    // league mode
    bool league = false;
    int num_pairs = 0;
    uint8_t pairs[CRL_PONG_OPP_MAX_PAIRS][2] = {};
    uint8_t* stack0 = nullptr;                 // seat 0's stacks (league) or the learner's rings, allocated on first use
    unsigned long long* pair_stats = nullptr;  // [CRL_PONG_OPP_MAX_PAIRS][4], allocated by the first crl_pong_opp_set_pairs
    // learner mode
    bool learner = false;
    bool learner_loaded = false;
    float* learner_net = nullptr;              // [NET_LRN]
    // self-play mode: league mode's pairings (a learner seat is PAIR_LEARNER), stacks and statistics
    bool selfplay = false;
    bool clear_rings = false;                  // a restart is pending: the next act zeroes every learner seat's ring
};

static const char* const SELFPLAY_REFUSAL = "self-play mode: use crl_pong_opp_act_selfplay (crl_pong_opp_set_pool leaves it)";

static OppArgs opp_args(const crl_pong_opp* h) {
    OppArgs a;
    memset(&a, 0, sizeof a);
    a.n = h->n; a.pool_size = h->pool_size; a.phase = h->phase; a.first_env = h->first_env; a.seed = h->seed; a.step = h->steps;
    memcpy(a.kind, h->kind, sizeof a.kind);
    memcpy(a.cum, h->cum, sizeof a.cum);
    a.ids = h->ids; a.stack = h->stack; a.ret = h->ret; a.episodes = h->episodes; a.stats = h->stats; a.nets = h->nets;
    return a;
}

extern "C" {

int crl_pong_opp_destroy(crl_pong_opp* h) {
    if (!h) return CRL_OK;
    CrlDeviceGuard guard(h->device);
    h->allocs.free_all();
    delete h;
    return CRL_OK;
}

int crl_pong_opp_create(int32_t num_envs, int32_t device, uint64_t seed, int64_t first_env, crl_pong_opp** out) {
    if (!out) return crl_set_error(CRL_E_INVALID, "null argument");
    *out = nullptr;
    if (num_envs <= 0) return crl_set_error(CRL_E_INVALID, "num_envs must be positive");
    if (int r = crl_check_device(device)) return r;
    CrlDeviceGuard guard(device);
    CUDA_TRY(guard.err);
    crl_pong_opp* h = new crl_pong_opp();
    h->n = num_envs; h->device = device; h->seed = seed; h->first_env = first_env;
    const size_t n = (size_t)num_envs;
    int sms = 0, per_sm = 0, per_sm_league = 0, per_sm_learner = 0, per_sm_selfplay = 0;
    cudaError_t err = cudaSuccess;
    auto alloc = [&](auto** p, size_t count) { if (err == cudaSuccess) err = h->allocs.alloc(p, count); };
    alloc(&h->nets, (size_t)NET_DEV * CRL_PONG_OPP_SLOTS);
    alloc(&h->learner_net, (size_t)NET_LRN);
    alloc(&h->ids, n); alloc(&h->stack, (size_t)STACK * FRAME * n); alloc(&h->ret, n); alloc(&h->episodes, n);
    alloc(&h->stats, 4 * CRL_PONG_OPP_MAX_POOL);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(pong_opp_act_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES);
    if (err == cudaSuccess)
        err = cudaFuncSetAttribute(pong_opp_act_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes<2>());
    if (err == cudaSuccess)
        err = cudaFuncSetAttribute(pong_opp_act_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)smem_bytes<1, true>());
    if (err == cudaSuccess)
        err = cudaFuncSetAttribute(pong_opp_act_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)smem_bytes<2, true>());
    if (err == cudaSuccess) err = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (err == cudaSuccess) err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pong_opp_act_kernel<1, false>, THREADS, SMEM_BYTES);
    if (err == cudaSuccess)
        err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_league, pong_opp_act_kernel<2, false>, THREADS, smem_bytes<2>());
    if (err == cudaSuccess)
        err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_learner, pong_opp_act_kernel<1, true>, THREADS,
                                                            smem_bytes<1, true>());
    if (err == cudaSuccess)
        err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_selfplay, pong_opp_act_kernel<2, true>, THREADS,
                                                            smem_bytes<2, true>());
    if (err == cudaSuccess) err = cudaDeviceSynchronize();
    if (err != cudaSuccess) {
        crl_pong_opp_destroy(h);
        return crl_set_error(CRL_E_CUDA, "crl_pong_opp_create: %s", cudaGetErrorString(err));
    }
    // one resident wave: every CTA owns an equal contiguous range of envs
    h->grid = (int)std::min<int64_t>((int64_t)std::max(per_sm, 1) * sms, num_envs);
    h->grid_league = (int)std::min<int64_t>((int64_t)std::max(per_sm_league, 1) * sms, num_envs);
    h->grid_learner = (int)std::min<int64_t>((int64_t)std::max(per_sm_learner, 1) * sms, num_envs);
    h->grid_selfplay = (int)std::min<int64_t>((int64_t)std::max(per_sm_selfplay, 1) * sms, num_envs);
    *out = h;
    return CRL_OK;
}

int crl_pong_opp_seed(crl_pong_opp* h, uint64_t seed) {
    if (!h) return crl_set_error(CRL_E_INVALID, "null handle");
    h->seed = seed;
    return CRL_OK;
}

// checks a state-dict image and copies it to dst in the device layout: a slot image (NET_DEV floats) or, with the
// critic, the learner's (NET_LRN).  Synchronises the stream.
static int load_image(float* dst, int floats, const float* params_host, size_t count, void* stream) {
    if (!params_host || count != (size_t)CRL_PONG_OPP_NET_FLOATS)
        return crl_set_error(CRL_E_INVALID, "a LightActorCritic parameter image has %d floats (got %zu)", CRL_PONG_OPP_NET_FLOATS, count);
    for (size_t k = 0; k < count; ++k)
        if (!std::isfinite(params_host[k])) return crl_set_error(CRL_E_INVALID, "network parameter %zu is not finite", k);
    std::vector<float> img(floats, 0.f);
    const float* p = params_host;
    for (int co = 0; co < C1; ++co)
        for (int t = 0; t < 64; ++t) img[OFF_W1 + t * C1 + co] = p[SD_W1 + co * 64 + t];     // [co][ci][kh][kw] -> [tap][co]
    for (int co = 0; co < C1; ++co) img[OFF_B1 + co] = p[SD_B1 + co];
    for (int co = 0; co < C2; ++co)
        for (int t = 0; t < 64; ++t) img[OFF_W2 + t * C2 + co] = p[SD_W2 + co * 64 + t];     // [co][ci][kh][kw], 16 x 4 taps
    for (int co = 0; co < C2; ++co) img[OFF_B2 + co] = p[SD_B2 + co];
    for (int k = 0; k < 3 * FEATS; ++k) img[OFF_WA + k] = p[SD_WA + k];
    for (int k = 0; k < 3; ++k) img[OFF_BA + k] = p[SD_BA + k];
    if (floats == NET_LRN) {
        for (int k = 0; k < FEATS; ++k) img[OFF_WC + k] = p[SD_WC + k];
        img[OFF_BC] = p[SD_BC];
    }
    CUDA_TRY(cudaMemcpyAsync(dst, img.data(), sizeof(float) * floats, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    return CRL_OK;
}

int crl_pong_opp_load_net(crl_pong_opp* h, int32_t slot, const float* params_host, size_t count, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (slot < 0 || slot >= CRL_PONG_OPP_SLOTS) return crl_set_error(CRL_E_INVALID, "network slot must be in [0, %d)", CRL_PONG_OPP_SLOTS);
    if (int r = load_image(h->nets + (size_t)slot * NET_DEV, NET_DEV, params_host, count, stream)) return r;
    h->loaded[slot] = true;
    return CRL_OK;
}

int crl_pong_opp_load_learner(crl_pong_opp* h, const float* params_host, size_t count, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (int r = load_image(h->learner_net, NET_LRN, params_host, count, stream)) return r;
    h->learner_loaded = true;
    return CRL_OK;
}

int crl_pong_opp_set_pool(crl_pong_opp* h, const int32_t* kinds_host, const double* weights_host, int32_t pool_size, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (!kinds_host || pool_size < 1 || pool_size > CRL_PONG_OPP_MAX_POOL)
        return crl_set_error(CRL_E_INVALID, "a pool has 1 to %d entries", CRL_PONG_OPP_MAX_POOL);
    double total = 0.0;
    for (int k = 0; k < pool_size; ++k) {
        const int kd = kinds_host[k];
        if (kd != CRL_PONG_OPP_RULE_BASED && kd != CRL_PONG_OPP_RANDOM && (kd < 0 || kd >= CRL_PONG_OPP_SLOTS))
            return crl_set_error(CRL_E_INVALID, "pool entry %d: kind %d is neither RULE_BASED, RANDOM nor a network slot", k, kd);
        if (kd >= 0 && !h->loaded[kd]) return crl_set_error(CRL_E_STATE, "pool entry %d: network slot %d was never loaded", k, kd);
        const double wk = weights_host ? weights_host[k] : 1.0;
        if (!(wk >= 0.0) || !std::isfinite(wk)) return crl_set_error(CRL_E_INVALID, "pool entry %d: weight must be finite and >= 0", k);
        total += wk;
    }
    if (!(total > 0.0)) return crl_set_error(CRL_E_INVALID, "the pool's weights sum to 0");
    double run = 0.0;
    int last = 0;
    for (int k = 0; k < pool_size; ++k)
        if ((weights_host ? weights_host[k] : 1.0) > 0.0) last = k;
    for (int k = 0; k < CRL_PONG_OPP_MAX_POOL; ++k) {
        h->kind[k] = k < pool_size ? (int8_t)kinds_host[k] : (int8_t)CRL_PONG_OPP_RULE_BASED;
        if (k < pool_size) run += weights_host ? weights_host[k] : 1.0;
        // r32 < cum[k] picks entry k first: a zero weight repeats the previous bound and is never drawn
        h->cum[k] = k >= last ? (1ull << 32) : (uint64_t)std::floor(run / total * 4294967296.0);
    }
    h->pool_size = pool_size;
    h->assigned = false;
    h->learner = false;
    CUDA_TRY(cudaMemsetAsync(h->stats, 0, sizeof(unsigned long long) * 4 * CRL_PONG_OPP_MAX_POOL, (cudaStream_t)stream));
    // leaving league or self-play mode: the per-env opponents start as on a fresh handle (the act count runs on)
    if (h->league || h->selfplay) {
        h->league = false;
        h->selfplay = false;
        CUDA_TRY(cudaMemsetAsync(h->ret, 0, sizeof(float) * h->n, (cudaStream_t)stream));
        CUDA_TRY(cudaMemsetAsync(h->stack, 0, (size_t)STACK * FRAME * h->n, (cudaStream_t)stream));
        h->phase = 0;
    }
    return CRL_OK;
}

int crl_pong_opp_assign(crl_pong_opp* h, const int32_t* ids_host, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (h->pool_size == 0) return crl_set_error(CRL_E_STATE, "crl_pong_opp_set_pool first");
    if (ids_host) {
        for (int i = 0; i < h->n; ++i)
            if (ids_host[i] < 0 || ids_host[i] >= h->pool_size)
                return crl_set_error(CRL_E_INVALID, "env %d: opponent id %d is not in [0, %d)", i, ids_host[i], h->pool_size);
        CUDA_TRY(cudaMemcpyAsync(h->ids, ids_host, sizeof(int32_t) * h->n, cudaMemcpyHostToDevice, (cudaStream_t)stream));
        CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    } else {
        LAUNCH((pong_opp_draw_kernel<<<(h->n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(opp_args(h)), cudaGetLastError()), 1);
    }
    h->assigned = true;
    return CRL_OK;
}

int crl_pong_opp_restart(crl_pong_opp* h, int32_t clear_stacks, void* stream) {
    CHECK_HANDLE(h, h->device);
    CUDA_TRY(cudaMemsetAsync(h->ret, 0, sizeof(float) * h->n, (cudaStream_t)stream));
    if (clear_stacks) {
        CUDA_TRY(cudaMemsetAsync(h->stack, 0, (size_t)STACK * FRAME * h->n, (cudaStream_t)stream));
        if (h->stack0) CUDA_TRY(cudaMemsetAsync(h->stack0, 0, (size_t)STACK * FRAME * h->n, (cudaStream_t)stream));
        h->phase = 0;
    } else if (h->learner) {   // a reset starts every learner episode afresh (FrameStackTensor.reset)
        CUDA_TRY(cudaMemsetAsync(h->stack0, 0, (size_t)STACK * FRAME * h->n, (cudaStream_t)stream));
    } else if (h->selfplay) {  // the same for every learner seat; pool seats keep their stacks
        h->clear_rings = true;
    }
    return CRL_OK;
}

int crl_pong_opp_act(crl_pong_opp* h, const uint8_t* obs1_dev, const float* rew_dev, const uint8_t* done_dev, int32_t resample,
                     int32_t* actions_dev, float* logits_dev, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (h->league) return crl_set_error(CRL_E_STATE, "league mode: use crl_pong_opp_act_pairs (crl_pong_opp_set_pool leaves it)");
    if (h->learner) return crl_set_error(CRL_E_STATE, "learner mode: use crl_pong_opp_act_learner (crl_pong_opp_set_pool leaves it)");
    if (h->selfplay) return crl_set_error(CRL_E_STATE, SELFPLAY_REFUSAL);
    if (!h->assigned) return crl_set_error(CRL_E_STATE, "crl_pong_opp_assign after every crl_pong_opp_set_pool");
    if (!obs1_dev || !actions_dev) return crl_set_error(CRL_E_INVALID, "null buffer");
    if ((rew_dev == nullptr) != (done_dev == nullptr)) return crl_set_error(CRL_E_INVALID, "rew_dev and done_dev go together");
    if (((uintptr_t)obs1_dev & 3) != 0) return crl_set_error(CRL_E_INVALID, "obs1_dev must be 4-byte aligned");
    OppArgs a = opp_args(h);
    a.resample = resample ? 1 : 0;
    a.obs1 = obs1_dev; a.rew = rew_dev; a.done = done_dev; a.actions = actions_dev; a.logits = logits_dev;
    LAUNCH((pong_opp_act_kernel<1, false><<<h->grid, THREADS, SMEM_BYTES, (cudaStream_t)stream>>>(a), cudaGetLastError()), 1);
    h->phase = (h->phase + 1) & 3;
    h->steps += 1;
    return CRL_OK;
}

// league and self-play modes: pairs_host validated by the caller (a learner seat is CRL_PONG_OPP_LEARNER).  Allocates
// what the modes share on first use, zeroes the pairing statistics, the reward sums and both stacks of every env, and
// stores the table; the caller sets the mode.
static int enter_pairs(crl_pong_opp* h, const int32_t* pairs_host, int32_t num_pairs, void* stream, const char* who) {
    if (!h->pair_stats) {
        const bool had_stack0 = h->stack0 != nullptr;   // learner mode came first
        cudaError_t err = h->allocs.alloc(&h->pair_stats, 4 * CRL_PONG_OPP_MAX_PAIRS);
        if (err == cudaSuccess && !had_stack0) err = h->allocs.alloc(&h->stack0, (size_t)STACK * FRAME * h->n);
        if (err != cudaSuccess) {   // both or neither: a failed call leaves the handle as it was
            h->allocs.free(h->pair_stats);
            h->pair_stats = nullptr;
            if (!had_stack0) h->stack0 = nullptr;
            return crl_set_error(CRL_E_CUDA, "%s: %s", who, cudaGetErrorString(err));
        }
    }
    const cudaStream_t s = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(h->pair_stats, 0, sizeof(unsigned long long) * 4 * CRL_PONG_OPP_MAX_PAIRS, s));
    CUDA_TRY(cudaMemsetAsync(h->ret, 0, sizeof(float) * h->n, s));
    CUDA_TRY(cudaMemsetAsync(h->stack, 0, (size_t)STACK * FRAME * h->n, s));
    CUDA_TRY(cudaMemsetAsync(h->stack0, 0, (size_t)STACK * FRAME * h->n, s));
    for (int p = 0; p < CRL_PONG_OPP_MAX_PAIRS; ++p)
        for (int seat = 0; seat < 2; ++seat) {
            const int32_t v = p < num_pairs ? pairs_host[2 * p + seat] : 0;
            h->pairs[p][seat] = v == CRL_PONG_OPP_LEARNER ? PAIR_LEARNER : (uint8_t)v;
        }
    h->num_pairs = num_pairs;
    h->phase = 0;
    h->league = false;
    h->learner = false;
    h->selfplay = false;
    h->clear_rings = false;
    return CRL_OK;
}

int crl_pong_opp_set_pairs(crl_pong_opp* h, const int32_t* pairs_host, int32_t num_pairs, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (h->pool_size == 0) return crl_set_error(CRL_E_STATE, "crl_pong_opp_set_pool first");
    if (!pairs_host || num_pairs < 1 || num_pairs > CRL_PONG_OPP_MAX_PAIRS)
        return crl_set_error(CRL_E_INVALID, "a league has 1 to %d pairings", CRL_PONG_OPP_MAX_PAIRS);
    for (int p = 0; p < num_pairs; ++p)
        for (int seat = 0; seat < 2; ++seat)
            if (pairs_host[2 * p + seat] < 0 || pairs_host[2 * p + seat] >= h->pool_size)
                return crl_set_error(CRL_E_INVALID, "pairing %d, seat %d: pool index %d is not in [0, %d)", p, seat,
                                     pairs_host[2 * p + seat], h->pool_size);
    if (int r = enter_pairs(h, pairs_host, num_pairs, stream, "crl_pong_opp_set_pairs")) return r;
    h->league = true;
    return CRL_OK;
}

int crl_pong_opp_set_selfplay(crl_pong_opp* h, const int32_t* pairs_host, int32_t num_pairs, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (h->pool_size == 0) return crl_set_error(CRL_E_STATE, "crl_pong_opp_set_pool first");
    if (!pairs_host || num_pairs < 1 || num_pairs > CRL_PONG_OPP_MAX_PAIRS)
        return crl_set_error(CRL_E_INVALID, "a self-play table has 1 to %d pairings", CRL_PONG_OPP_MAX_PAIRS);
    for (int p = 0; p < num_pairs; ++p)
        for (int seat = 0; seat < 2; ++seat) {
            const int32_t v = pairs_host[2 * p + seat];
            if (v != CRL_PONG_OPP_LEARNER && (v < 0 || v >= h->pool_size))
                return crl_set_error(CRL_E_INVALID,
                                     "pairing %d, seat %d: %d is neither CRL_PONG_OPP_LEARNER nor a pool index in [0, %d)",
                                     p, seat, v, h->pool_size);
        }
    if (int r = enter_pairs(h, pairs_host, num_pairs, stream, "crl_pong_opp_set_selfplay")) return r;
    h->selfplay = true;
    return CRL_OK;
}

int crl_pong_opp_act_pairs(crl_pong_opp* h, const uint8_t* obs0_dev, const uint8_t* obs1_dev, const float* rew_dev,
                           const uint8_t* done_dev, int32_t* actions_dev, float* logits_dev, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (h->selfplay) return crl_set_error(CRL_E_STATE, SELFPLAY_REFUSAL);
    if (!h->league) return crl_set_error(CRL_E_STATE, "crl_pong_opp_set_pairs first (league mode)");
    if (!obs0_dev || !obs1_dev || !actions_dev) return crl_set_error(CRL_E_INVALID, "null buffer");
    if ((rew_dev == nullptr) != (done_dev == nullptr)) return crl_set_error(CRL_E_INVALID, "rew_dev and done_dev go together");
    if (((uintptr_t)obs0_dev & 3) != 0 || ((uintptr_t)obs1_dev & 3) != 0)
        return crl_set_error(CRL_E_INVALID, "obs0_dev and obs1_dev must be 4-byte aligned");
    OppArgs a = opp_args(h);
    a.stats = h->pair_stats;
    a.num_pairs = h->num_pairs;
    memcpy(a.pairs, h->pairs, sizeof a.pairs);
    a.obs0 = obs0_dev; a.obs1 = obs1_dev; a.stack0 = h->stack0;
    a.rew = rew_dev; a.done = done_dev; a.actions = actions_dev; a.logits = logits_dev;
    LAUNCH((pong_opp_act_kernel<2, false><<<h->grid_league, THREADS, smem_bytes<2>(), (cudaStream_t)stream>>>(a), cudaGetLastError()), 1);
    h->phase = (h->phase + 1) & 3;
    h->steps += 1;
    return CRL_OK;
}

int crl_pong_opp_act_learner(crl_pong_opp* h, const uint8_t* obs0_dev, const uint8_t* obs1_dev, const float* rew_dev,
                             const uint8_t* done_dev, int32_t resample, int32_t sample, int32_t* actions_dev,
                             float* logp_value_dev, float* logits_dev, uint8_t* stack_out_dev, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (!h->learner_loaded) return crl_set_error(CRL_E_STATE, "crl_pong_opp_load_learner first");
    if (h->league) return crl_set_error(CRL_E_STATE, "league mode: use crl_pong_opp_act_pairs (crl_pong_opp_set_pool leaves it)");
    if (h->selfplay) return crl_set_error(CRL_E_STATE, SELFPLAY_REFUSAL);
    if (!h->assigned) return crl_set_error(CRL_E_STATE, "crl_pong_opp_assign after every crl_pong_opp_set_pool");
    if (!obs0_dev || !obs1_dev || !actions_dev || !logp_value_dev || !stack_out_dev) return crl_set_error(CRL_E_INVALID, "null buffer");
    if ((rew_dev == nullptr) != (done_dev == nullptr)) return crl_set_error(CRL_E_INVALID, "rew_dev and done_dev go together");
    if (((uintptr_t)obs0_dev & 3) != 0 || ((uintptr_t)obs1_dev & 3) != 0 || ((uintptr_t)stack_out_dev & 3) != 0)
        return crl_set_error(CRL_E_INVALID, "obs0_dev, obs1_dev and stack_out_dev must be 4-byte aligned");
    const cudaStream_t s = (cudaStream_t)stream;
    if (!h->learner) {   // entering learner mode: fresh rings
        if (!h->stack0) {
            const cudaError_t err = h->allocs.alloc(&h->stack0, (size_t)STACK * FRAME * h->n);
            if (err != cudaSuccess) {
                h->stack0 = nullptr;
                return crl_set_error(CRL_E_CUDA, "crl_pong_opp_act_learner: %s", cudaGetErrorString(err));
            }
        }
        CUDA_TRY(cudaMemsetAsync(h->stack0, 0, (size_t)STACK * FRAME * h->n, s));
        h->learner = true;
    }
    OppArgs a = opp_args(h);
    a.resample = resample ? 1 : 0;
    a.sample = sample ? 1 : 0;
    a.obs0 = obs0_dev; a.obs1 = obs1_dev; a.stack0 = h->stack0; a.learner = h->learner_net;
    a.rew = rew_dev; a.done = done_dev; a.actions = actions_dev;
    a.logp_value = logp_value_dev; a.learner_logits = logits_dev; a.stack_out = stack_out_dev;
    LAUNCH((pong_opp_act_kernel<1, true><<<h->grid_learner, THREADS, smem_bytes<1, true>(), s>>>(a), cudaGetLastError()), 1);
    h->phase = (h->phase + 1) & 3;
    h->steps += 1;
    return CRL_OK;
}

int crl_pong_opp_act_selfplay(crl_pong_opp* h, const uint8_t* obs0_dev, const uint8_t* obs1_dev, const float* rew_dev,
                              const uint8_t* done_dev, int32_t sample, int32_t* actions_dev, float* logp_value_dev,
                              float* logits_dev, uint8_t* stack_out_dev, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (!h->selfplay) return crl_set_error(CRL_E_STATE, "crl_pong_opp_set_selfplay first (self-play mode)");
    if (!h->learner_loaded) return crl_set_error(CRL_E_STATE, "crl_pong_opp_load_learner first");
    if (!obs0_dev || !obs1_dev || !actions_dev || !logp_value_dev || !stack_out_dev) return crl_set_error(CRL_E_INVALID, "null buffer");
    if ((rew_dev == nullptr) != (done_dev == nullptr)) return crl_set_error(CRL_E_INVALID, "rew_dev and done_dev go together");
    if (((uintptr_t)obs0_dev & 3) != 0 || ((uintptr_t)obs1_dev & 3) != 0 || ((uintptr_t)stack_out_dev & 3) != 0)
        return crl_set_error(CRL_E_INVALID, "obs0_dev, obs1_dev and stack_out_dev must be 4-byte aligned");
    OppArgs a = opp_args(h);
    a.stats = h->pair_stats;
    a.num_pairs = h->num_pairs;
    memcpy(a.pairs, h->pairs, sizeof a.pairs);
    a.sample = sample ? 1 : 0;
    a.clear_rings = h->clear_rings ? 1 : 0;
    a.obs0 = obs0_dev; a.obs1 = obs1_dev; a.stack0 = h->stack0; a.learner = h->learner_net;
    a.rew = rew_dev; a.done = done_dev; a.actions = actions_dev; a.logits = logits_dev;
    a.logp_value = logp_value_dev; a.stack_out = stack_out_dev;
    LAUNCH((pong_opp_act_kernel<2, true><<<h->grid_selfplay, THREADS, smem_bytes<2, true>(), (cudaStream_t)stream>>>(a),
            cudaGetLastError()), 1);
    h->clear_rings = false;
    h->phase = (h->phase + 1) & 3;
    h->steps += 1;
    return CRL_OK;
}

int crl_pong_opp_get_pair_stats(crl_pong_opp* h, uint64_t* stats_host, int32_t num_pairs, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (!stats_host) return crl_set_error(CRL_E_INVALID, "null buffer");
    if (num_pairs < 1 || num_pairs > CRL_PONG_OPP_MAX_PAIRS)
        return crl_set_error(CRL_E_INVALID, "num_pairs must be in [1, %d]", CRL_PONG_OPP_MAX_PAIRS);
    if (!h->pair_stats) return crl_set_error(CRL_E_STATE, "crl_pong_opp_set_pairs first (league mode)");
    return crl_read_counters(h->pair_stats, stats_host, 4 * num_pairs, (cudaStream_t)stream);
}

int crl_pong_opp_get_ids(crl_pong_opp* h, int32_t* ids_dev, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (!ids_dev) return crl_set_error(CRL_E_INVALID, "null buffer");
    CUDA_TRY(cudaMemcpyAsync(ids_dev, h->ids, sizeof(int32_t) * h->n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return CRL_OK;
}

int crl_pong_opp_get_stats(crl_pong_opp* h, uint64_t* stats_host, void* stream) {
    CHECK_HANDLE(h, h->device);
    if (!stats_host) return crl_set_error(CRL_E_INVALID, "null buffer");
    return crl_read_counters(h->stats, stats_host, 4 * CRL_PONG_OPP_MAX_POOL, (cudaStream_t)stream);
}

}  // extern "C"
