// car_physics.cu -- cCarRacing game core: track generation + reset (one warp per env, the next track ahead of time),
// the wheel-tile sensor overlaps (one thread per wheel) and the car-car manifolds (one thread per fixture pair) ahead of
// the step, and the per-step pipeline (one thread per car): action decode, wheel model, contact events / tile reward,
// Box2D-style joint + contact solver, done / TimeLimit logic.
//
// Replaces (paths relative to /root/reference/competitive_rl/):
//   car_racing/car_racing_multi_players.py  _create_track (262-452), reset (454-525), process_action (527-540),
//                                           step (542-620), FrictionDetector._contact (111-153)
//   car_racing/car_dynamics.py              Car.__init__ (55-129), gas/brake/steer (131-157), step (159-234)
//   car_racing/register.py                  max_episode_steps=1000 (gym TimeLimit) (8-26)
//   box2d-py 2.3 (un-vendored)              b2World::Step(1/50, 180, 60): b2Island::Solve + b2RevoluteJoint,
//                                           polygon mass data, sensor overlap -- restated from the published
//                                           algorithm (parity vs a real Box2D is unpinned, DESIGN.md section 9)
//
// Arithmetic: solver in fp32 exactly as Box2D (b2 float32), un-fused (-fmad=false); the Python-level
// wheel model and the track generator in fp64 like the reference's Python floats.
#include <math.h>

#include "car_common.cuh"
#include "car_spans.cuh"

namespace crl {

// ---- constants (car_dynamics.py:17-41, car_racing_multi_players.py:54-72) ----
#define CR_SIZE 0.02
#define CR_ENGINE_POWER (100000000 * CR_SIZE * CR_SIZE)
#define CR_WHEEL_MOI (4000 * CR_SIZE * CR_SIZE)
#define CR_FRICTION_LIMIT (1000000 * CR_SIZE * CR_SIZE)
#define CR_WHEEL_R 27
#define CR_WHEEL_W 14
#define CR_SCALE 6.0
#define CR_TRACK_RAD (900.0 / CR_SCALE)
#define CR_PLAYFIELD (2000.0 / CR_SCALE)
#define CR_FPS 50
#define CR_TRACK_DETAIL_STEP (21.0 / CR_SCALE)
#define CR_TRACK_TURN_RATE 0.31
#define CR_TRACK_WIDTH (40.0 / CR_SCALE)
#define CR_BORDER (8.0 / CR_SCALE)
#define CR_BORDER_MIN_COUNT 4
#define CR_PI 3.141592653589793

// Box2D 2.3 b2Settings.h
#define B2_PI 3.14159265359f
#define B2_LINEAR_SLOP 0.005f
#define B2_ANGULAR_SLOP (2.0f / 180.0f * B2_PI)
#define B2_POLYGON_RADIUS (2.0f * B2_LINEAR_SLOP)
#define B2_MAX_ANGULAR_CORRECTION (8.0f / 180.0f * B2_PI)
#define B2_MAX_TRANSLATION 2.0f
#define B2_MAX_ROTATION (0.5f * B2_PI)
#define B2_TIME_TO_SLEEP 0.5f
#define B2_LINEAR_SLEEP_TOL 0.01f
#define B2_ANGULAR_SLEEP_TOL (2.0f / 180.0f * B2_PI)

__constant__ float c_wheelpos[4][2] = {{-55, +80}, {+55, +80}, {-55, -82}, {+55, -82}};

struct F2 { float x, y; };
__device__ __forceinline__ F2 f2(float x, float y) { F2 r; r.x = x; r.y = y; return r; }
__device__ __forceinline__ F2 operator+(F2 a, F2 b) { return f2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ F2 operator-(F2 a, F2 b) { return f2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ F2 operator*(float s, F2 a) { return f2(s * a.x, s * a.y); }
__device__ __forceinline__ float dot(F2 a, F2 b) { return a.x * b.x + a.y * b.y; }
__device__ __forceinline__ float cross(F2 a, F2 b) { return a.x * b.y - a.y * b.x; }
__device__ __forceinline__ F2 cross_sv(float s, F2 a) { return f2(-s * a.y, s * a.x); }
struct Rot { float s, c; };
__device__ __forceinline__ Rot make_rot(float a) { Rot r; sincosf(a, &r.s, &r.c); return r; }
__device__ __forceinline__ F2 rmul(Rot q, F2 v) { return f2(q.c * v.x - q.s * v.y, q.s * v.x + q.c * v.y); }
__device__ __forceinline__ float clampf(float a, float lo, float hi) { return a < lo ? lo : (a > hi ? hi : a); }
__device__ __forceinline__ double signd(double v) { return (double)((v > 0) - (v < 0)); }

}  // namespace crl
#include "car_contact.cuh"
namespace crl {

// ------------------------------------------------------------------------------------------------
// track generator (fp64): one walk of the curve follower (_create_track :262-375), run by ONE lane.  The reference keeps
// all raw points and slices track[i1 : i2 - 1] afterwards (i2 = last, i1 = previous crossing of start_alpha).  Here the
// last CAR_RAW_RING raw points go to a ring in global memory (fire-and-forget stores off the dependent chain), which holds
// the slice whenever the walk ends within a lap of the last crossing -- always, unless the follower got stuck; then
// `emit_from/emit_to` select the raw points a second walk writes out.
struct WalkResult { int n_raw, i1, i2; };

__device__ WalkResult track_walk(const double* draws, double* ring /* [CAR_RAW_RING][3] or nullptr */, int emit_from, int emit_to,
                                 double* out /* [][3] beta,x,y or nullptr */) {
    double cp_alpha[CAR_CHECKPOINTS], cp_x[CAR_CHECKPOINTS], cp_y[CAR_CHECKPOINTS];
    double start_alpha = 0.0;
    for (int c = 0; c < CAR_CHECKPOINTS; ++c) {
        double alpha = 2 * CR_PI * c / CAR_CHECKPOINTS + draws[2 * c];
        double rad = draws[2 * c + 1];
        if (c == 0) { alpha = 0; rad = 1.5 * CR_TRACK_RAD; }
        if (c == CAR_CHECKPOINTS - 1) {
            alpha = 2 * CR_PI * c / CAR_CHECKPOINTS;
            start_alpha = 2 * CR_PI * (-0.5) / CAR_CHECKPOINTS;
            rad = 1.5 * CR_TRACK_RAD;
        }
        cp_alpha[c] = alpha; cp_x[c] = rad * cos(alpha); cp_y[c] = rad * sin(alpha);
    }
    double x = 1.5 * CR_TRACK_RAD, y = 0, beta = 0, prev_alpha = 0;
    int dest_i = 0, laps = 0, no_freeze = 2500, visited_other_side = 0, n_raw = 0;
    int last_cross = -1, prev_cross = -1;
    for (;;) {
        double alpha = atan2(y, x);
        if (visited_other_side && alpha > 0) { laps += 1; visited_other_side = 0; }
        if (alpha < 0) { visited_other_side = 1; alpha += 2 * CR_PI; }
        double dest_x, dest_y;
        for (;;) {
            bool failed = true;
            for (;;) {
                const int k = dest_i % CAR_CHECKPOINTS;
                dest_x = cp_x[k]; dest_y = cp_y[k];
                if (alpha <= cp_alpha[k]) { failed = false; break; }
                dest_i += 1;
                if (dest_i % CAR_CHECKPOINTS == 0) break;
            }
            if (!failed) break;
            alpha -= 2 * CR_PI;
        }
        const double r1x = cos(beta), r1y = sin(beta);
        const double p1x = -r1y, p1y = r1x;
        double proj = r1x * (dest_x - x) + r1y * (dest_y - y);
        while (beta - alpha > 1.5 * CR_PI) beta -= 2 * CR_PI;
        while (beta - alpha < -1.5 * CR_PI) beta += 2 * CR_PI;
        const double prev_beta = beta;
        proj *= CR_SCALE;
        if (proj > 0.3) beta -= fmin(CR_TRACK_TURN_RATE, fabs(0.001 * proj));
        if (proj < -0.3) beta += fmin(CR_TRACK_TURN_RATE, fabs(0.001 * proj));
        x += p1x * CR_TRACK_DETAIL_STEP;
        y += p1y * CR_TRACK_DETAIL_STEP;
        // raw point n_raw = (alpha, prev_beta*0.5 + beta*0.5, x, y)
        if (n_raw >= 1 && alpha > start_alpha && prev_alpha <= start_alpha) { prev_cross = last_cross; last_cross = n_raw; }
        if (ring != nullptr) {
            double* o = ring + 3 * (n_raw & (CAR_RAW_RING - 1));
            o[0] = prev_beta * 0.5 + beta * 0.5; o[1] = x; o[2] = y;
        }
        if (out != nullptr && n_raw >= emit_from && n_raw < emit_to) {
            double* o = out + 3 * (n_raw - emit_from);
            o[0] = prev_beta * 0.5 + beta * 0.5; o[1] = x; o[2] = y;
        }
        prev_alpha = alpha;
        n_raw += 1;
        if (laps > 4) break;
        no_freeze -= 1;
        if (no_freeze == 0) break;
    }
    WalkResult r;
    r.n_raw = n_raw; r.i2 = last_cross; r.i1 = prev_cross;
    return r;
}

// b2PolygonShape::Set hull of 5 points (gift wrapping, fp32)
__device__ int convex_hull5(const float* px, const float* py, float* ox, float* oy) {
    float qx[5], qy[5];
    int m = 0;
    for (int i = 0; i < 5; ++i) {
        bool unique = true;
        for (int k = 0; k < m; ++k) {
            const float dx = px[i] - qx[k], dy = py[i] - qy[k];
            if (dx * dx + dy * dy < 0.5f * B2_LINEAR_SLOP * 0.5f * B2_LINEAR_SLOP) { unique = false; break; }
        }
        if (unique) { qx[m] = px[i]; qy[m] = py[i]; ++m; }
    }
    if (m < 3) return 0;
    int i0 = 0;
    for (int i = 1; i < m; ++i)
        if (qx[i] > qx[i0] || (qx[i] == qx[i0] && qy[i] < qy[i0])) i0 = i;
    int hull[5], cnt = 0, ih = i0;
    for (;;) {
        hull[cnt] = ih;
        int ie = 0;
        for (int j = 1; j < m; ++j) {
            if (ie == ih) { ie = j; continue; }
            const float rx = qx[ie] - qx[hull[cnt]], ry = qy[ie] - qy[hull[cnt]];
            const float vx = qx[j] - qx[hull[cnt]], vy = qy[j] - qy[hull[cnt]];
            const float c = rx * vy - ry * vx;
            if (c < 0.0f) ie = j;
            if (c == 0.0f && vx * vx + vy * vy > rx * rx + ry * ry) ie = j;
        }
        ++cnt;
        ih = ie;
        if (ie == i0 || cnt >= 5) break;
    }
    for (int i = 0; i < cnt; ++i) { ox[i] = qx[hull[i]]; oy[i] = qy[hull[i]]; }
    return cnt;
}

// Car.__init__ (car_dynamics.py:55-129) of car `ci` at the track start, by the 32 lanes of a warp
__device__ void car_body_reset(const CarDev& p, int ci, double init_angle, double init_x, double init_y, int birth, int lane) {
    init_x -= birth % 2 * 5;
    init_y -= floor((double)(birth / 2)) * 10;
    float* b = p.body + (size_t)ci * 40;
    const CarHullConst* K = p.consts;
    const float a = (float)init_angle;
    if (lane == 0) {
        const Rot q = make_rot(a);
        const F2 lc = rmul(q, f2(K->hull_lcx, K->hull_lcy));
        b[0] = (float)init_x + lc.x; b[1] = (float)init_y + lc.y; b[2] = a; b[3] = b[4] = b[5] = 0.f; b[6] = 0.f; b[7] = 1.f;
    } else if (lane <= 4) {   // wheels are NOT placed rotated (car_dynamics.py:90); the joints pull them in
        const int k = lane - 1;
        float* w = b + 8 * (k + 1);
        w[0] = (float)(init_x + c_wheelpos[k][0] * CR_SIZE); w[1] = (float)(init_y + c_wheelpos[k][1] * CR_SIZE);
        w[2] = a; w[3] = w[4] = w[5] = 0.f; w[6] = 0.f; w[7] = 1.f;
    }
    if (lane < 24) p.joint[(size_t)ci * 24 + lane] = 0.f;
    if (lane < 8) p.wheel[(size_t)ci * 8 + lane] = 0.0;
    if (lane < 2) p.reward[2 * ci + lane] = 0.0;
    if (lane < 4) p.counters[4 * ci + lane] = 0;
    p.touching[(size_t)ci * 64 + lane] = 0u; p.touching[(size_t)ci * 64 + 32 + lane] = 0u;
    if (lane < 16) p.visited[(size_t)ci * 16 + lane] = 0u;
}

// One tile of the track (:399-445): convex hull + edge normals for the physics, road-map pixels for the renderer
__device__ void build_tile(const double* pts, int n, int i, uint8_t border_flag, CarTile* tiles, float2* centres) {
    const double* p1 = pts + 3 * i;
    const double* p2 = pts + 3 * ((i - 1 + n) % n);
    const double b1 = p1[0], x1 = p1[1], y1 = p1[2], b2 = p2[0], x2 = p2[1], y2 = p2[2];
    const double osc = (10 / (100 / sqrt(96.0))) * 1.8;
    const double cb1 = cos(b1), sb1 = sin(b1), cb2 = cos(b2), sb2 = sin(b2);
    const double dvx[5] = {x1 - CR_TRACK_WIDTH * cb1, x1 - CR_TRACK_WIDTH / 2 * cos(b1 - CR_PI / 2),
                           x1 + CR_TRACK_WIDTH * cb1, x2 + CR_TRACK_WIDTH * cb2, x2 - CR_TRACK_WIDTH * cb2};
    const double dvy[5] = {y1 - CR_TRACK_WIDTH * sb1, y1 - CR_TRACK_WIDTH / 2 * sin(b1 - CR_PI / 2),
                           y1 + CR_TRACK_WIDTH * sb1, y2 + CR_TRACK_WIDTH * sb2, y2 - CR_TRACK_WIDTH * sb2};
    float vx[5], vy[5];
    CarTile t;
    for (int k = 0; k < 5; ++k) {
        vx[k] = (float)dvx[k]; vy[k] = (float)dvy[k];
        // road-map pixels of the listed (fp64) vertices: obs_scale * -v + world_size / 2, truncated
        t.mx[k] = (int16_t)(int)(osc * -dvx[k] + 5000.0);
        t.my[k] = (int16_t)(int)(osc * -dvy[k] + 5000.0);
    }
    t.n = (uint8_t)convex_hull5(vx, vy, t.px, t.py);
    for (int k = t.n; k < 5; ++k) { t.px[k] = t.px[0]; t.py[k] = t.py[0]; }
    for (int k = 0; k < 5; ++k) {      // edge normals exactly as max_separation derives them (same fp32 operations)
        t.nx[k] = 3.0e38f; t.ny[k] = 0.f;
        if (k < t.n) {
            const int k2 = (k + 1 == t.n) ? 0 : k + 1;
            const float ex = t.px[k2] - t.px[k], ey = t.py[k2] - t.py[k];
            const float len = sqrtf(ex * ex + ey * ey);
            if (!(len < 1e-12f)) { t.nx[k] = ey / len; t.ny[k] = -ex / len; }
        }
    }
    t.flags = (uint8_t)(1 | (border_flag & 2) | ((i % 2 == 0) ? 4 : 0));
    t.pad = 0;
    t.cx = (float)x1; t.cy = (float)y1;
    centres[i] = make_float2(t.cx, t.cy);
    const double side = signd(b2 - b1);
    const double kdx[4] = {x1 + side * CR_TRACK_WIDTH * cb1, x1 + side * (CR_TRACK_WIDTH + CR_BORDER) * cb1,
                           x2 + side * (CR_TRACK_WIDTH + CR_BORDER) * cb2, x2 + side * CR_TRACK_WIDTH * cb2};
    const double kdy[4] = {y1 + side * CR_TRACK_WIDTH * sb1, y1 + side * (CR_TRACK_WIDTH + CR_BORDER) * sb1,
                           y2 + side * (CR_TRACK_WIDTH + CR_BORDER) * sb2, y2 + side * CR_TRACK_WIDTH * sb2};
    for (int k = 0; k < 4; ++k) {
        t.kmx[k] = (int16_t)(int)(osc * -kdx[k] + 5000.0);
        t.kmy[k] = (int16_t)(int)(osc * -kdy[k] + 5000.0);
    }
    tiles[i] = t;
}

// CarRacing.reset's track loop (:499-507) for env e into track slot `slot`, by one warp: lane 0 retries _create_track until
// an attempt succeeds (the curve walk is a serial fp64 chain); the kerb flags, tiles, prefilter samples and span tables
// that follow are spread over the lanes.  Returns the number of track points; 0 = failed 64 times (flagged);
// -1 = (for_pregen only) the injected draw table has no attempt left, nothing was written or consumed.
__device__ int generate_track_warp(const CarDev& p, int e, int slot, bool for_pregen, int lane) {
    double* pts = p.track_pts + (size_t)slot * CAR_MAX_TRACK * 3;
    CarTile* tiles = p.tiles + (size_t)slot * CAR_MAX_TRACK;
    float2* centres = p.tile_centres + (size_t)slot * CAR_MAX_TRACK;
    double* ring = p.raw_ring + (size_t)e * CAR_RAW_RING * 3;
    const uint64_t gi = (uint64_t)(p.first_env + e);
    int n = 0, ring_from = -1;
    if (p.fixed_tracks != nullptr && p.n_fixed > 0) {       // replay of a recorded track: no generation, no draws consumed
        const int k = (int)(gi % (uint64_t)p.n_fixed);
        n = min(max(p.fixed_counts[k], 0), CAR_MAX_TRACK);
        const double* src = p.fixed_tracks + (size_t)k * CAR_MAX_TRACK * 3;
        for (int i = lane; i < 3 * n; i += 32) pts[i] = src[i];
    } else {
        if (lane == 0) {
            for (int guard = 0; guard < 64 && n == 0; ++guard) {
                double draws[CAR_DRAWS];
                const int att = p.attempt_count[e];
                if (p.track_draws != nullptr) {
                    int k = att;
                    if (k >= p.k_draws) {
                        if (for_pregen) { n = -1; break; }          // the table is not ours to overrun ahead of time
                        *p.overrun = 1; k = p.k_draws - 1;
                    }
                    for (int i = 0; i < CAR_DRAWS; ++i) draws[i] = p.track_draws[((size_t)e * p.k_draws + k) * CAR_DRAWS + i];
                } else {
                    for (int i = 0; i < CAR_DRAWS; i += 2) {   // noise ~ U(0, 2pi/12), rad ~ U(R/3, R), :268-270
                        uint32_t r[4];
                        philox4x32_10((uint32_t)att, (uint32_t)(i / 2), (uint32_t)gi, (uint32_t)(gi >> 32), (uint32_t)p.seed,
                                      (uint32_t)(p.seed >> 32) ^ 0xC0FFEEu, r);
                        const double u0 = (double)((((uint64_t)r[0] >> 5) << 26) | ((uint64_t)r[1] >> 6)) * (1.0 / 9007199254740992.0);
                        const double u1 = (double)((((uint64_t)r[2] >> 5) << 26) | ((uint64_t)r[3] >> 6)) * (1.0 / 9007199254740992.0);
                        draws[i] = 0.0 + (2 * CR_PI * 1 / CAR_CHECKPOINTS - 0.0) * u0;
                        draws[i + 1] = CR_TRACK_RAD / 3 + (CR_TRACK_RAD - CR_TRACK_RAD / 3) * u1;
                    }
                }
                p.attempt_count[e] = att + 1;
                const WalkResult w = track_walk(draws, ring, 0, 0, nullptr);
                if (w.i1 < 0 || w.i2 < 0) continue;               // "return False  # Failed"
                const int cnt = (w.i2 - 1) - w.i1;                // track = track[i1:i2 - 1]
                if (cnt <= 8 || cnt > CAR_MAX_TRACK) continue;
                const double *first, *last;
                if (w.n_raw - w.i1 <= CAR_RAW_RING) {             // the slice is still in the ring
                    first = ring + 3 * (w.i1 & (CAR_RAW_RING - 1));
                    last = ring + 3 * ((w.i1 + cnt - 1) & (CAR_RAW_RING - 1));
                    ring_from = w.i1;
                } else {                                          // follower wandered off after its last lap: walk again
                    track_walk(draws, nullptr, w.i1, w.i1 + cnt, pts);
                    first = pts; last = pts + 3 * (cnt - 1);
                    ring_from = -1;
                }
                const double fb = first[0], fpx = cos(fb), fpy = sin(fb);
                const double gx = fpx * (first[1] - last[1]), gy = fpy * (first[2] - last[2]);
                if (sqrt(gx * gx + gy * gy) > CR_TRACK_DETAIL_STEP) continue;   // not well glued together
                n = cnt;
            }
            if (n == 0) *p.overrun = 2;   // cannot happen with sane draws; the env keeps its old track, flagged
        }
        __syncwarp();
        n = __shfl_sync(0xffffffffu, n, 0);
        ring_from = __shfl_sync(0xffffffffu, ring_from, 0);
        if (n <= 0) return n;
        if (ring_from >= 0)
            for (int i = lane; i < 3 * n; i += 32) pts[i] = ring[3 * ((ring_from + i / 3) & (CAR_RAW_RING - 1)) + i % 3];
    }
    __syncwarp();
    if (n <= 0) return 0;
    if (lane == 0) p.n_track[slot] = n;
    // red-white border on hard turns (:383-397): border[] kept in tile.flags bit 1
    for (int i = lane; i < n; i += 32) {
        bool good = true;
        int oneside = 0;
        for (int neg = 0; neg < CR_BORDER_MIN_COUNT; ++neg) {
            const double b1 = pts[3 * (((i - neg - 0) % n + n) % n)], b2 = pts[3 * (((i - neg - 1) % n + n) % n)];
            good = good && fabs(b1 - b2) > CR_TRACK_TURN_RATE * 0.2;
            oneside += (b1 - b2 > 0) - (b1 - b2 < 0);
        }
        good = good && abs(oneside) == CR_BORDER_MIN_COUNT;
        tiles[i].flags = good ? 3 : 1;
    }
    __syncwarp();
    // "border[i - neg] |= border[i]" in place, i ascending (:394-396): the marks i = 0..2 put on the last tiles through the
    // negative indices are seen again when the loop gets there, exactly like the reference's list -- serial, lane 0
    if (lane == 0)
        for (int i = 0; i < n; ++i)
            if (tiles[i].flags & 2)
                for (int neg = 0; neg < CR_BORDER_MIN_COUNT; ++neg) tiles[((i - neg) % n + n) % n].flags |= 2;
    __syncwarp();
    for (int i = lane; i < n; i += 32) build_tile(pts, n, i, tiles[i].flags, tiles, centres);
    for (int i = n + lane; i < CAR_MAX_TRACK; i += 32) tiles[i].flags = 0;
    // the tiles the prefilter's constant radii do not cover (CAR_WIDE_REACH / CAR_WIDE_GROUP), listed with their reach
    float4* wide = p.wide_tiles + (size_t)slot * CAR_MAX_WIDE;
    int n_wide = 0;
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;                       // the lane that built tile i above
        float4 w = make_float4(0.f, 0.f, -1.f, 0.f);
        if (i < n) {
            const CarTile& T = tiles[i];
            float reach = 0.f;
            for (int k = 0; k < T.n; ++k) reach = fmaxf(reach, sqrtf((T.px[k] - T.cx) * (T.px[k] - T.cx) + (T.py[k] - T.cy) * (T.py[k] - T.cy)));
            const int s = i - i % CAR_SAMPLE_STRIDE;
            const float gx = T.cx - (float)pts[3 * s + 1], gy = T.cy - (float)pts[3 * s + 2];
            if (reach > CAR_WIDE_REACH || gx * gx + gy * gy > CAR_WIDE_GROUP * CAR_WIDE_GROUP) w = make_float4(T.cx, T.cy, reach, (float)i);
        }
        const unsigned m = __ballot_sync(0xffffffffu, w.z >= 0.f);
        const int k = n_wide + __popc(m & ((1u << lane) - 1u));
        if (w.z >= 0.f && k < CAR_MAX_WIDE) wide[k] = w;   // more cannot come from a generated track; load_tracks refuses them
        n_wide += __popc(m);
    }
    for (int k = n_wide + lane; k < CAR_MAX_WIDE; k += 32) wide[k] = make_float4(0.f, 0.f, -1.f, 0.f);
    for (int s = lane; s < CAR_MAX_SAMPLES; s += 32) {
        const int i = s * CAR_SAMPLE_STRIDE;
        p.samples[(size_t)s * (2 * p.n) + slot] = (i < n) ? make_float2((float)pts[3 * i + 1], (float)pts[3 * i + 2])
                                                          : make_float2(1e30f, 1e30f);
    }
    if (lane < 3) p.start_pose[3 * slot + lane] = pts[lane];
    __syncwarp();
    paint_road_map(p, slot, n, lane);
    return n;
}

// Claim the generation of env e's next track (next_state 0 -> 1), or wait for whoever holds it.  A holder is a resident
// warp of car_pregen_kernel or car_reset_kernel, so it finishes on its own: the wait cannot deadlock.
// Returns true when this warp has to generate.
__device__ bool claim_next_track(const CarDev& p, int e, int lane, bool wait) {
    int st = 0;
    if (lane == 0) st = atomicCAS(p.next_state + e, 0, 1);
    st = __shfl_sync(0xffffffffu, st, 0);
    if (st == 0) return true;
    if (wait && st == 1) {
        if (lane == 0) {
            volatile int32_t* flag = p.next_state + e;
            while (*flag != 2) __nanosleep(500);
        }
        __syncwarp();
    }
    __threadfence();
    return false;
}

__device__ void publish_next_track(const CarDev& p, int e, int lane, bool ok) {
    __threadfence();
    __syncwarp();
    if (lane == 0) *(volatile int32_t*)(p.next_state + e) = ok ? 2 : 0;
}

// Next track of every env that has none, one warp per env.  Runs on a side stream behind the step, so that the
// auto-reset below finds the track ready: its inputs are only (seed, global env index, attempt_count).
__global__ void __launch_bounds__(64) car_pregen_kernel(CarDev p) {
    const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (e >= p.n) return;
    if (*(volatile int32_t*)(p.next_state + e) != 0) return;
    if (!claim_next_track(p, e, lane, false)) return;
    if (lane == 0) p.next_att0[e] = p.attempt_count[e];
    const int n = generate_track_warp(p, e, e + p.n * (1 - p.sel[e]), true, lane);
    publish_next_track(p, e, lane, n > 0);
}

// A pre-generated track that will not be used (seed / injection tables / fixed tracks changed): give its attempts back.
__global__ void car_discard_next_kernel(CarDev p) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.n) return;
    if (p.next_state[e] == 2) p.attempt_count[e] = p.next_att0[e];
    p.next_state[e] = 0;
}

// CarRacing.reset: new track (retry until an attempt succeeds, :499-507), cars at track[0] (:508-512).  One warp per env:
// the track is normally waiting in the env's other slot (car_pregen_kernel) and the reset is a slot swap + spawn.
__device__ void car_reset_env(const CarDev& p, int e, int only_done, int lane);

// only_done: the envs on the done list (grid-stride over the list, a warp per env); else every env, one warp each
__global__ void __launch_bounds__(64) car_reset_kernel(CarDev p, int only_done) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (!only_done) {
        if (w < p.n) car_reset_env(p, w, 0, lane);
        return;
    }
    const int count = min(*p.done_count, p.n), n_warps = (gridDim.x * blockDim.x) >> 5;
    for (int i = w; i < count; i += n_warps) car_reset_env(p, p.done_list[i], 1, lane);
}

__device__ void car_reset_env(const CarDev& p, int e, int only_done, int lane) {
    const int next_slot = e + p.n * (1 - p.sel[e]);
    bool have = true;
    const int st_before = *(volatile int32_t*)(p.next_state + e);
    if (only_done && st_before != 2 && lane == 0) atomicAdd(p.overrun + 3, 1);   // an auto-reset that found no track waiting
    if (claim_next_track(p, e, lane, true)) {          // not pre-generated (first reset, or an episode shorter than the generator)
        have = generate_track_warp(p, e, next_slot, false, lane) > 0;
        __threadfence();
    }
    __syncwarp();
    if (lane == 0) {
        if (have) p.sel[e] = 1 - p.sel[e];             // a failed generation (flagged) keeps the old track
        *(volatile int32_t*)(p.next_state + e) = 0;
    }
    const int slot = have ? next_slot : (next_slot >= p.n ? e : e + p.n);
    // cars: birth_place_indices = shuffle(arange(num_player)) (:508-512)
    int rc = 0;
    if (lane == 0) { rc = p.reset_count[e]; p.reset_count[e] = rc + 1; }
    rc = __shfl_sync(0xffffffffu, rc, 0);
    const uint64_t gi = (uint64_t)(p.first_env + e);
    int birth[CAR_MAX_PLAYERS] = {0, 1};
    if (p.players == 2) {
        if (p.birth != nullptr) {
            int k = rc;
            if (k >= p.k_birth) { if (lane == 0) *p.overrun = 1; k = p.k_birth - 1; }
            birth[0] = p.birth[((size_t)e * p.k_birth + k) * 2]; birth[1] = p.birth[((size_t)e * p.k_birth + k) * 2 + 1];
        } else {
            uint32_t r[4];
            philox4x32_10((uint32_t)rc, 0x5EEDu, (uint32_t)gi, (uint32_t)(gi >> 32), (uint32_t)p.seed,
                          (uint32_t)(p.seed >> 32) ^ 0xB1A7u, r);
            if (r[0] & 1u) { birth[0] = 1; birth[1] = 0; }
        }
    }
    const double sp0 = p.start_pose[3 * slot], sp1 = p.start_pose[3 * slot + 1], sp2 = p.start_pose[3 * slot + 2];
    for (int k = 0; k < p.players; ++k) car_body_reset(p, e * p.players + k, sp0, sp1, sp2, birth[k], lane);
    if (lane == 0) {
        p.step_count[e] = 0;
        p.elapsed[e] = 0;
        p.inv_dt0[e] = 0.f;
        if (p.n_contacts != nullptr) p.n_contacts[e] = 0;
    }
}

// ------------------------------------------------------------------------------------------------
// per-step pipeline, one thread per car

struct Joint {
    F2 rA;
    float k00, k01, k02, k11, k12, k22;   // symmetric K (ex.x, ey.x, ez.x, ey.y, ez.y, ez.z)
    float c33x, c33y, c33z, det33;        // b2Mat33::Solve33: cross(ey, ez) and 1 / det, the same every iteration of a step
    float motor_mass;
    float ix, iy, iz, motor_impulse, motor_speed;
    int limit_state;
};

// the part of Solve33 that does not depend on the right-hand side (same operations in the same order as Box2D's)
__device__ __forceinline__ void solve33_prepare(Joint& j) {
    const float ex0 = j.k00, ex1 = j.k01, ex2 = j.k02, ey0 = j.k01, ey1 = j.k11, ey2 = j.k12, ez0 = j.k02, ez1 = j.k12, ez2 = j.k22;
    j.c33x = ey1 * ez2 - ey2 * ez1; j.c33y = ey2 * ez0 - ey0 * ez2; j.c33z = ey0 * ez1 - ey1 * ez0;
    float det = ex0 * j.c33x + ex1 * j.c33y + ex2 * j.c33z;
    if (det != 0.0f) det = 1.0f / det;
    j.det33 = det;
}
__device__ __forceinline__ void solve33(const Joint& j, float b0, float b1, float b2, float& o0, float& o1, float& o2) {
    const float ex0 = j.k00, ex1 = j.k01, ex2 = j.k02, ey0 = j.k01, ey1 = j.k11, ey2 = j.k12, ez0 = j.k02, ez1 = j.k12, ez2 = j.k22;
    const float cx = j.c33x, cy = j.c33y, cz = j.c33z, det = j.det33;
    o0 = det * (b0 * cx + b1 * cy + b2 * cz);
    const float bx = b1 * ez2 - b2 * ez1, by = b2 * ez0 - b0 * ez2, bz = b0 * ez1 - b1 * ez0;
    o1 = det * (ex0 * bx + ex1 * by + ex2 * bz);
    const float dx = ey1 * b2 - ey2 * b1, dy = ey2 * b0 - ey0 * b2, dz = ey0 * b1 - ey1 * b0;
    o2 = det * (ex0 * dx + ex1 * dy + ex2 * dz);
}

__device__ __forceinline__ F2 solve22(float a11, float a12, float a21, float a22, F2 b) {
    float det = a11 * a22 - a12 * a21;
    if (det != 0.0f) det = 1.0f / det;
    return f2(det * (a22 * b.x - a12 * b.y), det * (a11 * b.y - a21 * b.x));
}

// One relaxation of a wheel joint inside a velocity iteration (b2RevoluteJoint::SolveVelocityConstraints: motor, then
// the limit's 3 x 3 block or the plain 2 x 2 point constraint).  MAY_LIMIT = false: no lane of the warp has this joint
// at its limit in this step (the limit state is fixed before the 180 iterations), so the branch and its code are
// left out of the loop altogether.
template <bool MAY_LIMIT>
__device__ __forceinline__ void relax_joint(Joint& j, F2& vA, float& wA, F2& vB, float& wB, float mA, float iA, float mB, float iB,
                                            float max_motor_impulse) {
    {   // motor
        const float Cdot = wB - wA - j.motor_speed;
        float impulse = -j.motor_mass * Cdot;
        const float old = j.motor_impulse;
        j.motor_impulse = clampf(old + impulse, -max_motor_impulse, max_motor_impulse);
        impulse = j.motor_impulse - old;
        wA -= iA * impulse;
        wB += iB * impulse;
    }
    if (MAY_LIMIT && j.limit_state != 0) {
        const F2 Cdot1 = (vB - vA) - cross_sv(wA, j.rA);
        const float Cdot2 = wB - wA;
        float i0, i1, i2;
        solve33(j, Cdot1.x, Cdot1.y, Cdot2, i0, i1, i2);
        i0 = -i0; i1 = -i1; i2 = -i2;
        const float ni = j.iz + i2;
        const bool release = (j.limit_state == 1) ? (ni < 0.0f) : (ni > 0.0f);
        if (release) {
            const F2 rhs = f2(-Cdot1.x + j.iz * j.k02, -Cdot1.y + j.iz * j.k12);
            const F2 red = solve22(j.k00, j.k01, j.k01, j.k11, rhs);
            i0 = red.x; i1 = red.y; i2 = -j.iz;
            j.ix += red.x; j.iy += red.y; j.iz = 0.0f;
        } else {
            j.ix += i0; j.iy += i1; j.iz += i2;
        }
        const F2 P = f2(i0, i1);
        vA = vA - mA * P;
        wA -= iA * (cross(j.rA, P) + i2);
        vB = vB + mB * P;
        wB += iB * i2;
    } else {
        const F2 Cdot = (vB - vA) - cross_sv(wA, j.rA);
        const F2 imp = solve22(j.k00, j.k01, j.k01, j.k11, f2(-Cdot.x, -Cdot.y));
        j.ix += imp.x; j.iy += imp.y;
        vA = vA - mA * imp;
        wA -= iA * cross(j.rA, imp);
        vB = vB + mB * imp;
    }
}

// polygons (with b2_polygonRadius skins) touch: max face separation below 2 * radius
__device__ float max_separation(const float* ax, const float* ay, int na, const float* bx, const float* by, int nb) {
    float best = -3.4e38f;
    for (int i = 0; i < na; ++i) {
        const int i2 = (i + 1 == na) ? 0 : i + 1;
        const float ex = ax[i2] - ax[i], ey = ay[i2] - ay[i];
        const float len = sqrtf(ex * ex + ey * ey);
        if (len < 1e-12f) continue;
        const float nx = ey / len, ny = -ex / len;
        float mn = 3.4e38f;
        for (int k = 0; k < nb; ++k) mn = fminf(mn, nx * (bx[k] - ax[i]) + ny * (by[k] - ay[i]));
        best = fmaxf(best, mn);
    }
    return best;
}

// the same with the face normals of A given (nx[i] > 1e38: degenerate edge, skipped like len < 1e-12 above)
__device__ __forceinline__ float max_separation_n(const float* ax, const float* ay, const float* nx, const float* ny, int na,
                                                  const float* bx, const float* by, int nb) {
    float best = -3.4e38f;
    for (int i = 0; i < na; ++i) {
        if (nx[i] > 1.0e38f) continue;
        float mn = 3.4e38f;
        for (int k = 0; k < nb; ++k) mn = fminf(mn, nx[i] * (bx[k] - ax[i]) + ny[i] * (by[k] - ay[i]));
        best = fmaxf(best, mn);
    }
    return best;
}

// max_separation_n(...) >= thr, i.e. some face of A keeps every vertex of B at least thr away (same arithmetic per face)
__device__ __forceinline__ bool separated_by_face(const float* ax, const float* ay, const float* nx, const float* ny, int na,
                                                  const float* bx, const float* by, int nb, float thr) {
    for (int i = 0; i < na; ++i) {
        if (nx[i] > 1.0e38f) continue;
        float mn = 3.4e38f;
        for (int k = 0; k < nb; ++k) mn = fminf(mn, nx[i] * (bx[k] - ax[i]) + ny[i] * (by[k] - ay[i]));
        if (!(mn < thr)) return true;
    }
    return false;
}

// Can any fixture pair of the two cars be within contact reach?  The cars as oriented boxes in their hull frames (hull
// polygons span x +-1.2, y -2.4..2.6; wheels reach x +-1.71 at any steering angle; 0.3 of slack for skins and joint
// error): separated boxes, no contact.  pose[0] / pose[5] = (cx, cy, angle) of the two hulls.  Right after a reset the
// wheels are not yet where the joints want them (Car.__init__ places them un-rotated, car_dynamics.py:90): plain
// distance gate for the first steps.
__device__ __forceinline__ bool cars_near(const float (*pose)[3], float hull_lcx, float hull_lcy, int step_count) {
    const Rot qa = make_rot(pose[0][2]), qb = make_rot(pose[5][2]);
    const F2 pa = f2(pose[0][0], pose[0][1]) + rmul(qa, f2(-hull_lcx, 0.1f - hull_lcy));
    const F2 pb = f2(pose[5][0], pose[5][1]) + rmul(qb, f2(-hull_lcx, 0.1f - hull_lcy));
    const F2 t = pb - pa;
    const float ex = 2.01f, ey = 2.8f;
    const float cxx = fabsf(qa.c * qb.c + qa.s * qb.s), cxy = fabsf(qa.s * qb.c - qa.c * qb.s);   // |ax.bx|, |ax.by| (= |ay.bx|)
    const float tax = fabsf(t.x * qa.c + t.y * qa.s), tay = fabsf(-t.x * qa.s + t.y * qa.c);
    const float tbx = fabsf(t.x * qb.c + t.y * qb.s), tby = fabsf(-t.x * qb.s + t.y * qb.c);
    const bool separated = tax > ex + ex * cxx + ey * cxy || tay > ey + ex * cxy + ey * cxx ||
                           tbx > ex + ex * cxx + ey * cxy || tby > ey + ex * cxy + ey * cxx;
    return (step_count < 4) ? (t.x * t.x + t.y * t.y < 8.0f * 8.0f) : !separated;
}

// b2ContactManager::Collide for the tile sensors of ONE wheel: the road tiles whose fixture overlaps the wheel box (SAT
// with the b2_polygonRadius skins), as a 512-bit set in now16[16] (global memory).  Candidates: every 8th track point
// within 36 units of the hull (transposed array: coalesced), then tile centres within 11.5 of the hull and 9 of the wheel;
// plus the slot's wide tiles (generate_track_warp), which those radii would miss.  `near_samples`: bit s set = track point 8 s lies within 36 units of the hull (0 = not known: scanned here).
__device__ void sensor_wheel_overlaps(const CarDev& p, int slot, int n_track, F2 hp, F2 wc, float wa, uint32_t* __restrict__ now16,
                                      unsigned long long near_samples, bool have_near) {
    const CarTile* tiles = p.tiles + (size_t)slot * CAR_MAX_TRACK;
    const float2* centres = p.tile_centres + (size_t)slot * CAR_MAX_TRACK;
    reinterpret_cast<uint4*>(now16)[0] = make_uint4(0u, 0u, 0u, 0u); reinterpret_cast<uint4*>(now16)[1] = make_uint4(0u, 0u, 0u, 0u);
    reinterpret_cast<uint4*>(now16)[2] = make_uint4(0u, 0u, 0u, 0u); reinterpret_cast<uint4*>(now16)[3] = make_uint4(0u, 0u, 0u, 0u);
    // wheel box in world coordinates and its face normals
    float wx[4], wy[4], wnx[4], wny[4];
    {
        const Rot q = make_rot(wa);
        const float hw = (float)(CR_WHEEL_W * CR_SIZE), hr = (float)(CR_WHEEL_R * CR_SIZE);
        const F2 l0 = rmul(q, f2(-hw, -hr)) + wc, l1 = rmul(q, f2(+hw, -hr)) + wc;
        const F2 l2 = rmul(q, f2(+hw, +hr)) + wc, l3 = rmul(q, f2(-hw, +hr)) + wc;
        wx[0] = l0.x; wy[0] = l0.y; wx[1] = l1.x; wy[1] = l1.y; wx[2] = l2.x; wy[2] = l2.y; wx[3] = l3.x; wy[3] = l3.y;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int i2 = (i + 1) & 3;
            const float ex = wx[i2] - wx[i], ey = wy[i2] - wy[i];
            const float len = sqrtf(ex * ex + ey * ey);
            wnx[i] = 3.0e38f; wny[i] = 0.f;
            if (!(len < 1e-12f)) { wnx[i] = ey / len; wny[i] = -ex / len; }
        }
    }
    const int n_samp = (n_track + CAR_SAMPLE_STRIDE - 1) / CAR_SAMPLE_STRIDE;
    if (!have_near) {
        near_samples = 0ull;
        for (int s = 0; s < n_samp; ++s) {
            const float2 sp = p.samples[(size_t)s * (2 * p.n) + slot];
            const float dx = sp.x - hp.x, dy = sp.y - hp.y;
            if (dx * dx + dy * dy < 36.0f * 36.0f) near_samples |= 1ull << s;
        }
    }
    // Candidates first (tile centre within 11.5 of the hull and 9 of the wheel: a few per wheel), tests second: the lanes of
    // a warp reach their candidates at different points of the walk, and testing on the spot would run the test once per
    // such point instead of once per round of "every lane's j-th candidate".  Up to six 10-bit tile ids in one word.
    unsigned long long cand = 0ull;
    int n_cand = 0;
    auto test_tile = [&](int t) {
        const CarTile* Tp = tiles + t;
        float tpx[5], tpy[5], tnx[5], tny[5];
#pragma unroll
        for (int i = 0; i < 5; ++i) { tpx[i] = Tp->px[i]; tpy[i] = Tp->py[i]; tnx[i] = Tp->nx[i]; tny[i] = Tp->ny[i]; }
        const int tn = Tp->n;
        // Cheap and safe reject: a tile face that keeps the wheel's centre more than the wheel's circumradius (0.6083)
        // plus 2 r away keeps every wheel vertex 2 r away (the 0.0067 of slack dwarfs fp32 rounding), so the exact
        // test below would find the same face separating.  Most candidates are the overlapped tile's neighbours.
        bool far_face = false;
#pragma unroll
        for (int i = 0; i < 5; ++i)
            if (i < tn && !(tnx[i] > 1.0e38f) && tnx[i] * (wc.x - tpx[i]) + tny[i] * (wc.y - tpy[i]) - 0.615f >= 2.0f * B2_POLYGON_RADIUS)
                far_face = true;
        if (far_face) return;
        // max(s1, s2) < 2 r  <=>  no face of either polygon separates them by 2 r or more: stop at the first that does
        if (!separated_by_face(wx, wy, wnx, wny, 4, tpx, tpy, tn, 2.0f * B2_POLYGON_RADIUS) &&
            !separated_by_face(tpx, tpy, tnx, tny, tn, wx, wy, 4, 2.0f * B2_POLYGON_RADIUS))
            now16[t >> 5] |= 1u << (t & 31);
    };
    while (near_samples) {
        const int s = __ffsll((long long)near_samples) - 1;
        near_samples &= near_samples - 1ull;
        const int t1 = min(n_track, (s + 1) * CAR_SAMPLE_STRIDE);
        for (int t = s * CAR_SAMPLE_STRIDE; t < t1; ++t) {
            const float2 tc = centres[t];
            const float tx = tc.x - hp.x, ty = tc.y - hp.y;
            if (!(tx * tx + ty * ty < 11.5f * 11.5f)) continue;
            const float ddx = tc.x - wc.x, ddy = tc.y - wc.y;
            if (!(ddx * ddx + ddy * ddy <= 9.0f * 9.0f)) continue;
            if (n_cand < 6) { cand |= (unsigned long long)t << (10 * n_cand); ++n_cand; }
            else test_tile(t);                                     // more candidates than the word holds: on the spot
        }
    }
    // tiles that reach farther than the radii above assume (the seam tile of every generated track): candidates whenever
    // the wheel box (circumradius 0.6083, two skins 0.02) can reach the tile's far vertex; a repeated test only sets its
    // bit again
    const float4* wide = p.wide_tiles + (size_t)slot * CAR_MAX_WIDE;
    for (int j = 0; j < CAR_MAX_WIDE; ++j) {
        const float4 wt = wide[j];
        if (!(wt.z >= 0.f)) break;
        const float dx = wt.x - wc.x, dy = wt.y - wc.y, r = wt.z + 0.65f;
        if (!(dx * dx + dy * dy <= r * r)) continue;
        if (n_cand < 6) { cand |= (unsigned long long)(int)wt.w << (10 * n_cand); ++n_cand; }
        else test_tile((int)wt.w);
    }
    for (int j = 0; j < n_cand; ++j) test_tile((int)((cand >> (10 * j)) & 1023ull));
}

// The tile-sensor overlaps of every wheel at the start of world.Step, one thread per (car, wheel), ahead of the step
// kernel: they depend only on the poses the previous step left behind, and one thread per car would walk its four
// wheels' candidates one after the other on the step's critical path.
__global__ void __launch_bounds__(128) car_sensor_kernel(CarDev p, int classify) {
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int ci = gt >> 2, k = gt & 3;
    if (ci >= p.n * p.players) return;
    const int e = ci / p.players;
    const float* b = p.body + (size_t)ci * 40;
    const Rot qh = make_rot(b[2]);
    const F2 hp = f2(b[0], b[1]) - rmul(qh, f2(p.consts->hull_lcx, p.consts->hull_lcy));
    const int slot = car_slot(p, e);
    // two-car envs: the env whose cars are near each other goes on the near list (car_collide_kernel, then car_step_kernel)
    if (classify && p.players == 2 && (gt & 7) == 0) {
        const float* b1 = b + 40;
        const float pose[10][3] = {{b[0], b[1], b[2]}, {}, {}, {}, {}, {b1[0], b1[1], b1[2]}, {}, {}, {}, {}};
        const bool near = cars_near(pose, p.consts->hull_lcx, p.consts->hull_lcy, p.step_count[e]);
        if (near) p.near_list[atomicAdd(p.near_count, 1)] = e;       // car_collide_kernel decides whether they touch
        else { p.deferred[e] = 0; p.n_contacts[e] = 0; }
    }
    // the prefilter on every 8th track point depends on the hull only: the four wheel lanes of a car take a quarter of the
    // (at most 64) points each and pool what they found
    const int n_track = p.n_track[slot];
    const int n_samp = (n_track + CAR_SAMPLE_STRIDE - 1) / CAR_SAMPLE_STRIDE;
    unsigned long long near_samples = 0ull;
    for (int s = k; s < n_samp; s += 4) {
        const float2 sp = p.samples[(size_t)s * (2 * p.n) + slot];
        const float dx = sp.x - hp.x, dy = sp.y - hp.y;
        if (dx * dx + dy * dy < 36.0f * 36.0f) near_samples |= 1ull << s;
    }
    const unsigned car_lanes = 0xFu << (threadIdx.x & 28);            // the four lanes of this car: in range together
    near_samples |= __shfl_xor_sync(car_lanes, near_samples, 1);
    near_samples |= __shfl_xor_sync(car_lanes, near_samples, 2);
    sensor_wheel_overlaps(p, slot, n_track, hp, f2(b[8 * (k + 1)], b[8 * (k + 1) + 1]), b[8 * (k + 1) + 2],
                          p.sensor_now + ((size_t)ci * 4 + k) * 16, near_samples, true);
}

__device__ __noinline__ void sensor_car_overlaps(const CarDev& p, int ci, int slot, int n_track, F2 hp, const F2* c, const float* a) {
    for (int k = 0; k < 4; ++k) sensor_wheel_overlaps(p, slot, n_track, hp, c[k + 1], a[k + 1], p.sensor_now + ((size_t)ci * 4 + k) * 16, 0ull, false);
}

// b2ContactManager::Collide between the two cars of every env on the NEAR list (the oriented-box gate of the sensor
// kernel), ahead of the step kernel and in parallel: one 64-thread block per env, one thread per allowed fixture pair
// (48: hull-hull 16, wheel-hull 2 x 16).  Like the tile sensors, the manifolds depend only on the poses the previous
// step left behind; inside the one-lane-per-car step kernel the 48 b2CollidePolygons calls ran one after the other and
// were the longest part of the slow physics pass (0.32 of 0.64 ms at config 5).  Same arithmetic and the same canonical
// record order as car_contacts_collide (which stays for the further sub-steps of action_repeat > 1).  Envs that come out
// with a touching pair go on the slow list (merged island: sequential contact pass); the others are stepped by the fast pass.
__global__ void __launch_bounds__(64) car_collide_kernel(CarDev p) {
    __shared__ Xf s_xf[10];
    __shared__ F2 s_wc[16];
    __shared__ int s_cnt0, s_nold;
    __shared__ uint8_t s_old_pair[CAR_MAX_CONTACTS], s_old_count[CAR_MAX_CONTACTS];
    __shared__ uint32_t s_old_id[CAR_MAX_CONTACTS][2];
    __shared__ float s_old_ni[CAR_MAX_CONTACTS][2], s_old_ti[CAR_MAX_CONTACTS][2];
    const CarHullConst* K = p.consts;
    const int t = threadIdx.x;
    const int n_near = min(*p.near_count, p.n);
    for (int li = blockIdx.x; li < n_near; li += gridDim.x) {
        const int e = p.near_list[li];
        CarContact* recs = p.contacts + (size_t)e * CAR_MAX_CONTACTS;
        if (t < 10) {
            const float* b = p.body + ((size_t)e * 2 + t / 5) * 40 + 8 * (t % 5);
            s_xf[t] = xf_of(f2(b[0], b[1]), b[2], body_lc(K, t));
        }
        if (t == 32) s_nold = min(max(p.n_contacts[e], 0), CAR_MAX_CONTACTS);
        if (t >= 48 && t < 48 + CAR_MAX_CONTACTS) {          // the previous step's records: what the warm start needs of them
            const CarContact* o = recs + (t - 48);
            s_old_pair[t - 48] = o->pair; s_old_count[t - 48] = o->count;
            s_old_id[t - 48][0] = o->id[0]; s_old_id[t - 48][1] = o->id[1];
            s_old_ni[t - 48][0] = o->ni[0]; s_old_ni[t - 48][1] = o->ni[1];
            s_old_ti[t - 48][0] = o->ti[0]; s_old_ti[t - 48][1] = o->ti[1];
        }
        __syncthreads();
        if (t < 16) {      // world centroids of the 8 fixtures of each car
            const int car = t >> 3, f = t & 7;
            const int b = 5 * car + (f < 4 ? 0 : f - 3), sh = f < 4 ? f : 4;
            s_wc[t] = xf_mul(s_xf[b], f2(K->fix_cx[sh], K->fix_cy[sh]));
        }
        __syncthreads();
        CarContact m;
        m.count = 0;
        int ba = 0, bb = 5;
        if (t < 48) {
            const int fa = t < 32 ? t >> 3 : 4 + ((t - 32) >> 2), fb = t < 32 ? t & 7 : (t - 32) & 3;
            ba = fa < 4 ? 0 : fa - 3; bb = 5 + (fb < 4 ? 0 : fb - 3);
            const int sa = fa < 4 ? fa : 4, sb = fb < 4 ? fb : 4;
            // quick reject of pairs farther apart than their bounding circles plus 0.15 (see car_contacts_collide)
            const F2 d = s_wc[8 + fb] - s_wc[fa];
            const float reach = K->fix_cradius[sa] + K->fix_cradius[sb] + 0.15f;
            if (!(dot(d, d) > reach * reach)) collide_polygons(&m, poly_ref(K, sa), s_xf[ba], poly_ref(K, sb), s_xf[bb]);
        }
        const bool touching = m.count != 0;
        const unsigned ball = __ballot_sync(0xffffffffu, touching);
        if (t == 0) s_cnt0 = __popc(ball);
        __syncthreads();
        const int rank = (t < 32 ? 0 : s_cnt0) + __popc(ball & ((1u << (t & 31)) - 1u));   // canonical order = pair index
        int n_new = s_cnt0;
        if (t >= 32) n_new += __popc(ball);
        n_new = __shfl_sync(0xffffffffu, n_new, 0);                                        // warp 1 holds the total
        if (touching) {
            if (rank >= CAR_MAX_CONTACTS) atomicAdd(p.contact_overflow, 1);
            else {
                m.pair = (uint8_t)t; m.ia = (uint8_t)ba; m.ib = (uint8_t)bb; m.vcount = m.count;
                for (int i = 0; i < m.count; ++i) { m.ni[i] = 0.f; m.ti[i] = 0.f; }
                for (int o = 0; o < s_nold; ++o) {
                    if (s_old_pair[o] != t) continue;
                    for (int i = 0; i < m.count; ++i)
                        for (int j = 0; j < s_old_count[o]; ++j)
                            if (s_old_id[o][j] == m.id[i]) { m.ni[i] = s_old_ni[o][j]; m.ti[i] = s_old_ti[o][j]; break; }
                }
                recs[rank] = m;
            }
        }
        if (t == 32) {                                       // a thread of warp 1: it knows the total
            const int kept = min(n_new, CAR_MAX_CONTACTS);
            p.n_contacts[e] = kept;
            p.deferred[e] = kept > 0 ? 1 : 0;
            if (kept > 0) p.slow_list[atomicAdd(p.slow_count, 1)] = e;
        }
        __syncthreads();
    }
}

// mode 0: every car.  mode 1 (fast pass): two-car envs whose cars are near each other are skipped: car_sensor_kernel put
// them on p.slow_list (p.deferred[env] = 1) -- their contact solve is several times longer than a plain step and would
// hold up the whole single-wave launch.  mode 2 (slow pass): the envs on p.slow_list, two lanes each; the two passes
// touch disjoint envs and run side by side on two streams.
__global__ void __launch_bounds__(64)
car_step_kernel(CarDev p, int mode, const float* __restrict__ actions, float* __restrict__ rew, uint8_t* __restrict__ done_out,
                int32_t* __restrict__ num_steps_out, uint8_t* __restrict__ truncated_out) {
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
    const int n_cars = p.n * p.players;
    int ci = gtid;
    bool active = ci < n_cars;
    if (mode == 2) {                 // slow pass: lane pair i takes env slow_list[i]
        active = (gtid >> 1) < *p.slow_count;
        ci = active ? p.slow_list[gtid >> 1] * 2 + (gtid & 1) : 0;
    }
    const int e = active ? ci / p.players : 0, player = active ? ci % p.players : 0;
    bool car_done = false;
    double step_reward = 0.0;
    int env_steps = 0;
    // two-car envs: the cars of an env sit on adjacent lanes (blockDim is even, ci = 2 * env + player) and exchange
    // their bodies through these blocks when they touch (car_contact.cuh)
    __shared__ float sh_pose[32][10][3];
    __shared__ float sh_vel[32][10][3];
    const unsigned pair_mask = 3u << (threadIdx.x & 30);
    float (*pose)[3] = sh_pose[threadIdx.x >> 1];
    float (*vel)[3] = sh_vel[threadIdx.x >> 1];
    bool deferred = false;
    if (active && p.players == 2 && mode != 2) {
        if (mode == 1) deferred = p.deferred[e] != 0;       // decided by car_sensor_kernel from the poses at the start of the step
        else if (player == 0) p.deferred[e] = 0;
    }
    active = active && !deferred;
    const unsigned warp_lanes = __ballot_sync(0xffffffffu, active);   // the lanes that run the per-car pipeline
    if (active) {
        const CarHullConst K = *p.consts;
        // ---- load ----
        F2 c[5], v[5];
        float a[5], w[5], sleep_t[5];
        bool awake[5];
        {
            const float* b = p.body + (size_t)ci * 40;
#pragma unroll
            for (int i = 0; i < 5; ++i) {
                c[i] = f2(b[8 * i], b[8 * i + 1]); a[i] = b[8 * i + 2]; v[i] = f2(b[8 * i + 3], b[8 * i + 4]);
                w[i] = b[8 * i + 5]; sleep_t[i] = b[8 * i + 6]; awake[i] = b[8 * i + 7] != 0.f;
            }
        }
        Joint J[4];
        {
            const float* j = p.joint + (size_t)ci * 24;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                J[k].ix = j[6 * k]; J[k].iy = j[6 * k + 1]; J[k].iz = j[6 * k + 2]; J[k].motor_impulse = j[6 * k + 3];
                J[k].limit_state = (int)j[6 * k + 4]; J[k].motor_speed = j[6 * k + 5];
            }
        }
        double omega[4], gas[2], brake, steer;
        {
            const double* wd = p.wheel + (size_t)ci * 8;
#pragma unroll
            for (int k = 0; k < 4; ++k) omega[k] = wd[k];
            gas[0] = wd[4]; gas[1] = wd[5]; brake = wd[6]; steer = wd[7];
        }
        double reward = p.reward[2 * ci], prev_reward = p.reward[2 * ci + 1];
        int32_t* cn = p.counters + 4 * ci;
        int tile_visited = cn[0], last_block = cn[1], has_block = cn[2];
        car_done = cn[3] != 0;
        uint32_t* touching = p.touching + (size_t)ci * 64;
        uint32_t* visited = p.visited + (size_t)ci * 16;
        const int slot = car_slot(p, e);
        const int n_track = p.n_track[slot];
        int step_count = p.step_count[e];
        float inv_dt0 = p.inv_dt0[e];
        const float hull_lcx = K.hull_lcx, hull_lcy = K.hull_lcy;

        // ---- process_action (:527-540) + Car.steer(-a0) / gas / brake (car_dynamics.py:131-157) ----
        {
            const double in0 = (double)actions[2 * ci], in1 = (double)actions[2 * ci + 1];
            const double a0 = fmax(fmin(in0, 1.0), -1.0);
            double a1 = fmax(fmin(in1, 1.0), -1.0), a2;
            if (a1 > 0) a2 = 0; else { a2 = a1; a1 = 0; }
            steer = -a0;
            const double g = fmin(fmax(fabs(a1), 0.0), 1.0);
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                double diff = g - gas[k];
                if (diff > 0.1) diff = 0.1;
                gas[k] += diff;
            }
            brake = fabs(a2);
        }

        const double dt = 1.0 / CR_FPS;
        const float h = 1.0f / CR_FPS;
        for (int rep = 0; rep < p.action_repeat; ++rep) {
            F2 force[5];
#pragma unroll
            for (int i = 0; i < 5; ++i) force[i] = f2(0.f, 0.f);
            int n_touch[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                int cnt = 0;
                for (int wd = 0; wd < 16; ++wd) cnt += __popc(touching[16 * k + wd]);
                n_touch[k] = cnt;
            }
            if (!car_done) {
                // ---- Car.step(1/FPS), car_dynamics.py:159-234 ----
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int bi = k + 1;
                    const double joint_angle = (double)(a[bi] - a[0] - 0.0f);
                    const double st = (k < 2) ? steer : 0.0;
                    const double dir = signd(st - joint_angle), val = fabs(st - joint_angle);
                    J[k].motor_speed = (float)(dir * fmin(50.0 * val, 3.0));
                    if (!awake[0]) { awake[0] = true; sleep_t[0] = 0.f; }      // SetMotorSpeed wakes both bodies
                    if (!awake[bi]) { awake[bi] = true; sleep_t[bi] = 0.f; }
                    double friction_limit = CR_FRICTION_LIMIT * 0.6;
                    if (n_touch[k] > 0) friction_limit = fmax(friction_limit, CR_FRICTION_LIMIT * 1.0);
                    const Rot q = make_rot(a[bi]);
                    const F2 forw = rmul(q, f2(0.f, 1.f)), side = rmul(q, f2(1.f, 0.f));
                    const double vf = (double)forw.x * (double)v[bi].x + (double)forw.y * (double)v[bi].y;
                    const double vs = (double)side.x * (double)v[bi].x + (double)side.y * (double)v[bi].y;
                    const double gk = (k >= 2) ? gas[k - 2] : 0.0;
                    omega[k] += dt * CR_ENGINE_POWER * gk / CR_WHEEL_MOI / (fabs(omega[k]) + 5.0);
                    if (brake >= 0.9) {
                        omega[k] = 0;
                    } else if (brake > 0) {
                        const double bdir = -signd(omega[k]);
                        double bval = 15 * brake;
                        if (fabs(bval) > fabs(omega[k])) bval = fabs(omega[k]);
                        omega[k] += bdir * bval;
                    }
                    const double vr = omega[k] * (CR_WHEEL_R * CR_SIZE);
                    double f_force = -vf + vr, p_force = -vs;
                    f_force *= 205000 * CR_SIZE * CR_SIZE;
                    p_force *= 205000 * CR_SIZE * CR_SIZE;
                    double frc = sqrt(f_force * f_force + p_force * p_force);
                    if (fabs(frc) > friction_limit) {
                        f_force /= frc; p_force /= frc;
                        frc = friction_limit;
                        f_force *= frc; p_force *= frc;
                    }
                    omega[k] -= dt * f_force * (CR_WHEEL_R * CR_SIZE) / CR_WHEEL_MOI;
                    const float fx = (float)(p_force * (double)side.x + f_force * (double)forw.x);
                    const float fy = (float)(p_force * (double)side.y + f_force * (double)forw.y);
                    force[bi] = force[bi] + f2(fx, fy);   // ApplyForceToCenter(.., True): wheel is awake by now
                }
                // ---- CarRacing.step bookkeeping (:581-598) ----
                reward -= 0.1 / p.action_repeat;
                step_reward += reward - prev_reward;
                prev_reward = reward;
                {
                    const Rot q = make_rot(a[0]);
                    const F2 pos = c[0] - rmul(q, f2(hull_lcx, hull_lcy));
                    if (tile_visited == n_track) car_done = true;
                    if (fabs((double)pos.x) > CR_PLAYFIELD || fabs((double)pos.y) > CR_PLAYFIELD) car_done = true;
                    if (step_count > 1000) car_done = true;
                }
            }
            // ================= world.Step(1/FPS, 180, 60) =================
            // ---- b2ContactManager::Collide: wheel-tile sensor contacts -> FrictionDetector._contact ----
            {
                // the overlap sets of the four wheels come from car_sensor_kernel (poses at the start of the step); a further
                // sub-step of the same action (action_repeat > 1) recomputes them here from the poses it now has
                if (rep > 0) {
                    const Rot qh = make_rot(a[0]);
                    sensor_car_overlaps(p, ci, slot, n_track, c[0] - rmul(qh, f2(hull_lcx, hull_lcy)), c, a);
                }
                const uint32_t* now = p.sensor_now + (size_t)ci * 64;
                // contact events wheel by wheel (FrictionDetector._contact), BeginContact in ascending block id
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    uint32_t was_w[16];
                    {
                        const uint4* tw = reinterpret_cast<const uint4*>(touching + 16 * k);
#pragma unroll
                        for (int i = 0; i < 4; ++i) { const uint4 q4 = tw[i]; was_w[4 * i] = q4.x; was_w[4 * i + 1] = q4.y; was_w[4 * i + 2] = q4.z; was_w[4 * i + 3] = q4.w; }
                    }
                    uint32_t now_k[16];
                    {
                        const uint4* nw = reinterpret_cast<const uint4*>(now + 16 * k);
#pragma unroll
                        for (int i = 0; i < 4; ++i) { const uint4 q4 = nw[i]; now_k[4 * i] = q4.x; now_k[4 * i + 1] = q4.y; now_k[4 * i + 2] = q4.z; now_k[4 * i + 3] = q4.w; }
                    }
#pragma unroll
                    for (int wd = 0; wd < 16; ++wd) {
                        const uint32_t was = was_w[wd], now_w = now_k[wd];
                        if (now_w == was) continue;                        // nothing begins or ends in these 32 tiles
                        uint32_t begins = now_w & ~was;
                        while (begins) {
                            const int bit = __ffs(begins) - 1;
                            begins &= begins - 1;
                            const int t = wd * 32 + bit;
                            if (!((visited[wd] >> bit) & 1u)) {
                                const int last_blk = has_block ? last_block : 0;
                                if (t - last_blk < 50) {
                                    last_block = t; has_block = 1;
                                    reward += 1000.0 / n_track;
                                }
                                visited[wd] |= 1u << bit;
                                tile_visited += 1;
                            }
                        }
                        touching[16 * k + wd] = now_w;                     // EndContact: tiles.remove
                    }
                }
            }
            // ---- b2ContactManager::Collide: car-car contacts (two-car envs).  n_con > 0 merges both cars into one island. ----
            int n_con = 0;
            CarContact* recs = nullptr;
            if (p.players == 2) {
#pragma unroll
                for (int i = 0; i < 5; ++i) { pose[player * 5 + i][0] = c[i].x; pose[player * 5 + i][1] = c[i].y; pose[player * 5 + i][2] = a[i]; }
                __syncwarp(pair_mask);
                recs = p.contacts + (size_t)e * CAR_MAX_CONTACTS;
                if (rep == 0) {
                    n_con = p.n_contacts[e];       // car_sensor_kernel (far: 0) / car_collide_kernel, from the poses at the start of the step
                } else {                           // a further sub-step of the same action: from the poses it now has
                    const bool near_each_other = cars_near(pose, hull_lcx, hull_lcy, step_count);
                    if (near_each_other) {
                        if (player == 0) {
                            n_con = car_contacts_collide(p.consts, pose, recs, p.n_contacts[e], p.contact_overflow);
                            p.n_contacts[e] = n_con;
                        }
                        n_con = __shfl_sync(pair_mask, n_con, threadIdx.x & 30);
                    } else if (player == 0) {
                        p.n_contacts[e] = 0;
                    }
                }
            }
            if (p.players == 2 && player == 0) p.n_contacts_step[e] = n_con;   // what crl_car_get_contacts reports (n_contacts is rewritten ahead of the next step)
            const bool merged = n_con > 0;
            // ---- b2Island::Solve for this car's island (bodies: hull + 4 wheels; joints relaxed in the
            //      order wheel 3, 2, 1, 0 -- the island order b2World::Solve's DFS produces) ----
            bool any_awake = awake[0] || awake[1] || awake[2] || awake[3] || awake[4];
            if (merged) any_awake = any_awake || __shfl_xor_sync(pair_mask, (int)any_awake, 1) != 0;
            // The lanes arrive here diverged (different numbers of candidate tiles, contact events, gate outcomes); left
            // alone, each group would run the 180-iteration solver loops on its own.  Reconverge the warp first.
            __syncwarp(warp_lanes);
            const unsigned awake_lanes = __ballot_sync(warp_lanes, any_awake);   // the lanes that run the solver loops
            if (any_awake) {
#pragma unroll
                for (int i = 0; i < 5; ++i)
                    if (!awake[i]) { awake[i] = true; sleep_t[i] = 0.f; }
                const float dt_ratio = inv_dt0 * h;
                const float mA = K.hull_inv_mass, iA = K.hull_inv_I, mB = K.wheel_inv_mass, iB = K.wheel_inv_I;
                const F2 c0h = c[0];
                (void)c0h;
#pragma unroll
                for (int i = 0; i < 5; ++i) {
                    const float im = (i == 0) ? mA : mB;
                    v[i] = v[i] + h * (im * force[i]);
                    // torque is never applied; damping is 0: v *= 1/(1 + h*0)
                    v[i] = (1.0f / (1.0f + h * 0.0f)) * v[i];
                    w[i] *= 1.0f / (1.0f + h * 0.0f);
                }
                if (merged) {   // contact constraints are initialised and warm-started before the joints (b2Island::Solve)
#pragma unroll
                    for (int i = 0; i < 5; ++i) { vel[player * 5 + i][0] = v[i].x; vel[player * 5 + i][1] = v[i].y; vel[player * 5 + i][2] = w[i]; }
                    __syncwarp(pair_mask);
                    if (player == 0) car_contacts_init(p.consts, recs, n_con, pose, vel, dt_ratio);
                    __syncwarp(pair_mask);
#pragma unroll
                    for (int i = 0; i < 5; ++i) { v[i] = f2(vel[player * 5 + i][0], vel[player * 5 + i][1]); w[i] = vel[player * 5 + i][2]; }
                }
                // InitVelocityConstraints (+ warm start), joints 3, 2, 1, 0
#pragma unroll
                for (int kk = 3; kk >= 0; --kk) {
                    Joint& j = J[kk];
                    const int bi = kk + 1;
                    // The wheel's anchor is its body origin = its centre of mass (localAnchorB = (0, 0), car_dynamics.py:101-110), so
                    // Box2D's rB = R(aB) * (0 - 0) is (+-0, +-0): every term it enters only adds a signed zero.  Those terms
                    // (and the sincosf of the wheel angle they need) are left out; results differ at most in the sign of a zero.
                    const Rot qA = make_rot(a[0]);
                    j.rA = rmul(qA, f2((float)(c_wheelpos[kk][0] * CR_SIZE), (float)(c_wheelpos[kk][1] * CR_SIZE)) - f2(hull_lcx, hull_lcy));
                    j.k00 = mA + mB + j.rA.y * j.rA.y * iA;
                    j.k01 = -j.rA.y * j.rA.x * iA;
                    j.k02 = -j.rA.y * iA;
                    j.k11 = mA + mB + j.rA.x * j.rA.x * iA;
                    j.k12 = j.rA.x * iA;
                    j.k22 = iA + iB;
                    solve33_prepare(j);
                    j.motor_mass = iA + iB;
                    if (j.motor_mass > 0.0f) j.motor_mass = 1.0f / j.motor_mass;
                    const float joint_angle = a[bi] - a[0] - 0.0f;
                    const float lower = -0.4f, upper = +0.4f;
                    if (joint_angle <= lower) {
                        if (j.limit_state != 1) j.iz = 0.0f;
                        j.limit_state = 1;
                    } else if (joint_angle >= upper) {
                        if (j.limit_state != 2) j.iz = 0.0f;
                        j.limit_state = 2;
                    } else {
                        j.limit_state = 0;
                        j.iz = 0.0f;
                    }
                    j.ix *= dt_ratio; j.iy *= dt_ratio; j.iz *= dt_ratio; j.motor_impulse *= dt_ratio;
                    const F2 P = f2(j.ix, j.iy);
                    v[0] = v[0] - mA * P;
                    w[0] -= iA * (cross(j.rA, P) + j.motor_impulse + j.iz);
                    v[bi] = v[bi] + mB * P;
                    w[bi] += iB * (j.motor_impulse + j.iz);
                }
                const float max_motor_impulse = h * (float)(180 * 900 * CR_SIZE * CR_SIZE);
                // Which joints are at a limit in ANY lane of the warp: decided once (InitVelocityConstraints fixed the limit
                // states), so that the 180 iterations run without the limit branch where no lane needs it.  Rear wheels
                // (joints 2, 3) are held at angle 0 by their motors and only leave it under a contact; front wheels reach
                // +-0.4 whenever the steering saturates.
                unsigned lim = 0u;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (__ballot_sync(awake_lanes, J[k].limit_state != 0) != 0u) lim |= 1u << k;
                auto contacts_after_joints = [&]() {   // merged island: contacts after the joints of both cars
#pragma unroll
                    for (int i = 0; i < 5; ++i) { vel[player * 5 + i][0] = v[i].x; vel[player * 5 + i][1] = v[i].y; vel[player * 5 + i][2] = w[i]; }
                    __syncwarp(pair_mask);
                    if (player == 0) car_contacts_solve_velocity(p.consts, recs, n_con, vel);
                    __syncwarp(pair_mask);
#pragma unroll
                    for (int i = 0; i < 5; ++i) { v[i] = f2(vel[player * 5 + i][0], vel[player * 5 + i][1]); w[i] = vel[player * 5 + i][2]; }
                };
#define CRL_VELOCITY_ITERATIONS(REAR, FRONT)                                                                        \
                _Pragma("unroll 1") for (int it = 0; it < 6 * 30; ++it) {                                            \
                    relax_joint<REAR>(J[3], v[0], w[0], v[4], w[4], mA, iA, mB, iB, max_motor_impulse);              \
                    relax_joint<REAR>(J[2], v[0], w[0], v[3], w[3], mA, iA, mB, iB, max_motor_impulse);              \
                    relax_joint<FRONT>(J[1], v[0], w[0], v[2], w[2], mA, iA, mB, iB, max_motor_impulse);             \
                    relax_joint<FRONT>(J[0], v[0], w[0], v[1], w[1], mA, iA, mB, iB, max_motor_impulse);             \
                    if (merged) contacts_after_joints();                                                             \
                }
                if (lim == 0u) { CRL_VELOCITY_ITERATIONS(false, false) }
                else if ((lim & 0xCu) == 0u) { CRL_VELOCITY_ITERATIONS(false, true) }
                else { CRL_VELOCITY_ITERATIONS(true, true) }
#undef CRL_VELOCITY_ITERATIONS
                // integrate positions
#pragma unroll
                for (int i = 0; i < 5; ++i) {
                    const F2 tr = h * v[i];
                    if (dot(tr, tr) > B2_MAX_TRANSLATION * B2_MAX_TRANSLATION) v[i] = (B2_MAX_TRANSLATION / sqrtf(dot(tr, tr))) * v[i];
                    const float r = h * w[i];
                    if (r * r > B2_MAX_ROTATION * B2_MAX_ROTATION) w[i] *= B2_MAX_ROTATION / fabsf(r);
                    c[i] = c[i] + h * v[i];
                    a[i] += h * w[i];
                }
                // position iterations
                bool position_solved = false;
#pragma unroll 1
                for (int it = 0; it < 2 * 30; ++it) {
                    bool ok = true;
                    if (merged) {   // contacts before the joints
#pragma unroll
                        for (int i = 0; i < 5; ++i) { pose[player * 5 + i][0] = c[i].x; pose[player * 5 + i][1] = c[i].y; pose[player * 5 + i][2] = a[i]; }
                        __syncwarp(pair_mask);
                        int cok = 1;
                        if (player == 0) cok = car_contacts_solve_position(p.consts, recs, n_con, pose) ? 1 : 0;
                        __syncwarp(pair_mask);
                        ok = __shfl_sync(pair_mask, cok, threadIdx.x & 30) != 0;
#pragma unroll
                        for (int i = 0; i < 5; ++i) { c[i] = f2(pose[player * 5 + i][0], pose[player * 5 + i][1]); a[i] = pose[player * 5 + i][2]; }
                    }
#pragma unroll
                    for (int kk = 3; kk >= 0; --kk) {
                        const Joint& j = J[kk];
                        const int bi = kk + 1;
                        F2 cA = c[0], cB = c[bi];
                        float aA = a[0], aB = a[bi];
                        float angular_error = 0.0f;
                        if (j.limit_state != 0) {
                            const float angle = aB - aA - 0.0f;
                            float limit_impulse;
                            if (j.limit_state == 1) {
                                float C = angle - (-0.4f);
                                angular_error = -C;
                                C = clampf(C + B2_ANGULAR_SLOP, -B2_MAX_ANGULAR_CORRECTION, 0.0f);
                                limit_impulse = -j.motor_mass * C;
                            } else {
                                float C = angle - 0.4f;
                                angular_error = C;
                                C = clampf(C - B2_ANGULAR_SLOP, 0.0f, B2_MAX_ANGULAR_CORRECTION);
                                limit_impulse = -j.motor_mass * C;
                            }
                            aA -= iA * limit_impulse;
                            aB += iB * limit_impulse;
                        }
                        const Rot qA = make_rot(aA);
                        const F2 rA = rmul(qA, f2((float)(c_wheelpos[kk][0] * CR_SIZE), (float)(c_wheelpos[kk][1] * CR_SIZE)) - f2(hull_lcx, hull_lcy));
                        const F2 C = (cB - cA) - rA;                                   // rB = (+-0, +-0), see above
                        const float position_error = sqrtf(dot(C, C));
                        const float k00 = mA + mB + iA * rA.y * rA.y;
                        const float k01 = -iA * rA.x * rA.y;
                        const float k11 = mA + mB + iA * rA.x * rA.x;
                        F2 imp = solve22(k00, k01, k01, k11, C);
                        imp = f2(-imp.x, -imp.y);
                        cA = cA - mA * imp;
                        aA -= iA * cross(rA, imp);
                        cB = cB + mB * imp;
                        c[0] = cA; a[0] = aA; c[bi] = cB; a[bi] = aB;
                        ok = (position_error <= B2_LINEAR_SLOP && angular_error <= B2_ANGULAR_SLOP) && ok;
                    }
                    if (merged) ok = __shfl_xor_sync(pair_mask, (int)ok, 1) != 0 && ok;
                    if (ok) { position_solved = true; break; }
                }
                // sleeping
                float min_sleep = 3.4e38f;
#pragma unroll
                for (int i = 0; i < 5; ++i) {
                    if (w[i] * w[i] > B2_ANGULAR_SLEEP_TOL * B2_ANGULAR_SLEEP_TOL || dot(v[i], v[i]) > B2_LINEAR_SLEEP_TOL * B2_LINEAR_SLEEP_TOL) {
                        sleep_t[i] = 0.0f;
                        min_sleep = 0.0f;
                    } else {
                        sleep_t[i] += h;
                        min_sleep = fminf(min_sleep, sleep_t[i]);
                    }
                }
                if (merged) min_sleep = fminf(min_sleep, __shfl_xor_sync(pair_mask, min_sleep, 1));
                if (min_sleep >= B2_TIME_TO_SLEEP && position_solved)
#pragma unroll
                    for (int i = 0; i < 5; ++i) { awake[i] = false; sleep_t[i] = 0.f; v[i] = f2(0.f, 0.f); w[i] = 0.f; }
            }
            inv_dt0 = 1.0f / h;
            step_count += 1;
            env_steps += 1;
        }
        // ---- store ----
        {
            float* b = p.body + (size_t)ci * 40;
#pragma unroll
            for (int i = 0; i < 5; ++i) {
                b[8 * i] = c[i].x; b[8 * i + 1] = c[i].y; b[8 * i + 2] = a[i]; b[8 * i + 3] = v[i].x; b[8 * i + 4] = v[i].y;
                b[8 * i + 5] = w[i]; b[8 * i + 6] = sleep_t[i]; b[8 * i + 7] = awake[i] ? 1.f : 0.f;
            }
            float* j = p.joint + (size_t)ci * 24;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                j[6 * k] = J[k].ix; j[6 * k + 1] = J[k].iy; j[6 * k + 2] = J[k].iz; j[6 * k + 3] = J[k].motor_impulse;
                j[6 * k + 4] = (float)J[k].limit_state; j[6 * k + 5] = J[k].motor_speed;
            }
            double* wd = p.wheel + (size_t)ci * 8;
#pragma unroll
            for (int k = 0; k < 4; ++k) wd[k] = omega[k];
            wd[4] = gas[0]; wd[5] = gas[1]; wd[6] = brake; wd[7] = steer;
            p.reward[2 * ci] = reward; p.reward[2 * ci + 1] = prev_reward;
            cn[0] = tile_visited; cn[1] = last_block; cn[2] = has_block; cn[3] = car_done ? 1 : 0;
        }
        rew[ci] = (float)step_reward;
    }
    // ---- env level: done = any(car done) (FlattenMultiAgentObservation.step, atari_wrappers.py:323-331),
    //      gym TimeLimit (register.py:14,21) ----
    bool any_done = car_done;
    if (p.players == 2) {   // done_mode 1: the env ends with car 0 (make_competitive_car_racing returns d[0], :29-33)
        const bool other = __shfl_xor_sync(0xffffffffu, (int)car_done, 1) != 0;
        if (p.done_mode == 0) any_done = any_done || other;
    }
    if (active && player == 0) {
        const int steps = p.step_count[e] + env_steps;
        p.step_count[e] = steps;
        p.inv_dt0[e] = 1.0f / (1.0f / CR_FPS);
        int el = p.elapsed[e] + 1;
        // gym TimeLimit.step: at the limit `info["TimeLimit.truncated"] = not done; done = True`.  With one car `done` is a
        // bool; with two it is CarRacing's {player: bool} dict, which is truthy, so the reference's flag is always False
        // there.  bit 1 = the limit was hit on this step (the key exists), bit 0 = its value.
        int trunc = 0;
        if (p.max_episode_steps > 0 && el >= p.max_episode_steps) {
            trunc = 2 | ((p.players == 1 && !any_done) ? 1 : 0);
            any_done = true;
        }
        p.elapsed[e] = el;
        done_out[e] = any_done ? 1 : 0;
        truncated_out[e] = (uint8_t)trunc;
        num_steps_out[e] = steps;
        p.env_done[e] = any_done ? 1 : 0;
        if (any_done) {
            atomicAdd(&p.stats[0], 1ull);
            atomicAdd(&p.stats[1], (unsigned long long)el);
            atomicAdd(&p.stats[2], (unsigned long long)p.counters[4 * ci]);
        }
    }
}

// state[car][24]: hull x, y, angle, vx, vy, w; wheel k: joint angle, omega, gas, #tiles; reward; tiles visited
__global__ void car_get_state_kernel(CarDev p, double* state) {
    const int ci = blockIdx.x * blockDim.x + threadIdx.x;
    if (ci >= p.n * p.players) return;
    const float* b = p.body + (size_t)ci * 40;
    const CarHullConst* K = p.consts;
    double* s = state + (size_t)ci * 24;
    const Rot q = make_rot(b[2]);
    const F2 pos = f2(b[0], b[1]) - rmul(q, f2(K->hull_lcx, K->hull_lcy));
    s[0] = pos.x; s[1] = pos.y; s[2] = b[2]; s[3] = b[3]; s[4] = b[4]; s[5] = b[5];
    const double* wd = p.wheel + (size_t)ci * 8;
    for (int k = 0; k < 4; ++k) {
        int cnt = 0;
        for (int i = 0; i < 16; ++i) cnt += __popc(p.touching[(size_t)ci * 64 + 16 * k + i]);
        s[6 + 4 * k] = (double)(b[8 * (k + 1) + 2] - b[2]);
        s[7 + 4 * k] = wd[k];
        s[8 + 4 * k] = (k >= 2) ? wd[4 + k - 2] : 0.0;
        s[9 + 4 * k] = cnt;
    }
    s[22] = p.reward[2 * ci];
    s[23] = p.counters[4 * ci];
}

// Put every car into a given state (debug / tests: renderer cross-checks on arbitrary states).  state[car][24] as
// car_get_state_kernel writes it; used: hull x, y, angle, vx, vy, w; per wheel joint angle, omega, gas; reward.  The
// wheels are placed on their joint anchors and move rigidly with the hull; joint impulses, contacts and the wheels'
// tile sets are cleared; tiles visited so far are kept.
__global__ void car_set_state_kernel(CarDev p, const double* state) {
    const int ci = blockIdx.x * blockDim.x + threadIdx.x;
    if (ci >= p.n * p.players) return;
    const double* s = state + (size_t)ci * 24;
    const CarHullConst* K = p.consts;
    float* b = p.body + (size_t)ci * 40;
    const float a = (float)s[2];
    const Rot q = make_rot(a);
    const F2 org = f2((float)s[0], (float)s[1]);
    const F2 com = org + rmul(q, f2(K->hull_lcx, K->hull_lcy));
    const F2 v0 = f2((float)s[3], (float)s[4]);
    const float w0 = (float)s[5];
    b[0] = com.x; b[1] = com.y; b[2] = a; b[3] = v0.x; b[4] = v0.y; b[5] = w0; b[6] = 0.f; b[7] = 1.f;
    double* wd = p.wheel + (size_t)ci * 8;
    for (int k = 0; k < 4; ++k) {
        float* w = b + 8 * (k + 1);
        const F2 wp = org + rmul(q, f2((float)(c_wheelpos[k][0] * CR_SIZE), (float)(c_wheelpos[k][1] * CR_SIZE)));
        const F2 vw = v0 + cross_sv(w0, wp - com);
        w[0] = wp.x; w[1] = wp.y; w[2] = a + (float)s[6 + 4 * k]; w[3] = vw.x; w[4] = vw.y; w[5] = w0; w[6] = 0.f; w[7] = 1.f;
        wd[k] = s[7 + 4 * k];
        if (k >= 2) wd[4 + k - 2] = s[8 + 4 * k];
    }
    wd[6] = 0.0; wd[7] = 0.0;
    float* j = p.joint + (size_t)ci * 24;
    for (int i = 0; i < 24; ++i) j[i] = 0.f;
    p.reward[2 * ci] = s[22]; p.reward[2 * ci + 1] = s[22];
    for (int i = 0; i < 64; ++i) p.touching[(size_t)ci * 64 + i] = 0u;
    if (p.n_contacts != nullptr && ci % p.players == 0) p.n_contacts[ci / p.players] = 0;
}

__global__ void car_random_actions_kernel(float* actions, int n_values, uint64_t seed, uint64_t step) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i * 4 >= n_values) return;
    uint32_t r[4];
    philox4x32_10((uint32_t)i, 1u, (uint32_t)step, (uint32_t)(step >> 32), (uint32_t)seed, (uint32_t)(seed >> 32), r);
    for (int k = 0; k < 4; ++k)
        if (i * 4 + k < n_values) actions[i * 4 + k] = (float)r[k] * (2.0f / 4294967296.0f) - 1.0f;   // U[-1, 1)
}

cudaError_t launch_car_reset(const CarDev& p, int only_done, cudaStream_t s) {
    const int blocks = only_done ? min((p.n + 1) / 2, 296) : (p.n + 1) / 2;   // a warp per env; auto-reset: over the done list
    car_reset_kernel<<<blocks, 64, 0, s>>>(p, only_done);
    return cudaGetLastError();
}

cudaError_t launch_car_pregen(const CarDev& p, cudaStream_t s) {
    car_pregen_kernel<<<(p.n + 1) / 2, 64, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_car_discard_next(const CarDev& p, cudaStream_t s) {
    car_discard_next_kernel<<<(p.n + 127) / 128, 128, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_car_step(const CarDev& p, int mode, const float* actions, float* rew, uint8_t* done, int32_t* num_steps,
                            uint8_t* truncated, cudaStream_t s) {
    const int n_cars = p.n * p.players;
    car_step_kernel<<<(n_cars + 63) / 64, 64, 0, s>>>(p, mode, actions, rew, done, num_steps, truncated);
    return cudaGetLastError();
}

cudaError_t launch_car_sensors(const CarDev& p, int classify, cudaStream_t s) {
    car_sensor_kernel<<<(p.n * p.players * 4 + 127) / 128, 128, 0, s>>>(p, classify);
    return cudaGetLastError();
}

cudaError_t launch_car_collide(const CarDev& p, cudaStream_t s) {
    if (p.players != 2) return cudaSuccess;
    car_collide_kernel<<<min(p.n, 148 * 16), 64, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_car_get_state(const CarDev& p, double* state, cudaStream_t s) {
    const int n_cars = p.n * p.players;
    car_get_state_kernel<<<(n_cars + 127) / 128, 128, 0, s>>>(p, state);
    return cudaGetLastError();
}

cudaError_t launch_car_set_state(const CarDev& p, const double* state, cudaStream_t s) {
    const int n_cars = p.n * p.players;
    car_set_state_kernel<<<(n_cars + 127) / 128, 128, 0, s>>>(p, state);
    return cudaGetLastError();
}

cudaError_t launch_car_random_actions(float* actions, int n_values, uint64_t seed, uint64_t step, cudaStream_t s) {
    car_random_actions_kernel<<<((n_values + 3) / 4 + 127) / 128, 128, 0, s>>>(actions, n_values, seed, step);
    return cudaGetLastError();
}

}  // namespace crl
