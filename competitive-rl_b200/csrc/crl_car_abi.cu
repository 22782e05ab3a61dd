// crl_car_abi.cu -- C ABI (include/crl_b200.h, crl_car_*) over the car-racing kernels. Host side only.
#include <math.h>
#include <string.h>

#include <vector>

#include "../../include/crl_b200.h"
#include "car_common.cuh"
#include "crl_host.h"

using namespace crl;

struct crl_car {
    crl_car_config cfg;
    CarDev dev;
    DeviceAllocs allocs;
    // crl_car_step of two-car envs: envs whose cars touch are stepped on a side stream while the others render
    SideStream side;
    // plain stack mode without a registered buffer rotation ("stack-shift"): the C - 1 frames that stay in the observation
    // are moved ring -> obs on this stream beside the render passes
    SideStream copy;
    // the sensor kernel of the NEXT step, started on its own stream as soon as this step's auto-resets are done
    SideStream sens;
    bool sensors_ahead = false;      // sensor_now (and, two-car envs, slow list / deferred) of the current poses are in flight or ready
    // next tracks are generated ahead of time on this stream (car_pregen_kernel); at most one launch in flight
    SideStream pregen;
    uint64_t pregen_launches = 0;
    bool was_reset = false;
    // crl_car_step_host staging
    float* actions_stage = nullptr;
    float* rew_stage = nullptr;
    uint8_t* done_stage = nullptr;
    int32_t* steps_stage = nullptr;
    uint8_t* trunc_stage = nullptr;
};

// ---- car body mass data: b2PolygonShape::Set + ComputeMass + b2Body::ResetMassData, fp32 ----
namespace {
struct P2 { float x, y; };

int hull_of(const P2* in, int n, P2* out) {   // gift wrapping exactly as b2PolygonShape::Set
    P2 ps[8];
    int m = 0;
    for (int i = 0; i < n; ++i) {
        bool unique = true;
        for (int k = 0; k < m; ++k) {
            const float dx = in[i].x - ps[k].x, dy = in[i].y - ps[k].y;
            if (dx * dx + dy * dy < 0.5f * 0.005f * 0.5f * 0.005f) { unique = false; break; }
        }
        if (unique) ps[m++] = in[i];
    }
    int i0 = 0;
    for (int i = 1; i < m; ++i)
        if (ps[i].x > ps[i0].x || (ps[i].x == ps[i0].x && ps[i].y < ps[i0].y)) i0 = i;
    int idx[8], cnt = 0, ih = i0;
    for (;;) {
        idx[cnt] = ih;
        int ie = 0;
        for (int j = 1; j < m; ++j) {
            if (ie == ih) { ie = j; continue; }
            const float rx = ps[ie].x - ps[idx[cnt]].x, ry = ps[ie].y - ps[idx[cnt]].y;
            const float vx = ps[j].x - ps[idx[cnt]].x, vy = ps[j].y - ps[idx[cnt]].y;
            const float c = rx * vy - ry * vx;
            if (c < 0.0f) ie = j;
            if (c == 0.0f && vx * vx + vy * vy > rx * rx + ry * ry) ie = j;
        }
        ++cnt;
        ih = ie;
        if (ie == i0) break;
    }
    for (int i = 0; i < cnt; ++i) out[i] = ps[idx[i]];
    return cnt;
}

void poly_mass(const P2* v, int n, float density, float* mass, P2* center, float* inertia) {
    volatile float cx = 0.f, cy = 0.f, sx = 0.f, sy = 0.f, area = 0.f, I = 0.f;
    const float inv3 = 1.0f / 3.0f;
    for (int i = 0; i < n; ++i) { sx = sx + v[i].x; sy = sy + v[i].y; }
    sx = (1.0f / n) * sx; sy = (1.0f / n) * sy;
    for (int i = 0; i < n; ++i) {
        const float e1x = v[i].x - sx, e1y = v[i].y - sy, e2x = v[(i + 1) % n].x - sx, e2y = v[(i + 1) % n].y - sy;
        volatile float D = e1x * e2y - e1y * e2x;
        volatile float tri = 0.5f * D;
        area = area + tri;
        volatile float k = tri * inv3;
        cx = cx + k * (e1x + e2x); cy = cy + k * (e1y + e2y);
        volatile float intx2 = e1x * e1x + e2x * e1x + e2x * e2x, inty2 = e1y * e1y + e2y * e1y + e2y * e2y;
        volatile float q = 0.25f * inv3 * D;
        I = I + q * (intx2 + inty2);
    }
    *mass = density * area;
    volatile float ia = 1.0f / area;
    cx = ia * cx; cy = ia * cy;
    center->x = cx + sx; center->y = cy + sy;
    volatile float in = density * I;
    volatile float d1 = center->x * center->x + center->y * center->y, d2 = cx * cx + cy * cy;
    *inertia = in + *mass * (d1 - d2);
}

// b2PolygonShape::Set after the hull: edge normals (b2Cross(edge, 1) normalised) and ComputeCentroid (pRef = origin)
void fixture_polygon(CarHullConst* K, int s, const P2* v, int n) {
    K->fix_n[s] = n;
    volatile float cx = 0.f, cy = 0.f, area = 0.f, r2 = 0.f;
    const float inv3 = 1.0f / 3.0f;
    for (int i = 0; i < n; ++i) {
        const P2 a = v[i], b = v[i + 1 < n ? i + 1 : 0];
        K->fix_vx[s][i] = a.x; K->fix_vy[s][i] = a.y;
        volatile float ex = b.x - a.x, ey = b.y - a.y;
        volatile float nx = 1.0f * ey, ny = -1.0f * ex;
        volatile float l2 = nx * nx, l2b = ny * ny;
        volatile float len = sqrtf(l2 + l2b);
        if (!(len < 1.1920929e-07f)) { volatile float inv = 1.0f / len; nx = nx * inv; ny = ny * inv; }
        K->fix_nx[s][i] = nx; K->fix_ny[s][i] = ny;
        volatile float t1 = a.x * b.y, t2 = a.y * b.x;
        volatile float D = t1 - t2;
        volatile float tri = 0.5f * D;
        area = area + tri;
        volatile float k = tri * inv3;
        volatile float sx = (0.0f + a.x) + b.x, sy = (0.0f + a.y) + b.y;
        volatile float kx = k * sx, ky = k * sy;
        cx = cx + kx; cy = cy + ky;
        volatile float q1 = a.x * a.x, q2 = a.y * a.y;
        volatile float d2 = q1 + q2;
        if (d2 > r2) r2 = d2;
    }
    volatile float ia = 1.0f / area;
    K->fix_cx[s] = ia * cx; K->fix_cy[s] = ia * cy;
    K->fix_radius[s] = sqrtf(r2);
    float c2 = 0.f;
    for (int i = 0; i < n; ++i) {
        const float dx = v[i].x - K->fix_cx[s], dy = v[i].y - K->fix_cy[s];
        if (dx * dx + dy * dy > c2) c2 = dx * dx + dy * dy;
    }
    K->fix_cradius[s] = sqrtf(c2) * 1.0001f;
}

uint8_t gray_of(double r, double g, double b) { return (uint8_t)(r * 0.299 + g * 0.587 + b * 0.114); }

void car_constants(CarHullConst* K) {
    static const float HP[4][8][2] = {
        {{-60, +130}, {+60, +130}, {+60, +110}, {-60, +110}},
        {{-15, +120}, {+15, +120}, {+20, +20}, {-20, 20}},
        {{+25, +20}, {+50, -10}, {+50, -40}, {+20, -90}, {-20, -90}, {-50, -40}, {-50, -10}, {-25, +20}},
        {{-50, -120}, {+50, -120}, {+50, -90}, {-50, -90}}};
    static const int HC[4] = {4, 4, 8, 4};
    float mass = 0.f, I = 0.f, lx = 0.f, ly = 0.f;
    for (int k = 0; k < 4; ++k) {
        P2 raw[8], hull[8];
        for (int i = 0; i < HC[k]; ++i) { raw[i].x = (float)(HP[k][i][0] * 0.02); raw[i].y = (float)(HP[k][i][1] * 0.02); }
        const int n = hull_of(raw, HC[k], hull);
        fixture_polygon(K, k, hull, n);
        float m, in;
        P2 c;
        poly_mass(hull, n, 1.0f, &m, &c, &in);
        mass += m; lx += m * c.x; ly += m * c.y; I += in;
    }
    const float inv_mass = 1.0f / mass;
    lx = inv_mass * lx; ly = inv_mass * ly;
    I -= mass * (lx * lx + ly * ly);
    K->hull_inv_mass = inv_mass; K->hull_inv_I = 1.0f / I; K->hull_lcx = lx; K->hull_lcy = ly;
    {
        const float hw = (float)(14 * 0.02), hr = (float)(27 * 0.02);
        P2 box[4] = {{+hw, -hr}, {+hw, +hr}, {-hw, +hr}, {-hw, -hr}};
        fixture_polygon(K, 4, box, 4);
        float m, in;
        P2 c;
        poly_mass(box, 4, 0.1f, &m, &c, &in);
        const float wl = c.x * c.x + c.y * c.y;
        K->wheel_inv_mass = 1.0f / m;
        K->wheel_inv_I = 1.0f / (in - m * wl);
    }
    uint8_t* g = K->gray;
    g[G_GRASS] = gray_of((int)(0.4 * 255), (int)(0.8 * 255), (int)(0.4 * 255));
    g[G_CHECK] = gray_of((int)(0.4 * 255), (int)(0.9 * 255), (int)(0.4 * 255));
    for (int k = 0; k < 3; ++k) { const double c = (int)(255 * (0.4 + 0.01 * k)); g[G_ROAD0 + k] = gray_of(c, c, c); }
    g[G_KERB_W] = gray_of(255, 255, 255); g[G_KERB_R] = gray_of(255, 0, 0);
    g[G_WHEEL] = gray_of(0, 0, 0); g[G_OWN] = gray_of((int)(0.8 * 255), 0, 0); g[G_OTHER] = gray_of(0, 0, 255);
    g[G_HUD] = gray_of(0, 0, 0); g[G_BLUE] = gray_of(0, 0, 255); g[G_BLUE2] = gray_of((int)(0.2 * 255), 0, 255);
    g[G_GREEN] = gray_of(0, 255, 0); g[G_RED] = gray_of(255, 0, 0); g[G_TEXT] = gray_of(255, 255, 255);
}

// Generate the next track of every env that has none, behind everything queued on `s` so far, on the handle's side
// stream.  Launched after every step: the host runs many steps ahead of the GPU, so "launch when the previous one has
// finished" would batch ~80 steps' worth of resets into one burst of curve walks; a launch per step keeps it at the
// handful of envs that just finished (the others' warps exit at once), and a launch that finds the previous one still
// walking simply queues behind it.  The main stream never waits for the side stream: an env that finishes again before
// its next track is ready generates it inside car_reset_kernel.  High stream priority: the few warps that have work
// live ~1.5 ms each (the walk is a serial fp64 chain) and should start at once.
int kick_pregen(crl_car* h, cudaStream_t s) {
    CUDA_TRY(h->pregen.fork(s));
    LAUNCH(launch_car_pregen(h->dev, h->pregen.stream), 1);
    h->pregen_launches += 1;
    return CRL_OK;
}

// The inputs of track generation changed (seed, injected tables, fixed tracks): tracks generated ahead are dropped
// and their attempts given back, so that what follows does not depend on how far the side stream had got.
int discard_pregen(crl_car* h, cudaStream_t s) {
    CUDA_TRY(h->pregen.sync());
    LAUNCH(launch_car_discard_next(h->dev, s), 1);
    return CRL_OK;
}

// Ahead-write stack mode: the buffer of this call must be the next one of the registered rotation (any of them at a reset).
int rotate_obs(crl_car* h, uint8_t* obs_dev, bool at_reset) {
    CarDev& d = h->dev;
    if (d.rot_n == 0) return CRL_OK;
    if (at_reset) {
        for (int i = 0; i < d.rot_n; ++i)
            if (d.rot[i] == obs_dev) { d.rot_pos = i; return CRL_OK; }
        return crl_set_error(CRL_E_INVALID, "obs_dev is not one of the %d buffers registered with crl_car_set_obs_rotation", d.rot_n);
    }
    const int next = (d.rot_pos + 1) % d.rot_n;
    if (d.rot[next] != obs_dev)
        return crl_set_error(CRL_E_INVALID, "obs_dev must be buffer %d of the registered rotation (the one after the last call's)", next);
    d.rot_pos = next;
    return CRL_OK;
}
bool moves_frames(const crl_car* h) { return !h->dev.ring_mode && h->dev.rot_n == 0 && h->dev.c >= 2; }   // internal ring + stack shift

// Stack mode: start moving the frames that stay in the observation (ring -> channels 0 .. C-2 of obs) on the copy stream,
// behind everything queued on `s` so far; finish_step makes `s` wait for it (before the auto-reset pass).
int fork_stack_shift(crl_car* h, uint8_t* obs_dev, cudaStream_t s) {
    if (!moves_frames(h)) return CRL_OK;
    CUDA_TRY(h->copy.ensure(false));
    CUDA_TRY(h->copy.fork(s));
    LAUNCH(launch_car_stack_shift(h->dev, obs_dev, h->copy.stream), 1);
    return CRL_OK;
}

// The wheel-tile overlaps (and, two-car envs, the slow list) the NEXT step needs depend only on the poses this step leaves
// behind: started on their own stream behind everything queued on `s` so far (the auto-reset spawns included), they run
// under the auto-reset render passes instead of at the head of the next step.
int sensors_ahead_of_next_step(crl_car* h, cudaStream_t s) {
    CUDA_TRY(h->sens.ensure(true));
    CUDA_TRY(h->sens.fork(s));
    if (h->dev.players == 2) CUDA_TRY(cudaMemsetAsync(h->dev.slow_count, 0, 2 * sizeof(int32_t), h->sens.stream));   // slow + near counts
    LAUNCH(launch_car_sensors(h->dev, h->dev.players == 2 ? 1 : 0, h->sens.stream), 1);
    if (h->dev.players == 2) LAUNCH(launch_car_collide(h->dev, h->sens.stream), 1);     // manifolds of the near envs -> slow list
    h->sensors_ahead = true;
    return CRL_OK;
}

// At the head of a step: wait for the sensors (and, two-car envs, the manifolds and the slow list) started ahead, or run
// them now (first step, after set_state / reset).
int sensors_for_this_step(crl_car* h, cudaStream_t s) {
    if (h->sensors_ahead) {
        CUDA_TRY(h->sens.join(s));
        h->sensors_ahead = false;
        return CRL_OK;
    }
    const int two = h->dev.players == 2 ? 1 : 0;
    if (two) CUDA_TRY(cudaMemsetAsync(h->dev.slow_count, 0, 2 * sizeof(int32_t), s));
    LAUNCH(launch_car_sensors(h->dev, two, s), 1);
    if (two) LAUNCH(launch_car_collide(h->dev, s), 1);
    return CRL_OK;
}

// Before anything that moves the cars between steps (reset, set_state): what was computed ahead no longer holds, and the
// kernel computing it must not be reading the bodies while they are rewritten.
int drop_sensors_ahead(crl_car* h, cudaStream_t s) {
    if (!h->sensors_ahead) return CRL_OK;
    CUDA_TRY(h->sens.join(s));
    h->sensors_ahead = false;
    return CRL_OK;
}

// The tail of every step: the auto-reset of finished envs and their reset observation, with the next step's sensors and
// tracks started ahead.
int finish_step(crl_car* h, uint8_t* obs_dev, cudaStream_t s) {
    if (moves_frames(h)) {
        CUDA_TRY(h->copy.join(s));                                             // it reads ring_pos; the auto-reset pass rewrites whole stacks
        LAUNCH(launch_car_ring_advance(h->dev, s), 1);
    }
    LAUNCH(launch_car_reset(h->dev, 1, s), 1);                                 // auto-reset of finished envs
    if (int r = sensors_ahead_of_next_step(h, s)) return r;
    LAUNCH(launch_car_render(h->dev, 1, 0, 1, obs_dev, nullptr, s), 3);        // their reset observation
    return kick_pregen(h, s);
}
}  // namespace

extern "C" {

int crl_car_destroy(crl_car* h) {
    if (!h) return CRL_OK;
    CrlDeviceGuard guard(h->cfg.device);
    SideStream* streams[] = {&h->side, &h->copy, &h->sens, &h->pregen};
    for (SideStream* st : streams) st->sync();      // kernels on them read the buffers freed below
    h->allocs.free_all();
    for (SideStream* st : streams) st->destroy();
    delete h;
    return CRL_OK;
}

int crl_car_create(const crl_car_config* cfg, crl_car** out) {
    if (!cfg || !out) return crl_set_error(CRL_E_INVALID, "null argument");
    *out = nullptr;
    if (cfg->num_envs <= 0) return crl_set_error(CRL_E_INVALID, "num_envs must be positive");
    if (cfg->num_players != 1 && cfg->num_players != 2) return crl_set_error(CRL_E_INVALID, "num_players must be 1 or 2");
    if (cfg->frame_stack < 0 || cfg->frame_stack > CAR_MAX_STACK)
        return crl_set_error(CRL_E_INVALID, "frame_stack must be in [0, %d]", CAR_MAX_STACK);
    if (cfg->stack_mode != 0 && cfg->stack_mode != 1) return crl_set_error(CRL_E_INVALID, "stack_mode must be 0 (stack) or 1 (ring)");
    if (cfg->stack_mode == 1 && cfg->frame_stack < 2) return crl_set_error(CRL_E_INVALID, "stack_mode ring needs frame_stack >= 2");
    if (cfg->done_mode != 0 && cfg->done_mode != 1) return crl_set_error(CRL_E_INVALID, "done_mode must be 0 (any car) or 1 (car 0)");
    if (int r = crl_check_device(cfg->device)) return r;
    CrlDeviceGuard guard(cfg->device);
    CUDA_TRY(guard.err);
    crl_car* h = new crl_car();
    h->cfg = *cfg;
    CarDev& d = h->dev;
    memset(&d, 0, sizeof d);
    const size_t n = (size_t)cfg->num_envs, P = (size_t)cfg->num_players, nc = n * P;
    d.n = cfg->num_envs; d.players = cfg->num_players; d.c = cfg->frame_stack > 0 ? cfg->frame_stack : 1;
    d.action_repeat = cfg->action_repeat > 0 ? cfg->action_repeat : 1;
    d.max_episode_steps = cfg->max_episode_steps;
    d.done_mode = cfg->done_mode;
    d.ring_mode = cfg->stack_mode == 1 ? 1 : 0;
    d.first_env = cfg->first_env; d.seed = cfg->seed;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](auto** p, size_t count) { if (e == cudaSuccess) e = h->allocs.alloc(p, count); };
    alloc(&d.n_track, 2 * n); alloc(&d.tiles, 2 * n * CAR_MAX_TRACK); alloc(&d.samples, 2 * n * CAR_MAX_SAMPLES);
    alloc(&d.start_pose, 2 * n * 3); alloc(&d.track_pts, 2 * n * CAR_MAX_TRACK * 3);
    alloc(&d.sel, n); alloc(&d.next_state, n); alloc(&d.next_att0, n); alloc(&d.raw_ring, n * CAR_RAW_RING * 3);
    alloc(&d.step_count, n); alloc(&d.elapsed, n); alloc(&d.reset_count, n);
    alloc(&d.attempt_count, n); alloc(&d.inv_dt0, n); alloc(&d.env_done, n); alloc(&d.ring_pos, n);
    alloc(&d.body, nc * 40); alloc(&d.joint, nc * 24); alloc(&d.wheel, nc * 8); alloc(&d.reward, nc * 2);
    alloc(&d.counters, nc * 4); alloc(&d.touching, nc * 64); alloc(&d.visited, nc * 16); alloc(&d.sensor_now, nc * 64);
    alloc(&d.overrun, 4); alloc(&d.stats, 8);
    alloc(&d.contact_overflow, 1);
    {
        uint8_t* fmraw = nullptr;
        alloc(&fmraw, nc * car_frame_map_bytes());
        d.frame_map = reinterpret_cast<FrameMap*>(fmraw);
        alloc(&d.frame_aux, nc * car_frame_aux_bytes());
    }
    alloc(&d.map_index, 2 * n * CAR_MAP_GRID * CAR_MAP_GRID); alloc(&d.map_blocks, 2 * n * CAR_MAP_MAX_BLOCKS * 256);
    alloc(&d.tile_centres, 2 * n * CAR_MAX_TRACK); alloc(&d.wide_tiles, 2 * n * CAR_MAX_WIDE);
    alloc(&h->actions_stage, nc * 2); alloc(&h->rew_stage, nc); alloc(&h->done_stage, n); alloc(&h->steps_stage, n); alloc(&h->trunc_stage, n);
    if (P == 2) { alloc(&d.contacts, n * CAR_MAX_CONTACTS); alloc(&d.n_contacts, n); alloc(&d.n_contacts_step, n); alloc(&d.slow_list, n); alloc(&d.slow_count, 2); d.near_count = d.slow_count + 1; alloc(&d.near_list, n); }
    alloc(&d.deferred, n);
    alloc(&d.done_list, n); alloc(&d.done_count, 1);
    CarHullConst* kdev = nullptr;
    alloc(&kdev, 1);
    if (e != cudaSuccess) {
        crl_car_destroy(h);
        return crl_set_error(CRL_E_CUDA, "cudaMalloc: %s", cudaGetErrorString(e));
    }
    CarHullConst K;
    memset(&K, 0, sizeof K);
    car_constants(&K);
    car_checker_table(K.checker);
    e = cudaMemcpy(kdev, &K, sizeof K, cudaMemcpyHostToDevice);
    {   // checker squares as byte flags over the road-map window (the same bounds on both axes, kept per axis anyway)
        std::vector<uint8_t> chk(2 * 2048, 0);
        for (int axis = 0; axis < 2; ++axis)
            for (int i = 0; i < 20; ++i)
                for (int v = K.checker[(axis * 20 + i) * 2]; v <= K.checker[(axis * 20 + i) * 2 + 1]; ++v)
                    if (v >= CAR_MAP_ORIGIN && v < CAR_MAP_ORIGIN + 2048) chk[axis * 2048 + v - CAR_MAP_ORIGIN] = 0xFF;
        uint8_t* cdev = nullptr;
        if (e == cudaSuccess) e = h->allocs.alloc(&cdev, chk.size());
        if (e == cudaSuccess) e = cudaMemcpy(cdev, chk.data(), chk.size(), cudaMemcpyHostToDevice);
        d.chk = cdev;
    }
    if (e == cudaSuccess) e = cudaMemset(d.ring_pos, 0xFF, n * sizeof(int32_t));
    if (e == cudaSuccess) e = car_raster_init();
    if (e != cudaSuccess) {
        crl_car_destroy(h);
        return crl_set_error(CRL_E_CUDA, "init: %s", cudaGetErrorString(e));
    }
    d.consts = kdev;
    e = h->pregen.ensure(true);
    if (e != cudaSuccess) {
        crl_car_destroy(h);
        return crl_set_error(CRL_E_CUDA, "pregen stream: %s", cudaGetErrorString(e));
    }
    *out = h;
    return CRL_OK;
}

int crl_car_load_glyphs(crl_car* h, const uint8_t* glyphs_host, size_t bytes, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!glyphs_host || bytes != (size_t)CRL_CAR_GLYPH_BYTES) return crl_set_error(CRL_E_INVALID, "glyph atlas must be %d bytes", CRL_CAR_GLYPH_BYTES);
    uint8_t* g = nullptr;
    CUDA_TRY(h->allocs.alloc(&g, bytes));
    CUDA_TRY(cudaMemcpyAsync(g, glyphs_host, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    const uint8_t* old = h->dev.glyphs;
    h->dev.glyphs = g;
    CUDA_TRY(h->allocs.free(old));
    return CRL_OK;
}

int crl_car_inject_tracks(crl_car* h, const double* draws_host, int32_t k_draws, const int32_t* birth_host,
                          int32_t k_birth, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!draws_host || k_draws < 1) return crl_set_error(CRL_E_INVALID, "need at least one attempt of draws per env");
    cudaStream_t s = (cudaStream_t)stream;
    double* dd = nullptr;
    const size_t cnt = (size_t)h->dev.n * k_draws * CAR_DRAWS;
    CUDA_TRY(h->allocs.alloc(&dd, cnt));
    CUDA_TRY(cudaMemcpyAsync(dd, draws_host, cnt * sizeof(double), cudaMemcpyHostToDevice, s));
    if (int r = discard_pregen(h, s)) return r;
    const void* old[2] = {h->dev.track_draws, nullptr};
    h->dev.track_draws = dd; h->dev.k_draws = k_draws;
    if (birth_host && k_birth > 0) {                // without one, the previous birth table stays
        int32_t* bb = nullptr;
        const size_t bc = (size_t)h->dev.n * k_birth * h->dev.players;
        CUDA_TRY(h->allocs.alloc(&bb, bc));
        CUDA_TRY(cudaMemcpyAsync(bb, birth_host, bc * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        old[1] = h->dev.birth;
        h->dev.birth = bb; h->dev.k_birth = k_birth;
    }
    CUDA_TRY(cudaMemsetAsync(h->dev.attempt_count, 0, (size_t)h->dev.n * sizeof(int32_t), s));
    CUDA_TRY(cudaMemsetAsync(h->dev.reset_count, 0, (size_t)h->dev.n * sizeof(int32_t), s));
    CUDA_TRY(cudaStreamSynchronize(s));
    for (const void* p : old) CUDA_TRY(h->allocs.free(p));
    return CRL_OK;
}

// Tiles of a recorded track (beta, x, y per point) that the kernel would list in wide_tiles (generate_track_warp), counted
// in fp64 with 0.05 units of margin on the kernel's fp32 thresholds, over the 5 listed vertices (the hull is a subset).
static int count_wide_tiles(const double* pts, int n) {
    const double w = 40.0 / 6.0, pi = 3.141592653589793;
    int wide = 0;
    for (int i = 0; i < n; ++i) {
        const double *p1 = pts + 3 * i, *p2 = pts + 3 * ((i - 1 + n) % n), *ps = pts + 3 * (i - i % CAR_SAMPLE_STRIDE);
        const double vx[5] = {p1[1] - w * cos(p1[0]), p1[1] - w / 2 * cos(p1[0] - pi / 2), p1[1] + w * cos(p1[0]),
                              p2[1] + w * cos(p2[0]), p2[1] - w * cos(p2[0])};
        const double vy[5] = {p1[2] - w * sin(p1[0]), p1[2] - w / 2 * sin(p1[0] - pi / 2), p1[2] + w * sin(p1[0]),
                              p2[2] + w * sin(p2[0]), p2[2] - w * sin(p2[0])};
        double reach = 0.0;
        for (int k = 0; k < 5; ++k) reach = fmax(reach, hypot(vx[k] - p1[1], vy[k] - p1[2]));
        if (reach > CAR_WIDE_REACH - 0.05 || hypot(p1[1] - ps[1], p1[2] - ps[2]) > CAR_WIDE_GROUP - 0.05) ++wide;
    }
    return wide;
}

int crl_car_load_tracks(crl_car* h, const double* pts_host, const int32_t* counts_host, int32_t n_tracks, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    cudaStream_t s = (cudaStream_t)stream;
    if (int r = discard_pregen(h, s)) return r;
    CUDA_TRY(cudaStreamSynchronize(s));
    const void* old[2] = {h->dev.fixed_tracks, h->dev.fixed_counts};
    if (n_tracks <= 0) {                       // back to generated tracks
        h->dev.fixed_tracks = nullptr; h->dev.fixed_counts = nullptr; h->dev.n_fixed = 0;
        for (const void* p : old) CUDA_TRY(h->allocs.free(p));
        return CRL_OK;
    }
    if (!pts_host || !counts_host) return crl_set_error(CRL_E_INVALID, "null track buffer");
    for (int k = 0; k < n_tracks; ++k)
        if (counts_host[k] < 9 || counts_host[k] > CAR_MAX_TRACK)
            return crl_set_error(CRL_E_INVALID, "track %d has %d points; need 9..%d", k, counts_host[k], CAR_MAX_TRACK);
    for (int k = 0; k < n_tracks; ++k) {
        const int wide = count_wide_tiles(pts_host + (size_t)k * CAR_MAX_TRACK * 3, counts_host[k]);
        if (wide > CAR_MAX_WIDE)
            return crl_set_error(CRL_E_INVALID, "track %d: %d tiles reach farther from their track point than the wheel-tile "
                                 "contact search covers (at most %d per track; points too far apart?)", k, wide, CAR_MAX_WIDE);
    }
    double* dp = nullptr;
    int32_t* dc = nullptr;
    CUDA_TRY(h->allocs.alloc(&dp, (size_t)n_tracks * CAR_MAX_TRACK * 3));
    CUDA_TRY(h->allocs.alloc(&dc, (size_t)n_tracks));
    CUDA_TRY(cudaMemcpyAsync(dp, pts_host, (size_t)n_tracks * CAR_MAX_TRACK * 3 * sizeof(double), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(dc, counts_host, (size_t)n_tracks * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    h->dev.fixed_tracks = dp; h->dev.fixed_counts = dc; h->dev.n_fixed = n_tracks;
    for (const void* p : old) CUDA_TRY(h->allocs.free(p));
    return CRL_OK;
}

int crl_car_reset(crl_car* h, uint8_t* obs_dev, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!obs_dev) return crl_set_error(CRL_E_INVALID, "null observation buffer");
    cudaStream_t s = (cudaStream_t)stream;
    if (int r = rotate_obs(h, obs_dev, true)) return r;
    if (int r = drop_sensors_ahead(h, s)) return r;
    if (!h->dev.ring_mode && h->dev.rot_n == 0 && h->dev.ring == nullptr)   // the internal frame ring of the plain stack mode, on first use (1.2 GB at config 5)
        CUDA_TRY(h->allocs.alloc(&h->dev.ring, (size_t)h->dev.n * h->dev.players * h->dev.c * CAR_PIX));
    CUDA_TRY(cudaMemsetAsync(h->dev.ring_pos, 0xFF, (size_t)h->dev.n * sizeof(int32_t), s));
    CUDA_TRY(cudaMemsetAsync(h->dev.env_done, 0, (size_t)h->dev.n, s));
    h->dev.ring_phase = 0;
    h->dev.fill_all = 1;      // until the next step: every frame written goes to all slots of its ring
    LAUNCH(launch_car_reset(h->dev, 0, s), 1);
    LAUNCH(launch_car_render(h->dev, 0, 0, 1, obs_dev, nullptr, s), 4);
    h->was_reset = true;
    return kick_pregen(h, s);
}

int crl_car_step_state(crl_car* h, const float* actions_dev, float* rew_dev, uint8_t* done_dev,
                       int32_t* num_steps_dev, uint8_t* truncated_dev, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!h->was_reset) return crl_set_error(CRL_E_STATE, "reset must be called before step");
    if (!actions_dev || !rew_dev || !done_dev || !num_steps_dev || !truncated_dev) return crl_set_error(CRL_E_INVALID, "null step buffer");
    h->dev.fill_all = 0;
    if (h->dev.ring_mode) h->dev.ring_phase = (h->dev.ring_phase + 1) % h->dev.c;
    if (int r = sensors_for_this_step(h, (cudaStream_t)stream)) return r;
    LAUNCH(launch_car_step(h->dev, 0, actions_dev, rew_dev, done_dev, num_steps_dev, truncated_dev, (cudaStream_t)stream), 1);
    return CRL_OK;
}

int crl_car_render_obs(crl_car* h, uint8_t* obs_dev, uint8_t* term_obs_dev, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!h->was_reset) return crl_set_error(CRL_E_STATE, "reset must be called before step");
    if (!obs_dev) return crl_set_error(CRL_E_INVALID, "null observation buffer");
    cudaStream_t s = (cudaStream_t)stream;
    if (int r = rotate_obs(h, obs_dev, false)) return r;
    if (moves_frames(h)) LAUNCH(launch_car_stack_shift(h->dev, obs_dev, s), 1);   // the frames that stay: ring -> obs
    CUDA_TRY(cudaMemsetAsync(h->dev.done_count, 0, sizeof(int32_t), s));
    h->dev.collect_done = 1;
    LAUNCH(launch_car_render(h->dev, 0, 0, 1, obs_dev, term_obs_dev, s), 4);   // post-step frame (terminal obs of finished envs)
    h->dev.collect_done = 0;
    LAUNCH(launch_car_reset(h->dev, 1, s), 1);                                 // auto-reset of finished envs
    LAUNCH(launch_car_render(h->dev, 1, 0, 1, obs_dev, nullptr, s), 3);        // their reset observation
    return kick_pregen(h, s);
}

int crl_car_step(crl_car* h, const float* actions_dev, uint8_t* obs_dev, float* rew_dev, uint8_t* done_dev,
                 int32_t* num_steps_dev, uint8_t* truncated_dev, uint8_t* term_obs_dev, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!h->was_reset) return crl_set_error(CRL_E_STATE, "reset must be called before step");
    if (!actions_dev || !obs_dev || !rew_dev || !done_dev || !num_steps_dev || !truncated_dev) return crl_set_error(CRL_E_INVALID, "null step buffer");
    cudaStream_t s = (cudaStream_t)stream;
    if (h->dev.players == 1) {
        if (int r = rotate_obs(h, obs_dev, false)) return r;      // after the argument checks: a refused call leaves the rotation where it was
        if (int r = crl_car_step_state(h, actions_dev, rew_dev, done_dev, num_steps_dev, truncated_dev, stream)) return r;
        if (int r = fork_stack_shift(h, obs_dev, s)) return r;                     // next to the render pass
        CUDA_TRY(cudaMemsetAsync(h->dev.done_count, 0, sizeof(int32_t), s));
        h->dev.collect_done = 1;
        LAUNCH(launch_car_render(h->dev, 0, 0, 0, obs_dev, term_obs_dev, s), 3);   // post-step frame (terminal obs of finished envs)
        h->dev.collect_done = 0;
        return finish_step(h, obs_dev, s);
    }
    // Two-car envs.  The step kernel is one wave of latency-bound threads; lane pairs whose cars touch run the sequential
    // contact solver and take several times longer than the rest.  So the sensor kernel lists the envs whose cars are near
    // each other, the listed envs are stepped on a side stream (slow pass) WHILE the main stream steps the others (fast
    // pass) and renders their frames; the frames of the listed envs follow.  Per env nothing changes; only the launch
    // schedule does.  (Without a registered buffer rotation the frames that stay in the observation stack move ring -> obs
    // on a third stream meanwhile.)
    CUDA_TRY(h->side.ensure(true));
    if (int r = rotate_obs(h, obs_dev, false)) return r;
    h->dev.fill_all = 0;
    if (h->dev.ring_mode) h->dev.ring_phase = (h->dev.ring_phase + 1) % h->dev.c;
    CUDA_TRY(cudaMemsetAsync(h->dev.done_count, 0, sizeof(int32_t), s));
    if (int r = sensors_for_this_step(h, s)) return r;                         // wheel-tile overlaps, manifolds, the slow list
    CUDA_TRY(h->side.fork(s));
    LAUNCH(launch_car_step(h->dev, 2, actions_dev, rew_dev, done_dev, num_steps_dev, truncated_dev, h->side.stream), 1);
    LAUNCH(launch_car_step(h->dev, 1, actions_dev, rew_dev, done_dev, num_steps_dev, truncated_dev, s), 1);
    // "stack-shift" only: the frames that stay in the stack, ring -> obs, next to the render passes (DRAM-bound beside
    // issue-bound; the step kernels before it fill the register files, so it is not started under them)
    if (int r = fork_stack_shift(h, obs_dev, s)) return r;
    h->dev.collect_done = 1;
    LAUNCH(launch_car_render(h->dev, 0, 1, 0, obs_dev, term_obs_dev, s), 3);   // frames of the envs stepped by the fast pass
    CUDA_TRY(h->side.join(s));
    LAUNCH(launch_car_render(h->dev, 0, 2, 0, obs_dev, term_obs_dev, s), 3);   // frames of the listed envs
    h->dev.collect_done = 0;
    return finish_step(h, obs_dev, s);
}

int crl_car_seed(crl_car* h, uint64_t seed, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (int r = discard_pregen(h, (cudaStream_t)stream)) return r;
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    h->dev.seed = seed;
    return CRL_OK;
}

int crl_car_set_elapsed(crl_car* h, const int32_t* elapsed_dev, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!elapsed_dev) return crl_set_error(CRL_E_INVALID, "null buffer");
    CUDA_TRY(cudaMemcpyAsync(h->dev.elapsed, elapsed_dev, (size_t)h->dev.n * sizeof(int32_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return CRL_OK;
}

int crl_car_step_host(crl_car* h, const float* actions_host, uint8_t* obs_dev, uint8_t* obs_host, float* rew_host,
                      uint8_t* done_host, int32_t* num_steps_host, uint8_t* truncated_host, uint8_t* term_obs_dev, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!actions_host || !obs_dev || !rew_host || !done_host) return crl_set_error(CRL_E_INVALID, "null host buffer");
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)h->dev.n, nc = n * h->dev.players;
    CUDA_TRY(cudaMemcpyAsync(h->actions_stage, actions_host, nc * 2 * sizeof(float), cudaMemcpyHostToDevice, s));
    if (int r = crl_car_step(h, h->actions_stage, obs_dev, h->rew_stage, h->done_stage, h->steps_stage, h->trunc_stage,
                             term_obs_dev, stream)) return r;
    CUDA_TRY(cudaMemcpyAsync(rew_host, h->rew_stage, nc * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(done_host, h->done_stage, n, cudaMemcpyDeviceToHost, s));
    if (num_steps_host) CUDA_TRY(cudaMemcpyAsync(num_steps_host, h->steps_stage, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (truncated_host) CUDA_TRY(cudaMemcpyAsync(truncated_host, h->trunc_stage, n, cudaMemcpyDeviceToHost, s));
    if (obs_host) CUDA_TRY(cudaMemcpyAsync(obs_host, obs_dev, nc * (h->dev.ring_mode ? 2 : 1) * h->dev.c * CAR_PIX, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return CRL_OK;
}

int crl_car_get_state(crl_car* h, double* state_dev, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!state_dev) return crl_set_error(CRL_E_INVALID, "null buffer");
    LAUNCH(launch_car_get_state(h->dev, state_dev, (cudaStream_t)stream), 1);
    return CRL_OK;
}

int crl_car_set_state(crl_car* h, const double* state_dev, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!state_dev) return crl_set_error(CRL_E_INVALID, "null buffer");
    if (!h->was_reset) return crl_set_error(CRL_E_STATE, "reset must be called before set_state");
    if (int r = drop_sensors_ahead(h, (cudaStream_t)stream)) return r;
    LAUNCH(launch_car_set_state(h->dev, state_dev, (cudaStream_t)stream), 1);
    return CRL_OK;
}

int crl_car_render_state(crl_car* h, uint8_t* obs_dev, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!h->was_reset) return crl_set_error(CRL_E_STATE, "reset must be called before rendering");
    if (!obs_dev) return crl_set_error(CRL_E_INVALID, "null observation buffer");
    if (int r = rotate_obs(h, obs_dev, false)) return r;
    h->dev.fill_all = 0;
    if (h->dev.ring_mode) h->dev.ring_phase = (h->dev.ring_phase + 1) % h->dev.c;
    if (moves_frames(h)) LAUNCH(launch_car_stack_shift(h->dev, obs_dev, (cudaStream_t)stream), 1);
    LAUNCH(launch_car_render(h->dev, 0, 0, 1, obs_dev, nullptr, (cudaStream_t)stream), 4);
    return CRL_OK;
}

int crl_car_set_obs_rotation(crl_car* h, uint8_t* const* obs_devs_host, int32_t count, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    CarDev& d = h->dev;
    if (count == 0) { d.rot_n = 0; d.rot_pos = 0; h->was_reset = false; return CRL_OK; }   // plain mode again, from the next reset on
    if (d.ring_mode) return crl_set_error(CRL_E_STATE, "stack_mode ring has no use for a buffer rotation");
    if (d.c < 2) return crl_set_error(CRL_E_STATE, "a buffer rotation needs frame_stack >= 2");
    if (!obs_devs_host || count < d.c + 1 || count > CAR_MAX_ROTATION)
        return crl_set_error(CRL_E_INVALID, "need frame_stack + 1 .. %d buffers, got %d", CAR_MAX_ROTATION, count);
    for (int i = 0; i < count; ++i) {
        if (!obs_devs_host[i]) return crl_set_error(CRL_E_INVALID, "null buffer %d", i);
        for (int k = 0; k < i; ++k)
            if (obs_devs_host[k] == obs_devs_host[i]) return crl_set_error(CRL_E_INVALID, "buffers %d and %d are the same", k, i);
    }
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    for (int i = 0; i < count; ++i) d.rot[i] = obs_devs_host[i];
    d.rot_n = count; d.rot_pos = 0;
    h->was_reset = false;                  // the stacks are rebuilt by the next reset
    return CRL_OK;
}

int crl_car_ring_phase(crl_car* h) {
    if (!h) return crl_set_error(CRL_E_INVALID, "null handle");
    if (!h->dev.ring_mode) return crl_set_error(CRL_E_STATE, "the handle was not created with stack_mode ring");
    return h->dev.ring_phase;
}

int crl_car_get_track(crl_car* h, int32_t env, int32_t* n_out, double* pts_host, int32_t max_points, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (env < 0 || env >= h->dev.n || !n_out) return crl_set_error(CRL_E_INVALID, "bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    int32_t n = 0, sel = 0;
    CUDA_TRY(cudaMemcpyAsync(&sel, h->dev.sel + env, sizeof sel, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    const size_t slot = (size_t)env + (size_t)h->dev.n * (sel ? 1 : 0);
    CUDA_TRY(cudaMemcpyAsync(&n, h->dev.n_track + slot, sizeof n, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    *n_out = n;
    if (pts_host) {
        const int m = n < max_points ? n : max_points;
        if (m > 0)
            CUDA_TRY(cudaMemcpy(pts_host, h->dev.track_pts + slot * CAR_MAX_TRACK * 3, (size_t)m * 3 * sizeof(double), cudaMemcpyDeviceToHost));
    }
    return CRL_OK;
}

int crl_car_random_actions(float* actions_dev, int32_t n_values, uint64_t seed, uint64_t step, void* stream) {
    if (!actions_dev || n_values <= 0) return crl_set_error(CRL_E_INVALID, "bad arguments");
    LAUNCH(launch_car_random_actions(actions_dev, n_values, seed, step, (cudaStream_t)stream), 1);
    return CRL_OK;
}

int crl_car_get_stats(crl_car* h, uint64_t* stats_host, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    if (!stats_host) return crl_set_error(CRL_E_INVALID, "null buffer");
    if (int r = crl_read_counters(h->dev.stats, stats_host, 8, (cudaStream_t)stream)) return r;
    int32_t flags[4] = {0, 0, 0, 0};
    CUDA_TRY(cudaMemcpyAsync(flags, h->dev.overrun, sizeof flags, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    stats_host[3] = (uint64_t)flags[3];
    stats_host[4] = (uint64_t)flags[2];
    stats_host[5] = h->pregen_launches;
    return CRL_OK;
}

int crl_car_get_contacts(crl_car* h, int32_t* counts_host, int32_t* overflow_host, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    cudaStream_t s = (cudaStream_t)stream;
    if (counts_host) {
        if (h->dev.n_contacts_step) CUDA_TRY(cudaMemcpyAsync(counts_host, h->dev.n_contacts_step, (size_t)h->dev.n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        else memset(counts_host, 0, (size_t)h->dev.n * sizeof(int32_t));
    }
    if (overflow_host) CUDA_TRY(cudaMemcpyAsync(overflow_host, h->dev.contact_overflow, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return CRL_OK;
}

int crl_car_check(crl_car* h, void* stream) {
    CHECK_HANDLE(h, h->cfg.device);
    int32_t flags[4] = {0, 0, 0, 0};
    CUDA_TRY(cudaMemcpyAsync(flags, h->dev.overrun, sizeof flags, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    const int32_t flag = flags[0];
    if (flag != 0 || flags[1] != 0)                                   // reported once: the flags are cleared ([2], [3] are statistics)
        CUDA_TRY(cudaMemsetAsync(h->dev.overrun, 0, 2 * sizeof(int32_t), (cudaStream_t)stream));
    if (flags[1] != 0) return crl_set_error(CRL_E_STATE, "road map: %d span(s) / block(s) of a track could not be painted (outside the 2048 px map window or block pool full)", flags[1]);
    if (flag == 1) return crl_set_error(CRL_E_SERVES, "injected track-draw / birth-place table exhausted");
    if (flag == 2) return crl_set_error(CRL_E_STATE, "track generation failed 64 times in a row");
    return CRL_OK;
}

}  // extern "C"
