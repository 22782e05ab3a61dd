// crl_abi.cu -- C ABI (include/crl_b200.h) over the Pong kernels.  Host-side only:
// allocation, table setup, launch sequencing.  No CPU fallback exists: every entry
// point needs a CUDA device.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cuda.h>

#include <atomic>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "../../include/crl_b200.h"
#include "crl_host.h"
#include "pong_common.cuh"

using namespace crl;

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

int crl_set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
void crl_count_launch(int n) { g_launches += (uint64_t)n; }

#define CUDA_TRY(expr)                                                                                \
    do {                                                                                              \
        cudaError_t _e = (expr);                                                                      \
        if (_e != cudaSuccess) return fail(CRL_E_CUDA, "%s: %s", #expr, cudaGetErrorString(_e));      \
    } while (0)

#define LAUNCH(expr)     \
    do {                 \
        CUDA_TRY(expr);  \
        g_launches += 1; \
    } while (0)

struct crl_pong {
    crl_pong_config cfg;
    PongDev dev;
    std::vector<void*> allocs;
    double* serves_dev = nullptr;
    uint8_t* atlas_dev = nullptr;
    uint8_t* text_tab_dev = nullptr;
    uint8_t* tmpl_dev = nullptr;
    AreaTabs* tabs_dev = nullptr;
    AreaTabs tabs_host;
    uint8_t* fast_tabs_dev = nullptr;
    int32_t* actions_stage = nullptr;   // device staging for crl_pong_step_host
    float* rew_stage = nullptr;
    uint8_t* done_stage = nullptr;
    int32_t* steps_stage = nullptr;
    float* real_stage = nullptr;
    bool atlas_loaded = false;
    bool was_reset = false;
    // crl_pong_step_host: the small results go back to the host on a side stream while the rasteriser runs
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_state = nullptr, ev_copied = nullptr;
    // crl_pong_set_obs_buffers: observation buffers whose contents the library tracks.  shown ([agent][c][n] FrameSpecs per
    // set) describes what the set's buffers hold while `valid`; renders into a valid set store only what changed.
    struct ObsSet {
        uint8_t* obs[2];
        FrameSpec* shown;
        bool valid;
    };
    std::vector<ObsSet> sets;
    FrameSpec* shown_dev = nullptr;
    bool full_obs = false;      // CRL_PONG_FULL_OBS: every render stores whole stacks
};

static size_t obs_bytes(const crl_pong* h) {
    return (size_t)h->dev.n * (h->dev.ring ? 2 * h->dev.c : h->dev.c) * h->dev.dim * h->dev.dim;
}

// [p, p + bytes) was written by something other than a tracked render: the sets it overlaps no longer know their contents
static void obs_written(crl_pong* h, const void* p, size_t bytes) {
    if (!p) return;
    const uintptr_t a = (uintptr_t)p, b = a + bytes, ob = obs_bytes(h);
    for (auto& st : h->sets)
        for (int k = 0; k < h->dev.n_agents; ++k)
            if (a < (uintptr_t)st.obs[k] + ob && (uintptr_t)st.obs[k] < b) st.valid = false;
}

// OpenCV computeResizeAreaTab (SURVEY.md A.2): scale and cell in double, alpha stored as float.
static bool build_axis(int ssize, int dsize, uint8_t* src0, uint8_t* cnt, float (*alpha)[MAX_TAPS], uint8_t* first,
                       uint8_t* last) {
    const double scale = (double)ssize / dsize;
    for (int s = 0; s < ssize; ++s) { first[s] = 255; last[s] = 0; }
    for (int dx = 0; dx < dsize; ++dx) {
        const double fsx1 = dx * scale, fsx2 = fsx1 + scale;
        const double cell = fmin(scale, ssize - fsx1);
        int sx1 = (int)ceil(fsx1), sx2 = (int)floor(fsx2);
        sx2 = sx2 < ssize - 1 ? sx2 : ssize - 1;
        sx1 = sx1 < sx2 ? sx1 : sx2;
        int n = 0, s0 = -1;
        auto emit = [&](int s, float a) -> bool {
            if (n == 0) s0 = s;
            if (n >= MAX_TAPS || s != s0 + n) return false;
            alpha[dx][n++] = a;
            if (first[s] == 255) first[s] = (uint8_t)dx;
            last[s] = (uint8_t)dx;
            return true;
        };
        if (sx1 - fsx1 > 1e-3 && !emit(sx1 - 1, (float)((sx1 - fsx1) / cell))) return false;
        for (int sx = sx1; sx < sx2; ++sx)
            if (!emit(sx, (float)(1.0 / cell))) return false;
        if (fsx2 - sx2 > 1e-3 && !emit(sx2, (float)(fmin(fmin(fsx2 - sx2, 1.0), cell) / cell))) return false;
        if (n == 0) return false;
        src0[dx] = (uint8_t)s0;
        cnt[dx] = (uint8_t)n;
        for (int k = n; k < MAX_TAPS; ++k) alpha[dx][k] = 0.f;
    }
    for (int s = 0; s < ssize; ++s)
        if (first[s] == 255) return false;   // every source index must feed some destination
    return true;
}

static bool build_tabs(int dim, AreaTabs* t) {
    memset(t, 0, sizeof *t);
    t->dim = dim;
    if (!build_axis(SCREEN_W, dim, t->x_src0, t->x_n, t->x_a, t->x_first, t->x_last)) return false;
    if (!build_axis(SCREEN_H, dim, t->y_src0, t->y_n, t->y_b, t->y_first, t->y_last)) return false;
    for (int dx = 0; dx < dim; ++dx)
        for (int k = 0; k < MAX_TAPS; ++k) {
            volatile float pa = 255.0f * t->x_a[dx][k];   // fl(fl(255) * alpha), single rounding in fp32
            t->x_pa[dx][k] = pa;
        }
    t->text_rows = t->y_last[ARENA_TOP - 1] + 1;
    return true;
}

template <typename T>
static cudaError_t dev_alloc(crl_pong* h, T** p, size_t count) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 16);
    if (e != cudaSuccess) return e;
    h->allocs.push_back(q);
    *p = (T*)q;
    return cudaMemset(q, 0, count * sizeof(T) + 16);
}

extern "C" {

int crl_abi_version(void) { return CRL_ABI_VERSION; }
const char* crl_last_error(void) { return g_err; }
uint64_t crl_launch_count(void) { return g_launches.load(); }

int crl_pong_destroy(crl_pong* h) {
    if (!h) return CRL_OK;
    CrlDeviceGuard guard(h->cfg.device);
    for (void* p : h->allocs) cudaFree(p);
    if (h->shown_dev) cudaFree(h->shown_dev);
    if (h->ev_state) cudaEventDestroy(h->ev_state);
    if (h->ev_copied) cudaEventDestroy(h->ev_copied);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    delete h;
    return CRL_OK;
}

int crl_pong_create(const crl_pong_config* cfg, crl_pong** out) {
    if (!cfg || !out) return fail(CRL_E_INVALID, "null argument");
    *out = nullptr;
    if (cfg->num_envs <= 0) return fail(CRL_E_INVALID, "num_envs must be positive");
    if (cfg->n_agents != 1 && cfg->n_agents != 2) return fail(CRL_E_INVALID, "n_agents must be 1 or 2");
    if (cfg->resized_dim < 8 || cfg->resized_dim > MAX_DIM || cfg->resized_dim % 2)
        return fail(CRL_E_INVALID, "resized_dim must be even and in [8, %d]", MAX_DIM);
    if (cfg->frame_stack < 0 || cfg->frame_stack > MAX_STACK)
        return fail(CRL_E_INVALID, "frame_stack must be in [0, %d]", MAX_STACK);
    if (cfg->stack_mode != 0 && cfg->stack_mode != 1) return fail(CRL_E_INVALID, "stack_mode must be 0 (stack) or 1 (ring)");
    if (cfg->stack_mode == 1 && cfg->frame_stack < 2) return fail(CRL_E_INVALID, "stack_mode ring needs frame_stack >= 2");
    if (cfg->max_num_rounds < 1 || cfg->max_num_rounds > ATLAS_SCORES - 1)
        return fail(CRL_E_INVALID, "max_num_rounds must be in [1, %d] (scoreboard atlas range)", ATLAS_SCORES - 1);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(CRL_E_CUDA, "no CUDA device available (%s); this library has no CPU path",
                    cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(CRL_E_INVALID, "device %d out of range", cfg->device);
    CrlDeviceGuard guard(cfg->device);
    CUDA_TRY(guard.err);
    AreaTabs tabs;
    if (!build_tabs(cfg->resized_dim, &tabs))
        return fail(CRL_E_INVALID, "resized_dim %d needs more than %d taps per pixel", cfg->resized_dim, MAX_TAPS);

    crl_pong* h = new crl_pong();
    h->cfg = *cfg;
    PongDev& d = h->dev;
    memset(&d, 0, sizeof d);
    const size_t n = (size_t)cfg->num_envs;
    d.n = cfg->num_envs;
    d.n_agents = cfg->n_agents;
    d.dim = cfg->resized_dim;
    d.c = cfg->frame_stack > 0 ? cfg->frame_stack : 1;
    d.max_rounds = cfg->max_num_rounds;
    d.ring = cfg->stack_mode == 1 ? 1 : 0;
    d.zero_on_done = cfg->zero_on_done ? 1 : 0;
    d.first_env = cfg->first_env;
    d.seed = cfg->seed;
    const int dd = d.dim * d.dim;
    d.text_stride = ((tabs.text_rows * d.dim + 15) / 16) * 16;
    if (d.text_stride > ((dd + 15) / 16) * 16) d.text_stride = ((dd + 15) / 16) * 16;
    d.text_w0 = 0; d.text_w1 = d.text_stride / 4;
#define ALLOC(ptr, count)                                                        \
    do {                                                                         \
        cudaError_t _e = dev_alloc(h, &(ptr), (count));                          \
        if (_e != cudaSuccess) {                                                 \
            crl_pong_destroy(h);                                                 \
            return fail(CRL_E_CUDA, "cudaMalloc: %s", cudaGetErrorString(_e));   \
        }                                                                        \
    } while (0)
    ALLOC(d.ball, n); ALLOC(d.vx, n); ALLOC(d.vy, n); ALLOC(d.bats, n); ALLOC(d.score, n);
    ALLOC(d.num_steps, n); ALLOC(d.clip_steps, n); ALLOC(d.serve_count, n); ALLOC(d.last_done, n);
    ALLOC(d.skipbuf, 2 * n); ALLOC(d.hist, d.c * n); ALLOC(d.term_hist, d.c * n);
    ALLOC(d.serve_overrun, 1);
    ALLOC(d.stats, 8);
    ALLOC(d.work_counter, 2);
    ALLOC(h->tabs_dev, 1);
    ALLOC(h->atlas_dev, (size_t)CRL_PONG_ATLAS_BYTES);
    ALLOC(h->text_tab_dev, (size_t)ATLAS_SCORES * ATLAS_SCORES * 3 * 2 * d.text_stride);
    ALLOC(h->tmpl_dev, (size_t)((dd + 15) / 16) * 16);
    ALLOC(h->actions_stage, 2 * n); ALLOC(h->rew_stage, 2 * n); ALLOC(h->done_stage, n);
    ALLOC(h->steps_stage, n); ALLOC(h->real_stage, 2 * n);
    h->tabs_host = tabs;
    const size_t ftb = pong_fast_tabs_bytes(d.dim);
    if (ftb) {
        std::vector<uint8_t> img(ftb);
        if (pong_fast_tabs_fill(tabs, d.text_stride, img.data())) {
            ALLOC(h->fast_tabs_dev, ftb);
            cudaError_t _e = cudaMemcpy(h->fast_tabs_dev, img.data(), ftb, cudaMemcpyHostToDevice);
            if (_e == cudaSuccess) _e = launch_pong_build_bat_lut(d.dim, h->fast_tabs_dev, 0);
            if (_e != cudaSuccess) {
                crl_pong_destroy(h);
                return fail(CRL_E_CUDA, "fast tabs upload: %s", cudaGetErrorString(_e));
            }
            g_launches += 1;
            d.fast_tabs = h->fast_tabs_dev;
            d.quad_ok = (pong_quad_ok(tabs) && getenv("CRL_PONG_NO_QUAD") == nullptr) ? 1 : 0;
            h->full_obs = getenv("CRL_PONG_FULL_OBS") != nullptr;   // A/B switch: no incremental stacks
        }
    }
    d.tabs = h->tabs_dev;
    d.atlas = h->atlas_dev;
    d.text_tab = h->text_tab_dev;
    d.tmpl = h->tmpl_dev;
#undef ALLOC
    e = cudaMemcpy(h->tabs_dev, &tabs, sizeof tabs, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = pong_raster_init(d.raster_grid);
    if (e == cudaSuccess) e = launch_pong_construct(d, 0);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        crl_pong_destroy(h);
        return fail(CRL_E_CUDA, "construct: %s", cudaGetErrorString(e));
    }
    g_launches += 1;
    *out = h;
    return CRL_OK;
}

#define CHECK_HANDLE(h)                                        \
    do {                                                       \
        if (!(h)) return fail(CRL_E_INVALID, "null handle");   \
    } while (0);                                               \
    CrlDeviceGuard crl_guard_((h)->cfg.device);                \
    CUDA_TRY(crl_guard_.err)

int crl_pong_load_atlas(crl_pong* h, const uint8_t* strips_host, size_t bytes, void* stream) {
    CHECK_HANDLE(h);
    if (!strips_host || bytes != (size_t)CRL_PONG_ATLAS_BYTES)
        return fail(CRL_E_INVALID, "atlas must be %d bytes ([22][22][34][160][3] uint8)", CRL_PONG_ATLAS_BYTES);
    cudaStream_t s = (cudaStream_t)stream;
    // The hot kernel treats source rows above the arena that share a destination row with arena
    // rows as pure white (true for any scoreboard that stays clear of the arena edge); otherwise
    // every frame takes the exact one-thread-per-pixel rasteriser.
    {
        const AreaTabs& t = h->tabs_host;
        const int first = t.y_src0[t.text_rows - 1];
        bool white = true;
        for (int pair = 0; pair < ATLAS_SCORES * ATLAS_SCORES && white; ++pair)
            for (int r = first; r < ATLAS_ROWS && white; ++r) {
                const uint8_t* row = strips_host + ((size_t)pair * ATLAS_ROWS + r) * SCREEN_W * 3;
                for (int i = 0; i < SCREEN_W * 3; ++i)
                    if (row[i] != 255) { white = false; break; }
            }
        h->dev.fast_ok = white ? 1 : 0;
    }
    CUDA_TRY(cudaMemcpyAsync(h->atlas_dev, strips_host, bytes, cudaMemcpyHostToDevice, s));
    LAUNCH(launch_pong_build_tables(h->dev, h->text_tab_dev, h->tmpl_dev, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    {   // The words of a scoreboard entry that differ between entries (any score pair, kind, agent) or from the template: the
        // score digits cover a few of the rows above the arena only, and the rest of an entry never needs copying.
        const int tw = h->dev.text_stride / 4;
        const size_t n_ent = (size_t)ATLAS_SCORES * ATLAS_SCORES * 3 * 2;
        std::vector<uint32_t> tt(n_ent * tw), tm(tw);
        CUDA_TRY(cudaMemcpy(tt.data(), h->text_tab_dev, tt.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(tm.data(), h->tmpl_dev, tm.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        int w0 = tw, w1 = 0;
        for (int w = 0; w < tw; ++w) {
            bool differs = tm[w] != tt[w];
            for (size_t e = 1; e < n_ent && !differs; ++e) differs = tt[e * tw + w] != tt[w];
            if (differs) { if (w < w0) w0 = w; w1 = w + 1; }
        }
        if (w1 <= w0) w0 = w1 = 0;
        if (getenv("CRL_PONG_TEXT_FULL") != nullptr) { w0 = 0; w1 = tw; }   // A/B switch: copy whole entries
        h->dev.text_w0 = w0; h->dev.text_w1 = w1;
    }
    h->atlas_loaded = true;
    for (auto& st : h->sets) st.valid = false;   // every frame may look different now
    return CRL_OK;
}

int crl_pong_inject_serves(crl_pong* h, const double* serves_host, int32_t k, void* stream) {
    CHECK_HANDLE(h);
    if (!serves_host || k < 3) return fail(CRL_E_INVALID, "serve table needs k >= 3 entries per env");
    cudaStream_t s = (cudaStream_t)stream;
    double* buf = nullptr;
    CUDA_TRY(dev_alloc(h, &buf, (size_t)h->dev.n * k * 2));
    CUDA_TRY(cudaMemcpyAsync(buf, serves_host, (size_t)h->dev.n * k * 2 * sizeof(double), cudaMemcpyHostToDevice, s));
    h->serves_dev = buf;
    h->dev.serves = buf;
    h->dev.serves_k = k;
    LAUNCH(launch_pong_construct(h->dev, s));   // constructors re-run: serves 0 and 1 from the table
    CUDA_TRY(cudaStreamSynchronize(s));
    h->was_reset = false;
    return CRL_OK;
}

int crl_pong_seed(crl_pong* h, uint64_t seed) {
    CHECK_HANDLE(h);
    h->dev.seed = seed;
    return CRL_OK;
}

static int need_ready(crl_pong* h, bool need_reset) {
    if (!h->atlas_loaded) return fail(CRL_E_STATE, "crl_pong_load_atlas must be called before reset/step");
    if (need_reset && !h->was_reset) return fail(CRL_E_STATE, "reset must be called before step");
    return CRL_OK;
}

int crl_pong_render_obs(crl_pong* h, uint8_t* obs0_dev, uint8_t* obs1_dev, void* stream) {
    CHECK_HANDLE(h);
    if (int r = need_ready(h, true)) return r;
    if (!obs0_dev || (h->dev.n_agents == 2 && !obs1_dev)) return fail(CRL_E_INVALID, "null observation buffer");
    if (h->dev.n_agents == 1) obs1_dev = obs0_dev;
    cudaStream_t s = (cudaStream_t)stream;
    crl_pong::ObsSet* set = nullptr;
    for (auto& st : h->sets)
        if (st.obs[0] == obs0_dev && (h->dev.n_agents == 1 || st.obs[1] == obs1_dev)) set = &st;
    const bool incremental = !h->full_obs && pong_raster_incremental_ok(h->dev, obs0_dev, obs1_dev);
    if (set && set->valid && incremental) {
        LAUNCH(launch_pong_raster(h->dev, h->dev.hist, obs0_dev, obs1_dev, set->shown, s));
        return CRL_OK;
    }
    LAUNCH(launch_pong_raster(h->dev, h->dev.hist, obs0_dev, obs1_dev, nullptr, s));
    if (!set) {
        obs_written(h, obs0_dev, obs_bytes(h));
        obs_written(h, obs1_dev, obs_bytes(h));
    } else if (incremental) {   // the set now holds hist: later renders into it can be incremental
        const size_t per_agent = (size_t)h->dev.c * h->dev.n;
        for (int k = 0; k < h->dev.n_agents; ++k)
            CUDA_TRY(cudaMemcpyAsync(set->shown + k * per_agent, h->dev.hist, per_agent * sizeof(FrameSpec),
                                     cudaMemcpyDeviceToDevice, s));
        set->valid = true;
    } else {
        set->valid = false;
    }
    return CRL_OK;
}

int crl_pong_set_obs_buffers(crl_pong* h, uint8_t* const* obs0_devs_host, uint8_t* const* obs1_devs_host, int32_t count,
                             void* stream) {
    CHECK_HANDLE(h);
    const int na = h->dev.n_agents;
    if (count != 0) {
        if (h->dev.ring) return fail(CRL_E_STATE, "stack_mode ring keeps its own frames: there are no buffer sets to register");
        if (count < 0 || count > CRL_PONG_MAX_OBS_SETS || !obs0_devs_host || (na == 2 && !obs1_devs_host))
            return fail(CRL_E_INVALID, "need 1 .. %d buffer sets (and obs1 buffers for cPongDouble), got %d",
                        CRL_PONG_MAX_OBS_SETS, count);
        std::vector<uint8_t*> all;
        for (int i = 0; i < count; ++i)
            for (int k = 0; k < na; ++k) {
                uint8_t* b = k ? obs1_devs_host[i] : obs0_devs_host[i];
                if (!b) return fail(CRL_E_INVALID, "null buffer in set %d", i);
                for (uint8_t* o : all)
                    if (o == b) return fail(CRL_E_INVALID, "a buffer appears twice in the sets");
                all.push_back(b);
            }
    }
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));   // no render in flight reads the old specs
    h->sets.clear();
    if (h->shown_dev) {
        CUDA_TRY(cudaFree(h->shown_dev));
        h->shown_dev = nullptr;
    }
    if (count == 0) return CRL_OK;
    const size_t per_set = (size_t)na * h->dev.c * h->dev.n;
    CUDA_TRY(cudaMalloc(&h->shown_dev, (size_t)count * per_set * sizeof(FrameSpec)));
    for (int i = 0; i < count; ++i)
        h->sets.push_back({{obs0_devs_host[i], na == 2 ? obs1_devs_host[i] : obs0_devs_host[i]}, h->shown_dev + i * per_set, false});
    return CRL_OK;
}

int crl_pong_forget_obs(crl_pong* h) {
    if (!h) return fail(CRL_E_INVALID, "null handle");
    for (auto& st : h->sets) st.valid = false;
    return CRL_OK;
}

int crl_pong_render_obs_generic(crl_pong* h, uint8_t* obs0_dev, uint8_t* obs1_dev, void* stream) {
    CHECK_HANDLE(h);
    if (int r = need_ready(h, true)) return r;
    if (!obs0_dev || (h->dev.n_agents == 2 && !obs1_dev)) return fail(CRL_E_INVALID, "null observation buffer");
    LAUNCH(launch_pong_raster_generic(h->dev, h->dev.hist, nullptr, h->dev.ring, obs0_dev, obs1_dev, (cudaStream_t)stream));
    obs_written(h, obs0_dev, obs_bytes(h));
    obs_written(h, obs1_dev, obs_bytes(h));
    return CRL_OK;
}

int crl_pong_render_obs_f32(crl_pong* h, int32_t terminal, const uint8_t* only_done_dev, float* obs0_dev, float* obs1_dev, void* stream) {
    CHECK_HANDLE(h);
    if (int r = need_ready(h, true)) return r;
    if (h->dev.ring) return fail(CRL_E_STATE, "float32 observations are plain stacks: create the handle with stack_mode 0");
    if (!obs0_dev || (h->dev.n_agents == 2 && !obs1_dev)) return fail(CRL_E_INVALID, "null observation buffer");
    LAUNCH(launch_pong_raster_f32(h->dev, terminal ? h->dev.term_hist : h->dev.hist, only_done_dev, obs0_dev, obs1_dev, (cudaStream_t)stream));
    obs_written(h, obs0_dev, 4 * obs_bytes(h));
    obs_written(h, obs1_dev, 4 * obs_bytes(h));
    return CRL_OK;
}

int crl_pong_reset_state(crl_pong* h, void* stream) {
    CHECK_HANDLE(h);
    if (int r = need_ready(h, false)) return r;
    LAUNCH(launch_pong_reset(h->dev, (cudaStream_t)stream));
    h->was_reset = true;
    h->dev.ring_phase = 0;
    h->dev.fill_all = 1;
    return CRL_OK;
}

int crl_pong_reset(crl_pong* h, uint8_t* obs0_dev, uint8_t* obs1_dev, void* stream) {
    CHECK_HANDLE(h);
    if (int r = need_ready(h, false)) return r;
    LAUNCH(launch_pong_reset(h->dev, (cudaStream_t)stream));
    h->was_reset = true;
    h->dev.ring_phase = 0;
    h->dev.fill_all = 1;      // until the next step: every ring is (re)written completely
    return crl_pong_render_obs(h, obs0_dev, obs1_dev, stream);
}

int crl_pong_step_state(crl_pong* h, const int32_t* actions_dev, float* rew_dev, uint8_t* done_dev,
                        int32_t* num_steps_dev, float* real_reward_dev, void* stream) {
    CHECK_HANDLE(h);
    if (int r = need_ready(h, true)) return r;
    if (!actions_dev || !rew_dev || !done_dev || !num_steps_dev || !real_reward_dev)
        return fail(CRL_E_INVALID, "null step buffer");
    h->dev.fill_all = 0;
    if (h->dev.ring) h->dev.ring_phase = (h->dev.ring_phase + 1) % h->dev.c;
    LAUNCH(launch_pong_step(h->dev, actions_dev, rew_dev, done_dev, num_steps_dev, real_reward_dev,
                            (cudaStream_t)stream));
    return CRL_OK;
}

int crl_pong_step(crl_pong* h, const int32_t* actions_dev, uint8_t* obs0_dev, uint8_t* obs1_dev, float* rew_dev,
                  uint8_t* done_dev, int32_t* num_steps_dev, float* real_reward_dev, void* stream) {
    if (int r = crl_pong_step_state(h, actions_dev, rew_dev, done_dev, num_steps_dev, real_reward_dev, stream))
        return r;
    return crl_pong_render_obs(h, obs0_dev, obs1_dev, stream);
}

int crl_pong_terminal_obs(crl_pong* h, const uint8_t* done_dev, uint8_t* term0_dev, uint8_t* term1_dev, void* stream) {
    CHECK_HANDLE(h);
    if (int r = need_ready(h, true)) return r;
    if (!done_dev || !term0_dev || (h->dev.n_agents == 2 && !term1_dev)) return fail(CRL_E_INVALID, "null buffer");
    LAUNCH(launch_pong_raster_generic(h->dev, h->dev.term_hist, done_dev, 0, term0_dev, term1_dev, (cudaStream_t)stream));
    obs_written(h, term0_dev, obs_bytes(h));
    obs_written(h, term1_dev, obs_bytes(h));
    return CRL_OK;
}

int crl_pong_step_host(crl_pong* h, const int32_t* actions_host, uint8_t* obs0_dev, uint8_t* obs1_dev,
                       uint8_t* obs0_host, uint8_t* obs1_host, float* rew_host, uint8_t* done_host,
                       int32_t* num_steps_host, float* real_reward_host, void* stream) {
    CHECK_HANDLE(h);
    if (!actions_host || !rew_host || !done_host) return fail(CRL_E_INVALID, "null host buffer");
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)h->dev.n;
    const size_t aw = h->dev.n_agents == 2 ? 2 : 1;
    if (!h->copy_stream) {
        CUDA_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&h->ev_state, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&h->ev_copied, cudaEventDisableTiming));
    }
    CUDA_TRY(cudaMemcpyAsync(h->actions_stage, actions_host, n * aw * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    if (int r = crl_pong_step_state(h, h->actions_stage, h->rew_stage, h->done_stage, h->steps_stage, h->real_stage, stream))
        return r;
    // rewards / dones / counters are final once the game-core kernel has run: copy them out on the side stream,
    // behind the rasteriser (which is the whole cost of the step)
    CUDA_TRY(cudaEventRecord(h->ev_state, s));
    CUDA_TRY(cudaStreamWaitEvent(h->copy_stream, h->ev_state, 0));
    cudaStream_t cs = h->copy_stream;
    CUDA_TRY(cudaMemcpyAsync(rew_host, h->rew_stage, n * 2 * sizeof(float), cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(cudaMemcpyAsync(done_host, h->done_stage, n, cudaMemcpyDeviceToHost, cs));
    if (num_steps_host)
        CUDA_TRY(cudaMemcpyAsync(num_steps_host, h->steps_stage, n * sizeof(int32_t), cudaMemcpyDeviceToHost, cs));
    if (real_reward_host)
        CUDA_TRY(cudaMemcpyAsync(real_reward_host, h->real_stage, n * 2 * sizeof(float), cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(cudaEventRecord(h->ev_copied, cs));
    if (int r = crl_pong_render_obs(h, obs0_dev, obs1_dev, stream)) return r;
    CUDA_TRY(cudaStreamWaitEvent(s, h->ev_copied, 0));
    const size_t ob = n * (h->dev.ring ? 2 * h->dev.c : h->dev.c) * h->dev.dim * h->dev.dim;
    if (obs0_host) CUDA_TRY(cudaMemcpyAsync(obs0_host, obs0_dev, ob, cudaMemcpyDeviceToHost, s));
    if (obs1_host && h->dev.n_agents == 2) CUDA_TRY(cudaMemcpyAsync(obs1_host, obs1_dev, ob, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return CRL_OK;
}

int crl_pong_ring_phase(crl_pong* h) {
    if (!h) return fail(CRL_E_INVALID, "null handle");
    if (!h->dev.ring) return fail(CRL_E_STATE, "the handle was not created with stack_mode ring");
    return h->dev.ring_phase;
}

int crl_pong_get_state(crl_pong* h, double* state_dev, void* stream) {
    CHECK_HANDLE(h);
    if (!state_dev) return fail(CRL_E_INVALID, "null buffer");
    LAUNCH(launch_pong_get_state(h->dev, state_dev, (cudaStream_t)stream));
    return CRL_OK;
}

int crl_pong_set_state(crl_pong* h, const double* state_dev, void* stream) {
    CHECK_HANDLE(h);
    if (!state_dev) return fail(CRL_E_INVALID, "null buffer");
    LAUNCH(launch_pong_set_state(h->dev, state_dev, (cudaStream_t)stream));
    return CRL_OK;
}

int crl_pong_render_raw(crl_pong* h, int32_t env, uint8_t* rgb0_dev, uint8_t* rgb1_dev, void* stream) {
    CHECK_HANDLE(h);
    if (int r = need_ready(h, false)) return r;
    if (env < 0 || env >= h->dev.n || !rgb0_dev) return fail(CRL_E_INVALID, "bad env index or null buffer");
    LAUNCH(launch_pong_raw_frame(h->dev, env, rgb0_dev, rgb1_dev, (cudaStream_t)stream));
    return CRL_OK;
}

int crl_pong_random_actions(int32_t* actions_dev, int32_t n_values, uint64_t seed, uint64_t step, void* stream) {
    if (!actions_dev || n_values <= 0) return fail(CRL_E_INVALID, "bad arguments");
    LAUNCH(launch_pong_random_actions(actions_dev, n_values, seed, step, (cudaStream_t)stream));
    return CRL_OK;
}

int crl_pong_get_stats(crl_pong* h, uint64_t* stats_host, void* stream) {
    CHECK_HANDLE(h);
    if (!stats_host) return fail(CRL_E_INVALID, "null buffer");
    unsigned long long raw[8];
    CUDA_TRY(cudaMemcpyAsync(raw, h->dev.stats, sizeof raw, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    for (int i = 0; i < 8; ++i) stats_host[i] = raw[i];
    return CRL_OK;
}

int crl_pong_check(crl_pong* h, void* stream) {
    CHECK_HANDLE(h);
    int32_t flag = 0;
    CUDA_TRY(cudaMemcpyAsync(&flag, h->dev.serve_overrun, sizeof flag, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    if (flag != 0) {   // reported once: the flag is cleared so that later checks see later steps only
        CUDA_TRY(cudaMemsetAsync(h->dev.serve_overrun, 0, sizeof flag, (cudaStream_t)stream));
        CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    }
    if (flag & 2) return fail(CRL_E_INVALID, "an action outside {0, 1, 2} (cPongDouble: or 999) was passed to step; it was played as 1 (stay)");
    if (flag & 1) return fail(CRL_E_SERVES, "injected serve table exhausted");
    return CRL_OK;
}

// ---- observation buffers in compressible memory (crl_obs_alloc / crl_obs_free) ----
// The driver calls come through cudaGetDriverEntryPointByVersion, so the library has no link dependency on libcuda.
struct ObsDriver {
    decltype(&::cuMemCreate) create = nullptr;
    decltype(&::cuMemRelease) release = nullptr;
    decltype(&::cuMemGetAllocationGranularity) granularity = nullptr;
    decltype(&::cuMemGetAllocationPropertiesFromHandle) properties = nullptr;
    decltype(&::cuMemAddressReserve) reserve = nullptr;
    decltype(&::cuMemAddressFree) address_free = nullptr;
    decltype(&::cuMemMap) map = nullptr;
    decltype(&::cuMemUnmap) unmap = nullptr;
    decltype(&::cuMemSetAccess) set_access = nullptr;
    bool ok = false;
};

static const ObsDriver& obs_driver() {
    static const ObsDriver d = [] {
        ObsDriver r;
        auto get = [](const char* name, auto& fn) {
            void* p = nullptr;
            cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
            if (cudaGetDriverEntryPointByVersion(name, &p, 12000, cudaEnableDefault, &q) != cudaSuccess ||
                q != cudaDriverEntryPointSuccess)
                return false;
            fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(p);
            return p != nullptr;
        };
        r.ok = get("cuMemCreate", r.create) && get("cuMemRelease", r.release) &&
               get("cuMemGetAllocationGranularity", r.granularity) &&
               get("cuMemGetAllocationPropertiesFromHandle", r.properties) && get("cuMemAddressReserve", r.reserve) &&
               get("cuMemAddressFree", r.address_free) && get("cuMemMap", r.map) && get("cuMemUnmap", r.unmap) &&
               get("cuMemSetAccess", r.set_access);
        return r;
    }();
    return d;
}

struct ObsAlloc {
    int device;
    size_t bytes;   // mapped size (VMM) or 0 (cudaMalloc)
};
static std::mutex g_obs_mu;
static std::unordered_map<void*, ObsAlloc> g_obs;

// A compressible VMM mapping of `bytes` on `device`, or nullptr when the driver does not provide one.
static void* obs_map_compressible(int device, size_t bytes, size_t* mapped, int32_t* compressed) {
    const ObsDriver& d = obs_driver();
    if (!d.ok) return nullptr;
    CUmemAllocationProp prop;
    memset(&prop, 0, sizeof prop);
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t g = 0;
    if (d.granularity(&g, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || g == 0) return nullptr;
    const size_t sz = (bytes + g - 1) / g * g;
    CUmemGenericAllocationHandle h;
    if (d.create(&h, sz, &prop, 0) != CUDA_SUCCESS) return nullptr;
    CUmemAllocationProp got;
    memset(&got, 0, sizeof got);
    CUdeviceptr va = 0;
    CUmemAccessDesc acc;
    memset(&acc, 0, sizeof acc);
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (d.properties(&got, h) != CUDA_SUCCESS || d.reserve(&va, sz, g, 0, 0) != CUDA_SUCCESS) {
        d.release(h);
        return nullptr;
    }
    if (d.map(va, sz, 0, h, 0) != CUDA_SUCCESS) {
        d.address_free(va, sz);
        d.release(h);
        return nullptr;
    }
    d.release(h);   // the mapping keeps the memory until it is unmapped
    if (d.set_access(va, sz, &acc, 1) != CUDA_SUCCESS) {
        d.unmap(va, sz);
        d.address_free(va, sz);
        return nullptr;
    }
    *mapped = sz;
    // the driver may grant an ordinary allocation (for instance when the device's compression resources are used up)
    *compressed = got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC ? 1 : 0;
    return reinterpret_cast<void*>(va);
}

int crl_obs_alloc(int32_t device, size_t bytes, void** ptr, int32_t* compressed) {
    if (!ptr || !compressed || bytes == 0) return fail(CRL_E_INVALID, "crl_obs_alloc: null output pointer or zero bytes");
    *ptr = nullptr;
    *compressed = 0;
    CrlDeviceGuard guard(device);
    CUDA_TRY(guard.err);
    int supported = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&supported, (cudaDeviceAttr)CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, device));
    void* p = nullptr;
    size_t mapped = 0;
    if (supported) p = obs_map_compressible(device, bytes, &mapped, compressed);
    if (p == nullptr) {
        *compressed = 0;
        CUDA_TRY(cudaMalloc(&p, bytes));
    }
    {
        std::lock_guard<std::mutex> lk(g_obs_mu);
        g_obs[p] = ObsAlloc{device, mapped};
    }
    *ptr = p;
    return CRL_OK;
}

int crl_obs_free(void* ptr) {
    if (!ptr) return CRL_OK;
    ObsAlloc a;
    {
        std::lock_guard<std::mutex> lk(g_obs_mu);
        auto it = g_obs.find(ptr);
        if (it == g_obs.end()) return fail(CRL_E_INVALID, "crl_obs_free: %p was not returned by crl_obs_alloc", ptr);
        a = it->second;
        g_obs.erase(it);
    }
    CrlDeviceGuard guard(a.device);
    CUDA_TRY(guard.err);
    if (a.bytes == 0) {
        CUDA_TRY(cudaFree(ptr));
        return CRL_OK;
    }
    CUDA_TRY(cudaDeviceSynchronize());   // a kernel may still be writing the buffer
    const ObsDriver& d = obs_driver();
    CUresult r = d.unmap(reinterpret_cast<CUdeviceptr>(ptr), a.bytes);
    if (r == CUDA_SUCCESS) r = d.address_free(reinterpret_cast<CUdeviceptr>(ptr), a.bytes);
    if (r != CUDA_SUCCESS) return fail(CRL_E_CUDA, "crl_obs_free: cuMemUnmap / cuMemAddressFree failed (CUresult %d)", (int)r);
    return CRL_OK;
}

}  // extern "C"
