// crl_torch.cpp -- the PyTorch C++ extension of the host layer: a thin binding of the C ABI (include/crl_b200.h) that
// takes and returns torch tensors.  No kernels here and no logic beyond argument checking: every function validates
// its tensors (device, dtype, contiguity, element count), picks up torch's current CUDA stream for the handle's
// device and makes ONE call into libcrl_b200.so, so a vec-env step costs one Python -> C++ crossing instead of a
// dozen ctypes pointer conversions.  Replaces nothing in the reference (which has no native layer): it is the
// "Python host layer = PyTorch C++/CUDA extension over a C-ABI" of BASELINE.json's north_star.
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/extension.h>

#include <algorithm>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/crl_b200.h"

namespace {

struct CrlError : public std::runtime_error {
    using std::runtime_error::runtime_error;
};

void check_rc(int rc) {
    if (rc != CRL_OK) throw CrlError("crl error " + std::to_string(rc) + ": " + crl_last_error());
}

void* stream_of(int device) { return (void*)c10::cuda::getCurrentCUDAStream((c10::DeviceIndex)device).stream(); }

// a device tensor the kernels can write / read directly
template <typename T>
T* dev_ptr(const at::Tensor& t, at::ScalarType dtype, int device, int64_t numel, const char* what) {
    TORCH_CHECK(t.is_cuda() && t.get_device() == device, what, ": expected a CUDA tensor on device ", device);
    TORCH_CHECK(t.scalar_type() == dtype, what, ": expected dtype ", dtype, ", got ", t.scalar_type());
    TORCH_CHECK(t.is_contiguous(), what, ": expected a contiguous tensor");
    TORCH_CHECK(numel < 0 || t.numel() == numel, what, ": expected ", numel, " elements, got ", t.numel());
    return reinterpret_cast<T*>(t.data_ptr());
}
template <typename T>
T* opt_dev_ptr(const c10::optional<at::Tensor>& t, at::ScalarType dtype, int device, int64_t numel, const char* what) {
    return t.has_value() ? dev_ptr<T>(*t, dtype, device, numel, what) : nullptr;
}
template <typename T>
const T* host_ptr(const at::Tensor& t, at::ScalarType dtype, const char* what) {
    TORCH_CHECK(!t.is_cuda() && t.scalar_type() == dtype && t.is_contiguous(), what, ": expected a contiguous CPU tensor of dtype ", dtype);
    return reinterpret_cast<const T*>(t.data_ptr());
}

// ------------------------------------------------------------------------------------------------ Pong
struct Pong {
    crl_pong* h = nullptr;
    crl_pong_config cfg{};
    int64_t obs_numel = 0;

    Pong(int64_t num_envs, int64_t n_agents, int64_t resized_dim, int64_t frame_stack, int64_t max_num_rounds, int64_t device,
         int64_t stack_mode, bool zero_on_done, uint64_t seed, int64_t first_env) {
        cfg.num_envs = (int32_t)num_envs; cfg.n_agents = (int32_t)n_agents; cfg.resized_dim = (int32_t)resized_dim;
        cfg.frame_stack = (int32_t)frame_stack; cfg.max_num_rounds = (int32_t)max_num_rounds; cfg.device = (int32_t)device;
        cfg.stack_mode = (int32_t)stack_mode; cfg.zero_on_done = zero_on_done ? 1 : 0; cfg.seed = seed; cfg.first_env = first_env;
        check_rc(crl_pong_create(&cfg, &h));
        const int64_t c = frame_stack > 0 ? frame_stack : 1;
        obs_numel = num_envs * (stack_mode == 1 ? 2 * c : c) * resized_dim * resized_dim;
    }
    ~Pong() { close(); }
    void close() {
        if (h) { crl_pong_destroy(h); h = nullptr; }
    }
    crl_pong* handle() const {
        TORCH_CHECK(h != nullptr, "the environment is closed");
        return h;
    }
    int dev() const { return cfg.device; }
    int64_t n() const { return cfg.num_envs; }
    uint8_t* obs1_ptr(const c10::optional<at::Tensor>& o1, const char* what) const {
        if (cfg.n_agents == 2) TORCH_CHECK(o1.has_value(), what, ": cPongDouble needs both agents' buffers");
        return opt_dev_ptr<uint8_t>(o1, at::kByte, dev(), obs_numel, what);
    }

    void load_atlas(const at::Tensor& strips) {
        check_rc(crl_pong_load_atlas(handle(), host_ptr<uint8_t>(strips, at::kByte, "atlas"), (size_t)strips.numel(), stream_of(dev())));
    }
    void inject_serves(const at::Tensor& serves) {
        TORCH_CHECK(serves.dim() == 3 && serves.size(0) == n() && serves.size(2) == 2, "serves must have shape (num_envs, K, 2)");
        check_rc(crl_pong_inject_serves(handle(), host_ptr<double>(serves, at::kDouble, "serves"), (int32_t)serves.size(1), stream_of(dev())));
    }
    void seed(uint64_t s) { check_rc(crl_pong_seed(handle(), s)); }
    void reset(const at::Tensor& obs0, const c10::optional<at::Tensor>& obs1) {
        check_rc(crl_pong_reset(handle(), dev_ptr<uint8_t>(obs0, at::kByte, dev(), obs_numel, "obs0"), obs1_ptr(obs1, "obs1"), stream_of(dev())));
    }
    // VecEnv.step: actions int32 (N, 2) / (N,) on the device; done is a torch.bool tensor (the kernel writes 0 / 1 bytes)
    void step(const at::Tensor& actions, const at::Tensor& obs0, const c10::optional<at::Tensor>& obs1, const at::Tensor& rew,
              const at::Tensor& done, const at::Tensor& num_steps, const at::Tensor& real_reward) {
        check_rc(crl_pong_step(handle(), dev_ptr<int32_t>(actions, at::kInt, dev(), n() * cfg.n_agents, "actions"),
                               dev_ptr<uint8_t>(obs0, at::kByte, dev(), obs_numel, "obs0"), obs1_ptr(obs1, "obs1"),
                               dev_ptr<float>(rew, at::kFloat, dev(), 2 * n(), "rew"), dev_ptr<uint8_t>(done, at::kBool, dev(), n(), "done"),
                               dev_ptr<int32_t>(num_steps, at::kInt, dev(), n(), "num_steps"),
                               dev_ptr<float>(real_reward, at::kFloat, dev(), 2 * n(), "real_reward"), stream_of(dev())));
    }
    // float32 observation mode (stock gym): game core, then the float rasteriser
    void reset_f32(const at::Tensor& obs0, const c10::optional<at::Tensor>& obs1) {
        check_rc(crl_pong_reset_state(handle(), stream_of(dev())));
        render_f32(false, c10::nullopt, obs0, obs1);
    }
    void step_f32(const at::Tensor& actions, const at::Tensor& obs0, const c10::optional<at::Tensor>& obs1, const at::Tensor& rew,
                  const at::Tensor& done, const at::Tensor& num_steps, const at::Tensor& real_reward) {
        check_rc(crl_pong_step_state(handle(), dev_ptr<int32_t>(actions, at::kInt, dev(), n() * cfg.n_agents, "actions"),
                                     dev_ptr<float>(rew, at::kFloat, dev(), 2 * n(), "rew"), dev_ptr<uint8_t>(done, at::kBool, dev(), n(), "done"),
                                     dev_ptr<int32_t>(num_steps, at::kInt, dev(), n(), "num_steps"),
                                     dev_ptr<float>(real_reward, at::kFloat, dev(), 2 * n(), "real_reward"), stream_of(dev())));
        render_f32(false, c10::nullopt, obs0, obs1);
    }
    void render_f32(bool terminal, const c10::optional<at::Tensor>& only_done, const at::Tensor& obs0, const c10::optional<at::Tensor>& obs1) {
        if (cfg.n_agents == 2) TORCH_CHECK(obs1.has_value(), "obs1: cPongDouble needs both agents' buffers");
        check_rc(crl_pong_render_obs_f32(handle(), terminal ? 1 : 0, opt_dev_ptr<uint8_t>(only_done, at::kBool, dev(), n(), "done"),
                                         dev_ptr<float>(obs0, at::kFloat, dev(), obs_numel, "obs0"),
                                         opt_dev_ptr<float>(obs1, at::kFloat, dev(), obs_numel, "obs1"), stream_of(dev())));
    }
    void render_obs_generic(const at::Tensor& obs0, const c10::optional<at::Tensor>& obs1) {
        check_rc(crl_pong_render_obs_generic(handle(), dev_ptr<uint8_t>(obs0, at::kByte, dev(), obs_numel, "obs0"), obs1_ptr(obs1, "obs1"),
                                             stream_of(dev())));
    }
    void terminal_obs(const at::Tensor& done, const at::Tensor& term0, const c10::optional<at::Tensor>& term1) {
        const int64_t c = cfg.frame_stack > 0 ? cfg.frame_stack : 1;
        const int64_t numel = n() * c * cfg.resized_dim * cfg.resized_dim;   // terminal observations are always plain stacks
        if (cfg.n_agents == 2) TORCH_CHECK(term1.has_value(), "term1: cPongDouble needs both agents' buffers");
        check_rc(crl_pong_terminal_obs(handle(), dev_ptr<uint8_t>(done, at::kBool, dev(), n(), "done"),
                                       dev_ptr<uint8_t>(term0, at::kByte, dev(), numel, "term0"),
                                       opt_dev_ptr<uint8_t>(term1, at::kByte, dev(), numel, "term1"), stream_of(dev())));
    }
    int64_t ring_phase() {
        const int k = crl_pong_ring_phase(handle());
        if (k < 0) check_rc(k);
        return k;
    }
    void get_state(const at::Tensor& state) {
        check_rc(crl_pong_get_state(handle(), dev_ptr<double>(state, at::kDouble, dev(), n() * CRL_PONG_STATE_DOUBLES, "state"), stream_of(dev())));
    }
    void set_state(const at::Tensor& state) {
        check_rc(crl_pong_set_state(handle(), dev_ptr<double>(state, at::kDouble, dev(), n() * CRL_PONG_STATE_DOUBLES, "state"), stream_of(dev())));
    }
    void render_raw(int64_t env, const at::Tensor& rgb0, const c10::optional<at::Tensor>& rgb1) {
        check_rc(crl_pong_render_raw(handle(), (int32_t)env, dev_ptr<uint8_t>(rgb0, at::kByte, dev(), 210 * 160 * 3, "rgb0"),
                                     opt_dev_ptr<uint8_t>(rgb1, at::kByte, dev(), 210 * 160 * 3, "rgb1"), stream_of(dev())));
    }
    void check() { check_rc(crl_pong_check(handle(), stream_of(dev()))); }
    // observation buffer sets whose contents the library tracks (crl_pong_set_obs_buffers); empty lists unregister
    void set_obs_buffers(const std::vector<at::Tensor>& obs0, const std::vector<at::Tensor>& obs1) {
        TORCH_CHECK(cfg.n_agents == 1 || obs1.size() == obs0.size(), "cPongDouble needs an obs1 buffer per set");
        std::vector<uint8_t*> p0, p1;
        for (const at::Tensor& t : obs0) p0.push_back(dev_ptr<uint8_t>(t, at::kByte, dev(), obs_numel, "obs0 buffer of a set"));
        for (const at::Tensor& t : obs1) p1.push_back(dev_ptr<uint8_t>(t, at::kByte, dev(), obs_numel, "obs1 buffer of a set"));
        check_rc(crl_pong_set_obs_buffers(handle(), p0.data(), cfg.n_agents == 2 ? p1.data() : nullptr, (int32_t)p0.size(),
                                          stream_of(dev())));
    }
    void forget_obs() { check_rc(crl_pong_forget_obs(handle())); }
    std::vector<uint64_t> stats() {
        std::vector<uint64_t> s(8);
        check_rc(crl_pong_get_stats(handle(), s.data(), stream_of(dev())));
        return s;
    }
    uint64_t raw_handle() const { return (uint64_t)(uintptr_t)h; }
};

// ------------------------------------------------------------------------------------------------ cars
struct Car {
    crl_car* h = nullptr;
    crl_car_config cfg{};
    int64_t obs_numel = 0, term_numel = 0;

    Car(int64_t num_envs, int64_t num_players, int64_t frame_stack, int64_t action_repeat, int64_t max_episode_steps, int64_t device,
        int64_t done_mode, int64_t stack_mode, uint64_t seed, int64_t first_env) {
        cfg.num_envs = (int32_t)num_envs; cfg.num_players = (int32_t)num_players; cfg.frame_stack = (int32_t)frame_stack;
        cfg.action_repeat = (int32_t)action_repeat; cfg.max_episode_steps = (int32_t)max_episode_steps; cfg.device = (int32_t)device;
        cfg.done_mode = (int32_t)done_mode; cfg.stack_mode = (int32_t)stack_mode; cfg.seed = seed; cfg.first_env = first_env;
        check_rc(crl_car_create(&cfg, &h));
        const int64_t c = frame_stack > 0 ? frame_stack : 1;
        term_numel = num_envs * num_players * c * 96 * 96;
        obs_numel = stack_mode == 1 ? 2 * term_numel : term_numel;
    }
    ~Car() { close(); }
    void close() {
        if (h) { crl_car_destroy(h); h = nullptr; }
    }
    crl_car* handle() const {
        TORCH_CHECK(h != nullptr, "the environment is closed");
        return h;
    }
    int dev() const { return cfg.device; }
    int64_t n() const { return cfg.num_envs; }
    int64_t cars() const { return (int64_t)cfg.num_envs * cfg.num_players; }

    void load_glyphs(const at::Tensor& g) {
        check_rc(crl_car_load_glyphs(handle(), host_ptr<uint8_t>(g, at::kByte, "glyphs"), (size_t)g.numel(), stream_of(dev())));
    }
    void inject_tracks(const at::Tensor& draws, const c10::optional<at::Tensor>& birth) {
        TORCH_CHECK(draws.dim() == 3 && draws.size(0) == n() && draws.size(2) == CRL_CAR_DRAWS, "draws must have shape (num_envs, K, 24)");
        const int32_t* b = nullptr;
        int32_t kb = 0;
        if (birth.has_value()) {
            TORCH_CHECK(birth->dim() == 3 && birth->size(0) == n() && birth->size(2) == cfg.num_players, "birth must have shape (num_envs, K, players)");
            b = host_ptr<int32_t>(*birth, at::kInt, "birth");
            kb = (int32_t)birth->size(1);
        }
        check_rc(crl_car_inject_tracks(handle(), host_ptr<double>(draws, at::kDouble, "draws"), (int32_t)draws.size(1), b, kb, stream_of(dev())));
    }
    void load_tracks(const at::Tensor& pts, const at::Tensor& counts, int64_t n_tracks) {
        check_rc(crl_car_load_tracks(handle(), host_ptr<double>(pts, at::kDouble, "pts"), host_ptr<int32_t>(counts, at::kInt, "counts"),
                                     (int32_t)n_tracks, stream_of(dev())));
    }
    void seed(uint64_t s) { check_rc(crl_car_seed(handle(), s, stream_of(dev()))); }
    void set_elapsed(const at::Tensor& el) {
        check_rc(crl_car_set_elapsed(handle(), dev_ptr<int32_t>(el, at::kInt, dev(), n(), "elapsed"), stream_of(dev())));
    }
    void reset(const at::Tensor& obs) {
        check_rc(crl_car_reset(handle(), dev_ptr<uint8_t>(obs, at::kByte, dev(), obs_numel, "obs"), stream_of(dev())));
    }
    void step(const at::Tensor& actions, const at::Tensor& obs, const at::Tensor& rew, const at::Tensor& done, const at::Tensor& num_steps,
              const at::Tensor& truncated, const c10::optional<at::Tensor>& term) {
        check_rc(crl_car_step(handle(), dev_ptr<float>(actions, at::kFloat, dev(), 2 * cars(), "actions"),
                              dev_ptr<uint8_t>(obs, at::kByte, dev(), obs_numel, "obs"), dev_ptr<float>(rew, at::kFloat, dev(), cars(), "rew"),
                              dev_ptr<uint8_t>(done, at::kBool, dev(), n(), "done"), dev_ptr<int32_t>(num_steps, at::kInt, dev(), n(), "num_steps"),
                              dev_ptr<uint8_t>(truncated, at::kByte, dev(), n(), "truncated"),
                              opt_dev_ptr<uint8_t>(term, at::kByte, dev(), term_numel, "terminal observation"), stream_of(dev())));
    }
    void set_obs_rotation(const std::vector<at::Tensor>& bufs) {
        std::vector<uint8_t*> ptrs;
        for (const at::Tensor& t : bufs) ptrs.push_back(dev_ptr<uint8_t>(t, at::kByte, dev(), obs_numel, "obs buffer of the rotation"));
        check_rc(crl_car_set_obs_rotation(handle(), ptrs.data(), (int32_t)ptrs.size(), stream_of(dev())));
    }
    int64_t ring_phase() {
        const int k = crl_car_ring_phase(handle());
        if (k < 0) check_rc(k);
        return k;
    }
    void get_state(const at::Tensor& state) {
        check_rc(crl_car_get_state(handle(), dev_ptr<double>(state, at::kDouble, dev(), cars() * CRL_CAR_STATE_DOUBLES, "state"), stream_of(dev())));
    }
    void set_state(const at::Tensor& state) {
        check_rc(crl_car_set_state(handle(), dev_ptr<double>(state, at::kDouble, dev(), cars() * CRL_CAR_STATE_DOUBLES, "state"), stream_of(dev())));
    }
    void render_state(const at::Tensor& obs) {
        check_rc(crl_car_render_state(handle(), dev_ptr<uint8_t>(obs, at::kByte, dev(), obs_numel, "obs"), stream_of(dev())));
    }
    at::Tensor get_track(int64_t env) {
        int32_t cnt = 0;
        at::Tensor pts = at::zeros({512, 3}, at::kDouble);
        check_rc(crl_car_get_track(handle(), (int32_t)env, &cnt, pts.data_ptr<double>(), 512, stream_of(dev())));
        return pts.narrow(0, 0, cnt).clone();
    }
    std::vector<uint64_t> stats() {
        std::vector<uint64_t> s(8);
        check_rc(crl_car_get_stats(handle(), s.data(), stream_of(dev())));
        return s;
    }
    std::pair<at::Tensor, int64_t> contacts() {
        at::Tensor counts = at::zeros({n()}, at::kInt);
        int32_t over = 0;
        check_rc(crl_car_get_contacts(handle(), counts.data_ptr<int32_t>(), &over, stream_of(dev())));
        return {counts, (int64_t)over};
    }
    void check() { check_rc(crl_car_check(handle(), stream_of(dev()))); }
    uint64_t raw_handle() const { return (uint64_t)(uintptr_t)h; }
};

// An uninitialised observation buffer: crl_obs_alloc's memory (compressible where the device grants it) viewed as a tensor
// that gives the memory back through crl_obs_free when its storage is released; with compressible=False, torch.empty.
// Returns (tensor, whether the memory is compressible).
std::pair<at::Tensor, bool> obs_empty(const std::vector<int64_t>& shape, at::ScalarType dtype, int64_t device, bool compressible) {
    const auto opts = at::TensorOptions().dtype(dtype).device(at::kCUDA, (c10::DeviceIndex)device);
    if (!compressible) return {at::empty(shape, opts), false};
    int64_t numel = 1;
    for (int64_t d : shape) {
        TORCH_CHECK(d >= 0, "obs_empty: negative dimension");
        numel *= d;
    }
    void* p = nullptr;
    int32_t compressed = 0;
    check_rc(crl_obs_alloc((int32_t)device, std::max<size_t>((size_t)numel * c10::elementSize(dtype), 1), &p, &compressed));
    return {torch::from_blob(p, shape, [](void* q) { crl_obs_free(q); }, opts), compressed != 0};
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
    m.doc() = "torch C++ extension over libcrl_b200.so (include/crl_b200.h)";
    py::register_exception<CrlError>(m, "CrlError", PyExc_RuntimeError);
    m.def("abi_version", []() { return crl_abi_version(); });
    m.def("launch_count", []() { return crl_launch_count(); });
    m.def("obs_empty", &obs_empty, py::arg("shape"), py::arg("dtype"), py::arg("device"), py::arg("compressible") = true);
    py::class_<Pong>(m, "Pong")
        .def(py::init<int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, bool, uint64_t, int64_t>())
        .def("close", &Pong::close)
        .def("load_atlas", &Pong::load_atlas)
        .def("inject_serves", &Pong::inject_serves)
        .def("seed", &Pong::seed)
        .def("reset", &Pong::reset)
        .def("step", &Pong::step)
        .def("render_obs_generic", &Pong::render_obs_generic)
        .def("reset_f32", &Pong::reset_f32)
        .def("step_f32", &Pong::step_f32)
        .def("render_f32", &Pong::render_f32)
        .def("terminal_obs", &Pong::terminal_obs)
        .def("ring_phase", &Pong::ring_phase)
        .def("get_state", &Pong::get_state)
        .def("set_state", &Pong::set_state)
        .def("render_raw", &Pong::render_raw)
        .def("check", &Pong::check)
        .def("set_obs_buffers", &Pong::set_obs_buffers)
        .def("forget_obs", &Pong::forget_obs)
        .def("stats", &Pong::stats)
        .def("raw_handle", &Pong::raw_handle);
    py::class_<Car>(m, "Car")
        .def(py::init<int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, uint64_t, int64_t>())
        .def("close", &Car::close)
        .def("load_glyphs", &Car::load_glyphs)
        .def("inject_tracks", &Car::inject_tracks)
        .def("load_tracks", &Car::load_tracks)
        .def("seed", &Car::seed)
        .def("set_elapsed", &Car::set_elapsed)
        .def("reset", &Car::reset)
        .def("step", &Car::step)
        .def("ring_phase", &Car::ring_phase)
        .def("set_obs_rotation", &Car::set_obs_rotation)
        .def("get_state", &Car::get_state)
        .def("set_state", &Car::set_state)
        .def("render_state", &Car::render_state)
        .def("get_track", &Car::get_track)
        .def("stats", &Car::stats)
        .def("contacts", &Car::contacts)
        .def("check", &Car::check)
        .def("raw_handle", &Car::raw_handle);
}
