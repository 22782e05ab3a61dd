"""bench.py -- cPongDouble env-steps/s at 84x84x4 observations (BASELINE.json metric), plus the car-racing
configurations (BASELINE configs 4 and 5) as sub-records of the same JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs-per-gpu E] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one vec-env step of the whole shard: every env advances 4 game frames and both
agents' (4, 84, 84) uint8 observations are produced (56 448 B per env-step).  Workload =
BASELINE config 3: 65 536 envs per GPU, device-side random actions, device-side serve RNG.
For N > 1 the driver launches one rank per GPU with torch.distributed.run; envs shard by
index, no collective on the step path ("scaling": "weak").

Prints ONE JSON line (rank 0).  Keys beyond the driver's contract:
  api_step     the same metric through the Python facade, envs.step(device_actions) (torch C++ extension)
  ring         cPongDouble with stack_mode="ring" (double-write ring view, 28 224 B per env-step)
  modes        resized_dim=42 (the make_envs default) in both stack modes
  car_single   cCarRacing-v0, 1024 envs (config 4); car_double: cCarRacingDouble-v0, 16 384 envs per GPU (config 5):
               steady state (envs pre-aged so that TimeLimit resets are spread over the steps, auto-resets inside the
               timed region), p50 / p99 / max step latency, per-kernel split, roofline, e2e, cpu_baseline
`--impl reference` times the CPU oracle port of the reference's path (the reference is Python + un-installable
wheels and cannot travel to the GPU box; see DESIGN.md) with all host threads on a bounded sample of the workload.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_ENV_STEP = 2 * 4 * 84 * 84          # SURVEY.md section 8(d): 56 448 B written per env-step
METRIC = "cPongDouble env-steps/sec at 84x84x4 obs"
UNIT = "env-steps/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--envs-per-gpu", type=int, default=65536)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--cpu-sample-envs", type=int, default=256)
    ap.add_argument("--cpu-sample-steps", type=int, default=0, help="0 = auto (about 10-20 s of CPU work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--car-steps", type=int, default=1100, help="timed steps of the car legs (0 = skip the cars)")
    ap.add_argument("--car-single-envs", type=int, default=1024)
    ap.add_argument("--car-double-envs", type=int, default=16384)
    ap.add_argument("--no-modes", action="store_true", help="skip the ring / 42x42 / api_step side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed cPongDouble step returned to "
                    "DIR/<name>.npy (float32 / float64), so that two builds can be compared output for output")
    return ap.parse_args()


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profiled_traffic(kernel_key, units):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel_key` from the committed ncu --set full capture
    (profiles/kernel_traffic.json: bytes per unit at a stated size), scaled to `units`; None when no capture is committed."""
    p = os.path.join(ROOT, "profiles", "kernel_traffic.json")
    try:
        rec = json.load(open(p))[kernel_key]
        return (rec["dram_read_bytes"] + rec["dram_write_bytes"]) / rec["units"] * units, rec.get("source")
    except Exception:  # noqa: BLE001
        return None, None


# --------------------------------------------------------------------------- CPU baselines
def cpu_baseline(sample_envs, sample_steps, threads, min_seconds=2.0):
    """The oracle port of the reference's path (oracle/pong_oracle.c: renders all four 210x160x3
    frames per env-step like the reference, max-pool, cv2-exact gray+area, per-agent 4-stack),
    envs split over `threads` host threads the way SubprocVecEnv splits them over processes."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import pong_oracle
    atlas = np.load(os.path.join(ROOT, "competitive-rl_b200", "data", "scoreboard_atlas.npz"))["strips"]
    pong_oracle.set_threads(threads)
    v = pong_oracle.PongOracleVec("cPongDouble-v0", sample_envs, 84, 4, 21, atlas, None, seed=1)
    v.reset()
    rng = np.random.default_rng(0)
    acts = rng.integers(0, 3, (64, sample_envs, 2)).astype(np.int32)
    for t in range(3):
        v.step(acts[t])
    if sample_steps <= 0:
        t0 = time.perf_counter()
        for t in range(4):
            v.step(acts[t])
        per = (time.perf_counter() - t0) / 4
        sample_steps = int(max(8, min(4000, 12.0 / max(per, 1e-6))))
    t0 = time.perf_counter()
    done = 0
    while done < sample_steps or time.perf_counter() - t0 < min_seconds:
        v.step(acts[done % 64])
        done += 1
    dt = time.perf_counter() - t0
    v.close()
    return {
        "value": sample_envs * done / dt, "unit": UNIT, "cores": threads, "kind": "port",
        "sample": "%d envs x %d vec-steps of cPongDouble 84x84x4, random actions, oracle/pong_oracle.c, %.1f s"
                  % (sample_envs, done, dt),
    }


def car_cpu_baseline(players, threads, seconds=6.0, render=True):
    """oracle/car_oracle.c (mini Box2D + the per-pixel renderer restatement) on `threads` host threads, one env
    each, uniform random actions.  With render=False the physics alone (the oracle's renderer evaluates every polygon
    per pixel -- a checker, not pygame's blitter -- so the rendering figure understates what the reference's CPU path does)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import car_oracle as C
    glyphs = C.load_glyphs(os.path.join(ROOT, "competitive-rl_b200", "data", "car_hud_glyphs.npz"))
    counts = [0] * threads
    stop = time.perf_counter() + seconds

    def work(k):
        rng = np.random.RandomState(100 + k)
        track, border, _ = C.make_track(rng)
        env = C.CarOracleEnv(players, 1, glyphs, render=render)
        env.reset(track, border, list(range(players)))
        n = 0
        while time.perf_counter() < stop:
            env.step(rng.uniform(-1, 1, (players, 2)))
            n += 1
            if n % 1000 == 0:
                env.reset(track, border, list(range(players)))
        counts[k] = n
        env.close()

    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(k,)) for k in range(threads)]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    dt = time.perf_counter() - t0
    return {"value": sum(counts) / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d envs (one per host thread) x %.1f s of %s, uniform random actions, oracle/car_oracle.c, %s"
                      % (threads, dt, "cCarRacingDouble-v0" if players == 2 else "cCarRacing-v0",
                         "physics + per-pixel observation renderer" if render else "physics only (no observation)")}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# --------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """nvidia-smi -lms loop running across the timed region; samples are filtered to the
    [mark_start, mark_stop] wall-clock window (B200_PROFILING.md clocks line)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index):
        self.index, self.proc, self.t0, self.t1 = index, None, None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:  # noqa: BLE001
            self.proc = None

    def mark_start(self):
        self.t0 = time.time()

    def mark_stop(self):
        self.t1 = time.time()

    def stop(self):
        import datetime
        lines = []
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
                lines = out.strip().splitlines()
            except Exception:  # noqa: BLE001
                self.proc.kill()
        inside, every = [], []
        for ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7 or not f[1].isdigit():
                continue
            every.append(f)
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                continue
            if self.t0 is not None and self.t0 - 0.05 <= ts <= self.t1 + 0.05:
                inside.append(f)
        use = inside if inside else every
        sm = sorted(int(s[1]) for s in use)
        mx = [int(s[2]) for s in use if s[2].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in use for n, v in zip(names, s[3:7]) if v.lower().startswith("active")})
        pw = [float(s[7]) for s in use if len(s) > 7 and s[7].replace(".", "", 1).isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(use), "samples_in_timed_region": len(inside),
                "power_w_max": max(pw) if pw else None}


class Ctx(object):
    """rank / device / collective helpers shared by the legs"""

    def __init__(self, a):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU path)"
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.stream = torch.cuda.current_stream(self.dev)
        self.sp = ctypes.c_void_p(self.stream.cuda_stream)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, vals):
        if self.world == 1:
            return [float(v) for v in vals]
        tt = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(tt, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in tt.tolist()]

    def sum_over_ranks(self, vals):
        if self.world == 1:
            return [float(v) for v in vals]
        tt = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(tt, op=self.dist.ReduceOp.SUM)
        return [float(x) for x in tt.tolist()]


def P(t):
    return ctypes.c_void_p(t.data_ptr())


# --------------------------------------------------------------------------- Pong: the headline leg
DUMP_ENVS = 1 << 19          # per-env arrays: 32 B per env with its index, 16.8 MB at most
DUMP_OBS_ENVS = 128          # both agents' (4, 84, 84) stacks as float32: 28.9 MB


def dump_outputs(d, N, obs0, obs1, rew, done, steps_t, real):
    """The arrays crl_pong_step_state + crl_pong_render_obs wrote, as float32 .npy files under d (under 64 MB in all).
    Envs are a fixed seeded sample: every env up to DUMP_ENVS for the per-env arrays, DUMP_OBS_ENVS of them for the
    observations; env_index / obs_env_index name the envs kept."""
    import numpy as np
    import torch
    perm = np.random.default_rng(0).permutation(N)
    env_idx, obs_idx = np.sort(perm[:DUMP_ENVS]), np.sort(perm[:DUMP_OBS_ENVS])

    def take(t, idx):
        return t.index_select(0, torch.from_numpy(idx).to(t.device)).to(torch.float32).cpu().numpy()
    out = {"env_index": env_idx.astype(np.float64), "reward": take(rew, env_idx), "done": take(done, env_idx),
           "num_steps": take(steps_t, env_idx), "real_reward": take(real, env_idx),
           "obs_env_index": obs_idx.astype(np.float64), "obs_agent0": take(obs0, obs_idx), "obs_agent1": take(obs1, obs_idx)}
    os.makedirs(d, exist_ok=True)
    for name, x in out.items():
        np.save(os.path.join(d, name + ".npy"), x)


def pong_leg(cx, a, N, dim=84, stack_mode="stack", steps=None, warmup=None, with_e2e=True, with_clocks=True, dump_dir=None):
    """Device-timed rollout through the C ABI (random actions + game core + rasteriser); returns a record.  With
    dump_dir, the outputs of the last timed step are written there (dump_outputs) before anything else runs."""
    import numpy as np
    from competitive_rl_b200 import _native, make_envs
    torch = cx.torch
    lib = _native.load()
    steps = a.steps if steps is None else steps
    warmup = max(3, a.warmup if warmup is None else warmup)
    envs = make_envs("cPongDouble-v0", seed=1000, log_dir=None, num_envs=N, asynchronous=True, resized_dim=dim,
                     frame_stack=4, first_env=cx.rank * N, n_buffers=1, stack_mode=stack_mode)
    envs.reset()
    h = envs._h
    stream, sp = cx.stream, cx.sp
    actions = torch.zeros((N, 2), dtype=torch.int32, device=cx.dev)
    obs0, obs1 = envs._store
    rew, done, steps_t, real = envs._rew, envs._done, envs._steps, envs._real
    act_seed = 1000 + cx.rank
    bytes_step = envs.bytes_per_env_step

    def one_step(t, ev=None):
        _native.check(lib.crl_pong_random_actions(P(actions), 2 * N, act_seed, t, sp))
        _native.check(lib.crl_pong_step_state(h, P(actions), P(rew), P(done), P(steps_t), P(real), sp))
        if ev is not None:
            ev[0].record(stream)
        _native.check(lib.crl_pong_render_obs(h, P(obs0), P(obs1), sp))
        if ev is not None:
            ev[1].record(stream)

    sampler = ClockSampler(cx.local) if with_clocks else None
    if sampler:
        sampler.start()
    t = 0
    for _ in range(warmup):
        one_step(t)
        t += 1
    # ---- timed region: device-resident inputs, CUDA events on the launching stream ----
    kern_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cx.barrier()
    if sampler:
        sampler.mark_start()
    l0 = _native.launch_count()
    e0.record(stream)
    for k in range(steps):
        one_step(t, kern_ev[k])
        t += 1
    e1.record(stream)
    cx.barrier()
    if sampler:
        sampler.mark_stop()
    launches = _native.launch_count() - l0
    clocks = sampler.stop() if sampler else None
    if dump_dir:
        dump_outputs(dump_dir, N, obs0, obs1, rew, done, steps_t, real)
    ms = e0.elapsed_time(e1)
    raster_ms = sum(x.elapsed_time(y) for x, y in kern_ev) / steps
    rec = {"ms": ms, "raster_ms": raster_ms, "launches": launches, "clocks": clocks, "steps": steps, "warmup": warmup,
           "bytes_per_env_step": bytes_step}

    if with_e2e:
        # ---- e2e: through the host-buffer C-ABI call (pinned host memory, copies inside the timed region) ----
        K2 = max(10, min(steps, 200))
        rng = np.random.default_rng(1000 + cx.rank)
        h_act = torch.from_numpy(rng.integers(0, 3, (N, 2)).astype(np.int32)).pin_memory()
        h_rew = torch.zeros((N, 2), dtype=torch.float32).pin_memory()
        h_done = torch.zeros((N,), dtype=torch.uint8).pin_memory()
        h_steps = torch.zeros((N,), dtype=torch.int32).pin_memory()
        h_real = torch.zeros((N, 2), dtype=torch.float32).pin_memory()

        def host_step(o0=None, o1=None):
            _native.check(lib.crl_pong_step_host(h, P(h_act), P(obs0), P(obs1), o0, o1, P(h_rew), P(h_done),
                                                 P(h_steps), P(h_real), sp))
        for _ in range(3):
            host_step()
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(K2):
            host_step()
        cx.barrier()
        rec["e2e_s"], rec["e2e_steps"] = time.perf_counter() - t0, K2
        rec["h2d"] = h_act.numel() * 4
        rec["d2h"] = h_rew.numel() * 4 + h_done.numel() + h_steps.numel() * 4 + h_real.numel() * 4
        # ---- the numpy-style call that also brings both observation stacks to the host ----
        if stack_mode == "stack":
            K3 = 3
            h_o0 = torch.empty(obs0.shape, dtype=torch.uint8).pin_memory()
            h_o1 = torch.empty(obs1.shape, dtype=torch.uint8).pin_memory()
            host_step(P(h_o0), P(h_o1))
            cx.barrier()
            t0 = time.perf_counter()
            for _ in range(K3):
                host_step(P(h_o0), P(h_o1))
            cx.barrier()
            rec["e2e_obs_s"], rec["e2e_obs_steps"], rec["obs_bytes"] = time.perf_counter() - t0, K3, 2 * obs0.numel()
            del h_o0, h_o1
        # ---- context for the roofline: what a plain fill of the same observation buffers sustains on this GPU (the
        #      path writes and never reads, so the pure-write rate, not the read+write copy rate, is its ceiling) ----
        fill_views = [obs0.view(torch.int32), obs1.view(torch.int32)]
        for _ in range(3):
            for v in fill_views:
                v.fill_(0)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(cx.dev)
        f0.record(stream)
        for _ in range(25):
            for v in fill_views:
                v.fill_(0)
        f1.record(stream)
        torch.cuda.synchronize(cx.dev)
        rec["fill_gbps"] = 25 * 2 * obs0.numel() / (f0.elapsed_time(f1) / 1e3) / 1e9
    envs.close()
    del envs, obs0, obs1
    torch.cuda.empty_cache()
    return rec


def api_leg(cx, N, steps, dim=84, stack_mode="stack"):
    """The same rollout through the Python facade: envs.step(device action tensor) -- what a torch trainer calls.
    Actions come from a pre-generated device tensor bank (the policy's output in a real loop)."""
    from competitive_rl_b200 import make_envs
    torch = cx.torch
    envs = make_envs("cPongDouble-v0", seed=1000, log_dir=None, num_envs=N, asynchronous=True, resized_dim=dim,
                     frame_stack=4, first_env=cx.rank * N, n_buffers=1, stack_mode=stack_mode)
    envs.reset()
    g = torch.Generator(device=cx.dev)
    g.manual_seed(1000 + cx.rank)
    bank = torch.randint(0, 3, (16, N, 2), dtype=torch.int32, device=cx.dev, generator=g)
    for k in range(10):
        envs.step(bank[k % 16])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cx.barrier()
    e0.record(cx.stream)
    for k in range(steps):
        obs, rew, done, infos = envs.step(bank[k % 16])
    e1.record(cx.stream)
    cx.barrier()
    ms = e0.elapsed_time(e1)
    envs.close()
    del envs, obs
    torch.cuda.empty_cache()
    return ms


# --------------------------------------------------------------------------- cars
def car_leg(cx, a, env_id, N, steps, stack_mode="stack"):
    """Steady-state rollout of the car path: the envs are pre-aged uniformly over the 1000-step TimeLimit so that about
    N / 1000 of them finish (terminal observation, auto-reset, reset frame) on EVERY step, inside the timed region."""
    import numpy as np
    from competitive_rl_b200 import _native, make_envs
    torch = cx.torch
    lib = _native.load()
    players = 2 if "Double" in env_id else 1
    envs = make_envs(env_id, num_envs=N, frame_stack=4, log_dir=None, seed=1, asynchronous=True, n_buffers=2,
                     first_env=cx.rank * N, stack_mode=stack_mode)
    envs.reset()
    rng = np.random.default_rng(7 + cx.rank)
    envs.set_elapsed(rng.integers(0, 1000, N))
    h = envs._h
    stream, sp = cx.stream, cx.sp
    actions = torch.zeros((N, players, 2), dtype=torch.float32, device=cx.dev)
    bytes_step = envs.bytes_per_env_step
    warm = 30

    def one(t):
        b = envs.next_set()     # stack mode: the next observation buffer of the rotation the env registered with the library
        _native.check(lib.crl_car_random_actions(P(actions), actions.numel(), 7 + cx.rank, t, sp))
        _native.check(lib.crl_car_step(h, P(actions), P(b["obs"]), P(b["rew"]), P(b["done"]), P(b["steps"]), P(b["trunc"]),
                                       P(b["term"]), sp))

    sampler = ClockSampler(cx.local)
    sampler.start()
    t = 0
    for _ in range(warm):
        one(t)
        t += 1
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    stats0 = envs.episode_stats()
    cx.barrier()
    sampler.mark_start()
    l0 = _native.launch_count()
    ev[0].record(stream)
    for k in range(steps):
        one(t)
        t += 1
        ev[k + 1].record(stream)
    cx.barrier()
    sampler.mark_stop()
    launches = _native.launch_count() - l0
    clocks = sampler.stop()
    ms = ev[0].elapsed_time(ev[steps])
    lat = sorted(ev[k].elapsed_time(ev[k + 1]) for k in range(steps))
    stats1 = envs.episode_stats()
    finished = stats1["episodes"] - stats0["episodes"]

    # ---- per-kernel split: the two halves back to back (the combined call of two-car envs overlaps them) ----
    K = min(steps, 200)
    sev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    for k in range(K):
        _native.check(lib.crl_car_random_actions(P(actions), actions.numel(), 7 + cx.rank, t, sp))
        t += 1
        b = envs.next_set()
        sev[k][0].record(stream)
        _native.check(lib.crl_car_step_state(h, P(actions), P(b["rew"]), P(b["done"]), P(b["steps"]), P(b["trunc"]), sp))
        sev[k][1].record(stream)
        _native.check(lib.crl_car_render_obs(h, P(b["obs"]), P(b["term"]), sp))
        sev[k][2].record(stream)
    cx.barrier()
    phys = sum(e[0].elapsed_time(e[1]) for e in sev) / K
    rend = sum(e[1].elapsed_time(e[2]) for e in sev) / K

    # ---- e2e: host actions in, rewards / dones / counters out, observations stay in HBM ----
    K2 = min(steps, 100)
    h_act = torch.from_numpy(rng.uniform(-1, 1, (N, players, 2)).astype(np.float32)).pin_memory()
    h_rew = torch.zeros((N, players), dtype=torch.float32).pin_memory()
    h_done = torch.zeros((N,), dtype=torch.uint8).pin_memory()
    h_steps = torch.zeros((N,), dtype=torch.int32).pin_memory()
    h_trunc = torch.zeros((N,), dtype=torch.uint8).pin_memory()

    def host_step():
        b = envs.next_set()
        _native.check(lib.crl_car_step_host(h, P(h_act), P(b["obs"]), None, P(h_rew), P(h_done), P(h_steps), P(h_trunc),
                                            P(b["term"]), sp))
    for _ in range(3):
        host_step()
    cx.barrier()
    t0 = time.perf_counter()
    for _ in range(K2):
        host_step()
    cx.barrier()
    e2e_s = time.perf_counter() - t0

    # ---- the Python API: envs.step(device actions) through the torch C++ extension (what a trainer calls) ----
    K3 = min(steps, 200)
    for k in range(5):
        _native.check(lib.crl_car_random_actions(P(actions), actions.numel(), 7 + cx.rank, t + k, sp))
        envs.step(actions if players == 2 else actions.view(N, 2))
    cx.barrier()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record(stream)
    for k in range(K3):
        _native.check(lib.crl_car_random_actions(P(actions), actions.numel(), 7 + cx.rank, t + 5 + k, sp))
        envs.step(actions if players == 2 else actions.view(N, 2))
    a1.record(stream)
    # ... and the C-ABI call over the next K3 steps of the same rollout (the workload drifts as episodes age: compare like with like)
    for k in range(K3):
        one(t + 5 + K3 + k)
    a2 = torch.cuda.Event(enable_timing=True)
    a2.record(stream)
    cx.barrier()
    api_ms, abi_ms = a0.elapsed_time(a1), a1.elapsed_time(a2)
    envs.check()
    envs.close()
    del envs
    torch.cuda.empty_cache()

    ms, phys, rend, e2e_s, p50, p99, pmax, api_ms, abi_ms = cx.max_over_ranks(
        [ms, phys, rend, e2e_s, lat[len(lat) // 2], lat[min(len(lat) - 1, int(len(lat) * 0.99))], lat[-1], api_ms, abi_ms])
    finished = int(cx.sum_over_ranks([finished])[0])
    peak, peak_src = measured_peak()
    total = N * cx.world
    achieved = bytes_step * N / (ms / steps / 1e3) / 1e9
    traffic, tsrc = profiled_traffic("car_render_kernel/%s/%s" % (env_id, stack_mode), 2 * N if players == 2 else N)
    rec = {
        "metric": "%s env-steps/sec at 96x96x%d obs" % (env_id, 4 * players), "value": total * steps / (ms / 1e3), "unit": UNIT,
        "n_gpus": cx.world, "steps": steps, "warmup": warm, "ms_per_step": ms / steps, "scaling": "weak",
        "step_latency_ms": {"p50": p50, "p99": p99, "max": pmax},
        "episodes_finished": finished, "resets_per_step": finished / steps,
        "resets_without_pregenerated_track": int(stats1["resets_without_pregenerated_track"]),   # auto-resets that had to build their track inside the step
        "config": {"workload": "%s, %d envs per GPU x %d GPU(s), frame_stack 4, action_repeat 1, uniform random actions "
                               "(device Philox), TimeLimit 1000 with envs pre-aged uniformly over [0, 1000): auto-resets "
                               "(terminal observation + new track + reset frame) inside the timed region on every step"
                               % (env_id, N, cx.world), "envs_per_gpu": N, "bytes_per_env_step": bytes_step,
                   "stack_mode": stack_mode,
                   "l2": "each step writes %.3f GB per GPU%s" % (bytes_step * N / 1e9, " (> 126 MB L2)" if bytes_step * N > 126e6
                                                                 else " (fits L2: figures are L2-resident)")},
        "kernel_ms": {"step_state (car_step_kernel)": phys, "render_obs (setup + render + auto-reset passes)": rend,
                      "note": "the two halves timed back to back over %d steps; ms_per_step times the combined crl_car_step "
                              "(two-car envs: touching cars on a side stream, overlapped with the render)" % K},
        "roofline": {"bound": "hbm", "limiter": "instruction issue (rasteriser) and dependent latency (180 + 60 solver "
                                                 "iterations per car): HBM is not the binding roof of this path",
                     "kernel": "crl_car_step (whole step)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "traffic_source": tsrc, "peak_source": peak_src,
                     "bytes_per_launch": bytes_step * N},
        "e2e": {"value": total * K2 / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h_act.numel() * 4 * cx.world,
                "d2h_bytes_per_step": (h_rew.numel() * 4 + 2 * N + 4 * N) * cx.world,
                "note": "crl_car_step_host: pinned host actions in; rewards, dones, num_steps, truncated out; observations "
                        "stay in HBM"},
        "api_step": {"value": total * K3 / (api_ms / 1e3), "unit": UNIT, "ms_per_step": api_ms / K3,
                     "ratio_to_c_abi_same_phase": abi_ms / api_ms,
                     "note": "envs.step(float32 device tensor) -> (obs, rew, done, infos) through the torch C++ extension, "
                             "device-timed over %d steps; the ratio compares it with crl_car_step over the next %d steps of the "
                             "same rollout (the workload drifts as the episodes age)" % (K3, K3)},
        "gpu_launches": int(launches), "clocks": clocks,
    }
    if cx.rank == 0 and not a.no_cpu_baseline and cx.world == 1:
        rec["cpu_baseline"] = car_cpu_baseline(players, host_threads(), seconds=5.0, render=True)
        rec["cpu_baseline_physics_only"] = car_cpu_baseline(players, host_threads(), seconds=3.0, render=False)
    return rec


# --------------------------------------------------------------------------- our arm
def run_ours(a):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.gpus > 1 and world == 1:   # plain `python bench.py --gpus N`: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(a.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000)] + sys.argv
        sys.exit(subprocess.call(cmd))
    cx = Ctx(a)
    world, rank = cx.world, cx.rank
    N = a.envs_per_gpu

    r = pong_leg(cx, a, N, dump_dir=a.dump_outputs if rank == 0 else None)
    ms, raster_ms, e2e_s, e2e_obs_s = cx.max_over_ranks([r["ms"], r["raster_ms"], r["e2e_s"], r["e2e_obs_s"]])
    total_envs = N * world
    value = total_envs * a.steps / (ms / 1e3)
    peak, peak_src = measured_peak()
    achieved = BYTES_PER_ENV_STEP * N / (raster_ms / 1e3) / 1e9
    traffic, tsrc = profiled_traffic("pong_raster_fast_kernel<84>/stack", N)
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": r["warmup"],
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8 obs / int32+f64 game state / f32 area-resize", "data": "synthetic",
        "config": {"workload": "cPongDouble-v0, %d envs per GPU x %d GPU(s), frameskip 4, 84x84x4 uint8 obs per agent, "
                               "device-side random actions (Philox) and serve RNG, auto-reset" % (N, world),
                   "envs_per_gpu": N, "bytes_per_env_step": BYTES_PER_ENV_STEP,
                   "l2": "each step writes %.2f GB per GPU (>> 126 MB L2); no flush needed"
                         % (BYTES_PER_ENV_STEP * N / 1e9)},
        "roofline": {"bound": "hbm", "kernel": "pong_raster_fast_kernel<84>", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak,
                     # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed ncu --set full
                     # capture (profiles/kernel_traffic.json names the .ncu-rep summary it was read from)
                     "traffic": traffic, "traffic_source": tsrc, "peak_source": peak_src,
                     "avg_launch_ms": raster_ms, "bytes_per_launch": BYTES_PER_ENV_STEP * N,
                     "sustained_fill_GBps": r["fill_gbps"], "frac_of_sustained_fill": achieved / r["fill_gbps"],
                     "note": "peak = read+write copy rate (MEASURED_PEAKS.json); sustained_fill = torch fill_ of the same "
                             "observation buffers, 25 back-to-back passes, measured in this run: the pure-write rate "
                             "a write-only path is bounded by (see profiles/r01_store_pattern_probe.txt)"},
        "e2e": {"value": total_envs * r["e2e_steps"] / e2e_s, "unit": UNIT, "h2d_bytes_per_step": r["h2d"] * world,
                "d2h_bytes_per_step": r["d2h"] * world,
                "note": "crl_pong_step_host (the C-ABI host-buffer call): pinned host actions in, rew/done/num_steps/real_reward "
                        "out (copied on a side stream behind the rasteriser, joined before the call returns); observations "
                        "stay in HBM (the API returns device tensors).  With the observations copied to the host as well "
                        "the same call is PCIe-bound: see e2e_host_obs"},
        "e2e_host_obs": {"value": total_envs * r["e2e_obs_steps"] / e2e_obs_s, "unit": UNIT,
                         "d2h_bytes_per_step": (r["d2h"] + r["obs_bytes"]) * world,
                         "note": "same call with both observation stacks copied to pinned host memory (PCIe-bound)"},
        "gpu_launches": int(r["launches"]), "clocks": r["clocks"],
    }

    if not a.no_modes:
        # ---- the Python facade (torch C++ extension): envs.step(device_actions) ----
        k_api = max(50, min(a.steps, 500))
        api_ms, = cx.max_over_ranks([api_leg(cx, N, k_api)])
        out["api_step"] = {"value": total_envs * k_api / (api_ms / 1e3), "unit": UNIT, "ms_per_step": api_ms / k_api,
                           "ratio_to_value": total_envs * k_api / (api_ms / 1e3) / value,
                           "note": "envs.step(int32 device tensor (N, 2)) -> (obs tuple, rew, done, infos) through the "
                                   "torch C++ extension, device-timed over %d steps" % k_api}
        # ---- opt-in double-write ring view of the same workload: the newest frame is written twice, 28 224 B ----
        k_m = max(50, min(a.steps, 500))
        rr = pong_leg(cx, a, N, 84, "ring", steps=k_m, warmup=10, with_e2e=False, with_clocks=False)
        rms, rras = cx.max_over_ranks([rr["ms"], rr["raster_ms"]])
        out["ring"] = {"value": total_envs * k_m / (rms / 1e3), "unit": UNIT, "ms_per_step": rms / k_m,
                       "bytes_per_env_step": rr["bytes_per_env_step"],
                       "roofline": {"bound": "hbm", "achieved": rr["bytes_per_env_step"] * N / (rras / 1e3) / 1e9, "peak": peak,
                                    "unit": "GB/s", "frac": rr["bytes_per_env_step"] * N / (rras / 1e3) / 1e9 / peak,
                                    "avg_launch_ms": rras},
                       "note": "stack_mode='ring': observations are strided views obs[:, k+1:k+5] of a (N, 8, 84, 84) ring "
                               "in which each new frame is stored at slots k and k+4; same frames, half the bytes"}
        modes = {}
        for sm in ("stack", "ring"):
            m = pong_leg(cx, a, N, 42, sm, steps=k_m, warmup=10, with_e2e=False, with_clocks=False)
            mms, mras = cx.max_over_ranks([m["ms"], m["raster_ms"]])
            modes["42x42x4/" + sm] = {
                "value": total_envs * k_m / (mms / 1e3), "unit": UNIT, "ms_per_step": mms / k_m,
                "bytes_per_env_step": m["bytes_per_env_step"],
                "roofline": {"bound": "hbm", "achieved": m["bytes_per_env_step"] * N / (mras / 1e3) / 1e9, "peak": peak,
                             "unit": "GB/s", "frac": m["bytes_per_env_step"] * N / (mras / 1e3) / 1e9 / peak,
                             "avg_launch_ms": mras}}
        out["modes"] = modes

    if a.car_steps > 0:
        if world == 1:
            out["car_single"] = car_leg(cx, a, "cCarRacing-v0", a.car_single_envs, a.car_steps)
        out["car_double"] = car_leg(cx, a, "cCarRacingDouble-v0", a.car_double_envs, a.car_steps)
        if not a.no_modes:
            ring = car_leg(cx, a, "cCarRacingDouble-v0", a.car_double_envs, min(a.car_steps, 300), stack_mode="ring")
            ring.pop("cpu_baseline", None)
            ring.pop("cpu_baseline_physics_only", None)
            out["car_double_ring"] = ring

    if rank == 0 and not a.no_cpu_baseline and world == 1:
        out["cpu_baseline"] = cpu_baseline(a.cpu_sample_envs, a.cpu_sample_steps, host_threads())
    if world > 1:
        cx.dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(out))


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    # one "step" here = one vec-step of the bounded sample; K steps timed after W warm-up
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import pong_oracle
    atlas = np.load(os.path.join(ROOT, "competitive-rl_b200", "data", "scoreboard_atlas.npz"))["strips"]
    pong_oracle.set_threads(threads)
    E = a.cpu_sample_envs
    v = pong_oracle.PongOracleVec("cPongDouble-v0", E, 84, 4, 21, atlas, None, seed=1)
    v.reset()
    rng = np.random.default_rng(0)
    acts = rng.integers(0, 3, (64, E, 2)).astype(np.int32)
    for t in range(max(3, a.warmup)):
        v.step(acts[t % 64])
    steps = a.steps
    t0 = time.perf_counter()
    for t in range(steps):
        v.step(acts[t % 64])
    dt = time.perf_counter() - t0
    val = E * steps / dt
    cb = {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
          "sample": "%d envs x %d vec-steps of cPongDouble 84x84x4 (oracle/pong_oracle.c, all host threads), %.1f s" % (E, steps, dt)}
    ref_py = None
    try:   # the reference's own Python, measured in the build container (it cannot travel): committed artefact
        ref_py = json.load(open(os.path.join(ROOT, "profiles", "r02_reference_make_envs_cpu.json")))
    except Exception:  # noqa: BLE001
        pass
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
        "warmup": max(3, a.warmup), "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8 obs / int32+f64 game state / f32 area-resize", "data": "synthetic",
        "config": {"workload": "cPongDouble-v0 frameskip 4, 84x84x4 uint8 obs per agent, random actions; CPU sample of "
                               "%d envs per vec-step on %d host threads" % (E, threads)},
        "cpu_baseline": cb,
        "reference_python_make_envs": ref_py,
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


if __name__ == "__main__":
    args = parse_args()
    if args.steps < 1:
        sys.exit("bench.py: --steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            sys.exit("bench.py: --dump-outputs writes the device path's outputs; it does not apply to --impl reference")
        run_reference(args)
    else:
        run_ours(args)
