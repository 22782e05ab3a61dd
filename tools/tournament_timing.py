"""cPongTournament-v0 step rate against built-in opponents: the uniform torch path against per-env opponents.

    python tools/tournament_timing.py [--envs 65536] [--steps 200] [--warmup 20] [--rounds 3]

42x42, frame_stack None, synthetic LightActorCritic weights saved as checkpoint-{weak,medium}.pkl in a temporary
directory.  Modes, run in alternating rounds in one process:
  (a) uniform  reset_opponent("WEAK"): DevicePolicy (torch roll + cuDNN fp32 convolutions + linear + argmax);
  (b) per-env  set_opponents with every env on WEAK (csrc/pong_opponent.cu);
  (c) mix      set_opponents over RULE_BASED / RANDOM / WEAK / MEDIUM, uniform draw, resample_on_done.
Reported per mode: the wrapper's env-steps/s (host clock over `steps` wrapper steps ending in a synchronise) and the
opponent's own time per step from CUDA events (a: the DevicePolicy call; b, c: the act kernel), plus, once, the bare
cPongDouble step.  The learner's actions are random device tensors generated before the timed window."""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

MACS_PER_ENV = 4 * 16 * 16 * 400 + 16 * 16 * 4 * 100 + 3 * 1600   # LightActorCritic: conv1 + conv2 + actor = 516 800


def synthetic(a, b):
    import torch
    from competitive_rl_b200.builtin_policies import LIGHT_ACTOR_CRITIC_LAYOUT
    sd = {}
    for k, (name, shape) in enumerate(LIGHT_ACTOR_CRITIC_LAYOUT):
        i = np.arange(int(np.prod(shape)), dtype=np.float64)
        sd[name] = torch.from_numpy((0.08 * np.sin(a * i + b * k)).astype(np.float32).reshape(shape))
    return {"model": sd}


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.current.sm", "--format=csv"],
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=30).stdout.strip()
    except Exception as exc:  # noqa: BLE001
        return "nvidia-smi unavailable: %r" % (exc,)


def configure(w, mode):
    if mode == "a_uniform_weak":
        w.reset_opponent("WEAK")
    elif mode == "b_per_env_weak":
        w.set_opponents(assignment=["WEAK"] * w.num_envs, pool=["WEAK"], seed=1)
    else:
        w.set_opponents(pool=["RULE_BASED", "RANDOM", "WEAK", "MEDIUM"], resample_on_done=True, seed=1)


def time_mode(w, mode, acts, steps, warmup):
    import torch
    configure(w, mode)
    stream = torch.cuda.current_stream()
    for t in range(warmup):
        w.step(acts[t % len(acts)])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for t in range(steps):
        w.step(acts[t % len(acts)])
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    # the opponent alone, CUDA events around each call (same state, separate window so the step rate is unperturbed)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    env = w.env
    for t in range(steps):
        ev[t][0].record(stream)
        if w.per_env:
            w._opp.act(env._obs[1], env._rew, env._done, w._resample, w._both, None)
        else:
            w.current_agent(w.prev_opponent_obs)
        ev[t][1].record(stream)
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    return w.num_envs * steps / wall, wall / steps * 1e3, sum(ms) / len(ms), ms[len(ms) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("tournament_timing needs a CUDA device")
    from competitive_rl_b200 import make_envs
    print(gpu_info(), flush=True)
    N = a.envs
    with tempfile.TemporaryDirectory() as res:
        torch.save(synthetic(0.37, 0.0), os.path.join(res, "checkpoint-weak.pkl"))
        torch.save(synthetic(0.23, 2.0), os.path.join(res, "checkpoint-medium.pkl"))
        w = make_envs("cPongTournament-v0", num_envs=N, resized_dim=42, log_dir=None, seed=7, resource_dir=res)
        g = torch.Generator(device=w.env.device)
        g.manual_seed(0)
        acts = [torch.randint(0, 3, (N,), dtype=torch.int32, device=w.env.device, generator=g) for _ in range(64)]
        w.reset()
        # the bare env step, for scale
        both = torch.zeros((N, 2), dtype=torch.int32, device=w.env.device)
        for t in range(a.warmup):
            w.env.step(both)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for t in range(a.steps):
            w.env.step(both)
        torch.cuda.synchronize()
        env_ms = (time.perf_counter() - t0) / a.steps * 1e3
        print("cPongDouble step alone (42x42, frame_stack None): %.4f ms/step, %.1f M env-steps/s" % (env_ms, N / env_ms / 1e3))
        modes = ["a_uniform_weak", "b_per_env_weak", "c_per_env_mix"]
        for r in range(a.rounds):
            for mode in modes:
                rate, ms_step, opp_ms, opp_med = time_mode(w, mode, acts, a.steps, a.warmup)
                extra = ""
                if mode != "a_uniform_weak":
                    nets = float((torch.tensor([k >= 2 for k in range(4)])[w.opponent_ids.long().cpu()]).float().mean()) \
                        if mode == "c_per_env_mix" else 1.0
                    fl = 2.0 * MACS_PER_ENV * N * nets
                    extra = "  network envs %.2f  %.1f TFLOP/s fp32 over the kernel" % (nets, fl / (opp_ms * 1e-3) / 1e12)
                print("round %d %-15s %8.2f M env-steps/s  %.4f ms/step  opponent %.4f ms (median %.4f)%s" % (
                    r + 1, mode, rate / 1e6, ms_step, opp_ms, opp_med, extra), flush=True)
        st = w.opponent_stats()
        print("mix stats after the run:", st)
        w.env.check()
        w.close()
    print(gpu_info(), flush=True)


if __name__ == "__main__":
    main()
