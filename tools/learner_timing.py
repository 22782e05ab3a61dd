"""PPO rollout step rate on cPongTournament-v0 with per-env opponents: a torch learner against the learner in the
opponents' kernel (TournamentEnvWrapper.learner_step, csrc/pong_opponent.cu learner mode).

    python tools/learner_timing.py [--envs 65536] [--steps 200] [--warmup 20] [--rounds 3]

42x42, frame_stack None, synthetic LightActorCritic weights (tournament_timing.synthetic) for WEAK, MEDIUM and the
learner.  Modes, each with two pools (mixed: RULE_BASED / RANDOM / WEAK / MEDIUM drawn uniformly with resample_on_done;
weak: every env on WEAK), run in alternating rounds in one process:
  (a) torch     today's loop: FrameStackTensor stacking of agent 0's frames (float32, zeroed on done), a torch
                LightActorCritic with default torch settings (cuDNN may use TF32), Categorical sampling and log-prob,
                then step() in per-env mode;
  (b) kernel    learner_step(): stacking, learner and opponents in one launch, then the env step;
  (c) control   step() in per-env mode with precomputed random learner actions (tournament_timing's mode).
Reported per mode: env-steps/s (host clock over `steps` steps ending in a synchronise) and, from CUDA events in a
separate window, the learner's work per step (a: stacking + network + sampling; b, c: the act kernel).  For (b) with
the weak pool, the kernel's fraction of the fp32 FMA bound: (2 x 516 800 + 1 600) MACs per env over
(SMs x 128 FMA/clk x max SM clock)."""
import argparse
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)

import league_timing as lt  # noqa: E402
import tournament_timing as tt  # noqa: E402

POOLS = {"mixed": dict(pool=["RULE_BASED", "RANDOM", "WEAK", "MEDIUM"], resample_on_done=True, seed=1),
         "weak": dict(pool=["WEAK"], seed=1)}


def configure(w, pool, learner):
    kw = dict(POOLS[pool])
    if pool == "weak":
        kw["assignment"] = ["WEAK"] * w.num_envs
    w.set_opponents(**kw)
    w.set_learner(learner)
    w.reset()


def events(steps):
    import torch
    return [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]


def summary(ev):
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    return sum(ms) / len(ms), ms[len(ms) // 2]


def time_torch(w, pool, learner, steps, warmup):
    """(a): the learner as a torch module over a FrameStackTensor stack, then step()."""
    import torch
    from torch.distributions import Categorical
    configure(w, pool, learner)
    n, dev = w.num_envs, w.env.device
    stack = torch.zeros((n, 4, 42, 42), dtype=torch.float32, device=dev)
    state = {"obs": w.env._obs[0], "done": None}

    def act():
        if state["done"] is not None:
            stack[state["done"]] = 0
        stack[:, :-1] = stack[:, 1:].clone()
        stack[:, -1] = state["obs"].reshape(n, 42, 42)
        with torch.no_grad():
            logits, value = learner(stack)
            dist = Categorical(logits=logits)
            a = dist.sample()
            dist.log_prob(a)
        return a

    def one():
        a = act()
        obs, rew, done, _ = w.step(a)
        state["obs"], state["done"] = obs, done[:, 0]

    for _ in range(warmup):
        one()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ev = events(steps)
    stream = torch.cuda.current_stream()
    for t in range(steps):
        ev[t][0].record(stream)
        act()
        ev[t][1].record(stream)
    torch.cuda.synchronize()
    return (n * steps / wall, wall / steps * 1e3) + summary(ev)


def time_kernel(w, pool, learner, steps, warmup):
    """(b): learner_step(), then the act_learner kernel alone under CUDA events."""
    import torch
    configure(w, pool, learner)
    n, env = w.num_envs, w.env
    for _ in range(warmup):
        w.learner_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        w.learner_step()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ev = events(steps)
    stream = torch.cuda.current_stream()
    both = torch.empty((n, 2), dtype=torch.int32, device=env.device)
    lpv = torch.empty((n, 2), dtype=torch.float32, device=env.device)
    out = torch.empty((n, 4, 42, 42), dtype=torch.uint8, device=env.device)
    for t in range(steps):       # no rew / done: the kernel alone, without crediting the last step's episodes again
        ev[t][0].record(stream)
        w._opp.act_learner(env._obs[0], env._obs[1], None, None, False, True, both, lpv, None, out)
        ev[t][1].record(stream)
    torch.cuda.synchronize()
    return (n * steps / wall, wall / steps * 1e3) + summary(ev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("learner_timing needs a CUDA device")
    from competitive_rl_b200 import make_envs
    from competitive_rl_b200.builtin_policies import LightActorCritic
    print(tt.gpu_info(), flush=True)
    clock = lt.max_sm_clock_hz()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = a.envs
    with tempfile.TemporaryDirectory() as res:
        torch.save(tt.synthetic(0.37, 0.0), os.path.join(res, "checkpoint-weak.pkl"))
        torch.save(tt.synthetic(0.23, 2.0), os.path.join(res, "checkpoint-medium.pkl"))
        w = make_envs("cPongTournament-v0", num_envs=n, resized_dim=42, log_dir=None, seed=7, resource_dir=res)
        learner = LightActorCritic().to(w.env.device)
        learner.load_state_dict(tt.synthetic(0.29, 1.0)["model"])
        g = torch.Generator(device=w.env.device)
        g.manual_seed(0)
        acts = [torch.randint(0, 3, (n,), dtype=torch.int32, device=w.env.device, generator=g) for _ in range(64)]
        w.reset()
        for r in range(a.rounds):
            for pool in ("mixed", "weak"):
                for mode in ("a_torch", "b_kernel", "c_control"):
                    extra = ""
                    if mode == "a_torch":
                        rate, ms_step, k_ms, k_med = time_torch(w, pool, learner, a.steps, a.warmup)
                    elif mode == "b_kernel":
                        rate, ms_step, k_ms, k_med = time_kernel(w, pool, learner, a.steps, a.warmup)
                        if pool == "weak":
                            macs = (2.0 * tt.MACS_PER_ENV + 1600) * n
                            extra = "  %.1f TFLOP/s fp32" % (2 * macs / (k_ms * 1e-3) / 1e12)
                            if clock:
                                extra += ", %.3f of the fp32 FMA bound (%d SMs x 128 x %.0f MHz)" % (
                                    macs / (sms * 128 * clock) / (k_ms * 1e-3), sms, clock / 1e6)
                    else:
                        rate, ms_step, k_ms, k_med = tt.time_mode(
                            w, "b_per_env_weak" if pool == "weak" else "c_per_env_mix", acts, a.steps, a.warmup)
                    print("round %d %-6s %-10s %8.2f M env-steps/s  %.4f ms/step  timed work %.4f ms "
                          "(median %.4f)%s" % (r + 1, pool, mode, rate / 1e6, ms_step, k_ms, k_med, extra), flush=True)
        print("opponent_stats of the last window:", w.opponent_stats())
        w.env.check()
        torch.cuda.synchronize()
        w.close()
    print(tt.gpu_info(), flush=True)


if __name__ == "__main__":
    main()
