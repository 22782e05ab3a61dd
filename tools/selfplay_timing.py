"""Self-play rollout step rate on cPongDouble-v0: a torch learner for both agents against the learner in the opponents'
kernel (SelfPlayEnvWrapper.learner_step, csrc/pong_opponent.cu self-play mode).

    python tools/selfplay_timing.py [--envs 65536] [--steps 200] [--warmup 20] [--rounds 3]

42x42, frame_stack None, synthetic LightActorCritic weights (tournament_timing.synthetic) for WEAK, MEDIUM and the
learner.  Modes, run in alternating rounds in one process:
  (a) torch     both agents' frames stacked in torch (float32, FrameStackTensor zeroing on done), a torch
                LightActorCritic with default torch settings (cuDNN may use TF32) on the 2N stacks, Categorical sampling
                and log-prob, then env.step;
  (b) self      learner_step() with every env on (LEARNER, LEARNER);
  (c) mixed     learner_step() with the pairings (L, L), (L, WEAK), (MEDIUM, L), (L, RULE_BASED);
  (d) control   league mode: act_pairs with WEAK / MEDIUM in both seats (all 4 pairings) + env.step, as
                tools/league_timing.py mode (b).
Reported per mode: env-steps/s (host clock over `steps` steps ending in a synchronise) and, from CUDA events in a
separate window, the work before the env step (a: stacking + network + sampling; b, c: the act_selfplay kernel; d: the
act_pairs kernel).  For (b), (c) and (d), the kernel's fraction of the fp32 FMA bound: the MACs per env (516 800 per
network seat, 1 600 more for a learner's critic) over (SMs x 128 FMA/clk x max SM clock)."""
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

TABLES = {"b_self": [("LEARNER", "LEARNER")],
          "c_mixed": [("LEARNER", "LEARNER"), ("LEARNER", "WEAK"), ("MEDIUM", "LEARNER"), ("LEARNER", "RULE_BASED")]}


def macs_per_env(table):
    """Mean MACs per env of a table whose pairings are played by equally many envs."""
    seat = {"LEARNER": tt.MACS_PER_ENV + 1600, "RULE_BASED": 0, "RANDOM": 0}
    return sum(seat.get(x, tt.MACS_PER_ENV) for pr in table for x in pr) / len(table)


def events(steps):
    import torch
    return [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]


def summary(ev):
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    return sum(ms) / len(ms), ms[len(ms) // 2]


def timed(one, kernel, steps, warmup):
    """(env-steps/s, ms per step) of `one` over `steps` steps, then (mean, median) ms of `kernel` under CUDA events."""
    import torch
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
        kernel()
        ev[t][1].record(stream)
    torch.cuda.synchronize()
    return (steps / wall, wall / steps * 1e3) + summary(ev)


def time_torch(env, learner, steps, warmup):
    """(a): both agents' stacks and the learner in torch, then env.step."""
    import torch
    from torch.distributions import Categorical
    n, dev = env.num_envs, env.device
    stack = torch.zeros((2 * n, 4, 42, 42), dtype=torch.float32, device=dev)
    env.reset()
    state = {"done": None}

    def act():
        if state["done"] is not None:
            stack[state["done"].repeat(2)] = 0
        stack[:, :-1] = stack[:, 1:].clone()
        stack[:, -1] = torch.cat([env._obs[0], env._obs[1]]).reshape(2 * n, 42, 42)
        with torch.no_grad():
            logits, value = learner(stack)
            dist = Categorical(logits=logits)
            a = dist.sample()
            dist.log_prob(a)
        return a.reshape(2, n).t().to(torch.int32).contiguous()

    def one():
        env.step(act())
        state["done"] = env._done

    return timed(one, act, steps, warmup)


def time_selfplay(w, table, steps, warmup):
    """(b), (c): learner_step(), then the act_selfplay kernel alone."""
    import torch
    w.set_league(table, seed=1)
    w.reset()
    env, n = w.env, w.num_envs
    both = torch.empty((n, 2), dtype=torch.int32, device=env.device)
    lpv = torch.empty((n, 2, 2), dtype=torch.float32, device=env.device)
    out = torch.empty((n, 2, 4, 42, 42), dtype=torch.uint8, device=env.device)

    def kernel():   # no rew / done: the kernel alone, without crediting the last step's episodes again
        w._opp.act_selfplay(env._obs[0], env._obs[1], None, None, True, both, lpv, None, out)

    return timed(lambda: w.learner_step(out), kernel, steps, warmup)


def time_league(env, opp, pairs, steps, warmup):
    """(d): act_pairs + env.step as evaluate_pool_in_batch runs them, then the act_pairs kernel alone."""
    import torch
    opp.set_pairs(torch.tensor(pairs, dtype=torch.int32))
    both = torch.zeros((env.num_envs, 2), dtype=torch.int32, device=env.device)
    env.reset()
    state = {"rew": None, "done": None}

    def one():
        opp.act_pairs(env._obs[0], env._obs[1], state["rew"], state["done"], both, None)
        env.step(both)
        state["rew"], state["done"] = env._rew, env._done

    return timed(one, lambda: opp.act_pairs(env._obs[0], env._obs[1], None, None, both, None), steps, warmup)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("selfplay_timing needs a CUDA device")
    from competitive_rl_b200 import _native, make_envs
    from competitive_rl_b200.builtin_policies import LightActorCritic, resolve_pool
    from competitive_rl_b200.selfplay import SelfPlayEnvWrapper
    print(tt.gpu_info(), flush=True)
    clock = lt.max_sm_clock_hz()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = a.envs
    with tempfile.TemporaryDirectory() as res:
        torch.save(tt.synthetic(0.37, 0.0), os.path.join(res, "checkpoint-weak.pkl"))
        torch.save(tt.synthetic(0.23, 2.0), os.path.join(res, "checkpoint-medium.pkl"))
        env = make_envs("cPongDouble-v0", num_envs=n, resized_dim=42, frame_stack=None, log_dir=None, seed=7)
        w = SelfPlayEnvWrapper(env, resource_dir=res)
        learner = LightActorCritic().to(env.device)
        learner.load_state_dict(tt.synthetic(0.29, 1.0)["model"])
        w.set_league(TABLES["b_self"])
        w.set_learner(learner)
        opp = _native.ext().PongOpponents(n, int(env.device.index), 1, int(env.first_env))
        _, kinds, images = resolve_pool(["WEAK", "MEDIUM"], None, res)
        for slot, image in enumerate(images):
            opp.load_net(slot, image)
        opp.set_pool(torch.tensor(kinds, dtype=torch.int32), None)
        net_pairs = [(x, y) for x in (0, 1) for y in (0, 1)]
        for r in range(a.rounds):
            for mode in ("a_torch", "b_self", "c_mixed", "d_control"):
                if mode == "a_torch":
                    rate, ms_step, k_ms, k_med = time_torch(env, learner, a.steps, a.warmup)
                    macs = None
                elif mode == "d_control":
                    rate, ms_step, k_ms, k_med = time_league(env, opp, net_pairs, a.steps, a.warmup)
                    macs = 2.0 * tt.MACS_PER_ENV
                else:
                    rate, ms_step, k_ms, k_med = time_selfplay(w, TABLES[mode], a.steps, a.warmup)
                    macs = macs_per_env(TABLES[mode])
                extra = ""
                if macs is not None:
                    extra = "  %.0f MACs/env, %.1f TFLOP/s fp32" % (macs, 2 * macs * n / (k_ms * 1e-3) / 1e12)
                    if clock:
                        extra += ", %.3f of the fp32 FMA bound (%d SMs x 128 x %.0f MHz)" % (
                            macs * n / (sms * 128 * clock) / (k_ms * 1e-3), sms, clock / 1e6)
                print("round %d %-10s %8.2f M env-steps/s  %.4f ms/step  timed work %.4f ms (median %.4f)%s" % (
                    r + 1, mode, rate * n / 1e6, ms_step, k_ms, k_med, extra), flush=True)
        print("pair_stats of the last c_mixed window:", w.pair_stats())
        env.check()
        torch.cuda.synchronize()
        opp.close()
        w.close()
    print(tt.gpu_info(), flush=True)


if __name__ == "__main__":
    main()
