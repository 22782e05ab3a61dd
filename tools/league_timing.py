"""League evaluation rate: every pairing of a pool in one batch (evaluate_pool_in_batch's loop, csrc/pong_opponent.cu
league mode) against the current way, one pairing per batch through torch DevicePolicy networks.

    python tools/league_timing.py [--envs 65536] [--steps 200] [--warmup 20] [--rounds 3]

42x42 cPongDouble, frame_stack None, synthetic LightActorCritic weights saved as checkpoint-{weak,medium}.pkl in a
temporary directory (tournament_timing.synthetic).  Modes, run in alternating rounds in one process:
  (a) league_mix   pool {RULE_BASED, RANDOM, WEAK, MEDIUM}, all 16 ordered pairings: act_pairs + env.step;
  (b) league_nets  pool {WEAK, MEDIUM}, all 4 pairings: both seats of every env are networks;
  (c) two_policies evaluate_two_policies_in_batch with two DevicePolicy networks (WEAK vs MEDIUM), one pairing;
  (d) per_env_weak tools/tournament_timing.py mode (b): cPongTournament, set_opponents with every env on WEAK.
Reported per mode: env-steps/s (host clock over `steps` steps ending in a synchronise) and the time of the opponents'
own work per step from CUDA events (a, b: the act_pairs kernel; c: the two DevicePolicy calls; d: the act kernel).  For
(b), the kernel's fraction of the fp32 FMA bound: 2 x 516 800 MACs per env over (SMs x 128 FMA/clk x max SM clock)."""
import argparse
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)

import tournament_timing as tt  # noqa: E402


class _Stop(Exception):
    pass


def max_sm_clock_hz():
    """clocks.max.sm of GPU 0 from nvidia-smi, in Hz, or None."""
    import subprocess
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout
        return float(out.strip().splitlines()[0]) * 1e6
    except Exception:  # noqa: BLE001
        return None


def time_league(env, opp, pairs, steps, warmup):
    """act_pairs + env.step as evaluate_pool_in_batch runs them, then the kernel alone under CUDA events."""
    import torch
    opp.set_pairs(torch.tensor(pairs, dtype=torch.int32))
    n = env.num_envs
    both = torch.zeros((n, 2), dtype=torch.int32, device=env.device)
    env.reset()
    rew = done = None
    for t in range(warmup + steps):
        if t == warmup:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
        opp.act_pairs(env._obs[0], env._obs[1], rew, done, both, None)
        env.step(both)
        rew, done = env._rew, env._done
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    stream = torch.cuda.current_stream()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    st = opp.pair_stats(len(pairs))
    for t in range(steps):          # no rew / done: the kernel alone, without crediting the last step's episodes again
        ev[t][0].record(stream)
        opp.act_pairs(env._obs[0], env._obs[1], None, None, both, None)
        ev[t][1].record(stream)
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    return n * steps / wall, wall / steps * 1e3, sum(ms) / len(ms), ms[len(ms) // 2], st


def time_two_policies(env, res, steps, warmup):
    """evaluate_two_policies_in_batch itself (WEAK vs MEDIUM DevicePolicy), stopped after warmup + steps steps."""
    import torch
    from competitive_rl_b200.builtin_policies import DevicePolicy
    from competitive_rl_b200.evaluate import evaluate_two_policies_in_batch
    n = env.num_envs
    p0 = DevicePolicy(n, os.path.join(res, "checkpoint-weak.pkl"), True, env.device)
    p1 = DevicePolicy(n, os.path.join(res, "checkpoint-medium.pkl"), True, env.device)
    stream = torch.cuda.current_stream()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    state = {"t": 0, "t0": None}

    def a0(obs):
        t = state["t"]
        if t == warmup:
            torch.cuda.synchronize()
            state["t0"] = time.perf_counter()
        if t == warmup + steps:
            torch.cuda.synchronize()
            state["wall"] = time.perf_counter() - state["t0"]
            raise _Stop()
        if t >= warmup:
            ev[t - warmup][0].record(stream)
        return p0(obs)

    def a1(obs):
        t = state["t"]
        out = p1(obs)
        if t >= warmup:
            ev[t - warmup][1].record(stream)
        state["t"] = t + 1
        return out

    try:
        evaluate_two_policies_in_batch(a0, a1, env, 10 ** 12)
    except _Stop:
        pass
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    wall = state["wall"]
    return n * steps / wall, wall / steps * 1e3, sum(ms) / len(ms), ms[len(ms) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("league_timing needs a CUDA device")
    from competitive_rl_b200 import _native, make_envs
    from competitive_rl_b200.builtin_policies import resolve_pool
    print(tt.gpu_info(), flush=True)
    clock = max_sm_clock_hz()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = a.envs
    ext = _native.ext()
    with tempfile.TemporaryDirectory() as res:
        torch.save(tt.synthetic(0.37, 0.0), os.path.join(res, "checkpoint-weak.pkl"))
        torch.save(tt.synthetic(0.23, 2.0), os.path.join(res, "checkpoint-medium.pkl"))
        env = make_envs("cPongDouble-v0", num_envs=n, resized_dim=42, frame_stack=None, log_dir=None, seed=7)
        opp = ext.PongOpponents(n, int(env.device.index), 1, int(env.first_env))
        _, kinds, images = resolve_pool(["RULE_BASED", "RANDOM", "WEAK", "MEDIUM"], None, res)
        for slot, image in enumerate(images):
            opp.load_net(slot, image)
        opp.set_pool(torch.tensor(kinds, dtype=torch.int32), None)
        mix_pairs = [(x, y) for x in range(4) for y in range(4)]
        net_pairs = [(x, y) for x in (2, 3) for y in (2, 3)]
        w = make_envs("cPongTournament-v0", num_envs=n, resized_dim=42, log_dir=None, seed=7, resource_dir=res)
        g = torch.Generator(device=w.env.device)
        g.manual_seed(0)
        acts = [torch.randint(0, 3, (n,), dtype=torch.int32, device=w.env.device, generator=g) for _ in range(64)]
        w.reset()
        modes = ["a_league_mix", "b_league_nets", "c_two_policies", "d_per_env_weak"]
        for r in range(a.rounds):
            for mode in modes:
                extra = ""
                if mode == "a_league_mix":
                    rate, ms_step, k_ms, k_med, _ = time_league(env, opp, mix_pairs, a.steps, a.warmup)
                elif mode == "b_league_nets":
                    rate, ms_step, k_ms, k_med, st = time_league(env, opp, net_pairs, a.steps, a.warmup)
                    macs = 2.0 * tt.MACS_PER_ENV * n
                    extra = "  %.1f TFLOP/s fp32" % (2 * macs / (k_ms * 1e-3) / 1e12)
                    if clock:
                        extra += ", %.3f of the fp32 FMA bound (%d SMs x 128 x %.0f MHz)" % (
                            macs / (sms * 128 * clock) / (k_ms * 1e-3), sms, clock / 1e6)
                elif mode == "c_two_policies":
                    rate, ms_step, k_ms, k_med = time_two_policies(env, res, a.steps, a.warmup)
                else:
                    rate, ms_step, k_ms, k_med = tt.time_mode(w, "b_per_env_weak", acts, a.steps, a.warmup)
                print("round %d %-15s %8.2f M env-steps/s  %.4f ms/step  opponents %.4f ms (median %.4f)%s" % (
                    r + 1, mode, rate / 1e6, ms_step, k_ms, k_med, extra), flush=True)
        print("league_nets pairing table of the last timed window, (episodes, wins, draws, losses) per pairing of "
              "WEAK / MEDIUM:", st)
        env.check()
        w.env.check()
        torch.cuda.synchronize()
        opp.close()
        env.close()
        w.close()
    print(tt.gpu_info(), flush=True)


if __name__ == "__main__":
    main()
