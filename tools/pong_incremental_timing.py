"""Render time of the 84x84 stack rasteriser: whole stacks against incremental stacks (crl_pong_set_obs_buffers), into
compressible (crl_obs_alloc, COMP_GENERIC) and ordinary (cudaMalloc) observation memory.

    python tools/pong_incremental_timing.py [--envs 65536] [--steps 1000] [--label NAME]

cPongDouble, random actions (crl_pong_random_actions), 4-frame stacks; CUDA events around every crl_pong_render_obs,
mean over the timed steps.  The build's compile-time switches (CRL_INC_TICKET, CRL_RASTER_NO_DRAIN) are
whatever libcrl_b200.so was built with; --label names the build in the output."""
import argparse
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def run(N, steps, warmup, compressible, full):
    import torch
    from competitive_rl_b200 import _native, make_envs
    lib, ext = _native.load(), _native.ext()
    os.environ.pop("CRL_PONG_FULL_OBS", None)
    if full:
        os.environ["CRL_PONG_FULL_OBS"] = "1"
    envs = make_envs("cPongDouble-v0", seed=1000, log_dir=None, num_envs=N, asynchronous=True, resized_dim=84,
                     frame_stack=4, n_buffers=1)
    os.environ.pop("CRL_PONG_FULL_OBS", None)
    h = envs._h
    bufs = [ext.obs_empty([N, 4, 84, 84], torch.uint8, envs.device.index, compressible) for _ in range(2)]
    obs = [b for b, _ in bufs]
    granted = all(c for _, c in bufs)
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    P = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731
    arr = (ctypes.c_void_p * 1)(obs[0].data_ptr()), (ctypes.c_void_p * 1)(obs[1].data_ptr())
    _native.check(lib.crl_pong_set_obs_buffers(h, arr[0], arr[1], 1, sp))
    _native.check(lib.crl_pong_reset(h, P(obs[0]), P(obs[1]), sp))
    actions = torch.zeros((N, 2), dtype=torch.int32, device=envs.device)
    rew, done, st, real = envs._rew, envs._done, envs._steps, envs._real
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for t in range(warmup + steps):
        _native.check(lib.crl_pong_random_actions(P(actions), 2 * N, 1000, t, sp))
        _native.check(lib.crl_pong_step_state(h, P(actions), P(rew), P(done), P(st), P(real), sp))
        if t >= warmup:
            ev[t - warmup][0].record(stream)
        _native.check(lib.crl_pong_render_obs(h, P(obs[0]), P(obs[1]), sp))
        if t >= warmup:
            ev[t - warmup][1].record(stream)
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    _native.check(lib.crl_pong_set_obs_buffers(h, None, None, 0, sp))
    envs.close()
    del obs, bufs
    torch.cuda.empty_cache()
    return sum(ms) / len(ms), ms[len(ms) // 2], granted


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--label", default="")
    a = ap.parse_args()
    import torch
    name = torch.cuda.get_device_name(0)
    for compressible in (True, False):
        for full in (True, False):
            mean, med, granted = run(a.envs, a.steps, a.warmup, compressible, full)
            print("%-14s %-12s %-11s render %.4f ms (median %.4f)  %s  %d envs x 2 agents" % (
                a.label, "compressible" if compressible else "cudaMalloc", "whole" if full else "incremental", mean, med,
                "granted" if granted == compressible else "NOT granted", a.envs, ) + "  " + name, flush=True)


if __name__ == "__main__":
    main()
