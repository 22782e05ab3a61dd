"""Incremental 84x84 observation stacks (crl_pong_set_obs_buffers): a render into a registered buffer set stores only
the chunks whose frames changed.  Every case runs the same seeded rollout on two handles, one with CRL_PONG_FULL_OBS=1
(whole stacks every render), and compares the observations byte for byte after every step."""
import ctypes
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

N, DIM, C = 256, 84, 4


def _make(env_id, full, **kw):
    from competitive_rl_b200 import make_envs
    old = os.environ.pop("CRL_PONG_FULL_OBS", None)
    if full:
        os.environ["CRL_PONG_FULL_OBS"] = "1"
    try:
        return make_envs(env_id, num_envs=N, resized_dim=DIM, frame_stack=C, log_dir=None, seed=11, asynchronous=True,
                         max_num_rounds=2, **kw)
    finally:
        os.environ.pop("CRL_PONG_FULL_OBS", None)
        if old is not None:
            os.environ["CRL_PONG_FULL_OBS"] = old


def _pair(env_id, **kw):
    return _make(env_id, False, **kw), _make(env_id, True, **kw)


def _np(obs):
    return [o.cpu().numpy() for o in (obs if isinstance(obs, tuple) else (obs,))]


def _same(a, b, what):
    for k, (x, y) in enumerate(zip(_np(a), _np(b))):
        assert np.array_equal(x, y), (what, k, int((x != y).sum()))


def _actions(rng, env_id):
    return rng.integers(0, 3, (N, 2) if env_id == "cPongDouble-v0" else (N,)).astype(np.int32)


def _random_state(env, rng):
    st = env.get_state().cpu().numpy()
    st[:, 0] = rng.integers(0, 157, N)
    st[:, 1] = rng.integers(30, 191, N)
    st[:, 4] = rng.integers(34, 180, N)
    st[:, 5] = rng.integers(34, 180, N)
    st[:, 6] = rng.integers(0, 2, N)
    st[:, 7] = rng.integers(0, 2, N)
    return st


@pytest.mark.parametrize("env_id", ["cPong-v0", "cPongDouble-v0"])
@pytest.mark.parametrize("zero_on_done", [False, True])
@pytest.mark.parametrize("n_buffers", [1, 2, 3])
def test_incremental_equals_full(env_id, zero_on_done, n_buffers):
    inc, full = _pair(env_id, zero_on_done=zero_on_done, n_buffers=n_buffers)
    _same(inc.reset(), full.reset(), "reset")
    rng = np.random.default_rng(3)
    done_seen = 0
    for t in range(160):
        if t == 70:      # reset in mid-run
            _same(inc.reset(), full.reset(), ("reset", t))
            continue
        if t == 110:     # new game states (hist keeps its frames; the next step's frame comes from them)
            st = _random_state(inc, rng)
            inc.set_state(st)
            full.set_state(st)
        a = _actions(rng, env_id)
        oi, _, di, _ = inc.step(a)
        of, _, df, _ = full.step(a)
        _same(oi, of, t)
        done_seen += int(di.sum())
    assert done_seen > 0          # max_num_rounds=2: resets and score changes happen inside the run
    inc.close()
    full.close()


def test_render_into_foreign_buffers_between_steps():
    from competitive_rl_b200 import _native
    lib = _native.load()
    inc, full = _pair("cPongDouble-v0", n_buffers=1)
    inc.reset(), full.reset()
    rng = np.random.default_rng(5)
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for t in range(60):
        a = _actions(rng, "cPongDouble-v0")
        oi, _, _, _ = inc.step(a)
        of, _, _, _ = full.step(a)
        _same(oi, of, t)
        if t % 7 == 3:   # an unregistered pair of buffers: rendered whole, the registered set stays valid
            foreign = [torch.zeros_like(o) for o in oi]
            assert lib.crl_pong_render_obs(inc._h, ctypes.c_void_p(foreign[0].data_ptr()),
                                           ctypes.c_void_p(foreign[1].data_ptr()), s) == 0, lib.crl_last_error()
            _same(tuple(foreign), of, ("foreign", t))
    inc.close()
    full.close()


def test_step_host():
    from competitive_rl_b200 import _native
    lib = _native.load()
    inc, full = _pair("cPongDouble-v0", n_buffers=1)
    inc.reset(), full.reset()
    rng = np.random.default_rng(6)
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731
    h_rew = torch.zeros((N, 2), dtype=torch.float32)
    h_done = torch.zeros((N,), dtype=torch.uint8)
    for t in range(80):
        h_act = torch.from_numpy(_actions(rng, "cPongDouble-v0"))
        for env in (inc, full):
            o0, o1 = env._obs
            assert lib.crl_pong_step_host(env._h, p(h_act), p(o0), p(o1), None, None, p(h_rew), p(h_done), None, None,
                                          s) == 0, lib.crl_last_error()
        _same(tuple(inc._obs), tuple(full._obs), t)
    inc.close()
    full.close()


def test_external_write_survives_until_forget_obs():
    """A template-only chunk (the bottom row, below the arena) is never stored by an incremental render: a byte written
    there by the caller survives a step, and forget_obs() makes the next render rewrite the buffer whole."""
    inc, full = _pair("cPongDouble-v0", n_buffers=1)
    inc.reset(), full.reset()
    rng = np.random.default_rng(7)
    for t in range(5):
        a = _actions(rng, "cPongDouble-v0")
        inc.step(a)
        full.step(a)
    for env in (inc, full):
        env._obs[0][:, :, DIM - 1, 40] = 123
    torch.cuda.synchronize()
    a = _actions(rng, "cPongDouble-v0")
    oi, _, _, _ = inc.step(a)
    of, _, _, _ = full.step(a)
    ref = of[0][:, :, DIM - 1, 40].cpu()
    assert (ref != 123).all()
    assert (oi[0][:, :, DIM - 1, 40].cpu() == 123).all()          # really incremental: the chunk was not stored
    oi[0][:, :, DIM - 1, 40] = ref.cuda()
    _same(oi, of, "restored")
    oi[0][:, :, DIM - 1, 40] = 123
    oi[1][:, :, 50, 50] = 7
    inc.forget_obs()
    a = _actions(rng, "cPongDouble-v0")
    oi, _, _, _ = inc.step(a)
    of, _, _, _ = full.step(a)
    _same(oi, of, "after forget_obs")
    inc.close()
    full.close()


def test_set_obs_buffers_arguments():
    from competitive_rl_b200 import _native
    lib = _native.load()
    env = _make("cPongDouble-v0", False, n_buffers=1)
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    o0, o1 = env._obs
    arr = lambda *ts: (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])   # noqa: E731
    assert lib.crl_pong_set_obs_buffers(env._h, arr(o0), arr(o0), 1, s) == _native.CRL_E_INVALID   # same buffer twice
    assert lib.crl_pong_set_obs_buffers(env._h, arr(o0), None, 1, s) == _native.CRL_E_INVALID      # Double needs obs1
    assert lib.crl_pong_set_obs_buffers(env._h, arr(o0), arr(o1), 1, s) == 0
    assert lib.crl_pong_set_obs_buffers(env._h, None, None, 0, s) == 0
    env.close()
    ring = _make("cPongDouble-v0", False, stack_mode="ring")
    r0, r1 = ring._ring
    assert lib.crl_pong_set_obs_buffers(ring._h, arr(r0), arr(r1), 1, s) == _native.CRL_E_STATE
    ring.close()
