"""The CUDA Pong path against the CPU oracle from designed states (oracle/pong_designed.py), bit for bit, at every
observation kernel the library can pick.

Per case: both simulators get the same injected serves and reset; a zero-buffer class row is written before the first
step (done on sub-step 0 or 1 while both MaxAndSkip buffers are still np.zeros); a few warm-up steps fill the buffers
with real, equal frames; then the score, jump and geometry classes are written in turn into both, each followed by
STEPS_PER_APP steps.  After every step: states, rewards, dones, num_steps, real_reward, observations and the terminal
observations of the finished envs; at the end, episode_stats() against a tally of the oracle's dones.  The oracle is
the reference throughout; the one-thread-per-pixel generic rasteriser is one more path under test (terminal
observations, and renders through the C ABI into buffers that are not 16-byte aligned).

Kernel per configuration (launch_pong_raster): 84x84 stack -> pong_raster_fast_kernel<84, false, true> (incremental)
after the first render into each buffer set, <84, false, false> (whole stacks) with CRL_PONG_FULL_OBS=1; 84x84 ring ->
<84, true, false>; 42x42 stack -> pong_raster_quad_kernel<42> (<42, false, false> with CRL_PONG_NO_QUAD=1); 42x42 ring
-> <42, true, false>."""
import ctypes
import os
import zlib

import numpy as np
import pytest

import pong_designed as D

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

MAX_ROUNDS = 21
WARMUP = 3
STEPS_PER_APP = 4
APPS = ("scores", "jump", "geometry", "scores", "jump")

# (env_id, dim, frame_stack, stack_mode, zero_on_done, n_buffers, N, switch): a pairwise cover of the configuration
# space; N * agents is odd or not a multiple of 4, N * C leaves a partial last quad at 42x42
CASES = [
    ("cPongDouble-v0", 84, 4, "stack", False, 1, 509, None),           # 84 incremental (every render after the first)
    ("cPong-v0", 84, None, "stack", True, 2, 61, None),
    ("cPongDouble-v0", 84, 7, "stack", True, 3, 3, None),
    ("cPong-v0", 84, 5, "stack", False, 1, 4099, None),
    ("cPongDouble-v0", 84, 2, "stack", False, 2, 61, "CRL_PONG_FULL_OBS"),   # 84 whole stacks
    ("cPong-v0", 84, 8, "stack", True, 1, 1, "CRL_PONG_FULL_OBS"),
    ("cPongDouble-v0", 84, 3, "ring", True, 2, 61, None),              # 84 ring
    ("cPong-v0", 84, 5, "ring", False, 2, 509, None),
    ("cPongDouble-v0", 84, 8, "ring", False, 2, 1, None),
    ("cPongDouble-v0", 42, None, "stack", False, 2, 509, None),        # quad: four envs per quad, partial last quad
    ("cPong-v0", 42, 3, "stack", True, 1, 4099, None),                 # quad: stacks straddle quads
    ("cPongDouble-v0", 42, 5, "stack", False, 3, 61, None),
    ("cPongDouble-v0", 42, 7, "stack", True, 1, 3, None),
    ("cPong-v0", 42, 2, "stack", False, 2, 1, None),
    ("cPong-v0", 42, 8, "stack", False, 2, 3, None),
    ("cPongDouble-v0", 42, 6, "stack", True, 2, 61, None),
    ("cPongDouble-v0", 42, 4, "stack", False, 2, 61, "CRL_PONG_NO_QUAD"),   # 42 one frame per warp, plain stacks
    ("cPongDouble-v0", 42, 4, "ring", False, 2, 509, None),            # 42 ring
    ("cPong-v0", 42, 7, "ring", True, 2, 61, None),
    ("cPongDouble-v0", 42, 2, "ring", True, 2, 3, None),
]


def _id(c):
    env, dim, fs, mode, zod, nb, n, sw = c
    return "%s-%d-fs%s-%s%s-nb%d-N%d%s" % ("double" if env == "cPongDouble-v0" else "single", dim, fs, mode,
                                          "-zod" if zod else "", nb, n, "-" + sw[9:].lower() if sw else "")


def _np(o, double):
    return np.stack([x.cpu().numpy() for x in o]) if double else o.cpu().numpy()[None]


def _onp(o, double):
    return np.stack(o) if double else o[None]


def _actions(rng, n, double):
    a = rng.integers(0, 3, (n, 2) if double else (n,)).astype(np.int32)
    if double:
        a[rng.random(a.shape) < 0.15] = 999     # the cheat action on the designed rows
    return a


class Tally(object):
    """episode statistics of the oracle's rollout, in crl_pong_get_stats' fields"""

    def __init__(self):
        self.d = {"episodes": 0, "sum_length": 0, "left_wins": 0, "right_wins": 0, "draws": 0, "sum_margin_biased": 0}

    def add(self, prev_state, done, real, steps):
        for i in np.nonzero(done)[0]:
            left = int(prev_state[i, 6]) + int(real[i] > 0)      # the episode's last point ends it: one per step at most
            right = int(prev_state[i, 7]) + int(real[i] < 0)
            self.d["episodes"] += 1
            self.d["sum_length"] += int(steps[i])
            self.d["left_wins" if left > right else "right_wins" if right > left else "draws"] += 1
            self.d["sum_margin_biased"] += left - right + 64


class Pair(object):
    """the CUDA env and the oracle, stepped with the same actions and compared after every step"""

    def __init__(self, case, atlas, monkeypatch):
        from competitive_rl_b200 import make_envs
        from pong_oracle import PongOracleVec, make_serve_table, set_threads
        env_id, dim, fs, mode, zod, nb, n, switch = case
        self.case, self.n, self.double = case, n, env_id == "cPongDouble-v0"
        self.ring = mode == "ring"
        serves = make_serve_table(n, 24, seed=n + dim)
        set_threads(os.cpu_count() or 1)
        if switch:
            monkeypatch.setenv(switch, "1")      # read when the handle is created
        self.g = make_envs(env_id, num_envs=n, resized_dim=dim, frame_stack=fs, log_dir=None, serves=serves,
                           max_num_rounds=MAX_ROUNDS, stack_mode=mode, zero_on_done=zod, n_buffers=nb)
        if switch:
            monkeypatch.delenv(switch)
        self.o = PongOracleVec(env_id, n, dim, fs, MAX_ROUNDS, atlas, serves)
        self.c, self.zod = fs or 1, zod
        self.tally = Tally()
        self.t = 0

    # zero_on_done (FrameStackTensor): a reset leaves zero frames in all but the newest slot, and steps push them out.
    # The oracle implements FrameStack, so its stacks are compared with their `z` oldest slots zeroed.
    def _mask(self, o, z):
        keep = (np.arange(self.c)[None, :] >= z[:, None]).astype(np.uint8)
        return o * keep[None, :, :, None, None] if self.zod else o

    def reset(self):
        og, oo = self.g.reset(), self.o.reset()
        self.z = np.full(self.n, self.c - 1)
        self.last_oracle_obs = oo
        self._obs(og, oo, "reset")

    def _obs(self, og, oo, what):
        g, o = _np(og, self.double), self._mask(_onp(oo, self.double), self.z)
        assert np.array_equal(g, o), (self.case, what, self.t, int((g != o).sum()))

    def write(self, rows):
        self.g.set_state(rows)          # raises if a row is outside the domain
        self.o.set_state(rows)
        assert np.array_equal(self.g.get_state().cpu().numpy(), self.o.get_state()), (self.case, "set_state")

    def step(self, rng):
        a = _actions(rng, self.n, self.double)
        prev = self.o.get_state()
        oo, ro, do, io = self.o.step(a)
        og, rg, dg, ig = self.g.step(a)
        self.t += 1
        what = (self.case, self.t)
        A = 2 if self.double else 1
        assert np.array_equal(self.g.get_state().cpu().numpy(), self.o.get_state()), what
        assert np.array_equal(rg.cpu().numpy().reshape(self.n, -1)[:, :A], ro.reshape(self.n, -1)[:, :A]), what
        d = dg.cpu().numpy().reshape(self.n, -1)[:, 0]
        assert np.array_equal(d, do), what
        assert np.array_equal(ig.num_steps.cpu().numpy(), io["num_steps"]), what
        real = io["real_reward"].reshape(self.n, -1)
        assert np.array_equal(ig.real_reward.cpu().numpy()[:, :A], real[:, :A]), what
        z_term = np.maximum(self.z - 1, 0)
        self.z = np.where(do, self.c - 1, z_term)
        self.last_oracle_obs = oo
        self._obs(og, oo, "step")
        if do.any():
            idx = np.nonzero(do)[0]
            tg = _np(ig.terminal_observation(), self.double)[:, idx]
            to = self._mask(_onp(io["terminal_observation"], self.double), z_term)[:, idx]
            assert np.array_equal(tg, to), (what, "terminal", int((tg != to).sum()))
        self.tally.add(prev, do, real[:, 0], io["num_steps"])
        return d

    def render_unaligned(self):
        """crl_pong_render_obs into buffers 4 bytes past a 16-byte boundary: the generic rasteriser's path"""
        if self.ring:
            return
        lib = self.g._lib
        nbytes = int(np.prod(self.g._obs[0].shape))
        raw = [torch.zeros(nbytes + 32, dtype=torch.uint8, device="cuda") for _ in range(2)]
        views = []
        for r in raw:
            off = (4 - r.data_ptr() % 16) % 16
            views.append(r[off:off + nbytes])
            assert views[-1].data_ptr() % 16 == 4
        s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        p1 = ctypes.c_void_p(views[1].data_ptr()) if self.double else None
        assert lib.crl_pong_render_obs(self.g._h, ctypes.c_void_p(views[0].data_ptr()), p1, s) == 0, lib.crl_last_error()
        torch.cuda.synchronize()
        shape = tuple(self.g._obs[0].shape)
        g = tuple(v.view(shape) for v in views[:2 if self.double else 1])
        g = np.stack([x.cpu().numpy() for x in g])
        o = self._mask(_onp(self.last_oracle_obs, self.double), self.z)
        assert np.array_equal(g, o), (self.case, self.t, "unaligned", int((g != o).sum()))


def _run_case(case, atlas, monkeypatch):
    from competitive_rl_b200.distributed import STAT_FIELDS
    p = Pair(case, atlas, monkeypatch)
    rng = np.random.default_rng(zlib.crc32(_id(case).encode()))
    p.reset()
    # zero-buffer class: right after construction and reset(), both MaxAndSkip buffers are np.zeros
    p.write(D.zero(rng, p.o.get_state(), MAX_ROUNDS, 0))
    p.step(rng)
    for _ in range(WARMUP):
        p.step(rng)
    for app, kind in enumerate(APPS):
        p.write(D.GENERATORS[kind](rng, p.o.get_state(), MAX_ROUNDS, app))
        for k in range(STEPS_PER_APP):
            p.step(rng)
            if k == 0:
                p.render_unaligned()
    stats = p.g.episode_stats()
    assert {k: stats[k] for k in STAT_FIELDS} == p.tally.d, (case, stats, p.tally.d)
    assert p.tally.d["episodes"] > 0
    p.g.check()
    p.g.close()
    p.o.close()


@pytest.mark.parametrize("case", CASES, ids=[_id(c) for c in CASES])
def test_designed_states_vs_oracle(case, atlas, monkeypatch):
    _run_case(case, atlas, monkeypatch)


def test_out_of_domain_rows_refused(atlas):
    """Rows outside the set_state domain are not applied: set_state raises CrlError, those envs keep their state, the
    rows inside the domain written by the same call are applied, and the next step is bit-exact against the oracle."""
    from competitive_rl_b200 import make_envs
    from competitive_rl_b200._native import CrlError
    from pong_oracle import PongOracleVec, make_serve_table, state_in_domain
    base = np.array([60, 100, 4.0, -2.0, 107, 107, 3, 4, 5, 6], np.float64)
    bad, _ = D.out_of_domain_rows(base, MAX_ROUNDS)
    n = 2 * len(bad)
    serves = make_serve_table(n, 16, seed=2)
    g = make_envs("cPongDouble-v0", num_envs=n, resized_dim=84, frame_stack=4, log_dir=None, serves=serves,
                  max_num_rounds=MAX_ROUNDS)
    o = PongOracleVec("cPongDouble-v0", n, 84, 4, MAX_ROUNDS, atlas, serves)
    g.reset(), o.reset()
    rng = np.random.default_rng(8)
    for _ in range(3):
        a = _actions(rng, n, True)
        g.step(a), o.step(a)
    before = g.get_state().cpu().numpy()
    good = D.geometry(rng, before, MAX_ROUNDS, 0)
    rows = good.copy()
    rows[0::2] = bad                       # even envs: one field outside the domain each; odd envs: designed rows
    assert not state_in_domain(rows[0::2], MAX_ROUNDS).any() and state_in_domain(rows[1::2], MAX_ROUNDS).all()
    with pytest.raises(CrlError, match="set_state domain"):
        g.set_state(rows)
    after = g.get_state().cpu().numpy()
    assert np.array_equal(after[0::2], before[0::2])
    assert np.array_equal(after[1::2], good[1::2])
    g.check()                              # reported once
    want = before.copy()
    want[1::2] = good[1::2]
    o.set_state(want)
    a = _actions(rng, n, True)
    og, rg, dg, _ = g.step(a)
    oo, ro, do, _ = o.step(a)
    assert np.array_equal(g.get_state().cpu().numpy(), o.get_state())
    assert np.array_equal(rg.cpu().numpy(), ro) and np.array_equal(dg.cpu().numpy()[:, 0], do)
    assert np.array_equal(_np(og, True), _onp(oo, True))
    g.check()
    # flags raised together are reported together: an invalid device action, then a refused row
    g.step(torch.full((n, 2), 7, dtype=torch.int32, device="cuda"))
    with pytest.raises(CrlError, match="set_state domain.*action outside"):
        g.set_state(np.concatenate([bad[:1], g.get_state().cpu().numpy()[1:]]))
    g.check()
    g.close()
