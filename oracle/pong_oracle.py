"""ctypes front-end of oracle/pong_oracle.c -- TEST INFRASTRUCTURE ONLY.

Importable only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline
legs.  The product package (competitive-rl_b200/) never imports this module.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libpong_oracle.so")
_lib = None


def build(force=False):
    """Compile the C restatement (gcc is in the image). Building the checker is not using it."""
    src = os.path.join(_HERE, "pong_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "libpong_oracle.so"])
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_LIB_PATH)
        c_u8p = ctypes.c_void_p
        L.pong_oracle_create.restype = ctypes.c_void_p
        L.pong_oracle_create.argtypes = [ctypes.c_int] * 6 + [c_u8p, ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64]
        L.pong_oracle_destroy.argtypes = [ctypes.c_void_p]
        L.pong_oracle_reset.argtypes = [ctypes.c_void_p, c_u8p]
        L.pong_oracle_step.argtypes = [ctypes.c_void_p] + [ctypes.c_void_p] * 7
        L.pong_oracle_get_state.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.pong_oracle_render_raw.argtypes = [ctypes.c_void_p, ctypes.c_int, c_u8p, c_u8p]
        L.pong_oracle_warp.argtypes = [c_u8p, ctypes.c_int, c_u8p]
        L.pong_oracle_resize_area.argtypes = [c_u8p, ctypes.c_int, ctypes.c_int, c_u8p, ctypes.c_int, ctypes.c_int]
        L.pong_oracle_set_threads.argtypes = [ctypes.c_int]
        L.pong_oracle_serve_overrun.argtypes = [ctypes.c_void_p]
        L.pong_oracle_serve_overrun.restype = ctypes.c_int
        L.pong_oracle_game_ptr.restype = ctypes.POINTER(Game)
        L.pong_oracle_game_ptr.argtypes = [ctypes.c_void_p, ctypes.c_int]
        _lib = L
    return _lib


class Game(ctypes.Structure):
    """pong_oracle.c's Game: one env's PongGame fields (pong_oracle_game_ptr)."""
    _fields_ = [("ball_x", ctypes.c_int), ("ball_y", ctypes.c_int), ("vx", ctypes.c_double),
                ("vy", ctypes.c_double), ("left_y", ctypes.c_int), ("right_y", ctypes.c_int),
                ("left_move", ctypes.c_int), ("right_move", ctypes.c_int), ("score_left", ctypes.c_int),
                ("score_right", ctypes.c_int), ("num_rounds", ctypes.c_int), ("num_steps", ctypes.c_int)]


# get_state() column -> Game field; vx / vy (columns 2, 3) are the float fields
STATE_FIELDS = ("ball_x", "ball_y", "vx", "vy", "left_y", "right_y", "score_left", "score_right", "num_rounds", "num_steps")


def state_in_domain(state, max_rounds=21):
    """(N,) bool: the rows of an (N, 10) get_state()-layout array inside the set_state domain of include/crl_b200.h
    (ball_x 0..156, ball_y 0..190, bats 0..255, finite |vx|, |vy| <= 64, scores 0..21, num_rounds 0..max_rounds-1,
    num_steps 0..10000, integer fields integral)."""
    s = np.asarray(state, np.float64).reshape(-1, 10)
    with np.errstate(invalid="ignore"):
        ok = (np.abs(s[:, 2]) <= 64) & (np.abs(s[:, 3]) <= 64)
        for col, hi in ((0, 156), (1, 190), (4, 255), (5, 255), (6, 21), (7, 21), (8, max_rounds - 1), (9, 10000)):
            v = s[:, col]
            ok &= (v >= 0) & (v <= hi) & (v == np.trunc(v))
    return ok


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def set_threads(n):
    lib().pong_oracle_set_threads(int(n))


def warp(rgb, dim):
    """cv2.cvtColor(RGB2GRAY) + cv2.resize(INTER_AREA) restated, one 210x160x3 frame."""
    rgb = np.ascontiguousarray(rgb, np.uint8)
    assert rgb.shape == (210, 160, 3)
    out = np.empty((dim, dim), np.uint8)
    lib().pong_oracle_warp(_p(rgb), dim, _p(out))
    return out


def resize_area(gray, dw, dh):
    gray = np.ascontiguousarray(gray, np.uint8)
    sh, sw = gray.shape
    out = np.empty((dh, dw), np.uint8)
    lib().pong_oracle_resize_area(_p(gray), sw, sh, _p(out), dw, dh)
    return out


class PongOracleVec(object):
    """Mirrors the reference vec-env protocol for cPong-v0 / cPongDouble-v0:
    reset() -> obs; step(actions) -> (obs, rew, done, info-arrays).

    obs: tuple of per-agent (N, C, D, D) uint8 for Double, one array for single.
    """

    def __init__(self, env_id="cPongDouble-v0", num_envs=1, resized_dim=84, frame_stack=None, max_rounds=21,
                 atlas=None, serves=None, render=True, seed=0):
        assert env_id in ("cPong-v0", "cPongDouble-v0")
        self.double = env_id == "cPongDouble-v0"
        self.n, self.dim = int(num_envs), int(resized_dim)
        self.c = int(frame_stack) if frame_stack else 1
        self.n_agents = 2 if self.double else 1
        self.render = bool(render)
        self._atlas = None if atlas is None else np.ascontiguousarray(atlas, np.uint8)
        if self._atlas is not None:
            assert self._atlas.shape == (22, 22, 34, 160, 3), self._atlas.shape
        self._serves = None if serves is None else np.ascontiguousarray(serves, np.float64)
        K = 0
        if self._serves is not None:
            assert self._serves.ndim == 3 and self._serves.shape[0] == self.n and self._serves.shape[2] == 2
            K = self._serves.shape[1]
        self._h = lib().pong_oracle_create(self.n, int(self.double), self.dim, int(frame_stack or 0), int(max_rounds),
                                           int(self.render), _p(self._atlas), _p(self._serves), K, int(seed))
        self._obs = np.zeros((self.n_agents, self.n, self.c, self.dim, self.dim), np.uint8)
        self._term = np.zeros_like(self._obs)
        self._rew = np.zeros((self.n, 2), np.float32)
        self._real = np.zeros((self.n, 2), np.float32)
        self._done = np.zeros((self.n,), np.uint8)
        self._steps = np.zeros((self.n,), np.int32)

    def close(self):
        if self._h:
            lib().pong_oracle_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _fmt_obs(self, arr):
        if self.double:
            return (arr[0].copy(), arr[1].copy())
        return arr[0].copy()

    def reset(self):
        lib().pong_oracle_reset(self._h, _p(self._obs) if self.render else None)
        return self._fmt_obs(self._obs) if self.render else None

    def step(self, actions):
        a = np.ascontiguousarray(actions, np.int32)
        assert a.shape == ((self.n, 2) if self.double else (self.n,)), a.shape
        lib().pong_oracle_step(self._h, _p(a), _p(self._obs) if self.render else None, _p(self._rew), _p(self._done),
                               _p(self._steps), _p(self._real), _p(self._term) if self.render else None)
        if lib().pong_oracle_serve_overrun(self._h):
            raise RuntimeError("serve table exhausted")
        rew = self._rew.copy() if self.double else self._rew[:, 0].copy()
        real = self._real.copy() if self.double else self._real[:, 0].copy()
        info = {"num_steps": self._steps.copy(), "real_reward": real,
                "terminal_observation": self._fmt_obs(self._term) if self.render else None}
        return (self._fmt_obs(self._obs) if self.render else None), rew, self._done.astype(bool), info

    def get_state(self):
        """(N, 10) float64: ball_x, ball_y, vx, vy, left_y, right_y, score_l, score_r, rounds, steps."""
        s = np.zeros((self.n, 10), np.float64)
        lib().pong_oracle_get_state(self._h, _p(s))
        return s

    def set_state(self, state):
        """Write (N, 10) game states in get_state()'s layout, as crl_pong_set_state does on the GPU: integer fields take
        the C (int) truncation, vx / vy are stored as given; Bat._current_move, the serve counter, ClipRewardEnv's step
        count, the MaxAndSkip buffers and the FrameStack deque keep what they held.  No domain check: the caller keeps
        the rows inside state_in_domain()."""
        s = np.asarray(state, np.float64).reshape(self.n, 10)
        for i in range(self.n):
            g = lib().pong_oracle_game_ptr(self._h, i).contents
            for k, name in enumerate(STATE_FIELDS):
                setattr(g, name, float(s[i, k]) if k in (2, 3) else int(s[i, k]))

    def render_raw(self, i):
        f0 = np.empty((210, 160, 3), np.uint8)
        f1 = np.empty((210, 160, 3), np.uint8)
        lib().pong_oracle_render_raw(self._h, int(i), _p(f0), _p(f1))
        return f0, f1


def make_serve_table(num_envs, K, seed=0, first_env=0):
    """serves[env, k] = (vx, vy) drawn with random.Random(seed*1000003 + global_env) in the reference's
    draw order (uniform, choice, choice) -- Ball.reset, pong/base_pong_env.py:314-320."""
    import random
    out = np.zeros((num_envs, K, 2), np.float64)
    for e in range(num_envs):
        r = random.Random(seed * 1000003 + first_env + e)
        for k in range(K):
            vy0 = r.uniform(4 * 0.3, 4)
            vx = r.choice([-4.0, 4.0])
            vy = r.choice([-vy0, vy0])
            out[e, k] = (vx, vy)
    return out
