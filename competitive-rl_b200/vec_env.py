"""Vec-env front end of the CUDA Pong simulator.

Mirrors the protocol of the reference's `VecEnv` (competitive_rl/utils/base_vec_env.py:63-252)
as implemented by `DummyVecEnv` (utils/dummy_vec_env.py:27-133) and `SubprocVecEnv`
(utils/subproc_vec_env.py:81-186) for the env ids `cPong-v0` / `cPongDouble-v0`, whose
per-env wrapper stack is `make_env_a2c_atari` (utils/atari_wrappers.py:40-53).

Differences a caller sees (all deliberate, see DESIGN.md):
  * observations / rewards / dones are torch CUDA tensors (pass `return_numpy=True` for
    host numpy arrays with exactly the reference's shapes and dtypes);
  * `infos` is a lazy sequence: `infos[i]` builds the reference's dict
    (`real_reward`, `num_steps`, `terminal_observation`) on demand;
  * cPongDouble accepts `frame_stack` (per-agent FrameStack; the reference asserts
    `frame_stack is None` because its FrameStack cannot stack tuples, make_envs.py:105-106).
"""
import ctypes
from abc import ABC, abstractmethod

import numpy as np
import torch

from . import _native
from . import spaces

CHEAT_CODES = 999  # pong/base_pong_env.py:9


def tile_images(img_nhwc):
    """Same contract as utils/base_vec_env.py:10-38: tile N images into one PxQ image."""
    img_nhwc = np.asarray(img_nhwc)
    n, h, w, c = img_nhwc.shape
    rows = int(np.ceil(np.sqrt(n)))
    cols = int(np.ceil(float(n) / rows))
    pad = np.zeros((rows * cols - n, h, w, c), img_nhwc.dtype)
    grid = np.concatenate([img_nhwc, pad]).reshape(rows, cols, h, w, c).transpose(0, 2, 1, 3, 4)
    return grid.reshape(rows * h, cols * w, c)


class AlreadySteppingError(Exception):
    def __init__(self):
        Exception.__init__(self, "already running an async step")


class NotSteppingError(Exception):
    def __init__(self):
        Exception.__init__(self, "not running an async step")


class VecEnv(ABC):
    """Abstract vectorised environment: same surface as utils/base_vec_env.py:63-252."""
    metadata = {"render.modes": ["human", "rgb_array"]}

    def __init__(self, num_envs, observation_space, action_space):
        self.num_envs = num_envs
        self.observation_space = observation_space
        self.action_space = action_space

    @abstractmethod
    def reset(self):
        pass

    @abstractmethod
    def step_async(self, actions):
        pass

    @abstractmethod
    def step_wait(self):
        pass

    @abstractmethod
    def close(self):
        pass

    @abstractmethod
    def get_attr(self, attr_name, indices=None):
        pass

    @abstractmethod
    def set_attr(self, attr_name, value, indices=None):
        pass

    @abstractmethod
    def env_method(self, method_name, *method_args, indices=None, **method_kwargs):
        pass

    @abstractmethod
    def seed(self, seed=None):
        pass

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def get_images(self, *args, **kwargs):
        raise NotImplementedError

    def render(self, mode="human", *args, **kwargs):
        try:
            imgs = self.get_images(*args, **kwargs)
        except NotImplementedError:
            return None
        big = tile_images(imgs)
        if mode == "human":
            import cv2
            cv2.imshow("vecenv", big[:, :, ::-1])
            cv2.waitKey(1)
        elif mode == "rgb_array":
            return big
        else:
            raise NotImplementedError

    @property
    def unwrapped(self):
        return self

    def _get_indices(self, indices):
        if indices is None:
            indices = range(self.num_envs)
        elif isinstance(indices, int):
            indices = [indices]
        return indices


class LazyInfos(object):
    """Sequence of per-env info dicts (`real_reward`, `num_steps`, and for finished
    episodes `terminal_observation`), materialised on access.  The vectorised fields are
    available without any host sync as `.num_steps`, `.real_reward`, `.done` (device tensors)."""

    def __init__(self, env, num_steps, real_reward, done):
        self._env = env
        self.num_steps, self.real_reward, self.done = num_steps, real_reward, done
        self._host = None
        self._term = None

    def __len__(self):
        return self._env.num_envs

    def _sync(self):
        if self._host is None:
            self._host = (self.num_steps.cpu().numpy(), self.real_reward.cpu().numpy(), self.done.cpu().numpy())
        return self._host

    def terminal_observation(self):
        """Device tensor(s) holding terminal observations in the rows where done is set."""
        if self._term is None:
            self._term = self._env._terminal_obs(self.done)
        return self._term

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        steps, real, done = self._sync()
        env = self._env
        rr = [float(real[i, 0]), float(real[i, 1])] if env.n_agents == 2 else float(real[i, 0])
        info = {"real_reward": rr, "num_steps": int(steps[i])}
        if done[i]:
            t = self.terminal_observation()
            if env.n_agents == 2:
                t = tuple(x[i] for x in t)
            else:
                t = t[i]
            info["terminal_observation"] = env._to_numpy(t) if env.return_numpy else t
        return info

    def __iter__(self):
        for i in range(len(self)):
            yield self[i]

    def copy(self):
        return self


class _EnvView(object):
    """`envs.envs[i]` of DummyVecEnv (used by vis.py:28-29, test/test_pong.py:13):
    a handle on one env of the batch."""

    def __init__(self, vec, index):
        self._vec, self._index = vec, index
        self.observation_space = vec.observation_space
        self.action_space = vec.action_space
        self.metadata = vec.metadata

    @property
    def unwrapped(self):
        return self

    def render(self, mode="rgb_array", **kwargs):
        img = self._vec.get_images(indices=[self._index])[0]
        if mode == "rgb_array":
            return img
        import cv2
        cv2.imshow("env%d" % self._index, img[:, :, ::-1])
        cv2.waitKey(1)

    def seed(self, seed=None):
        return None

    def close(self):
        pass


class CudaPongVecEnv(VecEnv):
    """cPong-v0 / cPongDouble-v0 batch on one GPU.

    reset() -> obs;  step(actions) -> (obs, rew, done, infos), auto-reset on done exactly
    like DummyVecEnv.step_wait (utils/dummy_vec_env.py:51-63).

    obs:   Double: tuple of two uint8 (N, C, D, D); single: one uint8 (N, C, D, D)
    rew:   `asynchronous=False` (DummyVecEnv convention): float32 (N, A);
           `asynchronous=True`  (SubprocVecEnv convention): (N, 2) for Double, (N,) for single
    done:  Dummy convention: bool (N, A); Subproc convention: bool (N,)
    actions: Double: int (N, 2) in {0, 1, 2, 999}; single: int (N,) in {0, 1, 2}.  An int32 CUDA tensor is consumed
             in place (no copy, no host sync).

    BUFFER LIFETIME (differs from the reference, which returns fresh numpy copies every step): the tensors returned by
    reset()/step() are owned by the env and rotate over `n_buffers` sets, so what step t returned is overwritten by
    step t + n_buffers.  Keep rollouts alive with a larger `n_buffers`, or pass `copy=True` to get fresh tensors from
    every call (one extra device copy of the observations per step).

    Do not write into the returned observation tensors.  At 84x84 with stack_mode="stack" and uint8 observations the
    buffer sets are registered with the library (crl_pong_set_obs_buffers), which then stores only the 16-byte chunks of
    each stack whose frames changed since that buffer was last rendered.  A caller that
    modifies a returned tensor in place must use `copy=True`, or call `forget_obs()` afterwards so that the next render
    into each buffer rewrites it whole.

    stack_mode="ring" (opt-in): the observations are strided VIEWS `ring[:, k+1 : k+1+C]` of an (N, 2C, D, D) ring per
    agent in which every new frame is stored twice (slots k and k + C), so a step writes 2 frames per agent instead of
    C -- same values, half the HBM traffic (SURVEY.md 8(d): 28 224 B instead of 56 448 B per env-step at 84x84x4).  The
    view returned by step t is valid until step t + 1 only (its oldest slot is the next one overwritten).

    obs_dtype="float32": the observations a STOCK gym install of the reference produces (gym's Box defaults to float32,
    SURVEY.md F7): unrounded fp32 area sums, rounded integers only in frames that came from reset().  A plain
    one-thread-per-pixel rasteriser, 4x the bytes: for parity with such an install, not for throughput.

    zero_on_done=True: FrameStackTensor's stacking (utils/utils.py:145-173) instead of FrameStack's: after a done the
    history is zeros and only the newest channel holds the reset observation.
    """

    def __init__(self, env_id="cPongDouble-v0", num_envs=1, resized_dim=42, frame_stack=None, seed=0,
                 asynchronous=False, device=None, max_num_rounds=21, atlas=None, serves=None, first_env=0,
                 return_numpy=False, n_buffers=2, stack_mode="stack", zero_on_done=False, copy=False, obs_dtype="uint8"):
        if env_id not in ("cPong-v0", "cPongDouble-v0"):
            raise ValueError("unsupported env id %r" % (env_id,))
        if stack_mode not in ("stack", "ring"):
            raise ValueError("stack_mode must be 'stack' or 'ring'")
        if obs_dtype not in ("uint8", "float32"):
            raise ValueError("obs_dtype must be 'uint8' or 'float32'")
        self.f32 = obs_dtype == "float32"
        if self.f32 and stack_mode == "ring":
            raise ValueError("obs_dtype='float32' needs stack_mode='stack'")
        if not torch.cuda.is_available():
            raise RuntimeError("CudaPongVecEnv needs a CUDA device: this simulator has no CPU path")
        ext = _native.ext()
        self._lib = _native.load()          # the plain C ABI, for callers that drive it directly (bench.py, tests)
        self.env_id = env_id
        self.n_agents = 2 if env_id == "cPongDouble-v0" else 1
        self.dim = int(resized_dim)
        self.c = int(frame_stack) if frame_stack else 1
        self.asynchronous = bool(asynchronous)
        self.return_numpy = bool(return_numpy)
        self.copy = bool(copy)
        self.stack_mode = stack_mode
        self.ring = stack_mode == "ring"
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        n = int(num_envs)
        box = spaces.Box(0, 255, (self.c, self.dim, self.dim), dtype=np.float32 if self.f32 else np.uint8)
        if self.n_agents == 2:
            obs_space = spaces.Tuple([box, box])
            act_space = spaces.Tuple([spaces.Discrete(3), spaces.Discrete(3)])
        else:
            obs_space, act_space = box, spaces.Discrete(3)
        VecEnv.__init__(self, n, obs_space, act_space)
        self.metadata = {"render.modes": ["human", "rgb_array"]}

        self._impl = ext.Pong(n, self.n_agents, self.dim, int(frame_stack or 0), int(max_num_rounds), int(self.device.index),
                              1 if self.ring else 0, bool(zero_on_done), int(seed) & (2 ** 64 - 1), int(first_env))
        self._h = ctypes.c_void_p(self._impl.raw_handle())
        if atlas is None:
            atlas = np.load(_native.DEFAULT_ATLAS)["strips"]
        atlas = np.ascontiguousarray(atlas, np.uint8)
        if atlas.shape != _native.ATLAS_SHAPE:
            raise ValueError("atlas must have shape %r" % (_native.ATLAS_SHAPE,))
        self._impl.load_atlas(torch.from_numpy(atlas))
        if serves is not None:
            self.inject_serves(serves)

        dev = self.device
        shape = (n, self.c, self.dim, self.dim)
        # Observation stacks and rings live in compressible memory where the device grants it (crl_obs_alloc): the frames
        # are mostly constant runs, so the rasteriser's writes reach DRAM in fewer bytes.  obs_compressed says whether
        # every one of them was granted compressible memory.
        self.obs_compressed = True

        def obs_buffer(shape, dtype):
            t, compressed = ext.obs_empty(list(shape), dtype, dev.index)
            self.obs_compressed = self.obs_compressed and compressed
            return t

        # the ring (one per agent) carries the frame history, so there is exactly one; the small outputs still rotate
        self._ring = [obs_buffer((n, 2 * self.c, self.dim, self.dim), torch.uint8)
                      for _ in range(self.n_agents)] if self.ring else None
        self._sets = []
        for _ in range(max(1, int(n_buffers))):
            self._sets.append(dict(
                obs=None if self.ring else [obs_buffer(shape, torch.float32 if self.f32 else torch.uint8)
                                            for _ in range(self.n_agents)],
                rew=torch.zeros((n, 2), dtype=torch.float32, device=dev),
                real=torch.zeros((n, 2), dtype=torch.float32, device=dev),
                done=torch.zeros((n,), dtype=torch.bool, device=dev),
                steps=torch.zeros((n,), dtype=torch.int32, device=dev)))
        self._tracked = not self.ring and not self.f32 and self.dim == 84
        if self._tracked:
            self._impl.set_obs_buffers([b["obs"][0] for b in self._sets],
                                       [b["obs"][1] for b in self._sets] if self.n_agents == 2 else [])
        self._cur = 0
        self._bind(0)
        self._actions = torch.zeros((n, 2) if self.n_agents == 2 else (n,), dtype=torch.int32, device=dev)
        self._waiting = False
        self.closed = False
        self.envs = _EnvList(self)

    # ------------------------------------------------------------------ plumbing
    @property
    def _store(self):
        """the two buffers the rasteriser writes: the observations themselves, or the rings (single: agent 0's twice)"""
        b = self._ring if self.ring else self._obs
        return [b[0], b[1 if self.n_agents == 2 else 0]]

    @property
    def bytes_per_env_step(self):
        """observation bytes the rasteriser writes per env-step (SURVEY.md section 8(d))"""
        return self.n_agents * (2 if self.ring else self.c) * self.dim * self.dim * (4 if self.f32 else 1)

    def _bind(self, k):
        b = self._sets[k]
        self._cur = k
        self._rew, self._real, self._done, self._steps = b["rew"], b["real"], b["done"], b["steps"]
        if not self.ring:
            self._obs = b["obs"]

    def _ring_views(self):
        k = self._impl.ring_phase()
        self._obs = [r[:, k + 1:k + 1 + self.c] for r in self._ring]

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _ptr(self, t):
        return ctypes.c_void_p(t.data_ptr())

    @staticmethod
    def _to_numpy(x):
        if isinstance(x, tuple):
            return tuple(t.cpu().numpy() for t in x)
        return x.cpu().numpy()

    def _fmt_obs(self):
        obs = tuple(self._obs) if self.n_agents == 2 else self._obs[0]
        if self.return_numpy:
            return self._to_numpy(obs)
        if self.copy:
            return tuple(o.clone() for o in obs) if self.n_agents == 2 else obs.clone()
        return obs

    def inject_serves(self, serves):
        """Validation mode: serves[env, k] = (vx, vy) of the k-th serve since construction
        (replaces the reference's stdlib-random draws, pong/base_pong_env.py:314-320)."""
        s = np.ascontiguousarray(serves, np.float64)
        if s.ndim != 3 or s.shape[0] != self.num_envs or s.shape[2] != 2:
            raise ValueError("serves must have shape (num_envs, K, 2)")
        self._impl.inject_serves(torch.from_numpy(s))

    # ------------------------------------------------------------------ VecEnv protocol
    def reset(self):
        self._bind((self._cur + 1) % len(self._sets))
        st = self._store
        (self._impl.reset_f32 if self.f32 else self._impl.reset)(st[0], st[1] if self.n_agents == 2 else None)
        if self.ring:
            self._ring_views()
        self._waiting = False
        return self._fmt_obs()

    def _coerce_actions(self, actions):
        want = self._actions.shape
        if isinstance(actions, torch.Tensor):
            # device-resident actions are validated on the device: see check()
            if actions.dtype == torch.int32 and actions.device == self.device and actions.is_contiguous() \
                    and actions.numel() == self._actions.numel():
                return actions
            a = actions
        else:
            arr = np.asarray(actions)
            # the reference raises on anything else: assert action_space.contains (cPong, base_pong_env.py:42),
            # BAT_DIRECTIONS[a] IndexError (cPongDouble, :124/:134; Python's negative indices are not honoured here)
            bad = (arr < 0) | (arr > 2)
            if self.n_agents == 2:
                bad &= arr != 999
            if bad.any():
                raise (IndexError if self.n_agents == 2 else AssertionError)(
                    "invalid Pong action %r (valid: 0, 1, 2%s)" % (arr[bad].ravel()[0].item(), ", 999" if self.n_agents == 2 else ""))
            a = torch.as_tensor(arr)
        if tuple(a.shape) != tuple(want):
            a = a.reshape(want)
        self._actions.copy_(a, non_blocking=True)   # casts to int32 and moves to the device
        return self._actions

    def step_async(self, actions):
        if self._waiting:
            raise AlreadySteppingError()
        a = self._coerce_actions(actions)
        self._bind((self._cur + 1) % len(self._sets))
        st = self._store
        (self._impl.step_f32 if self.f32 else self._impl.step)(a, st[0], st[1] if self.n_agents == 2 else None, self._rew,
                                                                 self._done, self._steps, self._real)
        if self.ring:
            self._ring_views()
        self._waiting = True

    def step_wait(self):
        if not self._waiting:
            raise NotSteppingError()
        self._waiting = False
        done_b, rew_t, steps, real = self._done, self._rew, self._steps, self._real
        if self.copy:
            done_b, rew_t, steps, real = done_b.clone(), rew_t.clone(), steps.clone(), real.clone()
        infos = LazyInfos(self, steps, real, done_b)
        if self.asynchronous:   # SubprocVecEnv: np.stack(rews) / np.stack(dones)
            rew = rew_t if self.n_agents == 2 else rew_t[:, 0]
            done = done_b
        else:                   # DummyVecEnv: buf_rews (N, A) float32, buf_dones (N, A) bool
            rew = rew_t[:, :self.n_agents]
            done = done_b[:, None].expand(-1, self.n_agents)
        if self.return_numpy:
            rew = rew.cpu().numpy()
            done = done.cpu().numpy().copy()
            if self.asynchronous:
                rew = rew.astype(np.float64)
            infos = list(infos) if not self.asynchronous else tuple(infos)
        return self._fmt_obs(), rew, done, infos

    def _terminal_obs(self, done):
        shape = (self.num_envs, self.c, self.dim, self.dim)
        term = [torch.zeros(shape, dtype=torch.float32 if self.f32 else torch.uint8, device=self.device) for _ in range(self.n_agents)]
        if self.f32:
            self._impl.render_f32(True, done.to(torch.bool), term[0], term[1] if self.n_agents == 2 else None)
        else:
            self._impl.terminal_obs(done.to(torch.bool), term[0], term[1] if self.n_agents == 2 else None)
        return tuple(term) if self.n_agents == 2 else term[0]

    def seed(self, seed=None):
        # reference: [env.seed(seed + idx)] -> PongSinglePlayerEnv._seed is `pass` -> [None]*N
        if seed is not None:
            self._impl.seed(int(seed) & (2 ** 64 - 1))
        return [None] * self.num_envs

    def close(self):
        if not self.closed and self._impl is not None:
            if torch.cuda.is_available():
                torch.cuda.synchronize(self.device)
            if self._tracked:
                self._impl.set_obs_buffers([], [])
            self._impl.close()
            self._h = None
            # the env's references to its buffers: the observation memory goes back once the caller's are gone too
            self._ring, self._sets, self._obs = None, [], None
        self.closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    # ------------------------------------------------------------------ state / debug access
    def get_state(self):
        """float64 (N, 10) device tensor: ball_x, ball_y, vx, vy, left_y, right_y, score_l, score_r,
        num_rounds, num_steps (the PongGame fields)."""
        s = torch.empty((self.num_envs, 10), dtype=torch.float64, device=self.device)
        self._impl.get_state(s)
        return s

    def set_state(self, state):
        s = torch.as_tensor(state, dtype=torch.float64).to(self.device).contiguous()
        assert tuple(s.shape) == (self.num_envs, 10)
        self._impl.set_state(s)
        torch.cuda.current_stream(self.device).synchronize()

    def forget_obs(self):
        """After writing into observation tensors this env returned: the next render into each buffer rewrites it whole."""
        self._impl.forget_obs()

    def check(self):
        """Raise if a device-side error flag is set (serve table overrun, invalid device action).  Synchronises; the flag
        is cleared once reported."""
        self._impl.check()

    def episode_stats(self):
        """Device-accumulated episode statistics of this shard as a dict (synchronises)."""
        from .distributed import stats_from_raw
        return stats_from_raw(list(self._impl.stats()))

    def render_obs_generic(self):
        """Observations through the one-thread-per-pixel reference rasteriser (cross-check); ring mode: the views of a
        completely rewritten scratch ring."""
        if self.ring:
            out = [torch.empty_like(r) for r in self._ring]
        else:
            out = [torch.empty_like(o) for o in self._obs]
        self._impl.render_obs_generic(out[0], out[1] if self.n_agents == 2 else None)
        if self.ring:
            k = self._impl.ring_phase()
            out = [r[:, k + 1:k + 1 + self.c] for r in out]
        return tuple(out) if self.n_agents == 2 else out[0]

    def get_images(self, indices=None, agent=0, **kwargs):
        """Raw 210x160x3 RGB frames (what the reference's env.render('rgb_array') returns)."""
        imgs = []
        for i in self._get_indices(indices):
            f0 = torch.empty((210, 160, 3), dtype=torch.uint8, device=self.device)
            f1 = torch.empty_like(f0)
            self._impl.render_raw(int(i), f0, f1)
            imgs.append((f1 if agent == 1 else f0).cpu().numpy())
        return imgs

    def render(self, mode="human", *args, **kwargs):
        if self.num_envs == 1:
            return self.envs[0].render(mode=mode)
        return super().render(mode, *args, **kwargs)

    def get_attr(self, attr_name, indices=None):
        return [getattr(self.envs[i], attr_name) for i in self._get_indices(indices)]

    def set_attr(self, attr_name, value, indices=None):
        for i in self._get_indices(indices):
            setattr(self.envs[i], attr_name, value)

    def env_method(self, method_name, *method_args, indices=None, **method_kwargs):
        return [getattr(self.envs[i], method_name)(*method_args, **method_kwargs) for i in self._get_indices(indices)]


class _EnvList(object):
    """Lazy `envs` list so a 65 536-env batch does not allocate 65 536 Python objects."""

    def __init__(self, vec):
        self._vec = vec
        self._cache = {}

    def __len__(self):
        return self._vec.num_envs

    def __getitem__(self, i):
        if i < 0:
            i += len(self)
        if not 0 <= i < len(self):
            raise IndexError(i)
        if i not in self._cache:
            self._cache[i] = _EnvView(self._vec, i)
        return self._cache[i]

    def __iter__(self):
        for i in range(len(self)):
            yield self[i]
