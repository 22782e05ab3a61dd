"""TournamentEnvWrapper: single-agent view of a Double vec-env whose agent 1 is played by a built-in opponent
(competitive_rl/pong/competitive_pong_env.py:9-53).  The opponent acts on the device (builtin_policies.py): its
observation, frame stack and action never visit the host.  Available opponents: RANDOM, RULE_BASED and every
network agent whose checkpoint file can be found (the reference ships WEAK and MEDIUM).

Two modes:
  * uniform (the reference's): one opponent plays every env; `reset_opponent(name)` switches it for the whole batch.
  * per-env (`set_opponents`): every env plays its own opponent from a pool, evaluated for the whole batch by one CUDA
    kernel per step (csrc/pong_opponent.cu, include/crl_b200.h crl_pong_opp_*).  See `set_opponents` for the rules.
    `reset_opponent` returns to uniform mode.

In per-env mode a LightActorCritic learner can also act in the same launch (`set_learner`, `learner_step`): it samples
its action and returns its log-probability, its value and the stacked observation it acted on, as a PPO rollout
stores them."""
import numpy as np
import torch

from . import _native
from .builtin_policies import (get_builtin_agent_names, get_compute_action_function, is_light_agent,
                               pack_light_actor_critic, resolve_pool)


class TournamentEnvWrapper(object):
    def __init__(self, env, num_envs, resource_dir=None):
        self.env = env
        self.num_envs = num_envs
        self._resource_dir = resource_dir
        self.agent_names = [n for n in get_builtin_agent_names(resource_dir) if n != "ALPHA_PONG"]
        self.agents = {}                      # built on first use: a network agent allocates its stack and weights
        self.current_agent_name = "RULE_BASED"
        self.current_agent = self._agent("RULE_BASED")
        self.observation_space = env.observation_space[0]
        self.action_space = env.action_space[0]
        self.prev_opponent_obs = None
        # per-env mode
        self.per_env = False
        self.opponent_logits = None           # float32 (N, 3) device tensor: per-env steps write the actor logits here
        self._added = {}                      # add_opponent: name -> packed LightActorCritic image
        self._opp = None                      # the kernel's handle (PongOpponents), created on first use
        self._pool, self._resample, self._seed = None, False, 0
        self._have_prev = False               # env._rew / env._done hold the outputs of a step played in per-env mode
        self._both = None                     # int32 (N, 2) step buffer of per-env mode: learner | opponent
        # learner
        self.learner_logits = None            # float32 (N, 3) device tensor: learner steps write the learner's logits here
        self._sample = None                   # set_learner's `sample`; None until a learner is loaded

    def _agent(self, name):
        if name not in self.agents:
            self.agents[name] = get_compute_action_function(name, self.num_envs, self.env.device, self._resource_dir)
        return self.agents[name]

    def get_agent_names(self):
        return self.agent_names

    def reset_opponent(self, agent_name=None):
        if agent_name is None:
            agent_name = self.agent_names[int(np.random.randint(len(self.agent_names)))]
        assert agent_name in self.agent_names, self.agent_names
        self.current_agent_name = agent_name
        self.current_agent = self._agent(agent_name)
        self.per_env = False

    # ------------------------------------------------------------------ per-env mode
    def add_opponent(self, name, state_dict_or_path):
        """Make a LightActorCritic-layout network available to per-env pools under `name`: a state dict, a module, a
        checkpoint dict ({"model": state_dict}) or the path of a file holding one (e.g. a snapshot of the learner).
        A name added here takes precedence over a built-in checkpoint of the same name.  Adding a name that is in the
        current pool again replaces its weights from the next step on."""
        if name in ("RULE_BASED", "RANDOM"):
            raise ValueError("%s is not a network" % name)
        state = state_dict_or_path
        if isinstance(state, str):
            state = torch.load(state, map_location="cpu", weights_only=True)
        self._added[name] = pack_light_actor_critic(state)
        if self.per_env and name in self._pool:
            self._load_pool_nets()

    def _default_pool(self):
        pool = ["RULE_BASED", "RANDOM"] + [n for n in self.agent_names if is_light_agent(n) and n not in self._added]
        return pool + list(self._added)

    def _load_pool_nets(self):
        for slot, image in enumerate(resolve_pool(self._pool, self._added, self._resource_dir)[2]):
            self._opp.load_net(slot, image)

    def set_opponents(self, assignment=None, pool=None, weights=None, resample_on_done=False, seed=None):
        """Enter (or re-configure) per-env mode: every env plays its own opponent, chosen from `pool`.

        pool: up to 16 names: "RULE_BASED", "RANDOM", and up to 8 LightActorCritic networks (WEAK / MEDIUM from their
            checkpoints, or names given to add_opponent).  ActorCritic agents (STRONG, ALPHA_PONG) are refused.  None:
            the current pool in per-env mode, else every opponent available.  Needs resized_dim 42 and uint8
            observations without frame_stack (the cPongTournament-v0 defaults).
        assignment: None draws every env's opponent from the pool with `weights` (None: uniform); otherwise N pool
            names or indices.  A draw uses Philox keyed by (seed, global env index, the env's count of finished
            episodes), so it does not depend on how a batch is sharded.
        resample_on_done: an env whose episode ended draws a new opponent before its next step.
        seed: keys the draws and RANDOM's actions (kept from the previous call if None; 0 initially).

        Semantics of a per-env step: each env keeps a uint8 stack of agent 1's last 4 observations, zeroed on entering
        per-env mode, pushed every step whatever the env's opponent is and never cleared on done or reset (like the
        reference's policy_serving.Policy).  RULE_BASED plays action 999, RANDOM a uniform draw from {0, 1, 2}, a
        network the argmax of its actor logits over stack / 255 (fp32; ties to the lowest action).  A finished episode
        is credited to the opponent that played it: agent 0 wins if its summed clipped reward is > 0, draws at 0 and
        loses below (evaluate.py).  opponent_stats() reads the tally; setting a pool restarts it."""
        if self.env.dim != 42 or self.env.c != 1 or self.env.f32 or self.env.ring:
            raise ValueError("per-env opponents need resized_dim=42, frame_stack=None and uint8 observations")
        if pool is None:
            pool = self._pool if self.per_env else self._default_pool()
        pool, kinds, images = resolve_pool(pool, self._added, self._resource_dir)   # refuses bad pools before any change
        if seed is not None:
            self._seed = int(seed) & (2 ** 64 - 1)
        ext = _native.ext()
        if self._opp is None:
            self._opp = ext.PongOpponents(self.num_envs, int(self.env.device.index), self._seed, int(self.env.first_env))
        self._opp.seed(self._seed)
        for slot, image in enumerate(images):
            self._opp.load_net(slot, image)
        w = None
        if weights is not None:
            w = torch.as_tensor(np.asarray(weights, np.float64).reshape(-1))
            if w.numel() != len(pool):
                raise ValueError("one weight per pool entry")
        self._opp.set_pool(torch.tensor(kinds, dtype=torch.int32), w)
        if assignment is None:
            self._opp.assign(None)
        else:
            ids = [pool.index(a) if isinstance(a, str) else int(a) for a in list(np.asarray(assignment, dtype=object).reshape(-1))]
            if len(ids) != self.num_envs:
                raise ValueError("assignment needs one opponent per env (%d)" % self.num_envs)
            self._opp.assign(torch.tensor(ids, dtype=torch.int32))
        if not self.per_env:                 # entering: fresh stacks and reward sums, no episode end carried over
            self._opp.restart(True)
            self._have_prev = False
            self._both = torch.zeros((self.num_envs, 2), dtype=torch.int32, device=self.env.device)
        self._pool, self._resample, self.per_env = pool, bool(resample_on_done), True

    @property
    def opponent_ids(self):
        """int32 (N,) device tensor: every env's current opponent, an index into the pool (a snapshot, stream-ordered)."""
        if self._opp is None or self._pool is None:
            raise RuntimeError("no per-env opponents: call set_opponents first")
        out = torch.empty((self.num_envs,), dtype=torch.int32, device=self.env.device)
        self._opp.ids(out)
        return out

    @property
    def opponent_pool(self):
        return list(self._pool) if self._pool is not None else None

    def opponent_stats(self):
        """{name: {"episodes", "wins", "draws", "losses"}} of the episodes finished in per-env mode since the pool was
        last set; wins / draws / losses are agent 0's (the learner's).  One host synchronisation."""
        if self._opp is None or self._pool is None:
            raise RuntimeError("no per-env opponents: call set_opponents first")
        s = self._opp.stats()
        return {name: dict(episodes=int(s[4 * k]), wins=int(s[4 * k + 1]), draws=int(s[4 * k + 2]), losses=int(s[4 * k + 3]))
                for k, name in enumerate(self._pool)}

    # ------------------------------------------------------------------ learner
    def set_learner(self, module_or_state_dict, sample=True):
        """Load the learner's weights for learner_step: a LightActorCritic module, its state dict or a checkpoint dict
        ({"model": state_dict}); ActorCritic layouts are refused.  Needs per-env mode (set_opponents).  Call it again
        after every update to refresh the weights (one host synchronisation); they take effect on the next
        learner_step.  sample: sample the action from the softmax of the logits, else take the argmax."""
        if not self.per_env:
            raise RuntimeError("set_learner needs per-env opponents: call set_opponents first")
        self._opp.load_learner(pack_light_actor_critic(module_or_state_dict))
        self._sample = bool(sample)

    def learner_step(self, stack_out=None):
        """One step in which the learner (set_learner) acts for agent 0 and the per-env opponents for agent 1, both in one
        kernel launch, then the env steps.  Returns (stack, action, log_prob, value, obs, reward, done, info):
          stack     uint8 (N, 4, 42, 42): the learner's last 4 observations, oldest first, that it acted on (zeroed
                    before the newest frame after a done, like FrameStackTensor); written into `stack_out` if given
          action    int32 (N,); log_prob and value float32 (N,)
          obs, reward, done, info   as step() returns them.
        The learner's frames are stacked by the kernel (include/crl_b200.h, learner mode); step() is refused once
        learner steps have started, until set_opponents is called again.  learner_logits, if set, receives the
        learner's logits; opponent_logits is not written by learner steps."""
        if not self.per_env or self._sample is None:
            raise RuntimeError("no learner: call set_opponents, then set_learner")
        env = self.env
        dev = env.device
        n = self.num_envs
        if stack_out is None:
            stack_out = torch.empty((n, 4, 42, 42), dtype=torch.uint8, device=dev)
        both = torch.empty((n, 2), dtype=torch.int32, device=dev)
        lpv = torch.empty((n, 2), dtype=torch.float32, device=dev)
        prev = (env._rew, env._done) if self._have_prev else (None, None)
        self._opp.act_learner(env._obs[0], env._obs[1], prev[0], prev[1], self._resample, self._sample, both, lpv,
                              self.learner_logits, stack_out)
        self._both = both
        out = self._env_step(both)
        return (stack_out, both[:, 0], lpv[:, 0], lpv[:, 1]) + out

    # ------------------------------------------------------------------ VecEnv protocol
    def step(self, action):
        a = torch.as_tensor(np.asarray(action) if not isinstance(action, torch.Tensor) else action)
        a = a.reshape(-1).to(self.env.device, dtype=torch.int32)
        if self.per_env:
            env = self.env
            self._both[:, 0].copy_(a)
            prev = (env._rew, env._done) if self._have_prev else (None, None)
            self._opp.act(env._obs[1], prev[0], prev[1], self._resample, self._both, self.opponent_logits)
            both = self._both
        else:
            both = torch.stack([a, self.current_agent(self.prev_opponent_obs).reshape(-1)], dim=1)
        return self._env_step(both)

    def _env_step(self, both):
        obs, rew, done, info = self.env.step(both)
        self._have_prev = self.per_env
        self.prev_opponent_obs = obs[1]
        if done.ndim == 2:
            done = done[:, 0]
        return obs[0], rew[:, 0].reshape(-1, 1), done.reshape(-1, 1), info

    def reset(self, **kwargs):
        obs = self.env.reset(**kwargs)
        self.prev_opponent_obs = obs[1]
        if self.per_env:                     # per-env reward sums restart; opponents and stacks stay
            self._opp.restart(False)
        self._have_prev = False
        return obs[0]

    def seed(self, s):
        self.env.seed(s)

    def close(self):
        if self._opp is not None:
            torch.cuda.synchronize(self.env.device)
            self._opp.close()
            self._opp = None
        self.env.close()
