"""SelfPlayEnvWrapper: self-play rollouts on a cPongDouble vec-env, with a LightActorCritic learner in either seat of a
league pairing and frozen snapshots or built-in opponents in the other.

Every seat of every env is played by the self-play mode of the per-env opponent kernel (csrc/pong_opponent.cu,
include/crl_b200.h crl_pong_opp_set_selfplay / crl_pong_opp_act_selfplay): one launch per step stacks both agents'
frames, runs the learner for every learner seat and the pool's networks for the others, samples the learner's actions
and returns what a PPO rollout stores for each learner seat (the stack it acted on, the action, its log-probability and
the value).  Env g = first_env + i plays pairing g mod P for the whole run."""
import numpy as np
import torch

from . import _native
from .builtin_policies import LEARNER, pack_light_actor_critic, resolve_pairs, resolve_pool


class SelfPlayEnvWrapper(object):
    def __init__(self, env, resource_dir=None):
        if env.dim != 42 or env.c != 1 or env.f32 or env.ring or getattr(env, "n_agents", 2) != 2:
            raise ValueError("self-play needs a cPongDouble env with resized_dim=42, frame_stack=None and uint8 "
                             "observations")
        self.env = env
        self.num_envs = env.num_envs
        self._resource_dir = resource_dir
        self._added = {}                      # add_opponent: name -> packed LightActorCritic image
        self._opp = None                      # the kernel's handle (PongOpponents), created by the first set_league
        self._pool = self._pairs = None       # pool names and the table of name pairs of the current league
        self._seed = 0
        self._sample = None                   # set_learner's `sample`; None until a learner is loaded
        self._have_prev = False               # env._rew / env._done hold the outputs of a learner step
        self._seats = None
        self.logits = None                    # float32 (N, 2, 3) device tensor: learner steps write each seat's logits

    def add_opponent(self, name, state_dict_or_path):
        """Make a LightActorCritic-layout network available to leagues under `name`: a state dict, a module, a
        checkpoint dict ({"model": state_dict}) or the path of a file holding one (e.g. a snapshot of the learner).
        A name added here takes precedence over a built-in checkpoint of the same name.  Adding a name that is in the
        current pool again replaces its weights from the next step on."""
        if name in ("RULE_BASED", "RANDOM"):
            raise ValueError("%s is not a network" % name)
        if name == LEARNER:
            raise ValueError("%s is reserved for the learner's seats: it cannot be a pool name" % LEARNER)
        state = state_dict_or_path
        if isinstance(state, str):
            state = torch.load(state, map_location="cpu", weights_only=True)
        self._added[name] = pack_light_actor_critic(state)
        if self._pool is not None and name in self._pool:
            for slot, image in enumerate(resolve_pool(self._pool, self._added, self._resource_dir)[2]):
                self._opp.load_net(slot, image)

    def set_league(self, pairs=((LEARNER, LEARNER),), seed=None):
        """Enter (or re-configure) a league: `pairs` is a list of (seat 0, seat 1) names, each "LEARNER" (the learner,
        set_learner) or a pool entry ("RULE_BASED", "RANDOM", WEAK / MEDIUM from their checkpoints, or a name given to
        add_opponent).  The pool is the distinct other names, in order of appearance: at most 16, of which at most 8
        networks; a table with learner seats only gets a RULE_BASED pool that no env plays.  At most 256 pairings; env
        g plays pairing g mod P for the whole run.  seed keys the learner's draws and RANDOM's actions (kept from the
        previous call if None; 0 initially).  Every ring and the pairing tally restart; the env is not reset.

        Semantics of a step: each env keeps a uint8 stack of each agent's last 4 observations.  A learner seat's stack
        is zeroed before the newest frame after a done and by reset() (FrameStackTensor); a pool seat's never is.  A pool
        seat plays as in evaluate.evaluate_pool_in_batch: RULE_BASED action 999, RANDOM a uniform draw, a network the
        argmax of its logits.  A finished episode is credited to the env's pairing from seat 0's side."""
        pairs = [tuple(pr) for pr in pairs]
        for pr in pairs:
            if not all(isinstance(x, str) for x in pr):
                raise ValueError("pairing %r: a seat is %r or a pool name" % (pr, LEARNER))
        names = []
        for pr in pairs:
            names += [x for x in pr if x != LEARNER and x not in names]
        pool, kinds, images = resolve_pool(names or ["RULE_BASED"], self._added, self._resource_dir)
        idx = resolve_pairs(pairs, pool, learner=True)   # refuses bad tables before any change
        if seed is not None:
            self._seed = int(seed) & (2 ** 64 - 1)
        ext = _native.ext()
        dev = self.env.device
        if self._opp is None:
            self._opp = ext.PongOpponents(self.num_envs, int(dev.index), self._seed, int(self.env.first_env))
        self._opp.seed(self._seed)
        for slot, image in enumerate(images):
            self._opp.load_net(slot, image)
        self._opp.set_pool(torch.tensor(kinds, dtype=torch.int32), None)
        self._opp.set_selfplay(torch.tensor(idx, dtype=torch.int32))
        self._pool, self._pairs, self._have_prev = pool, pairs, False
        table = torch.tensor(idx, dtype=torch.int32) == ext.OPP_LEARNER                    # [P, 2]
        g = int(self.env.first_env) + np.arange(self.num_envs, dtype=np.int64)
        self._seats = table[torch.from_numpy(g % len(idx))].to(dev)

    def set_learner(self, module_or_state_dict, sample=True):
        """Load the learner's weights for learner_step: a LightActorCritic module, its state dict or a checkpoint dict
        ({"model": state_dict}); ActorCritic layouts are refused.  Needs a league (set_league).  Call it again after
        every update to refresh the weights (one host synchronisation); they take effect on the next learner_step.
        sample: sample the learner's actions from the softmax of its logits, else take the argmax."""
        if self._opp is None:
            raise RuntimeError("set_learner needs a self-play league: call set_league first")
        self._opp.load_learner(pack_light_actor_critic(module_or_state_dict))
        self._sample = bool(sample)

    @property
    def learner_seats(self):
        """bool (N, 2) device tensor: which seats of every env the learner plays."""
        if self._seats is None:
            raise RuntimeError("no league: call set_league first")
        return self._seats

    def learner_step(self, stack_out=None):
        """One step in which every seat of every env acts in one kernel launch, then the env steps.  Returns
        (stack, action, log_prob, value, obs, reward, done, info):
          stack     uint8 (N, 2, 4, 42, 42): per learner seat the last 4 observations of its agent, oldest first, that it
                    acted on; written into `stack_out` if given.  Rows of pool seats are not written.
          action    int32 (N, 2): both seats' actions
          log_prob, value   float32 (N, 2): the learner seats' log pi(action) and value, 0 for pool seats
          obs, reward, done, info   as the env's step() returns them; reward holds both agents' clipped rewards, so
                    the transitions of a learner in seat 1 use column 1.
        learner_seats tells which (env, seat) rows are the learner's transitions.  logits, if set, receives each seat's
        logits (0 for RULE_BASED and RANDOM seats)."""
        if self._opp is None or self._sample is None:
            raise RuntimeError("no learner: call set_league, then set_learner")
        env = self.env
        dev = env.device
        n = self.num_envs
        if stack_out is None:
            stack_out = torch.empty((n, 2, 4, 42, 42), dtype=torch.uint8, device=dev)
        actions = torch.empty((n, 2), dtype=torch.int32, device=dev)
        lpv = torch.empty((n, 2, 2), dtype=torch.float32, device=dev)
        prev = (env._rew, env._done) if self._have_prev else (None, None)
        self._opp.act_selfplay(env._obs[0], env._obs[1], prev[0], prev[1], self._sample, actions, lpv, self.logits,
                               stack_out)
        obs, rew, done, info = env.step(actions)
        self._have_prev = True
        return (stack_out, actions, lpv[:, :, 0], lpv[:, :, 1], obs, rew, done, info)

    def pair_stats(self):
        """{(seat 0 name, seat 1 name): {"episodes", "wins", "draws", "losses"}} of the episodes finished since the
        league was set, counted from seat 0's side; repeated pairings add up.  One host synchronisation."""
        if self._opp is None or self._pairs is None:
            raise RuntimeError("no league: call set_league first")
        s = self._opp.pair_stats(len(self._pairs))
        out = {}
        for k, pr in enumerate(self._pairs):
            d = out.setdefault(pr, dict(episodes=0, wins=0, draws=0, losses=0))
            for j, key in enumerate(("episodes", "wins", "draws", "losses")):
                d[key] += int(s[4 * k + j])
        return out

    def reset(self):
        """Resets the env; every learner seat's stack and the per-env reward sums restart (pool seats keep theirs)."""
        obs = self.env.reset()
        if self._opp is not None:
            self._opp.restart(False)
        self._have_prev = False
        return obs

    def close(self):
        if self._opp is not None:
            torch.cuda.synchronize(self.env.device)
            self._opp.close()
            self._opp = None
        self.env.close()
