"""Built-in opponents of the tournament env, evaluated on the device (SURVEY section 8 row f2).

Replaces competitive_rl/pong/builtin_policies.py:47-91 + utils/policy_serving.py:10-66 for a batched, GPU-resident
vec-env: the opponent's observation never leaves the device, its frame stack is a device tensor and its action
comes back as a device int32 tensor.  RULE_BASED is the env's own action 999 (pong/base_pong_env.py:116-134),
RANDOM a device randint; WEAK / MEDIUM (LightActorCritic, utils/network.py:73-93) and STRONG / ALPHA_PONG
(ActorCritic, :14-56) are torch networks whose weights come from the reference's checkpoint files
(resources/pong/checkpoint-*.pkl, a dict with the state dict under "model").  Those files are the reference's data,
not part of this repository: point COMPETITIVE_RL_RESOURCES (or the resource_dir argument) at the directory that
holds them; agents whose checkpoint is missing are simply not offered (the reference itself ships only weak and
medium).  The convolutions / linear layers are plain torch (cuDNN / cuBLAS) library calls.

The per-env opponents of tournament.py (set_opponents) run LightActorCritic networks in the project's own CUDA kernel
instead; pack_light_actor_critic is the flat parameter image that kernel loads.
"""
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from .vec_env import CHEAT_CODES

BUILTIN_AGENT_NAMES = ["RANDOM", "WEAK", "MEDIUM", "STRONG", "RULE_BASED", "ALPHA_PONG"]
_CHECKPOINTS = {"WEAK": ("checkpoint-weak.pkl", True), "MEDIUM": ("checkpoint-medium.pkl", True),
                "STRONG": ("checkpoint-strong.pkl", False), "ALPHA_PONG": ("checkpoint-alphapong.pkl", False)}


class LightActorCritic(nn.Module):
    """4x42x42 -> conv 4x4/2 (16) -> conv 2x2/2 (16) -> 1600 features -> 3 logits, 1 value.  Parameter names are the
    checkpoint's (conv1, conv2, critic_linear, actor_linear)."""

    def __init__(self, input_shape=(4, 42, 42), num_actions=3):
        super().__init__()
        c, h, w = input_shape
        self.conv1 = nn.Conv2d(c, 16, kernel_size=4, stride=2)
        self.conv2 = nn.Conv2d(16, 16, kernel_size=2, stride=2)
        h1, w1 = (h - 4) // 2 + 1, (w - 4) // 2 + 1
        feats = 16 * ((h1 - 2) // 2 + 1) * ((w1 - 2) // 2 + 1)
        self.critic_linear = nn.Linear(feats, 1)
        self.actor_linear = nn.Linear(feats, num_actions)

    def forward(self, x):
        x = F.relu(self.conv1(x / 255.0))
        x = F.relu(self.conv2(x)).flatten(1)
        return self.actor_linear(x), self.critic_linear(x)


# LightActorCritic's parameters in state-dict order: the flat layout the per-env opponent kernel loads
# (include/crl_b200.h, CRL_PONG_OPP_NET_FLOATS).  The critic is carried so that the image is the whole state dict.
LIGHT_ACTOR_CRITIC_LAYOUT = [("conv1.weight", (16, 4, 4, 4)), ("conv1.bias", (16,)), ("conv2.weight", (16, 16, 2, 2)),
                             ("conv2.bias", (16,)), ("critic_linear.weight", (1, 1600)), ("critic_linear.bias", (1,)),
                             ("actor_linear.weight", (3, 1600)), ("actor_linear.bias", (3,))]
LIGHT_ACTOR_CRITIC_FLOATS = 8484


def pack_light_actor_critic(state):
    """float32 CPU tensor of LIGHT_ACTOR_CRITIC_FLOATS: the parameters of a LightActorCritic (a state dict, a checkpoint
    dict with the state dict under "model", or the module) concatenated row-major in LIGHT_ACTOR_CRITIC_LAYOUT order.
    ActorCritic (STRONG / ALPHA_PONG) and any other layout are refused with ValueError."""
    if isinstance(state, nn.Module):
        state = state.state_dict()
    if "model" in state and not isinstance(state["model"], torch.Tensor):
        state = state["model"]
    names = [n for n, _ in LIGHT_ACTOR_CRITIC_LAYOUT]
    if any(k.startswith("conv3.") for k in state) or tuple(state.get("conv2.weight", torch.empty(0)).shape) == (32, 16, 4, 4):
        raise ValueError("an ActorCritic network (STRONG / ALPHA_PONG layout) cannot play in a per-env pool: only the "
                         "LightActorCritic layout (WEAK / MEDIUM) is supported")
    if sorted(state) != sorted(names):
        raise ValueError("not a LightActorCritic state dict: expected parameters %s, got %s" % (names, sorted(state)))
    parts = []
    for name, shape in LIGHT_ACTOR_CRITIC_LAYOUT:
        t = torch.as_tensor(state[name])
        if tuple(t.shape) != shape:
            raise ValueError("LightActorCritic parameter %s has shape %s, expected %s" % (name, tuple(t.shape), shape))
        parts.append(t.detach().to("cpu", torch.float32).reshape(-1))
    return torch.cat(parts).contiguous()


def unpack_light_actor_critic(flat):
    """Inverse of pack_light_actor_critic: a state dict LightActorCritic.load_state_dict accepts."""
    flat = torch.as_tensor(flat, dtype=torch.float32).reshape(-1)
    if flat.numel() != LIGHT_ACTOR_CRITIC_FLOATS:
        raise ValueError("a LightActorCritic image has %d floats, got %d" % (LIGHT_ACTOR_CRITIC_FLOATS, flat.numel()))
    out, k = {}, 0
    for name, shape in LIGHT_ACTOR_CRITIC_LAYOUT:
        n = 1
        for d in shape:
            n *= d
        out[name] = flat[k:k + n].reshape(shape).clone()
        k += n
    return out


class ActorCritic(nn.Module):
    """4x42x42 -> conv 4x4/2 (16) -> conv 4x4/2 pad 2 (32) -> conv 11x11 (256) -> 3 logits, 1 value."""

    def __init__(self, input_shape=(4, 42, 42), num_actions=3):
        super().__init__()
        c, h, w = input_shape
        self.conv1 = nn.Conv2d(c, 16, kernel_size=4, stride=2)
        self.conv2 = nn.Conv2d(16, 32, kernel_size=4, stride=2, padding=2)
        self.conv3 = nn.Conv2d(32, 256, kernel_size=11, stride=1)
        h1, w1 = (h - 4) // 2 + 1, (w - 4) // 2 + 1
        h2, w2 = (h1 + 4 - 4) // 2 + 1, (w1 + 4 - 4) // 2 + 1
        feats = 256 * (h2 - 11 + 1) * (w2 - 11 + 1)
        self.critic_linear = nn.Linear(feats, 1)
        self.actor_linear = nn.Linear(feats, num_actions)

    def forward(self, x):
        x = F.relu(self.conv1(x / 255.0))
        x = F.relu(self.conv2(x))
        x = F.relu(self.conv3(x)).flatten(1)
        return self.actor_linear(x), self.critic_linear(x)


def find_resource_dir(resource_dir=None):
    """Directory holding the reference's checkpoint-*.pkl files, or None."""
    cands = [resource_dir, os.environ.get("COMPETITIVE_RL_RESOURCES")]
    try:
        import competitive_rl   # a stock install of the reference keeps them in <repo>/resources/pong
        cands.append(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(competitive_rl.__file__))), "resources", "pong"))
    except Exception:  # noqa: BLE001
        pass
    for c in cands:
        if c and os.path.isdir(c):
            return c
    return None


class DevicePolicy(object):
    """policy_serving.Policy on the device: keeps the opponent's own stack of the last `frame_stack` single frames
    (FrameStackTensor.update: roll, append; never reset on done, like the reference) and returns greedy actions."""

    def __init__(self, num_envs, checkpoint_path="", use_light_model=True, device="cuda", obs_shape=(1, 42, 42),
                 frame_stack=4, num_actions=3):
        self.num_envs, self.device = num_envs, torch.device(device)
        self.num_channels = obs_shape[0]
        shape = (obs_shape[0] * frame_stack, *obs_shape[1:])
        net = LightActorCritic if use_light_model else ActorCritic
        self.model = net(shape, num_actions).to(self.device)
        if checkpoint_path:
            # the reference's checkpoint-*.pkl files hold {"model": state_dict, ...} of plain tensors: no pickled code is needed
            state = torch.load(checkpoint_path, map_location=self.device, weights_only=True)
            self.model.load_state_dict(state["model"] if "model" in state else state)
        self.model.requires_grad_(False)
        self.stack = torch.zeros((num_envs, *shape), dtype=torch.float32, device=self.device)

    def reset(self):
        self.stack.zero_()

    @torch.no_grad()
    def logits(self, obs):
        obs = torch.as_tensor(obs).to(self.device, dtype=torch.float32).reshape(self.num_envs, self.num_channels, *self.stack.shape[2:])
        self.stack = self.stack.roll(shifts=-self.num_channels, dims=1)
        self.stack[:, -self.num_channels:] = obs
        # plain fp32 convolutions (cuDNN would otherwise take TF32 tensor-core paths on this GPU: the networks are tiny,
        # and a greedy argmax over near-tied logits should not depend on the conv algorithm's precision)
        with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
            return self.model(self.stack)[0]

    def __call__(self, obs):
        """-> int32 [num_envs] device tensor of greedy actions (Categorical(logits).probs.argmax, policy_serving.py:50-56)."""
        return self.logits(obs).argmax(dim=1).to(torch.int32)


def get_builtin_agent_names(resource_dir=None):
    """Agents that can actually be built here: RANDOM, RULE_BASED and every network agent whose checkpoint exists."""
    d = find_resource_dir(resource_dir)
    names = []
    for n in BUILTIN_AGENT_NAMES:
        if n in _CHECKPOINTS and not (d and os.path.isfile(os.path.join(d, _CHECKPOINTS[n][0]))):
            continue
        names.append(n)
    return names


def find_checkpoint(agent_name, resource_dir=None):
    """Path of a built-in network agent's checkpoint file, or None when it cannot be found."""
    d = find_resource_dir(resource_dir)
    if agent_name not in _CHECKPOINTS or not d:
        return None
    path = os.path.join(d, _CHECKPOINTS[agent_name][0])
    return path if os.path.isfile(path) else None


def is_light_agent(agent_name):
    """True for the built-in network agents with the LightActorCritic layout (WEAK, MEDIUM)."""
    return agent_name in _CHECKPOINTS and _CHECKPOINTS[agent_name][1]


def light_network_image(name, added=None, resource_dir=None):
    """The packed LightActorCritic image (pack_light_actor_critic) of the network pool entry `name`, as the opponent
    kernel loads it: added[name] when `added` (name -> packed image) has it, else the built-in agent's checkpoint.
    ValueError for an ActorCritic agent (STRONG / ALPHA_PONG) and for a name with neither."""
    if added and name in added:
        return added[name]
    if name in BUILTIN_AGENT_NAMES and not is_light_agent(name):
        raise ValueError("%s is an ActorCritic agent: per-env pools take RULE_BASED, RANDOM and LightActorCritic "
                         "networks (WEAK, MEDIUM or add_opponent) only" % name)
    path = find_checkpoint(name, resource_dir)
    if path is None:
        raise ValueError("unknown opponent %r: not RULE_BASED / RANDOM, not added with add_opponent, and no "
                         "checkpoint found" % (name,))
    return pack_light_actor_critic(torch.load(path, map_location="cpu", weights_only=True))


def resolve_pool(pool, added=None, resource_dir=None):
    """A pool of names as the opponent kernel takes it (include/crl_b200.h, crl_pong_opp_set_pool): (names, kinds,
    images).  kinds[k] is entry k's kind: CRL_PONG_OPP_RULE_BASED, CRL_PONG_OPP_RANDOM or a network slot.  Networks
    take slots 0, 1, ... in pool order, and images[s] is slot s's image (light_network_image, `added` first).
    ValueError, before anything is loaded, for a pool that is not 1 to 16 distinct names, for more than 8 networks and
    for a name light_network_image refuses."""
    from . import _native
    ext = _native.ext()
    names = [str(p) for p in pool]
    if not 1 <= len(names) <= ext.OPP_MAX_POOL or len(set(names)) != len(names):
        raise ValueError("a pool is 1 to %d distinct names" % ext.OPP_MAX_POOL)
    nets = [p for p in names if p not in ("RULE_BASED", "RANDOM")]
    if len(nets) > ext.OPP_SLOTS:
        raise ValueError("a pool holds at most %d networks" % ext.OPP_SLOTS)
    images = [light_network_image(p, added, resource_dir) for p in nets]
    kinds = [ext.OPP_RULE_BASED if p == "RULE_BASED" else ext.OPP_RANDOM if p == "RANDOM" else nets.index(p)
             for p in names]
    return names, kinds, images


LEARNER = "LEARNER"   # a learner seat of a self-play pairing (selfplay.SelfPlayEnvWrapper); not a pool name there


def resolve_pairs(pairs, pool, learner=False):
    """Pairings as the opponent kernel takes them (include/crl_b200.h, crl_pong_opp_set_pairs and
    crl_pong_opp_set_selfplay): a list of [seat 0, seat 1].  Each seat of `pairs` is a name in `pool` (the names
    resolve_pool returned) or an index into it; with learner=True, "LEARNER" is a learner seat (CRL_PONG_OPP_LEARNER)
    and may not also be a pool name.  ValueError, before anything is loaded, for a pairing that is not two seats, a name
    not in the pool, an index out of range and for other than 1 to 256 pairings."""
    from . import _native
    ext = _native.ext()
    m = len(pool)
    if learner and LEARNER in pool:
        raise ValueError("%s is reserved for the learner's seats: it cannot be a pool name" % LEARNER)
    idx = []
    for pr in pairs:
        pr = list(pr)
        if len(pr) != 2:
            raise ValueError("a pairing is (seat 0, seat 1)")
        for x in pr:
            if isinstance(x, str) and x not in pool and not (learner and x == LEARNER):
                raise ValueError("pairing %r: %r is not in the pool" % (tuple(pr), x))
        is_lrn = [learner and isinstance(x, str) and x == LEARNER for x in pr]
        k = [ext.OPP_LEARNER if lr else pool.index(x) if isinstance(x, str) else int(x) for x, lr in zip(pr, is_lrn)]
        if not all(lr or 0 <= v < m for v, lr in zip(k, is_lrn)):
            raise ValueError("pairing %r: pool indices must be in [0, %d)" % (tuple(pr), m))
        idx.append(k)
    if not 1 <= len(idx) <= ext.OPP_MAX_PAIRS:
        raise ValueError("a league has 1 to %d pairings (got %d)" % (ext.OPP_MAX_PAIRS, len(idx)))
    return idx


def get_compute_action_function(agent_name, num_envs=1, device="cuda", resource_dir=None):
    """Callable obs -> int32 [num_envs] device tensor (pong/builtin_policies.py:61-91)."""
    device = torch.device(device)
    if agent_name == "RULE_BASED":
        return lambda _obs: torch.full((num_envs,), CHEAT_CODES, dtype=torch.int32, device=device)
    if agent_name == "RANDOM":
        return lambda _obs: torch.randint(0, 3, (num_envs,), dtype=torch.int32, device=device)
    if agent_name in _CHECKPOINTS:
        d = find_resource_dir(resource_dir)
        fname, light = _CHECKPOINTS[agent_name]
        path = os.path.join(d, fname) if d else None
        if not path or not os.path.isfile(path):
            raise FileNotFoundError("checkpoint %s of built-in agent %s not found; set COMPETITIVE_RL_RESOURCES to the "
                                    "reference's resources/pong directory" % (fname, agent_name))
        return DevicePolicy(num_envs, path, light, device)
    raise ValueError("Unknown agent name: {}".format(agent_name))
