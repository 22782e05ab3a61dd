"""Host model of the learner mode of the per-env opponent kernel (csrc/pong_opponent.cu, include/crl_b200.h
crl_pong_opp_load_learner / crl_pong_opp_act_learner) -- TEST INFRASTRUCTURE ONLY.  Written from the header's semantics;
the Philox streams, the float64 actor and the seat-1 model are opponent_oracle's.

  value64, value_magnitude64   LightActorCritic's critic in float64, and its scale M (as forward64 / magnitude64)
  learner_u                    the learner's uniform draw u = r32 * 2^-32 (Philox tag 4)
  cdf64, sample64, logprob64   the inverse-CDF action and log pi(a) in float64 from given logits
  boundary_distance            how far u is from the nearest cumulative bound (the rows where fp32 may choose otherwise)
  HostLearner                  HostOpponents plus the learner's FrameStackTensor ring
"""
import numpy as np
import torch

from opponent_oracle import DIM, NET_FLOATS, HostOpponents, _patches, forward64, magnitude64, opp_rand

LEARNER_TAG = 4


# ---------------------------------------------------------------------------------------------------- critic
def _critic(x_u8, params, absolute, chunk=8192):
    x_u8 = torch.as_tensor(x_u8)
    dev = x_u8.device
    p = torch.as_tensor(np.asarray(params, dtype=np.float32) if not torch.is_tensor(params) else params)
    p = p.reshape(-1).to(device=dev, dtype=torch.float64)
    assert p.numel() == NET_FLOATS
    w1, b1 = p[0:1024].reshape(16, 64), p[1024:1040]
    w2, b2 = p[1040:2064].reshape(16, 64), p[2064:2080]
    wc, bc = p[2080:3680], p[3680]                            # critic_linear [1][1600], [1]
    if absolute:
        w1, b1, w2, b2, wc, bc = (t.abs() for t in (w1, b1, w2, b2, wc, bc))
    out = torch.empty((x_u8.shape[0],), dtype=torch.float64, device=dev)
    for s in range(0, x_u8.shape[0], chunk):
        x = x_u8[s:s + chunk].reshape(-1, 4, DIM, DIM).to(torch.float64) / 255.0
        h1 = torch.relu(w1 @ _patches(x, 4, 20) + b1[:, None])
        h2 = torch.relu(w2 @ _patches(h1.reshape(-1, 16, 20, 20), 2, 10) + b2[:, None])
        out[s:s + chunk] = h2.reshape(-1, 1600) @ wc + bc
    return out


def value64(x_u8, params):
    """LightActorCritic's value [B] (float64, on x's device) for uint8 stacks [B, 4, 42, 42]: the features of forward64
    through critic_linear."""
    return _critic(x_u8, params, False)


def value_magnitude64(x_u8, params):
    """The critic with |W|, |b| and |x|: the sum of the magnitudes of all products that reach the value."""
    return _critic(x_u8, params, True)


# ---------------------------------------------------------------------------------------------------- sampling
def learner_u(seed, g, ctr):
    """The learner's draw of global env(s) g at act count ctr: r32 * 2^-32 of the tag-4 stream (float64, exact)."""
    r = opp_rand(seed, g, LEARNER_TAG, ctr)
    return np.asarray(r, dtype=np.float64) * 2.0 ** -32


def cdf64(logits):
    """[B, 2] cumulative softmax bounds (c_0, c_1) in float64."""
    lg = np.asarray(logits, np.float64)
    e = np.exp(lg - lg.max(axis=1, keepdims=True))
    p = e / e.sum(axis=1, keepdims=True)
    return np.stack([p[:, 0], p[:, 0] + p[:, 1]], axis=1)


def sample64(logits, u):
    """Inverse-CDF action per row: the first k with u < c_k, else 2."""
    c = cdf64(logits)
    u = np.asarray(u, np.float64)
    return np.where(u < c[:, 0], 0, np.where(u < c[:, 1], 1, 2))


def boundary_distance(logits, u):
    """min_k |u - c_k| per row: a row closer than the fp32 rounding of c_k may be sampled differently in fp32."""
    c = cdf64(logits)
    return np.abs(np.asarray(u, np.float64)[:, None] - c).min(axis=1)


def logprob64(logits, actions):
    """log pi(a) = l_a - logsumexp(l) per row, float64."""
    lg = np.asarray(logits, np.float64)
    m = lg.max(axis=1)
    lse = m + np.log(np.exp(lg - m[:, None]).sum(axis=1))
    return lg[np.arange(len(lg)), np.asarray(actions)] - lse


# ---------------------------------------------------------------------------------------------------- handle model
class LearnerStep(object):
    """What one act_learner of HostLearner computed for the learner: the stack it acted on [n, 4, 42, 42] (uint8, on the
    model's device), the float64 logits [n, 3] and value [n] with their magnitudes, and the draw u [n] (float64).  The
    seat-1 step (opponent_oracle.Step) is `opp`."""

    def __init__(self, stack, ref, mag, value, value_mag, u, opp):
        self.stack, self.ref, self.mag, self.value, self.value_mag, self.u, self.opp = stack, ref, mag, value, value_mag, u, opp


class HostLearner(HostOpponents):
    """Host model of a crl_pong_opp handle in learner mode (include/crl_b200.h), written from the header's semantics:
    seat 1 is HostOpponents; seat 0 keeps an [n, 4, 42, 42] uint8 ring, oldest to newest, shifted on every push and
    zeroed before the push when the previous step's done is set; the ring is zeroed on entering learner mode and by
    every restart in learner mode."""

    def __init__(self, n, seed, first_env=0, device="cpu"):
        super().__init__(n, seed, first_env, device)
        self.learner = None
        self.in_learner_mode = False
        self.ring = torch.zeros((n, 4, DIM, DIM), dtype=torch.uint8, device=self.device)

    def load_learner(self, params):
        self.learner = torch.as_tensor(params, dtype=torch.float32).reshape(-1).clone()

    def set_pool(self, kinds, weights=None):
        super().set_pool(kinds, weights)
        self.in_learner_mode = False

    def restart(self, clear):
        super().restart(clear)
        if clear or self.in_learner_mode:
            self.ring.zero_()

    def act_learner(self, obs0, obs1, rew=None, done=None, resample=False):
        """obs0, obs1 uint8 [n, 42, 42] (any device); rew float32 [n, 2] and done [n] as numpy, or both None."""
        assert self.learner is not None
        if not self.in_learner_mode:
            self.ring.zero_()
            self.in_learner_mode = True
        if done is not None:
            d = torch.from_numpy(np.asarray(done).astype(bool)).to(self.device)
            self.ring[d] = 0
        frame = torch.as_tensor(obs0).to(self.device).reshape(self.n, 1, DIM, DIM)
        self.ring = torch.cat([self.ring[:, 1:], frame], dim=1)
        u = learner_u(self.seed_, self.g, self.acts)          # the act count before this act
        opp = self.act(obs1, rew, done, resample)
        x = self.ring
        return LearnerStep(x.clone(), forward64(x, self.learner).cpu().numpy(), magnitude64(x, self.learner).cpu().numpy(),
                           value64(x, self.learner).cpu().numpy(), value_magnitude64(x, self.learner).cpu().numpy(), u,
                           opp)
