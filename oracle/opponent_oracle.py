"""Independent reference of the per-env opponent kernel (csrc/pong_opponent.cu, include/crl_b200.h crl_pong_opp_*) --
TEST INFRASTRUCTURE ONLY.  Plain Python / numpy / torch; the network runs in float64 with the same code on the CPU or a
GPU.

Pieces:
  philox4x32_10, opp_rand, opp_draw, random_action   the kernel's Philox streams (pong_common.cuh, pong_opponent.cu)
  cum_bounds                                         crl_pong_opp_set_pool's draw bounds
  forward64, magnitude64                             LightActorCritic's actor logits in float64, and their scale M
  logit_ratio, greedy, decided                       the tolerance rule and the action rule below
  HostOpponents                                      a host model of one handle, written from the header's semantics

Tolerance of the network's logits
---------------------------------
The kernel computes in fp32: x = lut[byte] (byte / 255 rounded once), then conv1 as 64 chained FMAs per output, conv2 as
64 chained FMAs, the actor as strided FMA chains, a warp tree and 7 ordered adds (about 21 roundings on one path), plus
the bias.  Let M be the same network evaluated with |W|, |b| and |x| (magnitude64): the sum of the magnitudes of every
product that reaches a logit.  The worst-case bound on any such evaluation order is gamma_n * M with n ~ 150 roundings
on the longest chain, about 150 u M (u = 2^-24).  That is too loose to be useful: feeding byte / 256 instead of byte / 255
moves the logits by only 34 to 270 u M.

Rounding errors of a chained sum are not all of one sign and not all at the worst magnitude, and |partial sums| are far
below M once terms cancel.  Measured on CPU with random weights at PyTorch's default init scale and at 30x, on uniform
random, all-255 and sparse Pong-like frames (512 envs each), the largest |error| / (u M) is
(tests/test_opponent_oracle_cpu.py prints its own values):
    torch fp32 (any summation order it picks)            <= 0.07
    x / 256 instead of x / 255                           34 to 270
    two conv1 taps swapped, random frames               >= 2 500
    two conv1 taps swapped, all-255 frames               0 (a constant frame cannot see a tap permutation)
The rule is |got - ref| <= 4 u M per logit (TOL_ULPS = 4): 50x above what a correct fp32 evaluation shows, 8x below the
smallest input-scaling bug.  Tests use frames in which every byte varies, so that layout bugs are visible.

Action rule: the kernel's action must be exactly the argmax of the logits it returned (ties to the lowest index), and it
must equal argmax(ref) wherever ref's top-two margin exceeds the sum of those two logits' tolerances (`decided`).  There
is no allowance for flips beyond that.
"""
import numpy as np
import torch

U = 2.0 ** -24
TOL_ULPS = 4.0
RULE_BASED, RANDOM = -1, -2          # CRL_PONG_OPP_RULE_BASED / CRL_PONG_OPP_RANDOM
CHEAT_CODES = 999                    # RULE_BASED's action
SLOTS, MAX_POOL, NET_FLOATS = 8, 16, 8484
DIM = 42
_M32 = 0xFFFFFFFF


# ---------------------------------------------------------------------------------------------------- Philox
def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al., SC'11).  Works on Python ints, or on numpy uint64 arrays holding 32-bit values
    (the 32x32 -> 64-bit products fit).  Returns (r0, r1, r2, r3)."""
    for _ in range(10):
        p0 = 0xD2511F53 * c0
        p1 = 0xCD9E8D57 * c2
        c0, c1, c2, c3 = (p1 >> 32) ^ c1 ^ k0, p1 & _M32, (p0 >> 32) ^ c3 ^ k1, p0 & _M32
        k0 = (k0 + 0x9E3779B9) & _M32
        k1 = (k1 + 0xBB67AE85) & _M32
    return c0, c1, c2, c3


def opp_rand(seed, g, tag, ctr):
    """r32 of stream (global env g, tag) at counter ctr, keyed by seed: tag 1 = RANDOM's actions, tag 2 = draws.
    g and ctr may be arrays (numpy uint64 result) or ints (int result)."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    if np.isscalar(g) and np.isscalar(ctr):
        g, ctr = int(g) & 0xFFFFFFFFFFFFFFFF, int(ctr) & 0xFFFFFFFFFFFFFFFF
        return philox4x32_10(g & _M32, (g >> 32) ^ (tag << 24), ctr & _M32, ctr >> 32, seed & _M32, seed >> 32)[0]
    g = np.asarray(g, dtype=np.int64).astype(np.uint64)      # two's complement, as (uint64_t)g
    ctr = np.broadcast_to(np.asarray(ctr, dtype=np.uint64), g.shape)
    return philox4x32_10(g & np.uint64(_M32), (g >> np.uint64(32)) ^ np.uint64(tag << 24), ctr & np.uint64(_M32),
                         ctr >> np.uint64(32), np.uint64(seed & _M32), np.uint64(seed >> 32))[0]


def cum_bounds(weights):
    """crl_pong_opp_set_pool's bounds (a list of ints): entry k is drawn first when r32 < bound[k].  Entries from the
    last positive weight on get 2^32; the others floor(prefix / total * 2^32) in double, accumulated in pool order.
    (The ABI's NULL weights are a list of ones here.)"""
    w = [float(x) for x in weights]
    total = 0.0
    for x in w:
        total += x
    last = max(k for k, x in enumerate(w) if x > 0.0)
    out, run = [], 0.0
    for k, x in enumerate(w):
        run += x
        out.append(1 << 32 if k >= last else int(np.floor(run / total * 4294967296.0)))
    return out


def opp_draw(cum, seed, g, episode):
    """Pool index drawn for global env(s) g after `episode` finished episodes: the first k (< pool size - 1) with
    r32 < cum[k], else the last entry."""
    r = opp_rand(seed, g, 2, episode)
    if np.isscalar(r):
        k = 0
        while k < len(cum) - 1 and r >= cum[k]:
            k += 1
        return k
    k = np.zeros(r.shape, np.int64)
    for j in range(len(cum) - 1):
        k += (k == j) & (r >= np.uint64(cum[j]))
    return k


def random_action(seed, g, ctr):
    """RANDOM's action of global env(s) g at act count ctr: (r32 * 3) >> 32, in {0, 1, 2}."""
    r = opp_rand(seed, g, 1, ctr)
    if np.isscalar(r):
        return (r * 3) >> 32
    return ((r * np.uint64(3)) >> np.uint64(32)).astype(np.int64)


# ---------------------------------------------------------------------------------------------------- network
def _unflat(params, dev):
    """The flat state-dict image (pack_light_actor_critic order) as float64 matrices on dev."""
    p = torch.as_tensor(np.asarray(params, dtype=np.float32) if not torch.is_tensor(params) else params)
    p = p.reshape(-1).to(device=dev, dtype=torch.float64)
    assert p.numel() == NET_FLOATS
    w1, b1 = p[0:1024].reshape(16, 64), p[1024:1040]          # conv1.weight [co][ci][kh][kw], conv1.bias
    w2, b2 = p[1040:2064].reshape(16, 64), p[2064:2080]       # conv2.weight [co][ci][kh][kw], conv2.bias
    wa, ba = p[3681:8481].reshape(3, 1600), p[8481:8484]      # actor_linear (critic_linear 2080:3681 is skipped)
    return w1, b1, w2, b2, wa, ba


def _patches(x, k, out):
    """[B, C, H, W] -> [B, C*k*k, out*out]: stride-2 k x k windows, rows in (c, kh, kw) order, columns (y, x)."""
    span = 2 * (out - 1) + 1
    cols = [x[:, :, kh:kh + span:2, kw:kw + span:2] for kh in range(k) for kw in range(k)]
    return torch.stack(cols, 2).reshape(x.shape[0], x.shape[1] * k * k, out * out)


def _net(x_u8, params, absolute, chunk=8192):
    x_u8 = torch.as_tensor(x_u8)
    dev = x_u8.device
    w1, b1, w2, b2, wa, ba = _unflat(params, dev)
    if absolute:
        w1, b1, w2, b2, wa, ba = (t.abs() for t in (w1, b1, w2, b2, wa, ba))
    out = torch.empty((x_u8.shape[0], 3), dtype=torch.float64, device=dev)
    for s in range(0, x_u8.shape[0], chunk):
        x = x_u8[s:s + chunk].reshape(-1, 4, DIM, DIM).to(torch.float64) / 255.0      # |x| = x
        h1 = torch.relu(w1 @ _patches(x, 4, 20) + b1[:, None])                         # [B, 16, 400]
        h2 = torch.relu(w2 @ _patches(h1.reshape(-1, 16, 20, 20), 2, 10) + b2[:, None])   # [B, 16, 100]
        out[s:s + chunk] = h2.reshape(-1, 1600) @ wa.T + ba
    return out


def forward64(x_u8, params):
    """LightActorCritic's actor logits [B, 3] (float64, on x's device) for uint8 stacks x_u8 [B, 4, 42, 42] (oldest ->
    newest): x = byte / 255 -> conv 4x4/2 -> ReLU -> conv 2x2/2 -> ReLU -> flatten (c, y, x) -> actor_linear."""
    return _net(x_u8, params, False)


def magnitude64(x_u8, params):
    """The same network with |W|, |b| and |x|: per logit, the sum of the magnitudes of all products that reach it."""
    return _net(x_u8, params, True)


def logit_ratio(got, ref, mag):
    """|got - ref| / (u M), elementwise (float64 numpy).  The tolerance rule is logit_ratio <= TOL_ULPS."""
    got, ref, mag = (np.asarray(a, dtype=np.float64) for a in (got, ref, mag))
    return np.abs(got - ref) / (U * np.maximum(mag, np.finfo(np.float64).tiny))


def greedy(logits):
    """Argmax per row, ties to the lowest index."""
    return np.argmax(np.asarray(logits), axis=1)


def decided(ref, mag, ulps=TOL_ULPS):
    """Rows whose top-two reference margin exceeds the sum of those two logits' tolerances: there the greedy action of
    any logits within tolerance is argmax(ref)."""
    ref, mag = np.asarray(ref, np.float64), np.asarray(mag, np.float64)
    order = np.argsort(-ref, axis=1, kind="stable")
    rows = np.arange(len(ref))
    i1, i2 = order[:, 0], order[:, 1]
    return ref[rows, i1] - ref[rows, i2] > ulps * U * (mag[rows, i1] + mag[rows, i2])


# ---------------------------------------------------------------------------------------------------- test inputs
def random_params(gen, scale=1.0):
    """float32 [NET_FLOATS] image of a LightActorCritic at PyTorch's default init scale (every tensor, bias included,
    uniform in +-1/sqrt(fan_in): 64 for both convs, 1600 for the linears) times `scale`.  gen: a CPU torch.Generator."""
    parts = []
    for numel, fan_in in ((1024, 64), (16, 64), (1024, 64), (16, 64), (1600, 1600), (1, 1600), (4800, 1600), (3, 1600)):
        b = scale / np.sqrt(fan_in)
        parts.append((torch.rand(numel, generator=gen, dtype=torch.float64) * 2 - 1) * b)
    return torch.cat(parts).to(torch.float32)


FRAME_KINDS = ("random", "zeros", "full", "sparse")


def synthetic_frames(kind, n, gen, device="cpu"):
    """uint8 [n, 42, 42] frames: uniform random bytes, all 0, all 255, or sparse Pong-like frames (a random background
    per frame with two bats and a ball of random values and positions).  gen: a torch.Generator on `device`."""
    if kind == "zeros":
        return torch.zeros((n, DIM, DIM), dtype=torch.uint8, device=device)
    if kind == "full":
        return torch.full((n, DIM, DIM), 255, dtype=torch.uint8, device=device)

    def ri(lo, hi):
        return torch.randint(lo, hi, (n, 1, 1), generator=gen, device=device)

    if kind == "random":
        return torch.randint(0, 256, (n, DIM, DIM), generator=gen, device=device, dtype=torch.uint8)
    assert kind == "sparse", kind
    yy = torch.arange(DIM, device=device).view(1, DIM, 1)
    xx = torch.arange(DIM, device=device).view(1, 1, DIM)
    f = ri(0, 256).expand(n, DIM, DIM).clone()
    for y0, x0, h, w in ((ri(0, 35), 3, 7, 2), (ri(0, 35), 37, 7, 2), (ri(0, 40), ri(6, 35), 2, 2)):
        m = (yy >= y0) & (yy < y0 + h) & (xx >= x0) & (xx < x0 + w)
        f = torch.where(m, ri(0, 256).expand(n, DIM, DIM), f)
    return f.to(torch.uint8)


# ---------------------------------------------------------------------------------------------------- handle model
class Step(object):
    """What one act of HostOpponents computed: ids used (after redraws), the kind of each env's opponent, the action of
    each non-network env (-1 for network envs), and for network envs the float64 logits and their magnitudes (0
    elsewhere, like the kernel's logits)."""

    def __init__(self, ids, kind, actions, ref, mag):
        self.ids, self.kind, self.actions, self.ref, self.mag = ids, kind, actions, ref, mag
        self.net = kind >= 0


class HostOpponents(object):
    """Host model of one crl_pong_opp handle (include/crl_b200.h), written from the header's semantics and independent
    of the kernel's layout: the frame stack is an [n, 4, 42, 42] uint8 tensor, oldest to newest, shifted on every push.
    Per-env bookkeeping is numpy; the stack lives on `device`, where the networks run in float64."""

    def __init__(self, n, seed, first_env=0, device="cpu"):
        self.n, self.device = n, torch.device(device)
        self.seed_ = int(seed)
        self.g = int(first_env) + np.arange(n, dtype=np.int64)
        self.nets = {}
        self.kinds = self.cum = None
        self.assigned = False
        self.ids = np.zeros(n, np.int64)
        self.ret = np.zeros(n, np.float32)
        self.episodes = np.zeros(n, np.int64)
        self.stats = np.zeros((MAX_POOL, 4), np.int64)
        self.stack = torch.zeros((n, 4, DIM, DIM), dtype=torch.uint8, device=self.device)
        self.acts = 0

    def seed(self, s):
        self.seed_ = int(s)

    def load_net(self, slot, params):
        self.nets[slot] = torch.as_tensor(params, dtype=torch.float32).reshape(-1).clone()

    def set_pool(self, kinds, weights=None):
        self.kinds = np.asarray(kinds, np.int64)
        self.cum = cum_bounds(np.ones(len(kinds)) if weights is None else weights)
        self.stats[:] = 0
        self.assigned = False

    def assign(self, ids=None):
        self.ids = (np.asarray(ids, np.int64).copy() if ids is not None
                    else opp_draw(self.cum, self.seed_, self.g, self.episodes & _M32))
        self.assigned = True

    def restart(self, clear):
        self.ret[:] = 0
        if clear:
            self.stack.zero_()

    def act(self, obs1, rew=None, done=None, resample=False):
        """obs1 uint8 [n, 42, 42] (any device); rew float32 [n, 2] and done [n] as numpy, or both None."""
        assert self.assigned
        if rew is not None:
            r = (self.ret + np.asarray(rew, np.float32)[:, 0]).astype(np.float32)
            d = np.asarray(done).astype(bool)
            old, rd = self.ids[d], r[d]
            np.add.at(self.stats, (old, 0), 1)
            np.add.at(self.stats, (old, np.where(rd > 0, 1, np.where(rd == 0, 2, 3))), 1)
            r[d] = 0
            self.episodes[d] += 1
            if resample:
                self.ids[d] = opp_draw(self.cum, self.seed_, self.g[d], self.episodes[d] & _M32)
            self.ret = r
        frame = torch.as_tensor(obs1).to(self.device).reshape(self.n, 1, DIM, DIM)
        self.stack = torch.cat([self.stack[:, 1:], frame], dim=1)
        kind = self.kinds[self.ids]
        actions = np.full(self.n, -1, np.int64)
        actions[kind == RULE_BASED] = CHEAT_CODES
        rnd = kind == RANDOM
        actions[rnd] = random_action(self.seed_, self.g[rnd], self.acts)
        self.acts += 1
        ref = np.zeros((self.n, 3))
        mag = np.zeros((self.n, 3))
        for s in np.unique(kind[kind >= 0]):
            rows = np.flatnonzero(kind == s)
            x = self.stack[torch.from_numpy(rows).to(self.device)]
            ref[rows] = forward64(x, self.nets[int(s)]).cpu().numpy()
            mag[rows] = magnitude64(x, self.nets[int(s)]).cpu().numpy()
        return Step(self.ids.copy(), kind, actions, ref, mag)
