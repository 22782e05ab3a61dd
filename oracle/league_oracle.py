"""Host model of the league mode of the per-env opponent kernel (csrc/pong_opponent.cu, include/crl_b200.h
crl_pong_opp_set_pairs / crl_pong_opp_act_pairs / crl_pong_opp_get_pair_stats) -- TEST INFRASTRUCTURE ONLY.  Written from
the header's semantics; the Philox streams, the float64 network and the tolerance rule are opponent_oracle's.

  random_action   RANDOM's action of a seat: seat 1 draws from tag 1 (as crl_pong_opp_act), seat 0 from tag 3
  HostLeague      a host model of one handle in league mode
"""
import numpy as np
import torch

from opponent_oracle import CHEAT_CODES, DIM, RANDOM, RULE_BASED, forward64, magnitude64, opp_rand

MAX_PAIRS = 256                      # CRL_PONG_OPP_MAX_PAIRS


def random_action(seed, g, ctr, seat=1):
    """RANDOM's action of global env(s) g at act count ctr in `seat`: (r32 * 3) >> 32, in {0, 1, 2}.  Seat 1 is
    opponent_oracle.random_action's stream (tag 1); seat 0 has a stream of its own (tag 3)."""
    r = opp_rand(seed, g, 1 if seat == 1 else 3, ctr)
    if np.isscalar(r):
        return (r * 3) >> 32
    return ((r * np.uint64(3)) >> np.uint64(32)).astype(np.int64)


class LeagueStep(object):
    """What one act_pairs of HostLeague computed, per env and seat (axis 1 = seat 0, seat 1): the pairing, the kind of
    each seat's entry, the action of each non-network seat (-1 for network seats), and for network seats the float64
    logits and their magnitudes [n, 2, 3] (0 elsewhere, like the kernel's logits)."""

    def __init__(self, pairing, kind, actions, ref, mag):
        self.pairing, self.kind, self.actions, self.ref, self.mag = pairing, kind, actions, ref, mag
        self.net = kind >= 0


class HostLeague(object):
    """Host model of a crl_pong_opp handle in league mode (include/crl_b200.h, crl_pong_opp_set_pairs), written from the
    header's semantics: env g = first_env + i plays pairing g mod P; two [n, 4, 42, 42] uint8 stacks, oldest to newest,
    shifted on every push (seat 0 fed agent 0's frames, seat 1 agent 1's); the pairing tally counts seat 0's finished
    episodes.  `acts` is the handle's act count (every act or act_pairs since creation)."""

    def __init__(self, n, seed, first_env=0, device="cpu"):
        self.n, self.device = n, torch.device(device)
        self.seed_ = int(seed)
        self.g = int(first_env) + np.arange(n, dtype=np.int64)
        self.nets = {}
        self.kinds = self.pairs = self.pairing = None
        self.ret = np.zeros(n, np.float32)
        self.stats = None
        self.stacks = [torch.zeros((n, 4, DIM, DIM), dtype=torch.uint8, device=self.device) for _ in range(2)]
        self.acts = 0

    def seed(self, s):
        self.seed_ = int(s)

    def load_net(self, slot, params):
        self.nets[slot] = torch.as_tensor(params, dtype=torch.float32).reshape(-1).clone()

    def set_pool(self, kinds):
        self.kinds = np.asarray(kinds, np.int64)

    def set_pairs(self, pairs):
        self.pairs = np.asarray(pairs, np.int64).reshape(-1, 2)
        assert 1 <= len(self.pairs) <= MAX_PAIRS and ((self.pairs >= 0) & (self.pairs < len(self.kinds))).all()
        self.pairing = self.g % len(self.pairs)              # numpy's remainder has the divisor's sign: >= 0
        self.stats = np.zeros((len(self.pairs), 4), np.int64)
        self.ret[:] = 0
        for st in self.stacks:
            st.zero_()

    def restart(self, clear):
        self.ret[:] = 0
        if clear:
            for st in self.stacks:
                st.zero_()

    def act_pairs(self, obs0, obs1, rew=None, done=None):
        """obs0, obs1 uint8 [n, 42, 42] (any device); rew float32 [n, 2] and done [n] as numpy, or both None."""
        if rew is not None:
            r = (self.ret + np.asarray(rew, np.float32)[:, 0]).astype(np.float32)
            d = np.asarray(done).astype(bool)
            p, rd = self.pairing[d], r[d]
            np.add.at(self.stats, (p, 0), 1)
            np.add.at(self.stats, (p, np.where(rd > 0, 1, np.where(rd == 0, 2, 3))), 1)
            r[d] = 0
            self.ret = r
        for seat, obs in enumerate((obs0, obs1)):
            frame = torch.as_tensor(obs).to(self.device).reshape(self.n, 1, DIM, DIM)
            self.stacks[seat] = torch.cat([self.stacks[seat][:, 1:], frame], dim=1)
        kind = self.kinds[self.pairs[self.pairing]]              # [n, 2]
        actions = np.full((self.n, 2), -1, np.int64)
        ref = np.zeros((self.n, 2, 3))
        mag = np.zeros((self.n, 2, 3))
        for seat in range(2):
            k = kind[:, seat]
            a = actions[:, seat]
            a[k == RULE_BASED] = CHEAT_CODES
            rnd = k == RANDOM
            a[rnd] = random_action(self.seed_, self.g[rnd], self.acts, seat)
            for s in np.unique(k[k >= 0]):
                rows = np.flatnonzero(k == s)
                x = self.stacks[seat][torch.from_numpy(rows).to(self.device)]
                ref[rows, seat] = forward64(x, self.nets[int(s)]).cpu().numpy()
                mag[rows, seat] = magnitude64(x, self.nets[int(s)]).cpu().numpy()
        self.acts += 1
        return LeagueStep(self.pairing.copy(), kind, actions, ref, mag)
