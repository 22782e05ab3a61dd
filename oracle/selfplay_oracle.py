"""Host model of the self-play mode of the per-env opponent kernel (csrc/pong_opponent.cu, include/crl_b200.h
crl_pong_opp_set_selfplay / crl_pong_opp_act_selfplay) -- TEST INFRASTRUCTURE ONLY.  Written from the header's
semantics; league mode's model is league_oracle's, the float64 critic, sampler and log-prob are learner_oracle's.

  LEARNER          CRL_PONG_OPP_LEARNER, a learner seat in a pairing table
  learner_u        the learner's uniform draw u = r32 * 2^-32 of a seat: tag 4 in seat 0, tag 5 in seat 1
  HostSelfPlay     a host model of one handle in self-play mode
"""
import numpy as np
import torch

from learner_oracle import LEARNER_TAG, value64, value_magnitude64
from league_oracle import MAX_PAIRS, HostLeague, random_action
from opponent_oracle import CHEAT_CODES, DIM, RANDOM, RULE_BASED, forward64, magnitude64, opp_rand

LEARNER = -3                         # CRL_PONG_OPP_LEARNER
SEAT1_TAG = 5


def learner_u(seed, g, ctr, seat):
    """The learner's draw of global env(s) g at act count ctr in `seat`: r32 * 2^-32 (float64, exact) of the tag-4 stream
    in seat 0 (learner mode's) and of the tag-5 stream in seat 1."""
    r = opp_rand(seed, g, LEARNER_TAG if seat == 0 else SEAT1_TAG, ctr)
    return np.asarray(r, dtype=np.float64) * 2.0 ** -32


class SelfPlayStep(object):
    """What one act_selfplay of HostSelfPlay computed, per env and seat (axis 1 = seat 0, seat 1): the pairing, each
    seat's kind (LEARNER, RULE_BASED, RANDOM or a network slot), the action of each RULE_BASED / RANDOM seat (-1
    elsewhere), the float64 logits and magnitudes [n, 2, 3] of network and learner seats (0 elsewhere), the learner
    seats' float64 value and its magnitude and their draw u [n, 2] (0 elsewhere), and both stacks the seats acted on
    [n, 2, 4, 42, 42] (uint8, on the model's device)."""

    def __init__(self, pairing, kind, actions, ref, mag, value, value_mag, u, stack):
        self.pairing, self.kind, self.actions, self.ref, self.mag = pairing, kind, actions, ref, mag
        self.value, self.value_mag, self.u, self.stack = value, value_mag, u, stack
        self.learner = kind == LEARNER
        self.net = kind >= 0


class HostSelfPlay(HostLeague):
    """Host model of a crl_pong_opp handle in self-play mode (include/crl_b200.h), written from the header's semantics:
    league mode's pairings, stacks and tally (HostLeague), where a seat may be LEARNER.  A learner seat's ring is
    zeroed before the push when the previous step's done is set, and before the push that follows a restart; a pool
    seat's ring only by set_selfplay and restart(clear=True)."""

    def __init__(self, n, seed, first_env=0, device="cpu"):
        super().__init__(n, seed, first_env, device)
        self.learner = None
        self.pending_clear = False

    def load_learner(self, params):
        self.learner = torch.as_tensor(params, dtype=torch.float32).reshape(-1).clone()

    def set_selfplay(self, pairs):
        p = np.asarray(pairs, np.int64).reshape(-1, 2)
        assert 1 <= len(p) <= MAX_PAIRS and (((p >= 0) & (p < len(self.kinds))) | (p == LEARNER)).all()
        self.pairs = p
        self.pairing = self.g % len(p)
        self.stats = np.zeros((len(p), 4), np.int64)
        self.ret[:] = 0
        for st in self.stacks:
            st.zero_()
        self.pending_clear = False

    def restart(self, clear):
        super().restart(clear)
        self.pending_clear = True

    def act_selfplay(self, obs0, obs1, rew=None, done=None):
        """obs0, obs1 uint8 [n, 42, 42] (any device); rew float32 [n, 2] and done [n] as numpy, or both None."""
        assert self.learner is not None
        seats = self.pairs[self.pairing]                           # [n, 2] pool index or LEARNER
        if rew is not None:
            r = (self.ret + np.asarray(rew, np.float32)[:, 0]).astype(np.float32)
            d = np.asarray(done).astype(bool)
            p, rd = self.pairing[d], r[d]
            np.add.at(self.stats, (p, 0), 1)
            np.add.at(self.stats, (p, np.where(rd > 0, 1, np.where(rd == 0, 2, 3))), 1)
            r[d] = 0
            self.ret = r
        d = np.asarray(done).astype(bool) if done is not None else np.zeros(self.n, bool)
        for seat, obs in enumerate((obs0, obs1)):
            zero = (seats[:, seat] == LEARNER) & (d | self.pending_clear)
            self.stacks[seat][torch.from_numpy(zero).to(self.device)] = 0
            frame = torch.as_tensor(obs).to(self.device).reshape(self.n, 1, DIM, DIM)
            self.stacks[seat] = torch.cat([self.stacks[seat][:, 1:], frame], dim=1)
        self.pending_clear = False
        kind = np.where(seats == LEARNER, LEARNER, self.kinds[np.where(seats == LEARNER, 0, seats)])
        actions = np.full((self.n, 2), -1, np.int64)
        ref, mag = np.zeros((self.n, 2, 3)), np.zeros((self.n, 2, 3))
        value, value_mag, u = np.zeros((self.n, 2)), np.zeros((self.n, 2)), np.zeros((self.n, 2))
        for seat in range(2):
            k = kind[:, seat]
            a = actions[:, seat]
            a[k == RULE_BASED] = CHEAT_CODES
            rnd = k == RANDOM
            a[rnd] = random_action(self.seed_, self.g[rnd], self.acts, seat)
            for s in np.unique(k[(k >= 0) | (k == LEARNER)]):
                rows = np.flatnonzero(k == s)
                x = self.stacks[seat][torch.from_numpy(rows).to(self.device)]
                params = self.learner if s == LEARNER else self.nets[int(s)]
                ref[rows, seat] = forward64(x, params).cpu().numpy()
                mag[rows, seat] = magnitude64(x, params).cpu().numpy()
                if s == LEARNER:
                    value[rows, seat] = value64(x, params).cpu().numpy()
                    value_mag[rows, seat] = value_magnitude64(x, params).cpu().numpy()
                    u[rows, seat] = learner_u(self.seed_, self.g[rows], self.acts, seat)
        self.acts += 1
        stack = torch.stack([st.clone() for st in self.stacks], dim=1)
        return SelfPlayStep(self.pairing.copy(), kind, actions, ref, mag, value, value_mag, u, stack)
