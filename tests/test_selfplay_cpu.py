"""CPU checks of self-play mode's host side: the learner's seat-1 draws (Philox tag 5), the host model HostSelfPlay of
oracle/selfplay_oracle.py against the header's ring semantics and against HostLeague / HostLearner, the pairing parser
builtin_policies.resolve_pairs, and the argument checks of SelfPlayEnvWrapper (all made before any device work)."""
import numpy as np
import pytest

from conftest import reference_layout, synthetic_state_dict

torch = pytest.importorskip("torch")
import league_oracle as lgo  # noqa: E402
import learner_oracle as lro  # noqa: E402
import opponent_oracle as oo  # noqa: E402
import selfplay_oracle as so  # noqa: E402

L, RB, RND = so.LEARNER, oo.RULE_BASED, oo.RANDOM


def frames(n, gen):
    return torch.randint(0, 256, (n, oo.DIM, oo.DIM), generator=gen, dtype=torch.uint8)


def test_seat_one_draws_are_the_tag_5_philox_stream():
    """Seat 0 draws from learner mode's stream (tag 4), seat 1 from tag 5: exact r32 * 2^-32, the same from scalars,
    arrays and any slicing of the envs, and independent of the other streams."""
    seed, ctr = 0x5EED5EED1234, 23
    g = np.arange(2 ** 33 - 5, 2 ** 33 + 4000, dtype=np.int64)
    u1 = so.learner_u(seed, g, ctr, 1)
    assert np.array_equal(u1, oo.opp_rand(seed, g, 5, ctr).astype(np.float64) * 2.0 ** -32)
    assert np.array_equal(so.learner_u(seed, g, ctr, 0), lro.learner_u(seed, g, ctr))
    assert all(so.learner_u(seed, int(g[k]), ctr, 1) == u1[k] for k in (0, 11, 3999))
    assert np.array_equal(np.concatenate([so.learner_u(seed, g[:777], ctr, 1), so.learner_u(seed, g[777:], ctr, 1)]), u1)
    r5 = oo.opp_rand(seed, g, 5, ctr)
    for tag in (1, 2, 3, 4):
        assert (oo.opp_rand(seed, g, tag, ctr) != r5).mean() > 0.999
    assert (so.learner_u(seed, g, ctr + 1, 1) != u1).mean() > 0.999
    assert (u1 >= 0).all() and (u1 < 1).all()


def make_model(n, seed, first_env, pairs, nets):
    m = so.HostSelfPlay(n, seed, first_env)
    for s, img in enumerate(nets):
        m.load_net(s, img)
    m.set_pool([RB, RND] + list(range(len(nets))))
    m.load_learner(nets[-1])
    m.set_selfplay(pairs)
    return m


def test_host_selfplay_ring_semantics():
    """Learner seats' rings are zeroed before the push that follows a done and after restart(False); pool seats' rings
    are never cleared on done or restart(False); restart(True) and set_selfplay clear both."""
    n = 8
    gen = torch.Generator().manual_seed(0)
    img = oo.random_params(torch.Generator().manual_seed(1))
    pairs = [(L, L), (L, 2), (0, L), (2, 1)]           # env i plays pairing i % 4
    m = make_model(n, 3, 0, pairs, [img])
    learner = np.array([[p[0] == L, p[1] == L] for p in pairs] * 2)
    obs = [[frames(n, gen) for _ in range(10)] for _ in range(2)]
    z = np.zeros(n, bool)
    rew = np.zeros((n, 2), np.float32)
    done = np.array([1, 1, 1, 1, 0, 0, 0, 0], bool)
    for t in range(5):
        args = (None, None) if t == 0 else (rew, done if t == 3 else z)
        st = m.act_selfplay(obs[0][t], obs[1][t], *args)
    for i in range(n):
        for seat in range(2):
            x = st.stack[i, seat]
            if learner[i, seat] and done[i]:     # the done passed at t = 3: frames 3 and 4 only
                assert not x[:2].any() and torch.equal(x[2], obs[seat][3][i]) and torch.equal(x[3], obs[seat][4][i])
            else:
                assert all(torch.equal(x[k], obs[seat][1 + k][i]) for k in range(4)), (i, seat)
    m.restart(False)                   # learner seats restart at the next act; pool seats keep their frames
    st = m.act_selfplay(obs[0][5], obs[1][5])
    for seat in range(2):
        lr = torch.from_numpy(learner[:, seat])
        assert not st.stack[lr, seat, :3].any() and torch.equal(st.stack[:, seat, 3], obs[seat][5])
        assert torch.equal(st.stack[~lr, seat, :3], torch.stack([o[~lr] for o in obs[seat][2:5]], dim=1))
    st = m.act_selfplay(obs[0][6], obs[1][6], rew, z)     # the pending clear applied once
    assert torch.equal(st.stack[:, :, 2], torch.stack([obs[0][5], obs[1][5]], dim=1))
    m.restart(True)
    assert not any(s.any() for s in m.stacks)
    m.act_selfplay(obs[0][7], obs[1][7])
    m.set_selfplay(pairs)
    assert not any(s.any() for s in m.stacks)


def test_host_selfplay_against_league_and_learner_models():
    """Pool-only pairings play as HostLeague; a learner in seat 0 sees HostLearner's ring, logits, value and draws; the
    kinds, actions and tally follow the table."""
    n, seed, first = 24, 5, 2 ** 33 + 1
    gen = torch.Generator().manual_seed(2)
    nets = [oo.random_params(gen) for _ in range(3)]
    pool = [RB, RND, 0, 1]
    pairs = [(0, 2), (L, 1), (3, L), (1, 3), (L, L), (2, 2)]
    m = so.HostSelfPlay(n, seed, first)
    lg = lgo.HostLeague(n, seed, first)
    lr = lro.HostLearner(n, seed, first)
    for s in range(2):
        for h in (m, lg, lr):
            h.load_net(s, nets[s])
    for h in (m, lg, lr):
        h.set_pool(pool)
    m.load_learner(nets[2])
    lr.load_learner(nets[2])
    lr.assign(np.zeros(n, np.int64))
    m.set_selfplay(pairs)
    lg.set_pairs([(p[0] if p[0] != L else 0, p[1] if p[1] != L else 0) for p in pairs])
    rng = np.random.default_rng(0)
    rew = done = None
    for t in range(6):
        o0, o1 = frames(n, gen), frames(n, gen)
        a, b, c = m.act_selfplay(o0, o1, rew, done), lg.act_pairs(o0, o1, rew, done), lr.act_learner(o0, o1, rew, done)
        assert np.array_equal(a.pairing, b.pairing)
        seats = np.array(pairs)[a.pairing]
        assert np.array_equal(a.learner, seats == L)
        pool_only = ~a.learner.any(axis=1)
        assert np.array_equal(a.actions[pool_only], b.actions[pool_only])
        assert np.allclose(a.ref[pool_only], b.ref[pool_only], rtol=1e-12, atol=1e-12)
        s0 = a.learner[:, 0]
        assert torch.equal(a.stack[torch.from_numpy(s0), 0], c.stack[torch.from_numpy(s0)])
        assert np.allclose(a.ref[s0, 0], c.ref[s0], rtol=1e-12, atol=1e-12)
        assert np.allclose(a.value[s0, 0], c.value[s0], rtol=1e-12, atol=1e-12)
        assert np.array_equal(a.u[s0, 0], c.u[s0])
        s1 = a.learner[:, 1]
        assert np.array_equal(a.u[s1, 1], so.learner_u(seed, m.g[s1], t, 1))
        assert (a.value[~a.learner] == 0).all() and (a.u[~a.learner] == 0).all()
        assert (a.actions[a.learner] == -1).all()
        rew = np.stack([rng.integers(-1, 2, n), rng.normal(size=n)], axis=1).astype(np.float32)
        done = rng.random(n) < 0.3
    assert np.array_equal(m.stats, lg.stats) and m.stats[:, 0].sum() > 0


# ---------------------------------------------------------------------------------------------------- resolve_pairs
def test_resolve_pairs():
    from competitive_rl_b200.builtin_policies import resolve_pairs
    pool = ["RULE_BASED", "RANDOM", "WEAK"]
    assert resolve_pairs([("RANDOM", 0), (2, "WEAK")], pool) == [[1, 0], [2, 2]]
    assert resolve_pairs([("LEARNER", "WEAK"), ("LEARNER", "LEARNER")], pool, learner=True) == [[L, 2], [L, L]]
    with pytest.raises(ValueError, match="'LEARNER' is not in the pool"):
        resolve_pairs([("LEARNER", "WEAK")], pool)                   # league mode has no learner
    with pytest.raises(ValueError, match="'NOBODY' is not in the pool"):
        resolve_pairs([("LEARNER", "NOBODY")], pool, learner=True)
    with pytest.raises(ValueError, match="reserved"):
        resolve_pairs([("LEARNER", 0)], pool + ["LEARNER"], learner=True)
    for bad in ([(0, 3)], [(-1, 0)], [(L, 0)]):                     # an index is never a learner seat
        with pytest.raises(ValueError, match=r"pool indices must be in \[0, 3\)"):
            resolve_pairs(bad, pool, learner=True)
    with pytest.raises(ValueError, match="seat 0, seat 1"):
        resolve_pairs([("LEARNER",)], pool, learner=True)
    for p in ([], [("LEARNER", "LEARNER")] * 257):
        with pytest.raises(ValueError, match="1 to 256 pairings"):
            resolve_pairs(p, pool, learner=True)


# ---------------------------------------------------------------------------------------------------- the wrapper
class _FakeDouble(object):
    """Enough of a 42x42 cPongDouble vec-env for SelfPlayEnvWrapper's argument checks (made before device work)."""
    dim, c, f32, ring, first_env, n_agents = 42, 1, False, False, 0, 2
    device = torch.device("cpu")

    def __init__(self, num_envs=64, **kw):
        self.num_envs = num_envs
        for k, v in kw.items():
            setattr(self, k, v)


@pytest.mark.parametrize("attrs", [dict(dim=84), dict(c=4), dict(f32=True), dict(ring=True), dict(n_agents=1)])
def test_wrapper_refuses_other_envs(attrs):
    from competitive_rl_b200.selfplay import SelfPlayEnvWrapper
    with pytest.raises(ValueError, match="resized_dim=42, frame_stack=None and uint8"):
        SelfPlayEnvWrapper(_FakeDouble(**attrs))


def test_wrapper_argument_checks(tmp_path):
    from competitive_rl_b200.builtin_policies import ActorCritic, LightActorCritic
    from competitive_rl_b200.selfplay import SelfPlayEnvWrapper
    w = SelfPlayEnvWrapper(_FakeDouble(), resource_dir=str(tmp_path))
    light = synthetic_state_dict(reference_layout("LightActorCritic"))
    with pytest.raises(RuntimeError, match="set_league first"):
        w.set_learner(LightActorCritic())
    with pytest.raises(RuntimeError, match="set_league, then set_learner"):
        w.learner_step()
    with pytest.raises(RuntimeError, match="set_league first"):
        w.learner_seats
    with pytest.raises(RuntimeError, match="set_league first"):
        w.pair_stats()
    for name in ("RULE_BASED", "RANDOM"):
        with pytest.raises(ValueError, match="not a network"):
            w.add_opponent(name, light)
    with pytest.raises(ValueError, match="reserved"):
        w.add_opponent("LEARNER", light)
    with pytest.raises(ValueError, match="ActorCritic"):
        w.add_opponent("SNAP", ActorCritic().state_dict())
    torch.save({"model": ActorCritic().state_dict()}, str(tmp_path / "checkpoint-strong.pkl"))
    for k in range(9):
        w.add_opponent("N%d" % k, light)
    with pytest.raises(ValueError, match="unknown opponent"):
        w.set_league([("LEARNER", "NOBODY")])
    with pytest.raises(ValueError, match="ActorCritic"):
        w.set_league([("STRONG", "LEARNER")])
    with pytest.raises(ValueError, match="a seat is 'LEARNER' or a pool name"):
        w.set_league([("LEARNER", 0)])
    with pytest.raises(ValueError, match="seat 0, seat 1"):
        w.set_league([("LEARNER", "N0", "N1")])
    with pytest.raises(ValueError, match="at most 8 networks"):
        w.set_league([("LEARNER", "N%d" % k) for k in range(9)])
    with pytest.raises(ValueError, match="1 to 16 distinct names"):
        w.set_league([("N%d" % (k % 8), x) for k, x in enumerate(["RULE_BASED", "RANDOM"] + ["X%d" % k for k in range(15)])])
    with pytest.raises(ValueError, match="1 to 256 pairings"):
        w.set_league([("LEARNER", "N0")] * 257)
    with pytest.raises(ValueError, match="1 to 256 pairings"):
        w.set_league([])
    assert w._opp is None and w._pool is None           # nothing was created or loaded
