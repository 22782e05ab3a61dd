"""CPU checks of league mode's host side: the host model HostLeague (oracle/league_oracle.py) against the header's
semantics and against HostOpponents, and the argument checks of evaluate.evaluate_pool_in_batch (all made before any
device work)."""
import numpy as np
import pytest

from conftest import reference_layout, synthetic_state_dict

torch = pytest.importorskip("torch")
import league_oracle as lo  # noqa: E402
import opponent_oracle as oo  # noqa: E402

N = 24


def frames(n, gen):
    return torch.randint(0, 256, (n, oo.DIM, oo.DIM), generator=gen, dtype=torch.uint8)


@pytest.mark.parametrize("first_env,num_pairs", [(0, 5), (2 ** 33 + 3, 7), (11, 1), (0, 24)])
def test_pairing_is_global_index_mod_p(first_env, num_pairs):
    m = lo.HostLeague(N, 1, first_env)
    m.set_pool([oo.RULE_BASED, oo.RANDOM])
    pairs = np.random.default_rng(num_pairs).integers(0, 2, (num_pairs, 2))
    m.set_pairs(pairs)
    g = first_env + np.arange(N)
    assert np.array_equal(m.pairing, [int(x) % num_pairs for x in g])
    gen = torch.Generator().manual_seed(0)
    step = m.act_pairs(frames(N, gen), frames(N, gen))
    assert np.array_equal(step.pairing, m.pairing)
    want = np.array([[oo.RULE_BASED, oo.RANDOM][k] for k in pairs[m.pairing].reshape(-1)]).reshape(N, 2)
    assert np.array_equal(step.kind, want)


def test_seat_random_streams_differ():
    """RANDOM in both seats: seat 1 is crl_pong_opp_act's stream (tag 1), seat 0 a stream of its own (tag 3)."""
    n, seed, first = 4096, 77, 5
    m = lo.HostLeague(n, seed, first)
    m.set_pool([oo.RANDOM])
    m.set_pairs([(0, 0)])
    gen = torch.Generator().manual_seed(1)
    agree = 0
    for t in range(3):
        step = m.act_pairs(frames(n, gen), frames(n, gen))
        g = first + np.arange(n)
        assert np.array_equal(step.actions[:, 1], oo.random_action(seed, g, t))
        assert np.array_equal(step.actions[:, 0], lo.random_action(seed, g, t, seat=0))
        assert set(np.unique(step.actions).tolist()) == {0, 1, 2}
        agree += int((step.actions[:, 0] == step.actions[:, 1]).sum())
    assert abs(agree / (3 * n) - 1 / 3) < 0.03                 # independent uniform draws agree a third of the time
    # seat 1 is the stream of the per-env opponents' RANDOM
    g = first + np.arange(n)
    assert np.array_equal(lo.random_action(seed, g, 4), oo.random_action(seed, g, 4))


def test_pairing_tally_on_a_hand_made_sequence():
    """Four envs, two pairings (env i plays pairing i % 2).  Rewards are seat 0's (column 0); an episode is credited by
    the act_pairs that receives the done."""
    m = lo.HostLeague(4, 0)
    m.set_pool([oo.RULE_BASED, oo.RANDOM])
    m.set_pairs([(0, 1), (1, 0)])
    z = np.zeros((4, oo.DIM, oo.DIM), np.uint8)
    m.act_pairs(z, z)
    seq = [  # (rew of seat 0 per env, done per env)
        ([1, 0, -1, 0], [0, 0, 0, 0]),
        ([0, -1, 0, 0], [1, 0, 0, 1]),      # env 0 ends at +1 (win, pairing 0), env 3 ends at 0 (draw, pairing 1)
        ([-1, 0, 0, 1], [0, 1, 1, 0]),      # env 1 ends at -1 (loss, pairing 1), env 2 ends at -1 (loss, pairing 0)
        ([1, 1, 0, -1], [1, 1, 0, 1]),      # env 0: -1 + 1 = 0 draw; env 1: +1 win; env 3: +1 - 1 = 0 draw
        ([0, 0, -1, 0], [0, 0, 0, 0]),      # env 2's next episode starts at -1
    ]
    for rew, done in seq:
        r = np.stack([np.array(rew, np.float32), np.full(4, 5.0, np.float32)], axis=1)   # column 1 is not counted
        m.act_pairs(z, z, r, np.array(done, bool))
    assert m.stats.tolist() == [[3, 1, 1, 1], [4, 1, 2, 1]]
    assert m.ret.tolist() == [0, 0, -1, 0]


def test_seat_one_matches_host_opponents():
    """Every pairing with the same seat-1 entry: seat 1's actions, logits and magnitudes equal HostOpponents' for an
    assignment of that entry, and seat 0 sees its own stack."""
    n, seed, first = 40, 3, 17
    gen = torch.Generator().manual_seed(5)
    nets = [oo.random_params(gen) for _ in range(2)]
    league = lo.HostLeague(n, seed, first)
    single = oo.HostOpponents(n, seed, first)
    for s, img in enumerate(nets):
        league.load_net(s, img)
        single.load_net(s, img)
    pool = [oo.RULE_BASED, 0, oo.RANDOM, 1]
    league.set_pool(pool)
    single.set_pool(pool)
    for seat1 in (1, 2, 3):
        league.set_pairs([(0, seat1), (1, seat1), (2, seat1), (3, seat1), (1, seat1)])
        single.assign(np.full(n, seat1))
        single.restart(True)
        stack0 = torch.zeros((n, 4, oo.DIM, oo.DIM), dtype=torch.uint8)
        for t in range(6):
            o0, o1 = frames(n, gen), frames(n, gen)
            a = league.act_pairs(o0, o1)
            b = single.act(o1)
            stack0 = torch.cat([stack0[:, 1:], o0[:, None]], dim=1)
            assert np.array_equal(a.actions[:, 1], b.actions) and np.array_equal(a.ref[:, 1], b.ref)
            assert np.array_equal(a.mag[:, 1], b.mag) and np.array_equal(a.net[:, 1], b.net)
            rows = np.flatnonzero(a.kind[:, 0] == 0)
            assert np.array_equal(a.ref[rows, 0], oo.forward64(stack0[rows], nets[0]).numpy())


# ------------------------------------------------------------------------------------------- evaluate_pool_in_batch
class _FakeDouble(object):
    """Enough of a 42x42 cPongDouble vec-env for evaluate_pool_in_batch's argument checks (made before device work)."""
    dim, c, f32, ring, first_env, n_agents = 42, 1, False, False, 0, 2
    device = torch.device("cpu")

    def __init__(self, num_envs=64, **kw):
        self.num_envs = num_envs
        for k, v in kw.items():
            setattr(self, k, v)


def evaluate(pool, envs=None, **kw):
    from competitive_rl_b200.evaluate import evaluate_pool_in_batch
    return evaluate_pool_in_batch(pool, envs if envs is not None else _FakeDouble(), 1, **kw)


@pytest.mark.parametrize("attrs", [dict(dim=84), dict(c=4), dict(f32=True), dict(ring=True), dict(n_agents=1)])
def test_pool_evaluation_refuses_other_envs(attrs):
    with pytest.raises(ValueError, match="resized_dim=42"):
        evaluate(["RULE_BASED", "RANDOM"], _FakeDouble(**attrs))


def test_pool_evaluation_argument_checks(tmp_path):
    from competitive_rl_b200.builtin_policies import ActorCritic
    torch.save({"model": ActorCritic().state_dict()}, str(tmp_path / "checkpoint-strong.pkl"))
    light = synthetic_state_dict(reference_layout("LightActorCritic"))
    with pytest.raises(ValueError, match="unknown opponent"):
        evaluate(["RULE_BASED", "NOBODY"])
    with pytest.raises(ValueError, match="ActorCritic"):
        evaluate(["RULE_BASED", "STRONG"], resource_dir=str(tmp_path))
    with pytest.raises(ValueError, match="ActorCritic"):
        evaluate(["RULE_BASED", "SNAP"], networks={"SNAP": ActorCritic().state_dict()})
    with pytest.raises(ValueError, match="not a network"):
        evaluate(["RULE_BASED"], networks={"RANDOM": light})
    with pytest.raises(ValueError, match="distinct"):
        evaluate(["RANDOM", "RANDOM"])
    with pytest.raises(ValueError, match="distinct"):
        evaluate([])
    with pytest.raises(ValueError, match="at most 8 networks"):
        evaluate(["N%d" % k for k in range(9)], networks={"N%d" % k: light for k in range(9)})
    for bad in ([(0, 2)], [(-1, 0)], [("RANDOM", "NOBODY")], [(0, 1, 1)]):
        with pytest.raises(ValueError, match="pool indices|not in the pool|seat 0, seat 1"):
            evaluate(["RULE_BASED", "RANDOM"], pairs=bad)
    with pytest.raises(ValueError, match="1 to 256 pairings"):
        evaluate(["RULE_BASED", "RANDOM"], _FakeDouble(1000), pairs=[(0, 1)] * 257)
    with pytest.raises(ValueError, match="1 to 256 pairings"):
        evaluate(["RULE_BASED", "RANDOM"], pairs=[])
    with pytest.raises(ValueError, match="at least as many envs"):
        evaluate(["RULE_BASED", "RANDOM"], _FakeDouble(3))          # 4 pairings by default
    with pytest.raises(ValueError, match="at least as many envs"):
        evaluate(["RULE_BASED"], _FakeDouble(5), pairs=[(0, 0)] * 6)
