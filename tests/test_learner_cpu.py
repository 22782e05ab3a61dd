"""CPU checks of learner mode's host side: the float64 critic of oracle/learner_oracle.py against the torch module, the
host sampler's Philox draws and inverse CDF, the host model HostLearner against the header's ring semantics, and the
argument checks of TournamentEnvWrapper.set_learner / learner_step (all made before any device work)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
import learner_oracle as lo  # noqa: E402
import opponent_oracle as oo  # noqa: E402


def frames(n, gen):
    return torch.randint(0, 256, (n, oo.DIM, oo.DIM), generator=gen, dtype=torch.uint8)


@pytest.mark.parametrize("scale", [1.0, 30.0])
def test_critic_matches_the_module_in_float64(scale):
    from competitive_rl_b200.builtin_policies import LightActorCritic, unpack_light_actor_critic
    gen = torch.Generator().manual_seed(int(scale))
    img = oo.random_params(gen, scale)
    net = LightActorCritic().double()
    net.load_state_dict({k: v.double() for k, v in unpack_light_actor_critic(img).items()})
    x = torch.randint(0, 256, (96, 4, oo.DIM, oo.DIM), generator=gen, dtype=torch.uint8)
    x[:8] = 0
    x[8:16] = 255
    with torch.no_grad():
        logits, value = net(x.double())
    v = lo.value64(x, img)
    assert torch.allclose(v, value[:, 0], rtol=1e-12, atol=1e-12 * scale)
    assert torch.allclose(oo.forward64(x, img), logits, rtol=1e-12, atol=1e-12 * scale)
    mag = lo.value_magnitude64(x, img)
    assert (mag >= v.abs() - 1e-12).all() and (mag > 0).all()


def test_learner_draws_are_the_tag_4_philox_stream():
    """u = r32 * 2^-32 of stream (g, tag 4) at the act count: the same from scalars and arrays, from any slicing of the
    envs (shards), and a stream of its own (tags 1-3 are RANDOM's and the draws')."""
    seed, ctr = 0x5EED5EED1234, 17
    g = np.arange(2 ** 33 - 5, 2 ** 33 + 4000, dtype=np.int64)
    u = lo.learner_u(seed, g, ctr)
    r = oo.opp_rand(seed, g, 4, ctr)
    assert np.array_equal(u, r.astype(np.float64) * 2.0 ** -32)
    assert all(lo.learner_u(seed, int(g[k]), ctr) == u[k] for k in (0, 7, 3999))
    assert np.array_equal(np.concatenate([lo.learner_u(seed, g[:1234], ctr), lo.learner_u(seed, g[1234:], ctr)]), u)
    for tag in (1, 2, 3):
        assert (oo.opp_rand(seed, g, tag, ctr) != r).mean() > 0.999
    assert (lo.learner_u(seed, g, ctr + 1) != u).mean() > 0.999
    assert (u >= 0).all() and (u < 1).all()
    # r32 = 0 and r32 = 2^32 - 1 map to 0 and to just below 1, exactly
    assert lo.sample64([[0.0, 0.0, 0.0]], [0.0])[0] == 0
    assert lo.sample64([[0.0, 0.0, 0.0]], [(2 ** 32 - 1) * 2.0 ** -32])[0] == 2


def test_inverse_cdf_boundaries_and_log_prob():
    lg = np.log(np.array([[0.25, 0.5, 0.25]] * 6))
    u = np.array([0.0, 0.25 - 2 ** -40, 0.25, 0.75 - 2 ** -40, 0.75, 1 - 2 ** -32])
    assert lo.sample64(lg, u).tolist() == [0, 0, 1, 1, 2, 2]
    assert np.allclose(lo.boundary_distance(lg, u), [0.25, 2 ** -40, 0, 2 ** -40, 0, 0.25 - 2 ** -32])
    assert np.allclose(lo.logprob64(lg, [0, 1, 2, 0, 1, 2]), np.log([0.25, 0.5, 0.25, 0.25, 0.5, 0.25]), atol=1e-15)
    # large logits: no overflow, and a certain action has log-prob 0
    big = np.array([[1e4, -1e4, 3.0]])
    assert lo.sample64(big, [0.999999])[0] == 0 and lo.logprob64(big, [0])[0] == 0.0


def test_sampled_actions_follow_the_softmax():
    """Over 200 000 envs with one set of logits, the inverse-CDF actions of the Philox draws have the softmax's
    frequencies (chi-square, 2 degrees of freedom, p > 1e-4: statistic below 18.4)."""
    n = 200000
    lg = np.tile([[0.3, -1.2, 1.1]], (n, 1))
    a = lo.sample64(lg, lo.learner_u(99, np.arange(n), 5))
    p = np.exp(lg[0]) / np.exp(lg[0]).sum()
    counts = np.bincount(a, minlength=3)
    chi2 = (((counts - n * p) ** 2) / (n * p)).sum()
    assert chi2 < 18.4, (counts, n * p)


def test_host_learner_ring_semantics():
    """The ring pushes agent 0's frames oldest -> newest, zeroes an env's ring before the push that follows its done,
    is zeroed on entering learner mode (after set_pool) and by restart(False) in learner mode; seat 1 is HostOpponents."""
    n, seed = 6, 3
    gen = torch.Generator().manual_seed(0)
    m = lo.HostLearner(n, seed)
    ref = oo.HostOpponents(n, seed)
    img = oo.random_params(torch.Generator().manual_seed(1))
    for h in (m, ref):
        h.load_net(0, img)
        h.set_pool([oo.RULE_BASED, oo.RANDOM, 0])
        h.assign(np.arange(n) % 3)
    m.load_learner(img)
    obs0 = [frames(n, gen) for _ in range(8)]
    obs1 = [frames(n, gen) for _ in range(8)]
    rew = np.zeros((n, 2), np.float32)
    done = np.array([0, 1, 0, 0, 1, 0], bool)
    for t in range(5):
        args = (None, None) if t == 0 else (rew, done if t == 3 else np.zeros(n, bool))
        st = m.act_learner(obs0[t], obs1[t], *args)
        want = ref.act(obs1[t], *args)
        assert np.array_equal(st.opp.actions, want.actions) and np.array_equal(st.opp.ids, want.ids)
        assert np.array_equal(st.opp.ref, want.ref)
        assert np.allclose(st.ref, oo.forward64(st.stack, img).numpy()) and st.value.shape == (n,)
        assert np.array_equal(st.u, lo.learner_u(seed, np.arange(n), t))
    x = st.stack
    for i in range(n):
        if done[i]:      # the done of step 2 was passed at t = 3: the rings hold frames 3 and 4 only
            assert not x[i, :2].any() and torch.equal(x[i, 2], obs0[3][i]) and torch.equal(x[i, 3], obs0[4][i])
        else:
            assert all(torch.equal(x[i, k], obs0[1 + k][i]) for k in range(4))
    m.restart(False)
    assert not m.ring.any()
    st = m.act_learner(obs0[5], obs1[5])
    assert not st.stack[:, :3].any() and torch.equal(st.stack[:, 3], obs0[5])
    m.set_pool([oo.RULE_BASED])
    m.assign()
    m.restart(False)                 # not in learner mode: the ring stays
    assert m.ring.any()
    st = m.act_learner(obs0[6], obs1[6])
    assert not st.stack[:, :3].any() and torch.equal(st.stack[:, 3], obs0[6])


class _FakeDouble(object):
    dim, c, f32, ring, first_env = 42, 1, False, False, 0
    device = torch.device("cpu")
    observation_space = (None, None)
    action_space = (None, None)


class _FakeHandle(object):
    def __init__(self):
        self.images = []

    def load_learner(self, image):
        self.images.append(image)


def test_set_learner_argument_checks():
    from competitive_rl_b200.builtin_policies import ActorCritic, LightActorCritic, pack_light_actor_critic
    from competitive_rl_b200.tournament import TournamentEnvWrapper
    w = TournamentEnvWrapper(_FakeDouble(), 4)
    net = LightActorCritic()
    with pytest.raises(RuntimeError, match="set_opponents first"):
        w.set_learner(net)
    with pytest.raises(RuntimeError, match="set_learner"):
        w.learner_step()
    w.per_env, w._opp = True, _FakeHandle()          # per-env mode without a device
    with pytest.raises(RuntimeError, match="set_learner"):
        w.learner_step()
    with pytest.raises(ValueError, match="ActorCritic"):
        w.set_learner(ActorCritic())
    with pytest.raises(ValueError, match="ActorCritic"):
        w.set_learner({"model": ActorCritic().state_dict()})
    bad = net.state_dict()
    del bad["critic_linear.bias"]
    with pytest.raises(ValueError, match="not a LightActorCritic"):
        w.set_learner(bad)
    assert w._opp.images == [] and w._sample is None
    want = pack_light_actor_critic(net)
    w.set_learner(net)
    w.set_learner(net.state_dict(), sample=False)
    w.set_learner({"model": net.state_dict()})
    assert len(w._opp.images) == 3 and all(torch.equal(im, want) for im in w._opp.images)
    assert w._sample is True
    w.reset_opponent("RANDOM")                         # uniform mode: no learner steps
    with pytest.raises(RuntimeError, match="set_learner"):
        w.learner_step()
