"""CPU checks of the per-env opponent pool's host side: the LightActorCritic flat image the kernel loads
(builtin_policies.pack_light_actor_critic) and the refusal of ActorCritic layouts."""
import numpy as np
import pytest

from conftest import reference_layout, synthetic_state_dict

torch = pytest.importorskip("torch")


def test_pack_order_is_the_reference_state_dict_order():
    from competitive_rl_b200.builtin_policies import (LIGHT_ACTOR_CRITIC_FLOATS, LIGHT_ACTOR_CRITIC_LAYOUT, LightActorCritic,
                                                      pack_light_actor_critic)
    for key in ("LightActorCritic", "checkpoint-weak.pkl", "checkpoint-medium.pkl"):
        assert [(n, tuple(s)) for n, s in LIGHT_ACTOR_CRITIC_LAYOUT] == reference_layout(key)
    assert list(LightActorCritic().state_dict()) == [n for n, _ in LIGHT_ACTOR_CRITIC_LAYOUT]
    assert sum(int(np.prod(s)) for _, s in LIGHT_ACTOR_CRITIC_LAYOUT) == LIGHT_ACTOR_CRITIC_FLOATS
    sd = synthetic_state_dict(reference_layout("LightActorCritic"))
    flat = pack_light_actor_critic(sd)
    assert flat.dtype == torch.float32 and tuple(flat.shape) == (LIGHT_ACTOR_CRITIC_FLOATS,)
    k = 0
    for name, shape in reference_layout("LightActorCritic"):     # parameter by parameter, row-major, in file order
        n = int(np.prod(shape))
        assert torch.equal(flat[k:k + n], sd[name].reshape(-1)), name
        k += n


def test_pack_round_trip():
    from competitive_rl_b200.builtin_policies import LightActorCritic, pack_light_actor_critic, unpack_light_actor_critic
    torch.manual_seed(0)
    net = LightActorCritic()
    flat = pack_light_actor_critic(net)
    back = unpack_light_actor_critic(flat)
    ref = net.state_dict()
    assert list(back) == list(ref)
    for name in ref:
        assert torch.equal(back[name], ref[name]), name
    other = LightActorCritic()
    other.load_state_dict(back, strict=True)
    assert torch.equal(pack_light_actor_critic({"model": other.state_dict()}), flat)   # checkpoint-dict form
    with pytest.raises(ValueError):
        unpack_light_actor_critic(flat[:-1])


def test_actor_critic_layouts_are_refused():
    from competitive_rl_b200.builtin_policies import ActorCritic, pack_light_actor_critic
    with pytest.raises(ValueError, match="ActorCritic"):
        pack_light_actor_critic(synthetic_state_dict(reference_layout("ActorCritic")))
    with pytest.raises(ValueError, match="ActorCritic"):
        pack_light_actor_critic(ActorCritic())
    bad = synthetic_state_dict(reference_layout("LightActorCritic"))
    bad["actor_linear.weight"] = torch.zeros(4, 1600)
    with pytest.raises(ValueError, match="shape"):
        pack_light_actor_critic(bad)
    del bad["actor_linear.bias"]
    with pytest.raises(ValueError, match="not a LightActorCritic"):
        pack_light_actor_critic(bad)


class _FakeDouble(object):
    """Enough of a 42x42 cPongDouble vec-env for the wrapper's argument checks (which run before any device work)."""
    dim, c, f32, ring, first_env = 42, 1, False, False, 0
    device = torch.device("cpu")
    observation_space = (None, None)
    action_space = (None, None)


def test_wrapper_refuses_actor_critic_and_unknown_opponents(tmp_path):
    from competitive_rl_b200.builtin_policies import ActorCritic
    from competitive_rl_b200.tournament import TournamentEnvWrapper
    torch.save({"model": ActorCritic().state_dict()}, str(tmp_path / "checkpoint-strong.pkl"))
    w = TournamentEnvWrapper(_FakeDouble(), 4, resource_dir=str(tmp_path))
    assert "STRONG" in w.get_agent_names()
    with pytest.raises(ValueError, match="ActorCritic"):
        w.set_opponents(pool=["RULE_BASED", "STRONG"])
    with pytest.raises(ValueError, match="ActorCritic"):
        w.add_opponent("SNAPSHOT", ActorCritic().state_dict())
    with pytest.raises(ValueError, match="unknown opponent"):
        w.set_opponents(pool=["RULE_BASED", "NOBODY"])
    with pytest.raises(ValueError, match="distinct"):
        w.set_opponents(pool=["RANDOM", "RANDOM"])
    assert not w.per_env
    narrow = _FakeDouble()
    narrow.dim = 84
    with pytest.raises(ValueError, match="resized_dim=42"):
        TournamentEnvWrapper(narrow, 4).set_opponents(pool=["RANDOM"])
