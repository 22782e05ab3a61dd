"""Built-in tournament opponents (competitive-rl_b200/builtin_policies.py): the two network definitions against the
reference's own networks (utils/network.py) and shipped checkpoints -- their state-dict layouts
(tests/golden/reference_networks.json) and the logits they recorded in tests/golden/tournament_synth.npz (CPU) -- and
the device policy against a CPU evaluation of the same weights (GPU)."""
import numpy as np
import pytest

from conftest import load_golden, reference_layout, synthetic_state_dict

torch = pytest.importorskip("torch")


@pytest.mark.parametrize("name", ["weak", "medium"])
def test_light_network_matches_reference_checkpoint(name, tmp_path):
    """A checkpoint with the layout of the reference's checkpoint-<name>.pkl (its "model" state dict: every parameter
    name and shape) loads strictly into LightActorCritic, and DevicePolicy, which loads the real file the same way,
    computes exactly what the network computes with those weights."""
    from competitive_rl_b200.builtin_policies import DevicePolicy, LightActorCritic
    sd = synthetic_state_dict(reference_layout("checkpoint-%s.pkl" % name))
    ours = LightActorCritic((4, 42, 42), 3)
    ours.load_state_dict(sd, strict=True)
    path = str(tmp_path / ("checkpoint-%s.pkl" % name))
    torch.save({"model": sd, "optimizer": {}}, path)
    pol = DevicePolicy(64, path, use_light_model=True, device="cpu")
    x = torch.from_numpy(np.random.default_rng(0).integers(0, 256, (64, 4, 1, 42, 42)).astype(np.float32))
    for k in range(4):                           # four frames fill the policy's stack
        got = pol.logits(x[:, k])
    with torch.no_grad():
        want = ours(x[:, :, 0])[0]
    assert torch.equal(got, want)


def test_full_network_matches_reference_definition(atlas):
    """Replays the fixture's rollout on the CPU oracle (bit-exact to the reference's frames, checked on agent 0's
    observation every step) with the recorded opponent actions, and feeds the opponent's observations to LightActorCritic
    (WEAK) and ActorCritic (STRONG).  Their weights are the fixture's synthetic ones, built on the reference networks'
    own state-dict layouts and loaded strictly, so every parameter name, shape and the parameter order are pinned.
    WEAK's logits equal the recorded ones bit for bit; STRONG's 11x11x32 convolution sums in a library-chosen order, so
    its logits are held to a few fp32 ulps."""
    from competitive_rl_b200.builtin_policies import DevicePolicy
    from pong_oracle import PongOracleVec
    g = load_golden("tournament_synth")
    T, N = g["actions"].shape
    pols = {}
    for name, light in (("WEAK", True), ("STRONG", False)):
        pols[name] = DevicePolicy(N, "", use_light_model=light, device="cpu")
        layout = reference_layout("LightActorCritic" if light else "ActorCritic")
        pols[name].model.load_state_dict(synthetic_state_dict(layout), strict=True)
    orc = PongOracleVec("cPongDouble-v0", N, 42, None, 21, atlas, g["serves"])
    obs = orc.reset()
    assert np.array_equal(obs[0], g["obs0"][0])
    checked = {name: 0 for name in pols}
    for t in range(T):
        name = str(g["agent_at"][t])
        if name in pols:            # the opponent acts on the previous step's obs[1]; its stack rolls only when it acts
            got = pols[name].logits(torch.from_numpy(obs[1])).numpy()
            want = g["opp_logits"][t]
            if name == "WEAK":
                assert np.array_equal(got, want), (t, got, want)
            else:
                assert np.abs(got - want).max() <= 2e-6 * max(1.0, float(np.abs(want).max())), (t, got, want)
            checked[name] += 1
        obs, rew, done, _ = orc.step(np.stack([g["actions"][t], g["opp_actions"][t]], axis=1))
        assert np.array_equal(obs[0], g["obs0"][t + 1]) and np.array_equal(rew[:, :1], g["rew"][t]), t
        assert np.array_equal(done, g["done"][t][:, 0]), t
    orc.close()
    assert checked == {"WEAK": 75, "STRONG": 40}


def test_agent_names_follow_available_checkpoints(tmp_path):
    from competitive_rl_b200.builtin_policies import LightActorCritic, get_builtin_agent_names
    assert get_builtin_agent_names(str(tmp_path)) == ["RANDOM", "RULE_BASED"] or "WEAK" in get_builtin_agent_names(str(tmp_path))
    torch.save({"model": LightActorCritic().state_dict()}, str(tmp_path / "checkpoint-weak.pkl"))
    names = get_builtin_agent_names(str(tmp_path))
    assert "WEAK" in names and "RULE_BASED" in names and "RANDOM" in names


@pytest.mark.gpu
def test_device_policy_and_tournament_with_network_opponent(tmp_path):
    from competitive_rl_b200 import make_envs
    from competitive_rl_b200.builtin_policies import ActorCritic, DevicePolicy, LightActorCritic
    torch.manual_seed(3)
    torch.save({"model": LightActorCritic().state_dict()}, str(tmp_path / "checkpoint-weak.pkl"))
    torch.save({"model": ActorCritic().state_dict()}, str(tmp_path / "checkpoint-strong.pkl"))
    N = 256
    t = make_envs("cPongTournament-v0", num_envs=N, resized_dim=42, log_dir=None, seed=4, resource_dir=str(tmp_path))
    assert {"RANDOM", "RULE_BASED", "WEAK", "STRONG"} <= set(t.get_agent_names())
    o = t.reset()
    for name, light in (("WEAK", True), ("STRONG", False)):
        t.reset_opponent(name)
        gpu_pol = t.current_agent
        assert isinstance(gpu_pol, DevicePolicy)
        cpu_pol = DevicePolicy(N, str(tmp_path / ("checkpoint-%s.pkl" % name.lower())), light, "cpu")
        cpu_pol.stack.copy_(gpu_pol.stack.cpu())
        agree = total = 0
        for k in range(25):
            opp_obs = t.prev_opponent_obs.clone()
            expect = cpu_pol.logits(opp_obs.cpu())                       # same stack update, same weights, on the host
            o, r, d, info = t.step(np.random.randint(0, 3, N))
            assert tuple(o.shape) == (N, 1, 42, 42) and tuple(r.shape) == (N, 1) and tuple(d.shape) == (N, 1)
            assert torch.allclose(gpu_pol.stack.cpu(), cpu_pol.stack)     # the opponent's own frame stack
            got = gpu_pol.model(gpu_pol.stack)[0].cpu()
            assert torch.allclose(got, expect, rtol=1e-3, atol=1e-4)
            top2 = expect.topk(2, dim=1).values
            clear = (top2[:, 0] - top2[:, 1]) > 1e-3
            agree += int((got.argmax(1) == expect.argmax(1))[clear].sum())
            total += int(clear.sum())
        assert total > 0 and agree == total
    t.close()
