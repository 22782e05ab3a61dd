"""cPongTournament-v0 on the device against a rollout of the reference's OWN TournamentEnvWrapper + policy_serving.Policy
(tests/golden/tournament_synth.npz, oracle/gen_golden_tournament.py): opponent = RULE_BASED (action 999) and the
reference's two network classes carrying synthetic weights that this test re-creates from the same formula.

Checked per step: agent 0's observation (bit-exact), reward and done with the reference's (N, 1) shapes, and the
opponent: its logits against the reference's (fp32 tolerance) and its greedy action wherever the reference's logit margin
is not a near-tie.  The recorded opponent action is what is fed to the env (teacher forcing), so one flipped near-tie
cannot derail the comparison of everything after it.  Pins competitive_pong_env.py:9-53 + policy_serving.py:10-66: the
opponent sees the PREVIOUS step's obs[1]; its frame stack rolls on every call, is never reset on done and survives
reset_opponent; inputs / 255; argmax."""
import numpy as np
import pytest

from conftest import load_golden, reference_layout, synthetic_state_dict

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


class CheckedOpponent(object):
    def __init__(self, policy, g):
        self.policy, self.g, self.t, self.n_checked, self.n_flipped, self.worst = policy, g, 0, 0, 0, 0.0

    def __call__(self, obs):
        logits = self.policy.logits(obs).double().cpu().numpy()
        want = self.g["opp_logits"][self.t].astype(np.float64)
        self.worst = max(self.worst, float(np.abs(logits - want).max()))
        assert np.abs(logits - want).max() <= 2e-4 * max(1.0, float(np.abs(want).max())), (self.t, logits, want)
        srt = np.sort(want, axis=1)
        clear = (srt[:, -1] - srt[:, -2]) > 1e-3
        got = logits.argmax(axis=1)
        rec = self.g["opp_actions"][self.t]
        assert np.array_equal(got[clear], rec[clear]), (self.t, got, rec)
        self.n_checked += int(clear.sum())
        self.n_flipped += int((got != rec).sum())
        return torch.as_tensor(rec.astype(np.int32), device=self.policy.device)


def test_tournament_replays_reference_rollout():
    from competitive_rl_b200 import make_envs
    from competitive_rl_b200.builtin_policies import DevicePolicy
    g = load_golden("tournament_synth")
    T, N = g["actions"].shape
    env = make_envs("cPongTournament-v0", num_envs=N, resized_dim=42, log_dir=None, serves=g["serves"])
    assert tuple(env.observation_space.shape) == tuple(g["obs_space"]) and env.action_space.n == int(g["n_actions"])
    assert env.current_agent_name == "RULE_BASED" and "RULE_BASED" in env.get_agent_names() and "RANDOM" in env.get_agent_names()
    checked = {}
    for name, light in (("WEAK", True), ("STRONG", False)):
        pol = DevicePolicy(N, "", use_light_model=light, device=env.env.device)
        pol.model.load_state_dict(synthetic_state_dict(reference_layout("LightActorCritic" if light else "ActorCritic")),
                                  strict=True)
        checked[name] = CheckedOpponent(pol, g)
        env.agents[name] = checked[name]
        if name not in env.agent_names:
            env.agent_names.append(name)
    sched = dict(zip(g["schedule_t"].tolist(), [str(s) for s in g["schedule_name"]]))
    o = env.reset()
    assert o.dtype == torch.uint8 and np.array_equal(o.cpu().numpy(), g["obs0"][0])
    for t in range(T):
        if t in sched:
            env.reset_opponent(sched[t])
        assert env.current_agent_name == str(g["agent_at"][t])
        for c in checked.values():
            c.t = t
        o, r, d, info = env.step(g["actions"][t])
        assert tuple(r.shape) == (N, 1) and tuple(d.shape) == (N, 1)
        assert np.array_equal(o.cpu().numpy(), g["obs0"][t + 1]), t
        assert np.array_equal(r.cpu().numpy(), g["rew"][t]) and np.array_equal(d.cpu().numpy(), g["done"][t]), t
    assert int(g["done"].sum()) >= 1                       # the opponents' stacks lived through a done without a reset
    for name, c in checked.items():
        print("%s: %d actions checked, %d near-tie flips, worst logit error %.2e" % (name, c.n_checked, c.n_flipped, c.worst))
        assert c.n_checked > 50 and c.n_flipped <= 2
    env.env.check()
    env.close()
