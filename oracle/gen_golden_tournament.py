"""Generate tests/golden/tournament_synth.npz: the reference's OWN TournamentEnvWrapper (pong/competitive_pong_env.py:9-53)
driving its OWN policy_serving.Policy objects (utils/policy_serving.py:10-66, networks of utils/network.py) over the
reference's cPongDouble vec-env, with serves injected.  Build container only.

The reference's trained checkpoints (resources/pong/checkpoint-*.pkl) are its data and are not vendored, so the network
opponents of this fixture carry SYNTHETIC weights given by a closed formula (synthetic_state_dict in tests/conftest.py) that the GPU
test re-creates: what is pinned is everything around the weights -- the opponent sees obs[1] of the PREVIOUS step, its
own FrameStackTensor is rolled on every call and never reset on done or on reset_opponent, inputs / 255, greedy argmax,
action 999 for RULE_BASED, the (N, 1) reward / done shapes -- and the two network definitions themselves.
(tests/test_builtin_policies.py replays this fixture on the CPU oracle to check both network classes without a GPU.)

Two modifications to the reference objects, both forced by the tree itself: get_builtin_agent_names is narrowed (the
wrapper's constructor builds every agent and asserts on the STRONG / ALPHA_PONG checkpoint files, which the reference
does not ship), and the network agents' weights are overwritten with the synthetic ones."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))
import ref_loader  # noqa: E402
from conftest import synthetic_state_dict  # noqa: E402
from pong_oracle import make_serve_table  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def main():
    import torch
    torch.set_num_threads(1)
    ref_loader.install()
    import competitive_rl.utils as U
    from competitive_rl.utils.network import ActorCritic, LightActorCritic
    U.ActorCritic, U.LightActorCritic = ActorCritic, LightActorCritic
    import importlib.util
    spec = importlib.util.spec_from_file_location("_ref_utils_utils", os.path.join(ref_loader.REFERENCE_ROOT, "competitive_rl", "utils", "utils.py"))
    try:
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        U.FrameStackTensor = m.FrameStackTensor
    except Exception as exc:   # utils.py pulls optional packages at import: take the class text alone
        raise SystemExit("cannot import the reference's utils.py: %r" % (exc,))
    import competitive_rl.pong.builtin_policies as BP
    import competitive_rl.pong.competitive_pong_env as CP
    from competitive_rl.utils.policy_serving import Policy
    names = ["RANDOM", "WEAK", "MEDIUM", "RULE_BASED"]
    CP.get_builtin_agent_names = lambda: names
    N, T = 3, 180
    serves = make_serve_table(N, 200, seed=21)
    envs, inj = ref_loader.make_reference_vec_env("cPongDouble-v0", N, serves, resized_dim=42, frame_stack=None)
    w = CP.TournamentEnvWrapper(envs, N)
    assert isinstance(w.agents["WEAK"], Policy)
    # synthetic weights; "STRONG" = the reference's ActorCritic-based Policy, built the way get_compute_action_function does
    w.agents["STRONG"] = Policy(BP.single_obs_space, BP.single_act_space, N, "", use_light_model=False)
    w.agent_names.append("STRONG")
    for n in ("WEAK", "MEDIUM", "STRONG"):
        w.agents[n].model.load_state_dict(synthetic_state_dict([(k, p.shape) for k, p in w.agents[n].model.state_dict().items()]))
    schedule = [(0, "RULE_BASED"), (40, "WEAK"), (90, "STRONG"), (130, "WEAK"), (155, "RULE_BASED")]
    rng = np.random.default_rng(77)
    actions = rng.integers(0, 3, (T, N)).astype(np.int32)
    hold = rng.random((T, N)) < 0.6
    for t in range(1, T):
        actions[t][hold[t]] = actions[t - 1][hold[t]]
    obs0 = [np.array(w.reset())]
    rews, dones, opp_actions, opp_logits, agent_at = [], [], [], [], []
    orig_call = Policy.__call__
    last = {}

    def recording_call(self, obs):
        a = orig_call(self, obs)
        with torch.no_grad():
            last["logits"] = self.model(self.frame_stack.get())[0].numpy().copy()
        last["action"] = np.asarray(a).reshape(-1).copy()
        return a
    Policy.__call__ = recording_call
    try:
        for t in range(T):
            for t0, name in schedule:
                if t == t0:
                    w.reset_opponent(name)
            last.clear()
            o, r, d, info = w.step(actions[t])
            obs0.append(np.array(o))
            rews.append(np.array(r))
            dones.append(np.array(d))
            agent_at.append(w.current_agent_name)
            if "action" in last:
                opp_actions.append(last["action"])
                opp_logits.append(last["logits"])
            else:
                opp_actions.append(np.full(N, 999))
                opp_logits.append(np.zeros((N, 3), np.float32))
    finally:
        Policy.__call__ = orig_call
    path = os.path.join(OUT, "tournament_synth.npz")
    np.savez_compressed(path, serves=serves, actions=actions, obs0=np.array(obs0, np.uint8), rew=np.array(rews), done=np.array(dones),
                        opp_actions=np.array(opp_actions, np.int32), opp_logits=np.array(opp_logits, np.float32),
                        agent_at=np.array(agent_at), schedule_t=np.array([s[0] for s in schedule]),
                        schedule_name=np.array([s[1] for s in schedule]),
                        obs_space=np.array(w.observation_space.shape), n_actions=w.action_space.n)
    print("tournament_synth: obs0 %s rew %s done %s dones=%d opponent action histogram %s  %d KiB" % (
        np.array(obs0).shape, np.array(rews).shape, np.array(dones).shape, int(np.array(dones).sum()),
        np.unique(np.array(opp_actions), return_counts=True), os.path.getsize(path) // 1024))


if __name__ == "__main__":
    main()
