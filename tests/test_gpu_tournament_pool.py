"""Per-env opponents of cPongTournament-v0 (TournamentEnvWrapper.set_opponents, csrc/pong_opponent.cu) on the device.

1. the reference rollout of tests/golden/tournament_synth.npz from t = 40 on, every env on WEAK in per-env mode;
2. a mixed pool against torch LightActorCritic networks fed from a host-kept per-env stack;
3. resampling on done: which envs change, zero weights, same-seed and sharded reproducibility;
4. the per-opponent episode statistics against a host tally;
5. reset_opponent returns to the untouched uniform (torch) mode."""
import os

import numpy as np
import pytest

from conftest import load_golden, reference_layout, synthetic_state_dict

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TOL = 2e-4
MARGIN = 1e-3


def variant_state_dict(a, b):
    """LightActorCritic weights unlike the fixture's: parameter k, element i = float32(0.08 * sin(a * i + b * k + 1))."""
    sd = {}
    for k, (name, shape) in enumerate(reference_layout("LightActorCritic")):
        i = np.arange(int(np.prod(shape)), dtype=np.float64)
        sd[name] = torch.from_numpy((0.08 * np.sin(a * i + b * k + 1.0)).astype(np.float32).reshape(shape))
    return sd


@pytest.fixture
def resources(tmp_path):
    """A resource directory with checkpoint-weak.pkl (the fixture's synthetic weights) and checkpoint-medium.pkl."""
    torch.save({"model": synthetic_state_dict(reference_layout("LightActorCritic"))}, str(tmp_path / "checkpoint-weak.pkl"))
    torch.save({"model": variant_state_dict(0.23, 2.0)}, str(tmp_path / "checkpoint-medium.pkl"))
    return str(tmp_path)


def torch_net(sd, dev):
    from competitive_rl_b200.builtin_policies import LightActorCritic
    net = LightActorCritic().to(dev)
    net.load_state_dict(sd)
    net.requires_grad_(False)
    return net


@torch.no_grad()
def torch_logits(net, stack_u8):
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        return net(stack_u8.float())[0].double().cpu().numpy()


def check_logits(got, want, actions):
    """fp32 tolerance on the logits; the action must equal the argmax wherever the margin is not a near-tie.
    Returns (actions checked, near-tie flips)."""
    assert np.abs(got - want).max() <= TOL * max(1.0, float(np.abs(want).max())), (got, want)
    srt = np.sort(want, axis=1)
    clear = (srt[:, -1] - srt[:, -2]) > MARGIN
    ref = want.argmax(axis=1)
    assert np.array_equal(actions[clear], ref[clear]), (actions, ref)
    return int(clear.sum()), int((actions != ref).sum())


def make_tournament(n, seed=3, **kw):
    from competitive_rl_b200 import make_envs
    return make_envs("cPongTournament-v0", num_envs=n, resized_dim=42, log_dir=None, seed=seed, **kw)


def late_game(w, rows=None):
    """Put the envs (all, or `rows`) at num_rounds 20 of 21 so that their next point ends the episode."""
    st = w.env.get_state().cpu().numpy()
    rows = np.arange(len(st)) if rows is None else rows
    st[rows, 8] = 20
    st[rows, 6] = np.minimum(st[rows, 6], 10)
    st[rows, 7] = np.minimum(st[rows, 7], 10)
    w.env.set_state(st)


def learner_actions(n, t_max, seed):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 3, (t_max, n)).astype(np.int32)
    hold = rng.random((t_max, n)) < 0.6
    for t in range(1, t_max):
        a[t][hold[t]] = a[t - 1][hold[t]]
    return a


def test_per_env_replays_reference_rollout():
    """tournament_synth: RULE_BASED through reset_opponent for t < 40, then per-env mode with every env on WEAK (the
    fixture's synthetic weights).  The handle is driven with its logits output; the env is stepped with the recorded
    opponent actions (teacher forcing).  The fixture's WEAK stack is zero before t = 40, as per-env mode's is on entry."""
    g = load_golden("tournament_synth")
    T, N = g["actions"].shape
    w = make_tournament(N, serves=g["serves"])
    w.add_opponent("WEAK", synthetic_state_dict(reference_layout("LightActorCritic")))
    o = w.reset()
    assert np.array_equal(o.cpu().numpy(), g["obs0"][0])
    for t in range(40):
        assert str(g["agent_at"][t]) == "RULE_BASED"
        o, r, d, _ = w.step(g["actions"][t])
        assert np.array_equal(o.cpu().numpy(), g["obs0"][t + 1]), t
    w.set_opponents(assignment=["WEAK"] * N, pool=["WEAK"])
    assert w.per_env and w.opponent_ids.cpu().tolist() == [0] * N
    dev = w.env.device
    logits = torch.full((N, 3), float("nan"), dtype=torch.float32, device=dev)
    both = torch.zeros((N, 2), dtype=torch.int32, device=dev)
    checked = flipped = 0
    for t in range(40, 90):
        assert str(g["agent_at"][t]) == "WEAK"
        w._opp.act(w.env._obs[1], None, None, False, both, logits)
        got = logits.double().cpu().numpy()
        acts = both[:, 1].cpu().numpy()
        c, _ = check_logits(got, g["opp_logits"][t].astype(np.float64), acts)
        checked, flipped = checked + c, flipped + int((acts != g["opp_actions"][t]).sum())
        obs, r, d, _ = w.env.step(np.stack([g["actions"][t], g["opp_actions"][t]], axis=1).astype(np.int32))
        assert np.array_equal(obs[0].cpu().numpy(), g["obs0"][t + 1]), t
        assert np.array_equal(r[:, :1].cpu().numpy(), g["rew"][t]) and np.array_equal(d[:, :1].cpu().numpy(), g["done"][t]), t
    print("per-env WEAK: %d actions checked, %d near-tie flips" % (checked, flipped))
    assert checked > 50 and flipped <= 2
    w.env.check()
    w.close()


def test_mixed_pool_against_torch(resources):
    """N = 512, pool RULE_BASED / RANDOM / WEAK / MEDIUM / an added network, random assignment, 220 steps with dones.
    Every network env against torch on a host-kept stack; RULE_BASED exactly 999; RANDOM in {0, 1, 2} and, like every
    other action, identical in a second wrapper with the same seed."""
    N, T = 512, 220
    pool = ["RULE_BASED", "RANDOM", "WEAK", "MEDIUM", "SNAPSHOT"]
    added = variant_state_dict(0.41, -1.3)
    ws = []
    for _ in range(2):
        w = make_tournament(N, seed=9, resource_dir=resources)
        w.add_opponent("SNAPSHOT", added)
        w.reset()
        late_game(w)
        ws.append(w)
    dev = ws[0].env.device
    assign = np.random.default_rng(4).integers(0, len(pool), N)
    for w in ws:
        w.set_opponents(assignment=assign.tolist(), pool=pool, seed=77)
        w.opponent_logits = torch.zeros((N, 3), dtype=torch.float32, device=dev)
    assert np.array_equal(ws[0].opponent_ids.cpu().numpy(), assign)
    sds = {"WEAK": synthetic_state_dict(reference_layout("LightActorCritic")), "MEDIUM": variant_state_dict(0.23, 2.0),
           "SNAPSHOT": added}
    nets = {k: torch_net(sd, dev) for k, sd in sds.items()}
    rows = {k: np.flatnonzero(assign == pool.index(k)) for k in pool}
    assert all(len(r) > 50 for r in rows.values())
    stack = torch.zeros((N, 4, 42, 42), dtype=torch.uint8)
    acts_all = learner_actions(N, T, 5)
    checked = flipped = dones = 0
    seen_random = set()
    for t in range(T):
        stack = torch.cat([stack[:, 1:], ws[0].env._obs[1].cpu()], dim=1)
        outs = [w.step(acts_all[t]) for w in ws]
        opp = [w._both[:, 1].cpu().numpy() for w in ws]
        assert np.array_equal(opp[0], opp[1]), t
        for o0, o1 in zip(outs[0][:3], outs[1][:3]):
            assert torch.equal(o0, o1), t
        dones += int(outs[0][2].sum())
        got = ws[0].opponent_logits.double().cpu().numpy()
        assert np.all(opp[0][rows["RULE_BASED"]] == 999)
        ra = opp[0][rows["RANDOM"]]
        assert np.all((ra >= 0) & (ra <= 2))
        seen_random.update(ra.tolist())
        for k in ("WEAK", "MEDIUM", "SNAPSHOT"):
            want = torch_logits(nets[k], stack[rows[k]].to(dev))
            c, f = check_logits(got[rows[k]], want, opp[0][rows[k]])
            checked, flipped = checked + c, flipped + f
    print("mixed pool: %d network actions checked, %d near-tie flips, %d dones" % (checked, flipped, dones))
    assert seen_random == {0, 1, 2}
    assert dones >= N // 4 and checked > 0.9 * T * sum(len(rows[k]) for k in ("WEAK", "MEDIUM", "SNAPSHOT"))
    for w in ws:
        w.env.check()
        w.close()


def run_ids(ws, acts, T):
    """Step the wrappers `ws`, shards of one batch in env order, with that batch's learner actions; returns, per step,
    every shard's opponent ids used on that step and its dones."""
    ids, dones = [], []
    for t in range(T):
        if t % 50 == 0:
            for w in ws:
                late_game(w)
        outs, step_ids = [], []
        k = 0
        for w in ws:
            n = w.num_envs
            outs.append(w.step(acts[t][k:k + n]))
            step_ids.append(w.opponent_ids.cpu().numpy())
            k += n
        ids.append(step_ids)
        dones.append([o[2].cpu().numpy().reshape(-1) for o in outs])
    return ids, dones


def test_resampling_on_done(resources):
    """Ids change only in envs whose previous step was done; a zero weight is never drawn; the same seed gives the same
    id sequence; two shards of N/2 reproduce one N shard."""
    N, T = 256, 160
    pool = ["RULE_BASED", "RANDOM", "WEAK", "MEDIUM"]
    weights = [1.0, 2.0, 1.5, 0.0]
    acts = learner_actions(N, T, 8)
    groups = []
    for shards in ((0, N), (0, N), (0, N // 2, N)):
        g = []
        for a, b in zip(shards[:-1], shards[1:]):
            w = make_tournament(b - a, seed=13, first_env=a, resource_dir=resources)
            w.reset()
            w.set_opponents(pool=pool, weights=weights, resample_on_done=True, seed=21)
            g.append(w)
        groups.append(g)
    seqs = []
    for g in groups:
        ids, dones = run_ids(g, acts, T)
        seqs.append((np.array([np.concatenate(s) for s in ids]), np.array([np.concatenate(d) for d in dones])))
    ids, dones = seqs[0]
    assert (ids != 3).all()                                       # weight 0: MEDIUM never drawn
    changed = ids[1:] != ids[:-1]
    assert not (changed & ~dones[:-1]).any()                      # only envs done on the previous step redraw
    assert changed.sum() > 50 and dones[:-1].sum() > N
    assert set(np.unique(ids).tolist()) == {0, 1, 2}
    assert np.array_equal(seqs[1][0], ids) and np.array_equal(seqs[1][1], dones)      # same seed
    assert np.array_equal(seqs[2][0], ids) and np.array_equal(seqs[2][1], dones)      # sharded
    for g in groups:
        for w in g:
            w.close()


def test_opponent_stats_match_host_tally(resources):
    """opponent_stats() against a tally of rewards, dones and opponent_ids read back every step.  An episode that ends
    on step t is credited at step t + 1 (by that step's kernel launch), so the last step's dones are not counted."""
    N, T = 256, 160
    pool = ["RULE_BASED", "RANDOM", "WEAK", "MEDIUM"]
    w = make_tournament(N, seed=17, resource_dir=resources)
    w.reset()
    w.set_opponents(pool=pool, resample_on_done=True, seed=5)
    acts = learner_actions(N, T, 2)
    ret = np.zeros(N)
    tally = np.zeros((len(pool), 4), np.int64)
    for t in range(T):
        if t % 50 == 0:
            late_game(w)
        _, r, d, _ = w.step(acts[t])
        ids = w.opponent_ids.cpu().numpy()
        ret += r.cpu().numpy().reshape(-1)
        d = d.cpu().numpy().reshape(-1)
        if t < T - 1:
            for i in np.flatnonzero(d):
                tally[ids[i], 0] += 1
                tally[ids[i], 1 if ret[i] > 0 else 2 if ret[i] == 0 else 3] += 1
        ret[d] = 0
    st = w.opponent_stats()
    got = np.array([[st[k]["episodes"], st[k]["wins"], st[k]["draws"], st[k]["losses"]] for k in pool])
    print("stats", st)
    assert np.array_equal(got, tally)
    assert tally[:, 0].sum() > N and (tally[:, 1].sum() > 0) and (tally[:, 3].sum() > 0)
    w.close()


def test_reset_opponent_returns_to_uniform_mode(resources):
    """After per-env steps, reset_opponent("WEAK") plays through the torch DevicePolicy exactly as before: its stack and
    actions equal those of a fresh DevicePolicy fed the same observations."""
    from competitive_rl_b200.builtin_policies import DevicePolicy
    N = 64
    w = make_tournament(N, seed=1, resource_dir=resources)
    w.reset()
    w.set_opponents(pool=["RULE_BASED", "RANDOM", "WEAK"], resample_on_done=True)
    acts = learner_actions(N, 60, 3)
    for t in range(20):
        w.step(acts[t])
    w.reset_opponent("WEAK")
    assert not w.per_env and w.current_agent_name == "WEAK"
    fresh = DevicePolicy(N, os.path.join(resources, "checkpoint-weak.pkl"), True, w.env.device)
    for t in range(20, 60):
        want = fresh(w.prev_opponent_obs)
        w.step(acts[t])
        assert torch.equal(w.current_agent.stack, fresh.stack), t
        with torch.no_grad(), torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
            got = w.current_agent.model(w.current_agent.stack)[0].argmax(dim=1).to(torch.int32)
        assert torch.equal(got, want), t
    w.close()
