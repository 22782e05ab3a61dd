"""League mode of the opponent kernel (csrc/pong_opponent.cu, crl_pong_opp_set_pairs / act_pairs / get_pair_stats): both
seats of every env played from a pool, against the float64 reference and the host model HostLeague of
oracle/league_oracle.py, and through the game with evaluate.evaluate_pool_in_batch.

1. accuracy sweep over N: net / net (same and different slots), net / RULE_BASED, RANDOM / net, RULE_BASED / RANDOM
   pairings; every network logit of both seats within 4 u M of forward64 on that seat's stack, the action rules, and
   RULE_BASED / RANDOM exactly as HostLeague;
2. a whole-handle scenario against HostLeague (16-entry pool with all 8 slots, P = 256 and a P that divides no N) with
   synthetic rewards and dones: actions, logits and the pairing table at every step;
3. two shards against one handle, bit for bit, and their tables adding up;
4. the mode rules and the C ABI's argument checks;
5. through the game: evaluate_pool_in_batch against a twin env driven by HostLeague, and a network pool driven by the
   kernel's own actions with both seats' logits checked against host-kept stacks."""
import ctypes

import numpy as np
import pytest

from conftest import reference_layout

torch = pytest.importorskip("torch")
import league_oracle as lo  # noqa: E402
import opponent_oracle as oo  # noqa: E402

pytestmark = pytest.mark.gpu

SENTINEL = -7
DEV = "cuda"
WORST = {"ratio": 0.0}
RB, RND = oo.RULE_BASED, oo.RANDOM


def ext():
    from competitive_rl_b200 import _native
    return _native.ext()


@pytest.fixture(scope="module")
def nets():
    """8 distinct random LightActorCritic images: slots 0-3 at PyTorch's init scale, 4-7 at 30x."""
    gen = torch.Generator().manual_seed(2026)
    return [oo.random_params(gen, 1.0 if s < 4 else 30.0) for s in range(oo.SLOTS)]


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    print("\nlargest |logit error| / (u M) of the league kernel: %.3f" % WORST["ratio"])


def frames(n, gen):
    """uint8 [n, 42, 42] on the device: env i always gets frames of one kind (random bytes, all 0, all 255, sparse
    Pong-like), redrawn on every call."""
    kind = torch.as_tensor((np.arange(n) * 7 + np.arange(n) // 64) % 4, device=DEV).view(n, 1, 1)
    out = torch.zeros((n, oo.DIM, oo.DIM), dtype=torch.uint8, device=DEV)
    for k, name in enumerate(oo.FRAME_KINDS):
        out = torch.where(kind == k, oo.synthetic_frames(name, n, gen, DEV), out)
    return out.contiguous()


def new_handle(n, seed, first_env, images, kinds, pairs):
    h = ext().PongOpponents(n, 0, seed, first_env)
    for k, img in enumerate(images):
        h.load_net(k, img)
    h.set_pool(torch.tensor(kinds, dtype=torch.int32), None)
    h.set_pairs(torch.tensor(pairs, dtype=torch.int32))
    return h


def new_model(n, seed, first_env, images, kinds, pairs):
    m = lo.HostLeague(n, seed, first_env, DEV)
    for k, img in enumerate(images):
        m.load_net(k, img)
    m.set_pool(kinds)
    m.set_pairs(pairs)
    return m


def act_pairs(h, n, obs0, obs1, rew=None, done=None):
    """One act_pairs; returns (logits float32 [n, 2, 3], actions int32 [n, 2])."""
    actions = torch.full((n, 2), SENTINEL, dtype=torch.int32, device=DEV)
    logits = torch.full((n, 2, 3), float("nan"), dtype=torch.float32, device=DEV)
    h.act_pairs(obs0, obs1, rew, done, actions, logits)
    return logits, actions


def check_step(logits, actions, step, where=""):
    """Both seats against one step of HostLeague: non-network seats exact (logits 0); network seats within TOL_ULPS u M,
    action = greedy of its own logits, = argmax(ref) where decided."""
    lg = logits.cpu().numpy()
    ac = actions.cpu().numpy()
    for seat in range(2):
        net = step.net[:, seat]
        other = ~net
        assert np.array_equal(ac[other, seat], step.actions[other, seat]), (where, seat)
        assert (lg[other, seat] == 0).all(), (where, seat)
        if net.any():
            got, a, ref, mag = lg[net, seat], ac[net, seat], step.ref[net, seat], step.mag[net, seat]
            ratio = oo.logit_ratio(got, ref, mag)
            WORST["ratio"] = max(WORST["ratio"], float(ratio.max()))
            bad = np.flatnonzero((ratio > oo.TOL_ULPS).any(axis=1))
            assert len(bad) == 0, (where, seat, np.flatnonzero(net)[bad[:5]], got[bad[:5]], ref[bad[:5]], ratio[bad[:5]])
            assert np.array_equal(a, oo.greedy(got)), (where, seat)
            dec = oo.decided(ref, mag)
            assert np.array_equal(a[dec], ref[dec].argmax(axis=1)), (where, seat)


def bits(t):
    return t.contiguous().view(torch.int32).cpu()


def wave_n(offset):
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count * 64 + offset


SWEEP_N = [1, 3, 64, 65, 100, "wave-1", "wave+1", 65536, 65573]
SWEEP_POOL = list(range(oo.SLOTS)) + [RB, RND]            # pool index k < 8 is slot k; 8 = RULE_BASED, 9 = RANDOM
SWEEP_PAIRS = [(0, 0), (1, 5), (6, 2), (3, 8), (9, 7), (8, 9), (4, 4), (7, 1), (2, 9), (8, 6), (5, 3), (9, 8), (2, 0)]


@pytest.mark.parametrize("n", SWEEP_N, ids=[str(v) for v in SWEEP_N])
def test_accuracy_sweep(nets, n):
    """Six acts (the ring wraps) with 13 pairings that put every slot in both seats."""
    if isinstance(n, str):
        n = wave_n(-1 if n.endswith("-1") else 1)
    seed, first = 0x1EA6, 5
    h = new_handle(n, seed, first, nets, SWEEP_POOL, SWEEP_PAIRS)
    m = new_model(n, seed, first, nets, SWEEP_POOL, SWEEP_PAIRS)
    gen = torch.Generator(device=DEV).manual_seed(n)
    for t in range(6):
        o0, o1 = frames(n, gen), frames(n, gen)
        step = m.act_pairs(o0, o1)
        lg, ac = act_pairs(h, n, o0, o1)
        check_step(lg, ac, step, "N %d act %d" % (n, t))
    h.close()


SCENARIO_POOL = [RND, RB, 0, 1, 2, 3, RND, 4, 5, 6, 7, RB, RND, RB, RND, 7]


@pytest.mark.parametrize("n,steps,num_pairs", [(1000, 200, 256), (1000, 200, 7), (40000, 40, 256), (40000, 40, 7)])
def test_handle_scenario_against_host_model(nets, n, steps, num_pairs):
    """A 16-entry pool with all 8 slots (RULE_BASED / RANDOM / slot 7 repeated), first_env 2^33 + 7, P = 256 (every
    ordered pairing, shuffled) or 7 (dividing neither N), random rewards with about 5 % dones; mid-run restart(False)
    and restart(True).  Actions and logits every step, the pairing table exactly at every step."""
    seed, first = 0xBEEF, 2 ** 33 + 7
    rng = np.random.default_rng(n + num_pairs)
    every = [(a, b) for a in range(16) for b in range(16)]
    pairs = [every[k] for k in rng.permutation(256)[:num_pairs]]
    h = new_handle(n, seed, first, nets, SCENARIO_POOL, pairs)
    m = new_model(n, seed, first, nets, SCENARIO_POOL, pairs)
    gen = torch.Generator(device=DEV).manual_seed(n)
    fresh = True
    for t in range(steps):
        if t in (steps // 2, steps * 3 // 4):
            h.restart(t == steps * 3 // 4)
            m.restart(t == steps * 3 // 4)
            fresh = True
        o0, o1 = frames(n, gen), frames(n, gen)
        if fresh:
            r = d = rew = done = None
        else:
            r = np.stack([rng.integers(-1, 2, n), rng.normal(size=n)], axis=1).astype(np.float32)
            d = rng.random(n) < 0.05
            rew, done = torch.from_numpy(r).to(DEV), torch.from_numpy(d).to(DEV)
        step = m.act_pairs(o0, o1, r, d)
        lg, ac = act_pairs(h, n, o0, o1, rew, done)
        fresh = False
        check_step(lg, ac, step, "N %d P %d step %d" % (n, num_pairs, t))
        got = np.array(h.pair_stats(num_pairs), np.int64).reshape(num_pairs, 4)
        assert np.array_equal(got, m.stats), t
    assert m.stats[:, 0].sum() > 0 and (m.stats[:, 0] > 0).sum() >= min(num_pairs, 200)
    h.close()


def test_shards_reproduce_one_handle(nets):
    """first_env 0 and an odd split: the two shards' actions and logits equal the single handle's bit for bit, and
    their pairing tables add up to its table."""
    n, half, steps, seed = 5001, 2347, 30, 99
    pool = [RB, 0, RND, 5, 2]
    pairs = [(1, 3), (3, 1), (0, 4), (4, 2), (2, 2), (1, 1), (4, 0), (3, 3), (2, 1), (0, 2), (4, 4), (1, 0), (3, 2)]
    hs = [new_handle(n, seed, 0, nets, pool, pairs), new_handle(half, seed, 0, nets, pool, pairs),
          new_handle(n - half, seed, half, nets, pool, pairs)]
    parts = [slice(0, n), slice(0, half), slice(half, n)]
    rng = np.random.default_rng(3)
    gen = torch.Generator(device=DEV).manual_seed(3)
    rew = done = None
    for t in range(steps):
        o0, o1 = frames(n, gen), frames(n, gen)
        outs = [act_pairs(h, p.stop - p.start, o0[p], o1[p], None if rew is None else rew[p],
                          None if done is None else done[p]) for h, p in zip(hs, parts)]
        assert torch.equal(bits(torch.cat([outs[1][0], outs[2][0]])), bits(outs[0][0])), t
        assert torch.equal(torch.cat([outs[1][1], outs[2][1]]), outs[0][1]), t
        rew = torch.from_numpy(rng.integers(-1, 2, (n, 2)).astype(np.float32)).to(DEV)
        done = torch.from_numpy(rng.random(n) < 0.1).to(DEV)
    got = [np.array(h.pair_stats(len(pairs)), np.int64).reshape(-1, 4) for h in hs]
    assert got[0][:, 0].sum() > 0 and np.array_equal(got[1] + got[2], got[0])
    for h in hs:
        h.close()


def test_mode_rules_and_c_abi_argument_checks(nets):
    """Each refusal returns its code and sets crl_last_error without launching anything; after a league run,
    set_pool + assign gives seat-1 results bit-identical to a fresh handle's."""
    from competitive_rl_b200 import _native
    lib = _native.load()
    vp = ctypes.c_void_p
    n = 8

    def expect(rc, code, text):
        assert rc == code, (rc, code, text)
        assert text in lib.crl_last_error().decode(), (lib.crl_last_error(), text)

    h = vp()
    assert lib.crl_pong_opp_create(n, 0, 1, 0, ctypes.byref(h)) == 0 and h.value
    img = nets[0].numpy().copy()
    assert lib.crl_pong_opp_load_net(h, 0, img.ctypes.data, img.size, None) == 0
    obs = torch.zeros(n * 1764 + 4, dtype=torch.uint8, device=DEV)
    rew = torch.zeros((n, 2), dtype=torch.float32, device=DEV)
    done = torch.zeros(n, dtype=torch.uint8, device=DEV)
    actions = torch.full((n, 2), SENTINEL, dtype=torch.int32, device=DEV)
    p, r, d, a = obs.data_ptr(), rew.data_ptr(), done.data_ptr(), actions.data_ptr()
    stats = np.zeros(4 * 256, np.uint64)

    def act(obs_ptr, rew_ptr, done_ptr, act_ptr):
        return lib.crl_pong_opp_act(h, vp(obs_ptr), vp(rew_ptr), vp(done_ptr), 0, vp(act_ptr), None, None)

    def act_pairs(o0, o1, rew_ptr, done_ptr, act_ptr):
        return lib.crl_pong_opp_act_pairs(h, vp(o0), vp(o1), vp(rew_ptr), vp(done_ptr), vp(act_ptr), None, None)

    pairs = np.array([[0, 2], [2, 1], [1, 0]], np.int32)
    expect(lib.crl_pong_opp_set_pairs(h, pairs.ctypes.data, 3, None), _native.CRL_E_STATE, "set_pool first")
    expect(act_pairs(p, p, r, d, a), _native.CRL_E_STATE, "set_pairs first")
    expect(lib.crl_pong_opp_get_pair_stats(h, stats.ctypes.data, 3, None), _native.CRL_E_STATE, "set_pairs first")
    kinds = np.array([RB, RND, 0], np.int32)
    assert lib.crl_pong_opp_set_pool(h, kinds.ctypes.data, None, 3, None) == 0
    assert lib.crl_pong_opp_assign(h, None, None) == 0
    for size in (0, 257):
        big = np.zeros((257, 2), np.int32)
        expect(lib.crl_pong_opp_set_pairs(h, big.ctypes.data, size, None), _native.CRL_E_INVALID, "1 to 256 pairings")
    expect(lib.crl_pong_opp_set_pairs(h, None, 3, None), _native.CRL_E_INVALID, "1 to 256 pairings")
    for bad, text in ((3, "pairing 1, seat 0: pool index 3 is not in [0, 3)"), (-1, "pairing 1, seat 0: pool index -1")):
        b2 = pairs.copy()
        b2[1, 0] = bad
        expect(lib.crl_pong_opp_set_pairs(h, b2.ctypes.data, 3, None), _native.CRL_E_INVALID, text)
    b2 = pairs.copy()
    b2[2, 1] = 7
    expect(lib.crl_pong_opp_set_pairs(h, b2.ctypes.data, 3, None), _native.CRL_E_INVALID, "pairing 2, seat 1")
    assert act(p, 0, 0, a) == 0                                    # refused set_pairs calls left per-env mode in place
    assert lib.crl_pong_opp_set_pairs(h, pairs.ctypes.data, 3, None) == 0
    launches = lib.crl_launch_count()
    expect(act(p, r, d, a), _native.CRL_E_STATE, "league mode")
    expect(act_pairs(p, p, r, 0, a), _native.CRL_E_INVALID, "go together")
    expect(act_pairs(p, p, 0, d, a), _native.CRL_E_INVALID, "go together")
    expect(act_pairs(0, p, r, d, a), _native.CRL_E_INVALID, "null buffer")
    expect(act_pairs(p, 0, r, d, a), _native.CRL_E_INVALID, "null buffer")
    expect(act_pairs(p, p, r, d, 0), _native.CRL_E_INVALID, "null buffer")
    expect(act_pairs(p + 2, p, r, d, a), _native.CRL_E_INVALID, "4-byte aligned")
    expect(act_pairs(p, p + 1, r, d, a), _native.CRL_E_INVALID, "4-byte aligned")
    expect(lib.crl_pong_opp_get_pair_stats(h, None, 3, None), _native.CRL_E_INVALID, "null buffer")
    for k in (0, 257):
        expect(lib.crl_pong_opp_get_pair_stats(h, stats.ctypes.data, k, None), _native.CRL_E_INVALID, "num_pairs")
    assert lib.crl_launch_count() == launches
    assert act_pairs(p, p, 0, 0, a) == 0 and lib.crl_launch_count() == launches + 1
    torch.cuda.synchronize()
    got = actions.cpu().numpy()
    assert set(got.reshape(-1).tolist()) <= {0, 1, 2, 999} and got[0, 0] == 999 and got[2, 1] == 999
    assert lib.crl_pong_opp_get_pair_stats(h, stats.ctypes.data, 256, None) == 0 and not stats.any()
    # set_pool leaves league mode; assign must follow, as always
    assert lib.crl_pong_opp_set_pool(h, kinds.ctypes.data, None, 3, None) == 0
    expect(act(p, r, d, a), _native.CRL_E_STATE, "crl_pong_opp_assign after")
    expect(act_pairs(p, p, r, d, a), _native.CRL_E_STATE, "set_pairs first")
    assert lib.crl_pong_opp_destroy(h) == 0

    # seat 1 after a league run is a fresh handle's (pool without RANDOM: its stream is keyed by the act count)
    n, seed = 3000, 12
    pool = [RB, 0, 3, 6]
    gen = torch.Generator(device=DEV).manual_seed(12)
    used = ext().PongOpponents(n, 0, seed, 0)
    fresh = ext().PongOpponents(n, 0, seed, 0)
    for hh in (used, fresh):
        for k, img in enumerate(nets):
            hh.load_net(k, img)
    used.set_pool(torch.tensor([RB, RND, 0, 7], dtype=torch.int32), None)
    used.set_pairs(torch.tensor([(1, 2), (2, 3), (3, 1)], dtype=torch.int32))
    for t in range(5):
        both = torch.zeros((n, 2), dtype=torch.int32, device=DEV)
        rd = torch.from_numpy(np.random.default_rng(t).integers(-1, 2, (n, 2)).astype(np.float32)).to(DEV)
        used.act_pairs(frames(n, gen), frames(n, gen), rd if t else None, (rd[:, 0] != 0) if t else None, both, None)
    ids = torch.from_numpy(np.random.default_rng(1).integers(0, len(pool), n).astype(np.int32))
    for hh in (used, fresh):
        hh.set_pool(torch.tensor(pool, dtype=torch.int32), None)
        hh.assign(ids)
    for t in range(6):
        o1 = frames(n, gen)
        rd = torch.from_numpy(np.random.default_rng(10 + t).integers(-1, 2, (n, 2)).astype(np.float32)).to(DEV)
        outs = []
        for hh in (used, fresh):
            acts = torch.full((n, 2), SENTINEL, dtype=torch.int32, device=DEV)
            lg = torch.full((n, 3), float("nan"), dtype=torch.float32, device=DEV)
            hh.act(o1, rd if t else None, (rd[:, 0] != 0) if t else None, False, acts, lg)
            outs.append((bits(lg), acts.cpu()))
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]), t
    assert used.stats() == fresh.stats() and sum(fresh.stats()) > 0
    used.close()
    fresh.close()


# ------------------------------------------------------------------------------------------------ through the game
def make_double(n, seed):
    from competitive_rl_b200 import make_envs
    return make_envs("cPongDouble-v0", num_envs=n, resized_dim=42, frame_stack=None, log_dir=None, seed=seed)


def late_game(env, rows=None):
    """Put the envs (all, or `rows`) at num_rounds 20 of 21 so that their next point ends the episode."""
    st = env.get_state().cpu().numpy()
    rows = np.arange(len(st)) if rows is None else rows
    st[rows, 8] = 20
    st[rows, 6] = np.minimum(st[rows, 6], 10)
    st[rows, 7] = np.minimum(st[rows, 7], 10)
    env.set_state(st)


class LateGame(object):
    """A cPongDouble env whose reset() ends in late_game, so that every env's first episode ends within a test."""

    def __init__(self, env):
        self.__dict__["_env"] = env

    def __getattr__(self, name):
        return getattr(self._env, name)

    def reset(self):
        obs = self._env.reset()
        late_game(self._env)
        return obs


def tally(pairing, rew, done, ret, table):
    """Add the episodes that one step ended to table [P, 4] (seat 0's summed reward ret, updated in place)."""
    ret += rew[:, 0]
    for i in np.flatnonzero(done):
        table[pairing[i], 0] += 1
        table[pairing[i], 1 if ret[i] > 0 else 2 if ret[i] == 0 else 3] += 1
    ret[done] = 0


def by_entry(pairs, table, m):
    out = np.zeros((4, m, m), np.int64)
    for (a, b), row in zip(pairs, table):
        out[:, a, b] += row
    return out


def test_pool_evaluation_against_a_twin_env():
    """evaluate_pool_in_batch over [RULE_BASED, RANDOM] x [RULE_BASED, RANDOM] at N = 256 from late-game states, against
    a twin env of the same seed driven by HostLeague's actions: the same number of steps gives the same table."""
    from competitive_rl_b200.evaluate import evaluate_pool_in_batch
    n, seed, env_seed = 256, 31, 4
    pool = ["RULE_BASED", "RANDOM"]
    env = make_double(n, env_seed)
    out = evaluate_pool_in_batch(pool, LateGame(env), 12, seed=seed, check_every=16, max_steps=800)
    pairs = [(0, 0), (0, 1), (1, 0), (1, 1)]
    assert out["pool"] == pool and out["pairs"] == pairs
    twin = LateGame(make_double(n, env_seed))
    m = lo.HostLeague(n, seed, 0, DEV)
    m.set_pool([RB, RND])
    m.set_pairs(pairs)
    obs = twin.reset()
    rew = done = None
    table = np.zeros((4, 4), np.int64)
    ret = np.zeros(n, np.float32)
    for t in range(out["steps"]):
        step = m.act_pairs(obs[0], obs[1], rew, done)
        assert (step.actions >= 0).all()
        obs, r, d, _ = twin.step(step.actions.astype(np.int32))
        rew, done = r.cpu().numpy(), d.cpu().numpy()[:, 0].astype(bool)
        tally(m.pairing, rew.astype(np.float32), done, ret, table)
    want = by_entry(pairs, table, 2)
    print("pool table episodes", want[0].tolist(), "wins", want[1].tolist(), "steps", out["steps"])
    for k, key in enumerate(("episodes", "wins", "draws", "losses")):
        assert out[key].dtype == np.int64 and np.array_equal(out[key], want[k]), key
    assert want[0].sum() >= n // 2 and want[1].sum() > 0 and want[3].sum() > 0
    env.close()
    twin.close()


def variant_state_dict(a, b):
    sd = {}
    for k, (name, shape) in enumerate(reference_layout("LightActorCritic")):
        i = np.arange(int(np.prod(shape)), dtype=np.float64)
        sd[name] = torch.from_numpy((0.08 * np.sin(a * i + b * k + 1.0)).astype(np.float32).reshape(shape))
    return sd


def test_network_pool_through_the_game():
    """Pool [RULE_BASED, A, B] (two synthetic networks), all 9 pairings, N = 600 from late-game states.  The handle is
    driven directly and the env is stepped with the kernel's own actions; both seats' logits are checked against
    forward64 of host-kept stacks of the env's observations, the table against a host tally.  evaluate_pool_in_batch on
    a twin env of the same seed, for the same number of steps, returns that table."""
    from competitive_rl_b200.builtin_policies import pack_light_actor_critic
    from competitive_rl_b200.evaluate import evaluate_pool_in_batch
    n, seed, env_seed, steps = 600, 8, 21, 240
    sds = {"A": variant_state_dict(0.37, 0.0), "B": variant_state_dict(0.23, 2.0)}
    imgs = [pack_light_actor_critic(sds["A"]), pack_light_actor_critic(sds["B"])]
    pool = ["RULE_BASED", "A", "B"]
    pairs = [(a, b) for a in range(3) for b in range(3)]
    env = LateGame(make_double(n, env_seed))
    h = new_handle(n, seed, 0, imgs, [RB, 0, 1], pairs)
    pairing = np.arange(n) % 9
    kind = np.array([RB, 0, 1])[np.array(pairs)[pairing]]         # [n, 2]
    obs = env.reset()
    stacks = [torch.zeros((n, 4, 42, 42), dtype=torch.uint8, device=DEV) for _ in range(2)]
    both = torch.zeros((n, 2), dtype=torch.int32, device=DEV)
    logits = torch.zeros((n, 2, 3), dtype=torch.float32, device=DEV)
    rew = done = None
    table = np.zeros((9, 4), np.int64)
    ret = np.zeros(n, np.float32)
    for t in range(steps):
        h.act_pairs(env._obs[0], env._obs[1], rew, done, both, logits)
        for seat in range(2):
            stacks[seat] = torch.cat([stacks[seat][:, 1:], obs[seat].reshape(n, 1, 42, 42)], dim=1)
        lg, ac = logits.double().cpu().numpy(), both.cpu().numpy()
        for seat in range(2):
            assert (ac[kind[:, seat] == RB, seat] == 999).all() and (lg[kind[:, seat] == RB, seat] == 0).all(), t
            for s in (0, 1):
                rows = np.flatnonzero(kind[:, seat] == s)
                x = stacks[seat][torch.from_numpy(rows).to(DEV)]
                ref, mag = oo.forward64(x, imgs[s]).cpu().numpy(), oo.magnitude64(x, imgs[s]).cpu().numpy()
                ratio = oo.logit_ratio(lg[rows, seat], ref, mag)
                WORST["ratio"] = max(WORST["ratio"], float(ratio.max()))
                assert (ratio <= oo.TOL_ULPS).all(), (t, seat, s)
                assert np.array_equal(ac[rows, seat], oo.greedy(lg[rows, seat])), (t, seat, s)
                dec = oo.decided(ref, mag)
                assert np.array_equal(ac[rows, seat][dec], ref[dec].argmax(axis=1)), (t, seat, s)
        obs, r, d, _ = env.step(both)
        rew, done = env._rew, env._done
        tally(pairing, r.cpu().numpy().astype(np.float32), d.cpu().numpy()[:, 0].astype(bool), ret, table)
    h.act_pairs(env._obs[0], env._obs[1], rew, done, both, None)           # credits the last step's episodes
    got = np.array(h.pair_stats(9), np.int64).reshape(9, 4)
    print("network pool table", table.tolist())
    assert np.array_equal(got, table)
    assert table[:, 0].sum() >= n // 2 and (table[:, 0] > 0).all()
    h.close()
    env.close()
    twin = LateGame(make_double(n, env_seed))
    out = evaluate_pool_in_batch(pool, twin, 10 ** 9, networks=sds, seed=seed, check_every=steps, max_steps=steps)
    want = by_entry(pairs, table, 3)
    assert out["steps"] == steps
    for k, key in enumerate(("episodes", "wins", "draws", "losses")):
        assert np.array_equal(out[key], want[k]), key
    twin.close()
