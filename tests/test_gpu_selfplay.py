"""Self-play mode of the opponent kernel (csrc/pong_opponent.cu, crl_pong_opp_set_selfplay / act_selfplay): the learner in
either seat of a league pairing, against the float64 reference and the host model HostSelfPlay of
oracle/selfplay_oracle.py, against learner mode and league mode, and through the game with SelfPlayEnvWrapper.

1. accuracy sweep over N with (L, L), (L, pool), (pool, L) and (pool, pool) pairings, random and all-network pools and
   random dones: learner seats' stacks byte for byte, logits and value within 4 u M, log pi(a) and the sampled / greedy
   action as in learner mode's tests; pool seats as in league mode; pool seats' rows of stack_out untouched;
2. (LEARNER, X) in every env is bit-identical to learner mode with every env assigned X;
3. pool seats are bit-identical to league mode with the learner seats replaced by a pool entry;
4. learner seats' stacks against a twin cPongDouble env with frame_stack=4, zero_on_done=True over one-point games;
5. two shards against one handle, bit for bit, sampled actions included;
6. the mode rules and the C ABI's argument checks (no refusal launches anything);
7. SelfPlayEnvWrapper.learner_step with a torch LightActorCritic over full games: the pairing tally against a host
   tally, and a weight refresh taking effect on the next step.

The sampling rule and its margins are learner mode's (tests/test_gpu_learner.py): the action must equal the float64
inverse CDF of the returned logits wherever u is more than 2^-20 from a bound, and the reference's wherever u is more than
max(1e-5, 2 u max_j M_j + 2^-20) from a reference bound.  Rows nearer a bound are counted and printed."""
import copy
import ctypes

import numpy as np
import pytest

from conftest import reference_layout

torch = pytest.importorskip("torch")
import learner_oracle as lo  # noqa: E402
import opponent_oracle as oo  # noqa: E402
import selfplay_oracle as so  # noqa: E402

pytestmark = pytest.mark.gpu

DEV = "cuda"
L, RB, RND = so.LEARNER, oo.RULE_BASED, oo.RANDOM
NEAR_OWN = 2.0 ** -20
NEAR_REF = 1e-5
FILL = 77
REPORT = {"logit": 0.0, "value": 0.0, "logp": 0.0, "pool_logit": 0.0, "near_own": 0, "near_ref": 0, "sampled": 0}


def ext():
    from competitive_rl_b200 import _native
    return _native.ext()


@pytest.fixture(scope="module")
def nets():
    """8 pool networks (slots 0-3 at init scale, 4-7 at 30x) and two learners (init scale, 30x)."""
    gen = torch.Generator().manual_seed(909)
    return [oo.random_params(gen, 1.0 if s < 4 else 30.0) for s in range(oo.SLOTS)] + \
           [oo.random_params(gen, 1.0), oo.random_params(gen, 30.0)]


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    print("\nself-play kernel: largest |logit error| / (u M) learner %.3f, pool networks %.3f; |value error| / (u M) %.3f; "
          "|log-prob error| / tol %.3f; sampled learner actions %d, within 2^-20 of a bound of the returned logits %d, "
          "within the margin of a float64 bound %d" % (
              REPORT["logit"], REPORT["pool_logit"], REPORT["value"], REPORT["logp"], REPORT["sampled"],
              REPORT["near_own"], REPORT["near_ref"]))


def frames(n, gen):
    """uint8 [n, 42, 42]: env i always gets frames of one kind (random bytes, all 0, all 255, sparse Pong-like)."""
    kind = torch.as_tensor((np.arange(n) * 7 + np.arange(n) // 64) % 4, device=DEV).view(n, 1, 1)
    out = torch.zeros((n, oo.DIM, oo.DIM), dtype=torch.uint8, device=DEV)
    for k, name in enumerate(oo.FRAME_KINDS):
        out = torch.where(kind == k, oo.synthetic_frames(name, n, gen, DEV), out)
    return out.contiguous()


def wave_n(offset):
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count * 64 + offset


def new_handle(n, seed, first_env, images, learner, kinds):
    h = ext().PongOpponents(n, 0, seed, first_env)
    for k, img in enumerate(images):
        h.load_net(k, img)
    if learner is not None:
        h.load_learner(learner)
    h.set_pool(torch.tensor(kinds, dtype=torch.int32), None)
    return h


def mixed_table(rng, num_pairs, pool_size):
    """num_pairs pairings whose first four are (L, L), (L, pool), (pool, L), (pool, pool), the rest random with a
    learner seat half of the time."""
    t = np.where(rng.random((num_pairs, 2)) < 0.5, L, rng.integers(0, pool_size, (num_pairs, 2)))
    t[:4] = [[L, L], [L, 0], [0, L], [0, 0]]
    t[1:4] = np.where(t[1:4] == L, L, rng.integers(0, pool_size, (3, 2)))
    return t.astype(np.int32)


class Out(object):
    """The buffers of one act_selfplay: actions [n, 2], logp_value [n, 2, 2], logits [n, 2, 3], stack [n, 2, 4, 42, 42]."""

    def __init__(self, n):
        self.actions = torch.full((n, 2), -7, dtype=torch.int32, device=DEV)
        self.lpv = torch.full((n, 2, 2), float("nan"), dtype=torch.float32, device=DEV)
        self.logits = torch.full((n, 2, 3), float("nan"), dtype=torch.float32, device=DEV)
        self.stack = torch.full((n, 2, 4, 42, 42), FILL, dtype=torch.uint8, device=DEV)

    def bits(self):
        return [self.actions.cpu(), self.lpv.view(torch.int32).cpu(), self.logits.view(torch.int32).cpu(), self.stack.cpu()]


def act_selfplay(h, n, obs0, obs1, rew=None, done=None, sample=True):
    o = Out(n)
    h.act_selfplay(obs0, obs1, rew, done, sample, o.actions, o.lpv, o.logits, o.stack)
    return o


def logp_tol(lg, lp):
    """|log pi error| allowed from fp32 logits lg [B, 3] and log-prob lp [B]: 8 u (max |l| + |lp| + 1)."""
    return 8 * oo.U * (np.abs(lg).max(axis=1) + np.abs(lp) + 1.0)


def check_step(o, st, sample, where):
    """One act_selfplay against one step of HostSelfPlay."""
    lrn = st.learner                                            # [n, 2]
    lrn_t = torch.from_numpy(lrn).to(DEV)
    assert torch.equal(o.stack[lrn_t], st.stack.to(DEV)[lrn_t]), where
    assert (o.stack[~lrn_t] == FILL).all(), where               # pool seats' rows are not written
    lg_all = o.logits.double().cpu().numpy()
    act = o.actions.cpu().numpy()
    lpv = o.lpv.double().cpu().numpy()
    assert (lpv[~lrn] == 0).all(), where
    # pool seats: league mode's rules
    other = ~lrn & ~st.net
    assert np.array_equal(act[other], st.actions[other]) and (lg_all[other] == 0).all(), where
    if st.net.any():
        ratio = oo.logit_ratio(lg_all[st.net], st.ref[st.net], st.mag[st.net])
        REPORT["pool_logit"] = max(REPORT["pool_logit"], float(ratio.max()))
        assert (ratio <= oo.TOL_ULPS).all(), where
        assert np.array_equal(act[st.net], oo.greedy(lg_all[st.net])), where
        dec = oo.decided(st.ref[st.net], st.mag[st.net])
        assert np.array_equal(act[st.net][dec], st.ref[st.net][dec].argmax(axis=1)), where
    if not lrn.any():
        return
    # learner seats: learner mode's rules
    lg, ref, mag, a = lg_all[lrn], st.ref[lrn], st.mag[lrn], act[lrn]
    lp, v, u = lpv[lrn][:, 0], lpv[lrn][:, 1], st.u[lrn]
    ratio = oo.logit_ratio(lg, ref, mag)
    REPORT["logit"] = max(REPORT["logit"], float(ratio.max()))
    assert (ratio <= oo.TOL_ULPS).all(), (where, np.argwhere(ratio > oo.TOL_ULPS)[:5])
    vr = oo.logit_ratio(v, st.value[lrn], st.value_mag[lrn])
    REPORT["value"] = max(REPORT["value"], float(vr.max()))
    assert (vr <= oo.TOL_ULPS).all(), where
    assert set(np.unique(a).tolist()) <= {0, 1, 2}, where
    e = np.abs(lp - lo.logprob64(lg, a)) / logp_tol(lg, lp)
    REPORT["logp"] = max(REPORT["logp"], float(e.max()))
    assert (e <= 1).all(), where
    if not sample:
        assert np.array_equal(a, oo.greedy(lg)), where
        dec = oo.decided(ref, mag)
        assert np.array_equal(a[dec], ref[dec].argmax(axis=1)), where
        return
    REPORT["sampled"] += len(a)
    far = lo.boundary_distance(lg, u) > NEAR_OWN
    REPORT["near_own"] += int((~far).sum())
    assert np.array_equal(a[far], lo.sample64(lg[far], u[far])), where
    margin = np.maximum(NEAR_REF, 2 * oo.U * mag.max(axis=1) + NEAR_OWN)
    far = lo.boundary_distance(ref, u) > margin
    REPORT["near_ref"] += int((~far).sum())
    assert np.array_equal(a[far], lo.sample64(ref[far], u[far])), where


SWEEP_N = [1, 3, 64, 65, "wave-1", "wave+1", 65536, 65573]


@pytest.mark.parametrize("pool", ["mixed", "networks"])
@pytest.mark.parametrize("n", SWEEP_N, ids=[str(v) for v in SWEEP_N])
def test_accuracy_sweep(nets, n, pool):
    """Eight acts (the rings wrap twice) with about 10 % dones from the second on, sampling on six and greedy on two.
    The mixed pool is RULE_BASED / RANDOM and all 8 slots, the network pool the 8 slots; 37 pairings.  The learner is at
    init scale with the mixed pool and at 30x with the network pool."""
    if isinstance(n, str):
        n = wave_n(-1 if n.endswith("-1") else 1)
    seed, first = 0x5E1F, 2 ** 33 + 5
    learner = nets[8] if pool == "mixed" else nets[9]
    kinds = list(range(oo.SLOTS)) + ([RB, RND] if pool == "mixed" else [])
    rng = np.random.default_rng(n)
    table = mixed_table(rng, 37, len(kinds))
    h = new_handle(n, seed, first, nets[:8], learner, kinds)
    h.set_selfplay(torch.from_numpy(table))
    m = so.HostSelfPlay(n, seed, first, DEV)
    for s in range(oo.SLOTS):
        m.load_net(s, nets[s])
    m.load_learner(learner)
    m.set_pool(kinds)
    m.set_selfplay(table)
    gen = torch.Generator(device=DEV).manual_seed(n)
    r = d = None
    for t in range(8):
        sample = t % 4 != 2
        o0, o1 = frames(n, gen), frames(n, gen)
        st = m.act_selfplay(o0, o1, r, d)
        o = act_selfplay(h, n, o0, o1, None if r is None else torch.from_numpy(r).to(DEV),
                         None if d is None else torch.from_numpy(d).to(DEV), sample=sample)
        check_step(o, st, sample, "N %d %s act %d" % (n, pool, t))
        r = np.stack([rng.integers(-1, 2, n), rng.normal(size=n)], axis=1).astype(np.float32)
        d = rng.random(n) < 0.1
    st = np.array(h.pair_stats(len(table)), np.int64).reshape(-1, 4)
    assert np.array_equal(st, m.stats)
    h.close()


@pytest.mark.parametrize("opponent", ["RULE_BASED", "RANDOM", "network"])
def test_learner_seat_zero_is_learner_mode(nets, opponent):
    """(LEARNER, X) in every env against learner mode with every env assigned X, with dones and a restart(False): actions,
    log-prob, value, the learner's logits and stack bit for bit, and the tally equals X's per-entry statistics."""
    n, seed, first, steps = wave_n(1), 0xC0DE, 2 ** 32 - 9, 12
    kind = {"RULE_BASED": RB, "RANDOM": RND, "network": 5}[opponent]
    hs = new_handle(n, seed, first, nets[:8], nets[9], [kind])
    hl = new_handle(n, seed, first, nets[:8], nets[9], [kind])
    hs.set_selfplay(torch.tensor([[L, 0]], dtype=torch.int32))
    hl.assign(torch.zeros(n, dtype=torch.int32))
    hl.restart(True)
    rng = np.random.default_rng(1)
    gen = torch.Generator(device=DEV).manual_seed(1)
    rew = done = None
    for t in range(steps):
        if t == 7:
            hs.restart(False)
            hl.restart(False)
            rew = done = None
        sample = t != 4
        o0, o1 = frames(n, gen), frames(n, gen)
        a = act_selfplay(hs, n, o0, o1, rew, done, sample=sample)
        b_act = torch.full((n, 2), -7, dtype=torch.int32, device=DEV)
        b_lpv = torch.zeros((n, 2), dtype=torch.float32, device=DEV)
        b_lg = torch.zeros((n, 3), dtype=torch.float32, device=DEV)
        b_st = torch.zeros((n, 4, 42, 42), dtype=torch.uint8, device=DEV)
        hl.act_learner(o0, o1, rew, done, False, sample, b_act, b_lpv, b_lg, b_st)
        assert torch.equal(a.actions, b_act), t
        assert torch.equal(a.lpv[:, 0].view(torch.int32), b_lpv.view(torch.int32)), t
        assert torch.equal(a.logits[:, 0].view(torch.int32), b_lg.view(torch.int32)), t
        assert torch.equal(a.stack[:, 0], b_st) and (a.stack[:, 1] == FILL).all(), t
        assert not a.lpv[:, 1].any(), t
        rew = torch.from_numpy(rng.integers(-1, 2, (n, 2)).astype(np.float32)).to(DEV)
        done = torch.from_numpy(rng.random(n) < 0.1).to(DEV)
    assert hs.pair_stats(1) == hl.stats()[:4] and hs.pair_stats(1)[0] > 0
    hs.close()
    hl.close()


def test_pool_seats_are_league_mode(nets):
    """A self-play table against league mode with every learner seat replaced by pool entry 0: every pool seat's action
    and logits bit for bit (their stacks are fed and kept alike), and the pairing tally."""
    n, seed, first, steps = 20011, 0xFACE, 3, 10
    kinds = [RB, 0, RND, 6, 2, 7]
    table = mixed_table(np.random.default_rng(7), 19, len(kinds))
    league = np.where(table == L, 0, table).astype(np.int32)
    hs = new_handle(n, seed, first, nets[:8], nets[8], kinds)
    hp = new_handle(n, seed, first, nets[:8], None, kinds)
    hs.set_selfplay(torch.from_numpy(table))
    hp.set_pairs(torch.from_numpy(league))
    pool_seat = torch.from_numpy(table[(first + np.arange(n)) % len(table)] != L).to(DEV)
    rng = np.random.default_rng(2)
    gen = torch.Generator(device=DEV).manual_seed(2)
    rew = done = None
    for t in range(steps):
        o0, o1 = frames(n, gen), frames(n, gen)
        a = act_selfplay(hs, n, o0, o1, rew, done, sample=bool(t % 3))
        b_act = torch.full((n, 2), -7, dtype=torch.int32, device=DEV)
        b_lg = torch.zeros((n, 2, 3), dtype=torch.float32, device=DEV)
        hp.act_pairs(o0, o1, rew, done, b_act, b_lg)
        assert torch.equal(a.actions[pool_seat], b_act[pool_seat]), t
        assert torch.equal(a.logits.view(torch.int32)[pool_seat], b_lg.view(torch.int32)[pool_seat]), t
        rew = torch.from_numpy(rng.integers(-1, 2, (n, 2)).astype(np.float32)).to(DEV)
        done = torch.from_numpy(rng.random(n) < 0.1).to(DEV)
    assert hs.pair_stats(len(table)) == hp.pair_stats(len(table))
    hs.close()
    hp.close()


# ------------------------------------------------------------------------------------------------ through the game
def variant_state_dict(a, b):
    sd = {}
    for k, (name, shape) in enumerate(reference_layout("LightActorCritic")):
        i = np.arange(int(np.prod(shape)), dtype=np.float64)
        sd[name] = torch.from_numpy((0.08 * np.sin(a * i + b * k + 1.0)).astype(np.float32).reshape(shape))
    return sd


def double_env(n, seed, **kw):
    from competitive_rl_b200 import make_envs
    return make_envs("cPongDouble-v0", num_envs=n, resized_dim=42, frame_stack=None, log_dir=None, seed=seed, **kw)


def test_stacks_match_a_frame_stacked_twin_env():
    """learner_step over one-point games with a reset half-way and pairings (L, L), (L, RANDOM), (A, L), (RULE_BASED, A):
    every learner seat's stack equals its agent's observation of a twin cPongDouble env with frame_stack=4 and
    zero_on_done=True stepped with the same actions, byte for byte.  In the 3 steps after a reset the twin holds copies
    of the reset frame where the learner's history is zero (FrameStackTensor.reset): there the newest frames are compared
    and the learner's older slots must be zero."""
    from competitive_rl_b200 import make_envs
    from competitive_rl_b200.selfplay import SelfPlayEnvWrapper
    n, seed, steps = 512, 17, 400
    w = SelfPlayEnvWrapper(double_env(n, seed, max_num_rounds=1))
    twin = make_envs("cPongDouble-v0", num_envs=n, resized_dim=42, frame_stack=4, zero_on_done=True, log_dir=None,
                     seed=seed, max_num_rounds=1)
    w.add_opponent("A", variant_state_dict(0.37, 0.0))
    w.set_league([("LEARNER", "LEARNER"), ("LEARNER", "RANDOM"), ("A", "LEARNER"), ("RULE_BASED", "A")], seed=5)
    w.set_learner(variant_state_dict(0.23, 2.0))
    seats = w.learner_seats
    assert seats.shape == (n, 2) and seats.dtype == torch.bool
    assert seats.cpu().tolist()[:4] == [[True, True], [True, False], [False, True], [False, False]]
    episodes = np.zeros(n, np.int64)
    since = 0
    for t in range(steps):
        if t in (0, steps // 2):
            w.reset()
            tw = twin.reset()
            since = 0
        stack, act, lp, v, obs, rew, done, info = w.learner_step()
        k = max(0, 3 - since)
        for seat in range(2):
            s = seats[:, seat]
            assert torch.equal(stack[s, seat, k:], tw[seat][s, k:]) and not stack[s, seat, :k].any(), (t, seat)
        assert torch.isfinite(lp[seats]).all() and torch.isfinite(v[seats]).all()
        tw, r2, d2, _ = twin.step(act)
        assert torch.equal(rew, r2) and torch.equal(done, d2), t
        episodes += done[:, 0].cpu().numpy().astype(np.int64)
        since += 1
    print("episodes ended per env: mean %.2f, max %d" % (episodes.mean(), episodes.max()))
    assert episodes.sum() >= n and episodes.max() >= 3
    w.close()
    twin.close()


def test_shards_reproduce_one_handle(nets):
    """first_env 2^33 + 7 split at an odd point, 7 mixed pairings: the two shards' actions (sampled), log-probs, values,
    logits and stacks equal the single handle's bit for bit."""
    n, half, steps, seed, first = 5001, 2347, 12, 99, 2 ** 33 + 7
    kinds = [RB, 0, RND, 5, 2]
    table = torch.from_numpy(mixed_table(np.random.default_rng(5), 7, len(kinds)))
    hs = [new_handle(n, seed, first, nets[:8], nets[9], kinds), new_handle(half, seed, first, nets[:8], nets[9], kinds),
          new_handle(n - half, seed, first + half, nets[:8], nets[9], kinds)]
    parts = [slice(0, n), slice(0, half), slice(half, n)]
    for h in hs:
        h.set_selfplay(table)
    rng = np.random.default_rng(3)
    gen = torch.Generator(device=DEV).manual_seed(3)
    rew = done = None
    for t in range(steps):
        o0, o1 = frames(n, gen), frames(n, gen)
        outs = [act_selfplay(h, p.stop - p.start, o0[p], o1[p], None if rew is None else rew[p],
                             None if done is None else done[p], sample=t != 5)
                for h, p in zip(hs, parts)]
        for whole, a, b in zip(outs[0].bits(), outs[1].bits(), outs[2].bits()):
            assert torch.equal(torch.cat([a, b]), whole), t
        rew = torch.from_numpy(rng.integers(-1, 2, (n, 2)).astype(np.float32)).to(DEV)
        done = torch.from_numpy(rng.random(n) < 0.1).to(DEV)
    totals = np.array(hs[1].pair_stats(7)) + np.array(hs[2].pair_stats(7))
    assert totals.tolist() == hs[0].pair_stats(7)
    for h in hs:
        h.close()


def test_mode_rules_and_c_abi_argument_checks(nets):
    """Each refusal returns its code and sets crl_last_error without launching anything: set_selfplay without a pool and
    with bad tables; act_selfplay outside self-play mode, before load_learner and with bad buffers; act, act_pairs and
    act_learner in self-play mode; set_pairs refusing CRL_PONG_OPP_LEARNER.  set_pool and set_pairs leave the mode,
    reloading the learner does not."""
    from competitive_rl_b200 import _native
    lib = _native.load()
    vp = ctypes.c_void_p
    n = 8

    def expect(rc, code, text):
        assert rc == code, (rc, code, text)
        assert text in lib.crl_last_error().decode(), (lib.crl_last_error(), text)

    h = vp()
    assert lib.crl_pong_opp_create(n, 0, 1, 0, ctypes.byref(h)) == 0 and h.value
    img = nets[8].numpy().copy()
    obs = torch.zeros(n * 1764 + 4, dtype=torch.uint8, device=DEV)
    rew = torch.zeros((n, 2), dtype=torch.float32, device=DEV)
    done = torch.zeros(n, dtype=torch.uint8, device=DEV)
    actions = torch.full((n, 2), -7, dtype=torch.int32, device=DEV)
    lpv = torch.zeros((n, 2, 2), dtype=torch.float32, device=DEV)
    stack = torch.zeros(n * 2 * 7056 + 4, dtype=torch.uint8, device=DEV)
    stats = np.zeros((2, 4), np.uint64)
    p, r, d, a, q, s = obs.data_ptr(), rew.data_ptr(), done.data_ptr(), actions.data_ptr(), lpv.data_ptr(), stack.data_ptr()
    table = np.array([[L, L], [L, 1]], np.int32)
    kinds = np.array([RB, RND], np.int32)

    def act_selfplay(o0, o1, rew_ptr, done_ptr, act_ptr, lpv_ptr, stack_ptr):
        return lib.crl_pong_opp_act_selfplay(h, vp(o0), vp(o1), vp(rew_ptr), vp(done_ptr), 1, vp(act_ptr), vp(lpv_ptr),
                                             None, vp(stack_ptr), None)

    def set_selfplay(t, count):
        return lib.crl_pong_opp_set_selfplay(h, None if t is None else t.ctypes.data, count, None)

    act = lambda: lib.crl_pong_opp_act(h, vp(p), None, None, 0, vp(a), None, None)           # noqa: E731
    act_pairs = lambda: lib.crl_pong_opp_act_pairs(h, vp(p), vp(p), None, None, vp(a), None, None)   # noqa: E731
    act_learner = lambda: lib.crl_pong_opp_act_learner(h, vp(p), vp(p), None, None, 0, 1, vp(a), vp(q), None, vp(s),  # noqa: E731
                                                       None)

    start = lib.crl_launch_count()
    expect(set_selfplay(table, 2), _native.CRL_E_STATE, "crl_pong_opp_set_pool first")
    expect(act_selfplay(p, p, r, d, a, q, s), _native.CRL_E_STATE, "crl_pong_opp_set_selfplay first")
    assert lib.crl_pong_opp_set_pool(h, kinds.ctypes.data, None, 2, None) == 0
    for count in (0, 257):
        big = np.full((257, 2), L, np.int32)
        expect(set_selfplay(big, count), _native.CRL_E_INVALID, "a self-play table has 1 to 256 pairings")
    expect(set_selfplay(None, 2), _native.CRL_E_INVALID, "a self-play table has 1 to 256 pairings")
    for bad, where in ((2, "pairing 1, seat 0: 2 is neither"), (-1, "pairing 1, seat 0: -1 is neither"),
                       (-2, "pairing 1, seat 0: -2 is neither")):
        t2 = table.copy()
        t2[1, 0] = bad
        expect(set_selfplay(t2, 2), _native.CRL_E_INVALID, where)
    expect(lib.crl_pong_opp_set_pairs(h, table.ctypes.data, 2, None), _native.CRL_E_INVALID,
           "pairing 0, seat 0: pool index -3 is not in [0, 2)")
    expect(act_selfplay(p, p, r, d, a, q, s), _native.CRL_E_STATE, "crl_pong_opp_set_selfplay first")
    assert set_selfplay(table, 2) == 0
    expect(act_selfplay(p, p, r, d, a, q, s), _native.CRL_E_STATE, "crl_pong_opp_load_learner first")
    assert lib.crl_pong_opp_load_learner(h, img.ctypes.data, img.size, None) == 0
    for fn in (act, act_pairs, act_learner):
        expect(fn(), _native.CRL_E_STATE, "self-play mode: use crl_pong_opp_act_selfplay")
    expect(act_selfplay(p, p, r, 0, a, q, s), _native.CRL_E_INVALID, "go together")
    expect(act_selfplay(p, p, 0, d, a, q, s), _native.CRL_E_INVALID, "go together")
    for k in range(5):
        ptrs = [p, p, a, q, s]
        ptrs[k] = 0
        expect(act_selfplay(ptrs[0], ptrs[1], r, d, ptrs[2], ptrs[3], ptrs[4]), _native.CRL_E_INVALID, "null buffer")
    expect(act_selfplay(p + 1, p, r, d, a, q, s), _native.CRL_E_INVALID, "4-byte aligned")
    expect(act_selfplay(p, p + 2, r, d, a, q, s), _native.CRL_E_INVALID, "4-byte aligned")
    expect(act_selfplay(p, p, r, d, a, q, s + 3), _native.CRL_E_INVALID, "4-byte aligned")
    assert lib.crl_launch_count() == start
    assert act_selfplay(p, p, 0, 0, a, q, s) == 0 and lib.crl_launch_count() == start + 1
    assert lib.crl_pong_opp_load_learner(h, img.ctypes.data, img.size, None) == 0   # a refresh stays in self-play mode
    expect(act(), _native.CRL_E_STATE, "self-play mode")
    assert act_selfplay(p, p, r, d, a, q, s) == 0 and lib.crl_launch_count() == start + 2
    assert lib.crl_pong_opp_get_pair_stats(h, stats.ctypes.data, 2, None) == 0
    pairs = np.array([[0, 1]], np.int32)
    assert lib.crl_pong_opp_set_pairs(h, pairs.ctypes.data, 1, None) == 0          # set_pairs leaves it
    expect(act_selfplay(p, p, r, d, a, q, s), _native.CRL_E_STATE, "crl_pong_opp_set_selfplay first")
    assert act_pairs() == 0 and lib.crl_launch_count() == start + 3
    assert set_selfplay(table, 2) == 0
    assert lib.crl_pong_opp_set_pool(h, kinds.ctypes.data, None, 2, None) == 0     # and so does set_pool
    expect(act_selfplay(p, p, r, d, a, q, s), _native.CRL_E_STATE, "crl_pong_opp_set_selfplay first")
    assert lib.crl_pong_opp_assign(h, None, None) == 0
    assert act() == 0 and lib.crl_launch_count() == start + 5
    torch.cuda.synchronize()
    assert lib.crl_pong_opp_destroy(h) == 0


def test_learner_step_with_a_torch_learner():
    """SelfPlayEnvWrapper.learner_step with a torch LightActorCritic over full three-point games: the learner seats'
    logits and values match the module's own float64 forward within 4 u M, actions follow the tag-4 / tag-5 draws (the
    argmax after switching to sample=False), a weight refresh takes effect on the next step, and pair_stats() equals a
    host tally of the returned rewards and dones."""
    from competitive_rl_b200.builtin_policies import LightActorCritic, pack_light_actor_critic
    from competitive_rl_b200.selfplay import SelfPlayEnvWrapper
    n, seed, steps = 3000, 21, 700
    w = SelfPlayEnvWrapper(double_env(n, seed, max_num_rounds=3))
    table = [("LEARNER", "LEARNER"), ("LEARNER", "RULE_BASED"), ("B", "LEARNER"), ("RANDOM", "B"), ("LEARNER", "B")]
    w.add_opponent("B", variant_state_dict(0.41, 1.0))
    w.set_league(table, seed=7)
    nets_ = [LightActorCritic(), LightActorCritic()]
    for k, net in enumerate(nets_):
        net.load_state_dict(variant_state_dict(0.31 + 0.1 * k, k))
    w.logits = torch.zeros((n, 2, 3), dtype=torch.float32, device=DEV)
    w.set_learner(nets_[0])
    w.reset()
    seats = w.learner_seats.cpu().numpy()
    pairing = np.arange(n) % len(table)
    ret = np.zeros(n)
    tally = np.zeros((len(table), 4), np.int64)
    g = np.arange(n)
    switch = 12
    for t in range(steps):
        k = 0 if t < switch else 1
        if t == switch:
            w.set_learner(nets_[1], sample=False)
        stack, act, lp, v, obs, rew, done, info = w.learner_step()
        r, d = rew.cpu().numpy(), done[:, 0].cpu().numpy()
        if t < steps - 1:       # an episode is credited by the act after the step that ended it
            ret += r[:, 0]
            np.add.at(tally, (pairing[d], 0), 1)
            np.add.at(tally, (pairing[d], np.where(ret[d] > 0, 1, np.where(ret[d] == 0, 2, 3))), 1)
            ret[d] = 0
        if t > switch + 2:
            continue
        img = pack_light_actor_critic(nets_[k])
        lg_all, a_all = w.logits.double().cpu().numpy(), act.cpu().numpy()
        for seat in range(2):
            rows = seats[:, seat]
            x = stack[torch.from_numpy(rows).to(DEV), seat]
            with torch.no_grad():
                ref_l, ref_v = copy.deepcopy(nets_[k]).double().to(DEV)(x.double())
            ref_l, ref_v = ref_l.cpu().numpy(), ref_v[:, 0].cpu().numpy()
            lg, a = lg_all[rows, seat], a_all[rows, seat]
            mag = oo.magnitude64(x, img).cpu().numpy()
            assert (oo.logit_ratio(lg, ref_l, mag) <= oo.TOL_ULPS).all(), (t, seat)
            vm = lo.value_magnitude64(x, img).cpu().numpy()
            assert (oo.logit_ratio(v[:, seat].cpu().numpy()[rows], ref_v, vm) <= oo.TOL_ULPS).all(), (t, seat)
            if t == switch:    # the refreshed weights, not the old ones
                old = oo.forward64(x, pack_light_actor_critic(nets_[0])).cpu().numpy()
                assert (oo.logit_ratio(lg, old, mag) > oo.TOL_ULPS).any(axis=1).all()
            if k == 0:
                u = so.learner_u(7, g[rows], t, seat)
                far = lo.boundary_distance(lg, u) > NEAR_OWN
                assert np.array_equal(a[far], lo.sample64(lg[far], u[far])), (t, seat)
            else:
                assert np.array_equal(a, oo.greedy(lg)), (t, seat)
            lpn = lp[:, seat].double().cpu().numpy()[rows]
            assert (np.abs(lpn - lo.logprob64(lg, a)) <= logp_tol(lg, lpn)).all(), (t, seat)
            assert not lp[:, seat].cpu().numpy()[~rows].any()
    stats = w.pair_stats()
    want = {}
    for p, pr in enumerate(table):
        dct = want.setdefault(pr, dict(episodes=0, wins=0, draws=0, losses=0))
        for j, key in enumerate(("episodes", "wins", "draws", "losses")):
            dct[key] += int(tally[p, j])
    print("pair_stats:", stats)
    assert stats == want and all(s["episodes"] > 0 for s in stats.values())
    w.close()
