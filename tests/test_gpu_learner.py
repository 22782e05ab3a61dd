"""Learner mode of the opponent kernel (csrc/pong_opponent.cu, crl_pong_opp_load_learner / act_learner): a LightActorCritic
learner in seat 0 of the per-env opponents' launch, against the float64 reference and the host model HostLearner of
oracle/learner_oracle.py, and through the game with TournamentEnvWrapper.learner_step.

1. accuracy sweep over N, random and all-network pools, random dones: the learner's stacks byte for byte, logits and
   value within 4 u M, the sampled / greedy action and log pi(a) from the returned logits and against float64;
2. the stacks against a twin cPongDouble env with frame_stack=4, zero_on_done=True over full games with auto-resets;
3. seat 1 unchanged: actions, ids and statistics equal a per-env run without a learner;
4. two shards against one handle, bit for bit, sampled actions included;
5. the mode rules and the C ABI's argument checks (no refusal launches anything);
6. learner_step with a torch LightActorCritic, and a weight refresh taking effect on the next step.

Sampling rule.  The kernel draws u exactly (r32 * 2^-32) and compares it with fp32 cumulative bounds c_0, c_1 of the
softmax of its fp32 logits.  From the logits it returned, c_k in float64 differs from the kernel's fp32 c_k by a few
ulps, so the action must equal the float64 inverse CDF of the returned logits wherever u is more than 2^-20 from a
bound.  Against the float64 reference, each logit may be off by up to 4 u M_j and sum_j |dc_k / dl_j| <= 1/2, so c_k
may move by up to 2 u max_j M_j; the action must equal the reference's inverse CDF wherever u is more than
max(1e-5, 2 u max_j M_j + 2^-20) from a reference bound.  Rows nearer a bound are counted and printed, not excused silently."""
import copy
import ctypes

import numpy as np
import pytest

from conftest import reference_layout

torch = pytest.importorskip("torch")
import learner_oracle as lo  # noqa: E402
import opponent_oracle as oo  # noqa: E402

pytestmark = pytest.mark.gpu

DEV = "cuda"
RB, RND = oo.RULE_BASED, oo.RANDOM
NEAR_OWN = 2.0 ** -20
NEAR_REF = 1e-5
REPORT = {"logit": 0.0, "value": 0.0, "logp": 0.0, "dc": 0.0, "near_own": 0, "near_ref": 0, "sampled": 0}


def ext():
    from competitive_rl_b200 import _native
    return _native.ext()


@pytest.fixture(scope="module")
def nets():
    """8 pool networks (slots 0-3 at init scale, 4-7 at 30x) and two learners (init scale, 30x)."""
    gen = torch.Generator().manual_seed(808)
    return [oo.random_params(gen, 1.0 if s < 4 else 30.0) for s in range(oo.SLOTS)] + \
           [oo.random_params(gen, 1.0), oo.random_params(gen, 30.0)]


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    print("\nlearner kernel: largest |logit error| / (u M) %.3f, |value error| / (u M) %.3f, |log-prob error| / tol %.3f, "
          "largest |c_k(kernel logits) - c_k(float64)| %.3g; sampled actions %d, within 2^-20 of a bound of the "
          "returned logits %d, within the margin of a float64 bound %d" % (
              REPORT["logit"], REPORT["value"], REPORT["logp"], REPORT["dc"], REPORT["sampled"], REPORT["near_own"],
              REPORT["near_ref"]))


def frames(n, gen):
    """uint8 [n, 42, 42]: env i always gets frames of one kind (random bytes, all 0, all 255, sparse Pong-like)."""
    kind = torch.as_tensor((np.arange(n) * 7 + np.arange(n) // 64) % 4, device=DEV).view(n, 1, 1)
    out = torch.zeros((n, oo.DIM, oo.DIM), dtype=torch.uint8, device=DEV)
    for k, name in enumerate(oo.FRAME_KINDS):
        out = torch.where(kind == k, oo.synthetic_frames(name, n, gen, DEV), out)
    return out.contiguous()


def wave_n(offset):
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count * 64 + offset


def new_handle(n, seed, first_env, images, learner):
    h = ext().PongOpponents(n, 0, seed, first_env)
    for k, img in enumerate(images):
        h.load_net(k, img)
    if learner is not None:
        h.load_learner(learner)
    return h


class Out(object):
    """The buffers of one act_learner: actions [n, 2], logp_value [n, 2], logits [n, 3], stack [n, 4, 42, 42]."""

    def __init__(self, n):
        self.actions = torch.full((n, 2), -7, dtype=torch.int32, device=DEV)
        self.lpv = torch.full((n, 2), float("nan"), dtype=torch.float32, device=DEV)
        self.logits = torch.full((n, 3), float("nan"), dtype=torch.float32, device=DEV)
        self.stack = torch.full((n, 4, 42, 42), 77, dtype=torch.uint8, device=DEV)

    def bits(self):
        return [self.actions.cpu(), self.lpv.view(torch.int32).cpu(), self.logits.view(torch.int32).cpu(), self.stack.cpu()]


def act_learner(h, n, obs0, obs1, rew=None, done=None, resample=False, sample=True, logits=True):
    o = Out(n)
    h.act_learner(obs0, obs1, rew, done, resample, sample, o.actions, o.lpv, o.logits if logits else None, o.stack)
    return o


def logp_tol(lg, lp):
    """|log pi error| allowed from fp32 logits lg [B, 3] and log-prob lp [B]: 8 u (max |l| + |lp| + 1)."""
    return 8 * oo.U * (np.abs(lg).max(axis=1) + np.abs(lp) + 1.0)


def check_learner(o, st, sample, where):
    """The learner's outputs of one act against one step of HostLearner (see the module's sampling rule)."""
    stack = o.stack
    assert torch.equal(stack, st.stack), where
    lg = o.logits.double().cpu().numpy()
    a = o.actions[:, 0].cpu().numpy()
    lp, v = (t.double().cpu().numpy() for t in o.lpv.unbind(1))
    ratio = oo.logit_ratio(lg, st.ref, st.mag)
    REPORT["logit"] = max(REPORT["logit"], float(ratio.max()))
    assert (ratio <= oo.TOL_ULPS).all(), (where, np.argwhere(ratio > oo.TOL_ULPS)[:5])
    vr = oo.logit_ratio(v, st.value, st.value_mag)
    REPORT["value"] = max(REPORT["value"], float(vr.max()))
    assert (vr <= oo.TOL_ULPS).all(), (where, np.flatnonzero(vr > oo.TOL_ULPS)[:5])
    assert set(np.unique(a).tolist()) <= {0, 1, 2}, where
    e = np.abs(lp - lo.logprob64(lg, a)) / logp_tol(lg, lp)
    REPORT["logp"] = max(REPORT["logp"], float(e.max()))
    assert (e <= 1).all(), (where, np.flatnonzero(e > 1)[:5])
    if not sample:
        assert np.array_equal(a, oo.greedy(lg)), where
        dec = oo.decided(st.ref, st.mag)
        assert np.array_equal(a[dec], st.ref[dec].argmax(axis=1)), where
        return
    REPORT["sampled"] += len(a)
    REPORT["dc"] = max(REPORT["dc"], float(np.abs(lo.cdf64(lg) - lo.cdf64(st.ref)).max()))
    far = lo.boundary_distance(lg, st.u) > NEAR_OWN
    REPORT["near_own"] += int((~far).sum())
    assert np.array_equal(a[far], lo.sample64(lg[far], st.u[far])), where
    margin = np.maximum(NEAR_REF, 2 * oo.U * st.mag.max(axis=1) + NEAR_OWN)
    far = lo.boundary_distance(st.ref, st.u) > margin
    REPORT["near_ref"] += int((~far).sum())
    assert np.array_equal(a[far], lo.sample64(st.ref[far], st.u[far])), where


def check_seat1(o, step, where):
    """Seat 1 (no logits in learner mode): non-network actions exact, network actions the float64 argmax where decided."""
    a = o.actions[:, 1].cpu().numpy()
    other = ~step.net
    assert np.array_equal(a[other], step.actions[other]), where
    dec = oo.decided(step.ref, step.mag) & step.net
    assert np.array_equal(a[dec], step.ref[dec].argmax(axis=1)), where


SWEEP_N = [1, 3, 64, 65, 100, "wave-1", "wave+1", 65536, 65573]


@pytest.mark.parametrize("pool", ["mixed", "networks"])
@pytest.mark.parametrize("n", SWEEP_N, ids=[str(v) for v in SWEEP_N])
def test_accuracy_sweep(nets, n, pool):
    """Eight acts (the ring wraps twice) with about 10 % dones from the second on, sampling on six and greedy on two;
    the mixed pool has RULE_BASED / RANDOM and all 8 slots drawn at random, the network pool puts slot i % 8 in env i.
    The learner is at init scale with the mixed pool and at 30x with the network pool."""
    if isinstance(n, str):
        n = wave_n(-1 if n.endswith("-1") else 1)
    seed, first = 0x1EA2, 2 ** 33 + 3
    learner = nets[8] if pool == "mixed" else nets[9]
    kinds = list(range(oo.SLOTS)) + [RB, RND]
    rng = np.random.default_rng(n)
    ids = (rng.integers(0, len(kinds), n) if pool == "mixed" else np.arange(n) % 8).astype(np.int32)
    h = new_handle(n, seed, first, nets[:8], learner)
    m = lo.HostLearner(n, seed, first, DEV)
    for s in range(oo.SLOTS):
        m.load_net(s, nets[s])
    m.load_learner(learner)
    h.set_pool(torch.tensor(kinds, dtype=torch.int32), None)
    m.set_pool(kinds)
    h.assign(torch.from_numpy(ids))
    m.assign(ids)
    gen = torch.Generator(device=DEV).manual_seed(n)
    r = d = None
    for t in range(8):
        sample = t % 4 != 2
        o0, o1 = frames(n, gen), frames(n, gen)
        st = m.act_learner(o0, o1, r, d)
        o = act_learner(h, n, o0, o1, None if r is None else torch.from_numpy(r).to(DEV),
                        None if d is None else torch.from_numpy(d).to(DEV), sample=sample)
        where = "N %d %s act %d" % (n, pool, t)
        check_learner(o, st, sample, where)
        check_seat1(o, st.opp, where)
        r = np.stack([rng.integers(-1, 2, n), rng.normal(size=n)], axis=1).astype(np.float32)
        d = rng.random(n) < 0.1
    h.close()


# ------------------------------------------------------------------------------------------------ through the game
def variant_state_dict(a, b):
    sd = {}
    for k, (name, shape) in enumerate(reference_layout("LightActorCritic")):
        i = np.arange(int(np.prod(shape)), dtype=np.float64)
        sd[name] = torch.from_numpy((0.08 * np.sin(a * i + b * k + 1.0)).astype(np.float32).reshape(shape))
    return sd


def tournament(n, seed, **kw):
    from competitive_rl_b200 import make_envs
    return make_envs("cPongTournament-v0", num_envs=n, resized_dim=42, log_dir=None, seed=seed, **kw)


def test_stacks_match_a_frame_stacked_twin_env():
    """learner_step over one-point games (every env ends episodes and auto-resets), with a VecEnv reset half-way: every
    stack the learner acted on equals agent 0's observation of a twin cPongDouble env with frame_stack=4 and
    zero_on_done=True stepped with the same actions, byte for byte.  In the 3 steps after a reset the twin's history
    holds copies of the reset frame (FrameStack.reset) where the learner's is zero (FrameStackTensor.reset): there the
    newest frames are compared and the learner's older slots must be zero."""
    from competitive_rl_b200 import make_envs
    n, seed, steps = 512, 13, 400
    w = tournament(n, seed, max_num_rounds=1)
    twin = make_envs("cPongDouble-v0", num_envs=n, resized_dim=42, frame_stack=4, zero_on_done=True, log_dir=None,
                     seed=seed, max_num_rounds=1)
    w.add_opponent("A", variant_state_dict(0.37, 0.0))
    w.set_opponents(pool=["RULE_BASED", "RANDOM", "A"], resample_on_done=True, seed=5)
    w.set_learner(variant_state_dict(0.23, 2.0))
    episodes = np.zeros(n, np.int64)
    since = 0
    for t in range(steps):
        if t in (0, steps // 2):
            w.reset()
            tw = twin.reset()
            since = 0
        stack, act, lp, v, obs, rew, done, info = w.learner_step()
        k = max(0, 3 - since)
        assert torch.equal(stack[:, k:], tw[0][:, k:]) and not stack[:, :k].any(), t
        assert torch.equal(act, w._both[:, 0]) and torch.isfinite(lp).all() and torch.isfinite(v).all()
        tw, r2, d2, _ = twin.step(w._both)
        assert torch.equal(rew[:, 0], r2[:, 0]) and torch.equal(done[:, 0], d2[:, 0]), t
        episodes += done[:, 0].cpu().numpy().astype(np.int64)
        since += 1
    print("episodes ended per env: mean %.2f, max %d" % (episodes.mean(), episodes.max()))
    assert episodes.sum() >= n and episodes.max() >= 3
    w.close()
    twin.close()


def test_seat_one_is_unchanged_by_the_learner(nets):
    """A learner handle and a per-env handle of the same seeds, pool and assignment, with resample_on_done and random
    rewards / dones: seat 1's actions, the ids and the per-entry statistics are equal at every step."""
    n, seed, steps = wave_n(1), 0xABC, 30
    pool = [RND, RB, 0, 5, 7, RND, 2]
    weights = torch.tensor([1.0, 2.0, 1.0, 0.5, 1.0, 0.0, 3.0], dtype=torch.float64)
    hl = new_handle(n, seed, 9, nets[:8], nets[8])
    hp = new_handle(n, seed, 9, nets[:8], None)
    for h in (hl, hp):
        h.set_pool(torch.tensor(pool, dtype=torch.int32), weights)
        h.assign(None)
    rng = np.random.default_rng(4)
    gen = torch.Generator(device=DEV).manual_seed(4)
    rew = done = None
    for t in range(steps):
        o0, o1 = frames(n, gen), frames(n, gen)
        o = act_learner(hl, n, o0, o1, rew, done, resample=True, sample=bool(t % 2))
        ap = torch.full((n, 2), -7, dtype=torch.int32, device=DEV)
        hp.act(o1, rew, done, True, ap, None)
        assert torch.equal(o.actions[:, 1], ap[:, 1]) and (ap[:, 0] == -7).all(), t
        ids = [torch.empty(n, dtype=torch.int32, device=DEV) for _ in range(2)]
        hl.ids(ids[0])
        hp.ids(ids[1])
        assert torch.equal(ids[0], ids[1]), t
        rew = torch.from_numpy(rng.integers(-1, 2, (n, 2)).astype(np.float32)).to(DEV)
        done = torch.from_numpy(rng.random(n) < 0.1).to(DEV)
    assert hl.stats() == hp.stats() and sum(hl.stats()) > 0
    hl.close()
    hp.close()


def test_shards_reproduce_one_handle(nets):
    """first_env 2^33 + 7 split at an odd point: the two shards' actions (sampled), log-probs, values, logits and stacks
    equal the single handle's bit for bit."""
    n, half, steps, seed, first = 5001, 2347, 12, 99, 2 ** 33 + 7
    pool = torch.tensor([RB, 0, RND, 5, 2], dtype=torch.int32)
    hs = [new_handle(n, seed, first, nets[:8], nets[9]), new_handle(half, seed, first, nets[:8], nets[9]),
          new_handle(n - half, seed, first + half, nets[:8], nets[9])]
    parts = [slice(0, n), slice(0, half), slice(half, n)]
    for h in hs:
        h.set_pool(pool, None)
        h.assign(None)
    rng = np.random.default_rng(3)
    gen = torch.Generator(device=DEV).manual_seed(3)
    rew = done = None
    for t in range(steps):
        o0, o1 = frames(n, gen), frames(n, gen)
        outs = [act_learner(h, p.stop - p.start, o0[p], o1[p], None if rew is None else rew[p],
                            None if done is None else done[p], resample=True, sample=t != 5)
                for h, p in zip(hs, parts)]
        for whole, a, b in zip(outs[0].bits(), outs[1].bits(), outs[2].bits()):
            assert torch.equal(torch.cat([a, b]), whole), t
        rew = torch.from_numpy(rng.integers(-1, 2, (n, 2)).astype(np.float32)).to(DEV)
        done = torch.from_numpy(rng.random(n) < 0.1).to(DEV)
    for h in hs:
        h.close()


def test_mode_rules_and_c_abi_argument_checks(nets):
    """Each refusal returns its code and sets crl_last_error without launching anything: act_learner before
    load_learner, before assign and in league mode; act in learner mode; load_learner's checks; the buffers."""
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
    lpv = torch.zeros((n, 2), dtype=torch.float32, device=DEV)
    stack = torch.zeros(n * 7056 + 4, dtype=torch.uint8, device=DEV)
    p, r, d, a, q, s = obs.data_ptr(), rew.data_ptr(), done.data_ptr(), actions.data_ptr(), lpv.data_ptr(), stack.data_ptr()

    def act_learner(o0, o1, rew_ptr, done_ptr, act_ptr, lpv_ptr, stack_ptr):
        return lib.crl_pong_opp_act_learner(h, vp(o0), vp(o1), vp(rew_ptr), vp(done_ptr), 0, 1, vp(act_ptr), vp(lpv_ptr),
                                            None, vp(stack_ptr), None)

    def act():
        return lib.crl_pong_opp_act(h, vp(p), None, None, 0, vp(a), None, None)

    start = lib.crl_launch_count()
    expect(act_learner(p, p, r, d, a, q, s), _native.CRL_E_STATE, "crl_pong_opp_load_learner first")
    expect(lib.crl_pong_opp_load_learner(h, img.ctypes.data, img.size - 1, None), _native.CRL_E_INVALID, "has 8484 floats")
    expect(lib.crl_pong_opp_load_learner(h, None, img.size, None), _native.CRL_E_INVALID, "has 8484 floats")
    bad = img.copy()
    bad[2500] = np.inf                     # in the critic row, which the slots do not use
    expect(lib.crl_pong_opp_load_learner(h, bad.ctypes.data, bad.size, None), _native.CRL_E_INVALID,
           "parameter 2500 is not finite")
    expect(act_learner(p, p, r, d, a, q, s), _native.CRL_E_STATE, "crl_pong_opp_load_learner first")
    assert lib.crl_pong_opp_load_learner(h, img.ctypes.data, img.size, None) == 0
    expect(act_learner(p, p, r, d, a, q, s), _native.CRL_E_STATE, "crl_pong_opp_assign after")
    kinds = np.array([RB, RND], np.int32)
    assert lib.crl_pong_opp_set_pool(h, kinds.ctypes.data, None, 2, None) == 0
    expect(act_learner(p, p, r, d, a, q, s), _native.CRL_E_STATE, "crl_pong_opp_assign after")
    assert lib.crl_launch_count() == start
    assert lib.crl_pong_opp_assign(h, None, None) == 0
    launches = lib.crl_launch_count()
    expect(act_learner(p, p, r, 0, a, q, s), _native.CRL_E_INVALID, "go together")
    expect(act_learner(p, p, 0, d, a, q, s), _native.CRL_E_INVALID, "go together")
    for k in range(5):
        ptrs = [p, p, a, q, s]
        ptrs[k] = 0
        expect(act_learner(ptrs[0], ptrs[1], r, d, ptrs[2], ptrs[3], ptrs[4]), _native.CRL_E_INVALID, "null buffer")
    expect(act_learner(p + 1, p, r, d, a, q, s), _native.CRL_E_INVALID, "4-byte aligned")
    expect(act_learner(p, p + 2, r, d, a, q, s), _native.CRL_E_INVALID, "4-byte aligned")
    expect(act_learner(p, p, r, d, a, q, s + 3), _native.CRL_E_INVALID, "4-byte aligned")
    pairs = np.array([[0, 1]], np.int32)
    assert lib.crl_pong_opp_set_pairs(h, pairs.ctypes.data, 1, None) == 0
    expect(act_learner(p, p, r, d, a, q, s), _native.CRL_E_STATE, "league mode")
    assert lib.crl_launch_count() == launches
    # set_pool leaves league mode; act_learner enters learner mode, after which act is refused until set_pool
    assert lib.crl_pong_opp_set_pool(h, kinds.ctypes.data, None, 2, None) == 0
    assert lib.crl_pong_opp_assign(h, None, None) == 0
    assert act_learner(p, p, 0, 0, a, q, s) == 0 and lib.crl_launch_count() == launches + 2   # assign(NULL) + act_learner
    expect(act(), _native.CRL_E_STATE, "learner mode")
    assert lib.crl_pong_opp_load_learner(h, img.ctypes.data, img.size, None) == 0      # a refresh stays in learner mode
    expect(act(), _native.CRL_E_STATE, "learner mode")
    assert act_learner(p, p, r, d, a, q, s) == 0 and lib.crl_launch_count() == launches + 3
    assert lib.crl_pong_opp_set_pairs(h, pairs.ctypes.data, 1, None) == 0                # set_pairs leaves it too
    expect(act_learner(p, p, r, d, a, q, s), _native.CRL_E_STATE, "league mode")
    assert lib.crl_pong_opp_set_pool(h, kinds.ctypes.data, None, 2, None) == 0
    assert lib.crl_pong_opp_assign(h, None, None) == 0
    assert act() == 0 and lib.crl_launch_count() == launches + 5
    torch.cuda.synchronize()
    got = actions.cpu().numpy()
    assert set(got[:, 0].tolist()) <= {0, 1, 2} and set(got[:, 1].tolist()) <= {0, 1, 2, 999}
    assert lib.crl_pong_opp_destroy(h) == 0


def test_learner_step_with_a_torch_learner():
    """learner_step with a torch LightActorCritic: learner(stack / 255) in float64 (the module's own forward) matches the
    returned logits and value within 4 u M, the action is the inverse CDF of the returned logits at the tag-4 draw (the
    argmax with sample=False), and set_learner with new weights takes effect on the next step."""
    from competitive_rl_b200.builtin_policies import LightActorCritic, pack_light_actor_critic
    n, seed = 3000, 21
    w = tournament(n, seed)
    w.set_opponents(pool=["RULE_BASED", "RANDOM"], seed=7)
    nets_ = [LightActorCritic(), LightActorCritic()]
    for k, net in enumerate(nets_):
        net.load_state_dict(variant_state_dict(0.31 + 0.1 * k, k))
    w.learner_logits = torch.zeros((n, 3), dtype=torch.float32, device=DEV)
    w.set_learner(nets_[0])
    w.reset()
    acts = 0
    g = np.arange(n)
    for t in range(12):
        k = 0 if t < 6 else 1
        if t == 6:
            w.set_learner(nets_[1], sample=False)
        stack, act, lp, v, obs, rew, done, info = w.learner_step()
        acts += 1
        img = pack_light_actor_critic(nets_[k])
        with torch.no_grad():
            ref_l, ref_v = copy.deepcopy(nets_[k]).double().to(DEV)(stack.double())
        ref_l, ref_v = ref_l.cpu().numpy(), ref_v[:, 0].cpu().numpy()
        lg = w.learner_logits.double().cpu().numpy()
        mag = oo.magnitude64(stack, img).cpu().numpy()
        assert (oo.logit_ratio(lg, ref_l, mag) <= oo.TOL_ULPS).all(), t
        assert (oo.logit_ratio(v.cpu().numpy(), ref_v, lo.value_magnitude64(stack, img).cpu().numpy()) <= oo.TOL_ULPS).all(), t
        if t == 6:    # the refreshed weights, not the old ones
            old = oo.forward64(stack, pack_light_actor_critic(nets_[0])).cpu().numpy()
            assert (oo.logit_ratio(lg, old, mag) > oo.TOL_ULPS).any(axis=1).all()
        a = act.cpu().numpy()
        if k == 0:
            u = lo.learner_u(7, g, acts - 1)
            far = lo.boundary_distance(lg, u) > NEAR_OWN
            assert np.array_equal(a[far], lo.sample64(lg[far], u[far])), t
        else:
            assert np.array_equal(a, oo.greedy(lg)), t
        e = np.abs(lp.double().cpu().numpy() - lo.logprob64(lg, a)) / logp_tol(lg, lp.double().cpu().numpy())
        assert (e <= 1).all(), t
    w.close()
