"""The per-env opponent kernel (csrc/pong_opponent.cu) driven directly through _crl_torch.PongOpponents, with no env,
against the float64 reference and the host model of a handle in oracle/opponent_oracle.py.

1. accuracy sweep over N (one env per CTA, a short last chunk, several chunks per CTA): 8 distinct random networks at
   init scale and 30x, frames in which every byte varies, three assignment patterns; logits within 4 u M, the action
   rules, column 0 untouched, bit-identical logits against one-env handles and under a permutation of slot numbers;
2. exact ties of the argmax;
3. a whole-handle scenario (16-entry pool with zero weights and duplicates, first_env >= 2^33, seed / load_net /
   set_pool / restart mid-run) against HostOpponents, and two shards against one handle, bit for bit;
4. the C ABI's argument checks (every one returns before any launch)."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")
import opponent_oracle as oo  # noqa: E402

pytestmark = pytest.mark.gpu

SENTINEL = -7                      # column 0 of the action buffer: the learner's, never written by the kernel
DEV = "cuda"
WORST = {"ratio": 0.0}             # the largest |error| / (u M) seen in this module


def ext():
    from competitive_rl_b200 import _native
    return _native.ext()


@pytest.fixture(scope="module")
def nets():
    """8 distinct random LightActorCritic images: slots 0-3 at PyTorch's init scale, 4-7 at 30x."""
    gen = torch.Generator().manual_seed(2024)
    return [oo.random_params(gen, 1.0 if s < 4 else 30.0) for s in range(oo.SLOTS)]


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    print("\nlargest |logit error| / (u M) of the opponent kernel: %.3f" % WORST["ratio"])


def frames(n, gen):
    """uint8 [n, 42, 42] on the device: env i always gets frames of one kind (random bytes, all 0, all 255, sparse
    Pong-like), redrawn on every call, so that after 4 acts its whole stack is of that kind."""
    kind = torch.as_tensor((np.arange(n) * 7 + np.arange(n) // 64) % 4, device=DEV).view(n, 1, 1)
    out = torch.zeros((n, oo.DIM, oo.DIM), dtype=torch.uint8, device=DEV)
    for k, name in enumerate(oo.FRAME_KINDS):
        out = torch.where(kind == k, oo.synthetic_frames(name, n, gen, DEV), out)
    return out.contiguous()


def new_handle(n, seed, first_env, images, slots=None):
    """A PongOpponents with images[k] loaded into slot slots[k] (default: slot k)."""
    h = ext().PongOpponents(n, 0, seed, first_env)
    for k, img in enumerate(images):
        h.load_net(k if slots is None else slots[k], img)
    return h


def act(h, n, obs1, rew=None, done=None, resample=False):
    """One act; returns (logits float32 [n, 3], actions int32 [n, 2]) with column 0 prefilled with SENTINEL."""
    actions = torch.full((n, 2), SENTINEL, dtype=torch.int32, device=DEV)
    logits = torch.full((n, 3), float("nan"), dtype=torch.float32, device=DEV)
    h.act(obs1, rew, done, resample, actions, logits)
    return logits, actions


def check_step(logits, actions, step, where=""):
    """The kernel's logits and actions against one step of HostOpponents: column 0 untouched; non-network envs exact
    (logits 0); network envs within TOL_ULPS u M, action = greedy of its own logits, = argmax(ref) where decided."""
    lg = logits.cpu().numpy()
    ac = actions.cpu().numpy()
    assert (ac[:, 0] == SENTINEL).all(), where
    other = ~step.net
    assert np.array_equal(ac[other, 1], step.actions[other]), where
    assert (lg[other] == 0).all(), where
    if step.net.any():
        got, a, ref, mag = lg[step.net], ac[step.net, 1], step.ref[step.net], step.mag[step.net]
        ratio = oo.logit_ratio(got, ref, mag)
        WORST["ratio"] = max(WORST["ratio"], float(ratio.max()))
        bad = np.flatnonzero((ratio > oo.TOL_ULPS).any(axis=1))
        assert len(bad) == 0, (where, "envs", np.flatnonzero(step.net)[bad[:5]], got[bad[:5]], ref[bad[:5]],
                               ratio[bad[:5]])
        assert np.array_equal(a, oo.greedy(got)), where
        dec = oo.decided(ref, mag)
        assert np.array_equal(a[dec], ref[dec].argmax(axis=1)), where


def bits(t):
    return t.contiguous().view(torch.int32).cpu()


def wave_n(offset):
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count * 64 + offset


SWEEP_N = [1, 3, 64, 65, 100, "wave-1", "wave+1", 65536, 65573]


@pytest.mark.parametrize("n", SWEEP_N, ids=[str(v) for v in SWEEP_N])
def test_accuracy_sweep(nets, n):
    """Ten acts (the ring wraps twice) with the assignment cycling through i % 8 (all 8 slots in every 64-env chunk),
    sorted blocks (mostly one slot per chunk) and a random mix with RULE_BASED / RANDOM."""
    if isinstance(n, str):
        n = wave_n(-1 if n.endswith("-1") else 1)
    seed, first = 0x5EED, 11
    pool = list(range(oo.SLOTS)) + [oo.RULE_BASED, oo.RANDOM]
    perm = [3, 6, 0, 7, 2, 5, 1, 4]                      # network k lives in slot perm[k] of the permuted handle
    h = new_handle(n, seed, first, nets)
    hp = new_handle(n, seed, first, nets, perm)
    m = oo.HostOpponents(n, seed, first, DEV)
    for s, img in enumerate(nets):
        m.load_net(s, img)
    sampled = sorted({0, n // 2, n - 1})
    singles = [new_handle(1, seed, first + i, nets) for i in sampled]
    kinds = torch.tensor(pool, dtype=torch.int32)
    h.set_pool(kinds, None)
    hp.set_pool(torch.tensor(perm + pool[oo.SLOTS:], dtype=torch.int32), None)
    m.set_pool(pool)
    for s in singles:
        s.set_pool(kinds, None)
    idx = np.arange(n)
    patterns = [idx % 8, idx * 8 // n, np.random.default_rng(n).integers(0, len(pool), n)]
    gen = torch.Generator(device=DEV).manual_seed(n)
    for t in range(10):
        ids = patterns[t % 3].astype(np.int32)
        for hh in (h, hp):
            hh.assign(torch.from_numpy(ids))
        m.assign(ids)
        for s, i in zip(singles, sampled):
            s.assign(torch.from_numpy(ids[i:i + 1]))
        obs = frames(n, gen)
        step = m.act(obs)
        lg, ac = act(h, n, obs)
        check_step(lg, ac, step, "N %d act %d" % (n, t))
        lp, ap = act(hp, n, obs)
        assert torch.equal(bits(lp), bits(lg)) and torch.equal(ap, ac), (n, t)
        for s, i in zip(singles, sampled):
            l1, a1 = act(s, 1, obs[i:i + 1])
            assert torch.equal(bits(l1), bits(lg[i:i + 1])) and torch.equal(a1[:, 1], ac[i:i + 1, 1]), (n, t, i)
    for hh in [h, hp] + singles:
        hh.close()


def tied_net(base, rows, bias0=None):
    q = base.clone()
    wa = q[3681:8481].view(3, 1600)
    wa[rows[1]] = wa[rows[0]]
    q[8481 + rows[1]] = q[8481 + rows[0]]
    if bias0 is not None:
        q[8481] = bias0
    return q


def test_exact_ties_go_to_the_lowest_index(nets):
    """Equal actor rows and biases give bitwise-equal logits, and the argmax takes the lower index of a tie."""
    n = wave_n(1)
    gen = torch.Generator(device=DEV).manual_seed(7)
    h = new_handle(n, 1, 0, [tied_net(nets[0], (0, 1)), tied_net(nets[5], (0, 1)),
                             tied_net(nets[1], (1, 2), -1e3), tied_net(nets[6], (1, 2), -1e12)])
    h.set_pool(torch.tensor([0, 1, 2, 3], dtype=torch.int32), None)
    ids = np.arange(n) % 4
    h.assign(torch.from_numpy(ids.astype(np.int32)))
    for t in range(6):
        lg, ac = act(h, n, frames(n, gen))
        lg, a = lg.cpu(), ac[:, 1].cpu().numpy()
        b = bits(lg)
        first, second = ids < 2, ids >= 2
        assert torch.equal(b[first, 0], b[first, 1]) and (a[first] != 1).all(), t
        assert ((a[first] == 0) == (lg[first, 0] >= lg[first, 2]).numpy()).all(), t
        assert torch.equal(b[second, 1], b[second, 2]) and (a[second] == 1).all(), t
    h.close()


SCENARIO_POOL = [oo.RANDOM, oo.RULE_BASED, 0, 1, 2, 3, oo.RANDOM, 4, 5, 6, 7, oo.RULE_BASED, oo.RANDOM, oo.RULE_BASED,
                 oo.RANDOM, 7]
SCENARIO_WEIGHTS = [0.0, 1.0, 2.0, 1.0, 1.0, 0.5, 1.0, 1.0, 0.0, 1.0, 3.0, 1.0, 1.0, 0.5, 1.0, 0.0]
SMALL_POOL = [oo.RULE_BASED, 3, oo.RANDOM, 6, 0]
SMALL_WEIGHTS = [1.0, 2.0, 0.0, 1.0, 1.0]


@pytest.mark.parametrize("n,steps", [(1000, 200), (40000, 40)])
def test_handle_scenario_against_host_model(nets, n, steps):
    """A 16-entry pool (zero weights first, in the middle and last; RULE_BASED / RANDOM / network 7 twice), first_env
    2^33 + 7, random rewards with dones (about 5 %), and mid-run: resample toggled, seed(), load_net over a slot in use,
    set_pool to a smaller pool + assign(None), restart(False), restart(True).  Ids, non-network actions and stats are
    compared exactly, network logits and actions with the tolerance rule; two shards [0, N/2) and [N/2, N) reproduce
    the single handle bit for bit."""
    seed, first, half = 0xC0FFEE, 2 ** 33 + 7, n // 2
    ev = {"seed": steps * 3 // 10, "load": steps * 4 // 10, "pool": steps // 2, "restart": steps * 13 // 20,
          "clear": steps * 4 // 5}
    replacement = oo.random_params(torch.Generator().manual_seed(99), 3.0)
    hs = [new_handle(n, seed, first, nets), new_handle(half, seed, first, nets),
          new_handle(n - half, seed, first + half, nets)]
    parts = [slice(0, n), slice(0, half), slice(half, n)]
    m = oo.HostOpponents(n, seed, first, DEV)
    for s, img in enumerate(nets):
        m.load_net(s, img)

    def set_pool(kinds, weights):
        for h in hs:
            h.set_pool(torch.tensor(kinds, dtype=torch.int32), torch.tensor(weights, dtype=torch.float64))
            h.assign(None)
        m.set_pool(kinds, weights)
        m.assign(None)

    def check_stats(t):
        got = [np.array(h.stats(), np.int64).reshape(oo.MAX_POOL, 4) for h in hs]
        assert np.array_equal(got[0], m.stats), t
        assert np.array_equal(got[1] + got[2], got[0]), t

    set_pool(SCENARIO_POOL, SCENARIO_WEIGHTS)
    rng = np.random.default_rng(n)
    gen = torch.Generator(device=DEV).manual_seed(n)
    fresh = True                     # the first act after a (re)start has no reward / done
    resample = True
    for t in range(steps):
        if t == ev["seed"]:
            for h in hs:
                h.seed(seed + 1)
            m.seed(seed + 1)
        if t == ev["load"]:
            for h in hs:
                h.load_net(4, replacement)
            m.load_net(4, replacement)
        if t == ev["pool"]:
            set_pool(SMALL_POOL, SMALL_WEIGHTS)
        if t in (ev["restart"], ev["clear"]):
            for h in hs:
                h.restart(t == ev["clear"])
            m.restart(t == ev["clear"])
            fresh = True
        if t % max(1, steps // 8) == 0:
            resample = not resample
        obs = frames(n, gen)
        if fresh:
            rew = done = None
        else:
            r = np.stack([rng.integers(-1, 2, n), rng.normal(size=n)], axis=1).astype(np.float32)
            d = rng.random(n) < 0.05
            rew, done = torch.from_numpy(r).to(DEV), torch.from_numpy(d).to(DEV)
        step = m.act(obs, None if fresh else r, None if fresh else d, resample)
        outs = [act(h, p.stop - p.start, obs[p], None if fresh else rew[p], None if fresh else done[p], resample)
                for h, p in zip(hs, parts)]
        fresh = False
        ids = []
        for h, p in zip(hs, parts):
            out = torch.empty(p.stop - p.start, dtype=torch.int32, device=DEV)
            h.ids(out)
            ids.append(out.cpu().numpy())
        assert np.array_equal(ids[0], step.ids), t
        assert np.array_equal(np.concatenate(ids[1:]), ids[0]), t
        check_step(*outs[0], step, "N %d step %d" % (n, t))
        lg = torch.cat([outs[1][0], outs[2][0]])
        ac = torch.cat([outs[1][1], outs[2][1]])
        assert torch.equal(bits(lg), bits(outs[0][0])) and torch.equal(ac, outs[0][1]), t
        if t % 10 == 9:
            check_stats(t)
    check_stats(steps)
    assert m.stats[:, 0].sum() > 0 and len(np.unique(step.ids)) == len(SMALL_POOL) - 1
    for h in hs:
        h.close()


def test_c_abi_argument_checks(nets):
    """Every argument check of crl_pong_opp_* returns its code and sets crl_last_error; none reaches a kernel."""
    from competitive_rl_b200 import _native
    lib = _native.load()
    vp = ctypes.c_void_p
    n = 8

    def expect(rc, code, text):
        assert rc == code, (rc, code, text)
        assert text in lib.crl_last_error().decode(), (lib.crl_last_error(), text)

    h = vp()
    expect(lib.crl_pong_opp_create(0, 0, 1, 0, ctypes.byref(h)), _native.CRL_E_INVALID, "num_envs must be positive")
    expect(lib.crl_pong_opp_seed(None, 1), _native.CRL_E_INVALID, "null handle")
    assert lib.crl_pong_opp_create(n, 0, 1, 0, ctypes.byref(h)) == 0 and h.value
    img = nets[0].numpy().copy()
    obs = torch.zeros(n * 1764 + 4, dtype=torch.uint8, device=DEV)
    rew = torch.zeros((n, 2), dtype=torch.float32, device=DEV)
    done = torch.zeros(n, dtype=torch.uint8, device=DEV)
    actions = torch.full((n, 2), SENTINEL, dtype=torch.int32, device=DEV)
    p = obs.data_ptr()

    def act(obs_ptr, rew_ptr, done_ptr, act_ptr):
        return lib.crl_pong_opp_act(h, vp(obs_ptr), vp(rew_ptr), vp(done_ptr), 0, vp(act_ptr), None, None)

    # act and assign before any pool
    expect(act(p, rew.data_ptr(), done.data_ptr(), actions.data_ptr()), _native.CRL_E_STATE, "crl_pong_opp_assign after")
    expect(lib.crl_pong_opp_assign(h, None, None), _native.CRL_E_STATE, "set_pool first")
    # load_net
    for slot in (-1, 8):
        expect(lib.crl_pong_opp_load_net(h, slot, img.ctypes.data, img.size, None), _native.CRL_E_INVALID,
               "network slot must be in")
    expect(lib.crl_pong_opp_load_net(h, 0, img.ctypes.data, img.size - 1, None), _native.CRL_E_INVALID, "has 8484 floats")
    expect(lib.crl_pong_opp_load_net(h, 0, None, img.size, None), _native.CRL_E_INVALID, "has 8484 floats")
    bad = img.copy()
    bad[1234] = np.nan
    expect(lib.crl_pong_opp_load_net(h, 0, bad.ctypes.data, bad.size, None), _native.CRL_E_INVALID,
           "parameter 1234 is not finite")
    assert lib.crl_pong_opp_load_net(h, 0, img.ctypes.data, img.size, None) == 0
    # set_pool
    kinds = np.array([oo.RULE_BASED, oo.RANDOM, 0] + [oo.RANDOM] * 14, np.int32)
    w = np.ones(17, np.float64)
    for size in (0, 17):
        expect(lib.crl_pong_opp_set_pool(h, kinds.ctypes.data, w.ctypes.data, size, None), _native.CRL_E_INVALID,
               "a pool has 1 to 16 entries")
    for kd in (-3, 8):
        k2 = kinds.copy()
        k2[1] = kd
        expect(lib.crl_pong_opp_set_pool(h, k2.ctypes.data, w.ctypes.data, 3, None), _native.CRL_E_INVALID,
               "kind %d is neither" % kd)
    k2 = kinds.copy()
    k2[2] = 5
    expect(lib.crl_pong_opp_set_pool(h, k2.ctypes.data, w.ctypes.data, 3, None), _native.CRL_E_STATE,
           "network slot 5 was never loaded")
    for wk in (-1.0, np.nan, np.inf):
        w2 = w.copy()
        w2[1] = wk
        expect(lib.crl_pong_opp_set_pool(h, kinds.ctypes.data, w2.ctypes.data, 3, None), _native.CRL_E_INVALID,
               "pool entry 1: weight must be finite and >= 0")
    zero = np.zeros(3, np.float64)
    expect(lib.crl_pong_opp_set_pool(h, kinds.ctypes.data, zero.ctypes.data, 3, None), _native.CRL_E_INVALID, "sum to 0")
    assert lib.crl_pong_opp_set_pool(h, kinds.ctypes.data, w.ctypes.data, 3, None) == 0
    # assign
    expect(act(p, rew.data_ptr(), done.data_ptr(), actions.data_ptr()), _native.CRL_E_STATE, "crl_pong_opp_assign after")
    ids = np.array([0, 1, 2, 0, 1, 2, 3, 0], np.int32)
    expect(lib.crl_pong_opp_assign(h, ids.ctypes.data, None), _native.CRL_E_INVALID, "env 6: opponent id 3 is not in [0, 3)")
    ids[6] = -1
    expect(lib.crl_pong_opp_assign(h, ids.ctypes.data, None), _native.CRL_E_INVALID, "env 6: opponent id -1")
    ids[6] = 2
    assert lib.crl_pong_opp_assign(h, ids.ctypes.data, None) == 0
    # act
    launches = lib.crl_launch_count()
    expect(act(p, rew.data_ptr(), 0, actions.data_ptr()), _native.CRL_E_INVALID, "go together")
    expect(act(p, 0, done.data_ptr(), actions.data_ptr()), _native.CRL_E_INVALID, "go together")
    expect(act(0, rew.data_ptr(), done.data_ptr(), actions.data_ptr()), _native.CRL_E_INVALID, "null buffer")
    expect(act(p, rew.data_ptr(), done.data_ptr(), 0), _native.CRL_E_INVALID, "null buffer")
    expect(act(p + 1, rew.data_ptr(), done.data_ptr(), actions.data_ptr()), _native.CRL_E_INVALID, "4-byte aligned")
    expect(lib.crl_pong_opp_get_ids(h, None, None), _native.CRL_E_INVALID, "null buffer")
    expect(lib.crl_pong_opp_get_stats(h, None, None), _native.CRL_E_INVALID, "null buffer")
    assert lib.crl_launch_count() == launches
    # the handle still works after every refusal
    assert act(p, 0, 0, actions.data_ptr()) == 0 and lib.crl_launch_count() == launches + 1
    torch.cuda.synchronize()
    a = actions.cpu().numpy()
    assert (a[:, 0] == SENTINEL).all() and a[0, 1] == 999 and set(a[:, 1].tolist()) <= {0, 1, 2, 999}
    assert lib.crl_pong_opp_destroy(h) == 0
