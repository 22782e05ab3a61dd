"""CPU checks of the per-env opponent reference (oracle/opponent_oracle.py) itself, before it is used to judge the kernel:
Philox known answers, forward64 against the torch module, the tolerance rule's power to tell a correct fp32 evaluation
from subtly wrong ones, and the pool's draw bounds."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
import opponent_oracle as oo  # noqa: E402


# Random123's philox4x32-10 known-answer vectors (kat_vectors): counter, key -> output
PHILOX_KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


def test_philox_known_answers():
    for ctr, key, want in PHILOX_KAT:
        assert oo.philox4x32_10(*ctr, *key) == want
        arr = oo.philox4x32_10(*(np.full(3, c, np.uint64) for c in ctr), *(np.uint64(k) for k in key))
        assert all(np.array_equal(a, np.full(3, w, np.uint64)) for a, w in zip(arr, want))


def test_opp_rand_scalar_and_vector_agree():
    g = np.array([0, 1, 2 ** 32 + 5, 2 ** 33 + 7, -1], np.int64)
    ctr = np.array([0, 7, 2 ** 32 + 1, 3, 2 ** 63], np.uint64)
    for tag in (1, 2):
        vec = oo.opp_rand(0x123456789ABCDEF0, g, tag, ctr)
        assert [int(v) for v in vec] == [oo.opp_rand(0x123456789ABCDEF0, int(a), tag, int(b)) for a, b in zip(g, ctr)]
    # the key's high word, the env's high word and the tag all reach the output
    base = oo.opp_rand(5, 3, 1, 0)
    assert len({base, oo.opp_rand(5 + 2 ** 32, 3, 1, 0), oo.opp_rand(5, 3 + 2 ** 32, 1, 0), oo.opp_rand(5, 3, 2, 0),
                oo.opp_rand(5, 3, 1, 2 ** 32)}) == 5
    acts = oo.random_action(9, np.arange(4096), 11)
    assert set(np.unique(acts).tolist()) == {0, 1, 2}
    assert int(acts[17]) == oo.random_action(9, 17, 11)


def _module(params):
    from competitive_rl_b200.builtin_policies import LightActorCritic, unpack_light_actor_critic
    net = LightActorCritic()
    net.load_state_dict(unpack_light_actor_critic(params))
    return net.requires_grad_(False)


def _frames(kind, n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([oo.synthetic_frames(kind, n, g) for _ in range(4)], dim=1)


def test_forward64_matches_the_module_in_float64():
    gen = torch.Generator().manual_seed(1)
    for scale in (1.0, 30.0):
        p = oo.random_params(gen, scale)
        x = _frames("random", 64, 2)
        want = _module(p).double()(x.double())[0]
        got = oo.forward64(x, p)
        assert got.dtype == torch.float64 and tuple(got.shape) == (64, 3)
        assert torch.allclose(got, want, rtol=0, atol=1e-12 * max(1.0, float(want.abs().max())))
        mag = oo.magnitude64(x, p)
        assert (mag >= got.abs() - 1e-12).all() and (mag > 0).all()


def _fp32(params, x, input_scale=1.0):
    with torch.no_grad():
        return _module(params)(x.float() * input_scale)[0].double()


def _ratio(got, x, params):
    return oo.logit_ratio(got.numpy(), oo.forward64(x, params).numpy(), oo.magnitude64(x, params).numpy()).max()


def _swap_conv1_taps(params):
    """conv1 reads taps (ci 1, kh 2, kw 1) and (ci 1, kh 2, kw 2) of each other (a kernel's tap indexing bug)."""
    q = params.clone()
    w = q[:1024].view(16, 4, 4, 4)
    w[:, 1, 2, [1, 2]] = w[:, 1, 2, [2, 1]].clone()
    return q


def test_tolerance_separates_fp32_from_subtle_bugs():
    gen = torch.Generator().manual_seed(3)
    n = 512
    for scale in (1.0, 30.0):
        p = oo.random_params(gen, scale)
        for kind in ("random", "sparse", "full"):
            x = _frames(kind, n, 4)
            r = _ratio(_fp32(p, x), x, p)
            print("scale %g %s: torch fp32 %.3f u M" % (scale, kind, r))
            assert r <= 1.0, (scale, kind, r)
        x = _frames("random", n, 5)
        by256 = _ratio(_fp32(p, x, 255.0 / 256.0), x, p)
        swapped = _ratio(_fp32(_swap_conv1_taps(p), x), x, p)
        print("scale %g: x/256 %.1f u M, swapped conv1 taps %.1f u M" % (scale, by256, swapped))
        assert by256 > oo.TOL_ULPS and swapped > oo.TOL_ULPS
        full = _frames("full", 64, 6)        # a constant frame cannot see the swap: why the tests use varying frames
        assert _ratio(_fp32(_swap_conv1_taps(p), full), full, p) <= 1.0


def test_action_rule_helpers():
    ref = np.array([[1.0, 2.0, 0.0], [1.0, 1.0, 0.0], [0.0, 1.0, 1.0 - 1e-9], [3.0, 0.0, 0.0]])
    mag = np.ones_like(ref)
    assert oo.decided(ref, mag).tolist() == [True, False, False, True]
    assert oo.greedy(np.array([[1.0, 1.0, 0.0], [0.0, 2.0, 2.0], [5.0, 5.0, 5.0]], np.float32)).tolist() == [0, 1, 0]


def test_cum_bounds_frequencies_match_the_weights():
    from scipy.stats import chisquare
    w = [1.0, 2.0, 0.5, 3.0, 1.5]
    cum = oo.cum_bounds(w)
    assert cum[-1] == 2 ** 32 and all(a < b for a, b in zip(cum, cum[1:]))
    ids = oo.opp_draw(cum, 1234, np.arange(65536, dtype=np.int64) + 2 ** 33, 3)
    counts = np.bincount(ids, minlength=len(w))
    expected = np.array(w) / sum(w) * len(ids)
    stat, p = chisquare(counts, expected)
    print("draw counts", counts.tolist(), "expected", expected.round(1).tolist(), "p = %.3f" % p)
    assert p > 1e-3


@pytest.mark.parametrize("w", [[0.0, 1.0, 2.0], [1.0, 0.0, 0.0, 2.0], [1.0, 2.0, 0.0], [0.0, 1.0, 0.0, 3.0, 0.0, 0.0],
                              [0.0, 0.0, 1.0]])
def test_zero_weights_are_never_drawn(w):
    cum = oo.cum_bounds(w)
    g = np.arange(65536, dtype=np.int64)
    ids = np.concatenate([oo.opp_draw(cum, 77, g, ep) for ep in (0, 1)])
    pos = [k for k, x in enumerate(w) if x > 0]
    assert set(np.unique(ids).tolist()) == set(pos)
    if w == [0.0, 0.0, 1.0]:
        assert (ids == 2).all() and cum == [0, 0, 2 ** 32]
    assert oo.opp_draw(cum, 77, 5, 1) == ids[65536 + 5]


def test_host_model_bookkeeping():
    """The model's episode book on a hand-checked case: sums, classification, credit to the old id, redraw keys."""
    m = oo.HostOpponents(4, seed=3, first_env=10)
    m.set_pool([oo.RULE_BASED, oo.RANDOM], [1.0, 1.0])
    m.assign([0, 1, 0, 1])
    frame = torch.zeros((4, 42, 42), dtype=torch.uint8)
    s = m.act(frame)
    assert s.actions[0] == s.actions[2] == 999 and s.actions[1] == oo.random_action(3, 11, 0)
    rew = np.array([[1, 0], [-1, 0], [0, 0], [0, 0]], np.float32)
    m.act(frame, rew, np.array([0, 1, 1, 0]), resample=True)
    assert m.stats[0].tolist() == [1, 0, 1, 0] and m.stats[1].tolist() == [1, 0, 0, 1]
    assert m.ret.tolist() == [1, 0, 0, 0] and m.episodes.tolist() == [0, 1, 1, 0]
    assert m.ids[1] == oo.opp_draw(m.cum, 3, 11, 1) and m.ids[2] == oo.opp_draw(m.cum, 3, 12, 1) and m.ids[3] == 1
    s = m.act(frame, rew, np.array([1, 0, 0, 0]))
    assert m.stats[0].tolist() == [2, 1, 1, 0] and m.acts == 3
    assert s.actions[3] == oo.random_action(3, 13, 2)
