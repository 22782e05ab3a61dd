"""Re-uploaded tables through the C ABI: crl_pong_inject_serves, crl_car_inject_tracks and crl_car_load_tracks free the
table they supersede, so a loop that re-injects does not grow device memory; and a handle that was given a table many
times plays exactly like a fresh handle given the last table once."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

CALLS = 16
MB = 1 << 20


def _free_bytes():
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info()[0]


def _assert_no_growth(upload, table_bytes):
    """upload(k) is the k-th re-upload of a table of table_bytes: after the last call free device memory has not fallen
    by more than one table (plus allocation granularity) below where the first call left it"""
    assert table_bytes >= 64 * MB
    upload(0)
    first = _free_bytes()
    for k in range(1, CALLS):
        upload(k)
    fall = first - _free_bytes()
    assert fall <= table_bytes + 2 * MB, (fall, table_bytes)


def _equal(x, y):
    return all(torch.equal(a, b) for a, b in zip(x, y)) if isinstance(x, tuple) else torch.equal(x, y)


def _assert_same_rollout(a, b, actions):
    assert _equal(a.reset(), b.reset())
    for act in actions:
        oa, ra, da, _ = a.step(act)
        ob, rb, db, _ = b.step(act)
        assert _equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)


def _serves(n, k, seed):
    """(vx, vy) per serve as Ball.reset draws them: vx = +-4, |vy| ~ U(1.2, 4)"""
    rng = np.random.default_rng(seed)
    vx = rng.choice([-4.0, 4.0], (n, k))
    vy = rng.uniform(4 * 0.3, 4, (n, k)) * rng.choice([-1.0, 1.0], (n, k))
    return np.stack([vx, vy], axis=2)


def test_inject_serves_replaces_its_table():
    from competitive_rl_b200 import make_envs
    N, K = 65536, 64
    kw = dict(num_envs=N, resized_dim=42, frame_stack=None, log_dir=None)
    envs = make_envs("cPongDouble-v0", **kw)
    _assert_no_growth(lambda k: envs.inject_serves(_serves(N, K, k)), N * K * 2 * 8)
    fresh = make_envs("cPongDouble-v0", serves=_serves(N, K, CALLS - 1), **kw)
    rng = np.random.default_rng(1)
    _assert_same_rollout(envs, fresh, [rng.integers(0, 3, (N, 2)).astype(np.int32) for _ in range(6)])
    envs.close()
    fresh.close()


def _draws(n, k, seed):
    """k track attempts per env as _create_track draws them: per checkpoint noise ~ U(0, 2pi/12), rad ~ U(R/3, R)"""
    import car_oracle as C
    rng = np.random.default_rng(seed)
    d = np.empty((n, k, 2 * C.CHECKPOINTS))
    d[:, :, 0::2] = rng.uniform(0, 2 * np.pi / C.CHECKPOINTS, (n, k, C.CHECKPOINTS))
    d[:, :, 1::2] = rng.uniform(C.TRACK_RAD / 3, C.TRACK_RAD, (n, k, C.CHECKPOINTS))
    return d


def _car_actions(n, steps):
    rng = np.random.default_rng(2)
    return [np.stack([rng.uniform(-0.3, 0.3, n), rng.uniform(0.2, 0.8, n)], 1).astype(np.float32) for _ in range(steps)]


def test_inject_tracks_replaces_its_tables():
    from competitive_rl_b200 import make_envs
    N, K, KB = 64, 5462, 8
    kw = dict(num_envs=N, frame_stack=4, log_dir=None)
    birth = np.zeros((N, KB, 1), np.int32)
    envs = make_envs("cCarRacing-v0", **kw)
    _assert_no_growth(lambda k: envs.inject_tracks(_draws(N, K, k), birth), N * K * 24 * 8 + birth.nbytes)
    fresh = make_envs("cCarRacing-v0", track_draws=_draws(N, K, CALLS - 1), birth=birth, **kw)
    _assert_same_rollout(envs, fresh, _car_actions(N, 6))
    envs.close()
    fresh.close()


def test_load_tracks_replaces_its_tables():
    import car_oracle as C
    from competitive_rl_b200 import make_envs
    N, T = 16, 5462
    kw = dict(num_envs=N, frame_stack=4, log_dir=None, seed=3)
    track = C.make_track(np.random.RandomState(4))[0]
    envs = make_envs("cCarRacing-v0", **kw)
    _assert_no_growth(lambda k: envs.load_tracks([track] * T if k < CALLS - 1 else []), T * (512 * 3 * 8 + 4))
    fresh = make_envs("cCarRacing-v0", **kw)
    fresh.load_tracks([])
    _assert_same_rollout(envs, fresh, _car_actions(N, 6))
    envs.close()
    fresh.close()
