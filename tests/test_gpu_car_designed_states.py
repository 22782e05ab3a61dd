"""The car step kernel from designed states (oracle/car_designed.py) against the C oracle and the float64 references:
wheel-tile sensors (car_sensor_kernel and, for action_repeat > 1, the in-thread sensor_car_overlaps), the wheel model,
the tile ledger and reward rule, episode ends, and two cars from designed relative poses.

Measured maxima on the B200 (the bounds below are about 20x tighter than the 0.02 of test_gpu_car_parity.py or better):
  * per-wheel tile counts and tiles visited: identical to the oracle on every row, near-zero margins included;
  * omega after the first step against the float64 wheel model: relative 9.4e-6 (float32 wheel velocity, see
    test_car_designed_cpu.py), bound 2e-5;
  * hull pose after 1 / 2 / 5 steps of the wheel-model rows: 7.6e-6, bound WHEEL_POSE_TOL = 1e-4; two cars from
    designed contacts over 5 steps: 1.5e-5, bound PAIR_POSE_TOL = 1e-4; 40 steps after a playfield exit (car0 mode):
    bound 1e-3 (printed)."""
import numpy as np
import pytest

import car_designed as D

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ENV_IDS = ["cCarRacing-v0", "cCarRacingDouble-v0"]
N_TRACKS = 4
WHEEL_POSE_TOL = 1e-4        # position / angle after 1, 2, 5 steps; measured 7.6e-6 (velocity 1.5e-5, bound 2e-4)
PAIR_POSE_TOL = 1e-4         # measured 1.5e-5


@pytest.fixture(scope="module")
def tracks():
    return D.long_seam_tracks(N_TRACKS)


def _make(env_id, n, tracks, action_repeat=1, **kw):
    from competitive_rl_b200 import make_envs
    P = 2 if "Double" in env_id else 1
    draws = np.stack([np.tile(tracks[e % len(tracks)][2], (16, 1)) for e in range(n)])
    birth = np.tile(np.arange(P)[None, None], (n, 16, 1)).astype(np.int32)
    return make_envs(env_id, num_envs=n, log_dir=None, frame_stack=1, track_draws=draws, birth=birth,
                     action_repeat=action_repeat, **kw)


class _Oracles(object):
    """One oracle env per track, reset for every row (a fresh episode, like the vec-env's reset)."""

    def __init__(self, tracks, P, action_repeat=1):
        import car_oracle as C
        self.tracks, self.P = tracks, P
        self.envs = [C.CarOracleEnv(P, action_repeat, None, render=False) for _ in tracks]

    def run(self, e, state, actions_seq):
        k = e % len(self.tracks)
        o = self.envs[k]
        o.reset(self.tracks[k][0], self.tracks[k][1], list(range(self.P)))
        o.set_state(state)
        out = []
        for a in actions_seq:
            _, r, d, _ = o.step(np.asarray(a, np.float64).reshape(self.P, 2))
            out.append((o.get_state(), r.copy(), d.copy(), o.contacts()[0]))
        return out


def _sensor_batch(tracks, n, P, app, seed):
    """n env rows: car 0 from the designed sensor placements (all corners reached over the batch), car 1 far away."""
    rng = np.random.default_rng(seed)
    per = [D.sensor_rows(rng, tracks[k][0], (n + len(tracks) - 1) // len(tracks) + 1, app, None) for k in range(len(tracks))]
    st = np.zeros((n, P, 24))
    for e in range(n):
        k = e % len(tracks)
        st[e, 0] = per[k][e // len(tracks)]
        if P == 2:
            tr = tracks[k][0]
            st[e, 1] = D.road_row(tr, len(tr) // 2 + int(rng.integers(-20, 20)))
    return st


def _check_sensors(envs, orc, tracks, st, act, P):
    envs.set_state(st)
    envs.step(act if P == 2 else act[:, 0])
    sg = envs.get_state().cpu().numpy()
    polys = {}
    diff = 0
    for e in range(len(st)):
        so = orc.run(e, st[e], [act[e]])[0][0]
        for c in range(P):
            g, o = sg[e, c, [9, 13, 17, 21, 23]], so[c, [9, 13, 17, 21, 23]]
            if np.array_equal(g, o):
                continue
            # a difference is allowed only on a row with a margin within 1e-4 of zero where the oracle's own fp32 test
            # disagrees with the float64 reference
            k = e % len(tracks)
            polys.setdefault(k, D.tile_polygons(tracks[k][0]))
            cnt, tiles, near = D.sensor_reference(polys[k], st[e, c])
            assert near and not (np.array_equal(o[:4], cnt) and o[4] == len(tiles)), (e, c, g, o, cnt, st[e, c])
            diff += 1
    return diff


@pytest.mark.parametrize("env_id", ENV_IDS)
@pytest.mark.parametrize("n", [1, 33, 4099])
def test_sensor_counts_from_designed_placements(env_id, n, tracks):
    """set_state + one step: per-wheel tile counts [9 + 4k] and tiles visited [23] equal the oracle's, for wheels
    straddling tile edges, corners and bump vertices, on the seam tile, inside the sharpest turn and just off the road.
    Three applications per env (the visited bits of earlier ones carry over on both sides)."""
    P = 2 if "Double" in env_id else 1
    envs = _make(env_id, n, tracks)
    orc = _Oracles(tracks, P)
    envs.reset()
    for app in range(3 if n < 4099 else 1):
        envs.reset()
        st = _sensor_batch(tracks, n, P, app, 100 + app)
        act = np.zeros((n, P, 2), np.float32)
        _check_sensors(envs, orc, tracks, st, act, P)
    envs.check()
    envs.close()


@pytest.mark.parametrize("env_id", ENV_IDS)
@pytest.mark.parametrize("action_repeat", [2, 3])
def test_sensor_counts_in_thread_substeps(env_id, action_repeat, tracks):
    """action_repeat > 1: the later sub-steps recompute the overlaps inside the step kernel (sensor_car_overlaps).  The
    placements are at rest with the steering holding the front wheels, so they stay put through the sub-steps."""
    P = 2 if "Double" in env_id else 1
    n = 33
    envs = _make(env_id, n, tracks, action_repeat=action_repeat)
    orc = _Oracles(tracks, P, action_repeat)
    for app in range(2):
        envs.reset()
        st = _sensor_batch(tracks, n, P, app, 200 + app)
        act = np.zeros((n, P, 2), np.float32)
        r0, a0 = D.at_rest(st[:, 0])
        st[:, 0], act[:, 0] = r0, a0
        _check_sensors(envs, orc, tracks, st, act, P)
    envs.check()
    envs.close()


def test_coarse_loaded_track(tracks):
    """A recorded track with one point dropped has a second long tile besides the seam: the kernel lists both and the
    wheels on them match the oracle.  With every other point dropped the track has more such tiles than the kernel lists
    per track, and load_tracks refuses it."""
    import car_oracle as C
    tr = np.delete(tracks[0][0], 100, axis=0)
    bd = C.track_border(tr)
    n = 64
    envs = _make("cCarRacing-v0", n, tracks)
    envs.load_tracks([tr])
    envs.reset()
    assert np.array_equal(envs.get_track(0), tr[:, 1:])
    rng = np.random.default_rng(7)
    rows = D.sensor_rows(rng, tr, n, 0, None)
    p = tr[:, 2:4]
    for i in range(0, n, 2):                       # half the rows on the long tile (points 99 .. 100 of the new track)
        f, lat = rng.uniform(0.05, 0.95), rng.uniform(-0.8, 0.8)
        c = p[99] + f * (p[100] - p[99]) + lat * D.TRACK_WIDTH * np.array([np.cos(tr[100, 1]), np.sin(tr[100, 1])])
        rows[i] = D.placed_row(c, i // 2 % 4, rng.uniform(-np.pi, np.pi), rng.uniform(-0.5, 0.5))
    orc = _Oracles([(tr, bd, None)], 1)
    _check_sensors(envs, orc, [(tr, bd, None)], rows[:, None], np.zeros((n, 1, 2), np.float32), 1)
    with pytest.raises(Exception, match="reach farther"):
        envs.load_tracks([tracks[0][0][::2]])
    envs.close()


@pytest.mark.parametrize("env_id", ENV_IDS)
def test_wheel_model(env_id, tracks):
    """Wheel-model rows x actions (brake 0.3 / 0.89 / 0.9 / 1.0, steering past the joint limits, actions outside
    [-1, 1], -0.0 and 0): omega after step 1 against the float64 model, hull pose, velocity and omega against the oracle
    after 1, 2 and 5 steps (step 2 is the first with road friction)."""
    P = 2 if "Double" in env_id else 1
    acts = D.WHEEL_ACTIONS
    rows = D.wheel_rows(np.random.default_rng(11), tracks[0][0], 26, 0)
    n = len(rows) * len(acts) // 2
    st = np.zeros((n, P, 24))
    act = np.zeros((n, P, 2), np.float32)
    for e in range(n):
        st[e, 0] = rows[e % len(rows)]
        act[e, 0] = acts[(e // len(rows) * 2 + e % 2) % len(acts)]
        if P == 2:
            act[e, 1] = acts[(e + 3) % len(acts)]
    for e in range(n):                               # the tracks differ per env: car 0 onto its own track, car 1 far from it
        tr = tracks[e % N_TRACKS][0]
        t = int(e * 7 % len(tr))
        if P == 2:
            st[e, 1] = D.road_row(tr, (t + len(tr) // 2) % len(tr))
        st[e, 0, 0:2] = tr[t, 2:4]
        st[e, 0, 2] = tr[t, 1] + 0.1 * ((e % 5) - 2)
    envs = _make(env_id, n, tracks, max_episode_steps=0)
    orc = _Oracles(tracks, P)
    envs.reset()
    envs.set_state(st)
    ref = [orc.run(e, st[e], [act[e]] * 5) for e in range(n)]
    worst_om, worst = 0.0, np.zeros(3)
    for t in range(5):
        envs.step(act if P == 2 else act[:, 0])
        sg = envs.get_state().cpu().numpy()
        for e in range(n):
            so = ref[e][t][0]
            if t == 0:
                om = D.wheel_omega_step1(st[e, 0], act[e, 0])
                worst_om = max(worst_om, float((np.abs(sg[e][0, [7, 11, 15, 19]] - om) / np.maximum(1, np.abs(om))).max()))
            if ref[e][t][2].any():
                continue
            worst[0] = max(worst[0], np.abs(sg[e, :, :3] - so[:, :3]).max())
            worst[1] = max(worst[1], np.abs(sg[e, :, 3:6] - so[:, 3:6]).max())
            om_g, om_o = sg[e][:, [7, 11, 15, 19]], so[:, [7, 11, 15, 19]]
            worst[2] = max(worst[2], (np.abs(om_g - om_o) / np.maximum(1, np.abs(om_o))).max())
            if t in (0, 1, 4):
                assert np.abs(sg[e, :, :3] - so[:, :3]).max() <= WHEEL_POSE_TOL, (t, e, sg[e, :, :3], so[:, :3])
    print("wheel model: omega step 1 vs float64 %.3g; vs oracle pose %.3g, velocity %.3g, omega (rel) %.3g"
          % (worst_om, worst[0], worst[1], worst[2]))
    assert worst_om <= 2e-5
    assert worst[1] <= 2 * WHEEL_POSE_TOL and worst[2] <= 1e-3
    envs.check()
    envs.close()


def _ledger_orders(n):
    fwd = list(range(1, n)) + [0, 1, 2, 3]
    orders = {"forward": fwd, "backward": list(range(n - 1, 0, -1)), "seam_start": [0, n - 1, 1, n - 2, 2, 3, 0]}
    for j in (48, 49, 50, 51, 52):
        orders["jump%d" % j] = [1, 2, 3, 3 + j, 4 + j, 4 + 2 * j, 5 + 2 * j, 3 + 3 * j]
    return orders


def test_tile_ledger_by_teleport(tracks):
    """A car moved along its own track with set_state (the visited bits stay) and stepped each time: every tile forward
    through the seam to the lap-completion done, jumps of 48..52 tiles around the '< 50 tiles since the last rewarded
    tile' rule, backwards, and starting on the seam tile.  Per-step rewards, [22], tiles visited and done equal the oracle;
    episode_stats() equals a tally of the oracle's dones."""
    import car_oracle as C
    tr, bd, d = tracks[0]
    nt = len(tr)
    orders = _ledger_orders(nt)
    names = sorted(orders)
    n = len(names)
    envs = _make("cCarRacing-v0", n, [tracks[0]], max_episode_steps=0)
    envs.reset()
    orcs = [C.CarOracleEnv(1, 1, None, render=False) for _ in range(n)]
    for o in orcs:
        o.reset(tr, bd, [0])
    T = max(len(v) for v in orders.values()) + 1
    live = np.ones(n, bool)
    dones, tiles_at_done = 0, 0
    for t in range(T):
        sg0 = envs.get_state().cpu().numpy()
        st = sg0.copy()
        for e, name in enumerate(names):
            seq = orders[name]
            st[e, 0] = D.road_row(tr, seq[min(t, len(seq) - 1)]) if live[e] else D.road_row(tr, 0)
            st[e, 0, 22] = sg0[e, 0, 22]
        envs.set_state(st)
        _, r, dn, info = envs.step(np.zeros((n, 2), np.float32))
        rg, dg, sg = info.rewards.cpu().numpy()[:, 0], dn.cpu().numpy().reshape(n), envs.get_state().cpu().numpy()
        for e in range(n):
            if not live[e]:
                continue
            orcs[e].set_state(st[e])
            _, ro, do, _ = orcs[e].step(np.zeros((1, 2)))
            so = orcs[e].get_state()[0]
            assert abs(rg[e] - ro[0]) <= 1e-4, (names[e], t, rg[e], ro[0])
            assert bool(dg[e]) == bool(do[0]), (names[e], t)
            if do[0]:
                live[e] = False
                dones += 1
                tiles_at_done += int(so[23])
                continue
            assert sg[e, 0, 23] == so[23] and abs(sg[e, 0, 22] - so[22]) <= 1e-6, (names[e], t)
    assert not live[names.index("forward")]            # the forward lap completed
    es = envs.episode_stats()
    assert es["episodes"] == dones and es["mean_tiles"] * dones == tiles_at_done, (es, dones, tiles_at_done)
    envs.check()
    envs.close()


@pytest.mark.parametrize("done_mode", ["any", "car0"])
def test_playfield_exit(done_mode, tracks):
    """Car 1 put just outside (or inside) the playfield at rest, car 0 driving on the road.  'any': the env ends on the
    first step exactly when the oracle says car 1 left.  'car0': the env goes on; the finished car 1 is no longer driven,
    keeps being integrated and falls asleep -- both cars against the oracle for 40 steps."""
    rng = np.random.default_rng(13)
    rows = D.playfield_rows(rng, 16)
    n = len(rows)
    st = np.zeros((n, 2, 24))
    for e in range(n):
        tr = tracks[e % N_TRACKS][0]
        st[e, 0] = D.road_row(tr, 10 + e)
        st[e, 1] = rows[e]
    act = np.zeros((n, 2, 2), np.float32)
    act[:, 0] = [0.1, 0.4]
    act[:, 1] = [0.5, 1.0]
    envs = _make("cCarRacingDouble-v0", n, tracks, done_mode=done_mode, max_episode_steps=0)
    orc = _Oracles(tracks, 2)
    envs.reset()
    envs.set_state(st)
    T = 40 if done_mode == "car0" else 1
    ref = [orc.run(e, st[e], [act[e]] * T) for e in range(n)]
    outside = np.abs(rows[:, :2]).max(1) > D.PLAYFIELD
    worst = 0.0
    for t in range(T):
        _, _, dn, _ = envs.step(act)
        dg = dn.cpu().numpy().reshape(n)
        sg = envs.get_state().cpu().numpy()
        for e in range(n):
            so, ro, do, _ = ref[e][t]
            if t == 0:                               # rows just inside may be driven out later
                assert do[1] == outside[e] and not do[0], (e, t)
            assert bool(dg[e]) == (bool(do.any()) if done_mode == "any" else bool(do[0])), (e, t)
            if done_mode == "car0":
                worst = max(worst, np.abs(sg[e, :, :3] - so[:, :3]).max())
                assert np.abs(sg[e, :, :3] - so[:, :3]).max() <= 1e-3, (e, t)
                assert sg[e, 1, 22] == so[1, 22]
    print("playfield exit (%s): pose %.3g" % (done_mode, worst))
    envs.close()


@pytest.mark.parametrize("env_id", ENV_IDS)
def test_internal_step_count_done(env_id, tracks):
    """max_episode_steps=0 (no TimeLimit): the reference's own step_count > 1000 ends the episode on step 1002."""
    P = 2 if "Double" in env_id else 1
    n = 3
    envs = _make(env_id, n, tracks, max_episode_steps=0)
    envs.reset()
    import car_oracle as C
    orcs = [C.CarOracleEnv(P, 1, None, render=False) for _ in range(n)]
    for e, o in enumerate(orcs):
        o.reset(*tracks[e][:2], list(range(P)))
    a = np.zeros((n, P, 2), np.float32)
    done_at = []
    for t in range(1002):
        _, _, dn, info = envs.step(a if P == 2 else a[:, 0])
        if t >= 999:
            done_at.append(dn.cpu().numpy().reshape(n).copy())
    for o in orcs:
        for t in range(1002):
            _, _, do, ns = o.step(a[0].astype(np.float64))
            if t == 1000:
                assert not do.any()
        assert do.all() and ns == 1002
    assert not done_at[0].any() and not done_at[1].any() and done_at[2].all()
    envs.close()


PAIR_POSES = [  # (dx, dy, dangle) of car 1 in car 0's frame; lateral gaps between the wheel boxes -0.05, 0, 0.02, 0.2
    (2.76 - 0.05, 0.0, 0.0), (2.76, 0.0, 0.0), (2.76 + 0.02, 0.0, 0.0), (2.76 + 0.2, 0.0, 0.0),
    (0.0, 5.0 + 0.01, 0.0), (0.0, 5.0 - 0.05, 0.0), (0.0, -5.0 + 0.02, 0.0),        # nose to tail
    (1.2 + 1.64 + 0.27, 0.3, np.pi / 2), (1.2 + 1.64 + 0.3, -1.0, -np.pi / 2),     # a wheel of car 1 against car 0's side
]


def test_two_cars_from_designed_relative_poses(tracks):
    """Two cars side by side, nose to tail and wheel to hull, mixed with far-apart envs in one batch: the near list,
    car_collide_kernel and both stepping passes run in the same step.  First-step get_contacts() equals the oracle's
    contact count; poses stay within PAIR_POSE_TOL of the oracle for 5 steps."""
    n = 2 * len(PAIR_POSES) + 5
    st = np.zeros((n, 2, 24))
    act = np.zeros((n, 2, 2), np.float32)
    rng = np.random.default_rng(17)
    for e in range(n):
        tr = tracks[e % N_TRACKS][0]
        base = D.road_row(tr, 20 + 3 * e, lateral=-1.5)
        st[e, 0] = base
        if e < len(PAIR_POSES) * 2 and e % 2 == 0:
            dx, dy, da = PAIR_POSES[e // 2]
            c, s = np.cos(base[2]), np.sin(base[2])
            st[e, 1] = base
            st[e, 1, 0:2] = base[0:2] + np.array([c * dx - s * dy, s * dx + c * dy])
            st[e, 1, 2] = base[2] + da
        else:
            st[e, 1] = D.road_row(tr, 20 + 3 * e + 40)
        act[e] = rng.uniform(-0.3, 0.6, (2, 2))
    envs = _make("cCarRacingDouble-v0", n, tracks, max_episode_steps=0)
    orc = _Oracles(tracks, 2)
    envs.reset()
    envs.set_state(st)
    ref = [orc.run(e, st[e], [act[e]] * 5) for e in range(n)]
    worst = 0.0
    touched = 0
    for t in range(5):
        envs.step(act)
        sg = envs.get_state().cpu().numpy()
        cg, over = envs.get_contacts()
        assert over == 0
        for e in range(n):
            so, _, _, co = ref[e][t]
            if t == 0:
                assert cg[e] == co, (e, cg[e], co)
                touched += co > 0
            worst = max(worst, np.abs(sg[e, :, :3] - so[:, :3]).max())
            assert np.abs(sg[e, :, :3] - so[:, :3]).max() <= PAIR_POSE_TOL, (t, e)
    print("two cars: pose %.3g, envs touching %d" % (worst, touched))
    assert touched >= 5
    envs.check()
    envs.close()
