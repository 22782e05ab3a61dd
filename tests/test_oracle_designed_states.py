"""PongOracleVec.set_state, state_in_domain and the designed-state generators (oracle/pong_designed.py) that the GPU
parity file tests/test_gpu_pong_designed_states.py drives both simulators with."""
import numpy as np
import pytest

import pong_designed as D
from pong_oracle import PongOracleVec, lib, make_serve_table, state_in_domain


def _oracle(n, atlas, fs=4, dim=84, max_rounds=21, env_id="cPongDouble-v0"):
    v = PongOracleVec(env_id, n, dim, fs, max_rounds, atlas, make_serve_table(n, 16, seed=4))
    v.reset()
    return v


def test_set_state_round_trip(atlas):
    v = _oracle(4, atlas)
    v.step(np.ones((4, 2), np.int32))
    moves = [(lib().pong_oracle_game_ptr(v._h, i).contents.left_move, lib().pong_oracle_game_ptr(v._h, i).contents.right_move)
             for i in range(4)]
    rows = np.array([[1, 2, -4.0, 0.1, 34, 179, 0, 21, 20, 0],
                     [156, 190, 64.0, -64.0, 0, 255, 21, 21, 0, 10000],
                     [78, 0, 1e-3, 0.0, 107, 107, 5, 6, 7, 8],
                     [3.75, 100.5, -2.5, 3.25, 40.9, 50.2, 1.9, 2.1, 3.99, 9.5]], np.float64)
    v.set_state(rows)
    got = v.get_state()
    want = rows.copy()
    want[:, [0, 1, 4, 5, 6, 7, 8, 9]] = np.trunc(want[:, [0, 1, 4, 5, 6, 7, 8, 9]])   # C (int) truncation
    assert np.array_equal(got, want)
    assert got[0, 3] == 0.1 and got[2, 2] == 1e-3        # velocities stored as given
    # Bat._current_move is the game's, not the state's: set_state leaves it alone
    assert moves == [(lib().pong_oracle_game_ptr(v._h, i).contents.left_move, lib().pong_oracle_game_ptr(v._h, i).contents.right_move)
                     for i in range(4)]


@pytest.mark.parametrize("max_rounds", [21, 3])
def test_goal_on_sub_step_0(atlas, max_rounds):
    """A ball at x = 1 with vx = -4 leaves through the left goal line on sub-step 0: reward -1 for agent 0, done exactly
    when num_rounds = max_rounds - 1; the terminal observation's newest frame pools the previous step's buffers."""
    v = _oracle(2, atlas, max_rounds=max_rounds)
    for _ in range(3):
        prev, _, _, _ = v.step(np.ones((2, 2), np.int32))
    st = v.get_state()
    st[:, 0], st[:, 1], st[:, 2], st[:, 3] = 1, 100, -4.0, 2.0
    st[:, 6], st[:, 7] = 3, 4
    st[0, 8], st[1, 8] = max_rounds - 1, max_rounds - 2
    v.set_state(st)
    obs, rew, done, info = v.step(np.ones((2, 2), np.int32))
    assert rew[:, 0].tolist() == [-1.0, -1.0] and rew[:, 1].tolist() == [1.0, 1.0]
    assert done.tolist() == [True, False]
    assert info["num_steps"][0] == 4 and info["real_reward"][0].tolist() == [-1.0, 1.0]
    for a in range(2):
        term = info["terminal_observation"][a][0]
        assert np.array_equal(term[:3], prev[a][0][1:])   # FrameStack shifted once
        assert np.array_equal(term[3], prev[a][0][3])     # stale buffers: the same pooled frame again
        assert not np.array_equal(obs[a][1][3], prev[a][1][3])   # env 1 went on: its buffers are fresh
    s = v.get_state()
    assert s[0].tolist()[6:9] == [0, 0, 0]                        # env 0 was reset
    assert s[1].tolist()[6:9] == [3, 5, max_rounds - 1]           # env 1: a point for the right player, one round more


@pytest.mark.parametrize("max_rounds", [1, 2, 21])
@pytest.mark.parametrize("n", [1, 3, 61, 509])
def test_generated_rows_in_domain(max_rounds, n):
    rng = np.random.default_rng(n * 31 + max_rounds)
    state = np.zeros((n, 10))
    state[:, 6] = rng.integers(0, 22, n)
    state[:, 7] = rng.integers(0, 22, n)
    for app in range(12):
        for kind in D.KINDS:
            rows = D.GENERATORS[kind](rng, state, max_rounds, app)
            assert rows.shape == (n, 10)
            ok = state_in_domain(rows, max_rounds)
            assert ok.all(), (kind, app, rows[~ok][:3])


def test_generators_reach_their_corners():
    """Over its applications the geometry class visits every ball_x, and the score class the corner scores."""
    rng = np.random.default_rng(0)
    xs, pairs = set(), set()
    state = np.zeros((61, 10))
    for app in range(30):
        xs.update(D.geometry(rng, state, 21, app)[:, 0].astype(int).tolist())
        pairs.update(map(tuple, D.scores(rng, state, 21, app)[:, 6:8].astype(int).tolist()))
    assert set(range(157)) <= xs
    assert {(0, 21), (21, 0), (21, 21), (20, 21)} <= pairs
    # one env, the score class's applications of the GPU file (0 and 3): a 21 with a point coming each time
    for app in (0, 3):
        r = D.scores(rng, np.zeros((1, 10)), 21, app)[0]
        assert (r[6] == 21 and r[2] > 0) or (r[7] == 21 and r[2] < 0), (app, r)
        assert r[0] in [D.goal_row(k, s)[0] for k in range(4) for s in "LR"] and r[8] < 20


def test_state_in_domain_rejects_each_field():
    base = np.array([78, 112, 4.0, -2.0, 107, 107, 3, 4, 5, 6], np.float64)
    assert state_in_domain(base[None], 21).all()
    rows, _ = D.out_of_domain_rows(base, 21)
    assert not state_in_domain(rows, 21).any()
    edge = np.array([[0, 0, -64.0, 64.0, 0, 0, 0, 0, 0, 0], [156, 190, 64.0, -64.0, 255, 255, 21, 21, 20, 10000]])
    assert state_in_domain(edge, 21).all()
    assert not state_in_domain(edge, 20)[1]


def test_goal_rows_score_on_their_sub_step(atlas):
    """goal_row(k, side) leaves on sub-step k: the point is scored, and the ball re-served, within that step."""
    for k in range(4):
        for side in "LR":
            v = _oracle(1, atlas, fs=None, dim=42)
            st = v.get_state()
            st[0, 0], st[0, 2] = D.goal_row(k, side)
            st[0, 1], st[0, 3], st[0, 8] = 100, 1.5, 0
            v.set_state(st)
            _, rew, _, _ = v.step(np.ones((1, 2), np.int32))
            assert rew[0, 0] == (-1.0 if side == "L" else 1.0), (k, side)
            s = v.get_state()[0]
            assert s[8] == 1 and s[9] == 3 - k, (k, side, s)     # frames played in the new round
