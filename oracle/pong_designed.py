"""Designed Pong game states for the oracle-parity tests -- TEST INFRASTRUCTURE ONLY.

Every generator returns an (N, 10) float64 array in get_state()'s layout (ball_x, ball_y, vx, vy, left_y, right_y,
score_left, score_right, num_rounds, num_steps) whose rows lie inside the set_state domain (pong_oracle.state_in_domain,
include/crl_b200.h).  Each class starts with an explicit list of corner rows, cycled through by `app` (the how-many-th
application this is, so that repeated applications with few envs still reach every corner), and fills the remaining rows
from a seeded numpy Generator.

Goal geometry used below: the ball moves first and scores when ball_x < 0 (the right player scores) or ball_x + 4 > 160
(the left player scores).  With vx = -4 a ball at x = 4k + 1 leaves on sub-step k (k = 0..3) and never meets the left bat
(that needs ball_x > 21 before the move); with vx = +4 a ball at x = 153 - 4k leaves on sub-step k and never meets the
right bat (that needs ball_x + 4 < 139).
"""
import numpy as np

KINDS = ("scores", "jump", "zero", "geometry")


def goal_row(k, side):
    """(ball_x, vx) of a ball that leaves the arena on sub-step k (0..3): side 'L' through the left goal line (a point for
    the right player), 'R' through the right one (a point for the left player)."""
    return (4 * k + 1, -4.0) if side == "L" else (153 - 4 * k, 4.0)


def _base(rng, n, max_rounds):
    """Ordinary mid-game rows: ball in the arena, moderate speed, scores and rounds with room left."""
    s = np.zeros((n, 10), np.float64)
    s[:, 0] = rng.integers(30, 127, n)
    s[:, 1] = rng.integers(40, 181, n)
    s[:, 2] = rng.choice([-1.0, 1.0], n) * rng.uniform(1.0, 8.0, n)
    s[:, 3] = rng.choice([-1.0, 1.0], n) * rng.uniform(0.5, 6.0, n)
    s[:, 4] = rng.integers(34, 180, n)
    s[:, 5] = rng.integers(34, 180, n)
    s[:, 6] = rng.integers(0, 19, n)
    s[:, 7] = rng.integers(0, 19, n)
    s[:, 8] = rng.integers(0, max(1, max_rounds - 1), n)
    s[:, 9] = rng.integers(0, 60, n)
    return s


def _goal(s, i, k, side, rng):
    s[i, 0], s[i, 2] = goal_row(k, side)
    s[i, 1] = rng.integers(60, 171)
    s[i, 3] = rng.choice([-1.0, 1.0]) * rng.uniform(1.2, 4.0)


def scores(rng, state, max_rounds, app=0):
    """Scores over the whole atlas: the corners 0:21, 21:0, 21:21, 20:21; rows one point before a score change on each
    sub-step 0..3; and 21:x / x:21 rows with a point coming while rounds remain, whose next frames show a score of 22
    (outside the atlas: no text)."""
    n = len(state)
    s = _base(rng, n, max_rounds)
    s[:, 6] = rng.integers(0, 22, n)
    s[:, 7] = rng.integers(0, 22, n)
    s[:, 8] = rng.integers(0, max_rounds, n)
    # the rows that take a score to 22 come first, so that batches of one or three envs meet the blank-text rule too
    corners = []
    for k in range(4):
        corners += [(21, None, k, "R"), (None, 21, k, "L"), (21, 21, k, "R"), (21, 21, k, "L")]
    corners += [(0, 21, None, None), (21, 0, None, None), (21, 21, None, None), (20, 21, None, None)]
    for k in range(4):
        corners += [(None, None, k, "L"), (None, None, k, "R")]
    m = len(corners)
    for i in range(min(n, m)):
        l, r, k, side = corners[(i + app * n) % m]
        if l is not None:
            s[i, 6] = l
        if r is not None:
            s[i, 7] = r
        if k is not None:
            _goal(s, i, k, side, rng)
            if l == 21 or r == 21:      # the point takes a score to 22 and the game goes on
                s[i, 8] = rng.integers(0, max(1, max_rounds - 1))
    # the other rows: every fourth one scores on a random sub-step
    for i in range(m, n, 4):
        _goal(s, i, int(rng.integers(0, 4)), "L" if rng.random() < 0.5 else "R", rng)
    return s


def jump(rng, state, max_rounds, app=0):
    """Scores moved by >= 2 points from what the env shows, num_rounds = max_rounds - 1 and the ball one sub-step from
    a goal line: the done on sub-step 0..2 pools a fresh frame (or none) with a stale one from before the jump."""
    n = len(state)
    s = _base(rng, n, max_rounds)
    old = np.asarray(state, np.float64)[:, 6:8]
    for i in range(n):
        while True:
            l, r = rng.integers(0, 22, 2)
            if max(abs(l - old[i, 0]), abs(r - old[i, 1])) >= 2:
                break
        s[i, 6], s[i, 7] = l, r
        _goal(s, i, (i + app) % 3, "L" if (i // 3 + app) % 2 else "R", rng)
    s[:, 8] = max_rounds - 1
    return s


def zero(rng, state, max_rounds, app=0):
    """For the step right after construction and reset(): half the rows end the episode on sub-step 0 or 1, while both
    MaxAndSkip buffers still hold np.zeros frames, so the terminal observation's newest frame is the all-zero frame."""
    n = len(state)
    s = _base(rng, n, max_rounds)
    for i in range(0, n, 2):
        _goal(s, i, (i // 2 + app) % 2, "L" if (i // 4 + app) % 2 else "R", rng)
        s[i, 8] = max_rounds - 1
    return s


def geometry(rng, state, max_rounds, app=0):
    """Ball and bat geometry: every ball_x in [0, 156] over the applications; the ball above the arena (rows 0..33,
    under the scoreboard) and on the bottom border; the ball over each bat and each 4-column bat strip; the ball across
    the centre column agent 1's view mirrors about; bats at 34 and 179 (and at 0 / 255, which the next move clamps);
    large velocities; num_steps at the round's time limit."""
    n = len(state)
    s = _base(rng, n, max_rounds)
    sign = lambda: rng.choice([-1.0, 1.0])   # noqa: E731
    for i in range(n):
        j = i + app * n
        sub = j % 8
        if sub == 0:                                    # every ball_x
            s[i, 0] = (j // 8) % 157
            s[i, 2] = sign() * rng.uniform(0.25, 3.0)
        elif sub == 1:                                  # above the arena, drifting sideways
            s[i, 0] = rng.integers(0, 157)
            s[i, 1] = rng.integers(0, 34)
            s[i, 2] = sign() * rng.uniform(0.5, 4.0)
            s[i, 3] = rng.choice([0.0, 0.25, -0.25, 0.5])
        elif sub == 2:                                  # bottom border
            s[i, 1] = rng.integers(184, 191)
            s[i, 3] = sign() * rng.uniform(0.0, 6.0)
        elif sub in (3, 4):                             # over a bat / its destination strip
            left = sub == 3
            bat = int(rng.integers(34, 180))
            s[i, 4 if left else 5] = bat
            s[i, 0] = rng.integers(8, 29) if left else rng.integers(128, 150)
            s[i, 1] = min(190, max(0, bat + int(rng.integers(-4, 16))))
            s[i, 2] = sign() * rng.uniform(0.0, 1.0)
            s[i, 3] = sign() * rng.uniform(0.0, 1.0)
        elif sub == 5:                                  # across the mirror's centre column
            s[i, 0] = rng.integers(74, 83)
            s[i, 1] = rng.integers(34, 191)
            s[i, 2] = sign() * rng.uniform(0.0, 0.5)
        elif sub == 6:                                  # bats at the extremes, ball near a strip
            s[i, 4] = rng.choice([0, 34, 35, 178, 179, 255])
            s[i, 5] = rng.choice([0, 34, 35, 178, 179, 255])
            s[i, 0] = rng.choice([rng.integers(8, 29), rng.integers(128, 150)])
            s[i, 1] = rng.choice([rng.integers(30, 50), rng.integers(170, 191)])
            s[i, 2] = sign() * rng.uniform(0.0, 2.0)
        else:                                           # fast balls, the round's time limit
            s[i, 2] = sign() * rng.uniform(8.0, 64.0)
            s[i, 3] = sign() * rng.uniform(0.0, 64.0)
            s[i, 9] = rng.choice([9999, 10000])
    return s


GENERATORS = {"scores": scores, "jump": jump, "zero": zero, "geometry": geometry}


def out_of_domain_rows(base, max_rounds):
    """(rows, column changed) pairs: each row is `base` (a row inside the domain) with one field set just outside the
    set_state domain."""
    bad = [(0, 157), (0, -1), (1, 191), (1, 300), (1, -1), (2, np.nan), (3, np.inf), (2, 64.5), (3, -64.0001),
           (4, 256), (5, -1), (6, 22), (7, -1), (8, max_rounds), (9, 10001), (0, 3.5), (6, 0.5), (9, -0.25)]
    rows = []
    for col, v in bad:
        r = np.array(base, np.float64).copy()
        r[col] = v
        rows.append(r)
    return np.stack(rows), [c for c, _ in bad]
