"""The float64 references of oracle/car_designed.py against the C oracle, and the seam geometry the designed sensor
placements rely on.  CPU only: these validate the references before the GPU tests use them."""
import numpy as np
import pytest

import car_designed as D


@pytest.fixture(scope="module")
def tracks():
    return D.long_seam_tracks(3)


def test_sensor_reference_matches_oracle(tracks):
    """Per-wheel tile counts and tiles visited after set_state + one step, wherever every margin is more than 1e-4 from
    zero: the float64 SAT margins decide the same overlaps as the oracle's fp32 sensor test over its tile AABBs."""
    import car_oracle as C
    o = C.CarOracleEnv(1, 1, None, render=False)
    rng = np.random.default_rng(3)
    checked = seam = 0
    for tr, bd, _ in tracks:
        polys = D.tile_polygons(tr)
        for app in range(2):
            for r in D.sensor_rows(rng, tr, 90, app, polys):
                o.reset(tr, bd, [0])
                o.set_state(r[None])
                o.step(np.zeros((1, 2)))
                s = o.get_state()[0]
                cnt, tiles, near_zero = D.sensor_reference(polys, r)
                if near_zero:
                    continue
                assert np.array_equal(s[[9, 13, 17, 21]], cnt), (r, cnt)
                assert s[23] == len(tiles)
                checked += 1
                seam += 0 in tiles
    assert checked >= 450 and seam >= 100, (checked, seam)


def test_wheel_model_reference_matches_oracle(tracks):
    """omega of every wheel after the first step that follows set_state, float64 model against the oracle.  The oracle
    computes the wheel velocity in float32 (one ulp at 100 units/s is 8e-6, and d omega / d v_forward is 0.55 without
    the friction limit); measured worst relative difference 5.6e-6."""
    import car_oracle as C
    o = C.CarOracleEnv(1, 1, None, render=False)
    rng = np.random.default_rng(4)
    tr, bd, _ = tracks[0]
    worst = 0.0
    for app in range(2):
        rows = D.wheel_rows(rng, tr, 40, app)
        for i, r in enumerate(rows):
            for a in D.WHEEL_ACTIONS[(i + app) % 3::3]:
                o.reset(tr, bd, [0])
                o.set_state(r[None])
                o.step(a[None].astype(np.float64))
                om = o.get_state()[0, [7, 11, 15, 19]]
                ref = D.wheel_omega_step1(r, a)
                err = np.abs(om - ref) / np.maximum(1.0, np.abs(ref))
                worst = max(worst, float(err.max()))
    print("wheel model: worst relative omega difference %.3g" % worst)
    assert worst <= 2e-5


def test_seam_tile_reaches_past_the_prefilter_radius(tracks):
    """The designed seam placements reach the part of the seam tile that lies more than 9 units (the kernel's candidate
    radius around a tile's track point, less the wheel's 0.63 reach) from track point 0, while every other tile stays
    within the radius.  Measured on 300 generated tracks (RandomState(1)): non-seam reach <= 7.99, seam reach 8.4-17.3."""
    rng = np.random.default_rng(5)
    beyond = 0
    for tr, bd, _ in tracks:
        reach = D.tile_reach(tr)
        assert reach[1:].max() < 8.3 and reach[0] > 9.5, reach[0]
        polys = D.tile_polygons(tr)
        p0 = tr[0, 2:4]
        for r in D.sensor_rows(rng, tr, 60, 0, polys):
            m = D.wheel_tile_margins(polys, r)
            wp = D.wheel_poses(r)
            for k in range(4):
                if m[k, 0] < -1e-3 and np.hypot(*(wp[k, :2] - p0)) > 9.0 and (m[k, 1:] > 0).all():
                    beyond += 1
    assert beyond >= 10, beyond
    rs = np.random.RandomState(1)
    import car_oracle as C
    long_ = 0
    for _ in range(40):
        tr, _, _ = C.make_track(rs)
        reach = D.tile_reach(tr)
        assert reach[1:].max() < 8.3
        long_ += reach[0] > 8.37
    assert long_ >= 35, long_


def test_coarse_track_counts_wide_tiles():
    """A generated track with one point dropped has a second long tile (and its group neighbours); with every other point
    dropped it has far more than the kernel lists per track, and loading it must be refused."""
    tr = D.long_seam_tracks(1)[0][0]
    one = np.delete(tr, 100, axis=0)
    assert D.tile_reach(one)[100] > 9.0
    half = tr[::2]
    assert (D.tile_reach(half) > 8.25).sum() > 4
