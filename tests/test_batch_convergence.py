"""A batch handle's driver loop with one convergence monitor per trajectory (ConcatBatch.iterate_until,
icmslam_batch_iterate_until) against Engine.iterate_until on each trajectory alone (run with `-m gpu`)."""
import os

import numpy as np
import pytest

from helpers import CONFIG_ROS

pytestmark = pytest.mark.gpu

K, TK, MAX_SWEEPS = 7, 1024, 12
CFGD = dict(L=2048, cota=20.0)      # (room for the labels trajectory 2 creates every sweep)
TOL_XY, TOL_TH, TOL_MAP, TOL_CAMBIO = 1e-9, 1e-11, 1e-9, 1e-9      # the fp64 translation of each trajectory into its region


def _cfg():
    from icm_slam_b200.config import ConfigICM
    d = dict(CONFIG_ROS)
    d.update(CFGD)
    return ConfigICM.from_values(**d)


def _data():
    """K trajectories whose initial poses are perturbed by different amounts (so they converge after different numbers of
    sweeps), one with a missing landmark (its far observations create labels), one with empty scans inside it and one with a
    duplicated landmark (the two merge in the first sweep, so that trajectory's calc_cambio needs the full search)."""
    from icm_slam_b200.synthetic import make_synthetic_loop
    data = [make_synthetic_loop(16, T=TK, seed=20181 + 300 + i, init_pose_noise=(0.03 * (i + 1), 0.006 * (i + 1))) for i in range(K)]
    data[2]["map_init"] = np.delete(data[2]["map_init"], 5, axis=1)
    data[4]["observations"][:, 300:310] = 10.0
    data[5]["map_init"] = np.concatenate([data[5]["map_init"], data[5]["map_init"][:, 3:4] + np.array([[0.4], [0.0]])], axis=1)
    return data


def _alone(d):
    from icm_slam_b200.engine import Engine
    e = Engine(_cfg())
    e.load(d["observations"], d["odometry"], d["velocities"], precondition=True)
    e.extract()
    e.set_map(d["map_init"])
    e.set_poses(d["x_init"])
    return e


def _batch(data, env=None):
    from icm_slam_b200.batch import ConcatBatch
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        b = ConcatBatch(_cfg(), 0, 1, device=0)
        for i, d in enumerate(data):
            b.add(i, d["observations"], d["odometry"], d["velocities"], d["map_init"], d["x_init"])
        b.finalize()
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    return b


def _pick_tol(histories):
    """A tolerance that no sweep's largest change comes within 1 % of, chosen to spread the stopping sweeps widely."""
    allmax = np.concatenate([h[:, 1] for h in histories])
    best = None
    for tol in np.geomspace(allmax.min() * 1.5, allmax.max(), 400):
        if np.any(np.abs(allmax - tol) <= 0.01 * tol):
            continue
        n = [int(np.argmax(h[:, 1] <= tol)) + 1 if np.any(h[:, 1] <= tol) else len(h) for h in histories]
        if best is None or len(set(n)) > best[0]:
            best = (len(set(n)), float(tol))
    return best[1]


@pytest.fixture(scope="module")
def case():
    data = _data()
    hist = []
    for d in data:
        e = _alone(d)
        n, cam = e.iterate_until(d["odometry"][:, 0], MAX_SWEEPS, 0.0)
        assert n == MAX_SWEEPS
        hist.append(cam)
        e.close()
    tol = _pick_tol(hist)
    ref = []
    for d in data:
        e = _alone(d)
        n, cam = e.iterate_until(d["odometry"][:, 0], MAX_SWEEPS, tol)
        x1, m1 = e.get_poses(), e.get_map()
        e.iterate(None, d["odometry"][:, 0], 2)
        ref.append(dict(n=n, cambios=cam, x=x1, map=m1, x2=e.get_poses(), map2=e.get_map()))
        e.close()
    return data, tol, hist, ref


def _same_result(i, x, m, x1, m1):
    dx = np.abs(x - x1)
    assert dx[:2].max() <= TOL_XY and dx[2].max() <= TOL_TH, (i, dx.max(axis=1))
    assert m.shape == m1.shape, (i, m.shape, m1.shape)
    assert np.abs(m - m1).max() <= TOL_MAP, i


def test_batch_until_equals_each_trajectory_alone(case):
    data, tol, hist, ref = case
    allmax = np.concatenate([h[:, 1] for h in hist])
    assert not np.any(np.abs(allmax - tol) <= 0.01 * tol)
    assert len({r["n"] for r in ref}) >= 3, [r["n"] for r in ref]
    b = _batch(data)
    conv = b.iterate_until(MAX_SWEEPS, tol)
    got = b.results()
    for i in range(K):
        n, cam = conv[i]
        assert n == ref[i]["n"], (i, n, ref[i]["n"])
        assert cam.shape == (n, 3) and np.abs(cam - ref[i]["cambios"]).max() <= TOL_CAMBIO, (i, cam, ref[i]["cambios"])
        _same_result(i, got[i][0], got[i][1], ref[i]["x"], ref[i]["map"])
    assert b.engine.sweep_stats()["batch_until_fallbacks"] >= 1      # (the merge of trajectory 5 needs the full search)
    # after the call every trajectory sweeps again, as its own handle would after iterate_until
    b.iterate(2)
    got = b.results()
    for i in range(K):
        _same_result(i, got[i][0], got[i][1], ref[i]["x2"], ref[i]["map2"])
    b.close()


def test_batch_until_without_tolerance_is_the_fixed_loop():
    data = _data()
    a, c = _batch(data), _batch(data)
    conv = a.iterate_until(5, 0.0)
    c.iterate(5)
    assert np.array_equal(a.engine.get_poses(), c.engine.get_poses())
    assert np.array_equal(a.engine.get_map(), c.engine.get_map())
    assert np.array_equal(a.engine.associations(), c.engine.associations())
    a.close(); c.close()
    for i, d in enumerate(data):
        e = _alone(d)
        n, cam = e.iterate_until(d["odometry"][:, 0], 5, 0.0)
        e.close()
        assert conv[i][0] == n == 5
        assert np.abs(conv[i][1] - cam).max() <= TOL_CAMBIO, i


@pytest.mark.parametrize("env", [{"ICMSLAM_GRAPH": "0"}, {"ICMSLAM_STEADY": "0"}])
def test_batch_until_variants_agree(case, env):
    data, tol, _, _ = case
    out = []
    for e in (None, env):
        b = _batch(data, e)
        conv = b.iterate_until(MAX_SWEEPS, tol)
        out.append(({i: conv[i][0] for i in conv}, b.engine.get_poses(), b.engine.get_map()))
        b.close()
    assert out[0][0] == out[1][0], env
    assert np.array_equal(out[0][1], out[1][1]) and np.array_equal(out[0][2], out[1][2]), env


def test_batch_until_rejects_invalid_calls():
    from icm_slam_b200._lib import IcmSlamError
    data = _data()[:2]
    single = _alone(data[0])
    with pytest.raises(IcmSlamError) as ei:
        single.batch_iterate_until(3, 1e-3, 256.0, 64)
    assert ei.value.status == -1
    single.close()
    b = _batch(data)
    for args in ((3, 1e-3, 0.0, 64), (3, 1e-3, -256.0, 64), (-1, 1e-3, 256.0, 64)):
        with pytest.raises(IcmSlamError) as ei:
            b.engine.batch_iterate_until(*args)
        assert ei.value.status == -1, args
    m = b.engine.get_map()
    b.engine.set_map(np.concatenate([m, [[0.0], [256.0 * 5]]], axis=1))      # a landmark in region 320 of a 2-trajectory batch
    with pytest.raises(IcmSlamError) as ei:
        b.engine.batch_iterate_until(3, 1e-3, 256.0, 64)
    assert ei.value.status == -1
    b.close()
