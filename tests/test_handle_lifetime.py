"""Lifetime of a handle's buffers (run with `-m gpu`): a handle that is loaded and extracted again, that runs every call which
allocates on first use, or that is closed after all of them, gives bit for bit what a fresh handle gives for the same calls."""
import os

import numpy as np
import pytest

from helpers import CONFIG_ROS, c2_inputs, golden

pytestmark = pytest.mark.gpu


def _synth_b():
    g = golden("synth_b.npz")
    return dict(z=g["observations"].astype(np.float64), odo=g["odometry"], u=g["velocities"], map0=g["map_init"], x0=g["x_init"],
                cfg=dict(L=4096, cota=float(g["cfg_cota"])))      # (room for every label pass 0 creates)


def _synthetic():
    """16 record tiles: enough for a host sweep in four chunks of one tile or more."""
    from icm_slam_b200.synthetic import make_synthetic
    d = make_synthetic(256, T=2048, seed=20181 + 1)
    return dict(z=d["observations"], odo=d["odometry"], u=d["velocities"], map0=d["map_init"], x0=d["x_init"],
                cfg=dict(L=4096, cota=20.0))


CASES = {"synth_b": _synth_b, "synthetic": _synthetic}


@pytest.fixture(scope="module", params=sorted(CASES))
def case(request):
    return CASES[request.param]()


def _engine(c, env=None):
    from icm_slam_b200.config import ConfigICM
    from icm_slam_b200.engine import Engine
    d = dict(CONFIG_ROS)
    d.update(c["cfg"])
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        e = Engine(ConfigICM.from_values(**d))
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    return e


def _load(e, c):
    e.load(c["z"], c["odo"], c["u"], precondition=True)
    e.extract()


def _same(a, b, what):
    assert len(a) == len(b), what
    for k, (ra, rb) in enumerate(zip(a, b)):
        assert len(ra) == len(rb), (what, k)
        for i, (xa, xb) in enumerate(zip(ra, rb)):
            assert np.array_equal(np.asarray(xa), np.asarray(xb)), (what, k, i)


def _iterate3(e, c):
    e.set_map(c["map0"])
    e.set_poses(np.ascontiguousarray(c["x0"].copy()))
    e.iterate(None, c["odo"][:, 0], 3)      # (the second and third sweeps replay a captured graph)
    return [(e.get_poses(), e.get_map(), e.associations())]


def test_extract_again_then_graph_replay(case):
    """A second extraction replaces every buffer a captured sweep holds: the sweeps after it equal a fresh handle's."""
    e = _engine(case)
    _load(e, case)
    first = _iterate3(e, case)
    e.extract()
    again = _iterate3(e, case)
    e.close()
    f = _engine(case)
    _load(f, case)
    fresh = _iterate3(f, case)
    f.close()
    _same(first, fresh, "first extraction")
    _same(again, fresh, "second extraction")


def _pass0_then_modes(e, c):
    """Pass 0, two sequential RUNNING-view sweeps from its result, then two default sweeps: what each step returns."""
    x0 = c["odo"][:, 0]
    x, mapa = e.pass0(x0)
    out = [(x.copy(), mapa.copy(), e.associations())]
    e.landmarks_actuales = mapa.shape[1]
    for _ in range(2):
        st, Lout, mapa = e.sweep(mapa, x, x0, schedule="sequential", solver="nm", view="running")
        mapa = np.array(mapa, copy=True)
        out.append((x.copy(), mapa, e.associations(), np.array([st, Lout])))
    e.set_map(mapa)
    e.set_poses(x)
    e.iterate(None, x0, 2)
    out.append((e.get_poses(), e.get_map(), e.associations()))
    return out


def test_pass0_reference_modes_then_default_sweeps(case):
    """Pass 0 and the RUNNING view share the buffers of the matched landmarks; a reloaded handle repeats every step exactly."""
    f = _engine(case)
    _load(f, case)
    fresh = _pass0_then_modes(f, case)
    f.close()
    e = _engine(case)
    for r in range(2):
        _load(e, case)
        _same(_pass0_then_modes(e, case), fresh, "round %d" % r)
    e.close()


PIPE = {"ICMSLAM_PIPE_CHUNKS": "4", "ICMSLAM_PIPE_TILES": "1"}


def _every_lazy_call(e, c):
    """Every call that allocates on first use, in one handle."""
    x0 = c["odo"][:, 0]
    x, mapa = e.pass0(x0)
    out = [(x.copy(), mapa.copy())]
    e.landmarks_actuales = mapa.shape[1]
    st, Lout, mapa = e.sweep(mapa, x, x0, schedule="sequential", solver="nm", view="running")
    mapa = np.array(mapa, copy=True)
    out.append((x.copy(), mapa, e.associations()))
    assert e.sweep_stats()["n_tiles"] >= 4      # (the host sweeps of the chain below go through in four chunks)
    e.landmarks_actuales = mapa.shape[1]
    for _ in range(3):                          # the first link returns the map the next two continue from
        st, Lout, mapa = e.sweep(mapa, x, x0)
        mapa = np.array(mapa, copy=True)
        out.append((x.copy(), mapa, e.associations()))
    raw, _, _ = c2_inputs()
    out.append((e.filtrar_obs(raw, 10.0, 15),))
    ext = e.get_extraction()
    t = 1 + int(np.argmax(np.diff(ext["off"])[1:-1]))      # the inner scan with the most observations
    o0, o1 = int(ext["off"][t]), int(ext["off"][t + 1])
    z = np.stack([ext["d"][o0:o1], ext["beam"][o0:o1] * np.pi / 180.0], axis=1)
    seen = mapa[:, np.arange(o1 - o0) % mapa.shape[1]].T.copy()
    p, f, n = e.pose_eval("min_newton", z=z, seen=seen, x_ant=x[:, t - 1], x_pos=x[:, t + 1], u_ant=c["u"][:, t - 1],
                          u_act=c["u"][:, t], odo=c["odo"][:, t - 1:t + 2])
    out.append((p, np.array([f, n])))
    k = mapa.shape[1]
    e.landmarks_actuales = k
    y = np.zeros((2, e.L))
    y[:, :k] = mapa
    obs = np.concatenate([mapa[:, :8].T + 0.05, [[1e4, 1e4]]])      # near eight landmarks, and one far from all of them
    cl = e.associate(y, mapa, obs)
    out.append((y, cl))
    return out


def _loop_batch():
    from icm_slam_b200.config import ConfigICM
    from icm_slam_b200.synthetic import make_synthetic_loop
    from icm_slam_b200.batch import ConcatBatch
    d = dict(CONFIG_ROS)
    d.update(L=2048, cota=20.0)
    b = ConcatBatch(ConfigICM.from_values(**d), 0, 1, device=0)
    for i in range(3):
        t = make_synthetic_loop(16, T=1024, seed=20181 + 400 + i, init_pose_noise=(0.03 * (i + 1), 0.006 * (i + 1)))
        b.add(i, t["observations"], t["odometry"], t["velocities"], t["map_init"], t["x_init"])
    b.finalize()
    return b


def _batch_until_twice(b):
    """iterate_until twice: the first call allocates the freeze buffers, the second reuses them."""
    out = []
    for _ in range(2):
        conv = b.iterate_until(6, 1e-3)
        out.append(tuple(np.array([conv[i][0]]) for i in sorted(conv)) + tuple(conv[i][1] for i in sorted(conv)))
        out.append((b.engine.get_poses(), b.engine.get_map()))
    return out


def test_every_lazy_allocation_then_close():
    c = _synthetic()
    e = _engine(c, PIPE)
    _load(e, c)
    got = _every_lazy_call(e, c)
    e.close()
    b = _loop_batch()
    got_b = _batch_until_twice(b)
    b.close()
    f = _engine(c, PIPE)
    _load(f, c)
    _same(got, _every_lazy_call(f, c), "single handle")
    f.close()
    fb = _loop_batch()
    _same(got_b, _batch_until_twice(fb), "batch handle")
    fb.close()
