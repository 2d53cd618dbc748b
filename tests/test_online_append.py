"""Online ingestion on the device (icmslam_append + the resumable pass 0 walk, run with `-m gpu`): a log fed as one column plus
appends of mixed sizes holds what load + extract of the whole log hold, the walk after every advance equals pass 0 of the log cut
there, and sweeps on the fed handle equal sweeps on a handle loaded in one piece -- all bit for bit.  OnlineICM feeds the engine
after every pump call, so `positions` follows the messages."""
import ctypes as C

import numpy as np
import pytest

from helpers import CONFIG_ROS, c1_inputs, c2_inputs

pytestmark = pytest.mark.gpu

ERR_INVALID, ERR_UNSUPPORTED = -1, -7


def _cfg(**kw):
    from icm_slam_b200.config import ConfigICM
    d = dict(CONFIG_ROS)
    d.update(kw)
    return ConfigICM.from_values(**d)


def _empty_around(z, b):
    """Scans b - 1 and b have no observation (every range at the laser's maximum)."""
    z = z.copy()
    z[:, b - 1:b + 1] = CONFIG_ROS["rango_laser_max"]
    return z


def _log(name):
    if name == "c1":
        z, odo, u = c1_inputs()
    elif name == "c2":
        z, odo, u = c2_inputs()
    else:
        from icm_slam_b200.synthetic import make_synthetic_loop
        d = make_synthetic_loop(16, T=700, seed=20181 + 77)
        z, odo, u = d["observations"].astype(np.float64), d["odometry"], d["velocities"]
    return _empty_around(z, 41), odo, u          # (41 is a chunk boundary of every split below)


def _split(kind, T, seed=5):
    """Chunk sizes after the one column `load` takes."""
    if kind == "ones":
        return [1] * 40 + [T - 41]
    if kind == "one_chunk":
        return [40, T - 41]
    rng = np.random.default_rng(seed)
    sizes, left = [40], T - 41
    while left > 0:
        k = int(min(left, rng.integers(1, 400)))
        sizes.append(k)
        left -= k
    return sizes


def _engine(cfg):
    from icm_slam_b200.engine import Engine
    return Engine(cfg)


def _whole(cfg, z, odo, u):
    e = _engine(cfg)
    e.load(z, odo, u, precondition=True)
    e.extract()
    return e


def _fed(cfg, z, odo, u, sizes, each=None):
    """load of column 0, then one append per chunk; `each(engine, t)` after every append."""
    e = _engine(cfg)
    e.load(z[:, :1], odo[:, :1], u[:, :1], precondition=True)
    e.extract()
    t = 1
    if each:
        each(e, t)
    for k in sizes:
        e.append(z[:, t:t + k], odo[:, t:t + k], u[:, t:t + k])
        t += k
        if each:
            each(e, t)
    assert t == z.shape[1]
    return e


@pytest.mark.parametrize("name", ["c1", "c2", "loop"])
@pytest.mark.parametrize("kind", ["ones", "random", "one_chunk"])
def test_appended_extraction_equals_whole_log(name, kind):
    z, odo, u = _log(name)
    cfg = _cfg()
    ref = _whole(cfg, z, odo, u)
    e = _fed(cfg, z, odo, u, _split(kind, z.shape[1]))
    assert (e.n, e.n_empty, e.max_per_scan) == (ref.n, ref.n_empty, ref.max_per_scan)
    assert e.n_empty >= 2
    a, b = e.get_extraction(), ref.get_extraction()
    for k in ("off", "beam", "d", "bx", "by"):
        assert np.array_equal(a[k], b[k]), k
    e.close()
    ref.close()


def _pass0_prefix(ref, cfg, z, odo, u, t, x0):
    """pass 0 of the log cut at t: poses, filtered map (None when no landmark of a short prefix reaches cota: Mapa.filtrar
    raises after the walk), labels, raw map."""
    ref.load(z[:, :t], odo[:, :t], u[:, :t], precondition=True)
    ref.extract()
    try:
        x, mapa = ref.pass0(x0)
    except ValueError:
        x, mapa = ref.get_poses(), None
    return x, mapa, ref.associations(), ref.raw_map()


@pytest.mark.parametrize("name,kind", [("c1", "ones"), ("c1", "random"), ("c2", "random"), ("loop", "random")])
def test_walk_equals_pass0_of_every_prefix(name, kind):
    z, odo, u = _log(name)
    cfg = _cfg()
    x0 = odo[:, 0].copy()
    ref = _engine(cfg)
    other = []      # what the calls between two advances return: the walk must not change them, nor they the walk

    def each(e, t):
        if t == 1:
            assert e.pass0_begin(x0) == 0
        assert e.pass0_advance() == t
        xr, mr, cr, (rawr, cntr, rlr) = _pass0_prefix(ref, cfg, z, odo, u, t, x0)
        assert np.array_equal(e.get_poses()[:, :t], xr)
        assert np.array_equal(e.associations()[:cr.shape[0]], cr)
        raw, cnt, rl = e.raw_map()
        assert rl == rlr and np.array_equal(raw, rawr) and np.array_equal(cnt, cntr)
        if mr is not None and mr.shape[1] >= 2:        # calls that write the handle's raw map, counts and landmarks_actuales
            fm = e.filter_map(rawr, cntr)
            cc = e.calc_cambio(mr, mr[:, ::-1].copy())
            mapa = np.zeros((2, cfg.L))
            mapa[:, :mr.shape[1]] = mr
            e.landmarks_actuales = mr.shape[1]
            c = e.associate(mapa, mr, np.ascontiguousarray(mr.T[:2] + 0.05))
            other.append((fm[0].copy(), fm[2], cc, c.copy()))
            fm2 = ref.filter_map(rawr, cntr)
            cc2 = ref.calc_cambio(mr, mr[:, ::-1].copy())
            mapa2 = np.zeros((2, cfg.L))
            mapa2[:, :mr.shape[1]] = mr
            ref.landmarks_actuales = mr.shape[1]
            c2 = ref.associate(mapa2, mr, np.ascontiguousarray(mr.T[:2] + 0.05))
            assert np.array_equal(fm[0], fm2[0]) and fm[2] == fm2[2] and cc == cc2 and np.array_equal(c, c2)

    e = _fed(cfg, z, odo, u, _split(kind, z.shape[1]), each)
    x, mapa = e.pass0_finish()
    whole = _whole(cfg, z, odo, u)
    xw, mw = whole.pass0(x0)
    assert np.array_equal(x, xw) and np.array_equal(mapa, mw)
    assert e.landmarks_actuales == whole.landmarks_actuales == mw.shape[1]
    assert np.array_equal(e.counts(mw.shape[1]), whole.counts(mw.shape[1]))      # (cant_obs_i of the filtered map)
    assert np.array_equal(e.associations(), whole.associations())
    raw, cnt, rl = e.raw_map()
    raww, cntw, rlw = whole.raw_map()
    assert rl == rlw and np.array_equal(raw, raww) and np.array_equal(cnt, cntw)
    assert len(other) > 0
    for h in (e, ref, whole):
        h.close()


MODES = [dict(), dict(schedule="sequential", solver="nm", view="running")]


@pytest.mark.parametrize("name", ["c1", "loop"])
def test_sweeps_on_the_fed_handle_equal_the_whole_log(name):
    z, odo, u = _log(name)
    T = 500
    z, odo, u = z[:, :T], odo[:, :T], u[:, :T]
    cfg = _cfg()
    x0 = odo[:, 0].copy()
    whole = _whole(cfg, z, odo, u)
    xw, mw = whole.pass0(x0)
    e = _fed(cfg, z, odo, u, _split("random", T, seed=11))
    assert e.pass0_begin(x0) == 0 and e.pass0_advance() == T
    x, mapa = e.pass0_finish()
    assert np.array_equal(x, xw) and np.array_equal(mapa, mw)
    for mode in MODES:
        for h in (whole, e):
            h.set_map(mw)
            h.set_poses(xw.copy())
            h.iterate(None, x0, 5, **mode)
        assert np.array_equal(e.get_poses(), whole.get_poses()), mode
        assert np.array_equal(e.get_map(), whole.get_map()), mode
        assert np.array_equal(e.associations(), whole.associations()), mode
    res = []
    for h in (whole, e):
        h.set_map(mw)
        h.set_poses(xw.copy())
        res.append(h.iterate_until(x0, 12, 1e-9))
    assert res[0][0] == res[1][0] and np.array_equal(res[0][1], res[1][1])
    assert np.array_equal(e.get_poses(), whole.get_poses()) and np.array_equal(e.get_map(), whole.get_map())
    assert np.array_equal(e.associations(), whole.associations())
    e.close()
    whole.close()


def test_the_advance_that_crosses_the_label_cap_fails_as_pass0_does():
    z, odo, u = _log("c1")
    cfg = _cfg()
    x0 = odo[:, 0].copy()
    full = _whole(cfg, z, odo, u)
    full.pass0(x0)
    L = full.raw_map()[2] // 2
    full.close()
    cfg_s = _cfg(L=L)
    ref = _engine(cfg_s)
    sizes = _split("random", z.shape[1], seed=3)
    seen = []

    def each(e, t):
        if t == 1:
            assert e.pass0_begin(x0) == 0
        if "cap" in seen:
            with pytest.raises(Exception):        # (the walk ended: begin it again)
                e.pass0_advance()
            seen.append("ended")
            return
        ref.load(z[:, :t], odo[:, :t], u[:, :t], precondition=True)
        ref.extract()
        try:
            ref.pass0(x0)
            ok = True
        except ValueError:      # (the walk went through; no landmark of the short prefix reaches cota)
            ok = True
        except IndexError:
            ok = False
        if ok:
            assert e.pass0_advance() == t
            seen.append("ok")
        else:
            with pytest.raises(IndexError):
                e.pass0_advance()
            seen.append("cap")

    e = _fed(cfg_s, z, odo, u, sizes, each)
    assert "cap" in seen and seen[0] == "ok"
    assert e.pass0_begin(x0) == 0                 # begun again: the whole log crosses the cap in one advance
    with pytest.raises(IndexError):
        e.pass0_advance()
    e.close()
    ref.close()


def test_empty_first_scan_and_refusals():
    z, odo, u = _log("c1")
    T = 300
    z, odo, u = np.ascontiguousarray(z[:, :T]), np.ascontiguousarray(odo[:, :T]), np.ascontiguousarray(u[:, :T])
    cfg = _cfg()
    x0 = odo[:, 0].copy()
    e = _engine(cfg)
    lib, h = e.lib, e._h
    tn = C.c_int32(0)
    assert lib.icmslam_pass0_advance(h, C.byref(tn)) == ERR_INVALID          # before begin (and before load)
    p = lambda a: C.c_void_p(a.ctypes.data)
    assert lib.icmslam_append(h, p(z), 1, T, p(odo), T, p(u), T, 0) == ERR_INVALID       # before load
    e.load(_empty_around(z, 1)[:, 1:], odo[:, 1:], u[:, 1:], precondition=True)        # column 0 empty
    e.extract()
    assert e.pass0_begin(x0) == 1
    assert lib.icmslam_pass0_advance(h, C.byref(tn)) == ERR_INVALID
    e.load(z[:, :100], odo[:, :100], u[:, :100], precondition=True)
    e.extract()
    assert lib.icmslam_pass0_advance(h, C.byref(tn)) == ERR_INVALID          # a new log: begin again
    n0 = e.n
    assert lib.icmslam_append(h, p(z), 0, T, p(odo), T, p(u), T, 0) == ERR_INVALID
    assert lib.icmslam_append(h, p(z), -3, T, p(odo), T, p(u), T, 0) == ERR_INVALID
    e._extraction_size()
    assert e.n == n0
    # a batch handle and a segment handle refuse, and sweep as before
    twin = _whole(cfg, z[:, :100], odo[:, :100], u[:, :100])
    xs, ms = twin.pass0(x0)
    x0s = np.ascontiguousarray(np.stack([odo[:, 0], odo[:, 50]], axis=1))
    for h_ in (e, twin):
        h_.set_batch(50, x0s)
    assert lib.icmslam_append(h, p(z), 5, T, p(odo), T, p(u), T, 0) == ERR_UNSUPPORTED
    for h_ in (e, twin):
        h_.set_map(ms)
        h_.set_poses(xs.copy())
        h_.iterate(None, x0, 3)
    assert np.array_equal(e.get_poses(), twin.get_poses()) and np.array_equal(e.get_map(), twin.get_map())
    for h_ in (e, twin):
        h_.set_batch(0, None)
    assert lib.icmslam_set_segment(h, 0, 60, 1, 0) == 0
    assert lib.icmslam_append(h, p(z), 5, T, p(odo), T, p(u), T, 0) == ERR_UNSUPPORTED
    e._extraction_size()
    assert e.n == n0
    e.close()
    twin.close()


def test_online_icm_positions_follow_the_messages():
    from icm_slam_b200 import ros_ingest as ri
    from icm_slam_b200.icm import ICM_SLAM, Mapa
    z, odo, u = c1_inputs()
    T = 400
    z, odo, u = z[:, :T], odo[:, :T], u[:, :T]
    cfg = _cfg(**dict(N=3, topic_laser="/scan", topic_laser_msg="sensor_msgs/LaserScan", topic_odometry="/odom",
                      topic_odometry_msg="nav_msgs/Odometry"))
    raw = np.where(z >= cfg.rango_laser_max, np.nan, z - cfg.radio)
    online = ri.OnlineICM(cfg)
    client = ri.FakeRos()
    lt, ot = client.topic(cfg.topic_laser), client.topic(cfg.topic_odometry)
    bursts = [1, 7, 50]
    state = dict(t=0, k=0)
    snaps = []

    def pump(node):
        if node.positions is not None:
            snaps.append(node.positions.copy())
        t0 = state["t"]
        t1 = min(T, t0 + bursts[state["k"] % 3])
        for t in range(t0, t1):
            if t != 123:                                  # one laser message lost
                lt.publish(ri.laser_scan_msg(raw[:, t].tolist(), t))
            ot.publish(ri.odometry_msg(odo[:, t], u[:, t], t))
        state["t"], state["k"] = t1, state["k"] + 1
        if t1 == T:
            client.service("/icm_slam/iterative_flag").call({"data": True})
            return False
        return True

    mapa0, x0s = online.inicializar_online(client, pump)
    assert online.iterations_flag and online.lidar.warnings > 0
    Ta = online.mediciones.shape[1]
    assert x0s.shape == (3, Ta) and len(snaps) >= 10
    m_on, x_on = online.iterar(x0s.copy())
    off = ICM_SLAM(cfg, x0=np.array([online.odometria[:, 0]]).T)
    off.load_data(Mapa(cfg), online.mediciones.copy(), online.u.copy(), online.odometria.copy())
    mapa1, x1 = off.inicializar()
    assert np.array_equal(mapa0, mapa1) and np.array_equal(x0s, x1)
    for s in snaps:                                       # pass 0 is causal: every live estimate is a prefix of the offline one
        assert 0 < s.shape[1] <= Ta and np.array_equal(s, x1[:, :s.shape[1]])
    m_off, x_off = off.iterar(x1.copy())
    assert np.array_equal(m_on, m_off) and np.array_equal(x_on, x_off)
