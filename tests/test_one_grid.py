"""The landmark grid outside the fused sweep (the generic sweep's association, Mapa.filtrar's neighbour search, calc_cambio)
on large maps, against the CPU oracle or a numpy brute force.  And calc_cambio between two fused sweeps, and the callers of the
filter chain other than the fused sweep, leave the fused chain as it was."""
import numpy as np
import pytest

from helpers import CONFIG_ROS

pytestmark = pytest.mark.gpu

TOL_XY = 1e-6
TOL_TH = 1e-8
LARGE_K = 2048              # survivors of the large maps below (the golden fixtures' raw maps have at most 200 landmarks)


def _cfg(**kw):
    from icm_slam_b200.config import ConfigICM
    d = dict(CONFIG_ROS)
    d.update(kw)
    return ConfigICM.from_values(**d)


def _engine(cfg, z, odo, u):
    from icm_slam_b200.engine import Engine
    e = Engine(cfg)
    e.load(z, odo, u, precondition=True)
    e.extract()
    return e


def _cdist_min(new, old, chunk=1024):
    """min over the old landmarks of cdist(new, old), one value per new landmark: sqrt(dx*dx + dy*dy), each op rounded."""
    out = np.empty(new.shape[1])
    for s in range(0, new.shape[1], chunk):
        dx = new[0, s:s + chunk, None] - old[0, None, :]
        dy = new[1, s:s + chunk, None] - old[1, None, :]
        out[s:s + chunk] = np.sqrt(dx * dx + dy * dy).min(axis=1)
    return out


@pytest.mark.parametrize("view", ["prev", "running"])
def test_generic_sweeps_with_a_large_map_vs_oracle(view):
    """Two generic sweeps on a 2304-landmark field: the association and the filter's neighbour search both use the grid."""
    from icm_slam_b200.synthetic import make_synthetic
    from oracle import oracle as orc
    d = make_synthetic(2304, seed=20181 + 31)
    cfgd = dict(CONFIG_ROS, L=2 * 2304 + 64, cota=20.0)
    z, odo, u = d["observations"], d["odometry"], d["velocities"]
    ocfg = orc.make_cfg(**cfgd)
    ext = orc.extract_all(orc.precondition(z, ocfg.radio, ocfg.rango_laser_max), ocfg)
    e = _engine(_cfg(**cfgd), z, odo, u)
    mo = orc.Mapa(ocfg)
    map_o = d["map_init"].copy()
    map_g = d["map_init"].copy()
    mo.landmarks_actuales = map_o.shape[1]
    e.landmarks_actuales = map_g.shape[1]
    xo = np.ascontiguousarray(d["x_init"].copy())
    xg = xo.copy()
    for k in range(2):
        r = orc.sweep(ocfg, mo, ext, odo, u, odo[:, 0], map_o, xo, "redblack", "newton", view)
        st, Lout, mout = e.sweep(map_g, xg, odo[:, 0], schedule="redblack", solver="newton", view=view, fused=False,
                                 newton_tol=1e-12, newton_maxit=50)
        assert e.sweep_stats()["kept"] > LARGE_K
        assert np.array_equal(e.associations(), r["c"])
        assert Lout == r["map"].shape[1]
        dd = np.abs(xg - xo)
        assert dd[:2].max() <= TOL_XY and dd[2].max() <= TOL_TH, (k, dd.max(axis=1))
        assert np.max(np.abs(mout - r["map"])) <= TOL_XY
        map_o = r["map"]
        map_g = np.ascontiguousarray(mout.copy())
    e.close()


def test_filter_map_with_merges_vs_oracle():
    """Mapa.filtrar with merges, as the reference's K x K search does it: 3070 landmarks with planted close pairs, chains and
    exact ties (the grid search), and a map whose extent is below dist_thr but whose diameter is not, with coincident
    landmarks (the brute force of a degenerate map: a zero distance is replaced by the diameter, so a coincident pair with no
    other landmark within dist_thr stays two landmarks)."""
    from oracle import oracle as orc
    rng = np.random.default_rng(20181 + 32)
    G = 50
    gx, gy = np.meshgrid(np.arange(G), np.arange(G), indexing="xy")
    base = np.stack([3.0 * gx.ravel() + rng.uniform(-0.5, 0.5, G * G), 3.0 * gy.ravel() + rng.uniform(-0.5, 0.5, G * G)])
    pick = rng.choice(G * G, 500, replace=False)
    ang = rng.uniform(0.0, 2.0 * np.pi, 500)
    rad = rng.uniform(0.05, 1.2, 500)              # about a fifth of them beyond dist_thr = 1
    close = base[:, pick] + rad * np.stack([np.cos(ang), np.sin(ang)])
    chain = close[:, :50] + np.array([[0.6], [0.0]])                   # chains of three
    tie = base[:, pick[50:60]] + np.array([[0.0], [0.5]])
    tie2 = base[:, pick[50:60]] + np.array([[0.0], [-0.5]])            # equidistant pairs around the same landmark
    large = np.ascontiguousarray(np.concatenate([base, close, chain, tie, tie2], axis=1)[:, rng.permutation(3070)])
    large_counts = rng.integers(1, 60, large.shape[1]).astype(np.float64)
    assert int((large_counts >= 10.0).sum()) > LARGE_K
    far = 5.75 + rng.uniform(0.0, 0.15, (2, 20))
    small = np.concatenate([np.full((2, 2), 5.0), far, far[:, :3], np.full((2, 1), 5.9)], axis=1)
    small_counts = rng.integers(1, 60, small.shape[1]).astype(np.float64)
    small_counts[:2] = (20.0, 30.0)
    assert np.ptp(small, axis=1).max() < 1.0 <= np.hypot(0.9, 0.9)
    cfgd = dict(CONFIG_ROS, L=4096, cota=10.0)
    e = _engine_plain(cfgd)
    for mapa, counts in ((large, large_counts), (small, small_counts)):
        out, cnt, Lout = e.filter_map(mapa, counts)
        mo = orc.Mapa(orc.make_cfg(**cfgd))
        mo.landmarks_actuales = mapa.shape[1]
        mo.cant_obs_i[:] = 0.0
        mo.cant_obs_i[: mapa.shape[1]] = counts
        full = np.zeros((2, 4096))              # (the oracle's map has L columns)
        full[:, : mapa.shape[1]] = mapa
        ref = mo.filtrar(full)
        Lref = mo.landmarks_actuales
        assert Lref < int((counts >= 10.0).sum())         # merges happened
        assert Lout == Lref
        assert np.array_equal(cnt[:Lout], mo.cant_obs_i[:Lref])
        assert np.max(np.abs(out[:, :Lout] - ref[:, :Lref])) <= 1e-12
    assert Lout > 2 and np.array_equal(out[:, :2], np.full((2, 2), 5.0))      # (the coincident pair)
    e.close()


def _engine_plain(cfgd):
    from icm_slam_b200.engine import Engine
    return Engine(_cfg(**cfgd))


@pytest.mark.parametrize("spread", ["dense", "wide"])
def test_calc_cambio_vs_brute_force(spread):
    """calc_cambio of about 10^4 landmarks: some new ones far from every old one (the full scan), and (wide) an old map whose
    bounding box does not fit the cell budget at the smallest cell edge, so that the grid's cells are grown."""
    rng = np.random.default_rng(20181 + 33 + (spread == "wide"))
    n_old = 10000
    old = rng.uniform(0.0, 300.0, (2, n_old))
    if spread == "wide":
        old[:, :8] = rng.uniform(-1.0e5, 1.0e5, (2, 8))
    src = rng.integers(0, n_old, 9000)
    step = rng.uniform(0.0, 1.2, 9000) * np.array([[1.0], [0.0]])      # up to beyond dist_thr = 1
    new = old[:, src] + step
    new = np.concatenate([new, rng.uniform(-400.0, 700.0, (2, 1000)), old[:, :10]], axis=1)   # far ones, exact copies
    new = np.ascontiguousarray(new[:, rng.permutation(new.shape[1])])
    e = _engine_plain(dict(CONFIG_ROS, L=16384))
    got = e.calc_cambio(new, old)
    d = _cdist_min(new, old)
    assert (d > 1.05).sum() > 100 and (d == 0.0).sum() >= 10
    assert got[0] == d.min() and got[1] == d.max()
    assert abs(got[2] - d.mean()) <= 1e-12 * d.mean()      # (the device sums in another order)
    e.close()


def test_calc_cambio_between_fused_sweeps_leaves_the_chain():
    """calc_cambio builds its own grid: a fused chain with calls between its sweeps launches the same kernels and ends with
    the same poses and map as the chain without them."""
    from icm_slam_b200.synthetic import make_synthetic
    d = make_synthetic(625, T=4000, seed=20181 + 34)
    cfgd = dict(CONFIG_ROS, L=2 * 625 + 64, cota=20.0)
    z, odo, u = d["observations"], d["odometry"], d["velocities"]
    res = []
    for between in (False, True):
        e = _engine(_cfg(**cfgd), z, odo, u)
        e.set_map(d["map_init"]); e.set_poses(d["x_init"])
        n0 = e.launch_count()
        prev = d["map_init"]
        for k in range(4):
            e.iterate(None, odo[:, 0], 1)
            m = e.get_map()
            if between:
                e.calc_cambio(m, prev)
            prev = m
        res.append((e.launch_count() - n0, e.get_map(), e.get_poses(), e.sweep_stats()["epoch"]))
        e.close()
    (n_a, map_a, x_a, ep_a), (n_b, map_b, x_b, ep_b) = res
    assert n_a == n_b and ep_a == ep_b
    assert np.array_equal(map_a, map_b) and np.array_equal(x_a, x_b)


def test_filter_callers_leave_the_fused_sweep_counters():
    """Pass 0, Mapa.filtrar and a generic sweep run the fused tail's filter chain without closing a fused sweep: the sweep and
    peer-memory sequence numbers and the label-numbering epoch stay as the last fused sweep left them."""
    import ctypes as C
    from helpers import c1_inputs, golden
    g = golden("c1_ref.npz")
    z, odo, u = c1_inputs()
    e = _engine(_cfg(), z, odo, u)
    e.set_map(g["p0_map"]); e.set_poses(g["p0_x"])
    e.iterate(None, odo[:, 0], 2)

    def counters():
        trace, cn = (C.c_uint64 * 256)(), (C.c_uint32 * 3)()
        assert e.lib.icmslam_get_trace(e._h, trace, cn) == 0
        return list(cn), e.sweep_stats()["epoch"]

    before = counters()
    assert before[0][0] >= 2
    e.pass0(odo[:, 0])
    e.filter_map(g["p0_map"], np.full(g["p0_map"].shape[1], 400.0))
    e.landmarks_actuales = g["p0_map"].shape[1]
    x = np.ascontiguousarray(g["p0_x"].copy())
    e.sweep(g["p0_map"].copy(), x, odo[:, 0], fused=False)
    assert counters() == before
    e.close()
