"""Every sweep mode on a batch handle (ConcatBatch / icmslam_set_batch) against each trajectory swept alone, and the
reference's own mode (sequential, NM, running) inside a batch against the fixtures minted from the unmodified reference
(run with `-m gpu`)."""
import ctypes as C

import numpy as np
import pytest

from helpers import CONFIG_ROS, c1_inputs, golden

pytestmark = pytest.mark.gpu

SPACING = 256.0      # ConcatBatch's default region pitch
MODES = [("redblack", "newton", "prev"), ("redblack", "newton", "full"), ("redblack", "newton", "running"),
         ("sequential", "newton", "running"), ("redblack", "nm", "running"), ("sequential", "newton", "prev"),
         ("sequential", "nm", "running")]
K, N_SWEEPS = 5, 3
CFGD = dict(L=2048, cota=20.0)      # (room for the labels trajectory 1 creates every sweep)


def _cfg(**kw):
    from icm_slam_b200.config import ConfigICM
    d = dict(CONFIG_ROS)
    d.update(kw)
    return ConfigICM.from_values(**d)


def _offset(k):
    return np.array([(k % 64) * SPACING, (k // 64) * SPACING])


def _region(mapa):
    cell = np.rint(mapa / SPACING).astype(np.int64)
    return cell[1] * 64 + cell[0]


def _data(Tk):
    """K trajectories; trajectory 1 lacks a landmark of its map (its far observations create labels every sweep), trajectory 3
    has a run of empty scans inside it."""
    from icm_slam_b200.synthetic import make_synthetic_loop
    data = [make_synthetic_loop(16, T=Tk, seed=20181 + 400 + i, init_pose_noise=(0.03 * (i + 1), 0.006 * (i + 1))) for i in range(K)]
    data[1]["map_init"] = np.delete(data[1]["map_init"], 5, axis=1)
    data[3]["observations"][:, 200:206] = 10.0
    return data


def _alone(d, k, mode):
    """Trajectory d swept alone, translated by the offset ConcatBatch gives slot k (identical fp64 inputs)."""
    from icm_slam_b200.engine import Engine
    off = _offset(k)
    odo, x = d["odometry"].copy(), d["x_init"].copy()
    odo[0:2] += off[:, None]
    x[0:2] += off[:, None]
    e = Engine(_cfg(**CFGD))
    e.load(d["observations"], odo, d["velocities"], precondition=True)
    e.extract()
    e.set_map(d["map_init"] + off[:, None])
    e.set_poses(x)
    iters, far = [], []
    for _ in range(N_SWEEPS):
        e.iterate(None, odo[:, 0], 1, fused=False, stats=True, **mode)
        st = e.sweep_stats()
        iters.append(st["newton_iters"])
        far.append(st["n_far_scans"])
    mapa = e.get_map()
    out = dict(x=e.get_poses(), map=mapa, counts=e.counts(mapa.shape[1]), c=e.associations(), iters=iters, far=far)
    e.close()
    return out


def _same_labels_up_to_renumbering(cb, cs):
    """cb and cs label the same observations alike: a one-to-one map between their labels that keeps their order."""
    assert cb.shape == cs.shape
    pairs = np.unique(np.stack([cb, cs]), axis=1)      # (sorted by the batch label)
    assert len(np.unique(pairs[0])) == pairs.shape[1] and len(np.unique(pairs[1])) == pairs.shape[1]
    assert np.all(np.diff(pairs[1]) > 0)


@pytest.mark.parametrize("Tk", [512, 511])
@pytest.mark.parametrize("schedule,solver,view", MODES)
def test_batch_mode_equals_each_trajectory_alone(schedule, solver, view, Tk):
    from icm_slam_b200.batch import ConcatBatch
    mode = dict(schedule=schedule, solver=solver, view=view)
    data = _data(Tk)
    b = ConcatBatch(_cfg(**CFGD), 0, 1, device=0)
    for i, d in enumerate(data):
        b.add(i, d["observations"], d["odometry"], d["velocities"], d["map_init"], d["x_init"])
    b.finalize()
    iters = []
    for _ in range(N_SWEEPS):
        b.iterate(1, fused=False, stats=True, **mode)
        iters.append(b.engine.sweep_stats()["newton_iters"])
    x, mapa = b.engine.get_poses(), b.engine.get_map()
    counts, c = b.engine.counts(mapa.shape[1]), b.engine.associations()
    off = b.engine.get_extraction()["off"]
    kk = _region(mapa)
    b.close()
    alone = [_alone(d, k, mode) for k, d in enumerate(data)]
    assert iters == [sum(a["iters"][s] for a in alone) for s in range(N_SWEEPS)]
    assert all(a["iters"][0] > 0 for a in alone)
    assert min(alone[1]["far"]) > 0      # (trajectory 1 creates labels in every sweep)
    for k, a in enumerate(alone):
        xs, ms = x[:, k * Tk:(k + 1) * Tk], mapa[:, kk == k]
        _same_labels_up_to_renumbering(c[off[k * Tk]:off[(k + 1) * Tk]], a["c"])
        assert np.array_equal(counts[kk == k], a["counts"]), k
        assert ms.shape == a["map"].shape, (k, ms.shape, a["map"].shape)
        if view == "running":
            assert np.array_equal(xs, a["x"]), (k, np.abs(xs - a["x"]).max(axis=1))
            assert np.array_equal(ms, a["map"]), k
        else:
            # (the PREV and FULL means are float atomics: their summation order follows the warp schedule, batch or not)
            d = np.abs(xs - a["x"])
            assert d[:2].max() <= 1e-9 and d[2].max() <= 1e-11, (k, d.max(axis=1))
            assert np.abs(ms - a["map"]).max() <= 1e-9, k


@pytest.mark.parametrize("name", ["c1_ref.npz", "synth_a.npz"])
def test_reference_mode_in_slot_0_of_a_batch(name):
    """The reference's sweeps in (sequential, NM, running) with its log in slot 0 of a batch of four: slot 0 meets what the
    reference-mode test asserts for the log alone (labels, poses to 1e-6 m / 1e-8 rad, map to 1e-6 m)."""
    from icm_slam_b200.batch import ConcatBatch
    from icm_slam_b200.synthetic import make_synthetic_loop
    g = golden(name)
    if name == "c1_ref.npz":
        (z, odo, u), cfgd, map0 = c1_inputs(), {}, g["p0_map"]
    else:
        z, odo, u = g["observations"].astype(np.float64), g["odometry"], g["velocities"]
        cfgd, map0 = dict(L=int(g["cfg_L"]), cota=float(g["cfg_cota"])), g["map_init"]
    T = z.shape[1]
    b = ConcatBatch(_cfg(**cfgd), 0, 1, device=0)
    b.add(0, z, odo, u, map0, g["s1_x_in"])
    for i in range(1, 4):
        d = make_synthetic_loop(16, T=T, seed=20181 + 500 + i, beams=z.shape[0])
        b.add(i, d["observations"], d["odometry"], d["velocities"], d["map_init"], d["x_init"])
    b.finalize()
    e = b.engine
    n0 = int(e.get_extraction()["off"][T])
    x, mapa = e.get_poses(), e.get_map()
    gmap = map0
    for k in range(1, int(g["nsweeps"]) + 1):
        p = "s%d_" % k
        x[:, :T] = g[p + "x_in"]
        mapa = np.ascontiguousarray(np.concatenate([gmap, mapa[:, _region(mapa) != 0]], axis=1))
        L0, L_in = gmap.shape[1], mapa.shape[1]
        e.landmarks_actuales = L_in
        st, Lout, mout = e.sweep(mapa, x, b.x0s[:, 0], schedule="sequential", solver="nm", view="running")
        assert st == 0
        cg = g[p + "labels"].astype(np.int64)
        assert np.array_equal(e.associations()[:n0], np.where(cg >= L0, cg + (L_in - L0), cg))    # (new labels follow the batch's map)
        d = np.abs(x[:, :T] - g[p + "x_out"])
        assert d[:2].max() <= 1e-6 and d[2].max() <= 1e-8, d.max(axis=1)
        m0 = mout[:, _region(mout) == 0]
        assert m0.shape == g[p + "map_out"].shape
        assert np.max(np.abs(m0 - g[p + "map_out"])) <= 1e-6
        gmap, mapa = g[p + "map_out"], np.array(mout)
    b.close()


def test_batch_iterate_until_is_fused_mode_only():
    """The per-trajectory stop (icmslam_batch_iterate_until) freezes trajectories in the fused kernels only: every other mode,
    and the default mode with the fused path switched off, is refused with ICMSLAM_ERR_UNSUPPORTED."""
    from icm_slam_b200 import _lib
    from icm_slam_b200.batch import ConcatBatch
    data = _data(256)[:2]
    b = ConcatBatch(_cfg(**CFGD), 0, 1, device=0)
    for i, d in enumerate(data):
        b.add(i, d["observations"], d["odometry"], d["velocities"], d["map_init"], d["x_init"])
    b.finalize()
    e = b.engine
    n_done, n_run = np.zeros(2, np.int32), C.c_int32(0)
    for schedule, solver, view in MODES:
        for fused in ((0,) if (schedule, solver, view) == MODES[0] else (0, 1)):
            opts = _lib.SweepOpts(_lib.SCHED[schedule], _lib.SOLVER[solver], _lib.VIEW[view], 0, 0.0, fused, 0)
            st = e.lib.icmslam_batch_iterate_until(e._h, 3, 1e-3, SPACING, 64, C.byref(opts), None,
                                                   n_done.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(n_run))
            assert st == -7, (schedule, solver, view, fused)
    x = e.get_poses()
    b.iterate(1)       # (the handle is untouched: the default mode still sweeps)
    assert not np.array_equal(x, e.get_poses())
    b.close()
