"""Batch handles (ConcatBatch / icmslam_set_batch) in the default fused mode at odd and unaligned trajectory lengths: every
trajectory of the batch against its own handle and against the CPU oracle, the chain's variants (no graph, no steady tail, no
run records, host buffers in chunks), the per-trajectory stop, a batch of one, and set_batch's refusals (run with `-m gpu`).

The lengths put trajectory boundaries at many offsets inside the 128-scan run-record tiles and the 126-pose solve tiles; at an odd
length every odd-numbered trajectory starts on an odd column, so the red-black colours must follow trajectory-local time."""
import ctypes as C
import os

import numpy as np
import pytest

from helpers import CONFIG_ROS
from test_batch_modes import _same_labels_up_to_renumbering

pytestmark = pytest.mark.gpu

SPACING = 256.0      # ConcatBatch's default region pitch
K, N_SWEEPS = 5, 4
LENGTHS = [3, 127, 128, 129, 511, 513, 1021]
TOL_XY, TOL_TH, TOL_MAP = 1e-9, 1e-11, 1e-9      # the fp64 translation of each trajectory into its region
MAXIT = 20       # the fused solve's default Newton iteration cap
ST_OWN = 126     # poses a solve tile owns (solve.cuh)


def _cfgd(Tk):
    # (a landmark of a 3-scan trajectory is seen a handful of times: cota 20 would filter out every one)
    return dict(CONFIG_ROS, L=2048, cota=20.0 if Tk > 64 else 2.0)


def _cfg(Tk):
    from icm_slam_b200.config import ConfigICM
    return ConfigICM.from_values(**_cfgd(Tk))


def _offset(k):
    return np.array([(k % 64) * SPACING, (k // 64) * SPACING])


def _region(mapa):
    cell = np.rint(mapa / SPACING).astype(np.int64)
    return cell[1] * 64 + cell[0]


def _most_seen_from_start(d):
    """The landmark the first scan of trajectory d sees most often (by its true pose and true landmarks)."""
    from oracle import oracle as orc
    ocfg = orc.make_cfg(**CONFIG_ROS)
    ext = orc.extract_all(orc.precondition(d["observations"][:, :1], ocfg.radio, ocfg.rango_laser_max), ocfg)
    x, y, th = d["x_true"][:, 0]
    st, ct = np.sin(th - np.pi / 2), np.cos(th - np.pi / 2)
    wx, wy = ext["bx"] * ct - ext["by"] * st + x, ext["bx"] * st + ext["by"] * ct + y
    lm = d["landmarks_true"]
    near = np.argmin(np.hypot(wx[:, None] - lm[0], wy[:, None] - lm[1]), axis=1)
    return int(np.bincount(near).argmax())


def _data(Tk):
    """K trajectories of Tk scans.  Trajectory 1 lacks the landmark its first scan sees most (its far observations create labels
    from the first sweep on); trajectory 3 has an empty scan at local t = 1, next to its pinned first pose, and a run of empty
    scans in its middle."""
    from icm_slam_b200.synthetic import make_synthetic_loop
    data = [make_synthetic_loop(16, T=Tk, seed=20181 + 700 + i, init_pose_noise=(0.03 * (i + 1), 0.006 * (i + 1))) for i in range(K)]
    data[1]["map_init"] = np.delete(data[1]["map_init"], _most_seen_from_start(data[1]), axis=1)
    data[3]["observations"][:, 1] = 10.0
    if Tk >= 16:
        data[3]["observations"][:, Tk // 2 - 3:Tk // 2 + 3] = 10.0
    return data


def _with_env(env, make):
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        return make()
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _batch(data, Tk, env=None):
    """The batch handle, with `env` set while it is created (the library reads its switches then)."""
    from icm_slam_b200.batch import ConcatBatch

    def make():
        b = ConcatBatch(_cfg(Tk), 0, 1, device=0)
        for i, d in enumerate(data):
            b.add(i, d["observations"], d["odometry"], d["velocities"], d["map_init"], d["x_init"])
        b.finalize()
        return b
    return _with_env(env, make)


def _translated(d, k):
    """Trajectory d in the frame ConcatBatch gives slot k (identical fp64 inputs)."""
    off = _offset(k)
    odo, x = d["odometry"].copy(), d["x_init"].copy()
    odo[0:2] += off[:, None]
    x[0:2] += off[:, None]
    return odo, x, d["map_init"] + off[:, None]


def _engine(d, Tk, odo):
    from icm_slam_b200.engine import Engine
    e = Engine(_cfg(Tk))
    e.load(d["observations"], odo, d["velocities"], precondition=True)
    e.extract()
    return e


def _state(e):
    mapa = e.get_map()
    return dict(x=e.get_poses(), map=mapa, counts=e.counts(mapa.shape[1]), c=e.associations())


def _alone(d, k, Tk, n_sweeps):
    """Trajectory d on its own handle in slot k's frame: n_sweeps fused sweeps in one call (graph replay, steady tail), and the
    same sweeps one at a time with statistics."""
    odo, x, mapa = _translated(d, k)
    out = {}
    for stats in (False, True):
        e = _engine(d, Tk, odo)
        e.set_map(mapa)
        e.set_poses(x)
        if stats:
            out["iters"], out["far"] = [], []
            for _ in range(n_sweeps):
                e.iterate(None, odo[:, 0], 1, stats=True)
                st = e.sweep_stats()
                out["iters"].append(st["newton_iters"])
                out["far"].append(st["n_far_scans"])
        else:
            e.iterate(None, odo[:, 0], n_sweeps)
            out.update(_state(e))
        e.close()
    return out


def _n_halo_bound(Tk, K_):
    """Newton iterations the fused solve may spend on halo poses (re-solved by the tile next to their owner): the iteration
    count of a batch and of its trajectories alone may differ by this much, as their tiles fall differently."""
    nblk = lambda n: (n + ST_OWN - 1) // ST_OWN
    return MAXIT * (2 * nblk(K_ * Tk) + K_ * nblk(Tk))


def _same_trajectory(got, k, Tk, a, labels=True):
    """Slot k of a batch (_got) against trajectory k alone (_state)."""
    x, mapa, counts, c, off, kk = got
    xs, ms = x[:, k * Tk:(k + 1) * Tk], mapa[:, kk == k]
    if labels:
        _same_labels_up_to_renumbering(c[off[k * Tk]:off[(k + 1) * Tk]], a["c"])
        assert np.array_equal(counts[kk == k], a["counts"]), k
    assert ms.shape == a["map"].shape, (k, ms.shape, a["map"].shape)
    d = np.abs(xs - a["x"])
    assert d[:2].max() <= TOL_XY and d[2].max() <= TOL_TH, (k, d.max(axis=1))
    assert np.abs(ms - a["map"]).max() <= TOL_MAP, k


def _got(b):
    e = b.engine
    mapa = e.get_map()
    return e.get_poses(), mapa, e.counts(mapa.shape[1]), e.associations(), e.get_extraction()["off"], _region(mapa)


def _check_data(Tk, alone, data):
    assert alone[1]["far"][0] > 0      # (trajectory 1 creates labels)
    if Tk > 64:
        assert min(alone[1]["far"]) > 0, alone[1]["far"]       # (in every sweep)
    e = _engine(data[3], Tk, data[3]["odometry"])
    off = e.get_extraction()["off"]
    e.close()
    empty = np.flatnonzero(np.diff(off) == 0)
    assert 1 in empty and off[1] > off[0] and off[Tk] > off[Tk - 1], empty
    if Tk >= 16:
        assert set(range(Tk // 2 - 3, Tk // 2 + 3)) <= set(empty.tolist()), empty


@pytest.mark.parametrize("Tk", LENGTHS)
def test_fused_batch_equals_each_trajectory_alone(Tk):
    """N_SWEEPS sweeps of the batch in the default mode (graph capture, replay, steady tail) against each trajectory on its own
    handle: labels up to renumbering, counts and map sizes exact, poses and map within the translation's resolution; per sweep,
    the batch's far-observation count is the sum of the trajectories' (and its Newton iterations are, up to halo re-solves)."""
    data = _data(Tk)
    b = _batch(data, Tk)
    b.iterate(N_SWEEPS)
    got = _got(b)
    b.close()
    b = _batch(data, Tk)
    iters, far = [], []
    for _ in range(N_SWEEPS):
        b.iterate(1, stats=True)
        st = b.engine.sweep_stats()
        iters.append(st["newton_iters"])
        far.append(st["n_far_scans"])
    assert np.array_equal(b.engine.get_poses(), got[0]) and np.array_equal(b.engine.get_map(), got[1])      # (eager == graph)
    b.close()
    alone = [_alone(d, k, Tk, N_SWEEPS) for k, d in enumerate(data)]
    _check_data(Tk, alone, data)
    assert far == [sum(a["far"][s] for a in alone) for s in range(N_SWEEPS)], far
    assert all(a["iters"][0] > 0 for a in alone)
    for s in range(N_SWEEPS):
        assert abs(iters[s] - sum(a["iters"][s] for a in alone)) <= _n_halo_bound(Tk, K), (s, iters, [a["iters"] for a in alone])
    for k, a in enumerate(alone):
        _same_trajectory(got, k, Tk, a)


@pytest.mark.parametrize("Tk", [3, 129, 1021])
def test_fused_batch_vs_oracle(Tk):
    """Every trajectory of the batch, sweep by sweep, against the CPU oracle's (redblack, newton, prev) sweep of it alone: labels
    exact up to the batch's renumbering, landmark counts exact, poses within 1e-6 m / 1e-8 rad, map within 1e-6 m."""
    from oracle import oracle as orc
    data = _data(Tk)
    b = _batch(data, Tk)
    orcs = []
    for k, d in enumerate(data):
        odo, x, mapa = _translated(d, k)
        ocfg = orc.make_cfg(**_cfgd(Tk))
        ext = orc.extract_all(orc.precondition(d["observations"], ocfg.radio, ocfg.rango_laser_max), ocfg)
        mo = orc.Mapa(ocfg)
        mo.landmarks_actuales = mapa.shape[1]
        orcs.append(dict(cfg=ocfg, ext=ext, mapa=mo, odo=odo, u=d["velocities"], map=mapa, x=np.ascontiguousarray(x)))
    for s in range(3):
        b.iterate(1)
        x, mapa, _, c, off, kk = _got(b)
        for k, o in enumerate(orcs):
            r = orc.sweep(o["cfg"], o["mapa"], o["ext"], o["odo"], o["u"], o["odo"][:, 0], o["map"], o["x"], "redblack", "newton", "prev")
            o["map"] = r["map"]
            _same_labels_up_to_renumbering(c[off[k * Tk]:off[(k + 1) * Tk]], r["c"])
            ms = mapa[:, kk == k]
            assert ms.shape == r["map"].shape, (s, k, ms.shape, r["map"].shape)
            d = np.abs(x[:, k * Tk:(k + 1) * Tk] - o["x"])
            assert d[:2].max() <= 1e-6 and d[2].max() <= 1e-8, (s, k, d.max(axis=1))
            assert np.abs(ms - r["map"]).max() <= 1e-6, (s, k)
    b.close()


@pytest.mark.parametrize("env", [{"ICMSLAM_GRAPH": "0"}, {"ICMSLAM_STEADY": "0"}, {"ICMSLAM_RUNS": "0"}])
def test_fused_batch_variants_agree_at_odd_length(env):
    """Without the CUDA graph, the steady tail or the run records, the chain of an odd-length batch is the default chain bit for bit."""
    Tk = 513
    data = _data(Tk)
    out = []
    for e in (None, env):
        b = _batch(data, Tk, e)
        b.iterate(N_SWEEPS)
        out.append((b.engine.get_poses(), b.engine.get_map(), b.engine.associations()))
        b.close()
    for a, c in zip(out[0], out[1]):
        assert np.array_equal(a, c), env


def test_host_buffer_sweeps_on_a_batch_in_chunks():
    """Engine.sweep with host buffers on an odd-length batch handle: the chunk-pipelined sweep (4 chunks) equals the one-piece host
    sweep and the device-resident chain bit for bit."""
    Tk = 1021
    data = _data(Tk)
    b = _batch(data, Tk)
    b.iterate(N_SWEEPS)
    ref = (b.engine.get_poses(), b.engine.get_map(), b.engine.associations())
    b.close()
    outs = []
    for env in ({"ICMSLAM_PIPE_CHUNKS": "1"}, {"ICMSLAM_PIPE_CHUNKS": "4", "ICMSLAM_PIPE_TILES": "1"}):
        b = _batch(data, Tk, env)
        e = b.engine
        x, mapa = np.ascontiguousarray(e.get_poses()), np.ascontiguousarray(e.get_map())
        e.landmarks_actuales = mapa.shape[1]
        for _ in range(N_SWEEPS):
            st, _, mapa = e.sweep(mapa, x, b.x0s[:, 0], fused=True)
            assert st == 0
            mapa = np.ascontiguousarray(np.array(mapa, copy=True))
        outs.append((x.copy(), mapa, e.associations()))
        b.close()
    for a, c, r in zip(outs[0], outs[1], ref):
        assert np.array_equal(a, c)
        assert np.array_equal(a, r)


# ---- the per-trajectory stop at an odd length (the construction of test_batch_convergence) --------------------------------------
K_UNTIL, TK_UNTIL, MAX_SWEEPS = 7, 509, 12


def _until_data():
    from icm_slam_b200.synthetic import make_synthetic_loop
    data = [make_synthetic_loop(16, T=TK_UNTIL, seed=20181 + 300 + i, init_pose_noise=(0.03 * (i + 1), 0.006 * (i + 1)))
            for i in range(K_UNTIL)]
    data[2]["map_init"] = np.delete(data[2]["map_init"], 5, axis=1)
    data[4]["observations"][:, 300:310] = 10.0
    data[5]["map_init"] = np.concatenate([data[5]["map_init"], data[5]["map_init"][:, 3:4] + np.array([[0.4], [0.0]])], axis=1)
    return data


def test_batch_until_at_odd_length():
    """ConcatBatch.iterate_until at an odd length against Engine.iterate_until on each trajectory alone (n_done, cambios, poses,
    map), with stopping sweeps spread so that frozen and active trajectories share run tiles; then two more sweeps of everyone."""
    from test_batch_convergence import _pick_tol
    data = _until_data()
    hist = []
    for k, d in enumerate(data):
        odo, x, mapa = _translated(d, k)
        e = _engine(d, TK_UNTIL, odo)
        e.set_map(mapa); e.set_poses(x)
        n, cam = e.iterate_until(odo[:, 0], MAX_SWEEPS, 0.0)
        e.close()
        assert n == MAX_SWEEPS
        hist.append(cam)
    tol = _pick_tol(hist)
    ref = []
    for k, d in enumerate(data):
        odo, x, mapa = _translated(d, k)
        e = _engine(d, TK_UNTIL, odo)
        e.set_map(mapa); e.set_poses(x)
        n, cam = e.iterate_until(odo[:, 0], MAX_SWEEPS, tol)
        r = dict(n=n, cambios=cam, first=_state(e))
        e.iterate(None, odo[:, 0], 2)
        r["second"] = _state(e)
        ref.append(r)
        e.close()
    assert len({r["n"] for r in ref}) >= 3, [r["n"] for r in ref]
    b = _batch(data, TK_UNTIL)
    conv = b.iterate_until(MAX_SWEEPS, tol)
    got = _got(b)
    for k in range(K_UNTIL):
        n, cam = conv[k]
        assert n == ref[k]["n"], (k, n, ref[k]["n"])
        assert cam.shape == (n, 3) and np.abs(cam - ref[k]["cambios"]).max() <= 1e-9, (k, cam, ref[k]["cambios"])
        _same_trajectory(got, k, TK_UNTIL, ref[k]["first"], labels=False)
    b.iterate(2)
    got = _got(b)
    for k in range(K_UNTIL):
        _same_trajectory(got, k, TK_UNTIL, ref[k]["second"], labels=False)
    b.close()


@pytest.mark.parametrize("T", [129, 1021])
def test_batch_of_one_equals_the_plain_handle(T):
    """set_batch(T, x0) on a handle of one odd-length trajectory changes nothing: poses, map, labels and per-sweep statistics bit
    for bit, eager and replayed."""
    d = _data(T)[1]
    runs = []
    for batch in (False, True):
        e = _engine(d, T, d["odometry"])
        if batch:
            e.set_batch(T, d["odometry"][:, :1])
        e.set_map(d["map_init"]); e.set_poses(d["x_init"])
        stats = []
        for _ in range(3):
            e.iterate(None, d["odometry"][:, 0], 1, stats=True)
            st = e.sweep_stats()
            stats.append((st["newton_iters"], st["n_far_scans"]))
        e.iterate(None, d["odometry"][:, 0], 3)
        runs.append((stats, _state(e)))
        e.close()
    assert runs[0][0] == runs[1][0], (runs[0][0], runs[1][0])
    for key in ("x", "map", "counts", "c"):
        assert np.array_equal(runs[0][1][key], runs[1][1][key]), key


def _set_batch_status(e, traj_T, x0s):
    x0s = np.ascontiguousarray(x0s, dtype=np.float64)
    return e.lib.icmslam_set_batch(e._h, int(traj_T), C.c_void_p(x0s.ctypes.data), int(x0s.shape[1]), int(x0s.shape[1]))


def test_set_batch_refusals_leave_the_handle_as_it_was():
    """icmslam_set_batch refuses a trajectory length below 3 and one that does not divide the handle (ICMSLAM_ERR_INVALID), and
    a trajectory whose first or last scan is empty (ICMSLAM_ERR_UNSUPPORTED); the handle then sweeps as it did before."""
    from icm_slam_b200.engine import Engine
    Tk = 129
    data = _data(Tk)
    b, ref = _batch(data, Tk), _batch(data, Tk)
    e, T = b.engine, K * Tk
    x0s = b.x0s
    assert _set_batch_status(e, 1, np.repeat(x0s[:, :1], T, axis=1)) == -1            # traj_T < 3 (traj_T K = T)
    assert _set_batch_status(e, 2, np.repeat(x0s[:, :1], T // 2, axis=1)) == -1       # traj_T < 3 (and K traj_T != T)
    assert _set_batch_status(e, Tk, x0s[:, :K - 1]) == -1                               # traj_T K != T
    assert _set_batch_status(e, Tk + 1, x0s[:, :K - 1]) == -1
    b.iterate(2); ref.iterate(2)
    for a, c in zip(_state(b.engine).values(), _state(ref.engine).values()):
        assert np.array_equal(a, c)
    b.close(); ref.close()
    # three laps of trajectory 0 with the first scan of the third resp. the last scan of the second empty: refused, and the
    # handle sweeps as the single trajectory it still is
    d = data[0]
    for col in (2 * Tk, 2 * Tk - 1):
        z = np.tile(d["observations"], (1, 3))
        z[:, col] = 10.0
        odo, u, x = np.tile(d["odometry"], (1, 3)), np.tile(d["velocities"], (1, 3)), np.tile(d["x_init"], (1, 3))
        mapa = d["map_init"]
        runs = []
        for refuse in (True, False):
            h = Engine(_cfg(Tk))
            h.load(z, odo, u, precondition=True)
            h.extract()
            if refuse:
                assert _set_batch_status(h, Tk, odo[:, ::Tk]) == -7, col
            h.set_map(mapa); h.set_poses(x)
            h.iterate(None, odo[:, 0], 2)
            runs.append(_state(h))
            h.close()
        for key in ("x", "map", "counts", "c"):
            assert np.array_equal(runs[0][key], runs[1][key]), (col, key)
