"""Ragged batch handles (icmslam_set_batch_lengths / ConcatBatch with trajectories of different lengths): every trajectory of
the batch against its own handle and against the CPU oracle, in every sweep mode, with the chain's variants, the per-trajectory
stop, equal lengths through both entry points, and the refusals (run with `-m gpu`).

The lengths mix parities, so trajectories start on odd and even columns; their boundaries fall at many offsets inside the
128-scan run-record tiles and the 126-pose solve tiles, a 3-scan trajectory sits between two odd-length ones, and the record
tile of columns 128-255 holds three trajectories."""
import ctypes as C

import numpy as np
import pytest

from helpers import CONFIG_ROS
from test_batch_lengths import _most_seen_from_start, _with_env
from test_batch_modes import MODES, _same_labels_up_to_renumbering

pytestmark = pytest.mark.gpu

SPACING = 256.0      # ConcatBatch's default region pitch
LENGTHS = [129, 3, 1021, 128, 513, 127, 2048]
LENGTHS_MODES = [129, 3, 511, 128, 257, 127, 512]      # (the sequential Nelder-Mead walk is slow on long trajectories)
N_SWEEPS = 4
TOL_XY, TOL_TH, TOL_MAP = 1e-9, 1e-11, 1e-9      # the fp64 translation of each trajectory into its region
MAXIT = 20       # the fused solve's default Newton iteration cap
ST_OWN = 126     # poses a solve tile owns (solve.cuh)
# (a landmark of a 3-scan trajectory is seen a handful of times: cota 20 would filter out every one; L leaves room for the
#  labels trajectory 0 creates every sweep)
CFGD = dict(CONFIG_ROS, L=2048, cota=2.0)


def _cfg(**kw):
    from icm_slam_b200.config import ConfigICM
    d = dict(CFGD)
    d.update(kw)
    return ConfigICM.from_values(**d)


def _starts(lengths):
    return np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)


def _offset(k):
    return np.array([(k % 64) * SPACING, (k // 64) * SPACING])


def _region(mapa):
    cell = np.rint(mapa / SPACING).astype(np.int64)
    return cell[1] * 64 + cell[0]


def _data(lengths, seed=20181 + 900):
    """Trajectory 0 lacks the landmark its first scan sees most, and its scan 60 is turned by 40 beams: what that scan sees lies
    far from every landmark and is seen once, so cota 2 filters it out and it creates labels every sweep.  Trajectory 4 has an
    empty scan at local t = 1, next to its pinned first pose, and a run of empty scans in its middle."""
    from icm_slam_b200.synthetic import make_synthetic_loop
    data = [make_synthetic_loop(16, T=int(n), seed=seed + i, init_pose_noise=(0.03 * (i % 5 + 1), 0.006 * (i % 5 + 1)))
            for i, n in enumerate(lengths)]
    data[0]["map_init"] = np.delete(data[0]["map_init"], _most_seen_from_start(data[0]), axis=1)
    data[0]["observations"][:, 60] = np.roll(data[0]["observations"][:, 60], 40)
    n4 = int(lengths[4])
    data[4]["observations"][:, 1] = 10.0
    data[4]["observations"][:, n4 // 2 - 3:n4 // 2 + 3] = 10.0
    return data


def _batch(data, env=None, cfg=None):
    """The ConcatBatch of `data`, with `env` set while it is created (the library reads its switches then)."""
    from icm_slam_b200.batch import ConcatBatch

    def make():
        b = ConcatBatch(cfg or _cfg(), 0, 1, device=0)
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


def _engine(d, k, cfg=None):
    """Trajectory d alone, on its own handle in slot k's frame, with its map and poses set."""
    from icm_slam_b200.engine import Engine
    odo, x, mapa = _translated(d, k)
    e = Engine(cfg or _cfg())
    e.load(d["observations"], odo, d["velocities"], precondition=True)
    e.extract()
    e.set_map(mapa)
    e.set_poses(x)
    return e, odo


def _state(e):
    mapa = e.get_map()
    return dict(x=e.get_poses(), map=mapa, counts=e.counts(mapa.shape[1]), c=e.associations())


def _got(e):
    mapa = e.get_map()
    return e.get_poses(), mapa, e.counts(mapa.shape[1]), e.associations(), e.get_extraction()["off"], _region(mapa)


def _same_trajectory(got, k, starts, a, labels=True, exact=False):
    """Slot k of a batch (_got) against trajectory k alone (_state)."""
    x, mapa, counts, c, off, kk = got
    xs, ms = x[:, starts[k]:starts[k + 1]], mapa[:, kk == k]
    if labels:
        _same_labels_up_to_renumbering(c[off[starts[k]]:off[starts[k + 1]]], a["c"])
        assert np.array_equal(counts[kk == k], a["counts"]), k
    assert ms.shape == a["map"].shape, (k, ms.shape, a["map"].shape)
    if exact:
        assert np.array_equal(xs, a["x"]), (k, np.abs(xs - a["x"]).max(axis=1))
        assert np.array_equal(ms, a["map"]), k
    else:
        d = np.abs(xs - a["x"])
        assert d[:2].max() <= TOL_XY and d[2].max() <= TOL_TH, (k, d.max(axis=1))
        assert np.abs(ms - a["map"]).max() <= TOL_MAP, k


def _nblk(n):
    return (n + ST_OWN - 1) // ST_OWN


@pytest.fixture(scope="module")
def data():
    return _data(LENGTHS)


def test_ragged_layout_is_what_the_lengths_say(data):
    """The starts have both parities, a record tile holds three trajectories, trajectory 0 creates labels in every sweep and
    trajectory 4 has its empty scans where _data put them."""
    starts = _starts(LENGTHS)
    assert len({int(s) & 1 for s in starts[:-1]}) == 2
    assert sum(1 for k in range(len(LENGTHS)) if starts[k] < 256 and starts[k + 1] > 128) == 3
    e, odo = _engine(data[4], 4)
    off = e.get_extraction()["off"]
    e.close()
    n4 = LENGTHS[4]
    empty = set(np.flatnonzero(np.diff(off) == 0).tolist())
    assert 1 in empty and 0 not in empty and n4 - 1 not in empty
    assert set(range(n4 // 2 - 3, n4 // 2 + 3)) <= empty


def test_ragged_fused_batch_equals_each_trajectory_alone(data):
    """N_SWEEPS default-mode sweeps of the ragged batch (graph capture, replay, steady tail) against each trajectory on its own
    handle: labels up to renumbering, counts and map sizes exact, poses and map within the translation's resolution; per sweep,
    the batch's far-scan count is the sum of the trajectories' (and its Newton iterations are, up to halo re-solves)."""
    starts = _starts(LENGTHS)
    b = _batch(data)
    b.iterate(N_SWEEPS)
    got = _got(b.engine)
    b.close()
    b = _batch(data)
    iters, far = [], []
    for _ in range(N_SWEEPS):
        b.iterate(1, stats=True)
        st = b.engine.sweep_stats()
        iters.append(st["newton_iters"])
        far.append(st["n_far_scans"])
    assert np.array_equal(b.engine.get_poses(), got[0]) and np.array_equal(b.engine.get_map(), got[1])      # (eager == graph)
    b.close()
    alone = []
    for k, d in enumerate(data):
        a = {}
        e, odo = _engine(d, k)
        e.iterate(None, odo[:, 0], N_SWEEPS)
        a.update(_state(e))
        e.close()
        e, odo = _engine(d, k)
        a["iters"], a["far"] = [], []
        for _ in range(N_SWEEPS):
            e.iterate(None, odo[:, 0], 1, stats=True)
            st = e.sweep_stats()
            a["iters"].append(st["newton_iters"])
            a["far"].append(st["n_far_scans"])
        e.close()
        alone.append(a)
    assert min(alone[0]["far"]) > 0, alone[0]["far"]      # (trajectory 0 creates labels in every sweep)
    assert far == [sum(a["far"][s] for a in alone) for s in range(N_SWEEPS)], far
    bound = MAXIT * (2 * _nblk(int(starts[-1])) + 2 * sum(_nblk(n) for n in LENGTHS))
    for s in range(N_SWEEPS):
        assert abs(iters[s] - sum(a["iters"][s] for a in alone)) <= bound, (s, iters, [a["iters"] for a in alone])
    for k, a in enumerate(alone):
        _same_trajectory(got, k, starts, a)


def test_ragged_fused_batch_vs_oracle(data):
    """Every trajectory of the ragged batch, sweep by sweep, against the CPU oracle's (redblack, newton, prev) sweep of it alone:
    labels exact up to the batch's renumbering, map sizes exact, poses within 1e-6 m / 1e-8 rad, map within 1e-6 m."""
    from oracle import oracle as orc
    starts = _starts(LENGTHS)
    b = _batch(data)
    orcs = []
    for k, d in enumerate(data):
        odo, x, mapa = _translated(d, k)
        ocfg = orc.make_cfg(**CFGD)
        ext = orc.extract_all(orc.precondition(d["observations"], ocfg.radio, ocfg.rango_laser_max), ocfg)
        mo = orc.Mapa(ocfg)
        mo.landmarks_actuales = mapa.shape[1]
        orcs.append(dict(cfg=ocfg, ext=ext, mapa=mo, odo=odo, u=d["velocities"], map=mapa, x=np.ascontiguousarray(x)))
    for s in range(3):
        b.iterate(1)
        x, mapa, _, c, off, kk = _got(b.engine)
        for k, o in enumerate(orcs):
            r = orc.sweep(o["cfg"], o["mapa"], o["ext"], o["odo"], o["u"], o["odo"][:, 0], o["map"], o["x"], "redblack", "newton", "prev")
            o["map"] = r["map"]
            _same_labels_up_to_renumbering(c[off[starts[k]]:off[starts[k + 1]]], r["c"])
            ms = mapa[:, kk == k]
            assert ms.shape == r["map"].shape, (s, k, ms.shape, r["map"].shape)
            d = np.abs(x[:, starts[k]:starts[k + 1]] - o["x"])
            assert d[:2].max() <= 1e-6 and d[2].max() <= 1e-8, (s, k, d.max(axis=1))
            assert np.abs(ms - r["map"]).max() <= 1e-6, (s, k)
    b.close()


@pytest.mark.parametrize("schedule,solver,view", MODES)
def test_ragged_batch_mode_equals_each_trajectory_alone(schedule, solver, view):
    """Every sweep mode (the generic kernels) on a ragged batch against each trajectory alone: running views bit for bit, prev and
    full views within 1e-9 (their means are float atomics), labels up to renumbering, counts exact, and the batch's summed
    iteration counts equal to the sum of the single runs."""
    mode = dict(schedule=schedule, solver=solver, view=view)
    data = _data(LENGTHS_MODES, seed=20181 + 950)
    starts = _starts(LENGTHS_MODES)
    b = _batch(data)
    iters = []
    for _ in range(3):
        b.iterate(1, fused=False, stats=True, **mode)
        iters.append(b.engine.sweep_stats()["newton_iters"])
    got = _got(b.engine)
    b.close()
    alone = []
    for k, d in enumerate(data):
        e, odo = _engine(d, k)
        it = []
        for _ in range(3):
            e.iterate(None, odo[:, 0], 1, fused=False, stats=True, **mode)
            it.append(e.sweep_stats()["newton_iters"])
        a = _state(e)
        a["iters"] = it
        e.close()
        alone.append(a)
    assert iters == [sum(a["iters"][s] for a in alone) for s in range(3)], (iters, [a["iters"] for a in alone])
    assert all(a["iters"][0] > 0 for a in alone if len(a["x"][0]) > 3)
    for k, a in enumerate(alone):
        _same_trajectory(got, k, starts, a, exact=(view == "running"))


@pytest.mark.parametrize("Tk", [256, 257])
@pytest.mark.parametrize("mode", [{}, dict(schedule="sequential", solver="nm", view="running", fused=False)])
def test_equal_lengths_through_both_entry_points(Tk, mode):
    """Equal lengths given to icmslam_set_batch_lengths and to icmslam_set_batch are one layout: poses, map and labels bit for
    bit, in the default mode and in the reference's own (sequential, nm, running)."""
    data = _data([Tk] * 5, seed=20181 + 980)
    out = []
    for equal in (False, True):
        b = _batch(data, cfg=_cfg(cota=20.0))
        if equal:
            b.engine.set_batch(Tk, b.x0s)
        b.iterate(3, **mode)
        out.append(_state(b.engine))
        b.close()
    for key in ("x", "map", "counts", "c"):
        assert np.array_equal(out[0][key], out[1][key]), key


@pytest.mark.parametrize("env", [{"ICMSLAM_GRAPH": "0"}, {"ICMSLAM_STEADY": "0"}, {"ICMSLAM_RUNS": "0"}])
def test_ragged_variants_agree(data, env):
    """Without the CUDA graph, the steady tail or the run records, the chain of a ragged batch is the default chain bit for bit."""
    out = []
    for e in (None, env):
        b = _batch(data, e)
        b.iterate(N_SWEEPS)
        out.append((b.engine.get_poses(), b.engine.get_map(), b.engine.associations()))
        b.close()
    for a, c in zip(out[0], out[1]):
        assert np.array_equal(a, c), env


def test_ragged_host_buffer_sweeps_in_chunks(data):
    """Engine.sweep with host buffers on a ragged batch: the chunk-pipelined sweep (4 chunks) equals the one-piece host sweep and
    the device-resident chain bit for bit."""
    b = _batch(data)
    b.iterate(N_SWEEPS)
    ref = (b.engine.get_poses(), b.engine.get_map(), b.engine.associations())
    b.close()
    outs = []
    for env in ({"ICMSLAM_PIPE_CHUNKS": "1"}, {"ICMSLAM_PIPE_CHUNKS": "4", "ICMSLAM_PIPE_TILES": "1"}):
        b = _batch(data, env)
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


# ---- the per-trajectory stop on a ragged batch (the construction of test_batch_convergence) ------------------------------------
LENGTHS_UNTIL, MAX_SWEEPS = [509, 130, 257, 383, 1021, 128, 131], 12


def _until_data():
    from icm_slam_b200.synthetic import make_synthetic_loop
    data = [make_synthetic_loop(16, T=n, seed=20181 + 300 + i, init_pose_noise=(0.03 * (i + 1), 0.006 * (i + 1)))
            for i, n in enumerate(LENGTHS_UNTIL)]
    data[2]["map_init"] = np.delete(data[2]["map_init"], 5, axis=1)
    data[4]["observations"][:, 300:310] = 10.0
    data[5]["map_init"] = np.concatenate([data[5]["map_init"], data[5]["map_init"][:, 3:4] + np.array([[0.4], [0.0]])], axis=1)
    return data


def test_ragged_batch_until():
    """ConcatBatch.iterate_until on a ragged batch against Engine.iterate_until on each trajectory alone (n_done, cambios, poses,
    map), with stopping sweeps spread over three or more sweeps; then two more sweeps of everyone."""
    from test_batch_convergence import _pick_tol
    cfg = _cfg(cota=20.0)
    data = _until_data()
    starts = _starts(LENGTHS_UNTIL)
    hist = []
    for k, d in enumerate(data):
        e, odo = _engine(d, k, cfg)
        n, cam = e.iterate_until(odo[:, 0], MAX_SWEEPS, 0.0)
        e.close()
        assert n == MAX_SWEEPS
        hist.append(cam)
    tol = _pick_tol(hist)
    ref = []
    for k, d in enumerate(data):
        e, odo = _engine(d, k, cfg)
        n, cam = e.iterate_until(odo[:, 0], MAX_SWEEPS, tol)
        r = dict(n=n, cambios=cam, first=_state(e))
        e.iterate(None, odo[:, 0], 2)
        r["second"] = _state(e)
        ref.append(r)
        e.close()
    assert len({r["n"] for r in ref}) >= 3, [r["n"] for r in ref]
    b = _batch(data, cfg=cfg)
    conv = b.iterate_until(MAX_SWEEPS, tol)
    got = _got(b.engine)
    for k in range(len(data)):
        n, cam = conv[k]
        assert n == ref[k]["n"], (k, n, ref[k]["n"])
        assert cam.shape == (n, 3) and np.abs(cam - ref[k]["cambios"]).max() <= 1e-9, (k, cam, ref[k]["cambios"])
        _same_trajectory(got, k, starts, ref[k]["first"], labels=False)
    b.iterate(2)
    got = _got(b.engine)
    for k in range(len(data)):
        _same_trajectory(got, k, starts, ref[k]["second"], labels=False)
    b.close()


def _lengths_status(e, lengths, x0s):
    lengths = np.ascontiguousarray(lengths, dtype=np.int32)
    x0s = np.ascontiguousarray(x0s, dtype=np.float64)
    K = int(lengths.shape[0])
    return e.lib.icmslam_set_batch_lengths(e._h, C.c_void_p(lengths.ctypes.data), K, C.c_void_p(x0s.ctypes.data), max(K, 1))


def test_set_batch_lengths_refusals_leave_the_handle_as_it_was(data):
    """icmslam_set_batch_lengths refuses a length below 3, lengths whose sum is not T and K = 0 (ICMSLAM_ERR_INVALID), and a
    trajectory whose first or last scan is empty (ICMSLAM_ERR_UNSUPPORTED); the handle then sweeps exactly as before."""
    b, ref = _batch(data), _batch(data)
    e = b.engine
    L = list(LENGTHS)
    K = len(L)
    x0 = np.repeat(b.x0s[:, :1], K + 1, axis=1)
    assert _lengths_status(e, [2, L[0] - 2] + L[1:], x0[:, :K + 1]) == -1                # a length of 2
    assert _lengths_status(e, L[:-1] + [L[-1] - 1], x0[:, :K]) == -1                      # sum T - 1
    assert _lengths_status(e, L[:-1] + [L[-1] + 1], x0[:, :K]) == -1                      # sum T + 1
    assert _lengths_status(e, np.zeros(0, np.int32), x0[:, :1]) == -1                     # K = 0
    # trajectory 4's scan at local t = 1 is empty: as the first scan of a trajectory, and as the last one
    assert _lengths_status(e, L[:3] + [L[3] + 1, L[4] - 1] + L[5:], x0[:, :K]) == -7
    assert _lengths_status(e, L[:3] + [L[3] + 2, L[4] - 2] + L[5:], x0[:, :K]) == -7
    b.iterate(2)
    ref.iterate(2)
    for key, a in _state(b.engine).items():
        assert np.array_equal(a, _state(ref.engine)[key]), key
    b.close()
    ref.close()
