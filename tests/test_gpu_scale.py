"""Parity at the sizes the numbers are quoted on (run on the B200 box with `-m gpu`).

* C3 (BASELINE configs[2]: 100k poses / 10k landmarks): two chained fast-mode sweeps -- the first through the association
  kernel (grid search), the second on the certified run records -- against the CPU oracle's brute force over all landmarks:
  labels / counts bit-exact, poses <= 1e-6 m / 1e-8 rad, map <= 1e-6 m.
* C4 (BASELINE configs[3]: 1M poses / 99 856 landmarks, the headline): the oracle's brute force does not finish at this size, so
  one steady-state sweep is checked piecewise against the oracle's primitives: (a) the labels of >= 2000 random scans by
  brute force over ALL landmarks, (b) EVERY landmark mean and count recomputed from the GPU labels by an independent numpy
  bincount, (c) >= 2000 random poses re-solved with the oracle's exact Newton from the GPU's own neighbours.
* the real multi-rank path: 2 NCCL ranks under torchrun == the single engine, bit for bit (skipped with < 2 GPUs).
"""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import CONFIG_ROS

pytestmark = pytest.mark.gpu

TOL_XY = 1e-6
TOL_TH = 1e-8
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def test_c3_three_sweeps_vs_oracle_brute_force():
    from icm_slam_b200.synthetic import make_synthetic
    from oracle import oracle as orc
    L, T = 100 * 100, 100_000
    d = make_synthetic(L, T=T, seed=20181 + 3)
    cfgd = dict(CONFIG_ROS, L=2 * L, cota=20.0)
    z, odo, u = d["observations"], d["odometry"], d["velocities"]
    ocfg = orc.make_cfg(**cfgd)
    ext = orc.extract_all(orc.precondition(z, ocfg.radio, ocfg.rango_laser_max), ocfg)
    e = _engine(_cfg(**cfgd), z, odo, u)
    assert e.n == ext["n"]
    mo = orc.Mapa(ocfg)
    map_o = d["map_init"].copy()
    mo.landmarks_actuales = map_o.shape[1]
    xo = np.ascontiguousarray(d["x_init"].copy())
    e.set_map(d["map_init"])
    e.set_poses(xo.copy())
    dirty = []
    for k in range(3):
        r = orc.sweep(ocfg, mo, ext, odo, u, odo[:, 0], map_o, xo, "redblack", "newton", "prev")
        e.iterate(None, odo[:, 0], 1, stats=True)
        st = e.sweep_stats()
        dirty.append((st["dirty_tiles"], st["n_tiles"]))
        xg, mout = e.get_poses(), e.get_map()
        assert np.array_equal(e.associations(), r["c"]), k
        assert mout.shape == r["map"].shape, k
        assert np.array_equal(e.counts(mout.shape[1]), r["counts"]), k
        dd = np.abs(xg - xo)
        assert dd[:2].max() <= TOL_XY and dd[2].max() <= TOL_TH, (k, dd.max(axis=1))
        assert np.max(np.abs(mout - r["map"])) <= TOL_XY, k
        map_o = r["map"]
    assert dirty[0][0] == dirty[0][1]                 # first sweep: every tile through the association kernel
    assert dirty[1][0] == dirty[1][1]                 # second: the first filter renumbered the landmarks, its run records are void
    assert dirty[2][0] < dirty[2][1] // 4, dirty      # third sweep: (almost) every tile on its run records
    e.close()


def test_c4_steady_sweep_sampled_against_oracle_primitives():
    from icm_slam_b200.synthetic import make_synthetic
    from oracle import oracle as orc
    L, T = 316 * 316, 1_000_000
    d = make_synthetic(L, T=T, seed=20181 + 4)
    cfgd = dict(CONFIG_ROS, L=2 * L, cota=20.0)
    z, odo, u = d["observations"], d["odometry"], d["velocities"]
    ocfg = orc.make_cfg(**cfgd)
    e = _engine(_cfg(**cfgd), z, odo, u)
    x0 = odo[:, 0].copy()
    e.set_map(d["map_init"])
    e.set_poses(d["x_init"])
    e.iterate(None, x0, 3)                            # association kernel, then run records
    x_in, map_in = e.get_poses(), e.get_map()         # inputs of the sweep under test
    e.iterate(None, x0, 1, stats=True)
    st = e.sweep_stats()
    assert st["dirty_tiles"] < st["n_tiles"] // 4, st  # a steady-state sweep: the tiles ran on their records
    x_out, map_out = e.get_poses(), e.get_map()
    c = e.associations()
    raw, raw_cnt, raw_L = e.raw_map()
    g = e.get_extraction()
    off, bx, by, beam, dd = g["off"], g["bx"], g["by"], g["beam"], g["d"]
    Lin = map_in.shape[1]
    n = int(off[-1])
    assert n > 20_000_000 and Lin > 99_000
    rng = np.random.default_rng(20181)
    # ---- (a) labels of random scans: brute force over ALL landmarks of the input map --------------------------------
    scans = np.unique(np.concatenate([rng.integers(0, T, 2200), [0, 1, T - 2, T - 1]]))
    mo = orc.Mapa(ocfg)
    checked = 0
    for t in scans:
        a, b = int(off[t]), int(off[t + 1])
        if b == a:
            continue
        pose = x0 if t == 0 else x_in[:, t]
        wx, wy = orc.tras_rot(pose, bx[a:b], by[a:b])
        mo.clear_obs()
        mo.landmarks_actuales = Lin
        scratch = np.zeros((2, mo.L))
        _, cc = mo.actualizar(scratch, map_in, np.stack([wx, wy], axis=1))
        far_o, far_g = cc >= Lin, c[a:b] >= Lin
        assert np.array_equal(far_o, far_g), t
        assert np.array_equal(cc[~far_o], c[a:b][~far_g]), t
        checked += b - a
    assert checked > 40_000
    # ---- (b) every landmark mean and count from the GPU labels (independent numpy bincount) -------------------------
    scan_of = np.repeat(np.arange(T), np.diff(off))
    P = x_in.copy()
    P[:, 0] = x0
    th = P[2, scan_of] - np.pi / 2.0
    ct, sn = np.cos(th), np.sin(th)
    wx = bx * ct - by * sn + P[0, scan_of]
    wy = bx * sn + by * ct + P[1, scan_of]
    cnt = np.bincount(c, minlength=raw_L)[:raw_L]
    assert np.array_equal(cnt, raw_cnt.astype(np.int64))
    seen = cnt > 0
    mx = np.bincount(c, wx, minlength=raw_L)[:raw_L][seen] / cnt[seen]
    my = np.bincount(c, wy, minlength=raw_L)[:raw_L][seen] / cnt[seen]
    assert np.max(np.abs(raw[0][seen] - mx)) <= 1e-8 and np.max(np.abs(raw[1][seen] - my)) <= 1e-8
    # ... and the filtered map is those means for the landmarks that reach cota (nothing merges on this field)
    keep = cnt >= cfgd["cota"]
    assert map_out.shape[1] == int(keep.sum())
    assert np.max(np.abs(map_out[0] - (np.bincount(c, wx, minlength=raw_L)[:raw_L][keep] / cnt[keep]))) <= 1e-8
    # ---- (c) random poses re-solved with the oracle's exact Newton ----------------------------------------------------
    ang = g["beam"] * np.pi / 180.0
    seen_x = np.where(c < Lin, map_in[0][np.minimum(c, Lin - 1)], raw[0][np.minimum(c, raw_L - 1)])
    seen_y = np.where(c < Lin, map_in[1][np.minimum(c, Lin - 1)], raw[1][np.minimum(c, raw_L - 1)])
    worst = np.zeros(3)
    for t in np.unique(np.concatenate([rng.integers(1, T - 1, 2200), [1, 2, T - 2]])):
        a, b = int(off[t]), int(off[t + 1])
        if b == a:
            continue
        X = x_in if (t & 1) else x_out              # odd poses see the old even neighbours, even poses the new odd ones
        xa = X[:, t - 1]
        sol, _ = orc.solve_pose(ocfg, "newton", xa, X[:, t + 1], u[:, t - 1], u[:, t], odo[:, t - 1:t + 2], dd[a:b], ang[a:b],
                                seen_x[a:b], seen_y[a:b])
        worst = np.maximum(worst, np.abs(sol - x_out[:, t]))
    assert worst[:2].max() <= TOL_XY and worst[2] <= TOL_TH, worst
    e.close()


def result_hash(x, mapa, c):
    h = hashlib.sha256()
    for a in (np.ascontiguousarray(x, dtype=np.float64), np.ascontiguousarray(mapa, dtype=np.float64), np.ascontiguousarray(c, dtype=np.int32)):
        h.update(a.tobytes())
    return h.hexdigest()


def test_two_nccl_ranks_equal_the_single_engine_bit_for_bit(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = tmp_path / "seg.json"
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29517", os.path.join(ROOT, "tests", "nccl_segments_worker.py"), str(out)]
    subprocess.run(cmd, check=True, env=env, timeout=900, cwd=ROOT)
    import json
    res = json.loads(out.read_text())
    assert res["segmented_p2p"] == res["single"], res       # the library's exchange over peer memory (csrc/p2p.cuh)
    assert res["segmented_nccl"] == res["single"], res      # NCCL collectives between the segment calls
    assert res["fallback_exchange"] == "nccl" and res["segmented_fallback"] == res["single"], res   # one rank without peer memory
