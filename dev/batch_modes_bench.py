"""The reference's own sweep (sequential, NM, running) on many trajectories: one batch handle (ConcatBatch) against one handle
per trajectory (TrajectoryBatch), and the single-handle sequential pose kernel of this tree against another build's.

    python dev/batch_modes_bench.py [--n-traj 512] [--T 2048] [--sweeps 2] [--n-sub 16] [--baseline-lib PATH] [--reps 5]

* C5's shape: trajectories of T poses from make_synthetic_loop (16 landmarks, seeds 20181 + i).  ConcatBatch sweeps all
  n-traj in one handle; TrajectoryBatch sweeps the first n-sub of them, one handle each (their streams run concurrently), and
  its rate is scaled per trajectory: n-sub / (seconds per sweep).  Each arm: one warm-up sweep, then `sweeps` timed sweeps
  between device synchronisations.
* --baseline-lib: a libicmslam.so built from another tree (e.g. the parent commit).  One C1 (data_IJAC2018.mat) reference-mode
  sweep of a single handle, alternating the two libraries `reps` times from the same inputs: the sweep's wall time, the pose
  kernel's CUDA-event time, and whether poses and evaluation counts are identical.
Prints one JSON line with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

MODE = dict(schedule="sequential", solver="nm", view="running")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed_sweeps(torch, step, n):
    step()                                   # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        step()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n


def load_lib(path):
    """The ctypes library at `path`, with the argument types _lib gives this tree's library."""
    from icm_slam_b200 import _lib
    saved = _lib.LIB_PATH, _lib._lib
    _lib.LIB_PATH, _lib._lib = path, None
    try:
        return _lib.lib()
    finally:
        _lib.LIB_PATH, _lib._lib = saved


def engine_on(L, cfg):
    """An Engine whose handle lives in library L."""
    from icm_slam_b200 import _lib
    from icm_slam_b200.engine import Engine
    saved = _lib._lib
    _lib._lib = L
    try:
        return Engine(cfg)
    finally:
        _lib._lib = saved


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-traj", type=int, default=512)
    ap.add_argument("--T", type=int, default=2048)
    ap.add_argument("--sweeps", type=int, default=2)
    ap.add_argument("--n-sub", type=int, default=16)
    ap.add_argument("--baseline-lib", default=None)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    from icm_slam_b200 import _lib
    from icm_slam_b200.batch import ConcatBatch, TrajectoryBatch
    from icm_slam_b200.config import ConfigICM
    from icm_slam_b200.synthetic import make_synthetic_loop
    torch.zeros(1, device="cuda")
    out = {"gpu": card(), "mode": "/".join(MODE.values()), "n_traj": args.n_traj, "T": args.T, "timed_sweeps": args.sweeps}

    cfg = ConfigICM.from_values(N=1, L=64, cota=20.0)
    data = [make_synthetic_loop(16, T=args.T, seed=20181 + i) for i in range(args.n_traj)]
    b = ConcatBatch(cfg, 0, 1, device=0)
    for i, d in enumerate(data):
        b.add(i, d["observations"], d["odometry"], d["velocities"], d["map_init"], d["x_init"])
    b.finalize()
    s = timed_sweeps(torch, lambda: b.iterate(1, **MODE), args.sweeps)
    out["concat"] = {"trajectories": args.n_traj, "s_per_sweep": s, "trajectory_sweeps_per_s": args.n_traj / s,
                     "launches_per_sweep": None}
    lc = b.engine.launch_count()
    b.iterate(1, **MODE)
    out["concat"]["launches_per_sweep"] = b.engine.launch_count() - lc
    b.close()

    tb = TrajectoryBatch(cfg, 0, 1, device=0)
    for i in range(args.n_sub):
        d = data[i]
        tb.add(i, d["observations"], d["odometry"], d["velocities"], d["map_init"], d["x_init"])
    s = timed_sweeps(torch, lambda: tb.iterate(1, **MODE), args.sweeps)
    out["per_handle"] = {"trajectories": args.n_sub, "s_per_sweep": s, "trajectory_sweeps_per_s": args.n_sub / s,
                         "scaled": "rate of %d handles sweeping concurrently, per trajectory" % args.n_sub}
    tb.close()
    out["concat_over_per_handle"] = out["concat"]["trajectory_sweeps_per_s"] / out["per_handle"]["trajectory_sweeps_per_s"]

    if args.baseline_lib:
        from helpers import CONFIG_ROS, c1_inputs, golden
        g = golden("c1_ref.npz")
        z, odo, u = c1_inputs()
        ccfg = ConfigICM.from_values(**CONFIG_ROS)
        libs = {"this_tree": _lib.lib(), "baseline": load_lib(os.path.abspath(args.baseline_lib))}
        engines = {}
        for name, L in libs.items():
            e = engine_on(L, ccfg)
            e.load(z, odo, u, precondition=True)
            e.extract()
            engines[name] = e
        res = {name: {"wall_ms": [], "pose_kernel_ms": []} for name in libs}
        outs = {}
        for r in range(args.reps + 1):                       # (rep 0: warm-up)
            for name, e in engines.items():
                e.set_map(g["p0_map"])
                e.set_poses(np.ascontiguousarray(g["s1_x_in"]))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                e.iterate(None, odo[:, 0], 1, timing=True, stats=True, **MODE)
                e.synchronize()
                wall = 1e3 * (time.perf_counter() - t0)
                if r:
                    res[name]["wall_ms"].append(wall)
                    res[name]["pose_kernel_ms"].append(e.kernel_ms()[1])
                outs[name] = (e.get_poses(), e.sweep_stats()["newton_iters"], e.get_map())
        for name in libs:
            res[name] = {k: float(np.median(v)) for k, v in res[name].items()}
            res[name]["nev"] = int(outs[name][1])
        a, c = outs["this_tree"], outs["baseline"]
        res["identical_poses"] = bool(np.array_equal(a[0], c[0]))
        res["identical_map"] = bool(np.array_equal(a[2], c[2]))
        res["same_nev"] = a[1] == c[1]
        res["reference_nev"] = int(g["s1_nev"])
        res["max_dx_vs_reference"] = float(np.abs(a[0] - g["s1_x_out"]).max())
        res["new_over_old_pose_kernel"] = res["this_tree"]["pose_kernel_ms"] / res["baseline"]["pose_kernel_ms"]
        out["c1_single_handle"] = res
        for e in engines.values():
            e.close()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
