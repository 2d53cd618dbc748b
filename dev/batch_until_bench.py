"""Per-trajectory convergence of a C5-sized batch (ConcatBatch.iterate_until) against the fixed loop that runs every trajectory
as long as the slowest one (ConcatBatch.iterate(max n_done)).  Prints one JSON line.

    python dev/batch_until_bench.py [--n-traj 512] [--T 2048] [--max-sweeps 40] [--reps 3]

Trajectory i starts from poses perturbed by (0.01 + 0.15 i / n) m and (0.002 + 0.03 i / n) rad, so the trajectories need very
different numbers of sweeps.  The tolerance is chosen from the batch's own calc_cambio histories to spread the stopping sweeps.
Per-sweep times come from the difference of iterate_until calls with max_sweeps = s and s - 1 from the same start (map and
poses set again: a fresh map chain), each timed between device synchronisations."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-traj", type=int, default=512)
    ap.add_argument("--T", type=int, default=2048)
    ap.add_argument("--max-sweeps", type=int, default=40)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    from icm_slam_b200.batch import ConcatBatch
    from icm_slam_b200.config import ConfigICM
    from icm_slam_b200.synthetic import make_synthetic_loop

    n = args.n_traj
    cfg = ConfigICM.from_values(N=1, L=64, cota=20.0)
    b = ConcatBatch(cfg, 0, 1, device=0)
    for i in range(n):
        d = make_synthetic_loop(16, T=args.T, seed=20181 + i, init_pose_noise=(0.01 + 0.15 * i / n, 0.002 + 0.03 * i / n))
        b.add(i, d["observations"], d["odometry"], d["velocities"], d["map_init"], d["x_init"])
    b.finalize()
    e = b.engine
    map0, x0 = e.get_map(), e.get_poses()

    def reset():
        e.set_map(map0)
        e.set_poses(x0)
        torch.cuda.synchronize()

    def timed(fn):
        reset()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, out

    # the histories with no stopping, then a tolerance that spreads the stopping sweeps
    _, hist = timed(lambda: b.iterate_until(args.max_sweeps, 0.0))
    mx = np.stack([hist[i][1][:, 1] for i in range(n)])          # (n, max_sweeps) largest change per sweep
    # (a trajectory that never gets below tol runs all max_sweeps sweeps, as Engine.iterate_until would run it)
    best = None
    for tol in np.geomspace(np.percentile(mx, 1), np.percentile(mx, 95), 200):
        nd = np.where((mx <= tol).any(axis=1), np.argmax(mx <= tol, axis=1) + 1, args.max_sweeps)
        if best is None or np.std(nd) > best[0]:
            best = (float(np.std(nd)), float(tol), nd)
    _, tol, nd = best
    n_max = int(nd.max())
    b.iterate_until(n_max, tol)      # warm-up of the frozen path (its CUDA graph)
    b.iterate(n_max)
    t_until, t_fixed, fallbacks = [], [], []
    for _ in range(args.reps):
        t, conv = timed(lambda: b.iterate_until(n_max, tol))
        t_until.append(t)
        fallbacks.append(e.sweep_stats()["batch_until_fallbacks"])
        t_fixed.append(timed(lambda: b.iterate(n_max))[0])
    got = np.array([conv[i][0] for i in range(n)])
    # per-sweep time against the number of trajectories still active
    cum = np.zeros(n_max + 1)
    for s in range(1, n_max + 1):
        cum[s] = np.median([timed(lambda: b.iterate_until(s, tol))[0] for _ in range(args.reps)])
    per_sweep = [{"sweep": s, "active": int((nd >= s).sum()), "ms": round(1e3 * (cum[s] - cum[s - 1]), 4)} for s in range(1, n_max + 1)]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    out = {"gpu": gpu, "n_traj": n, "T": args.T, "tol": tol,
           "max_change_p5_p50_p95": {"first_sweep": np.percentile(mx[:, 0], [5, 50, 95]).tolist(),
                                     "last_sweep": np.percentile(mx[:, -1], [5, 50, 95]).tolist()},
           "n_done_min": int(nd.min()), "n_done_max": n_max,
           "n_done_hist": np.bincount(nd, minlength=n_max + 1)[1:].tolist(), "sweeps_run": n_max,
           "trajectory_sweeps_until": int(nd.sum()), "trajectory_sweeps_fixed": n * n_max,
           "until_s": t_until, "fixed_s": t_fixed, "until_over_fixed": float(np.median(t_until) / np.median(t_fixed)),
           "fallback_sweeps": fallbacks, "n_done_equals_histories": bool(np.array_equal(got, nd)),
           "per_sweep": per_sweep}
    print(json.dumps(out), flush=True)
    b.close()


if __name__ == "__main__":
    main()
