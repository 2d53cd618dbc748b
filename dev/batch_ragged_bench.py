"""Trajectories of different lengths in one batch handle: a ragged ConcatBatch against the equal-length batch of C5's shape and
against one handle per trajectory (TrajectoryBatch), in the default fused mode and in the reference's own mode.

    python dev/batch_ragged_bench.py [--n-traj 512] [--steps 20] [--ref-steps 2] [--n-sub 16] [--seed 20181]

* The ragged set: n-traj trajectories from make_synthetic_loop (16 landmarks, seeds seed + i) whose lengths are drawn uniformly
  from [1024, 3072] (numpy Generator seeded with `seed`) and then nudged so that they sum to n-traj x 2048, C5's column count.
* (a) the ragged ConcatBatch and (b) the equal-length n-traj x 2048 ConcatBatch (C5's batch) in the default mode
  (redblack, newton, prev); (c) the first n-sub ragged trajectories as a TrajectoryBatch, one handle each (their streams run
  concurrently), its rate scaled per trajectory; (a) and (c) again in the reference's mode (sequential, nm, running).
* Each configuration: one warm-up sweep, then the timed sweeps between a CUDA event recorded after a device synchronisation and
  one recorded after the closing device synchronisation (so the window covers every handle's stream).
Prints one JSON line with the card's name and power limit, trajectory-sweeps/s and pose-sweeps/s of each configuration."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

REFERENCE = dict(schedule="sequential", solver="nm", view="running")
T_MEAN, T_LO, T_HI = 2048, 1024, 3072


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def ragged_lengths(n, seed):
    """n lengths, uniform over [T_LO, T_HI], nudged to sum to n * T_MEAN."""
    rng = np.random.default_rng(seed)
    lengths = rng.integers(T_LO, T_HI + 1, n)
    i = 0
    while lengths.sum() != n * T_MEAN:
        step = 1 if lengths.sum() < n * T_MEAN else -1
        if T_LO <= lengths[i % n] + step <= T_HI:
            lengths[i % n] += step
        i += 1
    return lengths


def timed(torch, step, n):
    """Seconds per step: one warm-up, then n steps between CUDA events that bracket device synchronisations."""
    step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        step()
    torch.cuda.synchronize()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / n


def rates(n_traj, n_poses, s):
    return {"trajectories": int(n_traj), "poses": int(n_poses), "s_per_sweep": s, "trajectory_sweeps_per_s": n_traj / s,
            "pose_sweeps_per_s": n_poses / s}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-traj", type=int, default=512)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--ref-steps", type=int, default=2)
    ap.add_argument("--n-sub", type=int, default=16)
    ap.add_argument("--seed", type=int, default=20181)
    args = ap.parse_args()
    import torch
    from icm_slam_b200.batch import ConcatBatch, TrajectoryBatch
    from icm_slam_b200.config import ConfigICM
    from icm_slam_b200.synthetic import make_synthetic_loop
    torch.zeros(1, device="cuda")
    lengths = ragged_lengths(args.n_traj, args.seed)
    out = {"gpu": card(), "n_traj": args.n_traj, "lengths": {"min": int(lengths.min()), "max": int(lengths.max()),
           "mean": float(lengths.mean()), "sum": int(lengths.sum()), "odd": int((lengths & 1).sum())},
           "steps": args.steps, "ref_steps": args.ref_steps}
    cfg = ConfigICM.from_values(N=1, L=4 * 16, cota=20.0)      # (bench.py's C5 configuration)

    def concat(ls):
        b = ConcatBatch(cfg, 0, 1, device=0)
        data = []
        for i, n in enumerate(ls):
            d = make_synthetic_loop(16, T=int(n), seed=args.seed + i)
            b.add(i, d["observations"], d["odometry"], d["velocities"], d["map_init"], d["x_init"])
            data.append(d)
        b.finalize()
        return b, data

    b, data = concat(lengths)
    out["a_ragged_concat"] = rates(args.n_traj, lengths.sum(), timed(torch, lambda: b.iterate(1), args.steps))
    out["a_ragged_concat_reference_mode"] = rates(args.n_traj, lengths.sum(),
                                                  timed(torch, lambda: b.iterate(1, **REFERENCE), args.ref_steps))
    b.close()

    tb = TrajectoryBatch(cfg, 0, 1, device=0)
    for i in range(args.n_sub):
        d = data[i]
        tb.add(i, d["observations"], d["odometry"], d["velocities"], d["map_init"], d["x_init"])
    sub = int(lengths[:args.n_sub].sum())
    out["c_ragged_per_handle"] = rates(args.n_sub, sub, timed(torch, lambda: tb.iterate(1), args.steps))
    out["c_ragged_per_handle_reference_mode"] = rates(args.n_sub, sub, timed(torch, lambda: tb.iterate(1, **REFERENCE), args.ref_steps))
    out["c_scaled"] = "rate of %d handles sweeping concurrently, per trajectory" % args.n_sub
    tb.close()
    del data

    b, _ = concat([T_MEAN] * args.n_traj)
    out["b_equal_concat"] = rates(args.n_traj, T_MEAN * args.n_traj, timed(torch, lambda: b.iterate(1), args.steps))
    b.close()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
