"""Online ingestion on the device: the per-message cost of `Engine.append` (one column) + `Engine.pass0_advance` against a
full replay of the prefix (`load` + `extract` + `pass0`), on the palomar log (tests/golden/c2_inputs.npz: datos_palomar1's raw
scans through the filtrar_obs pre-pass, config_ros values) at T = 500, 1000 and 1833.

Each time is a host clock around work that ends in a device synchronise.  The incremental arm feeds the log one column at a
time through one handle and reports the median latency of the messages that bring columns T - 50 .. T - 1; the replay arm
reports the median of three replays of the prefix.  The fed walk's final pass-0 result is compared with the replay's bit for
bit.  Prints the card name and power limit of the same run.

    python dev/online_append_bench.py [--sizes 500,1000,1833] [--window 50] [--replays 3]
"""
from __future__ import annotations

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


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except Exception as e:       # (reported, not fatal: the timings stand without it)
        pl = "unknown (%s)" % e
    return name, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="500,1000,1833")
    ap.add_argument("--window", type=int, default=50)
    ap.add_argument("--replays", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from helpers import CONFIG_ROS, c2_inputs
    from icm_slam_b200.config import ConfigICM
    from icm_slam_b200.engine import Engine

    sizes = [int(s) for s in args.sizes.split(",")]
    cfg = ConfigICM.from_values(**CONFIG_ROS)
    raw, odo, u = c2_inputs()
    pre = Engine(cfg)
    z = np.ascontiguousarray(pre.filtrar_obs(raw, float(cfg.rango_laser_max), 15))      # filtrar_obs.m pre-pass
    pre.close()
    Tmax = max(sizes)
    assert Tmax <= z.shape[1]
    x0 = odo[:, 0].copy()

    # incremental: load column 0, then one append + advance per message
    e = Engine(cfg)
    e.load(z[:, :1], odo[:, :1], u[:, :1], precondition=True)
    e.extract()
    assert e.pass0_begin(x0) == 0
    e.pass0_advance()
    lat = np.zeros(Tmax)
    for t in range(1, Tmax):
        t0 = time.perf_counter()
        e.append(z[:, t:t + 1], odo[:, t:t + 1], u[:, t:t + 1])
        assert e.pass0_advance() == t + 1
        e.synchronize()
        lat[t] = time.perf_counter() - t0
    x_fed, m_fed = e.pass0_finish()

    rows = []
    ref = Engine(cfg)
    for T in sizes:
        reps = []
        for _ in range(args.replays):
            t0 = time.perf_counter()
            ref.load(z[:, :T], odo[:, :T], u[:, :T], precondition=True)
            ref.extract()
            xr, mr = ref.pass0(x0)
            ref.synchronize()
            reps.append(time.perf_counter() - t0)
        w = lat[max(1, T - args.window):T]
        rows.append({"T": T, "append_advance_ms_median": 1e3 * float(np.median(w)), "append_advance_ms_max": 1e3 * float(np.max(w)),
                     "replay_ms_median": 1e3 * float(np.median(reps)), "replay_ms_min": 1e3 * float(np.min(reps))})
        if T == Tmax:
            same = bool(np.array_equal(xr, x_fed) and np.array_equal(mr, m_fed))
    name, pl = card()
    out = {"card": name, "power_limit": pl, "log": "palomar (filtrar_obs pre-pass), config_ros", "rows": rows,
           "fed_equals_replay_at_T_%d" % Tmax: same, "message_budget_ms_at_10Hz": 100.0}
    print(json.dumps(out))
    for r in rows:
        print("T=%5d  append+advance %.3f ms (median of %d, max %.3f)   replay %.1f ms" % (
            r["T"], r["append_advance_ms_median"], args.window, r["append_advance_ms_max"], r["replay_ms_median"]))
    e.close()
    ref.close()


if __name__ == "__main__":
    main()
