"""Device memory of a handle and CUDA-event times of the paths outside the fused sweep (the generic sweep's association,
Mapa.filtrar, calc_cambio), for comparing two builds of the library.  Run it from each tree:

    python dev/generic_paths_time.py [--reps 10] [--out FILE.json]

Prints one JSON line: the card's name and power limit, the memory icmslam_create takes (cudaMemGetInfo around it) at
L = 4096 and at C4's L, and the median time of
  * a generic sweep (sequential, nm, running) on C1 (data_IJAC2018.mat, tests/golden) and on a 2304-landmark synthetic field
    (a quarter of the repetitions: its sequential schedule is slow),
  * pass 0 on C1,
  * calc_cambio of a C4-sized map (99 856 landmarks) against a copy moved by up to 0.1 m.
Each timed call runs on the handle's stream bracketed by CUDA events, host-memory inputs included."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def create_bytes(torch, Engine, cfg):
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    e = Engine(cfg)
    torch.cuda.synchronize()
    used = free0 - torch.cuda.mem_get_info()[0]
    e.close()
    return int(used)


def timed(torch, e, fn, reps):
    stream = torch.cuda.Stream()
    e.set_stream(stream.cuda_stream)
    fn()                                            # warm-up (module load, scan workspace)
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        ms.append(a.elapsed_time(b))
    e.set_stream(None)
    return round(float(np.median(ms)), 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from helpers import CONFIG_ROS, c1_inputs, golden
    from icm_slam_b200.config import ConfigICM
    from icm_slam_b200.engine import Engine
    from icm_slam_b200.synthetic import make_synthetic
    torch.cuda.init()
    torch.zeros(1, device="cuda")
    res = {"card": card(), "tree": ROOT}
    L_c4 = 2 * 316 * 316
    res["create_bytes"] = {"L=4096": create_bytes(torch, Engine, ConfigICM.from_values(**dict(CONFIG_ROS, L=4096))),
                           "L=%d (C4)" % L_c4: create_bytes(torch, Engine, ConfigICM.from_values(N=1, L=L_c4, cota=20.0))}

    def generic_sweep(cfgd, z, odo, u, map0, x0, reps):
        e = Engine(ConfigICM.from_values(**cfgd))
        e.load(z, odo, u, precondition=True)
        e.extract()

        def run():
            e.landmarks_actuales = map0.shape[1]
            x = np.ascontiguousarray(x0.copy())
            e.sweep(map0, x, odo[:, 0], schedule="sequential", solver="nm", view="running")
        t = timed(torch, e, run, reps)
        e.close()
        return t

    g = golden("c1_ref.npz")
    z, odo, u = c1_inputs()
    t = {"generic_sweep_c1_ms": generic_sweep(dict(CONFIG_ROS), z, odo, u, g["p0_map"], g["p0_x"], args.reps)}
    d = make_synthetic(2304, seed=20181 + 31)
    t["generic_sweep_synthetic_2304_ms"] = generic_sweep(dict(CONFIG_ROS, L=2 * 2304 + 64, cota=20.0), d["observations"], d["odometry"],
                                                         d["velocities"], d["map_init"], d["x_init"],
                                                         max(args.reps // 4, 2))      # (one warp walks the 23 040 poses)
    e = Engine(ConfigICM.from_values(**CONFIG_ROS))
    e.load(z, odo, u, precondition=True)
    e.extract()
    t["pass0_c1_ms"] = timed(torch, e, lambda: e.pass0(odo[:, 0]), args.reps)
    e.close()
    rng = np.random.default_rng(20181 + 35)
    gx, gy = np.meshgrid(np.arange(316), np.arange(316), indexing="xy")
    old = np.ascontiguousarray(np.stack([4.0 * gx.ravel(), 4.0 * gy.ravel()]) + rng.uniform(-0.75, 0.75, (2, 316 * 316)))
    new = np.ascontiguousarray(old + rng.uniform(-0.07, 0.07, old.shape))
    e = Engine(ConfigICM.from_values(N=1, L=L_c4, cota=20.0))
    t["calc_cambio_c4_map_ms"] = timed(torch, e, lambda: e.calc_cambio(new, old), args.reps)
    t["calc_cambio_c4_map_result"] = list(e.calc_cambio(new, old))
    e.close()
    res["times"] = t
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
