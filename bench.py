#!/usr/bin/env python
"""bench.py -- ICM sweeps/s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c3|c1|c5|ijac|palomar] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one ICM sweep (iterations_process_offline, sensors.py:125-168) over the whole
trajectory: projection, association, landmark statistics, pose update, map filter.  Scan
extraction (filtrar_z) is sweep-invariant and cached, as SURVEY.md 8(d) defines the metric; its
throughput is reported separately (`extraction`).

* `value`    : sweeps/s with poses, observations and map resident in HBM (icmslam_iterate), steady
               state (the sweeps after the first run on certified run records, runs.cuh); the first
               sweep of a map chain -- every tile through the association kernel -- is `cold_sweep_ms`.
* `e2e`      : the same sweep through the reference-facing call
               ICM_SLAM.iterations_process_offline(mapa_viejo, x) with HOST numpy buffers:
               poses + map go host->device and come back inside the timed region.
* `roofline` : the dominant kernel's algorithmic bytes / its CUDA-event duration vs the measured
               HBM copy bandwidth (MEASURED_PEAKS.json).
* `cpu_baseline` / `--impl reference`: the UNMODIFIED reference (baseline/_ref, copied by
               baseline/setup_ref.py; imported through oracle/ref_runner.py) on the host cores, on a
               bounded prefix of the same workload against the full map; extrapolated numbers say so.
* `result_sha256`: hash of poses + map + labels after warm-up + steps: identical for 1/2/4/8 GPUs.
* `--dump-outputs DIR`: the same poses, map and labels as .npy files (dump_outputs), so that two builds can be
               compared array by array; the inputs of a workload are the same on every run.

Workloads: c4 (default, the metric's configuration), c3, c1 (synthetic smoke), c5 (4096 independent
trajectories), ijac / palomar (the reference's two real logs: pass 0 + sweeps, as shipped).
Under torchrun (N > 1) the trajectory is split into N contiguous time segments, one per GPU.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (L_true, T, description)
    "c4": (316 * 316, 1_000_000, "synthetic 2D range-bearing: 1M poses / 99 856 (316^2) landmarks, 181-beam scans"),
    "c3": (100 * 100, 100_000, "synthetic 2D range-bearing: 100k poses / 10k landmarks, 181-beam scans"),
    "c1": (16 * 16, 2048, "synthetic 2D range-bearing: 2048 poses / 256 landmarks (smoke size)"),
    "c5": (16, 2048, "batch of independent synthetic trajectories (T = 2048, 16 landmarks each), 512 per GPU"),
    "ijac": (11, 1833, "data_IJAC2018.mat as shipped (T = 1833, 181 beams), config_ros.yaml values, pass 0 + sweeps"),
    "palomar": (11, 1833, "datos_palomar1.mat as shipped (raw log: filtrar_obs pre-pass), config_ros.yaml values, pass 0 + sweeps"),
}
REAL_LOGS = {"ijac": "data_IJAC2018.mat", "palomar": "datos_palomar1.mat"}
SEED = 20181
METRIC = "ICM sweeps/sec (1M poses,100k lmk) at 1/2/4/8 B200; % HBM roofline"
CONFIG_ROS = dict(N=30, deltat=0.1, L=1000, Q=[1, 1], R=[1, 1, 1], cte_odom=1.0, cota=300.0, dist_thr=1.0, dist_thr_obs=1.0,
                  rango_laser_max=10.0, radio=0.137)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def config_for(L_true, name="c4"):
    from icm_slam_b200.config import ConfigICM
    if name in REAL_LOGS:
        return ConfigICM.from_values(**CONFIG_ROS)
    return ConfigICM.from_values(N=1, L=2 * L_true, cota=20.0)


def ref_dir():
    for d in (os.path.join(ROOT, "baseline", "_ref", "scripts"), "/root/reference/scripts"):
        if os.path.isfile(os.path.join(d, "sensors.py")):
            return d
    return None


def make_data(name):
    """Synthetic workloads: the generator; real logs: the .mat file of the reference copy (baseline/_ref)."""
    t0 = time.time()
    if name in REAL_LOGS:
        from icm_slam_b200.icm import load_mat
        rd = ref_dir()
        if rd is None:
            raise SystemExit("workload %s needs the reference's logs under baseline/_ref (python baseline/setup_ref.py)" % name)
        z, odo, u = load_mat(os.path.join(rd, REAL_LOGS[name]))
        d = dict(observations=z, odometry=odo, velocities=u)
    else:
        from icm_slam_b200.synthetic import make_synthetic
        L_true, T, _ = WORKLOADS[name]
        d = make_synthetic(L_true, T=T, seed=SEED + {"c1": 1, "c3": 3, "c4": 4}[name])
    d["gen_s"] = time.time() - t0
    return d


def result_hash(x, mapa, c):
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(x, dtype=np.float64).tobytes())
    h.update(np.ascontiguousarray(mapa, dtype=np.float64).tobytes())
    h.update(np.ascontiguousarray(c, dtype=np.int32).tobytes())
    return h.hexdigest()


DUMP_COLUMNS = 1 << 20


def dump_outputs(out_dir, **arrays):
    """Writes each array as <out_dir>/<name>.npy in float64 (exact for the int32 labels).  An array of more than DUMP_COLUMNS
    columns keeps a sample of them drawn with SEED (the same columns for the same length), and the sampled column indices go
    to <name>_index.npy.  C4: the full 3 x 1M poses, the full map, 2^20 of the 25M labels; about 42 MB in all."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        n = a.shape[-1]
        if n > DUMP_COLUMNS:
            idx = np.sort(np.random.default_rng(SEED).choice(n, DUMP_COLUMNS, replace=False))
            a = a[..., idx]
            np.save(os.path.join(out_dir, name + "_index.npy"), idx.astype(np.float64))
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


class ClockSampler:
    """SM clock / power / throttle reasons sampled through NVML in a thread (every 5 ms) from start() to stop(): no child
    process -- forking a process that holds gigabytes of arrays next to the timed region stalls its CUDA launches for
    milliseconds, longer than a whole timed region at 8 GPUs.  start() is called BEFORE the warm-up sweeps and stop() after a short
    stretch of untimed sweeps that follows the timed region, so the samples cover the same load; `samples_timed` counts those
    that fell inside the timed region itself (mark_timed()).  Falls back to `nvidia-smi -lms` when NVML is not importable."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []          # (time, sm_mhz, max_mhz, watts, reasons bitmask)
        self.p = None
        self.h = None
        self.stop_flag = False
        self.t_timed = [None, None]

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(self.index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.h = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.p = None

    def mark_timed(self, which):
        self.t_timed[which] = time.perf_counter()

    def _poll(self):
        nv, h = self.nv, self.h
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((time.perf_counter(), float(sm), float(mx) if mx else None, pw, int(rs)))
            except Exception:
                pass
            time.sleep(0.005)

    def _read(self):
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        for line in self.p.stdout:
            f = [v.strip() for v in line.strip().split(",")]
            if len(f) < 7:
                continue
            try:
                rs = 0
                for n, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                    if v.lower().startswith("active"):
                        rs |= bits[n]
                self.rows.append((time.perf_counter(), float(f[0]), float(f[1]), float(f[2]), rs))
            except ValueError:
                continue

    def stop(self):
        if self.h is None and self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML and nvidia-smi unavailable"]}
        if self.p is not None:
            time.sleep(0.12)
            self.p.terminate()
            try:
                self.p.wait(timeout=2)
            except Exception:
                self.p.kill()
        else:
            self.stop_flag = True
            self.th.join(timeout=1)
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        sm = [r[1] for r in self.rows]
        mx = [r[2] for r in self.rows if r[2]]
        pw = [r[3] for r in self.rows]
        reasons = set()
        for r in self.rows:
            for bit, n in names.items():
                if r[4] & bit:
                    reasons.add(n)
        t0, t1 = self.t_timed
        inside = [r for r in self.rows if t0 is not None and t1 is not None and t0 <= r[0] <= t1]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "samples_timed": len(inside),
                "sampled_over": "warm-up + timed region + >= 0.15 s of untimed sweeps after it (NVML, 5 ms period)" if self.h is not None
                                else "nvidia-smi -lms 20 from before the warm-up",
                "reasons": sorted(reasons)}


def sweep_bytes(T, n, L):
    """SURVEY.md 8(d): compulsory traffic of one sweep (fp64 SoA, int32 indices)."""
    return 92 * T + 20 * n + 40 * L + 4


def runs_bytes(T, n, L):
    """Share of the run / association kernels: poses 24T + offsets 4(T+1) + observations 16n + map 16L in, labels 4n +
    statistics 24L out (the solve moves the rest: odometry 24T + controls 16T in, poses 24T out)."""
    return 24 * T + 4 * (T + 1) + 16 * n + 16 * L + 4 * n + 24 * L


# ------------------------------------------------------------------------------------------------
def cpu_reference_arm(name, d, budget_poses=None):
    """Times the UNMODIFIED reference (`ICM_ROS.iterations_process_offline`, sensors.py:125-168, imported from baseline/_ref)
    on the host.  Synthetic workloads: one sweep over a prefix of P poses against the FULL map (the reference cannot run
    the full size: ~0.2 s per pose at 1e5 landmarks), scaled linearly to T.  Real logs: one full sweep after its own pass 0.
    Returns (sweeps_per_s, sample, seconds, P, extrapolated)."""
    from oracle import ref_runner as rr
    import scipy
    L_true, T, _ = WORKLOADS[name]
    versions = "numpy %s / scipy %s, %d host cores, 1 used (the reference is single-threaded)" % (np.__version__, scipy.__version__, os.cpu_count())
    if name in REAL_LOGS:
        cfg = rr.make_config(**CONFIG_ROS)
        z = d["observations"]
        if name == "palomar":
            from oracle import oracle as orc
            z, _ = orc.filtrar_obs(z, 10.0, 15)       # (filtrar_obs.m is MATLAB: the restated pre-pass; not timed)
        s = rr.make_solver(cfg, rr.precondition(z, cfg), d["odometry"], d["velocities"])
        key = "_ref_p0_" + name
        if key not in d:
            t0 = time.perf_counter()
            d[key] = rr.pass0(s)
            d[key]["seconds"] = time.perf_counter() - t0
        else:
            s.mapa_obj.landmarks_actuales = d[key]["mapa"].shape[1]
        x = np.ascontiguousarray(d[key]["x"].copy())
        t0 = time.perf_counter()
        rr.sweep(s, d[key]["mapa"], x)
        dt = time.perf_counter() - t0
        sample = ("unmodified reference iterations_process_offline on the whole log (T = %d), %.1f s per sweep (after its own pass 0, "
                  "%.1f s, untimed); %s" % (T, dt, d[key]["seconds"], versions))
        return 1.0 / dt, sample, dt, T, False
    P = min(budget_poses or {"c4": 26, "c3": 60, "c1": 150}.get(name, 26), T)
    cfg = rr.make_config(L=2 * L_true, cota=20.0, N=1)
    zc = rr.precondition(d["observations"][:, :P + 1], cfg)
    import ICM_SLAM as ref_icm
    while P > 2 and np.size(ref_icm.filtrar_z(zc[:, P - 1], cfg)) == 0:      # the reference needs a non-empty last scan
        P -= 1
    s = rr.make_solver(cfg, zc[:, :P], d["odometry"][:, :P], d["velocities"][:, :P])
    s.mapa_obj.landmarks_actuales = d["map_init"].shape[1]
    x = np.ascontiguousarray(d["x_init"][:, :P].copy())
    t0 = time.perf_counter()
    try:
        rr.sweep(s, d["map_init"], x)
    except ValueError:
        pass   # a short prefix may leave no landmark above cota (ICM_SLAM.py:255); the timed work is already done
    dt = time.perf_counter() - t0
    sample = ("unmodified reference iterations_process_offline on the first %d of %d poses against the full %d-landmark map, %.2f s; "
              "sweeps/s EXTRAPOLATED linearly to the full trajectory (the reference cannot run this size); %s"
              % (P, T, d["map_init"].shape[1], dt, versions))
    return 1.0 / (dt * (T / P)), sample, dt, P, True


def run_reference(args, rank, world):
    if rank != 0:
        return
    name = args.workload
    if ref_dir() is None:
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref is missing (python baseline/setup_ref.py copies the reference where /root/reference exists)"}), flush=True)
        return
    d = make_data(name)
    real = name in REAL_LOGS
    steps, warm = (min(args.steps, 2), min(args.warmup, 0)) if real else (args.steps, args.warmup)
    vals, sample, extrap, P = [], "", True, 0
    for i in range(warm + steps):
        v, sample, dt, P, extrap = cpu_reference_arm(name, d, args.ref_poses)
        if i >= warm:
            vals.append(v)
    v = float(np.mean(vals))
    L_true, T, desc = WORKLOADS[name]
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": "sweeps/s", "n_gpus": args.gpus, "steps": steps,
           "warmup": warm, "ms_per_step": 1000.0 / v, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f64", "data": "real log" if real else "synthetic",
           "config": {"workload": desc, "T": T, "L_true": L_true, "seed": SEED, "sample_poses": P, "steps_requested": args.steps},
           "extrapolated": bool(extrap),
           "cpu_baseline": {"value": v, "unit": "sweeps/s", "cores": 1, "kind": "reference", "sample": sample, "extrapolated": bool(extrap)},
           "e2e": {"value": v, "unit": "sweeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------
def run_gpu(args, rank, world, local_rank):
    import torch
    from icm_slam_b200.engine import Engine
    from icm_slam_b200.icm import ICM_SLAM, Mapa

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libicmslam has no CPU fallback")
    torch.cuda.set_device(local_rank)
    name = args.workload
    if name == "c5":
        from icm_slam_b200 import batch
        return batch.bench(args, rank, world, local_rank, SEED, METRIC, peaks, ClockSampler, sweep_bytes, dump_outputs=dump_outputs)
    if world > 1:
        from icm_slam_b200 import multigpu
        return multigpu.bench(args, rank, world, local_rank, WORKLOADS, SEED, METRIC, sweep_bytes, peaks, ClockSampler, make_data,
                              config_for, result_hash, runs_bytes, dump_outputs)

    L_true, T, desc = WORKLOADS[name]
    real = name in REAL_LOGS
    d = make_data(name)
    cfg = config_for(L_true, name)
    x0 = d["odometry"][:, 0].copy()
    dev = torch.device("cuda", local_rank)
    B = int(d["observations"].shape[0])

    # ---- device-resident arm --------------------------------------------------------------------
    eng = Engine(cfg, device=local_rank)
    stream = torch.cuda.Stream(device=dev)          # (the legacy default stream cannot capture CUDA graphs)
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    z = d["observations"]
    if name == "palomar":
        z = eng.filtrar_obs(z, float(cfg.rango_laser_max), 15)       # filtrar_obs.m pre-pass on the GPU (row a1)
    t0 = time.time()
    eng.load(z, d["odometry"], d["velocities"], precondition=True)
    load_s = time.time() - t0
    # extraction (filtrar_z of every scan, once per dataset): CUDA events around the two passes, scans already in HBM
    ex0, ex1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ex0.record(stream)
    n = eng.extract()
    ex1.record(stream)
    torch.cuda.synchronize()
    extract_ms = ex0.elapsed_time(ex1)
    if real:
        x_init, map_init = eng.pass0(x0)              # the causal initialisation (sensors.py:51-123), native
    else:
        x_init, map_init = d["x_init"], d["map_init"]
    mode = dict(schedule="redblack", solver="newton", view="prev")
    # cold sweeps: a fresh map chain, every tile through the association kernel (what a 2-sweep config_default.yaml user gets)
    cold = []
    for _ in range(3):
        eng.set_poses(x_init)
        eng.set_map(map_init)
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        eng.iterate(None, x0, 1, **mode)
        c1.record(stream)
        torch.cuda.synchronize()
        cold.append(c0.elapsed_time(c1))
    eng.set_poses(x_init)                 # ICM.positions resident on the device
    eng.set_map(map_init)
    x_dev = None
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup + 2):      # (+2: the N > 1 arm runs two more untimed sweeps; result_sha256 is taken after the
        eng.iterate(x_dev, x0, 1, **mode)  #  same number of sweeps for every N, so the lines of a scaling run carry one hash)
    torch.cuda.synchronize()
    lc0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    sampler.mark_timed(0)
    ev0.record(stream)
    for _ in range(args.steps):
        eng.iterate(x_dev, x0, 1, **mode)        # steady state: one CUDA-graph replay per sweep
    ev1.record(stream)
    torch.cuda.synchronize()
    sampler.mark_timed(1)
    ms = ev0.elapsed_time(ev1) / args.steps
    launches = (eng.launch_count() - lc0) // max(args.steps, 1)
    L_now = eng.landmarks_actuales
    outputs = dict(poses=eng.get_poses(), map=eng.get_map(), associations=eng.associations())
    sha = result_hash(outputs["poses"], outputs["map"], outputs["associations"])
    t_load = time.perf_counter()          # the same load, untimed, for the clock sampler
    while time.perf_counter() - t_load < 0.15:
        eng.iterate(x_dev, x0, 20, **mode)
        torch.cuda.synchronize()
    clocks = sampler.stop()
    # kernel time of the dominant kernels, measured live with CUDA events on the handle's stream in a
    # separate short loop (reading the events synchronises, so it stays out of the timed region)
    kt, dirty = [], []
    for _ in range(max(3, min(args.steps, 10))):
        eng.iterate(x_dev, x0, 1, timing=True, stats=True, **mode)
        kt.append(eng.kernel_ms())
        st = eng.sweep_stats()
        dirty.append(st["dirty_tiles"])
        k_runs_only = st["k_runs_ns"] * 1e-6
    k_runs_ms = float(np.mean([a for a, _ in kt]))
    k_solve_ms = float(np.mean([b for _, b in kt]))
    B_sweep = sweep_bytes(T, n, L_true)
    peak, peak_src = peaks()
    dom_name, dom_ms, dom_bytes = "k_runs (+ k_assoc_tiles on the %d dirty of %d tiles)" % (int(np.max(dirty)), st["n_tiles"]), k_runs_ms, runs_bytes(T, n, L_true)
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    sweep_achieved = B_sweep / (ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(tp):
        try:
            with open(tp) as f:
                traffic = json.load(f).get(name, {}).get("k_runs")
        except Exception:
            traffic = None
    B_extract = 8 * B * T + 20 * n

    # ---- end-to-end arm: the reference-facing call with HOST buffers --------------------------------
    icm = ICM_SLAM(cfg, x0=x0)
    icm.mediciones, icm.odometria, icm.u = d["observations"], d["odometry"], d["velocities"]
    icm.mapa_obj = Mapa(cfg)
    icm.adopt_engine(eng)                                  # same device dataset; only the call path differs
    e2e_steps = max(3, min(args.steps, 10))

    def e2e_loop(x_host):
        mapa = np.array(map_init, copy=True)
        icm.mapa_obj.landmarks_actuales = mapa.shape[1]
        for _ in range(2):
            mapa, _ = icm.iterations_process_offline(mapa, x_host)
        torch.cuda.synchronize()
        tb0 = eng.transfer_bytes()             # bytes the library actually copies (a map fed back unchanged is not re-uploaded)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            mapa, _ = icm.iterations_process_offline(mapa, x_host)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / e2e_steps
        tb1 = eng.transfer_bytes()
        return dt, (tb1[0] - tb0[0]) // e2e_steps, (tb1[1] - tb0[1]) // e2e_steps

    x_pinned = torch.from_numpy(np.array(x_init, copy=True)).pin_memory().numpy()
    e2e_s, h2d, d2h = e2e_loop(x_pinned)
    e2e_pageable_s, _, _ = e2e_loop(np.array(x_init, copy=True))

    # ---- CPU baseline (rank 0, N = 1): bounded sample of the unmodified reference ---------------------------------
    cpu = None
    if not args.no_cpu_baseline and ref_dir() is not None:
        budget = args.ref_poses or {"c4": 100, "c3": 250, "c1": 600}.get(name)
        v, sample, dt, P, extrap = cpu_reference_arm(name, d, budget)
        cpu = {"value": v, "unit": "sweeps/s", "cores": 1, "kind": "reference", "sample": sample, "extrapolated": bool(extrap)}
    elif not args.no_cpu_baseline:
        cpu = {"value": None, "unit": "sweeps/s", "cores": 0, "kind": "reference", "sample": "baseline/_ref missing"}

    out = {
        "metric": METRIC, "value": 1000.0 / ms, "unit": "sweeps/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "real log" if real else "synthetic",
        "config": {"workload": desc, "T": T, "L_true": L_true, "n_obs": int(n), "landmarks_after": int(L_now), "beams": B,
                   "seed": SEED, "mode": "redblack/newton/prev", "partition": "1 time segment",
                   "l2": "inputs larger than L2 (run records %.0f MB + observations %.0f MB + poses/odometry/controls %.0f MB vs 126 MB L2)"
                         % (32 * 0.35 * n / 1e6, 16 * n / 1e6, 64 * T / 1e6) if not real else "whole problem L2-resident (a real log of 1833 scans)",
                   "prep_s": {"data": round(d["gen_s"], 2), "load_h2d": round(load_s, 2)}},
        "clocks": clocks,
        "cold_sweep_ms": float(np.min(cold)),
        "extraction": {"scans_per_s": T / (extract_ms * 1e-3), "ms": extract_ms, "algorithmic_bytes": int(B_extract),
                       "achieved_gbs": B_extract / (extract_ms * 1e-3) / 1e9, "frac": B_extract / (extract_ms * 1e-3) / 1e9 / peak,
                       "note": "filtrar_z of all T scans (two passes over the fp64 scan array + CSR build + host sync for the sizes), 8*B*T + 20*n bytes"},
        "e2e": {"value": 1.0 / e2e_s, "unit": "sweeps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "steps": e2e_steps, "pageable_caller_buffers": 1.0 / e2e_pageable_s,
                "call": "ICM_SLAM.iterations_process_offline(mapa_viejo, x) with pinned host numpy poses (value) / pageable ones"},
        "gpu_launches": int(launches) * args.steps,
        "gpu_launches_per_step": int(launches),
        "result_sha256": sha,
        "roofline": {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src, "kernel_ms": dom_ms, "algorithmic_bytes": int(dom_bytes),
                     "sweep": {"algorithmic_bytes": int(B_sweep), "achieved": sweep_achieved, "frac": sweep_achieved / peak,
                               "kernel_ms": {"k_runs": k_runs_only, "k_runs+k_assoc_tiles": k_runs_ms, "k_solve_tile": k_solve_ms},
                               "note": "whole sweep (all kernels of the graph replay) against the sweep's algorithmic bytes"}},
        "cpu_baseline": cpu,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, **outputs)
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--ref-poses", type=int, default=None, help="prefix length for the CPU arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the poses, map and labels of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "b200":
        args.warmup = max(args.warmup, 3)          # the first sweeps build the run records; steady state needs them
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU implementation computes; the reference arm times a prefix only")
    if args.dump_outputs and args.workload == "c5" and world > 1:
        ap.error("--dump-outputs with c5 needs one rank: each rank holds only its own trajectories")
    if args.impl == "reference":
        return run_reference(args, rank, world)
    return run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
