"""C5 of BASELINE.json / SURVEY.md section 8(e): a batch of INDEPENDENT trajectories (Monte-Carlo multi-start).

The path shards trivially: trajectory i belongs to rank i % world, every trajectory is one libicmslam handle (its own device
buffers, stream and CUDA graphs), and there is no data-path collective -- ranks never exchange anything while sweeping.  The
sweeps of a rank's handles are enqueued back to back on their own streams, so small trajectories overlap on the GPU.

    batch = ConcatBatch(config, rank, world)         # ONE handle for the rank's trajectories (or TrajectoryBatch: one handle each)
    for i in batch.owned(n_traj):
        batch.add(i, z_i, odo_i, u_i, map_i, x_i)
    batch.finalize()                                  # (ConcatBatch only)
    batch.iterate(30)                                 # a fixed number of sweeps of every trajectory (any sweep mode, below), or
    conv = batch.iterate_until(60, tol)               # each trajectory until its own largest landmark change is <= tol (the
                                                      # reference's stop rule, sensors.py:302-315): {i: (n_done, cambios (n_done, 3))}
    res = batch.results()          # {i: (x (3 x T), mapa (2 x L))}
    allres = gather_results(res)   # optional, for output only (torch.distributed all_gather_object)

iterate takes the sweep mode of Engine.iterate: schedule ("redblack" | "sequential"), solver ("newton" | "nm"), view ("prev" |
"full" | "running"); the default is the fast restated sweep (redblack, newton, prev).  Every mode sweeps each trajectory exactly
as it would be swept alone, so the reference's own sweep runs a whole batch in one handle:

    batch.iterate(30, schedule="sequential", solver="nm", view="running")      # the reference's ICM, one warp per trajectory

A ConcatBatch numbers new labels over the whole batch (each trajectory's labels keep their order) and its label cap applies to the
batch; iterate_until runs the default mode only.
"""
from __future__ import annotations

import numpy as np

from .engine import Engine


def owned_indices(n_traj: int, rank: int, world: int):
    """Round-robin shard: trajectory i runs on rank i % world (weak scaling: fixed work per trajectory)."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    return list(range(rank, int(n_traj), world))


class TrajectoryBatch:
    def __init__(self, config, rank: int = 0, world: int = 1, device=None):
        self.config, self.rank, self.world = config, int(rank), int(world)
        self.device = int(rank if device is None else device)
        self._eng = {}
        self._x0 = {}

    def owned(self, n_traj: int):
        return owned_indices(n_traj, self.rank, self.world)

    def add(self, idx: int, z, odometria, u, map_init, x_init, precondition=True):
        """Loads trajectory `idx` (raw ranges B x T, odometry 3 x T, controls 2 x T) with its initial map / poses."""
        if idx % self.world != self.rank:
            raise ValueError("trajectory %d belongs to rank %d" % (idx, idx % self.world))
        e = Engine(self.config, device=self.device)
        e.load(z, odometria, u, precondition=precondition)
        e.extract()
        e.set_map(map_init)
        e.set_poses(np.ascontiguousarray(x_init, dtype=np.float64))
        self._eng[idx] = e
        self._x0[idx] = np.ascontiguousarray(np.asarray(odometria, dtype=np.float64)[:, 0].copy())

    def iterate(self, n_sweeps: int = 1, **mode):
        """n_sweeps ICM sweeps of every owned trajectory; sweep k of all handles is enqueued before sweep k+1 (the calls
        are asynchronous: the handles' streams run concurrently)."""
        for _ in range(int(n_sweeps)):
            for idx, e in self._eng.items():
                e.iterate(None, self._x0[idx], 1, **mode)

    def iterate_until(self, max_sweeps: int, tol: float):
        """Engine.iterate_until of every owned trajectory: {trajectory index: (n_done, cambios (n_done, 3))}."""
        return {idx: e.iterate_until(self._x0[idx], int(max_sweeps), float(tol)) for idx, e in self._eng.items()}

    def results(self):
        return {idx: (e.get_poses(), e.get_map()) for idx, e in self._eng.items()}

    def n_observations(self):
        return sum(e.n for e in self._eng.values())

    def close(self):
        for e in self._eng.values():
            e.close()
        self._eng.clear()


class ConcatBatch:
    """The batch as ONE handle (icmslam_set_batch): the K owned trajectories (equal length) laid end to end and translated to
    disjoint regions of the plane -- their landmarks are farther apart than any gate, and the energy only sees differences of
    positions, so every trajectory is solved exactly as it would be alone -- with each trajectory's first pose pinned to its own x0.
    One sweep of the batch = one launch of each kernel over all K x T columns (TrajectoryBatch, one handle per trajectory, needs
    K x 15 small launches and is launch-bound).

        b = ConcatBatch(config_for_one_trajectory, rank, world)
        b.add(i, z_i, odo_i, u_i, map_i, x_i) ...; b.finalize(); b.iterate(30); res = b.results()

    Region k of the plane is the cell (k % 64, k // 64) of a grid of pitch `spacing` (default 256 m: a power of two, far more
    than a trajectory's extent); positions are translated in fp64, which costs < 1e-11 m of resolution at 16 km."""

    def __init__(self, config, rank: int = 0, world: int = 1, device=None, spacing: float = 256.0, labels_per_trajectory=None):
        self.config, self.rank, self.world = config, int(rank), int(world)
        self.device = int(rank if device is None else device)
        self.spacing = float(spacing)
        self.Lper = int(labels_per_trajectory if labels_per_trajectory is not None else config.L)
        self._items = []
        self.engine = None

    def owned(self, n_traj: int):
        return owned_indices(n_traj, self.rank, self.world)

    def _offset(self, k):
        return np.array([(k % 64) * self.spacing, (k // 64) * self.spacing])

    def add(self, idx: int, z, odometria, u, map_init, x_init):
        if idx % self.world != self.rank:
            raise ValueError("trajectory %d belongs to rank %d" % (idx, idx % self.world))
        if self.engine is not None:
            raise RuntimeError("finalize() was already called")
        self._items.append((int(idx), np.asarray(z, np.float64), np.asarray(odometria, np.float64), np.asarray(u, np.float64),
                            np.asarray(map_init, np.float64), np.asarray(x_init, np.float64)))

    def finalize(self, precondition=True):
        """Uploads the concatenated batch and extracts its scans."""
        from copy import copy
        K = len(self._items)
        if K == 0:
            raise ValueError("empty batch")
        Tk = self._items[0][1].shape[1]
        if any(it[1].shape[1] != Tk for it in self._items):
            raise ValueError("the trajectories of a ConcatBatch have the same length")
        if K > 64 * 64:
            raise ValueError("at most 4096 trajectories per handle")
        z = np.concatenate([it[1] for it in self._items], axis=1)
        odo = np.concatenate([it[2] for it in self._items], axis=1)
        u = np.concatenate([it[3] for it in self._items], axis=1)
        x = np.concatenate([it[5] for it in self._items], axis=1)
        maps, self._nl = [], []
        for k, it in enumerate(self._items):
            off = self._offset(k)
            odo[0:2, k * Tk:(k + 1) * Tk] += off[:, None]
            x[0:2, k * Tk:(k + 1) * Tk] += off[:, None]
            maps.append(it[4] + off[:, None])
            self._nl.append(it[4].shape[1])
        mapa = np.concatenate(maps, axis=1)
        cfg = copy(self.config)
        cfg.L = max(int(self.Lper) * K, mapa.shape[1] + K)
        self.K, self.Tk = K, Tk
        e = Engine(cfg, device=self.device)
        e.load(z, odo, u, precondition=precondition)
        e.extract()
        self.x0s = np.ascontiguousarray(np.stack([odo[:, k * Tk] for k in range(K)], axis=1))
        e.set_batch(Tk, self.x0s)
        e.set_map(mapa)
        e.set_poses(np.ascontiguousarray(x))
        self.engine = e
        self._items = [(it[0],) for it in self._items]
        return e.n

    def iterate(self, n_sweeps: int = 1, **mode):
        """n_sweeps sweeps of every trajectory in the sweep mode of Engine.iterate (schedule, solver, view, ...), each trajectory
        exactly as alone; e.g. iterate(n, schedule="sequential", solver="nm", view="running") for the reference's own ICM."""
        self.engine.iterate(None, self.x0s[:, 0], int(n_sweeps), **mode)

    def iterate_until(self, max_sweeps: int, tol: float):
        """Each trajectory sweeps until its own largest landmark change is <= tol (at most max_sweeps), exactly as
        Engine.iterate_until on it alone; a trajectory that has stopped is frozen on the device while the others sweep on
        (Engine.batch_iterate_until).  {trajectory index: (n_done, cambios (n_done, 3))}, keyed like results()."""
        _, n_done, cam = self.engine.batch_iterate_until(int(max_sweeps), float(tol), self.spacing, 64)
        return {it[0]: (int(n_done[k]), cam[k, : n_done[k]].copy()) for k, it in enumerate(self._items)}

    def results(self):
        """{trajectory index: (x (3 x T), mapa (2 x L))} in each trajectory's own frame; a landmark belongs to the region it lies in."""
        x = self.engine.get_poses()
        mapa = self.engine.get_map()
        cell = np.rint(mapa / self.spacing).astype(np.int64)      # (landmarks lie within spacing / 2 of their region's origin)
        kk = cell[1] * 64 + cell[0]
        out = {}
        for k, it in enumerate(self._items):
            off = self._offset(k)
            xs = x[:, k * self.Tk:(k + 1) * self.Tk].copy()
            xs[0:2] -= off[:, None]
            out[it[0]] = (xs, mapa[:, kk == k] - off[:, None])
        return out

    def n_observations(self):
        return self.engine.n

    def close(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None


def gather_results(local: dict, group=None):
    """All ranks' results as one dict (output only -- not part of the timed path)."""
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized():
        return dict(local)
    parts = [None] * dist.get_world_size(group)
    dist.all_gather_object(parts, local, group=group)
    out = {}
    for p in parts:
        out.update(p)
    return out


# ---- bench arm for the batch workload (called by bench.py --workload c5; one rank per GPU, no data-path collective) ---------
def bench(args, rank, world, local_rank, SEED, METRIC, peaks, ClockSampler, sweep_bytes, per_gpu=512, Tk=2048, L_true=16,
          dump_outputs=None):
    import json
    import time

    import torch

    from .config import ConfigICM
    from .synthetic import make_synthetic_loop

    dist = None
    if world > 1:
        import os
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(local_rank)
    n_traj = per_gpu * world
    cfg = ConfigICM.from_values(N=1, L=4 * L_true, cota=20.0)
    b = ConcatBatch(cfg, rank, world, device=local_rank)
    t0 = time.time()
    for i in b.owned(n_traj):
        d = make_synthetic_loop(L_true, T=Tk, seed=SEED + i)        # per-trajectory seeds 20181 + i (SURVEY.md 8d)
        b.add(i, d["observations"], d["odometry"], d["velocities"], d["map_init"], d["x_init"])
    gen_s = time.time() - t0
    stream = torch.cuda.Stream(device=dev, priority=-1)
    torch.cuda.set_stream(stream)
    n_obs = b.finalize()
    b.engine.set_stream(stream.cuda_stream)
    K = b.K
    sampler = ClockSampler(local_rank)     # (NVML polling thread, from before the warm-up to after the timed region)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        b.iterate(1)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
        torch.cuda.synchronize()
    lc0 = b.engine.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.mark_timed(0)
    ev0.record(stream)
    for _ in range(args.steps):
        b.iterate(1)
    ev1.record(stream)
    torch.cuda.synchronize()
    sampler.mark_timed(1)
    ms = ev0.elapsed_time(ev1) / args.steps
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        nt = torch.tensor([n_obs], dtype=torch.int64, device=dev)
        dist.all_reduce(nt)
        n_tot = int(nt.item())
    else:
        n_tot = n_obs
    launches = (b.engine.launch_count() - lc0) // max(args.steps, 1)
    outputs = dict(poses=b.engine.get_poses(), map=b.engine.get_map(), associations=b.engine.associations()) if args.dump_outputs else None
    t_load = time.perf_counter()          # the same load, untimed, for the clock sampler
    while time.perf_counter() - t_load < 0.15:
        b.iterate(20)
        torch.cuda.synchronize()
    clocks = sampler.stop()
    # end to end: every trajectory's poses and map go host -> device, one sweep, and come back, every step
    x_host = torch.from_numpy(b.engine.get_poses()).pin_memory().numpy()
    mapa = b.engine.get_map()
    e2e_steps = max(3, min(args.steps, 10))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    h2d = d2h = 0
    for _ in range(e2e_steps):
        b.engine.set_map(mapa)
        b.engine.set_poses(x_host)
        b.iterate(1)
        b.engine.get_poses(out=x_host)
        mapa = b.engine.get_map()
        h2d += mapa.nbytes + x_host.nbytes
        d2h += mapa.nbytes + x_host.nbytes
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    if dist is not None:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    if rank == 0:
        peak, peak_src = peaks()
        B_sweep = sweep_bytes(Tk * n_traj, n_tot, L_true * n_traj)
        achieved = B_sweep / (ms * 1e-3) / 1e9
        out = {
            "metric": METRIC, "value": n_traj * 1000.0 / ms, "unit": "trajectory-sweeps/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "batch of %d independent synthetic trajectories (T = %d, %d landmarks each, seeds %d + i), %d per GPU, one "
                                   "handle per GPU (icmslam_set_batch): a step = one ICM sweep of every trajectory" % (n_traj, Tk, L_true, SEED, per_gpu),
                       "n_trajectories": n_traj, "T_per_trajectory": Tk, "n_obs": n_tot, "mode": "redblack/newton/prev",
                       "partition": "trajectories round-robin over ranks, no data-path collective",
                       "l2": "inputs larger than L2 (%.0f MB of run records + poses per rank)" % ((24 * 0.35 * n_obs + 64 * Tk * K) / 1e6),
                       "prep_s": {"synthetic_gen": round(gen_s, 2)}},
            "clocks": clocks,
            "e2e": {"value": n_traj / e2e_s, "unit": "trajectory-sweeps/s", "h2d_bytes_per_step": int(h2d // e2e_steps) * world,
                    "d2h_bytes_per_step": int(d2h // e2e_steps) * world, "steps": e2e_steps,
                    "call": "Engine.set_map / set_poses / iterate / get_poses / get_map of the rank's concatenated batch with host buffers"},
            "gpu_launches": int(launches) * args.steps * world, "gpu_launches_per_step": int(launches),
            "roofline": {"bound": "hbm", "kernel": "whole sweep (all kernels of the graph replay)", "achieved": achieved, "peak": peak * world, "unit": "GB/s",
                         "frac": achieved / (peak * world), "traffic": None, "peak_source": peak_src, "kernel_ms": ms,
                         "algorithmic_bytes": int(B_sweep)},
            "cpu_baseline": None,
        }
        if outputs is not None:
            dump_outputs(args.dump_outputs, **outputs)
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    b.close()
