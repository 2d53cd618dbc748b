"""Time-segment partition of the ICM sweep over the GPUs of one node (one process per GPU).

The reference sweep is a sequential Gauss-Seidel in time (sensors.py:145-162) and does not partition;
the restated (red-black, exact inner solve, previous-map view) sweep does (DESIGN.md):

* the trajectory is cut into contiguous segments whose boundaries are even and balanced by the number
  of valid beams; segment r loads its own columns plus two halo columns on the left and one on the
  right (the poses its boundary poses are coupled to through the odometry terms);
* per sweep each rank runs the fused kernel on its segment, then the ranks
    1. all-gather a 16-double record with the number of scans that created a label, which gives the
       global numbering of the new labels (ICM_SLAM.py:174-182 is an exclusive prefix over time);
    2. sum-reduce the per-landmark statistics (int64 fixed point + int32 counts: exact and
       order-free, so the map is bit-identical for any number of GPUs) and the new labels' means;
  and every rank applies the same landmark update + Mapa.filtrar to the reduced statistics;
* BESIDE 1-2 and the map update (none of which reads the new poses), on the library's low-priority side
  stream and a second communicator: the pose solve of the segment, then an all-gather of its boundary
  poses (another 16-double record) that gives every rank its halo poses for the next sweep.

Two implementations of the exchange (SegmentedSolver(exchange=...), default from ICMSLAM_EXCHANGE, else "p2p"):

* "p2p"  -- the library's own kernels over peer memory (csrc/p2p.cuh): the ranks open each other's buffers once with CUDA IPC
  (the handles travel through one torch.distributed all-gather at set-up); after that a sweep is ONE call into the library per
  rank (icmslam_iterate: a CUDA graph with the solve and the halo exchange on a low-priority branch) and no collective: far
  counts, statistics (reduce-scatter by remote loads, the gather folded into the landmark update) and halo poses are NVLink
  loads / stores flagged with the sweep number.  GPUs of one node.
* "nccl" -- torch.distributed collectives between the library's seg_begin / seg_halo / seg_exchange / seg_finish calls, as
  described above (NCCL on GPUs; the host logic is exercised with gloo in tests/test_multigpu_cpu.py).

Both give bit-identical results (integer statistics), identical to one GPU.  All device work happens in libicmslam.so; this
module only moves pointers.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

SEG_REC = 16
PTR_SEG_REC, PTR_STAT_X, PTR_STAT_Y, PTR_STAT_N, PTR_NEW_LABELS, PTR_POSES, PTR_EXCHANGE, PTR_SEG_REC_POSE, PTR_SIDE_STREAM = range(9)


# ---- partition ---------------------------------------------------------------------------------------------
def plan_segments(T: int, world: int, weights=None, align: int = 2):
    """Global owned ranges [(g_lo, g_hi)] of the `world` segments: contiguous, covering [0, T), boundaries
    multiples of `align` (even: the red-black colours stay aligned with the global time index), balanced by the
    cumulative `weights` (per-pose work, e.g. valid beams per scan) or by pose count."""
    if world < 1 or T < 1:
        raise ValueError("need world >= 1 and T >= 1")
    align = max(2, int(align) + (int(align) & 1))
    w = np.ones(T) if weights is None else np.asarray(weights, dtype=np.float64) + 1.0
    cum = np.concatenate([[0.0], np.cumsum(w)])
    cuts = [0]
    for r in range(1, world):
        target = cum[-1] * r / world
        t = int(np.searchsorted(cum, target))
        t = int(round(t / align)) * align
        t = max(t, cuts[-1] + align)          # every segment owns at least `align` poses
        cuts.append(t)
    cuts.append(T)
    if any(b <= a for a, b in zip(cuts[:-1], cuts[1:])) or cuts[-2] > T - 3 and world > 1:
        raise ValueError("trajectory too short for %d segments" % world)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def local_columns(seg, r: int, world: int):
    """Columns [c_lo, c_hi) segment r loads (owned + halo) and its owned range in local indices."""
    g_lo, g_hi = seg[r]
    c_lo = g_lo - (0 if r == 0 else 2)
    c_hi = g_hi + (0 if r == world - 1 else 1)
    return c_lo, c_hi, g_lo - c_lo, g_hi - c_lo


def label_bases(far_totals):
    """New labels are numbered in time order: segment r starts after the scans-with-far-observations of the
    segments before it.  Returns (exclusive prefix, total)."""
    f = np.asarray(far_totals, dtype=np.int64)
    return np.concatenate([[0], np.cumsum(f)[:-1]]), int(f.sum())


def make_record(first_pose, second_last_pose, last_pose, far_total):
    rec = np.zeros(SEG_REC)
    rec[0:3] = first_pose
    rec[3:6] = second_last_pose
    rec[6:9] = last_pose
    rec[9] = float(far_total)
    return rec


def halo_from_records(all_recs, r: int, world: int):
    """What segment r reads from the gathered records: (left halo poses (3x2) or None, right halo pose (3,) or None)."""
    left = None if r == 0 else np.stack([all_recs[r - 1][3:6], all_recs[r - 1][6:9]], axis=1)
    right = None if r == world - 1 else np.array(all_recs[r + 1][0:3])
    return left, right


# ---- collectives (any torch.distributed backend) -----------------------------------------------------------
def gather_records(rec, group=None):
    """All-gather of one SEG_REC-double record per rank -> (world, SEG_REC) tensor on rec's device."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    out = torch.empty((world, SEG_REC), dtype=rec.dtype, device=rec.device)
    dist.all_gather_into_tensor(out, rec.reshape(1, SEG_REC).contiguous(), group=group) if rec.is_cuda else \
        dist.all_gather(list(out.unbind(0)), rec.reshape(SEG_REC).contiguous(), group=group)
    return out


def reduce_statistics(tensors, group=None):
    """Sum-reduction over the segments of the per-landmark statistics (integers: exact, order-free)."""
    import torch.distributed as dist
    works = [dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group, async_op=True) for t in tensors]
    for w in works:
        w.wait()


class _DevBuf:
    """Zero-copy view of a device buffer of the library for torch (CUDA array interface)."""

    def __init__(self, ptr, count, typestr):
        self.__cuda_array_interface__ = {"shape": (int(count),), "typestr": typestr, "data": (int(ptr), False), "version": 2}


# ---- the solver ------------------------------------------------------------------------------------------------
class SegmentedSolver:
    """One instance per rank.  `group` is a torch.distributed process group (default: the world)."""

    def __init__(self, config, rank: int, world: int, device: int = 0, group=None, halo_group=None, split_exchange=True, exchange=None):
        """halo_group: a second process group over the same ranks for the boundary-pose exchange that runs beside the label /
        statistics exchange (created with dist.new_group when None and world > 1: a collective call, like the constructor itself
        must then be).  split_exchange=False keeps everything on one stream and one communicator."""
        from .engine import Engine
        self.config, self.rank, self.world, self.device, self.group = config, int(rank), int(world), int(device), group
        self.halo_group = halo_group
        self.split_exchange = bool(split_exchange)
        import os
        self.exchange = (exchange or os.environ.get("ICMSLAM_EXCHANGE") or "p2p").lower()
        if self.exchange not in ("p2p", "nccl"):
            raise ValueError("exchange must be 'p2p' or 'nccl'")
        if self.world == 1:
            self.exchange = "nccl"        # (nothing to exchange: the segment calls run back to back)
        self._p2p_on = False
        self.engine = Engine(config, device=device)
        self._views = None
        self._graphs = {}
        self._steady = 0
        self._parity = 0
        self._launches = 0
        self._launches_per_sweep = 0

    # -- data -------------------------------------------------------------------------------------------------
    def load(self, scans, odometry, controls, precondition=True, weights=None):
        """Every rank passes the same full arrays (B x T, 3 x T, 2 x T); only its segment goes to its GPU."""
        T = int(scans.shape[1])
        if weights is None:
            weights = (np.nan_to_num(np.asarray(scans), nan=np.inf) < self.config.rango_laser_max - self.config.radio).sum(axis=0)
        self.T = T
        self.segments = plan_segments(T, self.world, weights)
        self.c_lo, self.c_hi, self.t_lo, self.t_hi = local_columns(self.segments, self.rank, self.world)
        sl = slice(self.c_lo, self.c_hi)
        e = self.engine
        e.load(np.ascontiguousarray(scans[:, sl]), np.ascontiguousarray(odometry[:, sl]), np.ascontiguousarray(controls[:, sl]),
               precondition=precondition)
        n = e.extract()
        from ._lib import check
        check(e.lib.icmslam_set_segment(e._h, self.t_lo, self.t_hi, int(self.rank == 0), int(self.rank == self.world - 1)), e._h)
        self.x0 = np.ascontiguousarray(np.asarray(odometry[:, 0], dtype=np.float64).reshape(3))
        self._last_map = None
        self._views = None
        self._graphs = {}
        self._steady = 0
        self._parity = 0
        self._launches = 0
        self._launches_per_sweep = 0
        return n

    def set_map(self, mapa):
        """mapa_viejo for the next sweep.  A caller that hands back the map `get_map()` gave it (mapa_viejo = mapa_refinado,
        sensors.py:315) continues the device-side map chain -- grid, proven radii, run records -- instead of starting a new one
        with a full re-association: the bytes are compared, as icmslam_sweep does for host-memory sweeps."""
        last = getattr(self, "_last_map", None)
        if last is not None and isinstance(mapa, np.ndarray) and mapa.shape == last.shape and np.array_equal(mapa, last):
            return False          # (nothing uploaded)
        self._last_map = None
        self.engine.set_map(mapa)
        self._steady = 0          # the next sweeps rebuild the grid eagerly ...
        self._graphs = {}         # ... and a captured graph bakes in which of the ping-pong buffers is current
        self._parity = 0
        return True

    def set_poses(self, x_full):
        self._graphs = {}
        self._parity = 0
        self.engine.set_poses(np.asarray(x_full)[:, self.c_lo:self.c_hi])      # (a strided view: copied by the library)

    # -- views of the library's exchange buffers ------------------------------------------------------------------
    def _ptr(self, which):
        from ._lib import check
        p, n = C.c_void_p(), C.c_int64()
        check(self.engine.lib.icmslam_device_ptr(self.engine._h, which, C.byref(p), C.byref(n)), self.engine._h)
        return p.value, n.value

    def _bind(self):
        import torch
        dev = "cuda:%d" % self.device
        mk = lambda which, ts: torch.as_tensor(_DevBuf(*self._ptr(which), ts), device=dev)
        self._views = dict(rec=mk(PTR_SEG_REC, "<f8"), sx=mk(PTR_STAT_X, "<i8"), sy=mk(PTR_STAT_Y, "<i8"), sn=mk(PTR_STAT_N, "<i4"),
                           new=mk(PTR_NEW_LABELS, "<f8"), all=mk(PTR_EXCHANGE, "<i8"), recp=mk(PTR_SEG_REC_POSE, "<f8"))

    # -- sweeps ---------------------------------------------------------------------------------------------------
    def _sweep_once(self, opts=None, stamps=None):
        """One sweep.  `stamps` (a list) receives CUDA events after each stage: begin (run / association / solve kernels),
        all-gather, exchange (label numbering), all-reduce, finish (map filter)."""
        from . import _lib
        from ._lib import check
        import torch
        e = self.engine
        v = self._views

        def stamp():
            if stamps is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(torch.cuda.current_stream(self.device))
                stamps.append(ev)

        split = self.split_exchange and self.world > 1 and stamps is None and opts is None
        if opts is None:
            opts = _lib.SweepOpts(_lib.SCHED["redblack"], _lib.SOLVER["newton"], _lib.VIEW["prev"], 0, 0.0, 1, 4 if split else 0)
        stamp()
        check(e.lib.icmslam_seg_begin(e._h, C.c_void_p(self.x0.ctypes.data), C.byref(opts)), e._h)
        stamp()
        if self.world > 1:
            import torch.distributed as dist
            if split:      # the solve is on the side stream: its boundary poses follow it there, beside everything below
                with torch.cuda.stream(self._side):
                    dist.all_gather_into_tensor(self._allpose, v["recp"].reshape(1, SEG_REC), group=self.halo_group)
                check(e.lib.icmslam_seg_halo(e._h, C.c_void_p(self._allpose.data_ptr()), self.rank, self.world), e._h)
            dist.all_gather_into_tensor(self._allrec, v["rec"].reshape(1, SEG_REC), group=self.group)
            stamp()
            check(e.lib.icmslam_seg_exchange(e._h, C.c_void_p(self._allrec.data_ptr()), self.rank, self.world), e._h)
            stamp()
            dist.all_reduce(v["all"], group=self.group)      # the four statistics buffers as one block of int64 words
            stamp()
        else:
            check(e.lib.icmslam_seg_exchange(e._h, C.c_void_p(v["rec"].data_ptr()), 0, 1), e._h)
        check(e.lib.icmslam_seg_finish(e._h), e._h)
        stamp()

    def timed_sweep(self):
        """One eager sweep with the library's kernel timers on (collective); returns engine.kernel_ms()."""
        from . import _lib
        import torch
        self._prepare()
        self._last_map = None
        if self._p2p_on:
            self.engine.iterate(None, self.x0, 1, timing=True)
        else:
            with torch.cuda.stream(self._stream):
                self._sweep_once(_lib.SweepOpts(_lib.SCHED["redblack"], _lib.SOLVER["newton"], _lib.VIEW["prev"], 0, 0.0, 1, 2))
            self._steady += 1
            self._parity ^= 1
            self._graphs = {}
        return self.engine.kernel_ms()

    def stage_times(self, n=5):
        """Mean milliseconds per stage over n eager sweeps (CUDA events on the solver's stream): what a step is made of."""
        import torch
        self._prepare()
        self._last_map = None
        if self._p2p_on:
            return None        # (no host-visible stages: the exchange happens inside the library's kernels)
        names = ["begin: k_runs + k_assoc_tiles + k_solve_tile + far scan", "all-gather (128 B per rank)", "exchange: halo unpack + new labels",
                 "all-reduce (statistics block)", "finish: landmark update + Mapa.filtrar + grid"] if self.world > 1 else \
                ["begin: k_runs + k_assoc_tiles + k_solve_tile + far scan", "exchange + finish"]
        acc = np.zeros(len(names))
        caller = torch.cuda.current_stream(self.device)
        self._stream.wait_stream(caller)
        with torch.cuda.stream(self._stream):
            for _ in range(n):
                st = []
                self._sweep_once(stamps=st)
                self._steady += 1
                self._parity ^= 1
                torch.cuda.synchronize()
                acc += np.array([st[i].elapsed_time(st[i + 1]) for i in range(len(st) - 1)])
        caller.wait_stream(self._stream)
        self._graphs = {}          # (an odd number of eager sweeps flips the ping-pong parity the graphs were captured for)
        return dict(zip(names, (acc / n).tolist()))

    def _prepare(self):
        import torch
        if self._views is None:
            self._bind()
        if getattr(self, "_allrec", None) is None:
            self._allrec = torch.empty((self.world, SEG_REC), dtype=torch.float64, device="cuda:%d" % self.device)
            self._allpose = torch.empty((self.world, SEG_REC), dtype=torch.float64, device="cuda:%d" % self.device)
            self._side = torch.cuda.ExternalStream(self._ptr(PTR_SIDE_STREAM)[0], device=self.device)
            if self.exchange == "nccl" and self.split_exchange and self.world > 1 and self.halo_group is None:
                import torch.distributed as dist
                self.halo_group = dist.new_group(ranks=list(range(self.world))) if self.group is None else None
                self._own_halo_group = self.halo_group is not None
                if self.halo_group is None:
                    self.split_exchange = False        # (a sub-group solver must be given its halo group)
        # The collectives run on torch's current stream over zero-copy views of the library's buffers, so the library must
        # enqueue on that same stream, or nothing orders its kernels against the collectives.  The solver owns one stream
        # for both (the legacy default stream cannot be captured into a graph) and orders it against the caller's.
        if getattr(self, "_stream", None) is None:
            self._stream = torch.cuda.Stream(device=self.device, priority=-1)   # (above the handle's low-priority solve stream)
            self.engine.set_stream(self._stream.cuda_stream)
        if self.exchange == "p2p" and not self._p2p_on:
            self._enable_p2p()
            if self.exchange == "nccl" and self.split_exchange and self.halo_group is None and self.world > 1:
                import torch.distributed as dist      # (the fall-back needs its second communicator after all)
                self.halo_group = dist.new_group(ranks=list(range(self.world))) if self.group is None else None
                self._own_halo_group = self.halo_group is not None
                if self.halo_group is None:
                    self.split_exchange = False

    def _enable_p2p(self):
        """Collective: every rank exports its three IPC handles, all ranks gather them and open each other's buffers.  If any
        rank cannot (no peer access, IPC not permitted in this container, ...) ALL ranks fall back to the NCCL exchange."""
        import torch
        import torch.distributed as dist
        from ._lib import check
        e = self.engine
        nbytes = 192
        dev = "cuda:%d" % self.device
        buf = C.create_string_buffer(nbytes)
        ok, why = 1, ""
        try:
            check(e.lib.icmslam_p2p_export(e._h, buf, nbytes), e._h)
            import os
            if os.environ.get("ICMSLAM_P2P_FAIL") == str(self.rank):      # (test hook: this rank pretends it cannot export)
                raise RuntimeError("peer memory switched off for this rank (ICMSLAM_P2P_FAIL)")
        except Exception as ex:      # noqa: BLE001
            ok, why = 0, str(ex)
        mine = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).to(dev)
        allh = torch.empty(self.world * nbytes, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allh, mine, group=self.group)
        raw = allh.cpu().numpy().tobytes()
        flag = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 1:
            try:
                check(e.lib.icmslam_p2p_import(e._h, self.rank, self.world, raw, len(raw)), e._h)
            except Exception as ex:      # noqa: BLE001
                ok, why = 0, str(ex)
            flag = torch.tensor([ok], dtype=torch.int32, device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        torch.cuda.synchronize(self.device)
        if int(flag.item()) != 1:
            # back to collectives on every rank (a rank that did import switches its peer tables off again)
            own = raw[self.rank * nbytes:(self.rank + 1) * nbytes]
            try:
                e.lib.icmslam_p2p_import(e._h, 0, 1, own, len(own))
            except Exception:            # noqa: BLE001
                pass
            self.exchange = "nccl"
            self.p2p_fallback_reason = why or "another rank could not open the peer buffers"
            return
        dist.barrier(group=self.group)         # every window is mapped everywhere before the first flag is written
        self._p2p_on = True

    def sweep(self, n_sweeps: int = 1, use_graph: bool = True):
        """n_sweeps sweeps of the whole trajectory (collective: every rank calls it).  In steady state two consecutive
        sweeps -- kernels of this library AND the NCCL collectives between them -- replay as one CUDA graph (two, because
        the pose and map buffers ping-pong)."""
        import torch
        self._prepare()
        self._last_map = None      # (the device map moves on: only a map fetched AFTER these sweeps continues the chain)
        caller = torch.cuda.current_stream(self.device)
        self._stream.wait_stream(caller)
        if self._p2p_on:      # the library exchanges by itself: one call, its own CUDA graph per sweep
            n0 = self.engine.launch_count()
            self.engine.iterate(None, self.x0, int(n_sweeps))
            self._launches += self.engine.launch_count() - n0
            self._launches_per_sweep = (self.engine.launch_count() - n0) // max(int(n_sweeps), 1)
            self._steady += int(n_sweeps)
            caller.wait_stream(self._stream)
            return
        with torch.cuda.stream(self._stream):
            done = 0
            while done < n_sweeps:
                left = n_sweeps - done
                if use_graph and left >= 2 and self._steady >= 2:
                    g = self._graphs.get(self._parity)
                    if g is None:            # one graph per ping-pong parity of the pose / map buffers
                        self._stream.synchronize()
                        g = torch.cuda.CUDAGraph()
                        side = torch.cuda.Stream(device=self.device, priority=-1)
                        self.engine.set_stream(side.cuda_stream)       # (before the capture starts: set_stream synchronises)
                        with torch.cuda.graph(g, stream=side):
                            self._sweep_once()
                            self._sweep_once()
                        self.engine.set_stream(self._stream.cuda_stream)
                        self._graphs[self._parity] = g                 # (capture records the work without running it)
                    g.replay()
                    self._launches += 2 * self._launches_per_sweep
                    done += 2
                    self._steady += 2
                else:
                    n0 = self.engine.launch_count()
                    self._sweep_once()
                    self._launches_per_sweep = self.engine.launch_count() - n0
                    self._launches += self._launches_per_sweep
                    self._steady += 1
                    self._parity ^= 1
                    done += 1
        caller.wait_stream(self._stream)

    @property
    def _graph(self):
        return next(iter(self._graphs.values()), None)

    def launch_count(self):
        """Kernels of the library enqueued by sweep() (replayed graphs included)."""
        return self._launches

    # -- results --------------------------------------------------------------------------------------------------
    def owned_poses(self, out_full=None):
        """Owned columns of the current poses; with out_full (3 x T host array) they are written in place there."""
        if out_full is not None:
            g_lo, g_hi = self.segments[self.rank]
            self.engine.get_poses(out=out_full[:, g_lo - self.t_lo:g_lo - self.t_lo + (self.c_hi - self.c_lo)])
            return out_full[:, g_lo:g_hi]
        return self.engine.get_poses()[:, self.t_lo:self.t_hi]

    def gather_poses(self):
        """Full 3 x T trajectory on every rank (host)."""
        import torch
        import torch.distributed as dist
        mine = self.owned_poses()
        if self.world == 1:
            return mine
        lens = [b - a for a, b in self.segments]
        m = max(lens)
        buf = torch.zeros((3, m), dtype=torch.float64)
        buf[:, : mine.shape[1]] = torch.from_numpy(np.ascontiguousarray(mine))
        dev = "cuda:%d" % self.device if dist.get_backend(self.group) == "nccl" else "cpu"
        buf = buf.to(dev)
        out = [torch.empty_like(buf) for _ in range(self.world)]
        dist.all_gather(out, buf, group=self.group)
        return np.concatenate([o.cpu().numpy()[:, :n] for o, n in zip(out, lens)], axis=1)

    def gather_ragged_int32(self, mine):
        """Concatenation over the ranks (in rank order) of one int32 vector per rank (host)."""
        import torch
        import torch.distributed as dist
        if self.world == 1:
            return np.asarray(mine, dtype=np.int32)
        dev = "cuda:%d" % self.device if dist.get_backend(self.group) == "nccl" else "cpu"
        n = torch.tensor([int(mine.shape[0])], dtype=torch.int64, device=dev)
        ns = [torch.zeros_like(n) for _ in range(self.world)]
        dist.all_gather(ns, n, group=self.group)
        lens = [int(v.item()) for v in ns]
        buf = torch.zeros(max(lens), dtype=torch.int32, device=dev)
        buf[: mine.shape[0]] = torch.from_numpy(np.ascontiguousarray(mine, dtype=np.int32)).to(dev)
        out = [torch.empty_like(buf) for _ in range(self.world)]
        dist.all_gather(out, buf, group=self.group)
        return np.concatenate([o.cpu().numpy()[:k] for o, k in zip(out, lens)])

    def get_map(self):
        m = self.engine.get_map()
        self._last_map = m.copy()
        return m

    def close(self):
        """Collective when the solver created its own halo group.  Captured graphs hold NCCL work of both communicators: they are
        dropped before a communicator goes (destroy_process_group otherwise waits forever on them)."""
        import torch
        self._graphs = {}
        if torch.cuda.is_available():
            torch.cuda.synchronize(self.device)
        if getattr(self, "_own_halo_group", False):
            import torch.distributed as dist
            dist.destroy_process_group(self.halo_group)
            self.halo_group, self._own_halo_group = None, False
        self.engine.close()


# ---- bench arm for N > 1 (called by bench.py under torchrun) -----------------------------------------------------
def bench(args, rank, world, local_rank, WORKLOADS, SEED, METRIC, sweep_bytes, peaks, ClockSampler, make_data, config_for, result_hash,
          runs_bytes, dump_outputs):
    import json
    import time

    import torch
    import torch.distributed as dist

    import os
    os.environ.setdefault("NCCL_DEBUG", "WARN")      # (NCCL's version banner goes to stdout: rank 0 must print ONE JSON line)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    name = args.workload
    L_true, T, desc = WORKLOADS[name]
    d = make_data(name)
    cfg = config_for(L_true, name)
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sol = SegmentedSolver(cfg, rank, world, device=local_rank)
    n_local = sol.load(d["observations"], d["odometry"], d["velocities"], precondition=True)
    sol.set_map(d["map_init"])
    sol.set_poses(d["x_init"])
    nt = torch.tensor([n_local, sol.t_hi - sol.t_lo], dtype=torch.int64, device=dev)
    dist.all_reduce(nt)
    sampler = ClockSampler(local_rank)     # (NVML polling thread, started before the warm-up: nothing is forked next to the timed region)
    sampler.start()
    for _ in range(args.warmup):
        sol.sweep()
    # two more untimed sweeps through the graph path: the two-sweep CUDA graph (kernels + NCCL) is captured and instantiated
    # HERE, not inside the timed region (capture costs tens of milliseconds of host time with the GPUs idle)
    sol.sweep(2)
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    lc0 = sol.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.mark_timed(0)
    ev0.record(stream)
    sol.sweep(args.steps)
    ev1.record(stream)
    torch.cuda.synchronize()
    sampler.mark_timed(1)
    dist.barrier()
    torch.cuda.synchronize()
    ms_t = torch.tensor([ev0.elapsed_time(ev1) / args.steps], dtype=torch.float64, device=dev)
    dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)           # device time, max over ranks
    ms = float(ms_t.item())
    launches = (sol.launch_count() - lc0) // max(args.steps, 1)
    # result hash: poses (gathered), map, labels of the owned scans (gathered) -- identical for any number of segments
    x_all = sol.gather_poses()
    offs = sol.engine.get_extraction()["off"]
    c_own = np.ascontiguousarray(sol.engine.associations()[offs[sol.t_lo]:offs[sol.t_hi]])
    c_all = sol.gather_ragged_int32(c_own)
    m_all = sol.get_map()
    sha = result_hash(x_all, m_all, c_all)
    t_load = time.perf_counter()          # the same load, untimed, for the clock sampler (a fixed number of sweeps: collective)
    sol.sweep(600)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    # run kernel time on this rank (separate short loop: reading the events synchronises)
    kt = []
    for _ in range(5):
        kt.append(sol.timed_sweep()[0])
    stages = sol.stage_times(6)
    # the same job with the exchange through NCCL collectives (a second solver): what the peer-memory kernels replace
    nccl_arm = None
    if sol.exchange == "p2p" and os.environ.get("ICMSLAM_BENCH_NCCL_ARM"):      # (opt-in: a second solver doubles the run's set-up time)
        sol2 = SegmentedSolver(cfg, rank, world, device=local_rank, exchange="nccl")
        sol2.load(d["observations"], d["odometry"], d["velocities"], precondition=True)
        sol2.set_map(d["map_init"])
        sol2.set_poses(d["x_init"])
        for _ in range(max(args.warmup, 3)):
            sol2.sweep()
        sol2.sweep(2)
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        sol2.sweep(args.steps)
        e1.record(stream)
        torch.cuda.synchronize()
        ms2 = torch.tensor([e0.elapsed_time(e1) / args.steps], dtype=torch.float64, device=dev)
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
        x2 = sol2.gather_poses()
        same = bool(np.array_equal(x2, x_all) and np.array_equal(sol2.get_map(), m_all))
        st2 = sol2.stage_times(6)
        nccl_arm = {"ms_per_step": float(ms2.item()), "stages_ms_rank0_eager": st2, "same_result": same}
        sol2.close()
    k_ms = torch.tensor([float(np.mean(kt))], dtype=torch.float64, device=dev)
    dist.all_reduce(k_ms, op=dist.ReduceOp.MAX)
    # end to end: host buffers in, host buffers out, every step
    x_host = torch.from_numpy(d["x_init"].copy()).pin_memory().numpy()
    mapa = d["map_init"].copy()
    e2e_steps = max(3, min(args.steps, 10))
    h2d = d2h = 0
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        uploaded = sol.set_map(mapa)
        sol.set_poses(x_host)
        h2d += (mapa.nbytes if uploaded else 0) + 24 * (sol.c_hi - sol.c_lo)
        sol.sweep()
        own = sol.owned_poses(out_full=x_host)      # D2H straight into the caller's 3 x T array
        mapa = sol.get_map()
        d2h += own.nbytes + mapa.nbytes
    torch.cuda.synchronize()
    dist.barrier()
    e2e_s = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device=dev)
    dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    bytes_t = torch.tensor([h2d // e2e_steps, d2h // e2e_steps], dtype=torch.int64, device=dev)
    dist.all_reduce(bytes_t)
    L_now = sol.engine.landmarks_actuales
    if rank == 0:
        n_tot, t_tot = int(nt[0].item()), int(nt[1].item())
        B_sweep = sweep_bytes(T, n_tot, L_true)
        peak, peak_src = peaks()
        # the dominant kernel's share of the sweep on one rank: its segment's bytes over its time
        Tseg = sol.t_hi - sol.t_lo
        seg_bytes = runs_bytes(Tseg, n_local, L_true)     # the run kernels' own share of this segment
        achieved = seg_bytes / (float(k_ms.item()) * 1e-3) / 1e9
        sweep_achieved = B_sweep / (ms * 1e-3) / 1e9
        out = {
            "metric": METRIC, "value": 1000.0 / ms, "unit": "sweeps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": desc, "T": T, "L_true": L_true, "n_obs": n_tot, "landmarks_after": int(L_now), "beams": 181,
                       "seed": SEED, "mode": "redblack/newton/prev",
                       "partition": "%d contiguous time segments (2+1 halo poses each), per sweep: far counts and halo poses between the ranks + "
                                    "sum-reduction of one block of 2.5 words per landmark slot (%d slots: int64 sums / fp64 new-label means sharing words, int32 counts); "
                                    "exchange by %s" % (world, L_true * 2, "the library's kernels over peer memory (NVLink loads/stores, csrc/p2p.cuh)" if sol.exchange == "p2p" else "NCCL collectives"),
                       "segments": [list(s) for s in sol.segments], "untimed_graph_capture_sweeps": 2,
                       "l2": "inputs larger than L2 (observations %.0f MB per rank vs 126 MB L2)" % (16 * n_tot / world / 1e6)},
            "clocks": clocks,
            "e2e": {"value": 1.0 / float(e2e_s.item()), "unit": "sweeps/s", "h2d_bytes_per_step": int(bytes_t[0].item()),
                    "d2h_bytes_per_step": int(bytes_t[1].item()), "steps": e2e_steps,
                    "call": "SegmentedSolver.set_map/set_poses/sweep/owned_poses/get_map with host numpy buffers on every rank"},
            "gpu_launches": int(launches) * args.steps * world, "gpu_launches_per_step": int(launches),
            "result_sha256": sha, "stages_ms_rank0_eager": stages, "exchange": sol.exchange, "nccl_exchange_arm": nccl_arm,
            "roofline": {"bound": "hbm", "kernel": "k_runs + k_assoc_tiles (rank 0's segment)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": None, "peak_source": peak_src, "kernel_ms": float(k_ms.item()),
                         "algorithmic_bytes": int(seg_bytes),
                         "sweep": {"algorithmic_bytes": int(B_sweep), "achieved": sweep_achieved, "frac": sweep_achieved / (peak * world),
                                   "note": "whole job: all segments' bytes over the max-over-ranks sweep time, vs %d x the HBM peak" % world}},
            "cpu_baseline": None,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, poses=x_all, map=m_all, associations=c_all)
        print(json.dumps(out), flush=True)
    dist.barrier()
    sol.close()
    # (the line is out and every rank is past the barrier: a communicator teardown that stalls must not hold the job)
    import threading
    guard = threading.Timer(30.0, lambda: os._exit(0))
    guard.daemon = True
    guard.start()
    dist.destroy_process_group()
