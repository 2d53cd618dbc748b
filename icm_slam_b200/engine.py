"""Thin object wrapper over the C ABI: one Engine == one icmslam_handle == one GPU.

Accepts numpy arrays (host buffers, copied inside the library) or torch CUDA tensors (device
buffers used in place).  All numerics happen in libicmslam.so; this file only marshals pointers.
"""
from __future__ import annotations

import os
import ctypes as C

import numpy as np

from . import _lib
from ._lib import HOST, DEVICE, IcmConfig, SweepOpts, check


def _diag(v, n):
    v = np.asarray(v, dtype=np.float64)
    return np.diag(v).copy() if v.ndim == 2 else v.reshape(n)


def make_c_config(config, device: int = 0, L: int | None = None) -> IcmConfig:
    q = _diag(config.Q, 2)
    r = _diag(config.R, 3)
    return IcmConfig(float(config.deltat), q[0], q[1], r[0], r[1], r[2], float(config.cte_odom), float(config.cota),
                     float(config.dist_thr), float(config.rango_laser_max), float(config.radio),
                     int(L if L is not None else config.L), int(device))


def _is_torch(a):
    return type(a).__module__.startswith("torch")


def _ptr(a):
    """(pointer, memspace) of a numpy array or a torch tensor."""
    if a is None:
        return None, HOST
    if _is_torch(a):
        return C.c_void_p(a.data_ptr()), (DEVICE if a.is_cuda else HOST)
    return C.c_void_p(a.ctypes.data), HOST


def _rows(a, nrows):
    """Checks a 2-D row-major fp64 array and returns its leading dimension in elements."""
    if _is_torch(a):
        import torch
        assert a.dtype == torch.float64 and a.dim() == 2 and a.shape[0] == nrows and a.stride(1) == 1, "need fp64 (%d, n) row-major" % nrows
        return int(a.stride(0)) if a.shape[0] > 1 else int(a.shape[1])
    assert a.dtype == np.float64 and a.ndim == 2 and a.shape[0] == nrows and a.strides[1] == 8, "need fp64 (%d, n) row-major" % nrows
    return int(a.strides[0] // 8) if a.shape[0] > 1 else int(a.shape[1])


class Engine:
    def __init__(self, config, device: int = 0, L: int | None = None):
        self.lib = _lib.lib()
        self.ccfg = make_c_config(config, device, L)
        self.L = int(self.ccfg.L)
        self.device = device
        self._h = C.c_void_p()
        st = self.lib.icmslam_create(C.byref(self.ccfg), C.byref(self._h))
        if st != 0:
            raise _lib.IcmSlamError(st, "icmslam_create failed (is a CUDA device visible? there is no CPU fallback)")
        self.T = 0
        self.B = 0
        self.n = 0

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.icmslam_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- stream ---------------------------------------------------------------------------------
    def set_stream(self, cuda_stream_ptr: int | None):
        check(self.lib.icmslam_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)), self._h)

    def synchronize(self):
        check(self.lib.icmslam_synchronize(self._h), self._h)

    # -- data -----------------------------------------------------------------------------------
    def load(self, scans, odometry, controls, precondition: bool = False):
        """scans B x T (already pre-conditioned unless precondition=True), odometry 3 x T, controls 2 x T."""
        if not _is_torch(scans):
            scans = np.ascontiguousarray(scans, dtype=np.float64)
            odometry = np.ascontiguousarray(odometry, dtype=np.float64)
            controls = np.ascontiguousarray(controls, dtype=np.float64)
        B, T = int(scans.shape[0]), int(scans.shape[1])
        ang = np.arange(B) * np.pi / 180.0            # exactly the reference's expression (ICM_SLAM.py:44)
        cb, sb = np.cos(ang), np.sin(ang)
        ps, ms = _ptr(scans)
        po, _ = _ptr(odometry)
        pu, _ = _ptr(controls)
        check(self.lib.icmslam_load(self._h, ps, B, T, _rows(scans, B), po, _rows(odometry, 3), pu, _rows(controls, 2),
                                    C.c_void_p(cb.ctypes.data), C.c_void_p(sb.ctypes.data), int(bool(precondition)), ms), self._h)
        self.B, self.T = B, T
        self.n = 0

    def extract(self):
        check(self.lib.icmslam_extract(self._h), self._h)
        n = C.c_int64()
        ne = C.c_int32()
        mx = C.c_int32()
        check(self.lib.icmslam_extraction_size(self._h, C.byref(n), C.byref(ne), C.byref(mx)), self._h)
        self.n, self.n_empty, self.max_per_scan = int(n.value), int(ne.value), int(mx.value)
        return self.n

    def get_extraction(self):
        off = np.empty(self.T + 1, np.int32)
        beam = np.empty(self.n, np.int32)
        d = np.empty(self.n)
        bx = np.empty(self.n)
        by = np.empty(self.n)
        check(self.lib.icmslam_get_extraction(self._h, _ptr(off)[0], _ptr(beam)[0], _ptr(d)[0], _ptr(bx)[0], _ptr(by)[0], HOST), self._h)
        return dict(off=off, beam=beam, d=d, bx=bx, by=by)

    # -- Mapa state -----------------------------------------------------------------------------
    @property
    def landmarks_actuales(self) -> int:
        v = C.c_int32()
        check(self.lib.icmslam_get_landmarks_actuales(self._h, C.byref(v)), self._h)
        return int(v.value)

    @landmarks_actuales.setter
    def landmarks_actuales(self, v: int):
        check(self.lib.icmslam_set_landmarks_actuales(self._h, int(v)), self._h)

    def counts(self, n=None):
        n = self.L if n is None else int(n)
        out = np.zeros(n)
        if n:
            check(self.lib.icmslam_get_counts(self._h, _ptr(out)[0], n, HOST), self._h)
        return out

    def set_batch(self, traj_T, x0s):
        """The loaded columns are K independent trajectories of traj_T columns each (x0s: 3 x K pinned first poses); traj_T = 0
        switches back to one trajectory."""
        if not traj_T:
            check(self.lib.icmslam_set_batch(self._h, 0, None, 0, 0), self._h)
            self.batch_K = 0
            return
        x0s = np.ascontiguousarray(x0s, dtype=np.float64)
        check(self.lib.icmslam_set_batch(self._h, int(traj_T), _ptr(x0s)[0], _rows(x0s, 3), int(x0s.shape[1])), self._h)
        self.batch_K = int(x0s.shape[1])

    def set_counts(self, counts=None):
        """cant_obs_i <- counts (rest zero); None: Mapa.clear_obs."""
        c = np.zeros(0) if counts is None else np.ascontiguousarray(counts, dtype=np.float64)
        n = min(int(c.shape[0]), self.L)
        check(self.lib.icmslam_set_counts(self._h, _ptr(c)[0] if n else None, n, HOST), self._h)

    # -- the sweep ------------------------------------------------------------------------------
    def sweep(self, map_in, x, x0, map_out=None, schedule="redblack", solver="newton", view="prev", newton_tol=0.0,
              newton_maxit=0, fused=True, want_L=True, stats=False):
        """One iterations_process_offline.  x (3 x T) is updated in place.  Returns (status, L_out);
        with map_out=None a fresh (2, L_out) array / tensor view is returned as third element."""
        opts = SweepOpts(_lib.SCHED[schedule], _lib.SOLVER[solver], _lib.VIEW[view], int(newton_maxit), float(newton_tol),
                         int(bool(fused)), 1 if stats else 0)
        px, ms = _ptr(x)
        ldx = _rows(x, 3)
        L_in = int(map_in.shape[1])
        pm, msm = _ptr(map_in)
        assert L_in == 0 or msm == ms, "map_in and x must live in the same memory space"
        ldm = _rows(map_in, 2) if L_in else 1
        x0 = np.ascontiguousarray(np.asarray(x0, dtype=np.float64).reshape(3))
        own_out = map_out is None
        if own_out:
            if ms == DEVICE:
                import torch
                map_out = torch.zeros((2, self.L), dtype=torch.float64, device=x.device)
            else:
                map_out = np.empty((2, self.L))       # (only the first L_out columns are written and returned)
        po, mso = _ptr(map_out)
        assert mso == ms
        cap = int(map_out.shape[1])
        ldo = _rows(map_out, 2)
        Lout = C.c_int32(-1)
        st = self.lib.icmslam_sweep(self._h, pm, L_in, ldm, px, ldx, C.c_void_p(x0.ctypes.data), po, cap, ldo,
                                    C.byref(Lout) if want_L else None, C.byref(opts), ms)
        check(st, self._h)
        if own_out:
            return st, int(Lout.value), (map_out[:, : int(Lout.value)] if want_L else map_out)
        return st, int(Lout.value)

    # -- the driver loop with the map resident on the device (sensors.py:302-315) ------------------
    def set_map(self, mapa):
        """mapa_viejo (2 x L_map) -> device; landmarks_actuales = L_map."""
        if not _is_torch(mapa):
            mapa = np.ascontiguousarray(mapa, dtype=np.float64)
        Lm = int(mapa.shape[1])
        pm, ms = _ptr(mapa)
        check(self.lib.icmslam_set_map(self._h, pm, Lm, _rows(mapa, 2) if Lm else 1, ms), self._h)

    def get_map(self):
        out = np.zeros((2, self.L))
        Lm = C.c_int32()
        check(self.lib.icmslam_get_map(self._h, _ptr(out)[0], self.L, self.L, C.byref(Lm), HOST), self._h)
        return out[:, : Lm.value].copy()

    def iterate(self, x, x0, n_sweeps=1, schedule="redblack", solver="newton", view="prev", newton_tol=0.0, newton_maxit=0,
                fused=True, timing=False, stats=False):
        """n_sweeps x iterations_process_offline on the device-resident map; x (3 x T, numpy or torch CUDA) in place,
        or x=None to sweep the poses uploaded with set_poses."""
        opts = SweepOpts(_lib.SCHED[schedule], _lib.SOLVER[solver], _lib.VIEW[view], int(newton_maxit), float(newton_tol),
                         int(bool(fused)), (1 if stats else 0) | (2 if timing else 0))
        px, ms = _ptr(x)
        x0 = np.ascontiguousarray(np.asarray(x0, dtype=np.float64).reshape(3))
        st = self.lib.icmslam_iterate(self._h, px, _rows(x, 3) if x is not None else 0, C.c_void_p(x0.ctypes.data), int(n_sweeps),
                                      C.byref(opts), ms)
        return check(st, self._h)

    def iterate_until(self, x0, max_sweeps, tol_max_change=0.0, schedule="redblack", solver="newton", view="prev", newton_tol=0.0,
                      newton_maxit=0, fused=True):
        """The driver loop with the convergence monitor (sensors.py:302-315): sweeps of the resident poses / map until the
        largest landmark change of a sweep (calc_cambio's maximum) is <= tol_max_change, at most max_sweeps.  Returns
        (sweeps run, cambios (n, 3): min / max / mean per sweep)."""
        opts = SweepOpts(_lib.SCHED[schedule], _lib.SOLVER[solver], _lib.VIEW[view], int(newton_maxit), float(newton_tol),
                         int(bool(fused)), 0)
        x0 = np.ascontiguousarray(np.asarray(x0, dtype=np.float64).reshape(3))
        n = C.c_int32(0)
        cam = np.zeros((3, max(int(max_sweeps), 1)))
        check(self.lib.icmslam_iterate_until(self._h, C.c_void_p(x0.ctypes.data), int(max_sweeps), float(tol_max_change), C.byref(opts),
                                             _ptr(cam)[0], C.byref(n)), self._h)
        return int(n.value), np.ascontiguousarray(cam[:, : n.value].T)

    def batch_iterate_until(self, max_sweeps, tol_max_change, region_pitch, region_cols, newton_tol=0.0, newton_maxit=0):
        """iterate_until for every trajectory of a batch handle (set_batch) on its own: trajectory k stops -- and is frozen on the
        device while the others sweep on -- after its first sweep whose largest landmark change is <= tol_max_change.  A landmark
        belongs to trajectory rint(y / region_pitch) * region_cols + rint(x / region_pitch).  Returns (sweeps the handle ran,
        n_done (K,), cambios (K, max_sweeps, 3): min / max / mean of trajectory k's sweep s for s < n_done[k])."""
        K = int(getattr(self, "batch_K", 0))
        opts = SweepOpts(_lib.SCHED["redblack"], _lib.SOLVER["newton"], _lib.VIEW["prev"], int(newton_maxit), float(newton_tol), 1, 0)
        m = max(int(max_sweeps), 1)
        cam = np.zeros((3, max(K, 1), m))
        n_done = np.zeros(max(K, 1), np.int32)
        n_run = C.c_int32(0)
        check(self.lib.icmslam_batch_iterate_until(self._h, int(max_sweeps), float(tol_max_change), float(region_pitch), int(region_cols),
                                                   C.byref(opts), _ptr(cam)[0], n_done.ctypes.data_as(C.POINTER(C.c_int32)),
                                                   C.byref(n_run)), self._h)
        return int(n_run.value), n_done[:K].copy(), np.ascontiguousarray(cam[:, :K, :].transpose(1, 2, 0))

    def associate(self, mapa, mapa_referencia, obs):
        """Mapa.actualizar for one scan (ICM_SLAM.py:128-201): `mapa` (2 x L, updated in place), `mapa_referencia` (2 x Lref),
        `obs` (n, 2) projected observations.  Returns the labels c (int64, like np.argmin).  landmarks_actuales and
        cant_obs_i live in the handle."""
        assert isinstance(mapa, np.ndarray) and mapa.dtype == np.float64 and mapa.ndim == 2 and mapa.shape[0] == 2 and mapa.strides[1] == 8
        ref = np.ascontiguousarray(mapa_referencia, dtype=np.float64)
        obs = np.asarray(obs, dtype=np.float64)
        n = int(obs.shape[0])
        ox, oy = np.ascontiguousarray(obs[:, 0]), np.ascontiguousarray(obs[:, 1])
        c = np.zeros(n, np.int32)
        Lr = int(ref.shape[1]) if ref.ndim == 2 else 0
        check(self.lib.icmslam_associate(self._h, _ptr(ref)[0] if Lr else None, Lr, _rows(ref, 2) if Lr else 1, _ptr(ox)[0], _ptr(oy)[0], n,
                                         _ptr(mapa)[0], min(int(mapa.shape[1]), self.L), _rows(mapa, 2), _ptr(c)[0], HOST), self._h)
        return c.astype(np.int64)

    POSE_OPS = {"energy": 0, "min_nm": 1, "min_newton": 2, "g": 3, "h": 4}

    def pose_eval(self, op, z=None, seen=None, x=None, x_ant=None, x_pos=None, u_ant=None, u_act=None, odo=None, newton_tol=0.0,
                  newton_maxit=0, model=0):
        """The reference's user-configurable model functions for one pose on the device (sensors.py:170-282; icmslam_pose_eval):
        op 'g' -> g(x_ant, u_ant); 'h' -> h(x, z) against `seen`; 'energy' -> fun_xn(x) (fun_x(x) when x_pos is None);
        'min_nm' / 'min_newton' -> the minimiser from the reference's start point.  z: (n, 2) [range, beam angle]; seen: (n, 2) matched
        landmark of each observation; odo: 3 x 3 (columns t-1, t, t+1) or 3 x 2.  Returns (pose (3,), energy, evaluations)."""
        f64 = lambda a, shape=None: None if a is None else np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(shape) if shape else np.asarray(a, dtype=np.float64))
        z = np.zeros((0, 2)) if z is None else np.asarray(z, dtype=np.float64).reshape(-1, 2)
        seen = np.zeros((0, 2)) if seen is None else np.asarray(seen, dtype=np.float64).reshape(-1, 2)
        n = int(z.shape[0])
        if seen.shape[0] != n:
            raise ValueError("one matched landmark per observation")
        zd, za = np.ascontiguousarray(z[:, 0]), np.ascontiguousarray(z[:, 1])
        sx, sy = np.ascontiguousarray(seen[:, 0]), np.ascontiguousarray(seen[:, 1])
        xx = np.zeros(3) if x is None else np.array(np.asarray(x, dtype=np.float64).reshape(3), copy=True)
        xa, xb, ua, uc = f64(x_ant, 3), f64(x_pos, 3), f64(u_ant, 2), f64(u_act, 2)
        od = None if odo is None else np.ascontiguousarray(np.asarray(odo, dtype=np.float64))
        p = lambda a: None if a is None or a.size == 0 else C.c_void_p(a.ctypes.data)
        opts = SweepOpts(_lib.SCHED["redblack"], _lib.SOLVER["newton"], _lib.VIEW["prev"], int(newton_maxit), float(newton_tol), 1, 0)
        f, nev = C.c_double(0.0), C.c_int32(0)
        check(self.lib.icmslam_pose_eval(self._h, int(model), self.POSE_OPS[op], n, p(zd), p(za), p(sx), p(sy), p(xa), p(xb), p(ua), p(uc), p(od),
                                         int(od.shape[1]) if od is not None else 0, C.c_void_p(xx.ctypes.data), C.byref(f), C.byref(nev),
                                         C.byref(opts)), self._h)
        return xx, float(f.value), int(nev.value)

    def set_poses(self, x):
        """ICM.positions (3 x T) -> device; iterate(None, ...) then sweeps them in place on the device."""
        if not _is_torch(x) and not (isinstance(x, np.ndarray) and x.dtype == np.float64 and x.ndim == 2 and x.strides[1] == 8):
            x = np.ascontiguousarray(x, dtype=np.float64)
        px, ms = _ptr(x)
        check(self.lib.icmslam_set_poses(self._h, px, _rows(x, 3), ms), self._h)

    def get_poses(self, out=None):
        if out is None:
            out = np.empty((3, self.T))
        check(self.lib.icmslam_get_poses(self._h, _ptr(out)[0], _rows(out, 3), HOST), self._h)
        return out

    def kernel_ms(self):
        out = np.zeros(2)
        check(self.lib.icmslam_get_kernel_ms(self._h, _ptr(out)[0]), self._h)
        return float(out[0]), float(out[1])

    def launch_count(self) -> int:
        v = C.c_int64()
        check(self.lib.icmslam_get_launch_count(self._h, C.byref(v)), self._h)
        return int(v.value)

    # -- pass 0 -----------------------------------------------------------------------------------------
    def pass0(self, x0):
        """inicializar_online replayed on the loaded log (sensors.py:51-123): returns (positions 3 x T, mapa_viejo 2 x L')."""
        x0 = np.ascontiguousarray(np.asarray(x0, dtype=np.float64).reshape(3))
        x = np.zeros((3, self.T))
        out = np.zeros((2, self.L))
        Lout = C.c_int32()
        st = self.lib.icmslam_pass0(self._h, C.c_void_p(x0.ctypes.data), _ptr(x)[0], self.T, _ptr(out)[0], self.L, self.L, C.byref(Lout), HOST)
        check(st, self._h)
        return x, out[:, : Lout.value].copy()

    def associations(self):
        c = np.empty(self.n, np.int32)
        if self.n:
            check(self.lib.icmslam_get_associations(self._h, _ptr(c)[0], HOST), self._h)
        return c

    def raw_map(self):
        raw = np.zeros((2, self.L))
        cnt = np.zeros(self.L)
        rl = C.c_int32()
        check(self.lib.icmslam_get_raw_map(self._h, _ptr(raw)[0], self.L, self.L, _ptr(cnt)[0], C.byref(rl), HOST), self._h)
        return raw[:, : rl.value].copy(), cnt[: rl.value].copy(), int(rl.value)

    def transfer_bytes(self):
        """(host->device, device->host) bytes copied so far by host-memory sweeps."""
        a, b = C.c_int64(), C.c_int64()
        check(self.lib.icmslam_get_transfer_bytes(self._h, C.byref(a), C.byref(b)), self._h)
        return int(a.value), int(b.value)

    def sweep_stats(self):
        v = (C.c_int64 * 17)()
        check(self.lib.icmslam_get_sweep_stats(self._h, v, 17), self._h)
        keys = ["newton_iters", "n_far_scans", "raw_L", "kept", "new_L", "n_ind", "lsearch", "status", "dirty_tiles", "epoch",
                "n_tiles", "stable_ids", "k_runs_ns", "n_dirty_now", "far_count", "steady_sweeps", "batch_until_fallbacks"]
        return dict(zip(keys, [int(t) for t in v]))

    # -- map utilities --------------------------------------------------------------------------
    def filter_map(self, mapa, counts):
        mapa = np.ascontiguousarray(mapa, dtype=np.float64)
        counts = np.ascontiguousarray(counts, dtype=np.float64)
        L_in = int(counts.shape[0])
        out = np.zeros((2, self.L))
        cout = np.zeros(self.L)
        Lout = C.c_int32()
        check(self.lib.icmslam_filter_map(self._h, _ptr(mapa)[0], _rows(mapa, 2), _ptr(counts)[0], L_in, _ptr(out)[0], self.L, self.L,
                                          _ptr(cout)[0], C.byref(Lout), HOST), self._h)
        return out, cout, int(Lout.value)

    def calc_cambio(self, y, mapa_viejo):
        y = np.ascontiguousarray(y, dtype=np.float64)
        old = np.ascontiguousarray(mapa_viejo, dtype=np.float64)
        out = np.zeros(3)
        check(self.lib.icmslam_calc_cambio(self._h, _ptr(y)[0], int(y.shape[1]), _rows(y, 2), _ptr(old)[0], int(old.shape[1]),
                                           _rows(old, 2), _ptr(out)[0], HOST), self._h)
        return float(out[0]), float(out[1]), float(out[2])

    def filtrar_obs(self, obs, max_dist=10.0, cant_max=15):
        obs = np.ascontiguousarray(obs, dtype=np.float64)
        B, T = obs.shape
        out = np.empty_like(obs)
        check(self.lib.icmslam_filtrar_obs(self._h, _ptr(obs)[0], B, T, T, float(max_dist), int(cant_max), _ptr(out)[0], T, HOST), self._h)
        return out
