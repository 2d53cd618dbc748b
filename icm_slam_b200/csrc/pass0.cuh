// pass0.cuh -- the causal initialisation pass ("iteracion ICM 0": ICM_ROS.inicializar_online /
// inicializar_online_process, sensors.py:51-123; legacy ICM_method.inicializar, ICM_SLAM_old.py:266-333)
// replayed on the loaded log.
//
// It is sequential by construction: scan t is associated against the map built from scans < t, which
// in turn was placed with pose t-1.  One block walks the time steps; inside a step the threads share
// the per-beam work (projection, nearest landmark of the map under construction, running means,
// ICM_SLAM.py:167-194) and ONE thread runs the reference's Nelder-Mead on fun_x (sensors.py:258-282)
// operation for operation, so the poses match the reference to 1e-6 m / 1e-8 rad.  Step 0 (Branch A of
// Mapa.actualizar, scipy's fcluster) runs on the host (fcluster.h) before the kernel.
// The walk can stop and resume: one launch takes the columns [t_lo, t_hi) and carries the last pose and landmarks_actuales
// in device memory (Pass0Carry) to the next launch, beside the map under construction and its counts, so that columns appended
// to a loaded log are walked as they arrive (icmslam_pass0_advance).
// Not a hot path: it runs once per column and is not part of the sweeps/s metric.
#pragma once
#include "common.cuh"
#include "assoc.cuh"
#include "pose.cuh"

// what the walk carries from one launch to the next: the pose of the last column walked, landmarks_actuales, columns walked
struct Pass0Carry { double x[3]; int lact; int t; };

struct Pass0Params {
    int t_lo, t_hi, Lcap;            // the columns this launch walks (t_lo >= 1)
    const int* off;
    const double *bx, *by, *d; const int* beam; const double* ang;
    const double* odo; int64_t ldo;
    const double* u; int64_t ldu;
    DevCfg cfg;
    int first;                       // t_lo == 1 after step 0: the carry starts from x0 / lact0 and x[:,0] = x0
    double x0[3];
    int lact0;                       // landmarks after scan 0
    Pass0Carry* carry;               // in (unless first) and out
    double* x; int64_t ldx;          // 3 x T poses (out: columns [t_lo, t_hi))
    double* y;                       // 2 x Lcap map under construction (in / out; after step 0: clusters of scan 0)
    double* cant;                    // Lcap observation counts (in / out; after step 0: cluster sizes)
    int* c;                          // labels per observation (out; scan 0 filled by the host)
    double *seen_x, *seen_y;         // per observation: its landmark's running mean after the scan
    DevState* st;
    unsigned long long* nev;         // energy evaluations (statistics)
};

// world coordinates of one scan's kept beams (tras_rot_z)
__global__ void k_project_scan(const int* __restrict__ off, int t, const double* __restrict__ bx, const double* __restrict__ by,
                               double px, double py, double th, double* __restrict__ wx, double* __restrict__ wy)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int o = off[t], n = off[t + 1] - o;
    if (i >= n) return;
    const Rot r = make_rot(th);
    project(r, px, py, bx[o + i], by[o + i], wx[i], wy[i]);
}

__global__ void __launch_bounds__(256)
k_pass0(const Pass0Params p)
{
    extern __shared__ double p0_smem[];
    const int tid = threadIdx.x, nth = blockDim.x;
    __shared__ double xt[3], xtc[3];
    __shared__ int s_lact, s_abort, s_nfar;
    const int cap = p.Lcap;
    double* wx = p0_smem;                    // world coordinates of the scan's beams
    double* wy = wx + 1024;
    int* cl = reinterpret_cast<int*>(wy + 1024);
    double* yx = p.y;
    double* yy = p.y + cap;
    if (tid == 0) {
        const double* x_last = p.first ? p.x0 : p.carry->x;
        xt[0] = x_last[0]; xt[1] = x_last[1]; xt[2] = x_last[2];
        s_lact = p.first ? p.lact0 : p.carry->lact;
        s_abort = 0;
    }
    if (p.first && tid < 3) p.x[tid * p.ldx] = p.x0[tid];
    __syncthreads();
    ObsArrays O;
    O.bx = p.bx; O.by = p.by; O.d = p.d; O.beam = p.beam; O.ang = p.ang;
    SeenSrc S;
    S.view = ICMSLAM_VIEW_RUNNING; S.c = p.c; S.seen_x = p.seen_x; S.seen_y = p.seen_y;
    S.raw_x = nullptr; S.raw_y = nullptr; S.min_x = nullptr; S.min_y = nullptr; S.lsearch_ptr = nullptr;
    int t = p.t_lo;
    for (; t < p.t_hi; ++t) {
        if (tid == 0) {
            const double ua[2] = {p.u[t - 1], p.u[p.ldu + t - 1]};
            g_step(xt, ua[0], ua[1], p.cfg.dt, xtc);               // sensors.py:111
            s_nfar = 0;
        }
        __syncthreads();
        const int o = p.off[t], n = p.off[t + 1] - o;
        if (n == 0) {                                              // sensors.py:114-117
            if (tid < 3) { xt[tid] = xtc[tid]; p.x[tid * p.ldx + t] = xtc[tid]; }
            __syncthreads();
            continue;
        }
        const int lact = s_lact;
        {   // tras_rot_z with the predicted pose, then cdist + argmin against the map under construction (:119-120)
            const Rot r = make_rot(xtc[2]);
            for (int i = tid; i < n; i += nth) {
                double ax, ay;
                project(r, xtc[0], xtc[1], p.bx[o + i], p.by[o + i], ax, ay);
                wx[i] = ax; wy[i] = ay;
                double best = INFINITY;
                int arg = 0;
                for (int l = 0; l < lact; ++l) {
                    const double dd = dist_rn(yx[l] - ax, yy[l] - ay);
                    if (dd < best) { best = dd; arg = l; }
                }
                if (best > p.cfg.dist_thr) { cl[i] = -1; atomicAdd(&s_nfar, 1); } else cl[i] = arg;
            }
        }
        __syncthreads();
        if (s_nfar > 0) {                                          // ICM_SLAM.py:174-182: one new label for the scan
            if (lact >= cap) { if (tid == 0) { s_abort = 1; p.st->status = ST_LABEL_CAP; } }
            else {
                for (int i = tid; i < n; i += nth) if (cl[i] < 0) cl[i] = lact;
                if (tid == 0) s_lact = lact + 1;
            }
        }
        __syncthreads();
        if (s_abort) break;
        // recursive running mean of every label seen in this scan (:184-194); the first beam of a label owns it
        for (int i = tid; i < n; i += nth) {
            const int lbl = cl[i];
            bool first = true;
            for (int j = 0; j < i; ++j) if (cl[j] == lbl) { first = false; break; }
            if (!first) continue;
            int k = 0;
            double sx = 0.0, sy = 0.0;
            for (int j = i; j < n; ++j)
                if (cl[j] == lbl) { sx = add_rn(sx, wx[j]); sy = add_rn(sy, wy[j]); ++k; }
            const double ni = p.cant[lbl], tot = ni + (double)k;
            yx[lbl] = add_rn(__ddiv_rn(sx, tot), __ddiv_rn(mul_rn(yx[lbl], ni), tot));
            yy[lbl] = add_rn(__ddiv_rn(sy, tot), __ddiv_rn(mul_rn(yy[lbl], ni), tot));
            p.cant[lbl] = tot;
        }
        __syncthreads();
        for (int i = tid; i < n; i += nth) {                       // y[:, c].T: what the pose is fitted against (:122)
            p.c[o + i] = cl[i];
            p.seen_x[o + i] = yx[cl[i]];
            p.seen_y[o + i] = yy[cl[i]];
        }
        __syncthreads();
        if (tid == 0) {                                            // minimizar_x: Nelder-Mead on fun_x (sensors.py:258-282)
            PoseProblem P;
            P.has_next = 0; P.o = o; P.n = n;
            for (int j = 0; j < 3; ++j) {
                P.a[j] = xt[j]; P.b[j] = 0.0;
                P.o0[j] = p.odo[j * p.ldo + t - 1]; P.o1[j] = p.odo[j * p.ldo + t]; P.o2[j] = 0.0;
            }
            P.ua[0] = p.u[t - 1]; P.ua[1] = p.u[p.ldu + t - 1];
            P.uc[0] = P.uc[1] = 0.0;
            double res[3];
            const int ne = nelder_mead(p.cfg, P, O, S, xtc, res);
            if (p.nev) *p.nev += (unsigned long long)ne;
            for (int j = 0; j < 3; ++j) { xt[j] = res[j]; p.x[j * p.ldx + t] = res[j]; }
        }
        __syncthreads();
    }
    if (tid == 0) {      // (on the label cap t is the column that could not be walked)
        p.carry->x[0] = xt[0]; p.carry->x[1] = xt[1]; p.carry->x[2] = xt[2];
        p.carry->lact = s_lact; p.carry->t = t;
        p.st->lact = s_lact; p.st->raw_l = s_lact;
    }
}

// the walk's construction becomes the handle's raw map (icmslam_get_raw_map): counts, width and landmarks_actuales (the map
// itself is copied beside this launch); the status word is cleared as a fresh pass 0 clears it
__global__ void k_walk_publish(const Pass0Carry* __restrict__ carry, const double* __restrict__ cant, int Lcap, int* __restrict__ rawcnt,
                               DevState* st)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l < Lcap) rawcnt[l] = (int)cant[l];
    if (l == 0) { st->lact = carry->lact; st->raw_l = carry->lact; st->status = 0; }
}
