// assoc.cuh -- data association, label assignment, landmark statistics
// (Mapa.actualizar Branch B, ICM_SLAM.py:167-194, for all scans of a sweep at once).
#pragma once
#include "common.cuh"
#include "fastgrid.cuh"

// Device-resident sweep state (no host round trip inside a sweep).
struct DevState {
    int lact;        // Mapa.landmarks_actuales
    int lsearch;     // min(lact, L_in): columns of map_in that are searched (ICM_SLAM.py:169)
    int lact0;       // lact at sweep start = first new label
    int raw_l;       // lact after association (before filtrar)
    int status;      // ST_*
    int n_far_scans;
    int kept;        // landmarks surviving cota
    int new_l;       // landmarks after filtrar
    int n_ind;       // landmarks with a neighbour closer than dist_thr
    int dirty_tiles; // record tiles that went through the association kernel this sweep (runs.cuh; filled on request)
    unsigned long long newton_iters;
    unsigned long long solved;
    double cambio[3]; // calc_cambio of the sweep's map against the previous one, accumulated by the fast tail: min, max, sum
    int cambio_unres; // new landmarks whose nearest old landmark the tail could not certify (then cambio[] is not usable)
    int cambio_pad;
};

// ---- association ---------------------------------------------------------------------------
// One warp per scan, lanes over the scan's kept observations.  Projects with the sweep's INPUT
// pose (sensors.py:141,153; each trajectory's first scan with its own x0, TrajLayout), finds the nearest of the first `lsearch` previous-map landmarks
// (cdist + argmin, ICM_SLAM.py:169-171), gates at dist_thr (strict >, :172).  Matched
// observations add into the per-label sums; far ones are marked -1 and counted per scan.
__global__ void __launch_bounds__(256)
k_assoc(int T, const int* __restrict__ off, const double* __restrict__ bx, const double* __restrict__ by,
        const double* __restrict__ x, int64_t ldx, const TrajLayout lay, const FGeom* __restrict__ geom,
        const int* __restrict__ cell_start, const double2* __restrict__ pts, const int* __restrict__ gidx, double thr2_hi,
        int* __restrict__ c, int* __restrict__ nfar, double* __restrict__ sum_x, double* __restrict__ sum_y, int* __restrict__ cnt)
{
    const int lane = threadIdx.x % WARP;
    const int wpb = blockDim.x / WARP;
    FGrid G;
    G.g = *geom; G.cell_start = cell_start; G.pts = pts; G.idx = gidx;
    for (int t = blockIdx.x * wpb + threadIdx.x / WARP; t < T; t += gridDim.x * wpb) {
        int o = off[t], e = off[t + 1];
        int far = 0;
        if (e > o) {
            double px, py, th;
            lay.scan_pose(x, ldx, t, px, py, th);
            Rot r = make_rot(th);
            for (int i = o + lane; i < e; i += WARP) {
                double wx, wy, best;
                project(r, px, py, bx[i], by[i], wx, wy);
                const int bk = fgrid_nearest(G, wx, wy, best);      // (an empty map: no candidate, best = INFINITY)
                if (best > thr2_hi) { c[i] = -1; ++far; }          // sqrt_rn(best) > dist_thr
                else {
                    const int arg = __ldg(gidx + bk);
                    c[i] = arg;
                    atomicAdd(sum_x + arg, wx);
                    atomicAdd(sum_y + arg, wy);
                    atomicAdd(cnt + arg, 1);
                }
            }
            far = warp_sum_i(far);
        }
        if (lane == 0) nfar[t] = far;
    }
}

// flag[t] = scan t has >= 1 far observation (each such scan creates exactly ONE new label,
// ICM_SLAM.py:174-182; SURVEY App. C.2).  Also used to turn counts into flags for cub scans.
__global__ void k_flag_positive(const int* __restrict__ v, int n, int* __restrict__ flag)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = v[i] > 0 ? 1 : 0;
}

// New labels: label(t) = lact0 + (number of earlier scans with a far observation).  One warp per
// scan that has far observations: rewrite c, and own the new label's statistics (no atomics).
__global__ void __launch_bounds__(256)
k_new_labels(int T, const int* __restrict__ off, const double* __restrict__ bx, const double* __restrict__ by,
             const double* __restrict__ x, int64_t ldx, const TrajLayout lay, DevState* st,
             const int* __restrict__ nfar, const int* __restrict__ far_prefix, int Lcap, int* __restrict__ c,
             double* __restrict__ sum_x, double* __restrict__ sum_y, int* __restrict__ cnt)
{
    const int lane = threadIdx.x % WARP;
    const int wpb = blockDim.x / WARP;
    const int lact0 = st->lact0;
    for (int t = blockIdx.x * wpb + threadIdx.x / WARP; t < T; t += gridDim.x * wpb) {
        if (t == T - 1 && lane == 0) {
            int total = far_prefix[t] + (nfar[t] > 0 ? 1 : 0);
            st->n_far_scans = total;
            st->raw_l = lact0 + total;
            if (lact0 + total > Lcap) st->status = ST_LABEL_CAP;   // IndexError at ICM_SLAM.py:191
        }
        if (nfar[t] == 0) continue;
        int label = lact0 + far_prefix[t];
        if (label >= Lcap) continue;
        int o = off[t], e = off[t + 1];
        double px, py, th;
        lay.scan_pose(x, ldx, t, px, py, th);
        Rot r = make_rot(th);
        double sx = 0.0, sy = 0.0;
        for (int i0 = o; i0 < e; i0 += WARP) {       // sequential-in-lane-order sum of the far points
            int i = i0 + lane;
            double wx = 0.0, wy = 0.0;
            bool isfar = false;
            if (i < e && c[i] < 0) {
                project(r, px, py, bx[i], by[i], wx, wy);
                c[i] = label;
                isfar = true;
            }
            unsigned bal = __ballot_sync(FULLMASK, isfar);
            while (bal) {                              // np.sum(obs[c==i], axis=0): in row order
                int src = __ffs(bal) - 1;
                sx += __shfl_sync(FULLMASK, wx, src);
                sy += __shfl_sync(FULLMASK, wy, src);
                bal &= bal - 1;
            }
        }
        if (lane == 0) { sum_x[label] = sx; sum_y[label] = sy; cnt[label] = nfar[t]; }
    }
}

// raw map = per-label mean (the value the recursive running mean of ICM_SLAM.py:191-194 ends at);
// labels never observed keep the zero column of `y` (sensors.py:132).
__global__ void k_means(const DevState* st, const double* __restrict__ sum_x, const double* __restrict__ sum_y,
                        const int* __restrict__ cnt, double* __restrict__ raw_x, double* __restrict__ raw_y, int Lcap)
{
    int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= Lcap) return;
    int k = l < st->raw_l ? cnt[l] : 0;
    raw_x[l] = k > 0 ? sum_x[l] / (double)k : 0.0;
    raw_y[l] = k > 0 ? sum_y[l] / (double)k : 0.0;
}

// ---- running view --------------------------------------------------------------------------
// Reference semantics of what a pose sees (sensors.py:154-156): the recursive running mean of its
// label INCLUDING the current scan.  Observations are sorted by (label, time) (stable radix sort
// of labels; CSR order is time order); one thread per label walks its segment, grouping by scan
// and applying ICM_SLAM.py:191-194 literally.  Also produces the reference-arithmetic raw map.
__global__ void k_running_mean(const DevState* st, const int* __restrict__ seg_start, const int* __restrict__ cnt,
                               const int* __restrict__ sorted_obs, const int* __restrict__ scan_of,
                               const double* __restrict__ bx, const double* __restrict__ by, const double* __restrict__ x,
                               int64_t ldx, const TrajLayout lay, double* __restrict__ seen_x,
                               double* __restrict__ seen_y, double* __restrict__ raw_x, double* __restrict__ raw_y, int Lcap)
{
    int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= Lcap) return;
    if (l >= st->raw_l || cnt[l] == 0) { raw_x[l] = 0.0; raw_y[l] = 0.0; return; }
    int s = seg_start[l], e = s + cnt[l];
    double mx = 0.0, my = 0.0, ni = 0.0;
    int j = s;
    while (j < e) {
        int t = scan_of[sorted_obs[j]];
        double px, py, th;
        lay.scan_pose(x, ldx, t, px, py, th);
        Rot r = make_rot(th);
        double sx = 0.0, sy = 0.0;
        int k = 0, j2 = j;
        while (j2 < e && scan_of[sorted_obs[j2]] == t) {
            int i = sorted_obs[j2];
            double wx, wy;
            project(r, px, py, bx[i], by[i], wx, wy);
            sx = add_rn(sx, wx); sy = add_rn(sy, wy);
            ++k; ++j2;
        }
        double tot = ni + (double)k;
        mx = add_rn(__ddiv_rn(sx, tot), __ddiv_rn(mul_rn(mx, ni), tot));
        my = add_rn(__ddiv_rn(sy, tot), __ddiv_rn(mul_rn(my, ni), tot));
        ni = tot;
        for (int q = j; q < j2; ++q) { seen_x[sorted_obs[q]] = mx; seen_y[sorted_obs[q]] = my; }
        j = j2;
    }
    raw_x[l] = mx; raw_y[l] = my;
}

// labels -> sort keys (far observations already relabelled)
__global__ void k_iota(int n, int* __restrict__ v)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = i;
}
