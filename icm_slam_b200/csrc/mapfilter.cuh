// mapfilter.cuh -- Mapa.filtrar (ICM_SLAM.py:204-265) and calc_cambio (ICM_SLAM.py:490-495).
//
// filtrar: (1) drop labels observed fewer than `cota` times; (2) every survivor whose nearest
// OTHER survivor is closer than dist_thr is visited in ascending index order and the class of
// that neighbour is renamed to the survivor's class (c[c==c[b[i]]] = c[i]); (3) classes are
// renumbered densely in ascending order; (4) each class becomes the count-weighted mean of its
// members.  The reference builds the full K x K distance matrix (O(K^2) memory, impossible at
// 1e5 landmarks); here the neighbour search scans the survivor's own cell of the landmark grid
// (fastgrid.cuh), and step (2) -- inherently sequential but touching only the few landmarks that
// do have a close neighbour -- is a directed union-find walked by one thread.  A brute-force path
// keeps the reference's exact corner cases (zero distances replaced by the map diameter, :242) for
// small or degenerate maps.
#pragma once
#include "common.cuh"
#include "assoc.cuh"
#include "fastgrid.cuh"

#define FILTER_SMALL_K 2048

// means + keep flag in one pass over the labels
__global__ void k_means_flags(const DevState* st, const double* __restrict__ sum_x, const double* __restrict__ sum_y,
                              const int* __restrict__ cnt, double cota, int running, double* __restrict__ raw_x,
                              double* __restrict__ raw_y, int* __restrict__ flag, int Lcap)
{
    int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= Lcap) return;
    int k = l < st->raw_l ? cnt[l] : 0;
    if (!running) {   // RUNNING view already wrote the reference-arithmetic means
        raw_x[l] = k > 0 ? sum_x[l] / (double)k : 0.0;
        raw_y[l] = k > 0 ? sum_y[l] / (double)k : 0.0;
    }
    flag[l] = (l < st->raw_l && !((double)k < cota)) ? 1 : 0;      // :232-236
}

// generic: flags (double counts) for icmslam_filter_map on caller data
__global__ void k_flags_from_counts(const double* __restrict__ counts, int n, double cota, int* __restrict__ flag, int Lcap)
{
    int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= Lcap) return;
    flag[l] = (l < n && !(counts[l] < cota)) ? 1 : 0;
}

__global__ void k_compact_kept(DevState* st, const int* __restrict__ flag, const int* __restrict__ pos,
                               const double* __restrict__ raw_x, const double* __restrict__ raw_y,
                               const int* __restrict__ cnt_i, const double* __restrict__ cnt_d, double* __restrict__ kx,
                               double* __restrict__ ky, double* __restrict__ kc, int* __restrict__ parent, int Lcap)
{
    int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= Lcap) return;
    if (flag[l]) {
        int p = pos[l];
        kx[p] = raw_x[l];
        ky[p] = raw_y[l];
        kc[p] = cnt_i ? (double)cnt_i[l] : cnt_d[l];
        parent[p] = p;
    }
    if (l == Lcap - 1) {
        st->kept = pos[l] + flag[l];
        st->n_ind = 0;
        if (st->kept == 0) st->status |= 4;   // ValueError in the reference (ICM_SLAM.py:241-255)
    }
}

__device__ __forceinline__ void atomic_max_pos(double* addr, double v)   // v >= 0
{
    atomicMax((unsigned long long*)addr, (unsigned long long)__double_as_longlong(v));
}
__device__ __forceinline__ void atomic_min_pos(double* addr, double v)   // v >= 0
{
    atomicMin((unsigned long long*)addr, (unsigned long long)__double_as_longlong(v));
}

// bb: bounding box of the survivors (the filter grid's, fastgrid.cuh k_fgrid_bbox)
__device__ __forceinline__ bool filter_small_path(const DevState* st, const unsigned long long* bb, double dist_thr)
{
    if (st->kept <= FILTER_SMALL_K) return true;
    const double extent = fmax(dkey_inv(bb[2]) - dkey_inv(bb[0]), dkey_inv(bb[3]) - dkey_inv(bb[1]));
    return !(extent >= dist_thr);
}

// brute-force path, step A: the map diameter amax (:242)
__global__ void k_filter_diameter(const DevState* st, const double* __restrict__ kx, const double* __restrict__ ky,
                                  const unsigned long long* __restrict__ bb, double dist_thr, double* __restrict__ amax)
{
    if (!filter_small_path(st, bb, dist_thr)) return;
    const int K = st->kept;
    double m = 0.0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < K; j += gridDim.x * blockDim.x)
        for (int i = 0; i < K; ++i) m = fmax(m, dist_rn(kx[i] - kx[j], ky[i] - ky[j]));
    m = warp_max(m);
    if ((threadIdx.x % WARP) == 0) atomic_max_pos(amax, m);
}

// nearest other survivor: amin / b (:243-245), flag = amin < dist_thr
__global__ void k_filter_nn(const DevState* st, const double* __restrict__ kx, const double* __restrict__ ky,
                            double dist_thr, const double* __restrict__ amax_p, const unsigned long long* __restrict__ bb,
                            const FGeom* __restrict__ geom, const int* __restrict__ cell_start, const double2* __restrict__ pts,
                            const int* __restrict__ gidx, int* __restrict__ nn, int* __restrict__ ind_flag, int Lcap)
{
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= Lcap) return;
    const int K = st->kept;
    if (j >= K) { ind_flag[j] = 0; return; }
    const double xj = kx[j], yj = ky[j];
    double best = INFINITY;
    int arg = 0;
    if (filter_small_path(st, bb, dist_thr)) {
        const double amax = *amax_p;
        for (int i = 0; i < K; ++i) {
            double dd = (i == j) ? 0.0 : dist_rn(kx[i] - xj, ky[i] - yj);
            if (dd == 0.0) dd = amax;                          // a[a==0] = max(a)
            if (dd < best) { best = dd; arg = i; }             // argmin: first minimum
        }
    } else {
        // diameter >= dist_thr here, so zero distances (replaced by it) can never pass the gate; the survivor's own cell holds
        // every survivor within dist_thr of it
        const FGeom g = *geom;
        const int c = fgrid_cell(g, xj, yj);
        for (int k = cell_start[c]; k < cell_start[c + 1]; ++k) {
            const double2 p = pts[k];
            const int id = gidx[k];
            const double dd = dist_rn(p.x - xj, p.y - yj);
            if (dd == 0.0) continue;
            if (dd < best || (dd == best && id < arg)) { best = dd; arg = id; }
        }
    }
    nn[j] = arg;
    ind_flag[j] = best < dist_thr ? 1 : 0;                     // :245 (strict <)
}

__global__ void k_ind_compact(DevState* st, const int* __restrict__ flag, const int* __restrict__ pos, int* __restrict__ ind,
                              int Lcap)
{
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= Lcap) return;
    if (flag[j]) ind[pos[j]] = j;
    if (j == Lcap - 1) st->n_ind = pos[j] + flag[j];
}

__device__ __forceinline__ int uf_find(const int* parent, int v)
{
    while (parent[v] != v) v = parent[v];
    return v;
}

// :247-249 -- for i in ind ascending: c[c == c[b[i]]] = c[i]   (class of the neighbour renamed)
__global__ void k_relabel(const DevState* st, const int* __restrict__ ind, const int* __restrict__ nn, int* parent)
{
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int n = st->n_ind;
    for (int q = 0; q < n; ++q) {
        int i = ind[q];
        int X = uf_find(parent, nn[i]), Y = uf_find(parent, i);
        if (X != Y) parent[X] = Y;
    }
}

__global__ void k_roots(const DevState* st, const int* __restrict__ parent, int* __restrict__ lab, int* __restrict__ used)
{
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= st->kept) return;
    int r = uf_find(parent, j);
    lab[j] = r;
    used[r] = 1;
}

// :251-260 -- dense renumbering (rank of the class label) + count-weighted mean
__global__ void k_merge_accumulate(const DevState* st, const int* __restrict__ lab, const int* __restrict__ rank,
                                   const double* __restrict__ kx, const double* __restrict__ ky, const double* __restrict__ kc,
                                   double* __restrict__ ox, double* __restrict__ oy, double* __restrict__ oc)
{
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= st->kept) return;
    int r = rank[lab[j]];
    if (lab[j] == j && st->n_ind == 0) {   // common case: nothing merged
        ox[r] = mul_rn(kx[j], kc[j]); oy[r] = mul_rn(ky[j], kc[j]); oc[r] = kc[j];
        return;
    }
    atomicAdd(ox + r, mul_rn(kx[j], kc[j]));
    atomicAdd(oy + r, mul_rn(ky[j], kc[j]));
    atomicAdd(oc + r, kc[j]);
}

__global__ void k_filter_finalize(DevState* st, const int* __restrict__ used, const int* __restrict__ rank,
                                  const double* __restrict__ ox, const double* __restrict__ oy, const double* __restrict__ oc,
                                  double* __restrict__ map_out, int cap_out, int64_t ld_out, double* __restrict__ counts_state,
                                  double* __restrict__ counts_out, int Lcap, int update_state)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= Lcap) return;
    const int K = st->kept;
    const int newL = K > 0 ? rank[K - 1] + used[K - 1] : 0;
    double c = r < newL ? oc[r] : 0.0;
    if (r < cap_out && map_out) {
        map_out[r] = r < newL ? ox[r] / c : 0.0;
        map_out[ld_out + r] = r < newL ? oy[r] / c : 0.0;
    }
    if (counts_state) counts_state[r] = c;
    if (counts_out && r < cap_out) counts_out[r] = c;
    if (r == 0) {
        st->new_l = newL;
        if (update_state) st->lact = newL;
    }
}

// ---- calc_cambio ---------------------------------------------------------------------------
// thread per NEW landmark: distance to the nearest OLD landmark.  The new landmark's cell of the grid over the old map holds every
// old landmark within dist_thr (1 + FG_MARGIN) of it (fastgrid.cuh: landmarks are registered with that radius plus a 2^-20 slack
// for the rounding of the cell arithmetic), so the nearest candidate within that reach is the nearest old landmark; otherwise,
// or with no candidate, a full scan.  The minimum of the rooted distances is the root of the minimum squared one (sqrt_rn is
// monotone), so the result does not depend on the path.
__global__ void k_cambio(const double* __restrict__ nx_, const double* __restrict__ ny_, int Ln, const double* __restrict__ oldx,
                         const double* __restrict__ oldy, int Lo, const FGeom* __restrict__ geom, const int* __restrict__ cell_start,
                         const double2* __restrict__ pts, double dist_thr, double* __restrict__ acc /* min,max,sum */)
{
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    double best = INFINITY;
    if (j < Ln) {
        const double xj = nx_[j], yj = ny_[j];
        const FGeom g = *geom;
        const int c = fgrid_cell(g, xj, yj);
        double s2 = INFINITY;
        for (int k = cell_start[c]; k < cell_start[c + 1]; ++k) {
            const double2 p = pts[k];
            s2 = fmin(s2, dist2_rn(p.x - xj, p.y - yj));
        }
        best = __dsqrt_rn(s2);
        if (!(best <= dist_thr + FG_MARGIN * dist_thr)) {
            best = INFINITY;
            for (int i = 0; i < Lo; ++i) best = fmin(best, dist_rn(oldx[i] - xj, oldy[i] - yj));
        }
    }
    double mn = warp_min(j < Ln ? best : INFINITY);
    double mx = warp_max(j < Ln ? best : 0.0);
    double sm = warp_sum(j < Ln ? best : 0.0);
    if ((threadIdx.x % WARP) == 0 && (j - (int)(threadIdx.x % WARP)) < Ln) {
        atomic_min_pos(acc + 0, mn);
        atomic_max_pos(acc + 1, mx);
        atomicAdd(acc + 2, sm);
    }
}

// ---- calc_cambio per trajectory of a batch handle (icmslam_batch_iterate_until) --------------------------------------------
// The tail (k_tail_nn / k_tail_steady) fills each trajectory's slots (Freeze::slots) with the changes it could certify.  A
// trajectory with an uncertified change (a landmark that left its proven radius, appeared or merged) gets the full search here,
// as calc_cambio computes it for the trajectory alone: every new landmark against every old landmark of the same region.  Brute
// force over the old map: it runs only on the sweeps that need it.
__global__ void k_fz_regions(const Freeze fz, const double* __restrict__ x, const double* __restrict__ y, int n, int* __restrict__ reg)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) reg[i] = fz.region(x[i], y[i]);
}

// the active trajectories with uncertified changes: need[k] = 1 and their min / max / sum / count slots cleared
__global__ void k_fz_need(const Freeze fz, unsigned char* __restrict__ need)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= fz.K) return;
    const bool nd = !fz.frozen[k] && fz.slots[4 * (size_t)fz.K + k] > 0.0;
    need[k] = nd ? 1 : 0;
    if (nd) {
        fz.slots[k] = INFINITY;
        for (int r = 1; r < 4; ++r) fz.slots[(size_t)r * fz.K + k] = 0.0;
    }
}

__global__ void k_cambio_regions(const Freeze fz, const unsigned char* __restrict__ need, const double* __restrict__ nx_,
                                 const double* __restrict__ ny_, int Ln, const double* __restrict__ oldx, const double* __restrict__ oldy,
                                 const int* __restrict__ oreg, int Lo)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= Ln) return;
    const double xj = nx_[j], yj = ny_[j];
    const int k = fz.region(xj, yj);
    if (k < 0 || !need[k]) return;
    double best = INFINITY;
    for (int i = 0; i < Lo; ++i)
        if (__ldg(oreg + i) == k) best = fmin(best, dist_rn(__ldg(oldx + i) - xj, __ldg(oldy + i) - yj));
    atomic_min_pos(fz.slots + k, best);
    atomic_max_pos(fz.slots + (size_t)fz.K + k, best);
    atomicAdd(fz.slots + 2 * (size_t)fz.K + k, best);
    atomicAdd(fz.slots + 3 * (size_t)fz.K + k, 1.0);
}
