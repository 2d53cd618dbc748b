// fastgrid.cuh -- the landmark grid: the association (ICM_SLAM.py:169-172), Mapa.filtrar's
// nearest-neighbour search (ICM_SLAM.py:241-245) and calc_cambio (ICM_SLAM.py:490-495).
//
// Contract: every landmark within dist_thr of a query point is visited, and ties are resolved
// exactly as cdist + np.argmin resolve them (the first minimum of the rooted distances).  Layout,
// made for the hot loop of the fused sweep:
//   * replicated binning: cell edge h >= 2*thr1 (thr1 = dist_thr*(1+2^-20)) and every landmark is
//     registered in each of the (at most 2 x 2) cells its thr1-disc overlaps, so a query reads ONE
//     cell -- the one containing the query point -- instead of a 3 x 3 block;
//   * a FIXED cell budget (NC cells, host constant) so the counting sort's scan has a host-known
//     length and no host round trip: the geometry kernel grows h until nx*ny <= NC;
//   * landmarks stored cell-sorted as double2 (one 16-byte load per candidate); the original index
//     is only fetched for the winner (and for exact tie resolution);
//   * squared distances are compared; the rooted values the reference compares are only formed when
//     two candidates are within 2^-50 relative (sqrt_rn is monotone, so this is exact), and the
//     gate `amin > dist_thr` becomes `s > thr2_hi` with thr2_hi the largest double whose rooted
//     value is <= dist_thr (computed on the host).
// Points outside the bounding box clamp to the border cells on both the build and the query side,
// so a grid whose geometry was fixed for an earlier map stays exact for a later one.
#pragma once
#include "common.cuh"

struct FGeom {
    double x0, y0, inv_h, delta;   // delta = thr1 * inv_h  (< 0.5)
    int nx, ny;
};

struct FGrid {
    FGeom g;
    const int* cell_start;     // nx*ny + 1 (within the NC + 2 allocation)
    const double2* pts;        // cell-sorted coordinates
    const int* idx;            // cell-sorted original indices
};

__device__ __forceinline__ unsigned long long dkey(double v)   // order-preserving double -> u64
{
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double dkey_inv(unsigned long long k)
{
    unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

// bb[0..3] = min x, min y, max x, max y as ordered keys; reset by k_fgrid_bbox_reset
__global__ void k_fgrid_bbox_reset(unsigned long long* bb)
{
    bb[0] = bb[1] = ~0ull;
    bb[2] = bb[3] = 0ull;
}

__global__ void __launch_bounds__(256)
k_fgrid_bbox(const double* __restrict__ px, const double* __restrict__ py, const int* __restrict__ n_ptr, unsigned long long* bb)
{
    const int n = *n_ptr;
    double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        double x = px[i], y = py[i];
        mnx = fmin(mnx, x); mxx = fmax(mxx, x);
        mny = fmin(mny, y); mxy = fmax(mxy, y);
    }
    mnx = warp_min(mnx); mny = warp_min(mny); mxx = warp_max(mxx); mxy = warp_max(mxy);
    if ((threadIdx.x % WARP) == 0 && mnx <= mxx) {
        atomicMin(bb + 0, dkey(mnx)); atomicMin(bb + 1, dkey(mny));
        atomicMax(bb + 2, dkey(mxx)); atomicMax(bb + 3, dkey(mxy));
    }
}

// A landmark is registered with the radius thr1 + FG_MARGIN * dist_thr: the cell lists then stay valid (supersets of what a query
// needs) while every landmark is within the margin of where it was when the grid was built, which lets a sweep that neither
// adds, drops nor merges a landmark keep the grid and only refresh the stored coordinates (tail.cuh k_tail_steady).
#define FG_MARGIN 0.05
// cell edge h = 2*(thr1 + margin)*(1+2^-20) grown by 25 % steps until the grid fits the cell budget
__device__ __forceinline__ FGeom fgrid_make_geom(double mnx, double mny, double mxx, double mxy, double dist_thr, int max_cells)
{
    const double thr1 = dist_thr * (1.0 + 9.5367431640625e-07) + FG_MARGIN * dist_thr;   // 1 + 2^-20, plus the margin
    double h = 2.0 * thr1 * (1.0 + 9.5367431640625e-07);
    if (!(h > 0.0)) h = 1.0;
    const double ex = mxx - mnx, ey = mxy - mny;
    for (;;) {
        double nxd = floor(ex / h) + 2.0, nyd = floor(ey / h) + 2.0;
        if (nxd * nyd <= (double)max_cells) break;
        h *= 1.25;
    }
    FGeom g;
    g.x0 = mnx; g.y0 = mny; g.inv_h = 1.0 / h; g.delta = thr1 * g.inv_h;
    g.nx = __double2int_rd((mxx - mnx) * g.inv_h) + 1;
    g.ny = __double2int_rd((mxy - mny) * g.inv_h) + 1;
    if (g.nx < 1) g.nx = 1;
    if (g.ny < 1) g.ny = 1;
    return g;
}

__global__ void k_fgrid_geom(const unsigned long long* bb, const int* n_ptr, double dist_thr, int max_cells, FGeom* out)
{
    double mnx = 0.0, mny = 0.0, mxx = 0.0, mxy = 0.0;
    if (*n_ptr > 0 && bb[0] != ~0ull) { mnx = dkey_inv(bb[0]); mny = dkey_inv(bb[1]); mxx = dkey_inv(bb[2]); mxy = dkey_inv(bb[3]); }
    *out = fgrid_make_geom(mnx, mny, mxx, mxy, dist_thr, max_cells);
}

// ---- replicated binning -------------------------------------------------------------------------
// Every landmark is registered in each cell its thr1-disc overlaps (at most 2 x 2 cells since
// h >= 2*thr1), so a query inspects exactly ONE cell: the one containing the query point.
__device__ __forceinline__ void fgrid_cell_range(const FGeom& g, double x, double y, int& cx0, int& cx1, int& cy0, int& cy1)
{
    const double fx = (x - g.x0) * g.inv_h, fy = (y - g.y0) * g.inv_h;
    cx0 = min(max(__double2int_rd(fx - g.delta), 0), g.nx - 1); cx1 = min(max(__double2int_rd(fx + g.delta), 0), g.nx - 1);
    cy0 = min(max(__double2int_rd(fy - g.delta), 0), g.ny - 1); cy1 = min(max(__double2int_rd(fy + g.delta), 0), g.ny - 1);
}

__device__ __forceinline__ int fgrid_cell(const FGeom& g, double x, double y)
{
    int cx = __double2int_rd((x - g.x0) * g.inv_h), cy = __double2int_rd((y - g.y0) * g.inv_h);
    cx = min(max(cx, 0), g.nx - 1);
    cy = min(max(cy, 0), g.ny - 1);
    return cy * g.nx + cx;
}

__global__ void __launch_bounds__(256)
k_fgrid_count(const double* __restrict__ px, const double* __restrict__ py, const int* __restrict__ n_ptr, const FGeom* __restrict__ geom,
              int* __restrict__ cell_cnt)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= *n_ptr) return;
    const FGeom g = *geom;
    int cx0, cx1, cy0, cy1;
    fgrid_cell_range(g, px[i], py[i], cx0, cx1, cy0, cy1);
    for (int cy = cy0; cy <= cy1; ++cy)
        for (int cx = cx0; cx <= cx1; ++cx) atomicAdd(cell_cnt + cy * g.nx + cx, 1);
}

__global__ void __launch_bounds__(256)
k_fgrid_fill(const double* __restrict__ px, const double* __restrict__ py, const int* __restrict__ n_ptr, const FGeom* __restrict__ geom,
             const int* __restrict__ cell_start, int* __restrict__ cell_fill, double2* __restrict__ pts, int* __restrict__ idx,
             int4* __restrict__ slots = nullptr /* where each landmark's (at most 4) entries went */, const int* skip = nullptr)
{
    if (skip && *skip) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= *n_ptr) return;
    const FGeom g = *geom;
    const double x = px[i], y = py[i];
    int cx0, cx1, cy0, cy1;
    fgrid_cell_range(g, x, y, cx0, cx1, cy0, cy1);
    int sl[4] = {-1, -1, -1, -1};
    int r = 0;
    for (int cy = cy0; cy <= cy1; ++cy)
        for (int cx = cx0; cx <= cx1; ++cx) {
            const int c = cy * g.nx + cx;
            const int p = cell_start[c] + atomicSub(cell_fill + c, 1) - 1;   // counts the cell back down to zero
            pts[p] = make_double2(x, y);
            idx[p] = i;
            if (r < 4) sl[r] = p;
            ++r;
        }
    if (slots) slots[i] = make_int4(sl[0], sl[1], sl[2], sl[3]);
}

// Nearest landmark of (wx, wy) among the cell's entries [s, e).  Returns the winner's position in the
// cell-sorted arrays (-1 if no candidate) and its squared distance `best` (INFINITY if none).
// Squared distances are compared against a 2^-50 window around the current best; only inside the
// window (an almost exact tie) are the rooted values formed, as cdist + np.argmin compare them.
__device__ __forceinline__ int fgrid_scan(const FGrid& G, double wx, double wy, int s, int e, double& best)
{
    best = INFINITY;
    double lo = INFINITY, hi = INFINITY;
    int bk = -1;
    for (int k = s; k < e; ++k) {
        const double2 p = __ldg(G.pts + k);
        const double s2 = dist2_rn(p.x - wx, p.y - wy);
        bool take = s2 < lo;
        if (!take && s2 <= hi && bk >= 0) {   // (almost) equidistant
            const double dk = __dsqrt_rn(s2), db = __dsqrt_rn(best);
            take = dk < db || (dk == db && __ldg(G.idx + k) < __ldg(G.idx + bk));
        }
        if (take) { best = s2; bk = k; lo = s2 * (1.0 - 8.8817841970012523e-16); hi = s2 * (1.0 + 8.8817841970012523e-16); }
    }
    return bk;
}

// The same scan with the cell's first entry already loaded (p0, id0): lets the caller issue the first
// gathers of several queries together before any of them is consumed.  `bid` = winner's original index.
__device__ __forceinline__ int fgrid_scan_pre(const FGrid& G, double wx, double wy, int s, int cnt, double2 p0, int id0, double& best,
                                              int& bid)
{
    best = INFINITY;
    bid = -1;
    if (cnt <= 0) return -1;
    best = dist2_rn(p0.x - wx, p0.y - wy);
    bid = id0;
    int bk = s;
    double lo = best * (1.0 - 8.8817841970012523e-16), hi = best * (1.0 + 8.8817841970012523e-16);
    for (int k = s + 1; k < s + cnt; ++k) {
        const double2 p = __ldg(G.pts + k);
        const double s2 = dist2_rn(p.x - wx, p.y - wy);
        bool take = s2 < lo;
        int id = -1;
        if (!take && s2 <= hi) {   // (almost) equidistant: decide on the rooted values like np.argmin over cdist
            const double dk = __dsqrt_rn(s2), db = __dsqrt_rn(best);
            id = __ldg(G.idx + k);
            take = dk < db || (dk == db && id < bid);
        }
        if (take) {
            best = s2; bk = k; bid = id >= 0 ? id : __ldg(G.idx + k);
            lo = s2 * (1.0 - 8.8817841970012523e-16); hi = s2 * (1.0 + 8.8817841970012523e-16);
        }
    }
    return bk;
}

__device__ __forceinline__ int fgrid_nearest(const FGrid& G, double wx, double wy, double& best)
{
    const int c = fgrid_cell(G.g, wx, wy);
    return fgrid_scan(G, wx, wy, __ldg(G.cell_start + c), __ldg(G.cell_start + c + 1), best);
}
