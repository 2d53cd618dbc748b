// mapfilter.cuh -- the entries of Mapa.filtrar (ICM_SLAM.py:204-265) for the callers other than the fused sweep, and
// calc_cambio (ICM_SLAM.py:490-495).
//
// Mapa.filtrar itself is the fused tail's filter chain (tail.cuh, k_tail_compact .. k_tail_nn); every caller runs it.  The
// fused sweep enters it through k_fused_means; the generic sweep through k_means_flags, icmslam_filter_map and pass 0 through
// k_flags_from_counts.  An entry leaves what the chain reads (filter_chain in icmslam.cu lists it): keep flags, kept landmarks
// per block, and the chain's per-call state reset.
#pragma once
#include "common.cuh"
#include "assoc.cuh"
#include "fastgrid.cuh"
#include "tail.cuh"

// The end of an entry, reached by every thread of the block: the block's kept landmarks (k_tail_compact takes its positions from
// them, so an entry is launched on k_tail_compact's grid, nblk(Lcap, 256) x 256), and the chain's per-call state as far_scan_block
// leaves it for the fused sweep: the survivors' bounding box empty, the merge counter zero, steady_ok = 0 (the chain runs).
__device__ __forceinline__ void filter_entry(int keep, int* __restrict__ blk_kept, unsigned long long* bb, TailState* ts)
{
    const int total = __syncthreads_count(keep);
    if (threadIdx.x == 0) {
        blk_kept[blockIdx.x] = total;
        if (blockIdx.x == 0) {
            bb[0] = bb[1] = ~0ull;
            bb[2] = bb[3] = 0ull;
            ts->n_ind = 0;
            ts->steady_ok = 0;
        }
    }
}

// generic sweep: means + keep flag in one pass over the labels
__global__ void k_means_flags(const DevState* st, const double* __restrict__ sum_x, const double* __restrict__ sum_y,
                              const int* __restrict__ cnt, double cota, int running, double* __restrict__ raw_x,
                              double* __restrict__ raw_y, int* __restrict__ flag, int Lcap, int* __restrict__ blk_kept,
                              unsigned long long* bb, TailState* ts)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    int keep = 0;
    if (l < Lcap) {
        const int k = l < st->raw_l ? cnt[l] : 0;
        if (!running) {   // RUNNING view already wrote the reference-arithmetic means
            raw_x[l] = k > 0 ? sum_x[l] / (double)k : 0.0;
            raw_y[l] = k > 0 ? sum_y[l] / (double)k : 0.0;
        }
        keep = (l < st->raw_l && !((double)k < cota)) ? 1 : 0;      // :232-236
        flag[l] = keep;
    }
    filter_entry(keep, blk_kept, bb, ts);
}

// icmslam_filter_map and pass 0: keep flags from double counts
__global__ void k_flags_from_counts(const double* __restrict__ counts, int n, double cota, int* __restrict__ flag, int Lcap,
                                    int* __restrict__ blk_kept, unsigned long long* bb, TailState* ts)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    int keep = 0;
    if (l < Lcap) {
        keep = (l < n && !(counts[l] < cota)) ? 1 : 0;
        flag[l] = keep;
    }
    filter_entry(keep, blk_kept, bb, ts);
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
