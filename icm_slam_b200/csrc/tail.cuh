// tail.cuh -- what follows the fused sweep kernel: new labels and Mapa.filtrar (ICM_SLAM.py:204-265),
// arranged so that the common case (no two surviving landmarks closer than dist_thr, i.e. nothing to
// merge) is a short fixed chain of small kernels with no host round trip, capturable in a CUDA
// graph, and so that the landmark grid built for the filter's neighbour search IS the association
// grid of the next sweep (same points: the filtered map).
//
//   far_scan_block   (by the last block of the association kernel to finish) exclusive scan of the per-tile counts of
//                    scans with far observations
//   k_tail_labels    one thread per far scan: label = lact0 + rank in time order (ICM_SLAM.py:174-182),
//                    statistics of the new label, rewrite of the scan's far labels
//   k_fused_means    raw map from the fixed-point statistics + keep flags (cota, :231-239) + kept landmarks per block
//   k_tail_compact   positions of the kept landmarks (each block sums the counts of the blocks before it), kept
//                    landmarks -> dense arrays + bounding box
//   k_tail_count     geometry of the grid over the survivors + entries per cell
//   k_cell_scan      single-pass exclusive scan of the cell counts (chained blocks)
//   k_fgrid_fill     (fastgrid.cuh)
//   k_tail_nn        nearest other survivor of every survivor (:241-245) through the grid; the survivors written as the
//                    new map on the assumption that nothing merges; the LAST block to finish checks the assumption and
//                    otherwise runs the reference's sequential relabelling (:247-260) and rebuilds the grid
// k_tail_compact .. k_tail_nn are Mapa.filtrar for every caller: the generic sweep, icmslam_filter_map and pass 0 enter them
// through the kernels of mapfilter.cuh instead of k_fused_means, and launch k_tail_nn<false>, without the sweep's bookkeeping.
// The chain keeps its own inputs clean for the next sweep (statistics, counts, far bits are zeroed by the kernel that
// consumes them last): a sweep needs no memset.
#pragma once
#include "common.cuh"
#include "assoc.cuh"
#include "fastgrid.cuh"
#include "p2p.cuh"

struct __align__(16) FarRec {
    int t, rank, n, pad;
    double sx, sy;
};

// Device-side scalars of the fast tail (one per handle).
struct TailState {
    int far_count;      // far records appended by the fused kernel this sweep
    int n_ind;          // survivors with a neighbour closer than dist_thr
    int degenerate;     // bounding box smaller than dist_thr: the reference's zero-distance rule matters
    int far_total;      // scans with far observations in THIS handle's segment
    int label_base;     // such scans in the segments before this one (0 on a single GPU)
    int remap_identity; // the filter kept every landmark of the previous map in place and no new label survived: labels below
                        // lsearch keep their meaning (labels created in the sweep may have come and gone)
    int epoch;          // label-numbering epoch: run records (runs.cuh) built in another epoch are void; bumped whenever landmark
                        // indices change (a merge or a drop in Mapa.filtrar, a map supplied by the caller)
    int n_dirty;        // tiles the steady-state kernel handed to the association kernel this sweep
    int assoc_ticket;   // blocks of the association kernel that have finished (the last one scans the far counts)
    int dirty_done;     // entries of the dirty list handled by earlier association launches of the same sweep
    int nn_ticket;      // blocks of k_tail_nn that have finished (the last one closes the sweep)
    int scan_ticket;    // blocks of k_cell_scan that have finished
    unsigned scan_seq;  // launch number of k_cell_scan: tags the block totals published through global memory (starts at 1)
    unsigned p2p_seq;   // number of the sweep in flight (starts at 1): tags the peer-memory flags of p2p.cuh
    unsigned halo_seq;  // ... of the halo exchange on the side stream (advanced by k_p2p_halo itself)
    int labels_ticket;  // blocks of k_tail_labels that have finished (p2p: the last one flags the statistics as final)
    int reduce_ticket;  // blocks of k_p2p_reduce that have finished
    // the steady tail (k_tail_steady): armed by a full chain that ended without a merge, for the K landmarks it left
    int steady_armed, steady_K, steady_fail, steady_ticket;
    int steady_ok;      // verdict of this sweep's k_tail_steady: 1 = the full chain has nothing to do
    int steady_cleared; // k_tail_steady moved this sweep's statistics to their shadow (the full chain reads them there)
    int steady_sweeps;  // sweeps closed by the steady tail since the handle was created (instrumentation)
    // instrumentation (ICMSLAM_TRACE=1): %globaltimer at the entry of the sweep's kernels, a ring over the last 32 sweeps
    // [0] k_runs [1] k_assoc_tiles [2] k_tail_labels [3] k_p2p_reduce [4] k_tail_steady [5] k_solve_tile [6] k_p2p_halo [7] end of k_tail_steady
    int trace_on; unsigned sweep_no;
    unsigned long long trace[32][8];
};

__device__ __forceinline__ unsigned long long globaltimer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void trace_mark(TailState* ts, int slot)
{
    if (ts->trace_on) ts->trace[ts->sweep_no & 31][slot] = globaltimer_ns();
}

// A landmark as the fused kernel reads it by label: position and the squared radius inside which an
// observation is PROVABLY nearest to it and inside the gate (see hint_radius2).
struct __align__(32) LmRec {
    double x, y, r2, r;     // r = sqrt(r2) rounded down: the radius the run records are certified against (runs.cuh)
};

// The per-sweep part of the device state (Mapa.clear_obs + the label bookkeeping of sensors.py:133-145): by k_sweep_begin, or by
// the first block of the run kernel when the sweep is a link of a chain.
__device__ __forceinline__ void sweep_begin_state(DevState* st, int L_in)
{
    st->cambio[0] = INFINITY; st->cambio[1] = 0.0; st->cambio[2] = 0.0; st->cambio_unres = 0;
    st->lact0 = st->lact;
    st->lsearch = min(st->lact, L_in);
    st->raw_l = st->lact;
    st->status = ST_OK;
    st->n_far_scans = 0;
    st->newton_iters = 0ull;
    st->solved = 0ull;
    st->dirty_tiles = 0;
}

// r2 = min(thr2_hi, (nnd/2)^2 (1 - 2^-30)) with nnd a lower bound of the distance to the nearest other
// landmark: an observation with |obs - A|^2 <= r2 has |obs - B| >= nnd - |obs - A| > |obs - A| for every other
// landmark B with a relative margin of 2^-31, far above the rounding of the distance computation, so
// argmin(cdist) == A with no tie, and sqrt_rn(|obs - A|^2) <= dist_thr.  nnd2_seen is the squared distance to
// the nearest other landmark found in the cells that were searched, reach2 the squared distance within which those
// cells are known to contain EVERY landmark (thr1^2 for the landmark's own cell list, (2 thr1)^2 for the 3 x 3 block
// around it, see nearest_other_wide): if none was found, nnd^2 > reach2.
__device__ __forceinline__ double hint_radius2(double nnd2_seen, double reach2, double thr2_hi)
{
    const double q = 0.25 * fmin(nnd2_seen, reach2) * (1.0 - 9.3132257461547852e-10);
    return fmin(q, thr2_hi);
}

// Squared distance from landmark j at (xj, yj) to the nearest OTHER landmark registered in the 3 x 3 block of cells around
// its own cell.  A cell is at least 2 thr1 wide and every landmark is registered (at least) in the cell that contains it,
// so the block holds every landmark within 2 thr1 of j: a landmark whose neighbours are all farther than that is the
// nearest landmark of every point within thr1 of it, i.e. its proven radius reaches the gate.
__device__ __forceinline__ double nearest_other_wide(const FGeom& g, const int* __restrict__ cell_start, const double2* __restrict__ pts,
                                                     const int* __restrict__ idx, int j, double xj, double yj)
{
    int cx = __double2int_rd((xj - g.x0) * g.inv_h), cy = __double2int_rd((yj - g.y0) * g.inv_h);
    cx = min(max(cx, 0), g.nx - 1); cy = min(max(cy, 0), g.ny - 1);
    double best = INFINITY;
    for (int yy = max(cy - 1, 0); yy <= min(cy + 1, g.ny - 1); ++yy)
        for (int xx = max(cx - 1, 0); xx <= min(cx + 1, g.nx - 1); ++xx) {
            const int c = yy * g.nx + xx;
            for (int k = cell_start[c]; k < cell_start[c + 1]; ++k) {
                if (idx[k] == j) continue;
                const double2 p = pts[k];
                best = fmin(best, dist2_rn(p.x - xj, p.y - yj));      // (a coincident landmark gives 0: its hints are never trusted)
            }
        }
    return best;
}

// What neighbouring time segments tell each other after a sweep (16 doubles per rank, all-gathered):
// [0..2] first owned pose, [3..5] second-to-last owned pose, [6..8] last owned pose, [9] far_total.
#define SEG_REC 16

// scans of tile i that created a label this sweep: one bit per scan of the tile (runs.cuh finalize_scan)
__device__ __forceinline__ int tile_far_count(const unsigned* __restrict__ farbits, int i)
{
    const uint4 w = *reinterpret_cast<const uint4*>(farbits + (size_t)i * 4);
    return __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
}

__device__ __forceinline__ int tile_far_count_cg(const unsigned* farbits, int i)     // (written by other blocks of the same launch)
{
    const uint4 w = __ldcg(reinterpret_cast<const uint4*>(farbits + (size_t)i * 4));
    return __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
}

// One block: exclusive scan over the tiles of the number of label-creating scans, and the sweep's label bookkeeping.
// The counts are first gathered into shared memory (cntb, cap bytes; every thread keeps 8 independent loads in flight), then
// each thread scans a contiguous range of them.  With at most FAR_DIRECT label-creating scans (every steady-state sweep) the
// scan is skipped: k_tail_labels counts the bits before each of them itself, and the total is the number of far records.
#define FAR_DIRECT 64
__device__ void far_scan_block(const unsigned* farbits, int n, int* __restrict__ blk_prefix, DevState* st, TailState* ts, int Lcap,
                               unsigned long long* bb, int* wsum /* >= 32 ints of shared memory */, unsigned char* cntb, int cap)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nth = blockDim.x, nw = nth >> 5;
    int carry = 0;
    const int nrec = *(volatile int*)&ts->far_count;
    if (nrec <= FAR_DIRECT) { carry = nrec; n = 0; }
    for (int s0 = 0; s0 < n; s0 += cap) {
        const int m = min(cap, n - s0);
        for (int i0 = tid; i0 < m; i0 += 8 * nth) {
            int c[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) { const int i = i0 + k * nth; c[k] = i < m ? tile_far_count_cg(farbits, s0 + i) : 0; }
#pragma unroll
            for (int k = 0; k < 8; ++k) { const int i = i0 + k * nth; if (i < m) cntb[i] = (unsigned char)c[k]; }     // (<= 128)
        }
        __syncthreads();
        const int per = (m + nth - 1) / nth;
        const int lo = min(tid * per, m), hi = min(lo + per, m);
        int sum = 0;
        for (int i = lo; i < hi; ++i) sum += cntb[i];
        int inc = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(FULLMASK, inc, d); if (lane >= d) inc += o; }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            int x = lane < nw ? wsum[lane] : 0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(FULLMASK, x, d); if (lane >= d) x += o; }
            wsum[lane] = x;
        }
        __syncthreads();
        int run = carry + inc - sum + (warp ? wsum[warp - 1] : 0);
        for (int i = lo; i < hi; ++i) { blk_prefix[s0 + i] = run; run += cntb[i]; }
        carry += wsum[nw - 1];
        __syncthreads();
    }
    if (tid == 0) {
        const int total = carry;
        ts->far_total = total;
        ts->label_base = 0;
        st->n_far_scans = total;              // (a segmented run overwrites these three in k_seg_unpack)
        st->raw_l = st->lact0 + total;
        if (st->lact0 + total > Lcap) st->status = ST_LABEL_CAP;   // IndexError at ICM_SLAM.py:191
        ts->n_ind = 0;
        ts->degenerate = 0;
        bb[0] = bb[1] = ~0ull;
        bb[2] = bb[3] = 0ull;
    }
}

__device__ __forceinline__ void far_label_write(const FarRec& r, int label, int Lcap, double* __restrict__ raw_x, double* __restrict__ raw_y,
                                                int* __restrict__ cnt)
{
    if (label >= Lcap) return;
    raw_x[label] = r.sx / (double)r.n;
    raw_y[label] = r.sy / (double)r.n;
    cnt[label] = r.n;
}

__global__ void __launch_bounds__(256)
k_tail_labels(TailState* ts, const FarRec* __restrict__ far, const int* __restrict__ blk_prefix, const unsigned* __restrict__ farbits, int tile,
              int t_start, const int* __restrict__ off, DevState* st, int Lcap, int* __restrict__ c, double* __restrict__ raw_x,
              double* __restrict__ raw_y, int* __restrict__ cnt, const P2PDev p2p)
{
    __shared__ int wsum[8];
    __shared__ int s_base;
    if (blockIdx.x == 0 && threadIdx.x == 0) trace_mark(ts, 2);
    const int nrec = ts->far_count;
    int label_base = ts->label_base;
    if (p2p.on) {
        // the global numbering of the sweep's new labels: every segment's count of label-creating scans, straight from the
        // windows (what k_seg_unpack derives from the all-gathered records on the NCCL path)
        if (threadIdx.x == 0) {
            int base = 0, total = 0;
            const bool ok = p2p_wait_far(p2p, *(volatile unsigned*)&ts->p2p_seq, base, total);
            s_base = base;
            if (blockIdx.x == 0) {
                ts->label_base = base;
                st->n_far_scans = total;
                st->raw_l = st->lact0 + total;
                if (st->lact0 + total > Lcap) st->status = ST_LABEL_CAP;
                if (!ok) st->status |= ST_P2P_TIMEOUT;
            }
        }
        __syncthreads();
        label_base = s_base;
    }
    const int lact0 = st->lact0 + label_base;
    // the scan's far observations: -1 from the association kernel, or the label an earlier sweep gave them when the scan
    // was certified on its run records (labels >= lsearch are exactly the labels created inside a sweep)
    const int ls = st->lsearch;
    if (nrec <= FAR_DIRECT) {
        // a block per record: rank in time order = label-creating scans of the tiles before its tile (counted here, all threads) +
        // those of its tile before the scan
        for (int k = blockIdx.x; k < nrec; k += gridDim.x) {
            const FarRec r = far[k];
            const int ti = (r.t - t_start) / tile, lt = (r.t - t_start) % tile;
            int part = 0;
            for (int i0 = threadIdx.x; i0 < ti; i0 += 8 * blockDim.x) {      // (eight independent loads in flight per thread)
                int c8[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) { const int i = i0 + q * blockDim.x; c8[q] = i < ti ? tile_far_count(farbits, i) : 0; }
#pragma unroll
                for (int q = 0; q < 8; ++q) part += c8[q];
            }
            part = warp_sum_i(part);
            __syncthreads();
            if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = part;
            __syncthreads();
            int rank = __popc(farbits[(size_t)ti * 4 + (lt >> 5)] & ((1u << (lt & 31)) - 1u));
            for (int q = 0; q < (lt >> 5); ++q) rank += __popc(farbits[(size_t)ti * 4 + q]);
            for (int q = 0; q < (int)(blockDim.x >> 5); ++q) rank += wsum[q];
            const int label = lact0 + rank;
            if (label >= Lcap) continue;
            if (threadIdx.x == 0) far_label_write(r, label, Lcap, raw_x, raw_y, cnt);
            for (int i = off[r.t] + threadIdx.x; i < off[r.t + 1]; i += blockDim.x)
                if (c[i] < 0 || c[i] >= ls) c[i] = label;
        }
    } else
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < nrec; k += gridDim.x * blockDim.x) {
        const FarRec r = far[k];
        // rank in time order: label-creating scans of the tiles before this one + those of this tile before the scan
        const int ti = (r.t - t_start) / tile, lt = (r.t - t_start) % tile;
        int rank = __popc(farbits[(size_t)ti * 4 + (lt >> 5)] & ((1u << (lt & 31)) - 1u));
        for (int q = 0; q < (lt >> 5); ++q) rank += __popc(farbits[(size_t)ti * 4 + q]);
        const int label = lact0 + blk_prefix[ti] + rank;
        if (label >= Lcap) continue;
        far_label_write(r, label, Lcap, raw_x, raw_y, cnt);
        for (int i = off[r.t]; i < off[r.t + 1]; ++i)
            if (c[i] < 0 || c[i] >= ls) c[i] = label;
    }
    if (p2p.on) {      // the last block to finish: this segment's exchange block (statistics + new labels) is final
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            s_base = atomicAdd(&ts->labels_ticket, 1) == (int)gridDim.x - 1;
            if (s_base) { ts->labels_ticket = 0; __threadfence_system(); }
        }
        __syncthreads();
        if (s_base) p2p_post_ready(p2p, *(volatile unsigned*)&ts->p2p_seq);
    }
}

// raw map of the previous-map landmarks from the fixed-point statistics + keep flags for all labels;
// clears the statistics for the next sweep.
__global__ void __launch_bounds__(256)
k_fused_means(const DevState* st, long long* fsum_x, long long* fsum_y, const int* cnt,
              const double* __restrict__ map_x, const double* __restrict__ map_y, double inv_scale, double cota,
              double* newraw /* 2 x Lcap: means of this sweep's new labels, zero elsewhere; cleared here.  ALIASES fsum_x / fsum_y
                                (old labels use a word as int64 sum, new labels as double mean: disjoint index ranges) */,
              double* __restrict__ raw_x, double* __restrict__ raw_y, int* __restrict__ flag, int Lcap, int* __restrict__ blk_kept,
              unsigned* __restrict__ farbits, int n_far_words, const P2PDev p2p, const TailState* ts, int* cnt_w, DevState* st_w,
              const long long* __restrict__ sh_x, const long long* __restrict__ sh_y, const int* __restrict__ sh_k,
              const Freeze fz, const double* __restrict__ counts_prev)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (ts->steady_ok) return;      // the steady tail closed the sweep (and cleared the statistics for the next one)
    if (fz.frozen) fz.reset_slots(l, gridDim.x * blockDim.x);      // (k_tail_steady may have filled them; k_tail_nn fills them again)
    const bool shadow = ts->steady_cleared != 0;      // k_tail_steady ran and said no: the (reduced) statistics are in its shadow arrays
    if (p2p.on && !shadow) {      // every segment's slice of the reduced statistics is in place (and nobody reads this segment's block any more)
        __shared__ int s_ok;
        if (threadIdx.x == 0) {
            s_ok = p2p_wait_all32(p2p.win[p2p.rank]->rs_done, p2p.world, *(const volatile unsigned*)&ts->p2p_seq) ? 1 : 0;
            if (!s_ok && blockIdx.x == 0) st_w->status |= ST_P2P_TIMEOUT;
            __threadfence_system();
        }
        __syncthreads();
    }
    for (int wd = l; wd < n_far_words; wd += gridDim.x * blockDim.x) farbits[wd] = 0u;      // (k_tail_labels was their last reader)
    int keep = 0;
    if (l < Lcap) {
    const int raw_l = st->raw_l, ls = st->lsearch;
    long long wx, wy;      // the landmark's two statistics words: int64 sums (l < ls) or the fp64 mean of a new label
    int kg;
    if (shadow) {
        wx = sh_x[l]; wy = sh_y[l]; kg = sh_k[l];
        cnt_w[l] = kg;
    } else if (p2p.on) {   // ... from the segment that reduced them (the layout of the exchange block: x | y | counts)
        wx = p2p_word(p2p, l); wy = p2p_word(p2p, (long long)Lcap + l);
        const long long cw = p2p_word(p2p, 2ll * Lcap + (l >> 1));
        kg = (int)((l & 1) ? (cw >> 32) : (cw & 0xffffffffll));
        cnt_w[l] = kg;     // (k_tail_compact reads the global count)
    } else {
        wx = fsum_x[l]; wy = fsum_y[l]; kg = cnt[l];
    }
    const int k = l < raw_l ? kg : 0;
    if (l < ls) {
        raw_x[l] = k > 0 ? map_x[l] + ((double)wx * inv_scale) / (double)k : 0.0;
        raw_y[l] = k > 0 ? map_y[l] + ((double)wy * inv_scale) / (double)k : 0.0;
    } else {
        const bool have = l < raw_l && k > 0;
        raw_x[l] = have ? __longlong_as_double(wx) : 0.0;
        raw_y[l] = have ? __longlong_as_double(wy) : 0.0;
    }
    newraw[l] = 0.0; newraw[Lcap + l] = 0.0;
    fsum_x[l] = 0; fsum_y[l] = 0;
    keep = (l < raw_l && !((double)k < cota)) ? 1 : 0;      // ICM_SLAM.py:232-236
    if (fz.frozen && l < ls && fz.landmark(map_x[l], map_y[l])) {
        // a frozen trajectory's landmark: no observation reached it; it keeps its position and its count, hence survives cota
        const int kp = (int)counts_prev[l];
        raw_x[l] = map_x[l]; raw_y[l] = map_y[l];
        cnt_w[l] = kp;
        keep = 1;
    }
    flag[l] = keep;
    }
    const int total = __syncthreads_count(keep);
    if (threadIdx.x == 0) blk_kept[blockIdx.x] = total;
}

// kept landmarks -> dense (kx, ky, kc), union-find parents, bounding box (ordered-key atomics, one set per block).  The position
// of a kept landmark = kept landmarks of the blocks before this one (blk_kept, from the entry kernel's grid of the same shape) +
// those before it in the block.  The counts are the observation counts cnt, moved to rawcnt and cleared for the next sweep; or,
// given cnt_d (icmslam_filter_map: a caller's counts, unrounded), cnt_d, with cnt and rawcnt left as they are.
__global__ void __launch_bounds__(256)
k_tail_compact(DevState* st, const int* __restrict__ flag, const int* __restrict__ blk_kept, int* __restrict__ pos,
               const double* __restrict__ raw_x, const double* __restrict__ raw_y, int* __restrict__ cnt, double* __restrict__ kx,
               double* __restrict__ ky, double* __restrict__ kc, int* __restrict__ parent, unsigned long long* bb, int Lcap,
               int* __restrict__ klab, int* __restrict__ rawcnt, const TailState* ts, const double* __restrict__ cnt_d)
{
    if (ts->steady_ok) return;
    __shared__ int wpart[8], wcnt[8];
    __shared__ double red[4][8];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int l = blockIdx.x * blockDim.x + tid;
    int part = 0;
    for (int b = tid; b < (int)blockIdx.x; b += blockDim.x) part += blk_kept[b];
    part = warp_sum_i(part);
    const int f = l < Lcap ? flag[l] : 0;
    const unsigned m = __ballot_sync(FULLMASK, f);
    if (lane == 0) { wpart[w] = part; wcnt[w] = __popc(m); }
    __syncthreads();
    int p = __popc(m & ((1u << lane) - 1u));
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) { p += wpart[k]; if (k < w) p += wcnt[k]; }
    double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    if (l < Lcap) {
        pos[l] = p;
        double c;
        if (cnt_d) {
            c = cnt_d[l];
        } else {
            const int k = cnt[l];
            rawcnt[l] = k;
            cnt[l] = 0;
            if (l == Lcap - 1) cnt[Lcap] = 0;
            c = (double)k;
        }
        if (f) {
            const double x = raw_x[l], y = raw_y[l];
            kx[p] = x; ky[p] = y; kc[p] = c;
            parent[p] = p;
            klab[p] = l;
            mnx = mxx = x; mny = mxy = y;
        }
        if (l == Lcap - 1) {
            st->kept = p + f;
            st->n_ind = 0;
            if (p + f == 0) st->status |= 4;   // ValueError in the reference (ICM_SLAM.py:241-255)
        }
    }
    mnx = warp_min(mnx); mny = warp_min(mny); mxx = warp_max(mxx); mxy = warp_max(mxy);
    if (lane == 0) { red[0][w] = mnx; red[1][w] = mny; red[2][w] = mxx; red[3][w] = mxy; }
    __syncthreads();
    if (tid == 0) {
        for (int k = 1; k < (int)(blockDim.x >> 5); ++k) {
            mnx = fmin(mnx, red[0][k]); mny = fmin(mny, red[1][k]); mxx = fmax(mxx, red[2][k]); mxy = fmax(mxy, red[3][k]);
        }
        if (mnx <= mxx) {
            atomicMin(bb + 0, dkey(mnx)); atomicMin(bb + 1, dkey(mny));
            atomicMax(bb + 2, dkey(mxx)); atomicMax(bb + 3, dkey(mxy));
        }
    }
}

// geometry of the grid over the kept landmarks (every block derives it from the bounding box; block 0 records it, with the
// degeneracy test: extent < dist_thr) and the number of entries of each cell
__global__ void __launch_bounds__(256)
k_tail_count(const double* __restrict__ kx, const double* __restrict__ ky, const DevState* st, TailState* ts, const unsigned long long* bb,
             double dist_thr, int max_cells, FGeom* out, int* __restrict__ cell_cnt)
{
    if (ts->steady_ok) return;
    __shared__ FGeom sg;
    const int n = st->kept;
    if (threadIdx.x == 0) {
        double mnx = 0.0, mny = 0.0, mxx = 0.0, mxy = 0.0;
        if (n > 0 && bb[0] != ~0ull) { mnx = dkey_inv(bb[0]); mny = dkey_inv(bb[1]); mxx = dkey_inv(bb[2]); mxy = dkey_inv(bb[3]); }
        sg = fgrid_make_geom(mnx, mny, mxx, mxy, dist_thr, max_cells);
        if (blockIdx.x == 0) { *out = sg; ts->degenerate = (fmax(mxx - mnx, mxy - mny) >= dist_thr) ? 0 : 1; }
    }
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const FGeom g = sg;
    int cx0, cx1, cy0, cy1;
    fgrid_cell_range(g, kx[i], ky[i], cx0, cx1, cy0, cy1);
    for (int cy = cy0; cy <= cy1; ++cy)
        for (int cx = cx0; cx <= cx1; ++cx) atomicAdd(cell_cnt + cy * g.nx + cx, 1);
}

// Exclusive scan of in[0..n) in one pass: a block scans its CS_THREADS * CS_ITEMS elements, publishes its total tagged with the
// launch number, and adds up the totals of the blocks before it as they appear (blocks start in index order, so the ones waited
// for are running or done).  The last block to finish advances the launch number.
#define CS_THREADS 1024
#define CS_ITEMS 8
__global__ void __launch_bounds__(CS_THREADS)
k_cell_scan(const int* __restrict__ in, int* __restrict__ out, int n, unsigned long long* state, TailState* ts)
{
    if (ts->steady_ok) return;
    __shared__ int wsum[32];
    __shared__ int s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, b = blockIdx.x;
    const unsigned seq = *(volatile unsigned*)&ts->scan_seq;
    const int i0 = (b * CS_THREADS + tid) * CS_ITEMS;
    int v[CS_ITEMS];
    if (i0 + CS_ITEMS <= n) {
        const int4 a = *reinterpret_cast<const int4*>(in + i0), c = *reinterpret_cast<const int4*>(in + i0 + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
    } else {
#pragma unroll
        for (int k = 0; k < CS_ITEMS; ++k) v[k] = (i0 + k < n) ? in[i0 + k] : 0;
    }
    int s = 0;
#pragma unroll
    for (int k = 0; k < CS_ITEMS; ++k) s += v[k];
    int inc = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(FULLMASK, inc, d); if (lane >= d) inc += o; }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int x = wsum[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(FULLMASK, x, d); if (lane >= d) x += o; }
        wsum[lane] = x;
        const int total = __shfl_sync(FULLMASK, x, 31);
        if (lane == 0) *(volatile unsigned long long*)(state + b) = ((unsigned long long)seq << 32) | (unsigned)total;
        int acc = 0;
        for (int p0 = 0; p0 < b; p0 += 32) {
            const int pb = p0 + lane;
            if (pb < b) {
                unsigned long long wv;
                do { wv = *(volatile unsigned long long*)(state + pb); } while ((unsigned)(wv >> 32) != seq);
                acc += (int)(unsigned)wv;
            }
        }
        acc = warp_sum_i(acc);
        if (lane == 0) s_base = acc;
    }
    __syncthreads();
    int run = s_base + (warp ? wsum[warp - 1] : 0) + inc - s;
    if (i0 + CS_ITEMS <= n) {
        int4 a, c;
        a.x = run; run += v[0]; a.y = run; run += v[1]; a.z = run; run += v[2]; a.w = run; run += v[3];
        c.x = run; run += v[4]; c.y = run; run += v[5]; c.z = run; run += v[6]; c.w = run;
        *reinterpret_cast<int4*>(out + i0) = a; *reinterpret_cast<int4*>(out + i0 + 4) = c;
    } else {
#pragma unroll
        for (int k = 0; k < CS_ITEMS; ++k) { if (i0 + k < n) out[i0 + k] = run; run += v[k]; }
    }
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(&ts->scan_ticket, 1) == (int)gridDim.x - 1) { ts->scan_ticket = 0; ts->scan_seq = seq + 1u; }
    }
}

// What the merge path (tail_slow_body) needs beyond the arguments of k_tail_nn.
struct SlowArgs {
    double dist_thr;
    int* parent; int* ind_pos; int* ind; int* lab; int* used; int* rank;
    double* ox; double* oy; double* oc;
    int max_cells; FGeom* geom; int* cell_cnt; int* cell_start; double2* pts; int* gidx;
    double2* gbuild; double* nnd0; int steady_enable;      // for the steady tail of the next sweeps
    Freeze fz;
};

// one landmark's calc_cambio term in its trajectory's slots (resolved: the change cd; not: it needs the fallback search)
__device__ __forceinline__ void fz_add(const Freeze& fz, int k, bool resolved, double cd)
{
    atomicAdd(fz.slots + 3 * (size_t)fz.K + k, 1.0);
    if (resolved) {
        atomic_min_pos(fz.slots + k, cd); atomic_max_pos(fz.slots + (size_t)fz.K + k, cd); atomicAdd(fz.slots + 2 * (size_t)fz.K + k, cd);
    } else {
        atomicAdd(fz.slots + 4 * (size_t)fz.K + k, 1.0);
    }
}

__device__ void tail_slow_body(DevState* st, TailState* ts, double dist_thr, double* kx, double* ky, double* kc, int* parent, int* nn, int* ind_flag,
            int* ind_pos, int* ind, int* lab, int* used, int* rank, double* ox, double* oy, double* oc, double* map_out, int cap_out,
            int64_t ld_out, double* counts_state, int Lcap, int max_cells, FGeom* geom, int* cell_cnt, int* cell_start, double2* pts, int* gidx,
            const int* kflag, const int* kpos, double thr1sq, double thr2_hi, LmRec* lmrec, int* remap, const Freeze& fz);

// Nearest OTHER survivor (zero distances are never neighbours, ICM_SLAM.py:242) within dist_thr, searched in the 3 x 3 block
// of cells around the survivor (three contiguous runs of the cell-sorted arrays, one per row of cells): the block holds
// every landmark within 2 thr1, so the same pass yields the distance the hint radius is derived from (see
// nearest_other_wide).  And, for free, calc_cambio (ICM_SLAM.py:490-495) of the new map against the previous one: the
// landmark a new landmark was updated from is its nearest old landmark whenever it stayed inside that landmark's proven
// radius r (<= half the distance to any other old landmark: |new - other| >= 2 r - d > d).
// The survivors are written as the new map (count-weighted mean of one member, :258-260) on the assumption that nothing
// merges; the last block to finish knows whether that held (n_ind == 0 and the map is not degenerate), closes the sweep's
// bookkeeping (FUSED: the instance the fused sweep launches; the other callers of the filter have no sweep in flight to close)
// and, if it did not, runs the reference's sequential relabelling over what the other blocks left.
template <bool FUSED>
__global__ void __launch_bounds__(256)
k_tail_nn(DevState* st, TailState* ts, double* __restrict__ kx, double* __restrict__ ky, double* __restrict__ kc, const FGeom* geom,
          const int* cell_start, const double2* pts, const int* idx, double thr2_lt, int* nn, int* ind_flag, int Lcap,
          const int* __restrict__ klab, const int* __restrict__ kflag, const int* __restrict__ kpos, const LmRec* __restrict__ lmrec_old,
          LmRec* lmrec_new, double* map_out, int cap_out, int64_t ld_out, double* counts_state, double thr1sq, double thr2_hi,
          int* remap, const SlowArgs sa)
{
    if (ts->steady_ok) return;
    __shared__ double red[3][8];
    __shared__ int redn[2][8];
    __shared__ int s_last, s_slow;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int K = st->kept;
    const bool act = j < Lcap && j < K && !ts->degenerate;
    double cd = 0.0, wide = 0.0;
    int cres = 0, cun = 0, nind = 0;
    const Freeze& fz = sa.fz;
    // a frozen trajectory's landmark keeps its exact position and never merges (every landmark near it is frozen as well)
    const bool frz = fz.frozen && j < Lcap && j < K && fz.landmark(kx[j], ky[j]);
    if (j < Lcap && !act) {
        ind_flag[j] = 0;
        if (j == 0 && K > 0) { cun = K; if (fz.frozen) for (int k = 0; k < fz.K; ++k) atomicAdd(fz.slots + 4 * (size_t)fz.K + k, 1.0); }
    }
    if (act) {
        const int l = klab[j];
        const double xj = kx[j], yj = ky[j];
        if (l < st->lsearch) {
            const LmRec o = lmrec_old[l];
            const double c = kc[j];
            const double d = dist_rn(mul_rn(xj, c) / c - o.x, mul_rn(yj, c) / c - o.y);      // (the map's own rounding, below)
            if (d < o.r * (1.0 - 1e-9)) { cres = 1; cd = d; }
        }
        cun = 1 - cres;
        const FGeom g = *geom;
        int cx = __double2int_rd((xj - g.x0) * g.inv_h), cy = __double2int_rd((yj - g.y0) * g.inv_h);
        cx = min(max(cx, 0), g.nx - 1); cy = min(max(cy, 0), g.ny - 1);
        const int xa = max(cx - 1, 0), xb = min(cx + 1, g.nx - 1);
        int rs[3], re[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            const int yy = cy - 1 + q;
            const bool in = yy >= 0 && yy < g.ny;
            rs[q] = in ? cell_start[yy * g.nx + xa] : 0;
            re[q] = in ? cell_start[yy * g.nx + xb + 1] : 0;
        }
        double best = INFINITY, lo = INFINITY, hi = INFINITY;
        int arg = -1;
        wide = INFINITY;
#pragma unroll
        for (int q = 0; q < 3; ++q)
            for (int k = rs[q]; k < re[q]; ++k) {
                const double2 p = pts[k];
                const int id = idx[k];
                if (id == j) continue;
                const double s2 = dist2_rn(p.x - xj, p.y - yj);
                wide = fmin(wide, s2);                  // (a coincident landmark gives 0: its hints are never trusted)
                if (s2 == 0.0) continue;
                bool take = s2 < lo;
                if (!take && s2 <= hi && arg >= 0) {
                    const double dk = __dsqrt_rn(s2), db = __dsqrt_rn(best);
                    take = dk < db || (dk == db && id < arg);
                }
                if (take) { best = s2; arg = id; lo = s2 * (1.0 - 8.8817841970012523e-16); hi = s2 * (1.0 + 8.8817841970012523e-16); }
            }
        const int f = (arg >= 0 && best <= thr2_lt && !frz) ? 1 : 0;      // amin < dist_thr (strict, :245)
        nn[j] = arg < 0 ? 0 : arg;
        ind_flag[j] = f;
        nind = f;
        if (fz.frozen && !frz) {      // the trajectory's calc_cambio; a merge in its region needs the fallback search
            const int k = fz.region(xj, yj);
            if (k >= 0) { fz_add(fz, k, cres != 0, cd); if (f) atomicAdd(fz.slots + 4 * (size_t)fz.K + k, 1.0); }
        }
    }
    if (j < Lcap) {      // the new map if nothing merges
        const bool have = j < K;
        const double c = have ? kc[j] : 0.0;
        const double mx = have ? (frz ? kx[j] : mul_rn(kx[j], c) / c) : 0.0, my = have ? (frz ? ky[j] : mul_rn(ky[j], c) / c) : 0.0;
        if (j < cap_out) { map_out[j] = mx; map_out[ld_out + j] = my; }
        counts_state[j] = c;
        LmRec rec;
        rec.x = mx; rec.y = my; rec.r2 = act ? hint_radius2(wide, 4.0 * thr1sq, thr2_hi) : 0.0; rec.r = __dsqrt_rd(rec.r2);
        lmrec_new[j] = rec;
        remap[j] = (j < st->raw_l && kflag[j]) ? kpos[j] : -1;      // label of this sweep -> index in the new map
        if (act) {      // what the steady tail of the next sweeps starts from (k_tail_steady)
            sa.gbuild[j] = make_double2(mx, my);
            sa.nnd0[j] = __dsqrt_rd(fmin(wide, 4.0 * thr1sq));
        }
    }
    // block totals -> one set of atomics per block
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const double mn = warp_min(cres ? cd : INFINITY), mx = warp_max(cres ? cd : 0.0), sm = warp_sum(cd);
    const int un = warp_sum_i(cun), ni = warp_sum_i(nind);
    if (lane == 0) { red[0][w] = mn; red[1][w] = mx; red[2][w] = sm; redn[0][w] = un; redn[1][w] = ni; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = red[0][0], b = red[1][0], c = red[2][0];
        int u = redn[0][0], n2 = redn[1][0];
        for (int k = 1; k < (int)(blockDim.x >> 5); ++k) { a = fmin(a, red[0][k]); b = fmax(b, red[1][k]); c += red[2][k]; u += redn[0][k]; n2 += redn[1][k]; }
        if (a < INFINITY) { atomic_min_pos(st->cambio + 0, a); atomic_max_pos(st->cambio + 1, b); atomicAdd(st->cambio + 2, c); }
        if (u) atomicAdd(&st->cambio_unres, u);
        if (n2) atomicAdd(&ts->n_ind, n2);
        __threadfence();
        const int last = atomicAdd(&ts->nn_ticket, 1) == (int)gridDim.x - 1;
        int slow = 0;
        if (last) {      // every other block's results are in global memory
            __threadfence();
            ts->nn_ticket = 0;
            const int n_ind = atomicAdd(&ts->n_ind, 0);
            slow = (n_ind != 0 || ts->degenerate) ? 1 : 0;
            if (!slow) { st->new_l = K; st->lact = K; st->n_ind = 0; }
            if (FUSED) {
                ts->far_count = 0; ts->n_dirty = 0;      // (consumed by k_tail_labels / the association kernel: ready for the next sweep)
                ts->p2p_seq += 1u;
                ts->sweep_no += 1u;
                // every old label survived in place (its position among the kept landmarks is its index) and nothing was added
                const int ls = st->lsearch, e = max(ls - 1, 0);
                const int identity = (!slow && ls > 0 && K == ls && kflag[e] && kpos[e] == e) ? 1 : 0;
                // run records (runs.cuh) name landmarks by index: void every one of them when landmark indices changed
                if (!identity) ts->epoch += 1;
                ts->remap_identity = identity;
                ts->steady_armed = (!slow && sa.steady_enable) ? 1 : 0;      // (a merged map is rebuilt by one block without the steady tail's inputs)
                ts->steady_K = K;
            }
        }
        s_last = last; s_slow = slow;
    }
    __syncthreads();
    if (!s_last || !s_slow) return;
    tail_slow_body(st, ts, sa.dist_thr, kx, ky, kc, sa.parent, nn, ind_flag, sa.ind_pos, sa.ind, sa.lab, sa.used, sa.rank, sa.ox, sa.oy, sa.oc,
                   map_out, cap_out, ld_out, counts_state, Lcap, sa.max_cells, sa.geom, sa.cell_cnt, sa.cell_start, sa.pts, sa.gidx, kflag, kpos,
                   thr1sq, thr2_hi, lmrec_new, remap, fz);
}


// ---- the steady tail ------------------------------------------------------------------------------------------------------
// A sweep that neither adds, drops nor merges a landmark -- every sweep of a converging run after the first few -- needs none
// of the filter's machinery: the new map is the means, in place; the landmark grid stays valid while every landmark is within
// FG_MARGIN * dist_thr of where it was when the grid was built (fastgrid.cuh) and only its stored coordinates are refreshed; and
// the proven radius follows from a bound instead of a neighbour search: with nnd0 a lower bound of the distance from landmark i
// to any other landmark at build time and D the displacement since then (<= margin for all of them),
// |p_i' - p_j'| >= nnd0_i - D_i - D_j >= nnd0_i - D_i - margin, which is also what rules out a merge (> dist_thr).
// Every thread checks its landmark and writes its results on the assumption that all checks pass (nothing it writes is an input of
// the full chain, which overwrites all of it); the last block to finish publishes the verdict in ts->steady_ok: 1 = done, the
// kernels of the full chain return at once (k_fused_means only clears the statistics); 0 = the full chain runs as if this
// kernel had not.  What is computed is bit-identical either way (same expressions for the map; the radius differs, and a radius
// only decides which exact path labels an observation).
struct SteadyArgs {
    long long* fsum_x; long long* fsum_y; int* cnt;
    long long* sh_x; long long* sh_y; int* sh_k;      // the statistics as this kernel found them (it clears them): what the full chain reads if it must run
    unsigned* farbits; int n_far_words;
    cudaGraphConditionalHandle cond; int use_cond;    // inside a CUDA graph the full chain is the body of an IF node: 1 = run it
    const double* map_x; const double* map_y;
    double inv_scale, cota, dist_thr, thr1sq, thr2_hi;
    const LmRec* lmrec_old; LmRec* lmrec_new;
    const double2* gbuild; const double* nnd0; const int4* gslots; double2* gpts;
    double* raw_x; double* raw_y; int* rawcnt;
    double* map_out; int cap_out; int64_t ld_out; double* counts_state; int* remap; int Lcap;
    double* cpart;      // 5 doubles per block: calc_cambio partials (min, max, sum, resolved?, unresolved)
    Freeze fz;
};

template <bool FZ>      // FZ: a batch with frozen trajectories (a.fz); the plain sweep launches the instance without the tests
__global__ void __launch_bounds__(256)
k_tail_steady(DevState* st, TailState* ts, const SteadyArgs a, const P2PDev p2p)
{
    __shared__ double red[3][8];
    __shared__ int redn[2][8];
    __shared__ int s_flag;
    const int K = ts->steady_K, ls = st->lsearch;
    if (blockIdx.x == 0 && threadIdx.x == 0) trace_mark(ts, 4);
    if (!(ts->steady_armed && ls == K && st->lact0 == K && K > 0)) {      // (the same for every block)
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            ts->steady_ok = 0; ts->steady_cleared = 0;
            if (a.use_cond) cudaGraphSetConditional(a.cond, 1u);
        }
        return;
    }
    if (p2p.on) {      // every segment's slice of the reduced statistics is in place
        if (threadIdx.x == 0) {
            s_flag = p2p_wait_all32(p2p.win[p2p.rank]->rs_done, p2p.world, *(const volatile unsigned*)&ts->p2p_seq) ? 1 : 0;
            if (!s_flag && blockIdx.x == 0) st->status |= ST_P2P_TIMEOUT;
            __threadfence_system();
        }
        __syncthreads();
    }
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    const int raw_l = st->raw_l;
    const double margin = FG_MARGIN * a.dist_thr;
    int fail = 0, cres = 0, cun = 0;
    double cd = 0.0;
    for (int wd = l; wd < a.n_far_words; wd += gridDim.x * blockDim.x) a.farbits[wd] = 0u;      // (k_tail_labels was their last reader)
    if (l < a.Lcap) {
        long long wx, wy;
        int kg;
        if (p2p.on) {
            wx = p2p_word(p2p, l); wy = p2p_word(p2p, (long long)a.Lcap + l);
            const long long cw = p2p_word(p2p, 2ll * a.Lcap + (l >> 1));
            kg = (int)((l & 1) ? (cw >> 32) : (cw & 0xffffffffll));
        } else {
            wx = a.fsum_x[l]; wy = a.fsum_y[l]; kg = a.cnt[l];
        }
        // the statistics move to their shadow and are cleared for the next sweep here: when the verdict is "done" nothing else
        // of the tail has to run
        a.sh_x[l] = wx; a.sh_y[l] = wy; a.sh_k[l] = kg;
        a.fsum_x[l] = 0; a.fsum_y[l] = 0; a.cnt[l] = 0;
        if (l == a.Lcap - 1) a.cnt[a.Lcap] = 0;
        const int k = l < raw_l ? kg : 0;
        LmRec rec;
        rec.x = 0.0; rec.y = 0.0; rec.r2 = 0.0; rec.r = 0.0;
        double mx = 0.0, my = 0.0, c = 0.0, rx = 0.0, ry = 0.0;
        if (l < ls) {
            const bool frz = FZ && a.fz.landmark(a.map_x[l], a.map_y[l]);
            if (!frz && (double)k < a.cota) fail = 1;                      // the landmark would be dropped (ICM_SLAM.py:232-236)
            else {
                if (frz) {      // (k_fused_means / k_tail_nn: position and count as they were)
                    c = a.counts_state[l];
                    kg = (int)c;
                    rx = a.map_x[l]; ry = a.map_y[l]; mx = rx; my = ry;
                } else {
                    c = (double)k;
                    rx = a.map_x[l] + ((double)wx * a.inv_scale) / c;      // k_fused_means
                    ry = a.map_y[l] + ((double)wy * a.inv_scale) / c;
                    mx = mul_rn(rx, c) / c; my = mul_rn(ry, c) / c;      // k_tail_nn (count-weighted mean of one member, :258-260)
                    const LmRec o = a.lmrec_old[l];
                    const double d = dist_rn(mx - o.x, my - o.y);
                    if (d < o.r * (1.0 - 1e-9)) { cres = 1; cd = d; }
                    cun = 1 - cres;
                    if (FZ) { const int kk = a.fz.region(mx, my); if (kk >= 0) fz_add(a.fz, kk, cres != 0, cd); }
                }
                const double2 gb = a.gbuild[l];
                const double D = dist_rn(mx - gb.x, my - gb.y) * (1.0 + 1e-12);
                const double nb = a.nnd0[l] - D - margin;             // lower bound of the distance to any other landmark now
                if (!(D <= margin) || !(nb > a.dist_thr * (1.0 + 1e-9))) fail = 1;
                rec.x = mx; rec.y = my;
                rec.r2 = nb > 0.0 ? hint_radius2(nb * nb, 4.0 * a.thr1sq, a.thr2_hi) : 0.0;
                rec.r = __dsqrt_rd(rec.r2);
                const int4 s4 = a.gslots[l];
                const double2 np_ = make_double2(mx, my);
                if (s4.x >= 0) a.gpts[s4.x] = np_;
                if (s4.y >= 0) a.gpts[s4.y] = np_;
                if (s4.z >= 0) a.gpts[s4.z] = np_;
                if (s4.w >= 0) a.gpts[s4.w] = np_;
            }
            a.remap[l] = l;
        } else {
            const bool have = l < raw_l && k > 0;
            if (l < raw_l && !((double)k < a.cota)) fail = 1;        // a label created in this sweep would be kept
            rx = have ? __longlong_as_double(wx) : 0.0;
            ry = have ? __longlong_as_double(wy) : 0.0;
            a.remap[l] = -1;
        }
        a.raw_x[l] = rx; a.raw_y[l] = ry; a.rawcnt[l] = kg;
        if (l < a.cap_out) { a.map_out[l] = mx; a.map_out[a.ld_out + l] = my; }
        a.counts_state[l] = c;
        a.lmrec_new[l] = rec;
    }
    // block partials of calc_cambio and of the verdict
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const double mn = warp_min(cres ? cd : INFINITY), mxv = warp_max(cres ? cd : 0.0), sm = warp_sum(cd);
    const int un = warp_sum_i(cun), fl = warp_sum_i(fail);
    if (lane == 0) { red[0][w] = mn; red[1][w] = mxv; red[2][w] = sm; redn[0][w] = un; redn[1][w] = fl; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double p0 = red[0][0], p1 = red[1][0], p2 = red[2][0];
        int u = redn[0][0], f = redn[1][0];
        for (int q = 1; q < (int)(blockDim.x >> 5); ++q) { p0 = fmin(p0, red[0][q]); p1 = fmax(p1, red[1][q]); p2 += red[2][q]; u += redn[0][q]; f += redn[1][q]; }
        double* cp = a.cpart + (size_t)blockIdx.x * 4;
        cp[0] = p0; cp[1] = p1; cp[2] = p2; cp[3] = (double)u;
        if (f) atomicOr(&ts->steady_fail, 1);
        __threadfence();
        s_flag = atomicAdd(&ts->steady_ticket, 1) == (int)gridDim.x - 1;
    }
    __syncthreads();
    if (!s_flag) return;
    // ---- last block: the verdict, and when it is "done" what the end of the full chain would have left ---------------------------
    __threadfence();
    const int ok = atomicOr(&ts->steady_fail, 0) == 0;
    double p0 = INFINITY, p1 = 0.0, p2 = 0.0, p3 = 0.0;
    if (ok)
        for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
            const double* cp = a.cpart + (size_t)b * 4;
            p0 = fmin(p0, __ldcg(cp)); p1 = fmax(p1, __ldcg(cp + 1)); p2 += __ldcg(cp + 2); p3 += __ldcg(cp + 3);
        }
    p0 = warp_min(p0); p1 = warp_max(p1); p2 = warp_sum(p2); p3 = warp_sum(p3);
    __syncthreads();
    if (lane == 0) { red[0][w] = p0; red[1][w] = p1; red[2][w] = p2; redn[0][w] = (int)p3; }
    __syncthreads();
    if (threadIdx.x == 0) {
        ts->steady_ticket = 0;
        ts->steady_fail = 0;
        ts->steady_ok = ok;
        ts->steady_cleared = 1;
        trace_mark(ts, 7);
        if (ok) ts->sweep_no += 1u;
        if (a.use_cond) cudaGraphSetConditional(a.cond, ok ? 0u : 1u);
        if (ok) {
            for (int q = 1; q < (int)(blockDim.x >> 5); ++q) { red[0][0] = fmin(red[0][0], red[0][q]); red[1][0] = fmax(red[1][0], red[1][q]); red[2][0] += red[2][q]; redn[0][0] += redn[0][q]; }
            if (red[0][0] < INFINITY) { st->cambio[0] = red[0][0]; st->cambio[1] = red[1][0]; st->cambio[2] = red[2][0]; }
            st->cambio_unres = redn[0][0];
            st->kept = K; st->new_l = K; st->lact = K; st->n_ind = 0;
            ts->n_ind = 0; ts->remap_identity = 1;
            ts->far_count = 0; ts->n_dirty = 0;
            ts->p2p_seq += 1u;
            ts->steady_sweeps += 1;
        }
    }
}

// landmark records of a map whose grid has just been built (first sweep on a caller-supplied map)
__global__ void __launch_bounds__(256)
k_lmrec_build(const double* __restrict__ mx, const double* __restrict__ my, const int* __restrict__ n_ptr, const FGeom* __restrict__ geom,
              const int* __restrict__ cell_start, const double2* __restrict__ pts, const int* __restrict__ idx, double thr1sq, double thr2_hi,
              LmRec* __restrict__ lmrec)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= *n_ptr) return;
    const FGeom g = *geom;
    const double xj = mx[j], yj = my[j];
    const double best = nearest_other_wide(g, cell_start, pts, idx, j, xj, yj);
    LmRec rec;
    rec.x = xj; rec.y = yj; rec.r2 = hint_radius2(best, 4.0 * thr1sq, thr2_hi); rec.r = __dsqrt_rd(rec.r2);
    lmrec[j] = rec;
}

// ---- the merge path: one block ------------------------------------------------------------------------
__device__ __forceinline__ int uf_find(const int* parent, int v)
{
    while (parent[v] != v) v = parent[v];
    return v;
}

// block-wide exclusive scan of v[0..n) (global memory) into out[0..n); returns the total to all threads
__device__ int block_exclusive_scan(const int* v, int* out, int n, int* wsum /* >= 33 ints of shared memory */)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nth = blockDim.x;
    const int per = (n + nth - 1) / nth;
    const int lo = min(tid * per, n), hi = min(lo + per, n);
    int s = 0;
    for (int i = lo; i < hi; ++i) s += v[i];
    int inc = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int o = __shfl_up_sync(FULLMASK, inc, d); if (lane >= d) inc += o; }
    __syncthreads();
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int x = lane < (nth >> 5) ? wsum[lane] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { int o = __shfl_up_sync(FULLMASK, x, d); if (lane >= d) x += o; }
        wsum[lane] = x;
    }
    __syncthreads();
    int run = inc - s + (warp ? wsum[warp - 1] : 0);
    for (int i = lo; i < hi; ++i) { const int a = v[i]; out[i] = run; run += a; }
    const int total = wsum[(nth >> 5) - 1];
    __syncthreads();
    return total;
}

__device__ void tail_slow_body(DevState* st, TailState* ts, double dist_thr, double* kx, double* ky, double* kc, int* parent, int* nn, int* ind_flag,
            int* ind_pos, int* ind, int* lab, int* used, int* rank, double* ox, double* oy, double* oc, double* map_out, int cap_out,
            int64_t ld_out, double* counts_state, int Lcap,
            // grid rebuild over the merged map
            int max_cells, FGeom* geom, int* cell_cnt, int* cell_start, double2* pts, int* gidx,
            const int* kflag, const int* kpos, double thr1sq, double thr2_hi, LmRec* lmrec, int* remap, const Freeze& fz)
{
    // (runs in the last block of k_tail_nn: everything it reads was written by other blocks of the same launch or before)
    __shared__ int wsum[34];
    __shared__ double red[4][32];
    const int tid = threadIdx.x, nth = blockDim.x;
    const int K = st->kept;
    if (ts->degenerate) {
        // the whole map fits in a dist_thr box: the reference's brute force with zero distances replaced by the
        // map diameter (:241-245)
        double m = 0.0;
        for (int j = tid; j < K; j += nth)
            for (int i = 0; i < K; ++i) m = fmax(m, dist_rn(kx[i] - kx[j], ky[i] - ky[j]));
        m = warp_max(m);
        if ((tid & 31) == 0) red[0][tid >> 5] = m;
        __syncthreads();
        double amax = 0.0;
        for (int w = 0; w < (nth >> 5); ++w) amax = fmax(amax, red[0][w]);
        for (int j = tid; j < K; j += nth) {
            double best = INFINITY;
            int arg = 0;
            for (int i = 0; i < K; ++i) {
                double dd = (i == j) ? 0.0 : dist_rn(kx[i] - kx[j], ky[i] - ky[j]);
                if (dd == 0.0) dd = amax;
                if (dd < best) { best = dd; arg = i; }
            }
            nn[j] = arg;
            ind_flag[j] = best < dist_thr ? 1 : 0;
        }
        for (int j = K + tid; j < Lcap; j += nth) ind_flag[j] = 0;
        __syncthreads();
    }
    // ordered list of the survivors that have a close neighbour
    const int n_ind = block_exclusive_scan(ind_flag, ind_pos, K, wsum);
    for (int j = tid; j < K; j += nth) {
        if (ind_flag[j]) ind[ind_pos[j]] = j;
        used[j] = 0; ox[j] = 0.0; oy[j] = 0.0; oc[j] = 0.0;
    }
    __syncthreads();
    if (tid == 0) {   // :247-249 -- for i in ind ascending: c[c == c[b[i]]] = c[i]
        for (int q = 0; q < n_ind; ++q) {
            const int i = ind[q];
            const int X = uf_find(parent, nn[i]), Y = uf_find(parent, i);
            if (X != Y) parent[X] = Y;
        }
    }
    __syncthreads();
    for (int j = tid; j < K; j += nth) {
        const int r = uf_find(parent, j);
        lab[j] = r;
        used[r] = 1;
    }
    __syncthreads();
    const int newL = block_exclusive_scan(used, rank, K, wsum);   // :251-253 dense renumbering in ascending order
    for (int j = tid; j < K; j += nth) {                           // :258-260 count-weighted means
        const int r = rank[lab[j]];
        atomicAdd(ox + r, mul_rn(kx[j], kc[j]));
        atomicAdd(oy + r, mul_rn(ky[j], kc[j]));
        atomicAdd(oc + r, kc[j]);
    }
    __syncthreads();
    for (int r = tid; r < Lcap; r += nth) {
        const double c = r < newL ? oc[r] : 0.0;
        if (r < cap_out) {
            map_out[r] = r < newL ? ox[r] / c : 0.0;
            map_out[ld_out + r] = r < newL ? oy[r] / c : 0.0;
        }
        counts_state[r] = c;
    }
    for (int l = tid; l < Lcap; l += nth) remap[l] = (l < st->raw_l && kflag[l]) ? rank[lab[kpos[l]]] : -1;
    if (fz.frozen) {      // a frozen landmark is a class of its own: its exact position, not the rounded count-weighted mean
        __syncthreads();
        for (int j = tid; j < K; j += nth)
            if (fz.landmark(kx[j], ky[j])) { const int r = rank[lab[j]]; if (r < cap_out) { map_out[r] = kx[j]; map_out[ld_out + r] = ky[j]; } }
    }
    if (tid == 0) { st->new_l = newL; st->lact = newL; st->n_ind = n_ind; st->cambio_unres += 1; }   // (merged map: calc_cambio needs the full search)
    __syncthreads();
    // ---- rebuild the landmark grid over the merged map (it is the next sweep's association grid) -------------
    {
        double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
        for (int r = tid; r < newL; r += nth) {
            const double x = map_out[r], y = map_out[ld_out + r];
            mnx = fmin(mnx, x); mxx = fmax(mxx, x); mny = fmin(mny, y); mxy = fmax(mxy, y);
        }
        mnx = warp_min(mnx); mny = warp_min(mny); mxx = warp_max(mxx); mxy = warp_max(mxy);
        if ((tid & 31) == 0) { red[0][tid >> 5] = mnx; red[1][tid >> 5] = mny; red[2][tid >> 5] = mxx; red[3][tid >> 5] = mxy; }
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < (nth >> 5); ++w) {
                red[0][0] = fmin(red[0][0], red[0][w]); red[1][0] = fmin(red[1][0], red[1][w]);
                red[2][0] = fmax(red[2][0], red[2][w]); red[3][0] = fmax(red[3][0], red[3][w]);
            }
            if (newL <= 0) { red[0][0] = red[1][0] = red[2][0] = red[3][0] = 0.0; }
            *geom = fgrid_make_geom(red[0][0], red[1][0], red[2][0], red[3][0], dist_thr, max_cells);
        }
        __syncthreads();
        const FGeom g = *geom;
        const int ncell = g.nx * g.ny;
        for (int c = tid; c <= max_cells; c += nth) cell_cnt[c] = 0;    // (the fill of the pre-merge grid left zeros; be explicit)
        __syncthreads();
        for (int r = tid; r < newL; r += nth) {
            int cx0, cx1, cy0, cy1;
            fgrid_cell_range(g, map_out[r], map_out[ld_out + r], cx0, cx1, cy0, cy1);
            for (int cy = cy0; cy <= cy1; ++cy)
                for (int cx = cx0; cx <= cx1; ++cx) atomicAdd(cell_cnt + cy * g.nx + cx, 1);
        }
        __syncthreads();
        block_exclusive_scan(cell_cnt, cell_start, ncell + 1, wsum);
        for (int c = ncell + 1 + tid; c <= max_cells; c += nth) cell_start[c] = cell_start[ncell];
        __syncthreads();
        for (int r = tid; r < newL; r += nth) {
            const double x = map_out[r], y = map_out[ld_out + r];
            int cx0, cx1, cy0, cy1;
            fgrid_cell_range(g, x, y, cx0, cx1, cy0, cy1);
            for (int cy = cy0; cy <= cy1; ++cy)
                for (int cx = cx0; cx <= cx1; ++cx) {
                    const int c = cy * g.nx + cx;
                    const int p = cell_start[c] + atomicSub(cell_cnt + c, 1) - 1;
                    pts[p] = make_double2(x, y);
                    gidx[p] = r;
                }
        }
        __syncthreads();
        for (int r = tid; r < Lcap; r += nth) {       // landmark records of the merged map
            LmRec rec;
            rec.x = 0.0; rec.y = 0.0; rec.r2 = 0.0; rec.r = 0.0;
            if (r < newL) {
                const double x = map_out[r], y = map_out[ld_out + r];
                const double best = nearest_other_wide(g, cell_start, pts, gidx, r, x, y);
                rec.x = x; rec.y = y; rec.r2 = hint_radius2(best, 4.0 * thr1sq, thr2_hi); rec.r = __dsqrt_rd(rec.r2);
            }
            lmrec[r] = rec;
        }
    }
}


// ---- time-segment partition (one segment per GPU) ---------------------------------------------------------
// after the run / association kernels: this segment's count of scans with far observations; after the solve: its boundary poses.
// `pose` and `far` select the part written (the two parts may be gathered separately: the poses beside the tail, on another stream)
__global__ void k_seg_pack(const double* __restrict__ x, int64_t ld, int t_lo, int t_hi, const TailState* ts, double* __restrict__ rec, int pose,
                           int far)
{
    const int i = threadIdx.x;
    if (pose && i < 3) {
        rec[i] = x[i * ld + t_lo];
        rec[3 + i] = x[i * ld + max(t_hi - 2, t_lo)];
        rec[6 + i] = x[i * ld + t_hi - 1];
    }
    if (far && i == 9) rec[9] = (double)ts->far_total;
    if (far && i > 9 && i < SEG_REC) rec[i] = 0.0;
}

// after the all-gather: neighbours' boundary poses into this segment's halo columns (0, 1 and T-1), and the
// global numbering of the new labels (exclusive prefix over the ranks of far_total, ICM_SLAM.py:174-182)
__global__ void k_seg_unpack(const double* __restrict__ all, int rank, int world, double* __restrict__ x, int64_t ld, int T, DevState* st,
                             TailState* ts, int Lcap, double4* __restrict__ ppar, int pose, int far)
{
    const int i = threadIdx.x;
    if (pose) {
        if (i < 3) {
            if (rank > 0) {
                const double* l = all + (size_t)(rank - 1) * SEG_REC;
                x[i * ld + 0] = l[3 + i];
                x[i * ld + 1] = l[6 + i];
            }
            if (rank + 1 < world) x[i * ld + T - 1] = all[(size_t)(rank + 1) * SEG_REC + i];
        }
        // projection parameters of the halo poses (the same expression the owner's solve used: bit-identical)
        if (i == 3 && rank > 0) { const double* l = all + (size_t)(rank - 1) * SEG_REC; ppar[0] = make_ppar(l[3], l[4], l[5]); }
        if (i == 4 && rank > 0) { const double* l = all + (size_t)(rank - 1) * SEG_REC; ppar[1] = make_ppar(l[6], l[7], l[8]); }
        if (i == 5 && rank + 1 < world) { const double* l = all + (size_t)(rank + 1) * SEG_REC; ppar[T - 1] = make_ppar(l[0], l[1], l[2]); }
    }
    if (far && i == 0) {
        int base = 0, total = 0;
        for (int r = 0; r < world; ++r) {
            const int f = (int)all[(size_t)r * SEG_REC + 9];
            if (r < rank) base += f;
            total += f;
        }
        ts->label_base = base;
        st->n_far_scans = total;
        st->raw_l = st->lact0 + total;
        if (st->lact0 + total > Lcap) st->status = ST_LABEL_CAP;
    }
}
