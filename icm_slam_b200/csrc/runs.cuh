// runs.cuh -- run records and the steady-state sweep kernel k_runs of the (REDBLACK, NEWTON, PREV) sweep.
//
// A RUN is a maximal group of consecutive kept beams of one scan that hit the same landmark (a trunk seen under ~3 beams).
// Everything the sweep needs from a run's observations is LINEAR in the sum of their body-frame points: with
// R = Rot(theta_t - pi/2), p = pose position, y = landmark (tras_rot_z ICM_SLAM.py:465-480, Mapa.actualizar :191-194, the
// energy's observation term sensors.py:194-204),
//     sum_i (w_i - y)            = R sum(b) + n (p - y)            -> the landmark update (running mean == sum / count)
//     sum_i (y - p), (y - p) (x) b_i = n (y - p), (y - p) (x) sum(b)   -> the six landmark moments of the pose's normal equations.
// So a run is kept as ONE 24-byte record (sum(b), n, label, a bound rho on |b_i - centroid|), built by the association
// kernel (assoc_tiles.cuh) whenever labels are (re)computed, and a sweep whose labels did not change reads ~0.31 records
// per observation instead of the observations themselves.
//
// "Did not change" is PROVEN every sweep, run by run, against the current poses and map: the landmark record carries the
// radius r inside which an observation is provably nearest to that landmark and inside the gate (tail.cuh hint_radius2);
// |w_i - y| <= |w_c - y| + |b_i - c| <= |S| / n + rho with S = sum_i (w_i - y), so |S| <= n (r - rho) certifies every label
// of the run exactly as the per-observation hint test would; a far run (its scan creates a label) is certified far through
// the landmark grid (run_provably_far).  A scan with a run that fails is marked dirty; the association kernel re-associates
// dirty tiles observation by observation in the same sweep and commits the dirty scans.
//
// LAYOUT: lanes are SCANS.  A slice is 32 scans of a tile (the tile's scans sorted by their number of runs, so that the lanes
// of a warp finish together: tile_perm); run k of the slice's scan j lives at slot
// (slice * maxr + k) * 32 + j of two arrays (sum(b): 16 B, packed label / slot / rho / n: 8 B), maxr = the largest number of
// kept beams of a scan.  A warp walks one slice, step k = run k of each of its 32 scans: the loads of a step are contiguous,
// slots past a scan's last run are never written nor read, and every lane accumulates ITS scan's moments in registers in run
// order -- no cross-lane reduction, and a result that depends on nothing but the scan (bit-identical for any tiling or GPU
// count).  The record names its landmark by the SLOT it has in the tile's table (assigned when the records were built): the
// block stages the landmark records of its slots in shared memory once, so a step's landmark look-up is a shared-memory read,
// and the fixed-point statistics of a run go to the slot's sums there -- 64-bit sums as two carry-free 32-bit limbs, so the adds
// are plain non-returning shared-memory atomics.  The block then adds one int64 pair + count per (tile, landmark) to the global
// statistics: integer addition is associative, so the landmark update is bit-reproducible as well.
#pragma once
#include "common.cuh"
#include "assoc.cuh"
#include "fastgrid.cuh"
#include "tail.cuh"

#define RT_TILE 128         // scans per record tile (= 4 slices = one block of k_runs)
#define RT_SLICES (RT_TILE / 32)
#define RT_RHO_UNIT 2048.0  // rho is kept as a 16-bit count of 1/2048 m (rounded up); RT_RHO_INF: not provable
#define RT_RHO_INF 65535
#define RUN_FAR 0xffffffu   // label field of a run of far observations (its scan creates a new label, ICM_SLAM.py:172-182)
#define RUN_MAX_LABEL 0xfffff0
#define RS_SLOTS 128        // landmark slots of a tile's statistics table; slot RS_NOSLOT: straight to the global sums
#define RS_NOSLOT 255
#define RS_MAX_ADDS 500     // runs per slot and tile (enforced when the records are built): with every one of them added and
                            // taken back once, a low limb stays below 2^32
#define RS_LO_BITS 22       // a sum is kept as (low 22 bits: unsigned limb, the rest: signed limb)
#define RS_MAX_BEAMS 255    // beams of a run that may use a slot: |S| <= n dist_thr, so its fixed-point value stays below 2^42 and
                            // the high limb below 2^20 * 1000 (longer runs go straight to the global sums)

#define RUN_RING 4          // steps of a slice in flight (cp.async ring, steady-state kernel)

// what a block keeps in shared memory for its tile: the statistics table and the landmark records of the table's slots
struct TileSmem {
    unsigned acc[RS_SLOTS][5];     // per slot: sum x (low, high limb), sum y (low, high limb), beams
    double2 lxy[RS_SLOTS];         // the slot's landmark
    double lr[RS_SLOTS];           // ... and its proven radius
};

// the records of the next RUN_RING steps of a warp's slice, brought in with cp.async: every lane copies and reads its own column
struct SliceRing {
    double2 sb[RUN_RING][32];
    int2 mt[RUN_RING][32];
};

__device__ __forceinline__ void ring_issue(SliceRing* R, const double2* sbp, const int2* mtp, int k, int nr, int lane)
{
    if (k < nr) {       // (nr = the slice's reserved steps for the first RUN_RING issues: they start before the scan's own count is known)
        const uint32_t d0 = (uint32_t)__cvta_generic_to_shared(&R->sb[k % RUN_RING][lane]);
        const uint32_t d1 = (uint32_t)__cvta_generic_to_shared(&R->mt[k % RUN_RING][lane]);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d0), "l"(sbp + (size_t)k * 32) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d1), "l"(mtp + (size_t)k * 32) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}

// packed half of a run record: x = label (24 bits) | slot << 24, y = rho code (16 bits) | beams << 16
__device__ __forceinline__ int2 run_meta_pack(int label, int slot, int rho_code, int n)
{
    return make_int2((int)(((unsigned)(label < 0 ? (int)RUN_FAR : label) & 0xffffffu) | ((unsigned)slot << 24)),
                     (int)((unsigned)rho_code | ((unsigned)n << 16)));
}

struct RunParams {
    int t_start, t_hi;                    // record tiles cover scans [t_start, t_hi): t_start = t_lo, or t_lo - 1 with a halo scan
    int halo_t;                           // the halo scan of a time segment (moments only: its statistics belong to the previous segment), or -1
    int maxr;                             // steps reserved per slice (>= runs of any scan)
    const double4* ppar;                  // projection parameters of the input poses (solve.cuh make_ppar)
    const LmRec* lmrec;                   // landmarks by label: position, hint radius^2, hint radius
    double2* rec_sb; int2* rec_meta;      // run records, slot (slice * maxr + k) * 32 + lane
    unsigned short* nruns;                // runs of each scan
    unsigned short* pos_nruns;            // RT_TILE entries per tile: runs of the scan at each (slice, lane) position
    unsigned char* tile_perm;             // RT_TILE entries per tile: the scan (relative to the tile) worked by each (slice, lane) position --
                                          // scans sorted by their number of runs, so that the lanes of a warp finish together
    int* tile_epoch;                      // label-numbering epoch the tile's records belong to
    double* dyn;                          // 6 doubles per pose: (Yx, Mxx, Mxy, Yy, Myx, Myy)
    long long* fsum_x; long long* fsum_y; int* cnt;   // per previous-map landmark statistics (fixed point)
    double fix_scale;
    int* tile_slots; int* tile_nslots;    // RS_SLOTS labels per tile: which landmark each slot of its statistics table stands for; slots in use
    FarRec* far_list; TailState* ts; unsigned* farbits;   // scans with far observations (each creates one label)
    DevState* st; int L_in;                               // the sweep's state, reset by the first block (tail.cuh sweep_begin_state)
    int slice0;                                           // first slice of this launch (a host-memory sweep launches the tiles in chunks)
    int* scan_dirty; int* tile_flag; int* dirty_list;     // steady state: what failed validation (tile_flag: 1 some scans, 2 all)
    const FGeom* geom; const int* cell_start; const double2* gpts;   // the landmark grid (fastgrid.cuh), for the far runs
    double dist_thr;
    Freeze fz;                            // a frozen trajectory's scans commit nothing (no moments, statistics or far records)
};

// A far run stays far if no landmark can be within the gate of any of its observations.  Every observation lies within rho of
// the run's centroid wc; if the square wc +- rho falls into ONE grid cell, that cell's list holds every landmark within thr1 >
// dist_thr of every observation (replicated binning, fastgrid.cuh), and a landmark e with |e - wc| > dist_thr + rho is
// farther than dist_thr from all of them: amin > dist_thr (ICM_SLAM.py:172) for the whole run, as the full search would find.
__device__ __forceinline__ bool run_provably_far(const RunParams& p, double wx, double wy, double rho)
{
    const FGeom g = *p.geom;
    const double r = rho * (1.0 + 1e-6) + 1e-9;
    const int cx0 = min(max(__double2int_rd((wx - r - g.x0) * g.inv_h), 0), g.nx - 1), cx1 = min(max(__double2int_rd((wx + r - g.x0) * g.inv_h), 0), g.nx - 1);
    const int cy0 = min(max(__double2int_rd((wy - r - g.y0) * g.inv_h), 0), g.ny - 1), cy1 = min(max(__double2int_rd((wy + r - g.y0) * g.inv_h), 0), g.ny - 1);
    if (cx0 != cx1 || cy0 != cy1) return false;
    const int c = cy0 * g.nx + cx0;
    const double lim = p.dist_thr * (1.0 + 1e-9) + r, lim2 = lim * lim;
    const int ke = __ldg(p.cell_start + c + 1);
    for (int k = __ldg(p.cell_start + c); k < ke; ++k) {
        const double2 e = __ldg(p.gpts + k);
        if (!(fma(e.x - wx, e.x - wx, (e.y - wy) * (e.y - wy)) > lim2)) return false;
    }
    return true;
}

// The run's statistics S = sum_i (w_i - y) in fixed point -> the tile's table in shared memory (sign = -1 takes a
// contribution back: the limbs are linear).
__device__ __forceinline__ void run_statistics(const RunParams& p, TileSmem& S, int label, int slot, double Sx, double Sy, int n, int sign)
{
    long long vx = __double2ll_rn(Sx * p.fix_scale), vy = __double2ll_rn(Sy * p.fix_scale);
    if (sign < 0) { vx = -vx; vy = -vy; n = -n; }
    if (slot != RS_NOSLOT) {
        const unsigned m = (1u << RS_LO_BITS) - 1u;
        atomicAdd(&S.acc[slot][0], (unsigned)vx & m); atomicAdd((int*)&S.acc[slot][1], (int)(vx >> RS_LO_BITS));
        atomicAdd(&S.acc[slot][2], (unsigned)vy & m); atomicAdd((int*)&S.acc[slot][3], (int)(vy >> RS_LO_BITS));
        atomicAdd((int*)&S.acc[slot][4], n);
    } else {
        atomicAdd((unsigned long long*)(p.fsum_x + label), (unsigned long long)vx);
        atomicAdd((unsigned long long*)(p.fsum_y + label), (unsigned long long)vy);
        atomicAdd(p.cnt + label, n);
    }
}

// the tile's table -> the global statistics: one int64 pair + count per landmark the tile saw (call between block barriers)
__device__ __forceinline__ void stats_flush(const RunParams& p, TileSmem& S, int tile, int nslots)
{
    for (int h = threadIdx.x; h < nslots; h += blockDim.x) {
        const int c = (int)S.acc[h][4];
        const long long vx = ((long long)(int)S.acc[h][1] << RS_LO_BITS) + (long long)S.acc[h][0];
        const long long vy = ((long long)(int)S.acc[h][3] << RS_LO_BITS) + (long long)S.acc[h][2];
        if (c != 0 || vx != 0 || vy != 0) {
            const int label = p.tile_slots[(size_t)tile * RS_SLOTS + h];
            atomicAdd((unsigned long long*)(p.fsum_x + label), (unsigned long long)vx);
            atomicAdd((unsigned long long*)(p.fsum_y + label), (unsigned long long)vy);
            atomicAdd(p.cnt + label, c);
        }
    }
}

// clears the table and stages the landmark records of the tile's slots (call before a block barrier)
__device__ __forceinline__ void tile_stage(const RunParams& p, TileSmem& S, int tile, int nslots)
{
    for (int h = threadIdx.x; h < nslots; h += blockDim.x) {
        const int label = p.tile_slots[(size_t)tile * RS_SLOTS + h];
        const double2* lp = reinterpret_cast<const double2*>(p.lmrec + label);
        S.lxy[h] = __ldg(lp);
        S.lr[h] = __ldg(lp + 1).y;
#pragma unroll
        for (int k = 0; k < 5; ++k) S.acc[h][k] = 0u;
    }
}

// everything one run contributes, from its record and the pose / landmark it names
struct RunEval {
    double Sx, Sy;          // sum of (observation - landmark)
    double rwx, rwy;        // sum of the rotated beams
    double yx, yy;          // landmark - pose
    double r;               // the landmark's proven radius
};

__device__ __forceinline__ RunEval run_eval(const RunParams& p, const TileSmem& S, const double2 sb, int label, int slot, bool matched, double nd,
                                            const double4 pp)
{
    RunEval e;
    double2 lm = make_double2(0.0, 0.0);
    e.r = 0.0;
    if (matched) {
        if (slot != RS_NOSLOT) { lm = S.lxy[slot]; e.r = S.lr[slot]; }       // (staged with the tile)
        else {
            const double2* lp = reinterpret_cast<const double2*>(p.lmrec + label);
            lm = __ldg(lp); e.r = __ldg(lp + 1).y;
        }
    }
    e.rwx = fma(pp.w, sb.x, -pp.z * sb.y); e.rwy = fma(pp.z, sb.x, pp.w * sb.y);
    e.yx = lm.x - pp.x; e.yy = lm.y - pp.y;
    e.Sx = e.rwx - nd * e.yx; e.Sy = e.rwy - nd * e.yy;
    return e;
}

// One slice (32 scans, one per lane) by one warp.  STEADY: every run is certified before it is committed; a scan with a run
// that cannot be certified takes back what it committed, is marked dirty and returns false for its lane.  !STEADY (the
// association kernel has just written the records): no certification; only the scans with commit_all or a dirty flag are
// committed.  FZ: the scans of frozen trajectories (p.fz) commit nothing (compiled out of the steady kernel of the plain sweep).
template <bool STEADY, bool FZ>
__device__ __forceinline__ bool process_slice(const RunParams& p, TileSmem& S, int slice, int tile, bool commit_all, SliceRing* ring = nullptr)
{
    const int lane = threadIdx.x & 31;
    const size_t base = (size_t)slice * p.maxr * 32 + lane;
    const double2* sbp = p.rec_sb + base;
    const int2* mtp = p.rec_meta + base;
    if (ring) {       // the first steps' records start their way before anything else is known about the slice
#pragma unroll
        for (int k = 0; k < RUN_RING; ++k) ring_issue(ring, sbp, mtp, k, p.maxr, lane);
    }
    const size_t ppos = (size_t)tile * RT_TILE + (slice - tile * RT_SLICES) * 32 + lane;
    const int lt = p.tile_perm[ppos];
    const int nr0 = p.pos_nruns[ppos];
    const int t = p.t_start + tile * RT_TILE + lt;
    const bool in = t < p.t_hi && !(FZ && p.fz.scan(t));
    const int nr = in ? nr0 : 0;
    const bool halo = t == p.halo_t;
    bool commit = in && nr > 0;
    if (!STEADY) commit = commit && (commit_all || p.scan_dirty[t] != 0);
    double4 pp = make_double4(0.0, 0.0, 0.0, 1.0);
    if (nr > 0) pp = ldg_ppar(p.ppar + t);
    double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0, m4 = 0.0, m5 = 0.0;
    double nfar = 0.0, fsx = 0.0, fsy = 0.0, FBx = 0.0, FBy = 0.0;
    bool ok = true;
    int kfail = 0;
    // (the records of the next steps are in flight while a step is worked: RUN_RING steps through the cp.async ring in the
    //  steady-state kernel, one step in registers otherwise)
    double2 sb = make_double2(0.0, 0.0);
    int2 mt = make_int2(0, 0);
    if (!ring && 0 < nr) { sb = __ldcg(sbp); mt = __ldcg(mtp); }
    const int steps = __reduce_max_sync(FULLMASK, nr);      // (also orders the staging of the tile's table before its first use)
    __syncwarp();
    for (int k = 0; k < steps; ++k) {
        double2 sb_c = sb;
        int2 mt_c = mt;
        if (ring) {
            asm volatile("cp.async.wait_group %0;" ::"n"(RUN_RING - 1) : "memory");
            sb_c = ring->sb[k % RUN_RING][lane]; mt_c = ring->mt[k % RUN_RING][lane];
            ring_issue(ring, sbp, mtp, k + RUN_RING, nr, lane);
        } else if (k + 1 < nr) { sb = __ldcg(sbp + (size_t)(k + 1) * 32); mt = __ldcg(mtp + (size_t)(k + 1) * 32); }
        if (k < nr && commit && ok) {
            const unsigned lab24 = (unsigned)mt_c.x & 0xffffffu;
            const bool matched = lab24 != RUN_FAR;
            const int label = (int)lab24, slot = (int)((unsigned)mt_c.x >> 24);
            const int rcode = (int)((unsigned)mt_c.y & 0xffffu), n = (int)((unsigned)mt_c.y >> 16);
            const double nd = (double)n;
            const RunEval e = run_eval(p, S, sb_c, label, slot, matched, nd, pp);
            if (STEADY) {
                const double rho = (double)rcode * (1.0 / RT_RHO_UNIT);
                if (rcode >= RT_RHO_INF) ok = false;
                else if (matched) { const double a = (e.r - rho) * nd; ok = a > 0.0 && fma(e.Sx, e.Sx, e.Sy * e.Sy) <= a * a * (1.0 - 1e-9); }
                else ok = run_provably_far(p, pp.x + e.rwx / nd, pp.y + e.rwy / nd, rho);
                if (!ok) kfail = k;
            }
            if (ok) {
                if (matched) {
                    m0 = fma(nd, e.yx, m0); m1 = fma(e.yx, sb_c.x, m1); m2 = fma(e.yx, sb_c.y, m2);
                    m3 = fma(nd, e.yy, m3); m4 = fma(e.yy, sb_c.x, m4); m5 = fma(e.yy, sb_c.y, m5);
                    if (!halo) run_statistics(p, S, label, slot, e.Sx, e.Sy, n, 1);
                } else {      // far run: statistics of the scan's new label (ICM_SLAM.py:174-194)
                    nfar += nd; fsx += fma(nd, pp.x, e.rwx); fsy += fma(nd, pp.y, e.rwy); FBx += sb_c.x; FBy += sb_c.y;
                }
            }
        }
    }
    if (STEADY && !ok) {
        // take back the statistics of the scan's runs before the one that failed; the association kernel commits the scan
        if (!halo) {
            for (int k = 0; k < kfail; ++k) {
                const double2 s2 = __ldcg(sbp + (size_t)k * 32);
                const int2 m2_ = __ldcg(mtp + (size_t)k * 32);
                const unsigned lab24 = (unsigned)m2_.x & 0xffffffu;
                if (lab24 == RUN_FAR) continue;
                const int n = (int)((unsigned)m2_.y >> 16);
                const int slot = (int)((unsigned)m2_.x >> 24);
                const RunEval e = run_eval(p, S, s2, (int)lab24, slot, true, (double)n, pp);
                run_statistics(p, S, (int)lab24, slot, e.Sx, e.Sy, n, -1);
            }
        }
        p.scan_dirty[t] = 1;
        if (atomicCAS(p.tile_flag + tile, 0, 1) == 0) p.dirty_list[atomicAdd(&p.ts->n_dirty, 1)] = tile;
        return false;
    }
    if (commit) {
        // the scan's totals: far observations see the mean of the scan's new label (PREV view), the scan is registered as
        // label-creating, and the six moments go to the solve
        if (nfar > 0.0) {
            const double yx = fsx / nfar - pp.x, yy = fsy / nfar - pp.y;
            m0 += nfar * yx; m3 += nfar * yy;
            m1 = fma(yx, FBx, m1); m2 = fma(yx, FBy, m2);
            m4 = fma(yy, FBx, m4); m5 = fma(yy, FBy, m5);
            if (!halo) {
                FarRec r;
                r.t = t; r.rank = 0; r.n = (int)nfar; r.pad = 0; r.sx = fsx; r.sy = fsy;
                p.far_list[atomicAdd(&p.ts->far_count, 1)] = r;
                atomicOr(p.farbits + (size_t)tile * 4 + (lt >> 5), 1u << (lt & 31));
            }
        }
        double2* d = reinterpret_cast<double2*>(p.dyn + (size_t)t * 6);
        d[0] = make_double2(m0, m1); d[1] = make_double2(m2, m3); d[2] = make_double2(m4, m5);
    }
    return true;
}

#define RUNS_THREADS 32

// steady state: one WARP per slice and block (no block barrier: a slice that needs more steps than its neighbours holds nobody
// up); every block stages its tile's slot table
template <bool FZ>      // FZ: a batch with frozen trajectories; 24 resident blocks per SM (80 registers)
__global__ void __launch_bounds__(RUNS_THREADS, 24)
k_runs(const RunParams p)
{
    __shared__ TileSmem S;
    __shared__ SliceRing ring;
    const int slice = p.slice0 + blockIdx.x, tile = slice / RT_SLICES;
    if (slice == 0 && threadIdx.x == 0) { sweep_begin_state(p.st, p.L_in); trace_mark(p.ts, 0); }      // (nothing in this launch reads it)
    const int nslots = p.tile_nslots[tile];
    if (p.tile_epoch[tile] != p.ts->epoch) {      // no records for this label numbering: the whole tile goes to the association kernel
        if (threadIdx.x == 0 && slice == tile * RT_SLICES) { p.tile_flag[tile] = 2; p.dirty_list[atomicAdd(&p.ts->n_dirty, 1)] = tile; }
        return;
    }
    tile_stage(p, S, tile, nslots);      // (its two dependent loads overlap those of process_slice's prologue: no barrier in between)
    process_slice<true, FZ>(p, S, slice, tile, true, &ring);
    __syncwarp();
    stats_flush(p, S, tile, nslots);
}

// every tile to the association kernel (ICMSLAM_RUNS=0: no steady-state shortcut)
__global__ void k_all_dirty(int* __restrict__ tile_flag, int* __restrict__ dirty_list, TailState* ts, int n_tiles, DevState* st, int L_in)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_tiles) { tile_flag[i] = 2; dirty_list[i] = i; }
    if (i == 0) { ts->n_dirty = n_tiles; sweep_begin_state(st, L_in); }
}
