// assoc_tiles.cuh -- k_assoc_tiles: data association observation by observation + construction of the run records.
//
// Runs over the tiles the steady-state kernel (runs.cuh k_runs) could not certify: every tile on the first sweep of a map
// chain or after landmarks were renumbered, afterwards only tiles with a run outside its landmark's proven radius or with far
// observations.  For every scan of the tile (sensors.py:146-154 restated per SURVEY.md App. A):
//   * the tile's contiguous slice of the observation records (bx, by) and last sweep's labels are staged in shared memory
//     with TMA bulk copies (cp.async.bulk + mbarrier); a tile whose observations exceed the budget goes in chunks of whole
//     scans;
//   * phase A -- LANES OVER CONSECUTIVE OBSERVATIONS (four per lane in flight): projection with the sweep's input pose
//     (tras_rot_z, ICM_SLAM.py:465-480, numpy's exact operation order); last sweep's label of the same observation is
//     accepted iff the point lies inside the landmark's proven-nearest radius (tail.cuh hint_radius2), else the landmark grid
//     (fastgrid.cuh) gives the nearest landmark by squared distance with the rooted values formed only inside a 2^-50 tie
//     window, and the gate s > thr2_hi <=> sqrt(s) > dist_thr: bit-exact cdist + argmin + gate (ICM_SLAM.py:169-172);
//   * pass 1 -- THREAD PAIR PER SCAN: each maximal group of beams with the same label becomes a run (sum of the body-frame
//     points, beam count, a bound rho on the distance of a beam from the centroid, runs.cuh), written to the scan's column of
//     its slice of the record arrays together with the landmark's slot in the tile's statistics table;
//   * the slices are then processed by the SAME code as the steady state (process_slice), so moments and statistics do not
//     depend on which of the two kernels handled a scan.
#pragma once
#include "common.cuh"
#include "assoc.cuh"
#include "fastgrid.cuh"
#include "tail.cuh"
#include "runs.cuh"

#define AT_THREADS (2 * RT_TILE)   // a thread pair per scan of the tile
#define AT_WARPS (AT_THREADS / 32)
#define AT_U 4                     // observations per lane in flight in phase A (pend bitmask: 64 / AT_U iterations per warp)
#define AT_OBS_BYTES 23            // staged bytes per observation: (bx, by) 16, label 4, cell entry count 2, scan 1
static_assert(AT_THREADS >= 32 * RT_SLICES, "a tile's slices are processed by the first warps of the block");
#define AT_HASH 256                // positions of the tile's landmark -> slot hash

struct AssocParams {
    int first_halo;                       // the first scan of tile 0 is the halo scan of a time segment (moments only)
    int T;                                // columns of the handle's trajectory
    const int* off;                       // CSR offsets of the kept observations (T + 1)
    const double2* bxy;                   // body-frame observations (bx, by), CSR order
    DevCfg cfg;
    double thr2_hi;                       // largest s with sqrt_rn(s) <= dist_thr
    const DevState* st;
    const FGeom* geom;
    const int* cell_start; const double2* gpts; const int* gidx;
    const int* remap;                     // last sweep's label -> this map's label (hints)
    int hints;                            // c[] holds last sweep's labels for this map chain
    int* c;                               // labels per observation (out)
    int obs_cap;                          // shared-memory capacity in observations
    int skip_hints;                       // debug (ICMSLAM_HINTS=0)
    int n_tiles; int* blk_prefix; int Lcap; unsigned long long* bb;      // for the scan of the far counts (tail.cuh far_scan_block)
    DevState* stw;                        // (= st, writable: the sweep's label bookkeeping)
    P2PDev p2p;                           // peer windows of a time-segmented run (p2p.cuh): the far count goes straight to every rank
    int final;                            // last launch of the sweep (a host-memory sweep launches one per chunk of tiles, each over the
                                          // tiles that turned dirty since the one before): scan the far counts
    RunParams R;
};

struct __align__(16) AssocSmem {
    double2 pp[RT_TILE];           // projection origin of each scan (self.x0 for scan 0)
    double2 rsc[RT_TILE];          // (sin, cos) of (projection heading - pi/2)
    int off[RT_TILE + 4];          // off[t] of the tile's scans
    // the tile's statistics slots: a small hash (landmark -> slot) filled while the runs are counted; slots are numbered densely
    int hkey[AT_HASH];             // landmark at each hash position (-1: free)
    int hid[AT_HASH];              // its slot (-1: not numbered yet)
    int hcnt[AT_HASH];             // runs that name it
    int slot_label[RS_SLOTS];      // landmark of each slot
    int nslots;
    int rtot[RT_TILE];             // runs of each scan
    unsigned char pos[RT_TILE];    // (slice, lane) position of each scan: its rank by number of runs (identity when the tile is staged in pieces)
    TileSmem tile;                 // the statistics table and the staged landmark records (runs.cuh)
    unsigned long long mbar;
};

// registers landmark `label` in the tile's hash (open addressing, at most 8 probes; a crowded table leaves it out)
__device__ __forceinline__ void slot_insert(AssocSmem& S, int label)
{
    unsigned h = ((unsigned)label * 2654435761u) >> 24;
#pragma unroll 1
    for (int q = 0; q < 8; ++q) {
        int key = ((volatile int*)S.hkey)[h];
        if (key == -1) {
            const int prev = atomicCAS(&S.hkey[h], -1, label);
            key = (prev == -1) ? label : prev;
        }
        if (key == label) return;
        h = (h + 1) & (AT_HASH - 1);
    }
}

// slot of landmark `label` for a run of n beams; RS_NOSLOT when the landmark is not in the table, the run is too long for the
// limbs or the slot already serves RS_MAX_ADDS runs (their statistics go straight to the global sums)
__device__ __forceinline__ int slot_of(AssocSmem& S, int label, int n)
{
    if (n > RS_MAX_BEAMS) return RS_NOSLOT;
    unsigned h = ((unsigned)label * 2654435761u) >> 24;
#pragma unroll 1
    for (int q = 0; q < 8; ++q) {
        const int key = S.hkey[h];
        if (key == label) {
            const int id = S.hid[h];
            return (id >= 0 && id < RS_SLOTS && atomicAdd(&S.hcnt[h], 1) < RS_MAX_ADDS) ? id : RS_NOSLOT;
        }
        if (key == -1) return RS_NOSLOT;
        h = (h + 1) & (AT_HASH - 1);
    }
    return RS_NOSLOT;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_wait(uint32_t mb, uint32_t parity)
{
    uint32_t done = 0;
    while (!done) {
        asm volatile("{\n.reg .pred P1;\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\nselp.u32 %0, 1, 0, P1;\n}"
                     : "=r"(done) : "r"(mb), "r"(parity) : "memory");
    }
}

__global__ void __launch_bounds__(AT_THREADS, 2)
k_assoc_tiles(const AssocParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    AssocSmem& S = *reinterpret_cast<AssocSmem*>(smem_raw);
    double2* sb = reinterpret_cast<double2*>(smem_raw + sizeof(AssocSmem));             // staged observations; later run sums
    int* sbk_raw = reinterpret_cast<int*>(sb + p.obs_cap);                               // hints in (TMA), labels out; +4 ints of alignment slack
    unsigned short* srn = reinterpret_cast<unsigned short*>(sbk_raw + p.obs_cap + 4);    // phase A: entries of the observation's grid cell
    unsigned char* slt = reinterpret_cast<unsigned char*>(srn + p.obs_cap);              // scan (relative to the tile) of each observation

    const RunParams& R = p.R;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t mb = smem_u32(&S.mbar);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mb));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint32_t parity = 0;
    FGrid G;
    G.g = *p.geom;
    G.cell_start = p.cell_start; G.pts = p.gpts; G.idx = p.gidx;
    const int lsearch = p.st->lsearch;
    const bool have_map = lsearch > 0;
    const bool ident = R.ts->remap_identity != 0;
    const bool use_hints = p.hints != 0 && have_map && !p.skip_hints;
    const int epoch = R.ts->epoch;
    const int n_dirty = R.ts->n_dirty;
    const int d_first = R.ts->dirty_done;
    if (blockIdx.x == 0 && tid == 0) trace_mark(R.ts, 1);
    const int q = tid >> 1, sub = tid & 1;          // scan of the tile worked by this thread pair, and the thread's half of it

    for (int di = d_first + blockIdx.x; di < n_dirty; di += gridDim.x) {
        const int tile = R.dirty_list[di];
        const int tb = R.t_start + tile * RT_TILE;
        const int nsc = min(RT_TILE, R.t_hi - tb);
        const bool commit_all = R.tile_flag[tile] == 2;
        const bool halo_tile = p.first_halo && tile == 0;
        // ---- tile loads -------------------------------------------------------------------------------------------
        for (int li = tid; li <= nsc; li += AT_THREADS) S.off[li] = p.off[tb + li];
        if (tid < nsc) {
            const double4 pq = ldg_ppar(R.ppar + tb + tid);
            S.pp[tid] = make_double2(pq.x, pq.y); S.rsc[tid] = make_double2(pq.z, pq.w);
        }
        for (int hh = tid; hh < AT_HASH; hh += AT_THREADS) { S.hkey[hh] = -1; S.hid[hh] = -1; S.hcnt[hh] = 0; }
        if (tid == 0) S.nslots = 0;
        __syncthreads();
        // ---- chunks of whole scans whose observations fit the shared-memory budget (normally one) -----------------
        for (int c_lo = 0; c_lo < nsc;) {
            int c_hi = nsc - 1;
            if (S.off[nsc] - S.off[c_lo] > p.obs_cap) {
                int lo = c_lo, hi = nsc - 1;
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (S.off[mid + 1] - S.off[c_lo] <= p.obs_cap) lo = mid; else hi = mid - 1;
                }
                c_hi = lo;
            }
            const int co = S.off[c_lo], ce = S.off[c_hi + 1];
            const int co4 = co & ~3;                         // 16-byte aligned start of the labels' slice
            int* sbk = sbk_raw + (co - co4);                 // label of each observation (-1 far), same slot as its hint
            if (tid == 0) {
                const uint32_t bytes = (uint32_t)(ce - co) * 16u;
                const uint32_t hbytes = (use_hints && ce > co) ? (uint32_t)((ce - co4 + 3) & ~3) * 4u : 0u;
                if (bytes + hbytes > 0) {
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes + hbytes) : "memory");
                    if (bytes) asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                            ::"r"(smem_u32(sb)), "l"(p.bxy + co), "r"(bytes), "r"(mb) : "memory");
                    // last sweep's labels of the same observations (the hints) land in the label array itself
                    if (hbytes) asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                             ::"r"(smem_u32(sbk_raw)), "l"(p.c + co4), "r"(hbytes), "r"(mb) : "memory");
                } else {
                    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mb) : "memory");
                }
            }
            // the pair's scan and this thread's half of it (indices relative to the chunk)
            const bool mine = q >= c_lo && q <= c_hi;
            int o = 0, e = 0;
            if (mine) {
                const int so = S.off[q] - co, se = S.off[q + 1] - co;
                const int h1 = (se - so + 1) >> 1;
                o = min(so + sub * h1, se);
                e = min(o + h1, se);
            }
            for (int i = o; i < e; ++i) slt[i] = (unsigned char)q;     // (while the bulk copies are in flight)
            mbar_wait(mb, parity);
            parity ^= 1u;
            __syncthreads();
            // ---- phase A: lanes over consecutive observations (adjacent lanes = adjacent beams), four per lane in flight --
            //   A0 (hints): last sweep's label of the same observation, carried through the filter's renumbering, is
            //       accepted when the observation lies inside the landmark's proven-nearest radius (tail.cuh hint_radius2):
            //       one staged value and one gather instead of the grid search.  Lanes it cannot settle stay pending for
            //   A1: project, locate the grid cell, fetch its entry range     (first level of gathers)
            //   A2: fetch the candidates, pick the nearest, gate, label      (second level of gathers)
            {
                const int m = ce - co;
                const int per = ((((m + AT_WARPS - 1) / AT_WARPS) + AT_U * 32 - 1) / (AT_U * 32)) * (AT_U * 32);
                const int wa = warp * per, wb = min(wa + per, m);
                unsigned long long pend = 0ull;
                int slot = 0;
                for (int b0 = wa; b0 < wb; b0 += AT_U * 32, slot += AT_U) {
                    int h_[AT_U];
                    double wx_[AT_U], wy_[AT_U];
#pragma unroll
                    for (int u = 0; u < AT_U; ++u) {
                        const int i = b0 + u * 32 + lane;
                        h_[u] = -1; wx_[u] = 0.0; wy_[u] = 0.0;
                        if (i < wb && use_hints) {
                            h_[u] = sbk[i];
                            if (h_[u] >= p.cfg.L) h_[u] = -1;          // (labels of scans this handle does not own are not maintained)
                            const double2 bq = sb[i];
                            const int lt = slt[i];
                            const double2 pq = S.pp[lt], rc = S.rsc[lt];
                            wx_[u] = add_rn(__fma_rn(bq.y, -rc.x, mul_rn(bq.x, rc.y)), pq.x);
                            wy_[u] = add_rn(__fma_rn(bq.y, rc.y, mul_rn(bq.x, rc.x)), pq.y);
                        }
                    }
                    if (!ident) {
#pragma unroll
                        for (int u = 0; u < AT_U; ++u) if (h_[u] >= 0) h_[u] = __ldg(p.remap + h_[u]);
                    }
                    double2 q_[AT_U];
                    double r2_[AT_U];
#pragma unroll
                    for (int u = 0; u < AT_U; ++u) {
                        q_[u] = make_double2(0.0, 0.0); r2_[u] = -1.0;
                        if (h_[u] >= 0 && h_[u] < lsearch) {
                            const double2* rp = reinterpret_cast<const double2*>(R.lmrec + h_[u]);
                            q_[u] = __ldg(rp); r2_[u] = __ldg(rp + 1).x;
                        }
                    }
#pragma unroll
                    for (int u = 0; u < AT_U; ++u) {
                        const int i = b0 + u * 32 + lane;
                        if (i < wb) {
                            const double d2 = dist2_rn(q_[u].x - wx_[u], q_[u].y - wy_[u]);
                            if (d2 <= r2_[u]) {
                                sbk[i] = h_[u];
                                if (!ident && !(halo_tile && slt[i] == 0)) p.c[co + i] = h_[u];    // (with the identity renumbering c[] already holds it)
                            } else pend |= 1ull << (slot + u);
                        }
                    }
                }
                const bool any_pend = __any_sync(FULLMASK, pend != 0ull);
                slot = 0;
                for (int b0 = wa; b0 < wb && any_pend; b0 += AT_U * 32, slot += AT_U) {
                    int s_[AT_U], e_[AT_U];
#pragma unroll
                    for (int u = 0; u < AT_U; ++u) {
                        const int i = b0 + u * 32 + lane;
                        s_[u] = 0; e_[u] = 0;
                        if (i < wb && have_map && ((pend >> (slot + u)) & 1ull)) {
                            const double2 bq = sb[i];
                            const int lt = slt[i];
                            const double2 pq = S.pp[lt], rc = S.rsc[lt];
                            const double wx = add_rn(__fma_rn(bq.y, -rc.x, mul_rn(bq.x, rc.y)), pq.x);
                            const double wy = add_rn(__fma_rn(bq.y, rc.y, mul_rn(bq.x, rc.x)), pq.y);
                            const int cc = fgrid_cell(G.g, wx, wy);
                            s_[u] = __ldg(G.cell_start + cc); e_[u] = __ldg(G.cell_start + cc + 1);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < AT_U; ++u) {
                        const int i = b0 + u * 32 + lane;
                        if (i < wb && ((pend >> (slot + u)) & 1ull)) { sbk[i] = s_[u]; srn[i] = (unsigned short)min(e_[u] - s_[u], 65535); }
                    }
                }
                slot = 0;
                for (int b0 = wa; b0 < wb && any_pend; b0 += AT_U * 32, slot += AT_U) {
                    double wx_[AT_U], wy_[AT_U];
                    double2 p_[AT_U];
                    int id_[AT_U], s_[AT_U], n_[AT_U];
#pragma unroll
                    for (int u = 0; u < AT_U; ++u) {
                        const int i = b0 + u * 32 + lane;
                        s_[u] = 0; n_[u] = 0; id_[u] = -1; p_[u] = make_double2(0.0, 0.0); wx_[u] = 0.0; wy_[u] = 0.0;
                        if (i < wb && ((pend >> (slot + u)) & 1ull)) {
                            s_[u] = sbk[i]; n_[u] = srn[i];
                            const double2 bq = sb[i];
                            const int lt = slt[i];
                            const double2 pq = S.pp[lt], rc = S.rsc[lt];
                            // tras_rot_z: numpy's matmul order, acc = a0*b0; acc = fma(a1, b1, acc); + translation
                            wx_[u] = add_rn(__fma_rn(bq.y, -rc.x, mul_rn(bq.x, rc.y)), pq.x);
                            wy_[u] = add_rn(__fma_rn(bq.y, rc.y, mul_rn(bq.x, rc.x)), pq.y);
                            if (n_[u] > 0) { p_[u] = __ldg(G.pts + s_[u]); id_[u] = __ldg(G.idx + s_[u]); }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < AT_U; ++u) {
                        const int i = b0 + u * 32 + lane;
                        if (i < wb && ((pend >> (slot + u)) & 1ull)) {
                            double best;
                            int bid;
                            const int bk = fgrid_scan_pre(G, wx_[u], wy_[u], s_[u], n_[u], p_[u], id_[u], best, bid);
                            const bool far = bk < 0 || best > p.thr2_hi;      // amin > dist_thr (ICM_SLAM.py:172)
                            sbk[i] = far ? -1 : bid;                          // the label (index in the previous map)
                            if (!(halo_tile && slt[i] == 0)) p.c[co + i] = far ? -1 : bid;    // the halo scan is not owned
                        }
                    }
                }
            }
            __syncthreads();     // the labels of the whole chunk are visible to the scan threads
            // ---- pass 1 (thread pair per scan): runs of equal labels -> run records ------------------------------------------
            // Each run goes straight to its slot: column (scan) of the scan's slice, row = index of the run in the scan.  rho: every
            // beam and the centroid lie in the run's bounding box, so the farthest box corner from the centroid bounds
            // |b_i - centroid| (float arithmetic with its rounding covered by the margins, then rounded up to 1/2048 m).
            int nr = 0;
            // (slot0 depends on the scan's position, known after the counting pass below)
            // (the first half's run count is needed for the second half's row offset: count first, then write)
            const bool halo_scan = halo_tile && q == 0;
            if (o < e) {
                int bk = sbk[o];
                if (bk >= 0 && !halo_scan) slot_insert(S, bk);
                for (int i = o + 1; i < e; ++i) {
                    const int b2 = sbk[i];
                    if (b2 != bk) { ++nr; if (b2 >= 0 && !halo_scan) slot_insert(S, b2); }
                    bk = b2;
                }
                ++nr;
            }
            const int nr_other = __shfl_xor_sync(FULLMASK, nr, 1);
            const int rtot = nr + nr_other;
            const bool whole = c_lo == 0 && c_hi == nsc - 1;      // the tile is staged in one piece: every scan's run count is known
            if (sub == 0 && q < RT_TILE) S.rtot[q] = mine ? rtot : 0;
            __syncthreads();
            // number the landmarks that entered the hash in this chunk
            if (tid < AT_HASH && S.hkey[tid] != -1 && S.hid[tid] < 0) {
                const int id = atomicAdd(&S.nslots, 1);
                S.hid[tid] = id;
                if (id < RS_SLOTS) S.slot_label[id] = S.hkey[tid];
            }
            // position of every scan: scans with fewer runs first (stable), so that a warp's 32 scans need about the same
            // number of steps
            if (c_lo == 0 && tid < RT_TILE) {
                int rank = tid;
                if (whole) {
                    const int mine_r = S.rtot[tid];
                    rank = 0;
                    for (int j = 0; j < RT_TILE; ++j) { const int rj = S.rtot[j]; rank += (rj < mine_r) || (rj == mine_r && j < tid); }
                }
                S.pos[tid] = (unsigned char)rank;
                R.tile_perm[(size_t)tile * RT_TILE + rank] = (unsigned char)tid;
                if (whole) R.pos_nruns[(size_t)tile * RT_TILE + rank] = (unsigned short)S.rtot[tid];
            }
            __syncthreads();
            if (o < e) {
                // (the next observation is fetched before the current one is consumed)
                const int ps = S.pos[q];
                const size_t slot0 = ((size_t)(tile * RT_SLICES + (ps >> 5)) * R.maxr) * 32 + (ps & 31);
                int k = sub ? nr_other : 0;
                int run_start = o, bk = sbk[o];
                double2 b = sb[o];
                double Sbx = 0.0, Sby = 0.0;
                float mnx = INFINITY, mxx = -INFINITY, mny = INFINITY, mxy = -INFINITY;
                for (int i = o; i < e; ++i) {
                    const int inx = min(i + 1, e - 1);
                    const double2 bn = sb[inx];
                    const int bkn = sbk[inx];
                    Sbx += b.x; Sby += b.y;
                    const float fx = (float)b.x, fy = (float)b.y;
                    mnx = fminf(mnx, fx); mxx = fmaxf(mxx, fx); mny = fminf(mny, fy); mxy = fmaxf(mxy, fy);
                    if (i + 1 == e || bkn != bk) {
                        const int n = i + 1 - run_start;
                        const float inv = 1.0f / (float)n, cx = (float)Sbx * inv, cy = (float)Sby * inv;
                        const float ex = fmaxf(mxx - cx, cx - mnx), ey = fmaxf(mxy - cy, cy - mny);
                        const float rho = sqrtf(fmaf(ex, ex, ey * ey)) * 1.0001f + 2e-5f;
                        const int rcode = min(__float2int_ru(rho * (float)RT_RHO_UNIT), RT_RHO_INF);
                        const int slot = (bk >= 0 && !halo_scan) ? slot_of(S, bk, n) : RS_NOSLOT;
                        if (k < R.maxr) {
                            R.rec_sb[slot0 + (size_t)k * 32] = make_double2(Sbx, Sby);
                            R.rec_meta[slot0 + (size_t)k * 32] = run_meta_pack(bk, slot, rcode, n);
                        }
                        ++k;
                        run_start = i + 1; Sbx = 0.0; Sby = 0.0; mnx = INFINITY; mxx = -INFINITY; mny = INFINITY; mxy = -INFINITY;
                    }
                    b = bn; bk = bkn;
                }
            }
            if (mine && sub == 0) {
                R.nruns[tb + q] = (unsigned short)rtot;
                if (!whole) R.pos_nruns[(size_t)tile * RT_TILE + q] = (unsigned short)rtot;      // (identity positions)
            }
            c_lo = c_hi + 1;
            if (c_lo < nsc) __syncthreads();   // the next chunk overwrites the staging buffers
        }
        __syncthreads();
        // ---- tile header, then the slices through the same code as the steady state -------------------------------------------
        const int nslots = min(S.nslots, RS_SLOTS);
        if (tid == 0) { R.tile_epoch[tile] = epoch; R.tile_nslots[tile] = nslots; }
        for (int hh = tid; hh < nslots; hh += AT_THREADS) R.tile_slots[(size_t)tile * RS_SLOTS + hh] = S.slot_label[hh];
        __syncthreads();     // the block's records and slot table are visible to its warps
        tile_stage(R, S.tile, tile, nslots);
        __syncthreads();
        if (warp < RT_SLICES) process_slice<false, true>(R, S.tile, tile * RT_SLICES + warp, tile, commit_all);
        __syncthreads();
        stats_flush(R, S.tile, tile, nslots);
        __syncthreads();
        if (tid < nsc) R.scan_dirty[tb + tid] = 0;
        if (tid == 0) R.tile_flag[tile] = 0;
    }
    // ---- the last block to finish numbers the sweep's label-creating scans (every tile's far bits are final by then) ----
    // (the tile loop's shared arrays are free again: no static shared memory, the dynamic allocation is the whole budget)
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        const int last = atomicAdd(&R.ts->assoc_ticket, 1) == (int)gridDim.x - 1;
        if (last) { __threadfence(); R.ts->assoc_ticket = 0; R.ts->dirty_done = p.final ? 0 : n_dirty; }
        S.nslots = last && p.final;
    }
    __syncthreads();
    if (S.nslots) {
        far_scan_block(R.farbits, p.n_tiles, p.blk_prefix, p.stw, R.ts, p.Lcap, p.bb, S.rtot, reinterpret_cast<unsigned char*>(sb), p.obs_cap * 16);
        if (p.p2p.on) {
            __syncthreads();
            p2p_post_far(p.p2p, *(volatile unsigned*)&R.ts->p2p_seq, *(volatile int*)&R.ts->far_total);
        }
    }
}

static size_t assoc_smem_bytes(int obs_cap)   // obs_cap is even
{
    return sizeof(AssocSmem) + (size_t)obs_cap * AT_OBS_BYTES + 16 + 64;
}
