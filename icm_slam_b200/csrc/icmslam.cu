// icmslam.cu -- C ABI (include/icmslam.h) and host orchestration of libicmslam.so.
// One translation unit: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo ...
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <new>
#include <utility>
#include <vector>

#include "common.cuh"
#include "assoc.cuh"
#include "extract.cuh"
#include "pose.cuh"
#include "mapfilter.cuh"
#include "fastgrid.cuh"
#include "tail.cuh"
#include "solve.cuh"
#include "runs.cuh"
#include "assoc_tiles.cuh"
#include "fcluster.h"
#include "pass0.cuh"

#define ASSOC_MAX_OBS 4096      // observations of one scan icmslam_associate accepts (a scan has at most B <= 1024 beams)

// ---- owners of the handle's CUDA resources: each is released by exactly one destructor ------------------------------------
// Nothing is allocated, freed or reassigned inside a graph capture (sweep_core and the fused_part_* functions under
// icmslam_iterate, and the icmslam_seg_* calls a caller captures together with its collectives): a captured graph holds the raw
// pointers, so whatever replaces a buffer a graph can hold calls drop_graphs before the old buffer is freed.
template <typename H, auto Release>
struct Owner {
    H p{};
    Owner() = default;
    Owner(Owner&& o) noexcept : p(o.p) { o.p = H{}; }
    Owner& operator=(Owner&& o) noexcept { if (this != &o) { reset(); p = o.p; o.p = H{}; } return *this; }
    ~Owner() { reset(); }
    void reset() { if (p) Release(p); p = H{}; }
    operator H() const { return p; }
};
using Stream = Owner<cudaStream_t, cudaStreamDestroy>;
using Event = Owner<cudaEvent_t, cudaEventDestroy>;
using GraphExec = Owner<cudaGraphExec_t, cudaGraphExecDestroy>;
using IpcMapping = Owner<void*, cudaIpcCloseMemHandle>;

// `count` elements of T in device memory (or, released with cudaFreeHost, in pinned host memory); alloc() frees what it held first
template <typename T, auto Release>
struct Buf : Owner<T*, Release> {
    cudaError_t alloc(size_t count)
    {
        this->reset();
        const size_t bytes = (count ? count : 1) * sizeof(T);
        const cudaError_t e = Release == cudaFreeHost ? cudaMallocHost((void**)&this->p, bytes) : cudaMalloc((void**)&this->p, bytes);
        if (e != cudaSuccess) this->p = nullptr;
        return e;
    }
    T* operator->() const { return this->p; }
};
template <typename T> using DevBuf = Buf<T, cudaFree>;
template <typename T> using PinnedBuf = Buf<T, cudaFreeHost>;

// A landmark grid (fastgrid.cuh): geometry, per-cell counts (all zero between builds: the fill pass counts them back down) and
// starts, the cell-sorted entries and the bounding box.  A handle has two.  `grid` indexes the map of the fused sweep's chain
// (Chain::grid_map) and is written by the filter chain; a caller other than the fused sweep invalidates ch.grid_map.  The two
// other readers (the generic sweep's association, calc_cambio) build `scratch_grid`.  calc_cambio runs between two fused sweeps
// of icmslam_iterate_until: were it to rebuild `grid`, the next sweep would find its grid stale, rebuild it and void every run
// record.
struct LandmarkGrid {
    DevBuf<FGeom> geom;
    DevBuf<int> cnt, start, idx;
    DevBuf<double2> pts;
    DevBuf<unsigned long long> bb;
    cudaError_t alloc(int cells, size_t entries)
    {
        cudaError_t e = geom.alloc(1);
        if (e == cudaSuccess) e = cnt.alloc((size_t)cells + 2);
        if (e == cudaSuccess) e = start.alloc((size_t)cells + 2);
        if (e == cudaSuccess) e = idx.alloc(entries);
        if (e == cudaSuccess) e = pts.alloc(entries);
        if (e == cudaSuccess) e = bb.alloc(4);
        if (e == cudaSuccess) e = cudaMemset(cnt, 0, ((size_t)cells + 2) * sizeof(int));
        return e;
    }
};

struct icmslam_handle {
    icmslam_config cfg;
    DevCfg dcfg;
    cudaStream_t stream = nullptr;
    Stream own_stream;                   // created with the handle; replaced by icmslam_set_stream
    // the pose solve does not feed the tail (labels, landmark update, Mapa.filtrar): on one GPU the two run concurrently,
    // the solve forked onto a side stream after the association kernel and joined at the end of the sweep (also inside the CUDA graph)
    Stream side_stream; Event ev_fork, ev_join, ev_tail; bool join_pending = false; int overlap_solve = 1;
    char err[512];
    // dataset
    int B = 0, T = 0, precondition = 0;
    int cap_T = 0;        // columns d_scans, d_odo, d_u and d_x have room for (their leading dimension): T after icmslam_load
                          // and after ensure_layout, grown by doubling when icmslam_append brings more
    struct Dataset {      // what icmslam_load allocates (B x cap_T, 3 x cap_T, ...) and ensure_layout sizes by T
        DevBuf<double> d_scans, d_odo, d_u, d_cos, d_sin, d_ang;
        DevBuf<int> d_nfar, d_flag, d_prefix;       // per scan workspace
        DevBuf<double> d_x /*3 x cap_T*/, d_x2 /*3 x T, pose double buffer*/, d_inc /*3 x T odometry increments*/;
        DevBuf<FarRec> d_far_list;
        DevBuf<int> d_blk_prefix;
    } ds;
    // extraction: the CSR arrays cover all T columns once `extracted`; what only the sweeps read follows on demand
    // (ensure_layout: `laid_out`)
    bool extracted = false, laid_out = false;
    int64_t n = 0, n_cap = 0;           // observations, and the room of the per-observation arrays (d_off has cap_T + 1 entries)
    std::vector<int> off_h;             // host copy of the T + 1 offsets
    int n_empty = 0, max_per_scan = 0;
    bool first_empty = false, last_empty = false;
    struct Extraction {   // what icmslam_extract / icmslam_append and ensure_layout allocate (some of it on first use)
        DevBuf<int> d_off, d_beam, d_scan_of;
        DevBuf<double> d_d, d_bx, d_by;
        DevBuf<double2> d_bxy;               // interleaved (bx, by) records for the TMA staging
        // per observation workspace
        DevBuf<int> d_c, d_keys_out, d_iota, d_sorted;
        DevBuf<double> d_seen_x, d_seen_y;
        // fused (REDBLACK, NEWTON, PREV) path: run records (runs.cuh) + association of dirty tiles (assoc_tiles.cuh) + solve (solve.cuh)
        DevBuf<double> d_bm;                 // 6 x T static body-frame moments + beam count
        DevBuf<double4> d_ppar[2];           // projection parameters of the poses in d_x / d_x2 (solve.cuh make_ppar)
        DevBuf<unsigned> d_farbits;          // 4 words per record tile: scans that created a label this sweep
        DevBuf<double2> d_rec_sb; DevBuf<int2> d_rec_meta;   // run records (runs.cuh)
        DevBuf<unsigned short> d_nruns;      // runs of each scan
        DevBuf<unsigned char> d_tile_perm;   // RT_TILE scan positions per record tile (runs.cuh)
        DevBuf<unsigned short> d_pos_nruns;  // ... and the runs of the scan at each position
        DevBuf<int> d_tile_slots, d_tile_nslots;   // RS_SLOTS labels per record tile, slots in use
        DevBuf<int> d_tile_epoch, d_tile_flag, d_dirty_list, d_scan_dirty;
        DevBuf<double> d_dyn;                // 6 landmark moments per pose
    } ex;
    // per label workspace (capacity Lcap)
    int Lcap = 0;
    DevBuf<double> d_sum_x, d_sum_y, d_raw /*2 x Lcap*/, d_counts;
    int* d_cnt = nullptr; DevBuf<int> d_seg;
    DevBuf<int> d_kflag, d_kpos, d_parent, d_nn, d_indflag, d_indpos, d_ind, d_lab, d_used, d_rank;
    DevBuf<double> d_kx, d_ky, d_kc, d_ox, d_oy, d_oc, d_acc;
    DevBuf<double> d_map_in /*2 x Lcap*/, d_map_out /*2 x Lcap*/;
    DevBuf<double> d_tmp_a, d_tmp_b; /* 2 x Lcap scratch for filter_map / calc_cambio inputs */
    // pass 0 as a resumable walk (icmslam_pass0_begin / _advance / _finish): its own map under construction (2 x Lcap) and
    // counts, which no other call writes, and the carried state; on the host the columns walked and x0
    struct Walk {
        DevBuf<double> y, cant;
        DevBuf<Pass0Carry> carry;
        bool on = false;
        int t = 0, lact = 0;
        double x0[3] = {0, 0, 0};
    } walk;
    // state
    DevBuf<DevState> d_st;
    PinnedBuf<DevState> h_st;   // pinned mirror
    int lact_host = 0;          // mirror of landmarks_actuales (valid when !ch.lact_dirty)
    DevBuf<unsigned char> d_cub;
    size_t cub_bytes = 0;
    DevBuf<unsigned char> d_sort_ws;
    size_t sort_bytes = 0;
    bool fused_ok = false;
    int trace_on = 0;                          // ICMSLAM_TRACE=1: %globaltimer marks of the sweep's kernels (icmslam_get_trace)
    int begin_L = 0;                           // landmarks_actuales bound of the sweep being issued (k_sweep_begin / sweep_begin_state)
    int n_tiles_alloc = 0;                     // tiles the per-tile arrays were allocated for
    int n_tiles = 0, n_solve_tiles = 0;        // record tiles (RT_TILE scans) / solve tiles (ST_OWN poses)
    int64_t rec_slots = 0; int rec_maxr = 1;   // run records (runs.cuh)
    DevBuf<TailState> d_ts;
    double thr2_lt = 0.0;        // largest s with sqrt_rn(s) < dist_thr
    DevBuf<LmRec> d_lmrec2[2];                 // landmarks of a map by label (position + hint radius): the current map's in
                                               // d_lmrec2[ch.lm_cur], the tail writes the new map's into the other one
    // the steady tail (tail.cuh k_tail_steady): where every landmark was when the grid was built, a lower bound of its distance to
    // any other landmark then, the positions of its grid entries, per-block calc_cambio partials
    DevBuf<double2> d_gbuild; DevBuf<double> d_nnd0; DevBuf<int4> d_gslots; DevBuf<double> d_cpart; int steady_enable = 1;
    DevBuf<long long> d_sh_x, d_sh_y; DevBuf<int> d_sh_k;      // shadow of the statistics (k_tail_steady clears the live ones)
    // inside the library's own CUDA graph the full chain is the body of an IF node (cudaGraphSetConditional in k_tail_steady)
    bool in_own_capture = false; int use_cond = 1; Stream cap_stream;
    DevBuf<int> d_blk_kept;                    // kept landmarks per block of k_fused_means
    DevBuf<int> d_rawcnt;                      // observation counts of the last fused sweep's raw map (the tail clears d_cnt)
    DevBuf<unsigned long long> d_scan_state;   // block totals of k_cell_scan
    DevBuf<int> d_remap;                // label of the last sweep -> label in the current map
    DevBuf<int> d_klab;                 // raw label of each kept landmark (fast tail)
    // batch of independent trajectories laid end to end (icmslam_set_batch / icmslam_set_batch_lengths): K + 1 column starts,
    // the trajectory of each column, 3 x K first poses; traj_odd: some trajectory starts on an odd column
    int traj_K = 0; bool traj_odd = false; DevBuf<int> d_traj_start, d_traj_of; DevBuf<double> d_x0s;
    // per-trajectory freezing (icmslam_batch_iterate_until): fz.frozen is null outside that call
    Freeze fz = {};
    DevBuf<unsigned char> d_fz_mask, d_fz_need; DevBuf<double> d_fz_slots; DevBuf<int> d_fz_reg; int fz_K = 0;
    int fz_fallbacks = 0;      // sweeps of the last icmslam_batch_iterate_until that needed the full calc_cambio search
    DevBuf<double> d_aobs; DevBuf<int> d_ac;   // icmslam_associate: one scan's observations (2 x ASSOC_MAX_OBS) and labels
    double thr1sq = 0.0;
    struct GraphSlot { GraphExec exec; const double* src = nullptr; const double* map_in = nullptr; double x0[3] = {0, 0, 0}; double tol = 0; int maxit = 0; int lm = 0; Freeze fz = {};
                       int launches = 0; };      // kernels of this library in the graph
    GraphSlot graphs[4];
    int use_graph = 1;
    int use_runs = 1;            // ICMSLAM_RUNS=0: every tile goes through the association kernel every sweep (no steady-state shortcut)
    int assoc_blocks = 0;        // grid of the (persistent) association kernel
    long long *d_fsum_x = nullptr, *d_fsum_y = nullptr;
    int fg_cells = 0;            // cell budget of the landmark grids (host constant)
    LandmarkGrid grid, scratch_grid;
    int obs_cap = 0, max_tile_obs = 0;
    // host-memspace sweeps: copy of the map returned by the last one (a caller that feeds it back continues the device-side
    // map chain: grid, hints and labels stay valid, sensors.py:315 `mapa_viejo = mapa_refinado`)
    PinnedBuf<double> h_map_pin;      // pinned 2 x Lcap: the map the last host-memory sweep returned (read back in one async copy; what
    int last_map_L = -1;              // the next call's mapa_viejo is compared with to continue the device-side map chain)
    int64_t bytes_h2d = 0, bytes_d2h = 0;      // copied by host-memspace sweeps (icmslam_get_transfer_bytes)
    // a host-memory sweep of a map chain goes through in chunks of tiles: upload, run kernel, solve and read-back of successive
    // chunks overlap (fused_part_a, HostPipe)
    Stream h2d_stream; Event ev_in[16], ev_out[16]; int pipe_chunks = 8; bool pipe_events = false;
    bool tail_wait_fork = false;
    int pipe_tiles_min = 64;
    double* d2h_x = nullptr; int64_t d2h_ld = 0; bool d2h_done = false;   // host destination of the sweep in flight's poses (fused path)
    // time-segment partition (icmslam_set_segment): this handle owns columns [seg_lo, seg_hi) of its T columns
    int seg_lo = 0, seg_hi = 0, seg_first = 1, seg_last = 1;
    double* d_newraw = nullptr;   // 2 x Lcap: means of the sweep's new labels (zero elsewhere)
    DevBuf<long long> d_exch;     // ONE block [fsum_x | fsum_y | cnt] (newraw aliases the first two): what the segments sum-reduce, viewed as int64
    int64_t exch_words = 0;
    DevBuf<double> d_seg_rec;     // SEG_REC doubles: what this segment tells its neighbours
    DevBuf<double> d_seg_rec_pose;      // ... the boundary poses on their own when they are gathered beside the tail (icmslam_seg_halo)
    // peer-memory exchange of a time-segmented run (p2p.cuh): this rank's window and result buffer, every rank's pointers
    P2PDev p2p = {0, 0, 1, nullptr, nullptr, nullptr, nullptr, 0, 0};
    DevBuf<P2PWin> d_win; DevBuf<long long> d_res;
    IpcMapping p2p_opened[3 * P2P_MAX_WORLD];      // mappings of the other ranks' buffers (cudaIpcOpenMemHandle)
    DevBuf<void*> d_p2p_ptrs;                      // device copy of the three pointer tables
    bool seg_split = false;       // the sweep in flight exchanges its halo poses through icmslam_seg_halo
    double* seg_dst = nullptr;    // output pose buffer of the segment sweep in flight
    size_t fused_smem = 0;
    double thr2_hi = 0.0, fix_scale = 1.0;
    Event ev[4];
    double last_runs_ms = 0.0;   // k_runs alone in the last timed fused sweep
    int64_t n_launch = 0;   // kernels of this library launched so far (cub's not counted)
    // what the host knows of the state the device carries from one sweep to the next (a graph capture leaves it as it found it)
    struct Chain {
        int x_cur = 0;                      // which pose buffer (d_x / d_x2) holds the resident poses
        const double* ppar_of = nullptr;    // the pose buffer whose projection parameters are current (nullptr: recompute)
        const double* grid_map = nullptr;   // the map buffer the fast grid currently indexes (nullptr: rebuild)
        const double* hint_map = nullptr;   // the map buffer for which c[] (through d_remap) holds last sweep's labels
        int lm_cur = 0;                     // d_lmrec2[lm_cur] holds the current map's landmarks
        bool stats_clean = false;           // statistics / counts / far bits are all zero (the fused tail leaves them so)
        bool rawcnt_valid = false;          // d_rawcnt holds the counts of the raw map
        bool timed_fused = false;           // the last sweep was a fused one (icmslam_get_kernel_ms reads its events)
        bool lact_dirty = false;            // lact_host is stale: the device changed landmarks_actuales
    };
    Chain ch;
};

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            snprintf(h->err, sizeof h->err, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return ICMSLAM_ERR_CUDA;                                                                     \
        }                                                                                                \
    } while (0)

static inline int nblk(int64_t n, int b) { return (int)((n + b - 1) / b); }

// the resident poses, the buffer the next sweep writes, and the projection parameters of a pose buffer (they ping-pong with it)
static double* cur_x(const icmslam_handle* h) { return h->ch.x_cur ? h->ds.d_x2 : h->ds.d_x; }
static double* next_x(const icmslam_handle* h) { return h->ch.x_cur ? h->ds.d_x : h->ds.d_x2; }
static double4* ppar_for(const icmslam_handle* h, const double* x) { return h->ex.d_ppar[x == h->ds.d_x2 ? 1 : 0]; }

// the default sweep (REDBLACK, NEWTON, PREV) on the fused path: run records, association of dirty tiles, tile solve, fused tail
static bool fused_mode(const icmslam_handle* h, const icmslam_sweep_opts& o)
{
    return h->fused_ok && o.fused && o.schedule == ICMSLAM_SCHED_REDBLACK && o.solver == ICMSLAM_SOLVER_NEWTON && o.map_view == ICMSLAM_VIEW_PREV;
}

// a fused sweep has been issued: its solve writes the poses in `xout` and their projection parameters (a segment's halo columns
// come from the exchange), its tail the map in `map_out` (nullptr: a buffer the grid does not index) and the raw counts
static void chain_advance(icmslam_handle* h, const double* xout, const double* map_out)
{
    icmslam_handle::Chain& c = h->ch;
    c.ppar_of = xout;
    c.grid_map = c.hint_map = map_out;      // the grid indexes the new map, and c[] / d_remap carry this sweep's labels into it
    c.lm_cur ^= 1;
    c.stats_clean = c.rawcnt_valid = c.timed_fused = c.lact_dirty = true;
}

// after a sweep of the resident poses: its poses become the resident ones, and mapa_viejo = mapa_refinado (sensors.py:315)
static void end_sweep(icmslam_handle* h)
{
    h->ch.x_cur ^= 1;
    std::swap(h->d_map_in, h->d_map_out);
}

extern "C" int icmslam_abi_version(void) { return ICMSLAM_ABI_VERSION; }

extern "C" const char* icmslam_strerror(int s)
{
    switch (s) {
    case ICMSLAM_OK: return "ok";
    case ICMSLAM_EMPTY_FIRST_SCAN: return "first scan has no observation; inputs returned unchanged (sensors.py:137-139)";
    case ICMSLAM_ERR_INVALID: return "invalid argument or call order";
    case ICMSLAM_ERR_LABEL_CAP: return "label capacity L exceeded (reference: IndexError, ICM_SLAM.py:191)";
    case ICMSLAM_ERR_EMPTY_LAST: return "last scan has no observation (reference: IndexError, sensors.py:148)";
    case ICMSLAM_ERR_EMPTY_MAP: return "no landmark reaches cota (reference: ValueError, ICM_SLAM.py:241-255)";
    case ICMSLAM_ERR_ALLOC: return "allocation failed";
    case ICMSLAM_ERR_CUDA: return "CUDA error";
    case ICMSLAM_ERR_UNSUPPORTED: return "unsupported";
    default: return "unknown status";
    }
}

extern "C" const char* icmslam_last_error(const icmslam_handle* h) { return h ? h->err : "null handle"; }

// (a captured sweep holds the freeze arguments it was captured with)
static bool same_freeze(const Freeze& a, const Freeze& b)
{
    return a.frozen == b.frozen && a.traj == b.traj && a.K == b.K && a.cols == b.cols && a.pitch == b.pitch && a.slots == b.slots;
}

static void drop_graphs(icmslam_handle* h)
{
    for (auto& g : h->graphs) g.exec.reset();
}

// a fresh extraction: graphs that hold the old buffers go first, and nothing the host knew of the old observations stays (a
// pass-0 walk over them included)
static void reset_extraction(icmslam_handle* h)
{
    drop_graphs(h);
    h->ex = icmslam_handle::Extraction();
    h->ch.ppar_of = nullptr;
    h->ch.grid_map = nullptr;
    h->ch.hint_map = nullptr;
    h->fused_ok = false;
    h->extracted = false;
    h->laid_out = false;
    h->n = 0; h->n_cap = 0;
    h->off_h.clear();
    h->n_empty = 0; h->max_per_scan = 0;
    h->walk.on = false;
}

static void free_dataset(icmslam_handle* h)
{
    reset_extraction(h);
    h->ds = icmslam_handle::Dataset();
    h->cap_T = 0;
    h->ch.x_cur = 0;
    h->last_map_L = -1;
    h->traj_K = 0; h->traj_odd = false;
    h->d_traj_start.reset(); h->d_traj_of.reset(); h->d_x0s.reset();
    h->d_fz_mask.reset(); h->d_fz_need.reset(); h->d_fz_slots.reset(); h->d_fz_reg.reset(); h->fz_K = 0;
}

extern "C" int icmslam_destroy(icmslam_handle* h)
{
    if (!h) return ICMSLAM_OK;
    cudaSetDevice(h->cfg.device);
    delete h;
    return ICMSLAM_OK;
}

static int ensure_cub(icmslam_handle* h, size_t bytes)
{
    if (bytes <= h->cub_bytes) return ICMSLAM_OK;
    // captured graphs have the old workspace pointer baked in: they must not be replayed after it is freed
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (h->stream && cudaStreamIsCapturing(h->stream, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone) {
        snprintf(h->err, sizeof h->err, "scan workspace too small inside a graph capture (%zu > %zu bytes)", bytes, h->cub_bytes);
        return ICMSLAM_ERR_CUDA;
    }
    drop_graphs(h);
    h->cub_bytes = 0;
    CK(h->d_cub.alloc(bytes));
    h->cub_bytes = bytes;
    return ICMSLAM_OK;
}

static int exclusive_sum(icmslam_handle* h, const int* in, int* out, int n)
{
    size_t bytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, n, h->stream));
    int rc = ensure_cub(h, bytes);
    if (rc) return rc;
    CK(cub::DeviceScan::ExclusiveSum(h->d_cub, bytes, in, out, n, h->stream));
    return ICMSLAM_OK;
}

extern "C" int icmslam_create(const icmslam_config* cfg, icmslam_handle** out)
{
    if (!cfg || !out || cfg->L <= 0) return ICMSLAM_ERR_INVALID;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= cfg->device || cfg->device < 0) return ICMSLAM_ERR_CUDA;
    icmslam_handle* h = new (std::nothrow) icmslam_handle();
    if (!h) return ICMSLAM_ERR_ALLOC;
    h->err[0] = 0;
    h->cfg = *cfg;
    h->dcfg.dt = cfg->deltat; h->dcfg.q1 = cfg->q1; h->dcfg.q2 = cfg->q2;
    h->dcfg.r1 = cfg->r1; h->dcfg.r2 = cfg->r2; h->dcfg.r3 = cfg->r3;
    h->dcfg.kod = cfg->cte_odom; h->dcfg.cota = cfg->cota; h->dcfg.dist_thr = cfg->dist_thr;
    h->dcfg.rmax = cfg->rango_laser_max; h->dcfg.radio = cfg->radio; h->dcfg.L = cfg->L;
    h->Lcap = cfg->L;
    const size_t L = (size_t)h->Lcap;
    cudaError_t e = cudaSetDevice(cfg->device);
    if (e == cudaSuccess) e = h->d_sum_x.alloc(L);
    if (e == cudaSuccess) e = h->d_sum_y.alloc(L);
    if (e == cudaSuccess) e = h->d_raw.alloc(2 * L);
    if (e == cudaSuccess) e = h->d_counts.alloc(L);
    {   // exchange block (see icmslam_device_ptr): 64-bit words
        const size_t wcnt = (L + 2) / 2;
        // [fsum_x | fsum_y | cnt].  The means of the sweep's NEW labels (doubles, indices >= lsearch) live in the same words as the
        // fixed-point sums of the OLD labels (int64, indices < lsearch): the two index ranges are disjoint, every new label is
        // written by exactly one segment, and adding the all-zero words of the other segments to a double's bit pattern as an
        // integer leaves it unchanged -- so the segments sum-reduce 2.5 words per landmark instead of 4.5.
        h->exch_words = (int64_t)(2 * L + wcnt);
        if (e == cudaSuccess) e = h->d_exch.alloc((size_t)h->exch_words);
        if (e == cudaSuccess) e = cudaMemset(h->d_exch, 0, (size_t)h->exch_words * 8);
        h->d_fsum_x = h->d_exch; h->d_fsum_y = h->d_exch + L; h->d_newraw = (double*)h->d_exch.p; h->d_cnt = (int*)(h->d_exch + 2 * L);
    }
    if (e == cudaSuccess) e = h->d_seg.alloc(L + 1);
    if (e == cudaSuccess) e = h->d_kflag.alloc(L);
    if (e == cudaSuccess) e = h->d_kpos.alloc(L);
    if (e == cudaSuccess) e = h->d_parent.alloc(L);
    if (e == cudaSuccess) e = h->d_nn.alloc(L);
    if (e == cudaSuccess) e = h->d_indflag.alloc(L);
    if (e == cudaSuccess) e = h->d_indpos.alloc(L);
    if (e == cudaSuccess) e = h->d_ind.alloc(L);
    if (e == cudaSuccess) e = h->d_lab.alloc(L);
    if (e == cudaSuccess) e = h->d_used.alloc(L);
    if (e == cudaSuccess) e = h->d_rank.alloc(L);
    if (e == cudaSuccess) e = h->d_kx.alloc(L);
    if (e == cudaSuccess) e = h->d_ky.alloc(L);
    if (e == cudaSuccess) e = h->d_kc.alloc(L);
    if (e == cudaSuccess) e = h->d_ox.alloc(L);
    if (e == cudaSuccess) e = h->d_oy.alloc(L);
    if (e == cudaSuccess) e = h->d_oc.alloc(L);
    if (e == cudaSuccess) e = h->d_acc.alloc(8);
    if (e == cudaSuccess) e = h->d_map_in.alloc(2 * L);
    if (e == cudaSuccess) e = h->d_map_out.alloc(2 * L);
    if (e == cudaSuccess) e = h->d_tmp_a.alloc(2 * L);
    if (e == cudaSuccess) e = h->d_tmp_b.alloc(2 * L);
    if (e == cudaSuccess) e = h->walk.y.alloc(2 * L);
    if (e == cudaSuccess) e = h->walk.cant.alloc(L);
    if (e == cudaSuccess) e = h->walk.carry.alloc(1);
    h->fg_cells = (int)(4 * L > 4096 ? 4 * L : 4096);
    if (e == cudaSuccess) e = h->grid.alloc(h->fg_cells, 4 * L);    // replicated binning: <= 4 cells per landmark
    if (e == cudaSuccess) e = h->scratch_grid.alloc(h->fg_cells, 4 * L);
    if (e == cudaSuccess) e = h->d_ts.alloc(1);
    if (e == cudaSuccess) e = h->d_seg_rec.alloc(SEG_REC);
    if (e == cudaSuccess) e = h->d_seg_rec_pose.alloc(SEG_REC);
    if (e == cudaSuccess) e = cudaMemset(h->d_seg_rec_pose, 0, SEG_REC * sizeof(double));
    if (e == cudaSuccess) e = h->d_lmrec2[0].alloc(L);
    if (e == cudaSuccess) e = h->d_lmrec2[1].alloc(L);
    if (e == cudaSuccess) e = h->d_blk_kept.alloc((size_t)nblk((int)L, 256) + 1);
    if (e == cudaSuccess) e = h->d_rawcnt.alloc(L);
    if (e == cudaSuccess) e = h->d_gbuild.alloc(L);
    if (e == cudaSuccess) e = h->d_nnd0.alloc(L);
    if (e == cudaSuccess) e = h->d_gslots.alloc(L);
    if (e == cudaSuccess) e = h->d_cpart.alloc((size_t)4 * (nblk((int)L, 256) + 1));
    if (e == cudaSuccess) e = h->d_sh_x.alloc(L);
    if (e == cudaSuccess) e = h->d_sh_y.alloc(L);
    if (e == cudaSuccess) e = h->d_sh_k.alloc(L);
    { const char* es = getenv("ICMSLAM_STEADY"); if (es) h->steady_enable = atoi(es) != 0; }
    { const char* es = getenv("ICMSLAM_TRACE"); if (es && atoi(es)) h->trace_on = 1; }
    { const char* es = getenv("ICMSLAM_COND"); if (es) h->use_cond = atoi(es) != 0; }
    if (e == cudaSuccess) e = h->d_scan_state.alloc((size_t)nblk(h->fg_cells + 1, CS_THREADS * CS_ITEMS) + 1);
    if (e == cudaSuccess) e = h->d_remap.alloc(L);
    if (e == cudaSuccess) e = h->d_klab.alloc(L);
    if (e == cudaSuccess) e = h->d_aobs.alloc((size_t)2 * ASSOC_MAX_OBS);
    if (e == cudaSuccess) e = h->d_ac.alloc((size_t)ASSOC_MAX_OBS);
    if (e == cudaSuccess) e = cudaMemset(h->d_lmrec2[0], 0, L * sizeof(LmRec));
    if (e == cudaSuccess) e = cudaMemset(h->d_lmrec2[1], 0, L * sizeof(LmRec));
    if (e == cudaSuccess) e = cudaMemset(h->d_scan_state, 0, ((size_t)nblk(h->fg_cells + 1, CS_THREADS * CS_ITEMS) + 1) * sizeof(unsigned long long));
    { const double t1 = cfg->dist_thr * (1.0 + 9.5367431640625e-07); h->thr1sq = t1 * t1; }
    if (e == cudaSuccess) e = cudaMemset(h->d_ts, 0, sizeof(TailState));
    if (e == cudaSuccess) { const unsigned one = 1u; e = cudaMemcpy(&h->d_ts->scan_seq, &one, sizeof one, cudaMemcpyHostToDevice); }
    if (e == cudaSuccess) { const unsigned one = 1u; e = cudaMemcpy(&h->d_ts->p2p_seq, &one, sizeof one, cudaMemcpyHostToDevice); }
    if (e == cudaSuccess) { const unsigned one = 1u; e = cudaMemcpy(&h->d_ts->halo_seq, &one, sizeof one, cudaMemcpyHostToDevice); }
    if (e == cudaSuccess && h->trace_on) { const int one = 1; e = cudaMemcpy(&h->d_ts->trace_on, &one, sizeof one, cudaMemcpyHostToDevice); }
    { const char* eg = getenv("ICMSLAM_GRAPH"); if (eg) h->use_graph = atoi(eg); }
    { const char* er = getenv("ICMSLAM_RUNS"); if (er) h->use_runs = atoi(er) != 0; }
    if (e == cudaSuccess) {
        int sms = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device);
        h->assoc_blocks = 2 * (sms > 0 ? sms : 1);
    }
    {   // gate and fixed-point scale of the fused path
        const double thr = cfg->dist_thr;
        double s2 = thr * thr;
        while (sqrt(nextafter(s2, INFINITY)) <= thr) s2 = nextafter(s2, INFINITY);
        while (s2 > 0.0 && sqrt(s2) > thr) s2 = nextafter(s2, -INFINITY);
        h->thr2_hi = s2;
        double s3 = thr * thr;
        while (sqrt(s3) >= thr && s3 > 0.0) s3 = nextafter(s3, -INFINITY);
        while (sqrt(nextafter(s3, INFINITY)) < thr) s3 = nextafter(s3, INFINITY);
        h->thr2_lt = s3;
        int ex = thr > 1.0 ? ilogb(thr) + 1 : 0;
        h->fix_scale = ldexp(1.0, 34 - ex);      // 2^-34 m per unit: a run's sum fits the two 32-bit limbs of runs.cuh
    }
    if (e == cudaSuccess) e = h->d_st.alloc(1);
    if (e == cudaSuccess) e = h->h_st.alloc(1);
    for (int i = 0; i < 4 && e == cudaSuccess; ++i) e = cudaEventCreate(&h->ev[i].p);
    if (e == cudaSuccess) {     // the tail's small kernels (main stream, highest priority) are dispatched ahead of the waves of the solve
        int lo = 0, hi = 0;     // (side stream, lowest): with equal priorities the solve's pending blocks keep the tail out until it ends
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        e = cudaStreamCreateWithPriority(&h->own_stream.p, cudaStreamNonBlocking, hi);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&h->side_stream.p, cudaStreamNonBlocking, lo);
    }
    { const char* ec = getenv("ICMSLAM_PIPE_CHUNKS"); if (ec) { int c = atoi(ec); h->pipe_chunks = c < 1 ? 1 : (c > 16 ? 16 : c); } }
    { const char* ec = getenv("ICMSLAM_PIPE_TILES"); if (ec && atoi(ec) > 0) h->pipe_tiles_min = atoi(ec); }

    if (e == cudaSuccess) h->stream = h->own_stream;
    if (e == cudaSuccess) { int lo = 0, hi = 0; cudaDeviceGetStreamPriorityRange(&lo, &hi); e = cudaStreamCreateWithPriority(&h->cap_stream.p, cudaStreamNonBlocking, hi); }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fork.p, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_join.p, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_tail.p, cudaEventDisableTiming);
    { const char* eo = getenv("ICMSLAM_OVERLAP"); if (eo) h->overlap_solve = atoi(eo) != 0; }
    if (e == cudaSuccess) e = cudaMemset(h->d_st, 0, sizeof(DevState));
    if (e == cudaSuccess) e = cudaMemset(h->d_counts, 0, L * sizeof(double));
    if (e != cudaSuccess) {
        delete h;
        return e == cudaErrorMemoryAllocation ? ICMSLAM_ERR_ALLOC : ICMSLAM_ERR_CUDA;
    }
    *out = h;
    return ICMSLAM_OK;
}

extern "C" int icmslam_set_stream(icmslam_handle* h, void* s)
{
    if (!h) return ICMSLAM_ERR_INVALID;
    if (h->stream) cudaStreamSynchronize(h->stream);
    h->stream = s ? (cudaStream_t)s : h->own_stream;   // NULL: back to the handle's own stream
    drop_graphs(h);
    return ICMSLAM_OK;
}

extern "C" int icmslam_synchronize(icmslam_handle* h)
{
    if (!h) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    return ICMSLAM_OK;
}

// the scans' workspace for the largest scan of a sweep, so that nothing allocates inside a graph capture
static int size_cub(icmslam_handle* h)
{
    size_t need = 0, b = 0;
    const int lens[3] = {h->Lcap + 1, h->fg_cells + 2, h->T + 1};
    for (int k = 0; k < 3; ++k) { CK(cub::DeviceScan::ExclusiveSum(nullptr, b, (const int*)nullptr, (int*)nullptr, lens[k], h->stream)); if (b > need) need = b; }
    return ensure_cub(h, need);
}

// a rows x new_ld buffer in place of `b`, with the first `cols` columns of each row of b (leading dimension ld) copied over
template <typename E>
static cudaError_t regrow(icmslam_handle* h, DevBuf<E>& b, int rows, int64_t ld, int64_t cols, int64_t new_ld)
{
    DevBuf<E> nb;
    cudaError_t e = nb.alloc((size_t)rows * new_ld);
    if (e == cudaSuccess && cols > 0 && b)
        e = cudaMemcpy2DAsync(nb, (size_t)new_ld * sizeof(E), b, (size_t)ld * sizeof(E), (size_t)cols * sizeof(E), rows, cudaMemcpyDeviceToDevice,
                              h->stream);
    if (e == cudaSuccess) b = std::move(nb);      // (cudaFree waits for the copy out of the old buffer)
    return e;
}

extern "C" int icmslam_load(icmslam_handle* h, const double* scans, int32_t B, int32_t T, int64_t ld_scans,
                            const double* odo, int64_t ld_odo, const double* u, int64_t ld_u, const double* cos_tab,
                            const double* sin_tab, int32_t precondition, int32_t memspace)
{
    if (!h || !scans || !odo || !u || B <= 0 || B > 1024 || T <= 0 || ld_scans < T || ld_odo < T || ld_u < T)
        return ICMSLAM_ERR_INVALID;
    (void)memspace;   // cudaMemcpyDefault resolves host / device pointers (UVA)
    CK(cudaSetDevice(h->cfg.device));
    free_dataset(h);
    h->B = B; h->T = T; h->cap_T = T; h->precondition = precondition;
    CK(h->ds.d_scans.alloc((size_t)B * T));
    CK(h->ds.d_odo.alloc((size_t)3 * T));
    CK(h->ds.d_u.alloc((size_t)2 * T));
    CK(h->ds.d_cos.alloc((size_t)B));
    CK(h->ds.d_sin.alloc((size_t)B));
    CK(h->ds.d_ang.alloc((size_t)B));
    CK(h->ds.d_x.alloc((size_t)3 * T));
    h->seg_lo = 0; h->seg_hi = T; h->seg_first = 1; h->seg_last = 1;
    int rc = size_cub(h);
    if (rc) return rc;
    const size_t w = (size_t)T * sizeof(double);
    CK(cudaMemcpy2DAsync(h->ds.d_scans, w, scans, (size_t)ld_scans * sizeof(double), w, B, cudaMemcpyDefault, h->stream));
    CK(cudaMemcpy2DAsync(h->ds.d_odo, w, odo, (size_t)ld_odo * sizeof(double), w, 3, cudaMemcpyDefault, h->stream));
    CK(cudaMemcpy2DAsync(h->ds.d_u, w, u, (size_t)ld_u * sizeof(double), w, 2, cudaMemcpyDefault, h->stream));
    std::vector<double> ang(B), cb(B), sb(B);
    for (int i = 0; i < B; ++i) {
        ang[i] = ((double)i * ICM_PI) / 180.0;                 // nind*np.pi/180.0 (ICM_SLAM.py:44,51)
        cb[i] = cos_tab ? cos_tab[i] : cos(ang[i]);
        sb[i] = sin_tab ? sin_tab[i] : sin(ang[i]);
    }
    CK(cudaMemcpyAsync(h->ds.d_ang, ang.data(), B * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->ds.d_cos, cb.data(), B * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->ds.d_sin, sb.data(), B * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));   // the host staging vectors and caller buffers may go away
    return ICMSLAM_OK;
}

// filtrar_z of the columns [t_lo, T): all of them after reset_extraction, or those an append brought.  The offsets of the
// window continue from the h->n observations before it, and the per-observation arrays grow (by doubling) to hold the new ones.
static int extract_window(icmslam_handle* h, int t_lo)
{
    const int B = h->B, T = h->T, W = T - t_lo;
    const int nwords = (B + 31) / 32;
    cudaStream_t s = h->stream;
    DevBuf<uint32_t> d_masks;
    DevBuf<int> d_counts;
    CK(d_masks.alloc((size_t)W * nwords));
    CK(d_counts.alloc((size_t)W + 1));
    if (!h->ex.d_off) CK(h->ex.d_off.alloc((size_t)h->cap_T + 1));
    CK(cudaMemsetAsync(d_counts, 0, ((size_t)W + 1) * sizeof(int), s));
    const size_t smem = extract_smem_bytes(B);
    CK(cudaFuncSetAttribute(k_extract<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaFuncSetAttribute(k_extract<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int blocks = nblk(W, EX_TILE);
    k_extract<1><<<blocks, EX_THREADS, smem, s>>>(h->ds.d_scans, B, t_lo, T, h->cap_T, h->ds.d_cos, h->ds.d_sin, h->dcfg, h->precondition,
                                                  nwords, d_masks, d_counts, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
    CK(cudaGetLastError());
    {   // off[t_lo .. T] = n + exclusive sum of the window's counts
        size_t bytes = 0;
        CK(cub::DeviceScan::ExclusiveScan(nullptr, bytes, (const int*)d_counts, h->ex.d_off + t_lo, cub::Sum(), (int)h->n, W + 1, s));
        int rc = ensure_cub(h, bytes);
        if (rc) return rc;
        CK(cub::DeviceScan::ExclusiveScan(h->d_cub, bytes, (const int*)d_counts, h->ex.d_off + t_lo, cub::Sum(), (int)h->n, W + 1, s));
    }
    std::vector<int>& off = h->off_h;
    off.resize((size_t)T + 1);
    CK(cudaMemcpyAsync(off.data() + t_lo, h->ex.d_off + t_lo, ((size_t)W + 1) * sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    for (int t = t_lo; t < T; ++t) {
        int k = off[t + 1] - off[t];
        if (k == 0) ++h->n_empty;
        if (k > h->max_per_scan) h->max_per_scan = k;
    }
    h->first_empty = off[1] == off[0];
    h->last_empty = off[T] == off[T - 1];
    const int64_t n0 = h->n, n = off[T];
    if (n > h->n_cap || !h->ex.d_beam) {
        const int64_t cap = std::max(2 * h->n_cap, n);
        CK(regrow(h, h->ex.d_beam, 1, n0, n0, cap)); CK(regrow(h, h->ex.d_scan_of, 1, n0, n0, cap)); CK(regrow(h, h->ex.d_d, 1, n0, n0, cap));
        CK(regrow(h, h->ex.d_bx, 1, n0, n0, cap + 2)); CK(regrow(h, h->ex.d_by, 1, n0, n0, cap + 2));
        CK(regrow(h, h->ex.d_c, 1, n0, n0, cap + 8));      // (+ slack: the fused kernel stages 16-byte aligned slices of it)
        if (h->ex.d_seen_x) { CK(regrow(h, h->ex.d_seen_x, 1, n0, n0, cap)); CK(regrow(h, h->ex.d_seen_y, 1, n0, n0, cap)); }
        h->n_cap = cap;
    }
    CK(cudaMemsetAsync(h->ex.d_bx + n, 0, 2 * sizeof(double), s));
    CK(cudaMemsetAsync(h->ex.d_by + n, 0, 2 * sizeof(double), s));
    k_extract<2><<<blocks, EX_THREADS, smem, s>>>(h->ds.d_scans, B, t_lo, T, h->cap_T, h->ds.d_cos, h->ds.d_sin, h->dcfg, h->precondition,
                                                  nwords, d_masks, nullptr, h->ex.d_off, h->ex.d_beam, h->ex.d_d, h->ex.d_bx, h->ex.d_by,
                                                  h->ex.d_scan_of);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(s));      // (the masks and counts go when this returns)
    h->n = n;
    h->extracted = true;
    h->laid_out = false;
    return ICMSLAM_OK;
}

// the resident poses into d_x (a sweep may have left them in the double buffer)
static int poses_home(icmslam_handle* h)
{
    if (h->ch.x_cur) CK(cudaMemcpyAsync(h->ds.d_x, h->ds.d_x2, (size_t)3 * h->cap_T * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    h->ch.x_cur = 0;
    h->ch.ppar_of = nullptr;
    return ICMSLAM_OK;
}

// What the sweeps read beyond the extraction, laid out for the T columns loaded: the pose, odometry and control arrays with
// leading dimension T, the odometry increments, the per-scan workspaces, run records and tiles, projection parameters, body
// moments and the association kernel's shared-memory budget.  Done by icmslam_extract, and by the first call after an append
// that sweeps or sets what a sweep reads (a walk of pass 0 needs none of it).
static int ensure_layout(icmslam_handle* h)
{
    if (!h->extracted || h->laid_out) return ICMSLAM_OK;
    drop_graphs(h);
    const int T = h->T;
    cudaStream_t s = h->stream;
    int rc = poses_home(h);
    if (rc) return rc;
    if (h->cap_T != T) {      // (an append left the columns in larger buffers)
        CK(regrow(h, h->ds.d_scans, h->B, h->cap_T, T, T));
        CK(regrow(h, h->ds.d_odo, 3, h->cap_T, T, T));
        CK(regrow(h, h->ds.d_u, 2, h->cap_T, T, T));
        CK(regrow(h, h->ds.d_x, 3, h->cap_T, T, T));
        h->cap_T = T;
    }
    CK(h->ds.d_x2.alloc((size_t)3 * T));
    CK(h->ds.d_inc.alloc((size_t)3 * T));
    k_odo_increments<<<nblk(T, 256), 256, 0, s>>>(h->ds.d_odo, T, T, h->ds.d_inc, T);
    CK(cudaGetLastError());
    CK(h->ds.d_nfar.alloc((size_t)T + 1));
    CK(h->ds.d_flag.alloc((size_t)T + 1));
    CK(h->ds.d_prefix.alloc((size_t)T + 1));
    CK(h->ds.d_far_list.alloc((size_t)T));
    CK(h->ds.d_blk_prefix.alloc((size_t)nblk(T + 1, RT_TILE) + 2));
    h->n_tiles = nblk(h->seg_hi - (h->seg_lo - (h->seg_first ? 0 : 1)), RT_TILE);
    h->n_solve_tiles = nblk(h->seg_hi - h->seg_lo, ST_OWN);
    h->ex.d_keys_out.reset(); h->ex.d_iota.reset(); h->ex.d_sorted.reset();      // (the running view sizes them by n on first use)
    const size_t n = (size_t)h->n;
    CK(h->ex.d_bxy.alloc(n + 2));
    k_interleave<<<nblk((int64_t)n, 256), 256, 0, s>>>(h->ex.d_bx, h->ex.d_by, (int64_t)n, h->ex.d_bxy);
    CK(cudaGetLastError());
    {   // run records and their bookkeeping (runs.cuh): slice s (32 scans) owns slots [s * maxr * 32, (s + 1) * maxr * 32)
        const size_t nt = (size_t)nblk(T + 1, RT_TILE) + 2;      // (+1 scan: a segment's tiling may start one scan earlier)
        h->n_tiles_alloc = (int)nt;
        h->ch.stats_clean = false;
        h->rec_maxr = h->max_per_scan > 0 ? h->max_per_scan : 1;
        h->rec_slots = (int64_t)(nt * RT_SLICES) * h->rec_maxr * 32;
        CK(h->ex.d_rec_sb.alloc((size_t)h->rec_slots)); CK(h->ex.d_rec_meta.alloc((size_t)h->rec_slots));
        CK(h->ex.d_nruns.alloc(nt * RT_TILE));
        CK(h->ex.d_tile_perm.alloc(nt * RT_TILE));
        CK(h->ex.d_pos_nruns.alloc(nt * RT_TILE));
        CK(cudaMemsetAsync(h->ex.d_pos_nruns, 0, nt * RT_TILE * sizeof(unsigned short), s));
        CK(cudaMemsetAsync(h->ex.d_tile_perm, 0, nt * RT_TILE, s));      // (rewritten with every tile's records; never read before)
        CK(h->ex.d_ppar[0].alloc((size_t)T)); CK(h->ex.d_ppar[1].alloc((size_t)T));
        CK(h->ex.d_farbits.alloc(nt * 4)); CK(h->ex.d_tile_epoch.alloc(nt));
        CK(h->ex.d_tile_flag.alloc(nt)); CK(h->ex.d_dirty_list.alloc(nt)); CK(h->ex.d_tile_slots.alloc(nt * RS_SLOTS)); CK(h->ex.d_tile_nslots.alloc(nt));
        CK(cudaMemsetAsync(h->ex.d_tile_nslots, 0, nt * sizeof(int), s));
        CK(h->ex.d_scan_dirty.alloc(nt * RT_TILE));
        CK(cudaMemsetAsync(h->ex.d_nruns, 0, nt * RT_TILE * sizeof(unsigned short), s));
        CK(cudaMemsetAsync(h->ex.d_tile_epoch, 0xff, nt * sizeof(int), s));       // epoch -1: no tile holds records
        CK(cudaMemsetAsync(h->ex.d_tile_flag, 0, nt * sizeof(int), s));
        CK(cudaMemsetAsync(h->ex.d_farbits, 0, nt * 4 * sizeof(unsigned), s));
        CK(cudaMemsetAsync(h->ex.d_scan_dirty, 0, nt * RT_TILE * sizeof(int), s));
    }
    CK(h->ex.d_bm.alloc((size_t)6 * T));
    CK(h->ex.d_dyn.alloc((size_t)6 * T));
    CK(cudaMemsetAsync(h->ex.d_dyn, 0, (size_t)6 * T * sizeof(double), s));
    k_body_moments<<<nblk(T, 128), 128, 0, s>>>(h->ex.d_off, h->ex.d_bxy, T, h->ex.d_bm, T);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(s));
    {   // shared-memory budget of the association kernel: observations of one tile of RT_TILE scans
        int mx = 0;
        const std::vector<int>& off = h->off_h;
        for (int tb = 0; tb < T; ++tb) {   // (any tile origin: a later icmslam_set_segment may shift the tiling)
            int t1 = tb + RT_TILE < T ? tb + RT_TILE : T;
            int m = off[t1] - off[tb];
            if (m > mx) mx = m;
        }
        h->max_tile_obs = mx;
        int blocks_per_sm = 2;
        const size_t fixed = sizeof(AssocSmem);
        const char* envb = getenv("ICMSLAM_BLOCKS_PER_SM");
        if (envb && atoi(envb) > 0) blocks_per_sm = atoi(envb);
        const size_t per_block = (size_t)233472 / blocks_per_sm - 1024 - 512;   // 228 KB per SM, 1 KB reserved per block
        int cap = (int)((per_block - fixed - 96) / AT_OBS_BYTES);
        const char* env = getenv("ICMSLAM_OBS_CAP");
        if (env && atoi(env) > 0) cap = atoi(env);
        const int cap_max = (int)((232448 - fixed - 96) / AT_OBS_BYTES);
        if (cap > cap_max) cap = cap_max;
        if (cap > mx) cap = mx;                                    // the whole tile fits: one chunk
        if (cap < h->max_per_scan) cap = h->max_per_scan;          // a chunk holds at least one whole scan
        if (cap < 2) cap = 2;
        h->obs_cap = (cap + 1) & ~1;
        h->fused_smem = assoc_smem_bytes(h->obs_cap);
        // (a per-function, per-device attribute shared by every handle of the process: opt in to the maximum)
        CK(cudaFuncSetAttribute(k_assoc_tiles, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
        h->fused_ok = h->max_per_scan <= 65535 && h->Lcap <= RUN_MAX_LABEL;
    }
    h->laid_out = true;
    return ICMSLAM_OK;
}

extern "C" int icmslam_extract(icmslam_handle* h)
{
    if (!h || !h->ds.d_scans) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    reset_extraction(h);
    int rc = extract_window(h, 0);
    if (rc) return rc;
    return ensure_layout(h);
}

extern "C" int icmslam_append(icmslam_handle* h, const double* scans, int32_t n_new, int64_t ld_scans, const double* odometry,
                              int64_t ld_odo, const double* controls, int64_t ld_u, int32_t memspace)
{
    if (!h || !h->ds.d_scans || !scans || !odometry || !controls || n_new <= 0 || ld_scans < n_new || ld_odo < n_new || ld_u < n_new)
        return ICMSLAM_ERR_INVALID;
    if ((int64_t)h->T + n_new > INT32_MAX) return ICMSLAM_ERR_INVALID;
    if (h->traj_K > 0 || h->seg_lo != 0 || h->seg_hi != h->T || !h->seg_first || !h->seg_last || h->p2p.on) return ICMSLAM_ERR_UNSUPPORTED;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    // captured graphs, the map chain and the projection parameters hold buffers that move or columns that change (the odometry
    // increment of the old last column reads the new first one)
    drop_graphs(h);
    h->ch.grid_map = nullptr; h->ch.hint_map = nullptr;
    int rc = poses_home(h);
    if (rc) return rc;
    const int T0 = h->T, T = T0 + n_new;
    const int t_lo = h->extracted ? T0 : 0;      // (a log loaded but not extracted yet is extracted whole)
    if (T > h->cap_T) {
        const int cap = std::max(2 * h->cap_T, T);
        CK(regrow(h, h->ds.d_scans, h->B, h->cap_T, T0, cap));
        CK(regrow(h, h->ds.d_odo, 3, h->cap_T, T0, cap));
        CK(regrow(h, h->ds.d_u, 2, h->cap_T, T0, cap));
        CK(regrow(h, h->ds.d_x, 3, h->cap_T, T0, cap));
        if (h->ex.d_off) CK(regrow(h, h->ex.d_off, 1, (int64_t)T0 + 1, h->extracted ? (int64_t)T0 + 1 : 0, (int64_t)cap + 1));
        h->cap_T = cap;
    }
    const size_t ld = (size_t)h->cap_T * sizeof(double), w = (size_t)n_new * sizeof(double);
    CK(cudaMemcpy2DAsync(h->ds.d_scans + T0, ld, scans, (size_t)ld_scans * sizeof(double), w, h->B, cudaMemcpyDefault, h->stream));
    CK(cudaMemcpy2DAsync(h->ds.d_odo + T0, ld, odometry, (size_t)ld_odo * sizeof(double), w, 3, cudaMemcpyDefault, h->stream));
    CK(cudaMemcpy2DAsync(h->ds.d_u + T0, ld, controls, (size_t)ld_u * sizeof(double), w, 2, cudaMemcpyDefault, h->stream));
    h->T = T;
    h->seg_hi = T;
    h->laid_out = false;
    rc = size_cub(h);
    if (rc) return rc;
    return extract_window(h, t_lo);      // (ends in a stream synchronise: the caller's buffers may go away)
}

extern "C" int icmslam_extraction_size(const icmslam_handle* h, int64_t* n_obs, int32_t* n_empty, int32_t* max_per_scan)
{
    if (!h || !h->extracted) return ICMSLAM_ERR_INVALID;
    if (n_obs) *n_obs = h->n;
    if (n_empty) *n_empty = h->n_empty;
    if (max_per_scan) *max_per_scan = h->max_per_scan;
    return ICMSLAM_OK;
}

extern "C" int icmslam_get_extraction(icmslam_handle* h, int32_t* off, int32_t* beam, double* d, double* bx, double* by,
                                      int32_t memspace)
{
    if (!h || !h->extracted) return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    const size_t n = (size_t)h->n;
    if (off) CK(cudaMemcpyAsync(off, h->ex.d_off, ((size_t)h->T + 1) * sizeof(int), cudaMemcpyDefault, h->stream));
    if (beam) CK(cudaMemcpyAsync(beam, h->ex.d_beam, n * sizeof(int), cudaMemcpyDefault, h->stream));
    if (d) CK(cudaMemcpyAsync(d, h->ex.d_d, n * sizeof(double), cudaMemcpyDefault, h->stream));
    if (bx) CK(cudaMemcpyAsync(bx, h->ex.d_bx, n * sizeof(double), cudaMemcpyDefault, h->stream));
    if (by) CK(cudaMemcpyAsync(by, h->ex.d_by, n * sizeof(double), cudaMemcpyDefault, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return ICMSLAM_OK;
}

// ---- Mapa state ------------------------------------------------------------------------------
__global__ void k_set_lact(DevState* st, int v) { st->lact = v; }

static int sync_state(icmslam_handle* h)
{
    CK(cudaMemcpyAsync(h->h_st, h->d_st, sizeof(DevState), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->lact_host = h->h_st->lact;
    h->ch.lact_dirty = false;
    return ICMSLAM_OK;
}

extern "C" int icmslam_set_landmarks_actuales(icmslam_handle* h, int32_t lact)
{
    if (!h || lact < 0 || lact > h->Lcap) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    if (h->last_map_L >= 0 && lact == h->last_map_L) {      // what the last host-memspace sweep left on the device: nothing to do,
        h->lact_host = lact;                                 // and the map chain stays alive (see icmslam_sweep)
        return ICMSLAM_OK;
    }
    k_set_lact<<<1, 1, 0, h->stream>>>(h->d_st, lact);
    CK(cudaGetLastError());
    h->ch.grid_map = nullptr;
    h->ch.hint_map = nullptr;
    h->last_map_L = -1;
    h->lact_host = lact;
    h->ch.lact_dirty = false;
    return ICMSLAM_OK;
}

extern "C" int icmslam_get_landmarks_actuales(const icmslam_handle* hc, int32_t* lact)
{
    icmslam_handle* h = const_cast<icmslam_handle*>(hc);
    if (!h || !lact) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    if (h->ch.lact_dirty) { int rc = sync_state(h); if (rc) return rc; }
    *lact = h->lact_host;
    return ICMSLAM_OK;
}

extern "C" int icmslam_get_counts(icmslam_handle* h, double* out, int32_t n, int32_t memspace)
{
    if (!h || !out || n < 0 || n > h->Lcap) return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpyAsync(out, h->d_counts, (size_t)n * sizeof(double), cudaMemcpyDefault, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return ICMSLAM_OK;
}

extern "C" int icmslam_set_counts(icmslam_handle* h, const double* in, int32_t n, int32_t memspace)
{
    if (!h || n < 0 || n > h->Lcap || (n > 0 && !in)) return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemsetAsync(h->d_counts, 0, (size_t)h->Lcap * sizeof(double), h->stream));      // Mapa.clear_obs (ICM_SLAM.py:119-126) + the given prefix
    if (n > 0) CK(cudaMemcpyAsync(h->d_counts, in, (size_t)n * sizeof(double), cudaMemcpyDefault, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return ICMSLAM_OK;
}

// landmark grid G (fastgrid.cuh) over the first *n_ptr points of (px, py): five kernels (the caller counts them).  G.cnt is all
// zero on entry and on exit (the fill pass counts it back down), so no per-build memset is needed.
static int build_fgrid(icmslam_handle* h, LandmarkGrid& G, const double* px, const double* py, const int* n_ptr, int n_cap)
{
    cudaStream_t s = h->stream;
    k_fgrid_bbox_reset<<<1, 1, 0, s>>>(G.bb);
    CK(cudaGetLastError());
    int nb = nblk(n_cap, 256);
    if (nb > 148 * 2) nb = 148 * 2;
    k_fgrid_bbox<<<nb, 256, 0, s>>>(px, py, n_ptr, G.bb);
    CK(cudaGetLastError());
    k_fgrid_geom<<<1, 1, 0, s>>>(G.bb, n_ptr, h->dcfg.dist_thr, h->fg_cells, G.geom);
    CK(cudaGetLastError());
    k_fgrid_count<<<nblk(n_cap, 256), 256, 0, s>>>(px, py, n_ptr, G.geom, G.cnt);
    CK(cudaGetLastError());
    int rc = exclusive_sum(h, G.cnt, G.start, h->fg_cells + 1);
    if (rc) return rc;
    k_fgrid_fill<<<nblk(n_cap, 256), 256, 0, s>>>(px, py, n_ptr, G.geom, G.start, G.cnt, G.pts, G.idx);
    CK(cudaGetLastError());
    return ICMSLAM_OK;
}

// ---- Mapa.filtrar (ICM_SLAM.py:204-265) for every caller: the filter chain of tail.cuh ---------------------------------------
// k_tail_compact -> k_tail_count -> k_cell_scan -> k_fgrid_fill -> k_tail_nn over the raw map (raw_x, raw_y): the filtered map
// to map_out, its counts to d_counts, its width to st->new_l and st->lact, and h->grid built over it.  What the chain reads is
// left by its entry (k_fused_means and far_scan_block in the fused sweep, k_means_flags or k_flags_from_counts otherwise):
//   * raw_x / raw_y hold the raw means, st->raw_l their number;
//   * d_kflag holds the keep flags, d_blk_kept the kept landmarks per 256-thread block, counted on a grid of k_tail_compact's
//     shape (the compaction takes its positions from them);
//   * d_cnt holds the int observation counts (k_tail_compact moves them to d_rawcnt and clears d_cnt), unless cnt_d gives
//     double counts, which are taken as they are (d_cnt and d_rawcnt then stay as they were);
//   * h->grid's bounding box is reset, ts->n_ind is 0, and ts->steady_ok is 0 (otherwise every kernel of the chain returns at
//     once);
//   * h->grid's cell counts are all zero (every build leaves them so).
// `fused` launches k_tail_nn<true>, which also closes the fused sweep's bookkeeping (sequence numbers, epoch, steady tail).  Any
// other caller invalidates ch.grid_map and ch.hint_map: the grid, d_remap and the landmark records the chain writes then belong
// to no map chain, and the next fused sweep rebuilds them.
//
// Why the chain gives the reference's result (a K x K search) at every map size:
//   * the grid is searched unless the map is degenerate (extent < dist_thr), where tail_slow_body runs the reference's brute
//     force.  With an extent >= dist_thr the map diameter is >= dist_thr, and the reference substitutes the diameter for zero
//     distances, so a substituted value never passes the strict gate.  The nearest neighbour is read only for survivors that pass
//     the gate, and on those the grid's rule (rooted distances, the lowest index on ties) is argmin's first minimum;
//   * with no merge the new map is mul_rn(x, c) / c and c, as the reference's count-weighted mean of one member;
//   * with merges the merged means are accumulated with fp64 atomics in no fixed order: equal up to the rounding of that order.
static int filter_chain(icmslam_handle* h, const double* raw_x, const double* raw_y, const double* cnt_d, double* dmap_out, int out_cap,
                        int64_t out_ld, cudaStream_t s, bool fused)
{
    const int L = h->Lcap;
    DevState* st = h->d_st;
    TailState* ts = h->d_ts;
    k_tail_compact<<<nblk(L, 256), 256, 0, s>>>(st, h->d_kflag, h->d_blk_kept, h->d_kpos, raw_x, raw_y, h->d_cnt, h->d_kx, h->d_ky, h->d_kc,
                                                h->d_parent, h->grid.bb, L, h->d_klab, h->d_rawcnt, ts, cnt_d);
    CK(cudaGetLastError());
    k_tail_count<<<nblk(L, 256), 256, 0, s>>>(h->d_kx, h->d_ky, st, ts, h->grid.bb, h->dcfg.dist_thr, h->fg_cells, h->grid.geom, h->grid.cnt);
    CK(cudaGetLastError());
    k_cell_scan<<<nblk(h->fg_cells + 1, CS_THREADS * CS_ITEMS), CS_THREADS, 0, s>>>(h->grid.cnt, h->grid.start, h->fg_cells + 1, h->d_scan_state, ts);
    CK(cudaGetLastError());
    k_fgrid_fill<<<nblk(L, 256), 256, 0, s>>>(h->d_kx, h->d_ky, &st->kept, h->grid.geom, h->grid.start, h->grid.cnt, h->grid.pts,
                                              h->grid.idx, h->d_gslots, &ts->steady_ok);
    CK(cudaGetLastError());
    SlowArgs sa;
    sa.dist_thr = h->dcfg.dist_thr; sa.parent = h->d_parent; sa.ind_pos = h->d_indpos; sa.ind = h->d_ind; sa.lab = h->d_lab; sa.used = h->d_used;
    sa.rank = h->d_rank; sa.ox = h->d_ox; sa.oy = h->d_oy; sa.oc = h->d_oc; sa.max_cells = h->fg_cells; sa.geom = h->grid.geom;
    sa.cell_cnt = h->grid.cnt; sa.cell_start = h->grid.start; sa.pts = h->grid.pts; sa.gidx = h->grid.idx;
    sa.gbuild = h->d_gbuild; sa.nnd0 = h->d_nnd0; sa.steady_enable = h->steady_enable; sa.fz = h->fz;
    auto nn = fused ? k_tail_nn<true> : k_tail_nn<false>;
    nn<<<nblk(L, 256), 256, 0, s>>>(st, ts, h->d_kx, h->d_ky, h->d_kc, h->grid.geom, h->grid.start, h->grid.pts, h->grid.idx, h->thr2_lt,
                                    h->d_nn, h->d_indflag, L, h->d_klab, h->d_kflag, h->d_kpos, h->d_lmrec2[h->ch.lm_cur],
                                    h->d_lmrec2[h->ch.lm_cur ^ 1], dmap_out, out_cap, out_ld, h->d_counts, h->thr1sq, h->thr2_hi, h->d_remap, sa);
    CK(cudaGetLastError());
    return ICMSLAM_OK;
}

// (a fused sweep on a map whose grid is in place does without this launch: k_runs' first block resets the sweep's state,
// tail.cuh sweep_begin_state, and the tail's last block has left the two counters at zero)
__global__ void k_sweep_begin(DevState* st, TailState* ts, int L_in)
{
    ts->far_count = 0;
    ts->n_dirty = 0;
    sweep_begin_state(st, L_in);
}

static int status_from_state(const DevState* s)
{
    if (s->status & ST_P2P_TIMEOUT) return ICMSLAM_ERR_CUDA;      // a peer never posted its flag (p2p.cuh): the ranks are out of step
    if (s->status & ST_LABEL_CAP) return ICMSLAM_ERR_LABEL_CAP;
    if (s->status & 4) return ICMSLAM_ERR_EMPTY_MAP;
    return ICMSLAM_OK;
}

static void default_opts(icmslam_sweep_opts& o, const icmslam_sweep_opts* opts)
{
    o.schedule = ICMSLAM_SCHED_REDBLACK; o.solver = ICMSLAM_SOLVER_NEWTON; o.map_view = ICMSLAM_VIEW_PREV;
    o.newton_maxit = 0; o.newton_tol = 0.0; o.fused = 1; o.reserved = 0;
    if (opts) o = *opts;
    if (o.newton_maxit <= 0) o.newton_maxit = 20;
    if (!(o.newton_tol > 0.0)) o.newton_tol = 1e-7;    // Newton is quadratic: the step after |dtheta| <= 1e-7 is ~1e-14
}

// (a map from outside: run records are void, and so is what the steady tail remembers of the grid the previous chain built)
__global__ void k_epoch_bump(TailState* ts) { ts->epoch += 1; ts->steady_armed = 0; }
__global__ void k_note_dirty(DevState* st, const TailState* ts) { st->dirty_tiles = ts->n_dirty; }

static TrajLayout traj_layout(const icmslam_handle* h, const double* x0)
{
    TrajLayout L;
    L.first = h->seg_first; L.K = h->traj_K; L.start = h->d_traj_start; L.traj = h->d_traj_of; L.x0s = h->d_x0s; L.ldx0s = h->traj_K;
    L.x0[0] = x0[0]; L.x0[1] = x0[1]; L.x0[2] = x0[2];
    return L;
}

// projection parameters (solve.cuh make_ppar) of the poses in `x`, unless the solve of the previous sweep already left them
static int ensure_ppar(icmslam_handle* h, const double* x, int64_t ldx, const double* x0, double4* dst)
{
    if (h->ch.ppar_of == x && x != nullptr) return ICMSLAM_OK;
    k_ppar_init<<<nblk(h->T, 256), 256, 0, h->stream>>>(x, ldx, 0, h->T, traj_layout(h, x0), dst);
    CK(cudaGetLastError());
    h->n_launch += 1;
    h->ch.ppar_of = x;
    return ICMSLAM_OK;
}

// The fused tail zeroes the landmark statistics, the observation counts and the far bits as it consumes them; anything else that
// wrote them (the reference-mode sweep, pass 0, a fresh extraction) leaves a memset to the next fused sweep.
static int ensure_stats_clean(icmslam_handle* h)
{
    if (h->ch.stats_clean) return ICMSLAM_OK;
    cudaStream_t s = h->stream;
    CK(cudaMemsetAsync(h->d_cnt, 0, ((size_t)h->Lcap + 1) * sizeof(int), s));
    if (h->d_fsum_x) CK(cudaMemsetAsync(h->d_fsum_x, 0, (size_t)2 * h->Lcap * sizeof(long long), s));
    if (h->ex.d_farbits) CK(cudaMemsetAsync(h->ex.d_farbits, 0, (size_t)h->n_tiles_alloc * 4 * sizeof(unsigned), s));
    h->ch.stats_clean = true;
    return ICMSLAM_OK;
}

// ---- the fused (REDBLACK, NEWTON, PREV) sweep in three parts; a time-segmented run (one segment per GPU)
// exchanges data with the other segments between them ----------------------------------------------------
// part A: (grid of the previous map if it is not there yet) + the run kernel + the association kernel over the tiles the run
// kernel could not certify + the pose solve (forked beside the tail when `overlap`) + the scan of far-scan counts
struct HostPipe { double* x; int64_t ld; int chunks; };      // the caller's host poses (in and out) of a chunk-pipelined sweep

static bool pipe_ready(icmslam_handle* h);

static void launch_runs(int blocks, cudaStream_t s, const RunParams& R)
{
    if (R.fz.frozen) k_runs<true><<<blocks, RUNS_THREADS, 0, s>>>(R);
    else k_runs<false><<<blocks, RUNS_THREADS, 0, s>>>(R);
}

static void launch_solve(const icmslam_handle* h, int blocks, cudaStream_t s, const SolveParams& P)
{
    if (h->traj_odd) {      // a batch with a trajectory that starts on an odd column: colours by trajectory-local time
        if (P.fz.frozen) k_solve_tile<true, true><<<blocks, ST_THREADS, 0, s>>>(P);
        else k_solve_tile<false, true><<<blocks, ST_THREADS, 0, s>>>(P);
    } else if (P.fz.frozen) k_solve_tile<true><<<blocks, ST_THREADS, 0, s>>>(P);
    else k_solve_tile<false><<<blocks, ST_THREADS, 0, s>>>(P);
}

static int fused_part_a(icmslam_handle* h, const double* xin, int64_t ldin, double* kout, int64_t kld, const double* x0,
                        const icmslam_sweep_opts& o, int n_search_cap, bool overlap = false, const HostPipe* hp = nullptr)
{
    h->tail_wait_fork = false;
    const int T = h->T, L = h->Lcap;
    cudaStream_t s = h->stream;
    DevState* st = h->d_st;
    const double* min_x = h->d_map_in;
    const double* min_y = h->d_map_in + L;
    const bool timing = (o.reserved & 2) != 0;
    if (h->ch.grid_map != h->d_map_in) {      // the grid of the previous sweep's tail does not index this map: build it
        int rc = build_fgrid(h, h->grid, min_x, min_y, &st->lsearch, n_search_cap);
        if (rc) return rc;
        k_lmrec_build<<<nblk(n_search_cap, 256), 256, 0, s>>>(min_x, min_y, &st->lsearch, h->grid.geom, h->grid.start, h->grid.pts, h->grid.idx,
                                                              h->thr1sq, h->thr2_hi, h->d_lmrec2[h->ch.lm_cur]);
        CK(cudaGetLastError());
        k_epoch_bump<<<1, 1, 0, s>>>(h->d_ts);      // a map from outside: its labels are a new numbering, run records are void
        CK(cudaGetLastError());
        h->n_launch += 7;      // the grid (5), k_lmrec_build, k_epoch_bump
        h->ch.hint_map = nullptr;
    }
    double4* pp_in = ppar_for(h, xin);
    double4* pp_out = h->ex.d_ppar[pp_in == h->ex.d_ppar[0] ? 1 : 0];      // (the other one, whatever buffer kout is)
    if (!hp) {
        int rc = ensure_ppar(h, xin, ldin, x0, pp_in);
        if (rc) return rc;
    }
    const int t_start = h->seg_lo - (h->seg_first ? 0 : 1);     // a later segment also forms the moments of its odd halo pose
    RunParams R;
    R.t_start = t_start; R.t_hi = h->seg_hi; R.halo_t = h->seg_first ? -1 : t_start; R.maxr = h->rec_maxr; R.ppar = pp_in; R.lmrec = h->d_lmrec2[h->ch.lm_cur];
    R.rec_sb = h->ex.d_rec_sb; R.rec_meta = h->ex.d_rec_meta; R.nruns = h->ex.d_nruns; R.tile_perm = h->ex.d_tile_perm; R.pos_nruns = h->ex.d_pos_nruns; R.tile_epoch = h->ex.d_tile_epoch; R.dyn = h->ex.d_dyn;
    R.fsum_x = h->d_fsum_x; R.fsum_y = h->d_fsum_y; R.cnt = h->d_cnt; R.fix_scale = h->fix_scale; R.tile_slots = h->ex.d_tile_slots; R.tile_nslots = h->ex.d_tile_nslots;
    R.far_list = h->ds.d_far_list; R.ts = h->d_ts; R.farbits = h->ex.d_farbits;
    R.scan_dirty = h->ex.d_scan_dirty; R.tile_flag = h->ex.d_tile_flag; R.dirty_list = h->ex.d_dirty_list;
    R.geom = h->grid.geom; R.cell_start = h->grid.start; R.gpts = h->grid.pts; R.dist_thr = h->dcfg.dist_thr;
    R.st = st; R.L_in = h->begin_L; R.slice0 = 0; R.fz = h->fz;
    AssocParams A;
    A.first_halo = h->seg_first ? 0 : 1; A.T = T; A.off = h->ex.d_off; A.bxy = h->ex.d_bxy; A.cfg = h->dcfg; A.thr2_hi = h->thr2_hi; A.st = st; A.geom = h->grid.geom;
    A.cell_start = h->grid.start; A.gpts = h->grid.pts; A.gidx = h->grid.idx; A.remap = h->d_remap;
    { const char* eh = getenv("ICMSLAM_HINTS"); A.skip_hints = (eh && atoi(eh) == 0) ? 1 : 0; }
    A.hints = (h->ch.hint_map == h->d_map_in) ? 1 : 0;
    A.c = h->ex.d_c; A.obs_cap = h->obs_cap; A.R = R;
    A.n_tiles = h->n_tiles; A.blk_prefix = h->ds.d_blk_prefix; A.Lcap = L; A.bb = h->grid.bb; A.stw = st; A.final = 1; A.p2p = h->p2p;
    const int nb = h->assoc_blocks < h->n_tiles ? h->assoc_blocks : h->n_tiles;      // grid of the association kernel
    SolveParams P;
    P.T = T; P.t_lo = h->seg_lo; P.t_hi = h->seg_hi; P.lay = traj_layout(h, x0);
    P.xin = xin; P.ldin = ldin; P.xout = kout; P.ldout = kld;
    P.inc = h->ds.d_inc; P.ldinc = T; P.u = h->ds.d_u; P.ldu = T; P.bm = h->ex.d_bm; P.ldbm = T; P.dyn = h->ex.d_dyn;
    P.ppin = pp_in; P.ppout = pp_out; P.cfg = h->dcfg; P.tol = o.newton_tol; P.maxit = o.newton_maxit;
    P.iters = (o.reserved & 1) ? &st->newton_iters : nullptr; P.tile0 = 0;
    P.trace_row = h->trace_on ? &h->d_ts->trace[0][0] : nullptr; P.trace_seq = h->p2p.on ? &h->d_ts->halo_seq : &h->d_ts->sweep_no;
    P.fz = h->fz;
    if (hp) {
        // ---- chunks of tiles: upload | projection parameters, run kernel, association of the tiles it hands over, solve of the
        //      poses whose moments are complete | read-back, on three streams ---------------------------------------------------
        P.iters = nullptr; P.trace_row = nullptr; P.trace_seq = nullptr;
        const int C = hp->chunks, per = (h->n_tiles + C - 1) / C;
        cudaStream_t sin = h->h2d_stream, sout = h->side_stream;
        CK(cudaEventRecord(h->ev_fork, s));
        CK(cudaStreamWaitEvent(sin, h->ev_fork, 0));
        CK(cudaStreamWaitEvent(sout, h->ev_fork, 0));
        for (int c = 0; c < C; ++c) {
            const int a = c * per * RT_TILE, b = (c + 1) * per * RT_TILE < T ? (c + 1) * per * RT_TILE : T;
            if (b > a) CK(cudaMemcpy2DAsync((double*)xin + a, (size_t)ldin * 8, hp->x + a, (size_t)hp->ld * 8, (size_t)(b - a) * 8, 3, cudaMemcpyHostToDevice, sin));
            CK(cudaEventRecord(h->ev_in[c], sin));
        }
        int solved = 0;
        for (int c = 0; c < C; ++c) {
            const int tile_a = c * per, tile_b = (c + 1) * per < h->n_tiles ? (c + 1) * per : h->n_tiles;
            const int a = tile_a * RT_TILE, b = tile_b * RT_TILE < T ? tile_b * RT_TILE : T;
            const bool last = c == C - 1;
            CK(cudaStreamWaitEvent(s, h->ev_in[c], 0));
            if (tile_b > tile_a) {
                k_ppar_init<<<nblk(b - a, 256), 256, 0, s>>>(xin, ldin, a, b, P.lay, pp_in);
                R.slice0 = tile_a * RT_SLICES;
                launch_runs((tile_b - tile_a) * RT_SLICES, s, R);
                h->n_launch += 2;
            }
            A.final = last ? 1 : 0;
            k_assoc_tiles<<<nb, AT_THREADS, h->fused_smem, s>>>(A);
            CK(cudaGetLastError());
            h->n_launch += 1;
            // solve tiles whose poses (own range + the staged margin) are uploaded and whose moments are final
            int ready = last ? h->n_solve_tiles : (b >= ST_XT ? (b - ST_XT) / ST_OWN + 1 : 0);
            if (ready > h->n_solve_tiles) ready = h->n_solve_tiles;
            if (ready > solved) {
                P.tile0 = solved;
                launch_solve(h, ready - solved, s, P);
                CK(cudaGetLastError());
                h->n_launch += 1;
                CK(cudaEventRecord(h->ev_out[c], s));
                CK(cudaStreamWaitEvent(sout, h->ev_out[c], 0));
                const int ca = h->seg_lo + solved * ST_OWN, cb = h->seg_lo + ready * ST_OWN < h->seg_hi ? h->seg_lo + ready * ST_OWN : h->seg_hi;
                if (cb > ca) CK(cudaMemcpy2DAsync(hp->x + ca, (size_t)hp->ld * 8, kout + ca, (size_t)kld * 8, (size_t)(cb - ca) * 8, 3, cudaMemcpyDeviceToHost, sout));
                solved = ready;
            }
        }
        CK(cudaEventRecord(h->ev_join, sout));
        CK(cudaEventRecord(h->ev_fork, s));      // (what a tail on another stream waits for: the last chunk's kernels)
        h->join_pending = true;
        h->d2h_done = true;
        return ICMSLAM_OK;
    }
    if (timing) CK(cudaEventRecord(h->ev[0], s));
    if (h->use_runs) {
        launch_runs(h->n_tiles * RT_SLICES, s, R);
    } else {
        k_all_dirty<<<nblk(h->n_tiles, 256), 256, 0, s>>>(h->ex.d_tile_flag, h->ex.d_dirty_list, h->d_ts, h->n_tiles, st, h->begin_L);
    }
    CK(cudaGetLastError());
    if (timing) CK(cudaEventRecord(h->ev[2], s));
    k_assoc_tiles<<<nb, AT_THREADS, h->fused_smem, s>>>(A);
    CK(cudaGetLastError());
    if (o.reserved & 1) { k_note_dirty<<<1, 1, 0, s>>>(st, h->d_ts); CK(cudaGetLastError()); }
    if (timing) CK(cudaEventRecord(h->ev[3], s));
    h->n_launch += 2;
    cudaStream_t ss = s;
    const bool fork = overlap && h->overlap_solve && !timing && h->side_stream;
    if (fork) {      // the tail does not depend on the new poses: solve beside it
        CK(cudaEventRecord(h->ev_fork, s));
        CK(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
        ss = h->side_stream;
    }
    launch_solve(h, h->n_solve_tiles, ss, P);
    CK(cudaGetLastError());
    if (h->d2h_x) {      // a host-memory caller: its poses start their way back as soon as they are solved, beside the tail
        CK(cudaMemcpy2DAsync(h->d2h_x, (size_t)h->d2h_ld * 8, kout, (size_t)kld * 8, (size_t)T * 8, 3, cudaMemcpyDeviceToHost, ss));
        h->d2h_done = true;
    }
    if (h->p2p.on) {     // the segment's boundary poses to its neighbours, theirs into the halo columns: behind the solve
        k_p2p_halo<<<1, 32, 0, ss>>>(h->p2p, &h->d_ts->halo_seq, kout, kld, T, h->seg_lo, h->seg_hi, pp_out, st,
                                     h->trace_on ? &h->d_ts->trace[0][0] : nullptr);
        CK(cudaGetLastError());
        h->n_launch += 1;
    }
    if (fork) {
        CK(cudaEventRecord(h->ev_join, ss));
        h->join_pending = true;
    }
    h->n_launch += 1;
    if (timing) CK(cudaEventRecord(h->ev[1], s));
    return ICMSLAM_OK;
}

// part B: the sweep's new labels (needs the label numbering: on several GPUs, after the exchange)
static int fused_part_b(icmslam_handle* h, cudaStream_t s)
{
    const int L = h->Lcap;
    const int t_start = h->seg_lo - (h->seg_first ? 0 : 1);
    k_tail_labels<<<148, 256, 0, s>>>(h->d_ts, h->ds.d_far_list, h->ds.d_blk_prefix, h->ex.d_farbits, RT_TILE, t_start, h->ex.d_off, h->d_st, L, h->ex.d_c,
                                              h->d_newraw, h->d_newraw + L, h->d_cnt, h->p2p);
    CK(cudaGetLastError());
    h->n_launch += 1;
    if (h->p2p.on) {      // this rank's slice of every rank's statistics (a reduce-scatter by remote loads, p2p.cuh)
        const long long mine = h->p2p.per;
        int nb = (int)((mine + 255) / 256);
        if (nb > 148 * 4) nb = 148 * 4;
        if (nb < 1) nb = 1;
        k_p2p_reduce<<<nb, 256, 0, s>>>(h->p2p, &h->d_ts->p2p_seq, &h->d_ts->reduce_ticket, h->d_st, h->trace_on ? &h->d_ts->trace[0][0] : nullptr);
        CK(cudaGetLastError());
        h->n_launch += 1;
    }
    return ICMSLAM_OK;
}

// part C: landmark update, Mapa.filtrar and the grid of the new map (needs the statistics of ALL segments); `xout` is the pose
// buffer part A's solve wrote
static int full_chain(icmslam_handle* h, double* dmap_out, int out_cap, int64_t out_ld, cudaStream_t s);

static int fused_part_c(icmslam_handle* h, const double* xout, double* dmap_out, int out_cap, int64_t out_ld, cudaStream_t s)
{
    const int L = h->Lcap;
    DevState* st = h->d_st;
    TailState* ts = h->d_ts;
    const double* min_x = h->d_map_in;
    const double* min_y = h->d_map_in + L;
    double* raw_x = h->d_raw;
    double* raw_y = h->d_raw + L;
    {
        SteadyArgs a;
        a.fsum_x = h->d_fsum_x; a.fsum_y = h->d_fsum_y; a.cnt = h->d_cnt; a.map_x = min_x; a.map_y = min_y;
        a.inv_scale = 1.0 / h->fix_scale; a.cota = h->dcfg.cota; a.dist_thr = h->dcfg.dist_thr; a.thr1sq = h->thr1sq; a.thr2_hi = h->thr2_hi;
        a.lmrec_old = h->d_lmrec2[h->ch.lm_cur]; a.lmrec_new = h->d_lmrec2[h->ch.lm_cur ^ 1];
        a.gbuild = h->d_gbuild; a.nnd0 = h->d_nnd0; a.gslots = h->d_gslots; a.gpts = h->grid.pts;
        a.raw_x = raw_x; a.raw_y = raw_y; a.rawcnt = h->d_rawcnt;
        a.map_out = dmap_out; a.cap_out = out_cap; a.ld_out = out_ld; a.counts_state = h->d_counts; a.remap = h->d_remap; a.Lcap = L;
        a.cpart = h->d_cpart; a.fz = h->fz;
        a.sh_x = h->d_sh_x; a.sh_y = h->d_sh_y; a.sh_k = h->d_sh_k; a.farbits = h->ex.d_farbits; a.n_far_words = h->n_tiles * 4;
        a.use_cond = 0;
        memset(&a.cond, 0, sizeof a.cond);
        // Inside the library's own graph capture the rest of the chain becomes the body of an IF node whose condition the steady
        // kernel sets (1 = it could not close the sweep): a steady sweep then launches nothing after it.
        cudaGraph_t cgraph = nullptr;
        const cudaGraphNode_t* deps = nullptr;
        size_t ndeps = 0;
        if (h->in_own_capture && h->use_cond && h->steady_enable && h->cap_stream) {
            cudaStreamCaptureStatus cst = cudaStreamCaptureStatusNone;
            unsigned long long cid = 0;
            if (cudaStreamGetCaptureInfo_v2(s, &cst, &cid, &cgraph, &deps, &ndeps) == cudaSuccess && cst == cudaStreamCaptureStatusActive && cgraph &&
                cudaGraphConditionalHandleCreate(&a.cond, cgraph, 1, cudaGraphCondAssignDefault) == cudaSuccess)
                a.use_cond = 1;
            else { cudaGetLastError(); cgraph = nullptr; }
        }
        if (a.fz.frozen) k_tail_steady<true><<<nblk(L, 256), 256, 0, s>>>(st, ts, a, h->p2p);
        else k_tail_steady<false><<<nblk(L, 256), 256, 0, s>>>(st, ts, a, h->p2p);
        CK(cudaGetLastError());
        h->n_launch += 1;
        if (a.use_cond) {
            cudaStreamCaptureStatus cst2 = cudaStreamCaptureStatusNone;
            unsigned long long cid2 = 0;
            CK(cudaStreamGetCaptureInfo_v2(s, &cst2, &cid2, &cgraph, &deps, &ndeps));      // (now: the steady kernel's node)
            cudaGraphNodeParams np = {};
            np.type = cudaGraphNodeTypeConditional;
            np.conditional.handle = a.cond; np.conditional.type = cudaGraphCondTypeIf; np.conditional.size = 1;
            cudaGraphNode_t cnode = nullptr;
            CK(cudaGraphAddNode(&cnode, cgraph, deps, ndeps, &np));
            CK(cudaStreamBeginCaptureToGraph(h->cap_stream, np.conditional.phGraph_out[0], nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal));
            int rc = full_chain(h, dmap_out, out_cap, out_ld, h->cap_stream);
            cudaError_t ce = cudaStreamEndCapture(h->cap_stream, nullptr);
            if (rc) return rc;
            CK(ce);
            CK(cudaStreamUpdateCaptureDependencies(s, &cnode, 1, cudaStreamSetCaptureDependencies));
            // (the body's six kernels are not counted: they launch only in a sweep the steady kernel could not close)
        } else {
            int rc = full_chain(h, dmap_out, out_cap, out_ld, s);
            if (rc) return rc;
            h->n_launch += 6;
        }
    }
    chain_advance(h, xout, (out_ld == L && out_cap == L) ? dmap_out : nullptr);
    if (h->join_pending) { CK(cudaStreamWaitEvent(s, h->ev_join, 0)); h->join_pending = false; }
    return ICMSLAM_OK;
}

// the full chain (tail.cuh): everything after k_tail_steady -- the fused entry, then the filter chain
static int full_chain(icmslam_handle* h, double* dmap_out, int out_cap, int64_t out_ld, cudaStream_t s)
{
    const int L = h->Lcap;
    DevState* st = h->d_st;
    double* raw_x = h->d_raw;
    double* raw_y = h->d_raw + L;
    k_fused_means<<<nblk(L, 256), 256, 0, s>>>(st, h->d_fsum_x, h->d_fsum_y, h->d_cnt, h->d_map_in, h->d_map_in + L, 1.0 / h->fix_scale, h->dcfg.cota,
                                               h->d_newraw, raw_x, raw_y, h->d_kflag, L, h->d_blk_kept, h->ex.d_farbits, h->n_tiles * 4, h->p2p, h->d_ts,
                                               h->d_cnt, st, h->d_sh_x, h->d_sh_y, h->d_sh_k, h->fz, h->d_counts);
    CK(cudaGetLastError());
    return filter_chain(h, raw_x, raw_y, nullptr, dmap_out, out_cap, out_ld, s, true);
}

// streams and events of the chunk-pipelined host sweep, created on first use
static bool pipe_ready(icmslam_handle* h)
{
    if (h->pipe_events) return true;
    if (cudaStreamCreateWithFlags(&h->h2d_stream.p, cudaStreamNonBlocking) != cudaSuccess) { h->pipe_chunks = 1; return false; }
    for (int i = 0; i < 16; ++i)
        if (cudaEventCreateWithFlags(&h->ev_in[i].p, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&h->ev_out[i].p, cudaEventDisableTiming) != cudaSuccess) { h->pipe_chunks = 1; return false; }
    h->pipe_events = true;
    return true;
}

// the landmark each observation was matched with, for the RUNNING view (pass 0, reference-mode sweeps): allocated on first use
static int ensure_seen(icmslam_handle* h)
{
    if (h->ex.d_seen_x && h->ex.d_seen_y) return ICMSLAM_OK;
    CK(h->ex.d_seen_x.alloc((size_t)h->n_cap));      // (the room of the per-observation arrays: an append grows them together)
    CK(h->ex.d_seen_y.alloc((size_t)h->n_cap));
    return ICMSLAM_OK;
}

// One sweep on device-resident data.  The previous map is in h->d_map_in (2 x Lcap); L_in is its
// width known on the host, or -1 when only the device knows it (= landmarks_actuales, chained
// sweeps).  Poses are read from xin (3 x T, ldin) and the updated poses written to xout (3 x T,
// ldout); xin == xout is allowed (the fused path then goes through the internal double buffer).
// The filtered map goes to dmap_out.
static int sweep_core(icmslam_handle* h, const double* xin, int64_t ldin, double* xout, int64_t ldout, const double* x0,
                      const icmslam_sweep_opts& o, int L_in, double* dmap_out, int out_cap, int64_t out_ld, const HostPipe* hp = nullptr)
{
    const int T = h->T, L = h->Lcap;
    const int64_t n = h->n;
    cudaStream_t s = h->stream;
    DevState* st = h->d_st;
    const double* min_x = h->d_map_in;
    const double* min_y = h->d_map_in + L;
    double* raw_x = h->d_raw;
    double* raw_y = h->d_raw + L;
    const bool timing = (o.reserved & 2) != 0;
    const bool collect = (o.reserved & 1) != 0;
    unsigned long long* iters = collect ? &st->newton_iters : nullptr;
    const bool use_fused = fused_mode(h, o);
    const int n_search_cap = L_in < 0 ? L : (L_in > 0 ? L_in : 1);

    h->begin_L = L_in < 0 ? L : L_in;
    if (!(use_fused && h->ch.grid_map == h->d_map_in)) {
        k_sweep_begin<<<1, 1, 0, s>>>(st, h->d_ts, h->begin_L);
        CK(cudaGetLastError());
        h->n_launch += 1;
    }
    int rc;
    if (use_fused) {
        rc = ensure_stats_clean(h);
        if (rc) return rc;
        double* kout = xout;
        int64_t kld = ldout;
        if (xin == xout) { kout = (xin == h->ds.d_x2) ? h->ds.d_x : h->ds.d_x2; kld = T; }
        rc = fused_part_a(h, xin, ldin, kout, kld, x0, o, n_search_cap, /*overlap=*/kout == xout, hp);
        if (rc) return rc;
        if (kout != xout) CK(cudaMemcpy2DAsync(xout, (size_t)ldout * 8, kout, (size_t)kld * 8, (size_t)T * 8, 3, cudaMemcpyDeviceToDevice, s));
        // The tail's chain of small kernels runs beside the solve's waves only if the block scheduler prefers it: on the handle's
        // own highest-priority stream (the solve is on the lowest-priority side stream).  A caller's stream joins both at the end.
        cudaStream_t ts_ = s;
        if (h->join_pending && h->own_stream && s != h->own_stream) {
            ts_ = h->own_stream;
            CK(cudaStreamWaitEvent(ts_, h->ev_fork, 0));
        } else if (h->tail_wait_fork) {
            CK(cudaStreamWaitEvent(ts_, h->ev_fork, 0));      // (chunked: the last association launch is on another stream)
        }
        rc = fused_part_b(h, ts_);
        if (rc) return rc;
        rc = fused_part_c(h, kout, dmap_out, out_cap, out_ld, ts_);
        if (rc) return rc;
        if (ts_ != s) { CK(cudaEventRecord(h->ev_tail, ts_)); CK(cudaStreamWaitEvent(s, h->ev_tail, 0)); }
        return ICMSLAM_OK;
    } else {
        h->ch.stats_clean = false;
        CK(cudaMemsetAsync(h->d_cnt, 0, ((size_t)L + 1) * sizeof(int), s));
        CK(cudaMemsetAsync(h->d_counts, 0, (size_t)L * sizeof(double), s));
        if (xin != xout) CK(cudaMemcpy2DAsync(xout, (size_t)ldout * 8, xin, (size_t)ldin * 8, (size_t)T * 8, 3, cudaMemcpyDeviceToDevice, s));
        double* dx = xout;
        const int64_t ldx = ldout;
        CK(cudaMemsetAsync(h->d_sum_x, 0, (size_t)L * 8, s));
        CK(cudaMemsetAsync(h->d_sum_y, 0, (size_t)L * 8, s));
        LandmarkGrid& G = h->scratch_grid;
        rc = build_fgrid(h, G, min_x, min_y, &st->lsearch, n_search_cap);
        if (rc) return rc;
        h->n_launch += 5;
        // (the generic sweep covers the handle's whole trajectory, or the whole batch: column 0 is a first pose either way)
        TrajLayout lay = traj_layout(h, x0);
        lay.first = 1;
        PoseArrays A;
        A.x = dx; A.ldx = ldx; A.odo = h->ds.d_odo; A.ldo = T; A.u = h->ds.d_u; A.ldu = T;
        A.lay = lay;
        A.off = h->ex.d_off; A.T = T;
        if (timing) CK(cudaEventRecord(h->ev[0], s));
        k_assoc<<<148 * 8, 256, 0, s>>>(T, h->ex.d_off, h->ex.d_bx, h->ex.d_by, dx, ldx, lay, G.geom, G.start, G.pts, G.idx,
                                        h->thr2_hi, h->ex.d_c, h->ds.d_nfar, h->d_sum_x, h->d_sum_y, h->d_cnt);
        CK(cudaGetLastError());
        h->n_launch += 1;
        if (timing) CK(cudaEventRecord(h->ev[1], s));
        // new labels: one per scan that has a far observation, numbered in time order
        k_flag_positive<<<nblk(T, 256), 256, 0, s>>>(h->ds.d_nfar, T, h->ds.d_flag);
        CK(cudaGetLastError());
        rc = exclusive_sum(h, h->ds.d_flag, h->ds.d_prefix, T);
        if (rc) return rc;
        k_new_labels<<<148 * 4, 256, 0, s>>>(T, h->ex.d_off, h->ex.d_bx, h->ex.d_by, dx, ldx, lay, st, h->ds.d_nfar, h->ds.d_prefix,
                                             L, h->ex.d_c, h->d_sum_x, h->d_sum_y, h->d_cnt);
        CK(cudaGetLastError());
        h->n_launch += 2;
        const bool running = o.map_view == ICMSLAM_VIEW_RUNNING;
        if (running) {
            if (!h->ex.d_sorted) {
                CK(h->ex.d_keys_out.alloc((size_t)n)); CK(h->ex.d_iota.alloc((size_t)n)); CK(h->ex.d_sorted.alloc((size_t)n));
                k_iota<<<nblk(n, 256), 256, 0, s>>>((int)n, h->ex.d_iota);
                CK(cudaGetLastError());
            }
            rc = ensure_seen(h);
            if (rc) return rc;
            rc = exclusive_sum(h, h->d_cnt, h->d_seg, L);
            if (rc) return rc;
            int end_bit = 1;
            while ((1ll << end_bit) < (long long)L + 1 && end_bit < 32) ++end_bit;
            size_t bytes = 0;
            CK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const unsigned*)h->ex.d_c.p, (unsigned*)h->ex.d_keys_out.p, h->ex.d_iota.p, h->ex.d_sorted.p,
                                               (int)n, 0, end_bit, s));
            if (bytes > h->sort_bytes) {      // (its own workspace: never invalidates the scans' one that captured graphs use)
                h->sort_bytes = 0;
                CK(h->d_sort_ws.alloc(bytes));
                h->sort_bytes = bytes;
            }
            CK(cub::DeviceRadixSort::SortPairs(h->d_sort_ws, bytes, (const unsigned*)h->ex.d_c.p, (unsigned*)h->ex.d_keys_out.p, h->ex.d_iota.p, h->ex.d_sorted.p,
                                               (int)n, 0, end_bit, s));
            k_running_mean<<<nblk(L, 128), 128, 0, s>>>(st, h->d_seg, h->d_cnt, h->ex.d_sorted, h->ex.d_scan_of, h->ex.d_bx, h->ex.d_by, dx, ldx,
                                                        lay, h->ex.d_seen_x, h->ex.d_seen_y, raw_x, raw_y, L);
            CK(cudaGetLastError());
            h->n_launch += 1;
        }
        k_means_flags<<<nblk(L, 256), 256, 0, s>>>(st, h->d_sum_x, h->d_sum_y, h->d_cnt, h->dcfg.cota, running ? 1 : 0, raw_x, raw_y,
                                                   h->d_kflag, L, h->d_blk_kept, h->grid.bb, h->d_ts);
        CK(cudaGetLastError());
        h->n_launch += 1;
        ObsArrays O;
        O.bx = h->ex.d_bx; O.by = h->ex.d_by; O.d = h->ex.d_d; O.beam = h->ex.d_beam; O.ang = h->ds.d_ang;
        SeenSrc S;
        S.view = o.map_view; S.c = h->ex.d_c; S.seen_x = h->ex.d_seen_x; S.seen_y = h->ex.d_seen_y;
        S.raw_x = raw_x; S.raw_y = raw_y; S.min_x = min_x; S.min_y = min_y;
        S.lsearch_ptr = &st->lsearch;
        if (timing) CK(cudaEventRecord(h->ev[2], s));
        if (o.schedule == ICMSLAM_SCHED_REDBLACK) {
            k_pose_colour<<<nblk(T, 128), 128, 0, s>>>(1, h->dcfg, A, O, S, o.solver, o.newton_tol, o.newton_maxit, iters);
            CK(cudaGetLastError());
            k_pose_colour<<<nblk(T, 128), 128, 0, s>>>(0, h->dcfg, A, O, S, o.solver, o.newton_tol, o.newton_maxit, iters);
            CK(cudaGetLastError());
            h->n_launch += 2;
        } else {
            k_pose_walk<<<h->traj_K > 0 ? h->traj_K : 1, WARP, 0, s>>>(h->dcfg, A, O, S, o.solver, o.newton_tol, o.newton_maxit, iters);
            CK(cudaGetLastError());
            h->n_launch += 1;
        }
        if (timing) CK(cudaEventRecord(h->ev[3], s));
    }
    h->ch.timed_fused = false;
    h->ch.grid_map = nullptr;
    h->ch.hint_map = nullptr;
    // Mapa.filtrar (sensors.py:165-166)
    rc = filter_chain(h, raw_x, raw_y, nullptr, dmap_out, out_cap, out_ld, s, false);
    if (rc) return rc;
    h->n_launch += 5;
    h->ch.rawcnt_valid = true;
    h->ch.lact_dirty = true;
    return ICMSLAM_OK;
}

extern "C" int icmslam_sweep(icmslam_handle* h, const double* map_in, int32_t L_in, int64_t ld_map_in, double* x, int64_t ld_x,
                             const double* x0, double* map_out, int32_t cap_out, int64_t ld_map_out, int32_t* L_out,
                             const icmslam_sweep_opts* opts, int32_t memspace)
{
    if (!h || !h->extracted || !x || !x0 || L_in < 0 || L_in > h->Lcap || ld_x < h->T || (L_in > 0 && (!map_in || ld_map_in < L_in)))
        return ICMSLAM_ERR_INVALID;
    if (map_out && (cap_out <= 0 || ld_map_out < cap_out)) return ICMSLAM_ERR_INVALID;
    icmslam_sweep_opts o;
    default_opts(o, opts);
    CK(cudaSetDevice(h->cfg.device));
    {
        int rc = ensure_layout(h);
        if (rc) return rc;
    }
    const int T = h->T, L = h->Lcap;
    cudaStream_t s = h->stream;
    if (h->first_empty) {   // sensors.py:137-139: inputs returned unchanged
        // Mapa.clear_obs (sensors.py:133) happens before the early return of :137-139 (a sweep rewrites every count itself)
        CK(cudaMemsetAsync(h->d_counts, 0, (size_t)L * sizeof(double), s));
        if (map_out && L_in > 0) {
            int w = L_in < cap_out ? L_in : cap_out;
            CK(cudaMemcpy2DAsync(map_out, (size_t)ld_map_out * 8, map_in, (size_t)ld_map_in * 8, (size_t)w * 8, 2, cudaMemcpyDefault, s));
            CK(cudaStreamSynchronize(s));
        }
        if (L_out) *L_out = L_in;
        return ICMSLAM_EMPTY_FIRST_SCAN;
    }
    if (h->last_empty && T > 1) return ICMSLAM_ERR_EMPTY_LAST;
    const double* xin = x;
    double* xout = x;
    int64_t ldin = ld_x, ldout = ld_x;
    bool continued = false;
    if (memspace == ICMSLAM_HOST && L_in > 0 && L_in == h->last_map_L && h->ch.grid_map != nullptr && h->ch.grid_map == h->d_map_in &&
        h->h_map_pin && memcmp(map_in, h->h_map_pin, (size_t)L_in * 8) == 0 &&
        memcmp(map_in + ld_map_in, h->h_map_pin + L, (size_t)L_in * 8) == 0) {
        // the caller hands back the map the previous sweep returned: it is already on the device (the current map buffer),
        // with its grid, hints and run records
        continued = true;
    }
    h->last_map_L = -1;
    // a link of a map chain in the default mode: the poses go up, through the kernels and back in chunks (fused_part_a)
    HostPipe pipe;
    const bool piped = continued && fused_mode(h, o) && o.reserved == 0 && h->use_runs && h->side_stream && h->seg_first && h->seg_last &&
                       h->seg_lo == 0 && h->pipe_chunks > 1 && h->n_tiles >= h->pipe_tiles_min * h->pipe_chunks && pipe_ready(h);
    if (memspace == ICMSLAM_HOST) {
        if (!piped) CK(cudaMemcpy2DAsync(h->ds.d_x, (size_t)T * 8, x, (size_t)ld_x * 8, (size_t)T * 8, 3, cudaMemcpyHostToDevice, s));
        h->bytes_h2d += (int64_t)3 * T * 8;
        h->ch.ppar_of = nullptr;
        xin = h->ds.d_x; ldin = T;
        xout = h->ds.d_x2; ldout = T;
        pipe.x = x; pipe.ld = ld_x; pipe.chunks = h->pipe_chunks;
    }
    if (!continued) {
        if (L_in > 0) {
            CK(cudaMemcpy2DAsync(h->d_map_in, (size_t)L * 8, map_in, (size_t)ld_map_in * 8, (size_t)L_in * 8, 2, cudaMemcpyDefault, s));
            if (memspace == ICMSLAM_HOST) h->bytes_h2d += (int64_t)2 * L_in * 8;
        }
        h->ch.grid_map = nullptr;
        h->ch.hint_map = nullptr;
    }
    const bool own_out = (memspace == ICMSLAM_HOST || !map_out);
    h->d2h_done = false;
    if (memspace == ICMSLAM_HOST) { h->d2h_x = x; h->d2h_ld = ld_x; }
    int rc = sweep_core(h, xin, ldin, xout, ldout, x0, o, L_in, own_out ? h->d_map_out : map_out, own_out ? L : cap_out,
                        own_out ? (int64_t)L : ld_map_out, piped ? &pipe : nullptr);
    h->d2h_x = nullptr;
    if (rc) return rc;
    if (own_out) {      // mapa_refinado becomes the handle's current map (icmslam_get_map, and the map chain a caller may continue)
        std::swap(h->d_map_in, h->d_map_out);
    }
    if (memspace == ICMSLAM_HOST) {
        if (!h->d2h_done) CK(cudaMemcpy2DAsync(x, (size_t)ld_x * 8, xout, (size_t)T * 8, (size_t)T * 8, 3, cudaMemcpyDeviceToHost, s));
        h->bytes_d2h += (int64_t)3 * T * 8 + (int64_t)sizeof(DevState);
        // the whole map buffer comes back with the state in ONE asynchronous copy into pinned memory (its width is only known on
        // the device until then); the caller's array -- usually pageable -- is then filled by a host copy
        if (map_out && !h->h_map_pin) CK(h->h_map_pin.alloc((size_t)2 * L));
        if (map_out) {
            CK(cudaMemcpyAsync(h->h_map_pin, h->d_map_in, (size_t)2 * L * sizeof(double), cudaMemcpyDeviceToHost, s));
            h->bytes_d2h += (int64_t)2 * L * 8;       // (what actually crosses the bus: the whole buffer, not only the live columns)
        }
        rc = sync_state(h);
        if (rc) return rc;
        int status = status_from_state(h->h_st);
        if (status) return status;
        const int newL = h->h_st->new_l;
        if (map_out) {
            int w = newL < cap_out ? newL : cap_out;
            if (w > 0) {
                memcpy(map_out, h->h_map_pin, (size_t)w * 8);
                memcpy(map_out + ld_map_out, h->h_map_pin + L, (size_t)w * 8);
                if (w == newL) h->last_map_L = newL;       // the caller received all of it (see `continued` above)
            }
        }
        if (L_out) *L_out = newL;
        return ICMSLAM_OK;
    }
    if (L_out) {   // device buffers, but the caller wants the new width now: one 4-byte round trip
        rc = sync_state(h);
        if (rc) return rc;
        int status = status_from_state(h->h_st);
        if (status) return status;
        *L_out = h->h_st->new_l;
    }
    return ICMSLAM_OK;
}

// ---- the driver loop (sensors.py:302-315): N sweeps with everything resident on the device -------
extern "C" int icmslam_set_map(icmslam_handle* h, const double* map, int32_t L_map, int64_t ld, int32_t memspace)
{
    if (!h || L_map < 0 || L_map > h->Lcap || (L_map > 0 && (!map || ld < L_map))) return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    int rc = ensure_layout(h);
    if (rc) return rc;
    if (L_map > 0)
        CK(cudaMemcpy2DAsync(h->d_map_in, (size_t)h->Lcap * 8, map, (size_t)ld * 8, (size_t)L_map * 8, 2, cudaMemcpyDefault, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->ch.grid_map = nullptr;
    h->ch.hint_map = nullptr;
    return icmslam_set_landmarks_actuales(h, L_map);
}

extern "C" int icmslam_get_map(icmslam_handle* h, double* map, int32_t cap, int64_t ld, int32_t* L_map, int32_t memspace)
{
    if (!h || !L_map) return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    int rc = sync_state(h);
    if (rc) return rc;
    int status = status_from_state(h->h_st);
    if (status) return status;
    *L_map = h->lact_host;
    int w = h->lact_host < cap ? h->lact_host : cap;
    if (map && w > 0) {
        CK(cudaMemcpy2DAsync(map, (size_t)ld * 8, h->d_map_in, (size_t)h->Lcap * 8, (size_t)w * 8, 2, cudaMemcpyDefault, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return ICMSLAM_OK;
}

// Poses resident on the device between calls (ICM.positions, sensors.py:104): icmslam_set_poses uploads
// x (3 x T); icmslam_iterate with x == NULL then sweeps the resident poses with no copies at all;
// icmslam_get_poses reads them back.
extern "C" int icmslam_set_poses(icmslam_handle* h, const double* x, int64_t ld_x, int32_t memspace)
{
    if (!h || !h->ds.d_x || !x || ld_x < h->T) return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    int rc = ensure_layout(h);
    if (rc) return rc;
    const int T = h->T;
    CK(cudaMemcpy2DAsync(h->ds.d_x, (size_t)T * 8, x, (size_t)ld_x * 8, (size_t)T * 8, 3, cudaMemcpyDefault, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->ch.x_cur = 0;
    h->ch.ppar_of = nullptr;
    return ICMSLAM_OK;
}

extern "C" int icmslam_get_poses(icmslam_handle* h, double* x, int64_t ld_x, int32_t memspace)
{
    if (!h || !h->ds.d_x || !x || ld_x < h->T) return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    const int T = h->T;      // (the resident poses have leading dimension cap_T, which is T unless an append grew the log)
    CK(cudaMemcpy2DAsync(x, (size_t)ld_x * 8, cur_x(h), (size_t)h->cap_T * 8, (size_t)T * 8, 3, cudaMemcpyDefault, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return ICMSLAM_OK;
}

extern "C" int icmslam_iterate(icmslam_handle* h, double* x, int64_t ld_x, const double* x0, int32_t n_sweeps,
                               const icmslam_sweep_opts* opts, int32_t memspace)
{
    if (!h || !h->extracted || !x0 || (x && ld_x < h->T) || n_sweeps < 0) return ICMSLAM_ERR_INVALID;
    icmslam_sweep_opts o;
    default_opts(o, opts);
    CK(cudaSetDevice(h->cfg.device));
    {
        int rc = ensure_layout(h);
        if (rc) return rc;
    }
    const int T = h->T, L = h->Lcap;
    cudaStream_t s = h->stream;
    h->last_map_L = -1;
    if (h->seg_first && h->first_empty) return ICMSLAM_EMPTY_FIRST_SCAN;
    if (h->seg_last && h->last_empty && T > 1) return ICMSLAM_ERR_EMPTY_LAST;
    const bool fused = fused_mode(h, o);
    if (h->p2p.on && !fused) return ICMSLAM_ERR_UNSUPPORTED;      // only the restated parallel sweep partitions in time
    if (x) {
        CK(cudaMemcpy2DAsync(h->ds.d_x, (size_t)T * 8, x, (size_t)ld_x * 8, (size_t)T * 8, 3, cudaMemcpyDefault, s));
        h->ch.x_cur = 0;
        h->ch.ppar_of = nullptr;
    }
    const bool graph_ok = fused && h->use_graph && s != nullptr && (o.reserved & 3) == 0;
    for (int k = 0; k < n_sweeps; ++k) {
        double* src = cur_x(h);
        double* dst = next_x(h);
        if (fused) {      // (outside the graph) projection parameters of poses that did not come out of the previous sweep's solve, and
                          // clean statistics after a sweep of another mode
            int rc = ensure_ppar(h, src, T, x0, ppar_for(h, src));
            if (rc) return rc;
            rc = ensure_stats_clean(h);
            if (rc) return rc;
        }
        if (graph_ok && h->ch.grid_map == h->d_map_in) {
            // steady state: the whole sweep (memsets + 15 kernels) replays as one CUDA graph
            icmslam_handle::GraphSlot* slot = nullptr;
            for (auto& g : h->graphs)
                if (g.exec && g.src == src && g.map_in == h->d_map_in && g.x0[0] == x0[0] && g.x0[1] == x0[1] && g.x0[2] == x0[2] &&
                    g.tol == o.newton_tol && g.maxit == o.newton_maxit && g.lm == h->ch.lm_cur && same_freeze(g.fz, h->fz)) slot = &g;
            if (!slot) {
                for (auto& g : h->graphs) if (!g.exec) { slot = &g; break; }
                if (!slot) { drop_graphs(h); slot = &h->graphs[0]; }
                cudaGraph_t graph = nullptr;
                const int64_t nl0 = h->n_launch;
                const icmslam_handle::Chain ch0 = h->ch;      // (the capture only records the sweep: each launch below advances the chain)
                CK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
                h->in_own_capture = true;
                int rc = sweep_core(h, src, T, dst, T, x0, o, -1, h->d_map_out, L, L);
                cudaError_t ce = cudaStreamEndCapture(s, &graph);
                h->in_own_capture = false;
                h->ch = ch0;
                const int launches = (int)(h->n_launch - nl0);
                h->n_launch = nl0;
                if (rc || ce != cudaSuccess || !graph) {
                    if (graph) cudaGraphDestroy(graph);
                    cudaGetLastError();
                    if (!rc) snprintf(h->err, sizeof h->err, "graph capture of the sweep failed (%s)", cudaGetErrorString(ce));
                    return rc ? rc : ICMSLAM_ERR_CUDA;
                }
                ce = cudaGraphInstantiate(&slot->exec.p, graph, cudaGraphInstantiateFlagUseNodePriority);   // (nodes keep the priority of the stream they were captured on)
                cudaGraphDestroy(graph);
                if (ce != cudaSuccess) { slot->exec.p = nullptr; snprintf(h->err, sizeof h->err, "cudaGraphInstantiate: %s", cudaGetErrorString(ce)); return ICMSLAM_ERR_CUDA; }
                slot->src = src; slot->map_in = h->d_map_in; slot->x0[0] = x0[0]; slot->x0[1] = x0[1]; slot->x0[2] = x0[2];
                slot->tol = o.newton_tol; slot->maxit = o.newton_maxit; slot->lm = h->ch.lm_cur; slot->fz = h->fz; slot->launches = launches;
            }
            CK(cudaGraphLaunch(slot->exec, s));
            h->n_launch += slot->launches;
            chain_advance(h, dst, h->d_map_out);
        } else {
            int rc = sweep_core(h, src, T, dst, T, x0, o, -1, h->d_map_out, L, L);
            if (rc) return rc;
        }
        end_sweep(h);
    }
    if (x) {
        CK(cudaMemcpy2DAsync(x, (size_t)ld_x * 8, cur_x(h), (size_t)T * 8, (size_t)T * 8, 3, cudaMemcpyDefault, s));
        if (memspace == ICMSLAM_HOST) {
            int rc = sync_state(h);
            if (rc) return rc;
            return status_from_state(h->h_st);
        }
    }
    return ICMSLAM_OK;
}

// ---- a batch of independent trajectories in one handle (BASELINE configs[4]) ---------------------------------------------
// Trajectory k covers columns start[k] .. start[k+1]-1 (start[0] = 0, start[K] = T).  The caller has checked the arguments; this
// checks the scans and changes the handle only when it accepts the layout.
static int set_layout(icmslam_handle* h, const std::vector<int>& start, const double* x0s, int64_t ld_x0s)
{
    const int K = (int)start.size() - 1;
    // every trajectory needs a non-empty first and last scan (the reference returns early / raises otherwise, sensors.py:137, :148)
    std::vector<int> off((size_t)h->T + 1);
    CK(cudaMemcpyAsync(off.data(), h->ex.d_off, ((size_t)h->T + 1) * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    bool odd = false;
    std::vector<int> traj((size_t)h->T);
    for (int k = 0; k < K; ++k) {
        const int a = start[k], b = start[k + 1] - 1;
        if (off[a + 1] == off[a] || off[b + 1] == off[b]) return ICMSLAM_ERR_UNSUPPORTED;
        odd = odd || (a & 1);
        std::fill(traj.begin() + a, traj.begin() + b + 1, k);
    }
    DevBuf<int> d_start, d_traj; DevBuf<double> d_x0;
    CK(d_start.alloc((size_t)K + 1)); CK(d_traj.alloc((size_t)h->T)); CK(d_x0.alloc((size_t)3 * K));
    CK(cudaMemcpyAsync(d_start, start.data(), ((size_t)K + 1) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d_traj, traj.data(), (size_t)h->T * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpy2DAsync(d_x0, (size_t)K * 8, x0s, (size_t)ld_x0s * 8, (size_t)K * 8, 3, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    drop_graphs(h);      // (before the old buffers go: graphs hold them)
    h->d_traj_start = std::move(d_start); h->d_traj_of = std::move(d_traj); h->d_x0s = std::move(d_x0);
    h->traj_K = K; h->traj_odd = odd;
    h->first_empty = false; h->last_empty = false;
    h->ch.ppar_of = nullptr;
    return ICMSLAM_OK;
}

extern "C" int icmslam_set_batch(icmslam_handle* h, int32_t traj_T, const double* x0s, int64_t ld_x0s, int32_t K)
{
    if (!h || !h->extracted) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    int rc = ensure_layout(h);
    if (rc) return rc;
    if (traj_T <= 0) {
        drop_graphs(h);
        h->traj_K = 0; h->traj_odd = false; h->d_traj_start.reset(); h->d_traj_of.reset(); h->d_x0s.reset();
        h->ch.ppar_of = nullptr;
        return ICMSLAM_OK;
    }
    if (!x0s || K <= 0 || ld_x0s < K || (int64_t)traj_T * K != h->T || traj_T < 3 || !h->fused_ok) return ICMSLAM_ERR_INVALID;
    std::vector<int> start((size_t)K + 1);
    for (int k = 0; k <= K; ++k) start[k] = k * traj_T;
    return set_layout(h, start, x0s, ld_x0s);
}

extern "C" int icmslam_set_batch_lengths(icmslam_handle* h, const int32_t* lengths, int32_t K, const double* x0s, int64_t ld_x0s)
{
    if (!h || !h->extracted) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    int rc = ensure_layout(h);
    if (rc) return rc;
    if (!lengths || !x0s || K <= 0 || ld_x0s < K || !h->fused_ok) return ICMSLAM_ERR_INVALID;
    std::vector<int> start((size_t)K + 1, 0);
    int64_t sum = 0;
    for (int k = 0; k < K; ++k) {
        if (lengths[k] < 3) return ICMSLAM_ERR_INVALID;
        sum += lengths[k];
        if (sum > h->T) return ICMSLAM_ERR_INVALID;
        start[k + 1] = (int)sum;
    }
    if (sum != h->T) return ICMSLAM_ERR_INVALID;
    return set_layout(h, start, x0s, ld_x0s);
}

// ---- time-segment partition: one handle per GPU owns columns [t_lo, t_hi) of the T columns it loaded ------
extern "C" int icmslam_set_segment(icmslam_handle* h, int32_t t_lo, int32_t t_hi, int32_t is_first, int32_t is_last)
{
    if (!h || !h->extracted || t_lo < 0 || t_hi > h->T || t_lo >= t_hi || (t_lo & 1)) return ICMSLAM_ERR_INVALID;
    if ((!is_first && t_lo < 2) || (!is_last && t_hi > h->T - 1)) return ICMSLAM_ERR_INVALID;   // halo columns must exist
    int rc = ensure_layout(h);
    if (rc) return rc;
    h->seg_lo = t_lo; h->seg_hi = t_hi; h->seg_first = is_first ? 1 : 0; h->seg_last = is_last ? 1 : 0;
    h->n_tiles = nblk(t_hi - (t_lo - (is_first ? 0 : 1)), RT_TILE);
    h->n_solve_tiles = nblk(t_hi - t_lo, ST_OWN);
    // the record tiling moved: no tile holds records (epoch -1)
    CK(cudaMemsetAsync(h->ex.d_tile_epoch, 0xff, ((size_t)nblk(h->T + 1, RT_TILE) + 2) * sizeof(int), h->stream));
    drop_graphs(h);
    return ICMSLAM_OK;
}

extern "C" int icmslam_device_ptr(icmslam_handle* h, int32_t which, void** ptr, int64_t* count)
{
    if (!h || !ptr || !count) return ICMSLAM_ERR_INVALID;
    int rc = ensure_layout(h);      // (the poses with leading dimension T)
    if (rc) return rc;
    const int64_t L = h->Lcap;
    switch (which) {
    case ICMSLAM_PTR_SEG_REC: *ptr = h->d_seg_rec; *count = SEG_REC; break;
    case ICMSLAM_PTR_STAT_X: *ptr = h->d_fsum_x; *count = L; break;
    case ICMSLAM_PTR_STAT_Y: *ptr = h->d_fsum_y; *count = L; break;
    case ICMSLAM_PTR_STAT_N: *ptr = h->d_cnt; *count = L; break;
    case ICMSLAM_PTR_NEW_LABELS: *ptr = h->d_newraw; *count = 2 * L; break;
    case ICMSLAM_PTR_POSES: *ptr = cur_x(h); *count = 3 * (int64_t)h->T; break;
    case ICMSLAM_PTR_EXCHANGE: *ptr = h->d_exch; *count = h->exch_words; break;
    case ICMSLAM_PTR_SEG_REC_POSE: *ptr = h->d_seg_rec_pose; *count = SEG_REC; break;
    case ICMSLAM_PTR_SIDE_STREAM: *ptr = (void*)h->side_stream; *count = 1; break;
    default: return ICMSLAM_ERR_INVALID;
    }
    return ICMSLAM_OK;
}

// ---- peer-memory exchange (p2p.cuh): the ranks of a node open each other's exchange block, window and result buffer ---------
// icmslam_p2p_export: 3 CUDA IPC handles (64 bytes each: exchange block, window, result buffer) of this rank.
extern "C" int icmslam_p2p_export(icmslam_handle* h, void* handles, int64_t cap_bytes)
{
    if (!h || !handles || cap_bytes < (int64_t)(3 * sizeof(cudaIpcMemHandle_t)) || !h->d_exch) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    if (!h->d_win) {
        CK(h->d_win.alloc(1));
        CK(cudaMemset(h->d_win, 0, sizeof(P2PWin)));
        CK(h->d_res.alloc((size_t)h->exch_words));
        CK(cudaMemset(h->d_res, 0, (size_t)h->exch_words * 8));
    }
    cudaIpcMemHandle_t* out = (cudaIpcMemHandle_t*)handles;
    CK(cudaIpcGetMemHandle(&out[0], h->d_exch));
    CK(cudaIpcGetMemHandle(&out[1], h->d_win));
    CK(cudaIpcGetMemHandle(&out[2], h->d_res));
    return ICMSLAM_OK;
}

// icmslam_p2p_import: `all` = world x 3 handles in rank order (every rank's icmslam_p2p_export, gathered by the caller).  From then
// on icmslam_iterate on a segment handle (icmslam_set_segment) exchanges with the other ranks by itself: every rank must call it
// with the same number of sweeps, and no NCCL collective is needed inside a sweep.  Same node only (NVLink / PCIe peer access).
extern "C" int icmslam_p2p_import(icmslam_handle* h, int32_t rank, int32_t world, const void* all, int64_t bytes)
{
    if (!h || !all || world < 1 || world > P2P_MAX_WORLD || rank < 0 || rank >= world || !h->d_win ||
        bytes < (int64_t)world * 3 * (int64_t)sizeof(cudaIpcMemHandle_t))
        return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    drop_graphs(h);      // (before the old mappings are closed: graphs of the old exchange hold them through the pointer table)
    const cudaIpcMemHandle_t* hs = (const cudaIpcMemHandle_t*)all;
    void* tab[3 * P2P_MAX_WORLD] = {};
    for (int r = 0; r < world; ++r) {
        for (int k = 0; k < 3; ++k) {
            void* ptr = nullptr;
            if (r == rank) ptr = k == 0 ? (void*)h->d_exch : (k == 1 ? (void*)h->d_win : (void*)h->d_res);
            else {
                h->p2p_opened[3 * r + k].reset();
                CK(cudaIpcOpenMemHandle(&ptr, hs[3 * r + k], cudaIpcMemLazyEnablePeerAccess));
                h->p2p_opened[3 * r + k].p = ptr;
            }
            tab[k * P2P_MAX_WORLD + r] = ptr;      // three tables of P2P_MAX_WORLD pointers: exchange blocks, windows, result buffers
        }
    }
    if (!h->d_p2p_ptrs) CK(h->d_p2p_ptrs.alloc(3 * P2P_MAX_WORLD));
    CK(cudaMemcpy(h->d_p2p_ptrs, tab, sizeof tab, cudaMemcpyHostToDevice));
    P2PDev& p = h->p2p;
    p.on = world > 1 ? 1 : 0; p.rank = rank; p.world = world;
    p.exch = (const long long* const*)h->d_p2p_ptrs.p;
    p.win = (P2PWin* const*)(h->d_p2p_ptrs + P2P_MAX_WORLD);
    p.res = (const long long* const*)(h->d_p2p_ptrs + 2 * P2P_MAX_WORLD);
    p.my_res = h->d_res;
    p.words = h->exch_words;
    p.per = (h->exch_words + world - 1) / world;
    return ICMSLAM_OK;
}

// Sweep of one segment, part 1: the fused kernel on the resident poses; leaves this segment's record
// (boundary poses, far-scan count) in the ICMSLAM_PTR_SEG_REC buffer for the all-gather.
extern "C" int icmslam_seg_begin(icmslam_handle* h, const double* x0, const icmslam_sweep_opts* opts)
{
    if (!h || !h->extracted || !x0) return ICMSLAM_ERR_INVALID;
    {
        CK(cudaSetDevice(h->cfg.device));
        int rc = ensure_layout(h);
        if (rc) return rc;
    }
    if (!h->fused_ok) return ICMSLAM_ERR_INVALID;
    icmslam_sweep_opts o;
    default_opts(o, opts);
    if (!fused_mode(h, o)) return ICMSLAM_ERR_UNSUPPORTED;     // only the restated parallel sweep partitions in time (DESIGN.md)
    if (h->p2p.on) return ICMSLAM_ERR_UNSUPPORTED;      // (peer-memory exchange: the sweeps go through icmslam_iterate)
    h->last_map_L = -1;
    CK(cudaSetDevice(h->cfg.device));
    const int T = h->T, L = h->Lcap;
    cudaStream_t s = h->stream;
    if (h->seg_first && h->first_empty) return ICMSLAM_EMPTY_FIRST_SCAN;
    if (h->seg_last && h->last_empty && T > 1) return ICMSLAM_ERR_EMPTY_LAST;
    double* src = cur_x(h);
    double* dst = next_x(h);
    int rc = ensure_stats_clean(h);
    if (rc) return rc;
    h->begin_L = L;
    if (h->ch.grid_map != h->d_map_in) {
        k_sweep_begin<<<1, 1, 0, s>>>(h->d_st, h->d_ts, L);
        CK(cudaGetLastError());
    }
    // opts.reserved & 4: the caller gathers the boundary poses separately (icmslam_seg_halo) on the side stream, where the solve
    // then runs beside the label exchange, the reduction of the statistics and the tail
    h->seg_split = (o.reserved & 4) != 0 && h->side_stream && h->overlap_solve && (o.reserved & 2) == 0;
    rc = fused_part_a(h, src, T, dst, T, x0, o, L, /*overlap=*/h->seg_split);
    if (rc) return rc;
    if (h->seg_split) {
        k_seg_pack<<<1, 32, 0, s>>>(dst, T, h->seg_lo, h->seg_hi, h->d_ts, h->d_seg_rec, 0, 1);
        CK(cudaGetLastError());
        k_seg_pack<<<1, 32, 0, h->side_stream>>>(dst, T, h->seg_lo, h->seg_hi, h->d_ts, h->d_seg_rec_pose, 1, 0);
        CK(cudaGetLastError());
        CK(cudaEventRecord(h->ev_join, h->side_stream));
        h->n_launch += 1;
    } else {
        k_seg_pack<<<1, 32, 0, s>>>(dst, T, h->seg_lo, h->seg_hi, h->d_ts, h->d_seg_rec, 1, 1);
        CK(cudaGetLastError());
    }
    h->seg_dst = dst;
    h->n_launch += 1;
    return ICMSLAM_OK;
}

// part 1b (only after icmslam_seg_begin with opts.reserved & 4): `gathered` = the all-gather of every segment's
// ICMSLAM_PTR_SEG_REC_POSE record, issued by the caller on the handle's side stream (ICMSLAM_PTR_SIDE_STREAM).  Fills this
// segment's halo poses there; icmslam_seg_finish joins the side stream.
extern "C" int icmslam_seg_halo(icmslam_handle* h, const double* gathered, int32_t rank, int32_t world)
{
    if (!h || !gathered || !h->seg_dst || !h->seg_split || rank < 0 || rank >= world) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    k_seg_unpack<<<1, 32, 0, h->side_stream>>>(gathered, rank, world, h->seg_dst, h->T, h->T, h->d_st, h->d_ts, h->Lcap,
                                               ppar_for(h, h->seg_dst), 1, 0);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev_join, h->side_stream));
    h->n_launch += 1;
    return ICMSLAM_OK;
}

// part 2: `gathered` = world x SEG_REC doubles (device), the all-gather of every segment's record.  Fills this
// segment's halo poses, numbers its new labels globally and writes their statistics.  After this call the
// caller sum-reduces ICMSLAM_PTR_STAT_X / _Y / _N / _NEW_LABELS over the segments.
extern "C" int icmslam_seg_exchange(icmslam_handle* h, const double* gathered, int32_t rank, int32_t world)
{
    if (!h || !gathered || !h->seg_dst || rank < 0 || rank >= world) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    k_seg_unpack<<<1, 32, 0, h->stream>>>(gathered, rank, world, h->seg_dst, h->T, h->T, h->d_st, h->d_ts, h->Lcap,
                                          ppar_for(h, h->seg_dst), h->seg_split ? 0 : 1, 1);
    CK(cudaGetLastError());
    h->n_launch += 1;
    return fused_part_b(h, h->stream);
}

// part 3: landmark update + Mapa.filtrar on the reduced statistics (identical on every segment).
extern "C" int icmslam_seg_finish(icmslam_handle* h)
{
    if (!h || !h->seg_dst) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    const int L = h->Lcap;
    int rc = fused_part_c(h, h->seg_dst, h->d_map_out, L, L, h->stream);
    if (rc) return rc;
    h->seg_dst = nullptr;
    end_sweep(h);
    return ICMSLAM_OK;
}

// elapsed milliseconds of the dominant kernels of the LAST sweep run with opts.reserved & 2:
// out[0] = association (or the fused sweep kernel), out[1] = pose kernels (0 when fused).
extern "C" int icmslam_get_kernel_ms(icmslam_handle* h, double* out2)
{
    if (!h || !out2) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    float a = 0.f, b = 0.f;
    if (h->ch.timed_fused) {      // fused path: k_runs + k_assoc_tiles | k_solve_tile
        CK(cudaEventElapsedTime(&a, h->ev[0], h->ev[3]));
        CK(cudaEventElapsedTime(&b, h->ev[3], h->ev[1]));
        float r = 0.f;
        CK(cudaEventElapsedTime(&r, h->ev[0], h->ev[2]));
        h->last_runs_ms = r;
    } else {
        CK(cudaEventElapsedTime(&a, h->ev[0], h->ev[1]));
        if (!h->ch.timed_fused) CK(cudaEventElapsedTime(&b, h->ev[2], h->ev[3]));
    }
    out2[0] = a; out2[1] = b;
    return ICMSLAM_OK;
}

extern "C" int icmslam_get_transfer_bytes(icmslam_handle* h, int64_t* h2d, int64_t* d2h)
{
    if (!h || !h2d || !d2h) return ICMSLAM_ERR_INVALID;
    *h2d = h->bytes_h2d; *d2h = h->bytes_d2h;
    return ICMSLAM_OK;
}

extern "C" int icmslam_get_launch_count(icmslam_handle* h, int64_t* n)
{
    if (!h || !n) return ICMSLAM_ERR_INVALID;
    *n = h->n_launch;
    return ICMSLAM_OK;
}

extern "C" int icmslam_get_associations(icmslam_handle* h, int32_t* c, int32_t memspace)
{
    if (!h || !h->extracted || !c) return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaMemcpyAsync(c, h->ex.d_c, (size_t)h->n * sizeof(int), cudaMemcpyDefault, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return ICMSLAM_OK;
}

__global__ void k_counts_to_int(const double* __restrict__ cnt, int n, int* __restrict__ out)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int)cnt[i];
}

__global__ void k_counts_to_double(const int* __restrict__ cnt, int n, double* __restrict__ out)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)cnt[i];
}

extern "C" int icmslam_get_raw_map(icmslam_handle* h, double* raw_map, int32_t cap, int64_t ld, double* raw_counts, int32_t* raw_L,
                                   int32_t memspace)
{
    if (!h) return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    int rc = sync_state(h);
    if (rc) return rc;
    const int rl = h->h_st->raw_l;
    if (raw_L) *raw_L = rl;
    const int w = rl < cap ? rl : cap;
    if (raw_map && w > 0)
        CK(cudaMemcpy2DAsync(raw_map, (size_t)ld * 8, h->d_raw, (size_t)h->Lcap * 8, (size_t)w * 8, 2, cudaMemcpyDefault, h->stream));
    if (raw_counts && w > 0) {
        k_counts_to_double<<<nblk(w, 256), 256, 0, h->stream>>>(h->ch.rawcnt_valid ? h->d_rawcnt : h->d_cnt, w, h->d_tmp_a);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(raw_counts, h->d_tmp_a, (size_t)w * 8, cudaMemcpyDefault, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return ICMSLAM_OK;
}

// ---- the user-configurable model functions of the reference (sensors.py:170-282: h, g, fun_xn, fun_x, minimizar_xn, minimizar_x)
// for ONE pose, on the device, with every input given explicitly (the reference reads them from attributes of the object)
struct PoseEvalArgs {
    int op, n, has_next, maxit;
    double tol;
    const double* zd; const double* zang; const double* sx; const double* sy;   // n each (device)
    int* iota; double* bx; double* by;                                           // n each (device scratch)
    double xa[3], xb[3], ua[2], uc[2], o0[3], o1[3], o2[3], x[3];
    double* out;       // [0..2] pose, [3] energy, [4] evaluations / iterations
};

__global__ void k_pose_eval(const DevCfg cfg, const PoseEvalArgs a)
{
    for (int i = 0; i < a.n; ++i) {      // (one thread: the reference evaluates these one pose at a time)
        a.iota[i] = i;
        double s, c;
        sincos(a.zang[i], &s, &c);
        a.bx[i] = mul_rn(a.zd[i], c); a.by[i] = mul_rn(a.zd[i], s);      // ICM_SLAM.py:52-53
    }
    PoseProblem P;
    ObsArrays O;
    SeenSrc S;
    for (int j = 0; j < 3; ++j) { P.a[j] = a.xa[j]; P.b[j] = a.xb[j]; P.o0[j] = a.o0[j]; P.o1[j] = a.o1[j]; P.o2[j] = a.o2[j]; }
    P.ua[0] = a.ua[0]; P.ua[1] = a.ua[1]; P.uc[0] = a.uc[0]; P.uc[1] = a.uc[1];
    P.has_next = a.has_next; P.o = 0; P.n = a.n;
    O.bx = a.bx; O.by = a.by; O.d = a.zd; O.beam = a.iota; O.ang = a.zang;
    S.view = ICMSLAM_VIEW_RUNNING; S.c = nullptr; S.seen_x = a.sx; S.seen_y = a.sy; S.raw_x = S.raw_y = S.min_x = S.min_y = nullptr; S.lsearch_ptr = nullptr;
    double x[3] = {a.x[0], a.x[1], a.x[2]};
    double f = 0.0, cnt = 0.0;
    if (a.op == ICMSLAM_POSE_G) {                                   // g(xt, ut), sensors.py:206-211
        g_step(P.a, P.ua[0], P.ua[1], cfg.dt, x);
    } else if (a.op == ICMSLAM_POSE_H) {                            // h(xt, zt) with mapa_visto, sensors.py:175-204
        for (int i = 0; i < a.n; ++i) {
            double s, c;
            sincos(a.zang[i] + x[2] - ICM_HALFPI, &s, &c);
            const double dx = (x[0] + a.zd[i] * c) - a.sx[i], dy = (x[1] + a.zd[i] * s) - a.sy[i];
            f += dx * cfg.q1 * dx;
            f += dy * cfg.q2 * dy;
        }
    } else if (a.op == ICMSLAM_POSE_ENERGY) {                       // fun_xn / fun_x at x, sensors.py:224-282
        f = pose_energy(cfg, P, O, S, x);
    } else {
        double start[3];
        if (P.has_next) { for (int j = 0; j < 3; ++j) start[j] = (P.a[j] + P.b[j]) / 2.0; }      // sensors.py:221
        else g_step(P.a, P.ua[0], P.ua[1], cfg.dt, start);                                       // sensors.py:262
        if (a.op == ICMSLAM_POSE_MIN_NM) {
            cnt = (double)nelder_mead(cfg, P, O, S, start, x);
        } else {
            Moments M;
            moments_zero(M);
            for (int i = 0; i < a.n; ++i) moments_add(M, a.bx[i], a.by[i], a.sx[i] - start[0], a.sy[i] - start[1]);
            cnt = (double)newton_moments(cfg, P, M, start[0], start[1], start[2], a.tol, a.maxit, x);
        }
        f = pose_energy(cfg, P, O, S, x);
    }
    a.out[0] = x[0]; a.out[1] = x[1]; a.out[2] = x[2]; a.out[3] = f; a.out[4] = cnt;
}

extern "C" int icmslam_pose_eval(icmslam_handle* h, int32_t model, int32_t op, int32_t n, const double* z_d, const double* z_ang,
                                 const double* seen_x, const double* seen_y, const double* x_ant, const double* x_pos, const double* u_ant,
                                 const double* u_act, const double* odo, int64_t ld_odo, double* x, double* f, int32_t* n_eval,
                                 const icmslam_sweep_opts* opts)
{
    if (!h || n < 0 || !x || op < ICMSLAM_POSE_ENERGY || op > ICMSLAM_POSE_H) return ICMSLAM_ERR_INVALID;
    if (model != ICMSLAM_MODEL_UNICYCLE_LASER2D) return ICMSLAM_ERR_UNSUPPORTED;      // the one model the reference ships (and the sweep kernels implement)
    if (n > 0 && (!z_d || !z_ang || !seen_x || !seen_y)) return ICMSLAM_ERR_INVALID;
    const bool needs_prev = op != ICMSLAM_POSE_H;
    if (needs_prev && (!x_ant || !u_ant)) return ICMSLAM_ERR_INVALID;
    const bool full = op == ICMSLAM_POSE_ENERGY || op == ICMSLAM_POSE_MIN_NM || op == ICMSLAM_POSE_MIN_NEWTON;
    if (full && (!odo || ld_odo < (x_pos ? 3 : 2) || (x_pos && !u_act))) return ICMSLAM_ERR_INVALID;
    icmslam_sweep_opts o;
    default_opts(o, opts);
    CK(cudaSetDevice(h->cfg.device));
    cudaStream_t s = h->stream;
    const size_t nn = (size_t)(n > 0 ? n : 1);
    DevBuf<double> dbuf;
    DevBuf<int> ibuf;
    CK(dbuf.alloc(6 * nn + 8));
    if (ibuf.alloc(nn) != cudaSuccess) return ICMSLAM_ERR_ALLOC;
    PoseEvalArgs a;
    memset(&a, 0, sizeof a);
    a.op = op; a.n = n; a.has_next = x_pos ? 1 : 0; a.maxit = o.newton_maxit; a.tol = o.newton_tol;
    double* dz = dbuf; double* dang = dbuf + nn; double* dsx = dbuf + 2 * nn; double* dsy = dbuf + 3 * nn;
    a.zd = dz; a.zang = dang; a.sx = dsx; a.sy = dsy; a.bx = dbuf + 4 * nn; a.by = dbuf + 5 * nn; a.out = dbuf + 6 * nn; a.iota = ibuf;
    if (n > 0) {
        CK(cudaMemcpyAsync(dz, z_d, (size_t)n * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dang, z_ang, (size_t)n * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dsx, seen_x, (size_t)n * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dsy, seen_y, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    }
    for (int j = 0; j < 3; ++j) {
        a.x[j] = x[j];
        if (x_ant) a.xa[j] = x_ant[j];
        if (x_pos) a.xb[j] = x_pos[j];
        if (odo) { a.o0[j] = odo[j * ld_odo + 0]; a.o1[j] = odo[j * ld_odo + 1]; if (x_pos) a.o2[j] = odo[j * ld_odo + 2]; }
    }
    if (u_ant) { a.ua[0] = u_ant[0]; a.ua[1] = u_ant[1]; }
    if (u_act) { a.uc[0] = u_act[0]; a.uc[1] = u_act[1]; }
    double out[5] = {0, 0, 0, 0, 0};
    k_pose_eval<<<1, 1, 0, s>>>(h->dcfg, a);
    CK(cudaGetLastError());
    h->n_launch += 1;
    CK(cudaMemcpyAsync(out, a.out, sizeof out, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (op != ICMSLAM_POSE_ENERGY && op != ICMSLAM_POSE_H) { x[0] = out[0]; x[1] = out[1]; x[2] = out[2]; }
    if (f) *f = out[3];
    if (n_eval) *n_eval = (int32_t)out[4];
    return ICMSLAM_OK;
}

// instrumentation: the ring of %globaltimer marks (32 sweeps x 8 marks, nanoseconds; TailState::trace) and the sweep counters
extern "C" int icmslam_get_trace(icmslam_handle* h, uint64_t* out256, uint32_t* counters3)
{
    if (!h || !out256) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    TailState hts;
    CK(cudaMemcpy(&hts, h->d_ts, sizeof(TailState), cudaMemcpyDeviceToHost));
    memcpy(out256, hts.trace, sizeof hts.trace);
    if (counters3) { counters3[0] = hts.sweep_no; counters3[1] = hts.p2p_seq; counters3[2] = hts.halo_seq; }
    return ICMSLAM_OK;
}

extern "C" int icmslam_get_sweep_stats(icmslam_handle* h, int64_t* stats, int32_t n)
{
    if (!h || !stats || n < 0) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    int rc = sync_state(h);
    if (rc) return rc;
    const DevState* s = h->h_st;
    TailState hts;
    CK(cudaMemcpy(&hts, h->d_ts, sizeof(TailState), cudaMemcpyDeviceToHost));
    int64_t v[17] = {(int64_t)s->newton_iters, s->n_far_scans, s->raw_l, s->kept, s->new_l, s->n_ind, s->lsearch, s->status, s->dirty_tiles,
                     hts.epoch, (int64_t)h->n_tiles, hts.remap_identity, (int64_t)(h->last_runs_ms * 1e6), hts.n_dirty, hts.far_count, hts.steady_sweeps,
                     h->fz_fallbacks};
    for (int i = 0; i < n && i < 17; ++i) stats[i] = v[i];
    return ICMSLAM_OK;
}

__global__ void k_set_raw_l(DevState* st, int v) { st->raw_l = v; st->status = 0; }

extern "C" int icmslam_filter_map(icmslam_handle* h, const double* map_in, int64_t ld_in, const double* counts_in, int32_t L_in,
                                  double* map_out, int32_t cap_out, int64_t ld_out, double* counts_out, int32_t* L_out,
                                  int32_t memspace)
{
    if (!h || !map_in || !counts_in || L_in <= 0 || L_in > h->Lcap || ld_in < L_in || !L_out) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    const int L = h->Lcap;
    cudaStream_t s = h->stream;
    CK(cudaMemcpy2DAsync(h->d_tmp_a, (size_t)L * 8, map_in, (size_t)ld_in * 8, (size_t)L_in * 8, 2, cudaMemcpyDefault, s));
    CK(cudaMemcpyAsync(h->d_tmp_b, counts_in, (size_t)L_in * 8, cudaMemcpyDefault, s));
    k_set_raw_l<<<1, 1, 0, s>>>(h->d_st, L_in);
    CK(cudaGetLastError());
    k_flags_from_counts<<<nblk(L, 256), 256, 0, s>>>(h->d_tmp_b, L_in, h->dcfg.cota, h->d_kflag, L, h->d_blk_kept, h->grid.bb, h->d_ts);
    CK(cudaGetLastError());
    // (the result goes through the handle's spare map buffer and rewrites the Mapa state: whatever map chain the handle was
    //  continuing -- grid, hints, run records, the copy of the last returned map -- no longer describes that buffer)
    h->ch.grid_map = nullptr; h->ch.hint_map = nullptr; h->last_map_L = -1;
    int rc = filter_chain(h, h->d_tmp_a, h->d_tmp_a + L, h->d_tmp_b, h->d_map_out, L, L, s, false);
    if (rc) return rc;
    rc = sync_state(h);
    if (rc) return rc;
    int status = status_from_state(h->h_st);
    if (status) return status;
    const int newL = h->h_st->new_l;
    *L_out = newL;
    (void)memspace;
    int w = newL < cap_out ? newL : cap_out;
    if (map_out && w > 0)
        CK(cudaMemcpy2DAsync(map_out, (size_t)ld_out * 8, h->d_map_out, (size_t)L * 8, (size_t)w * 8, 2, cudaMemcpyDefault, s));
    if (counts_out && w > 0) CK(cudaMemcpyAsync(counts_out, h->d_counts, (size_t)w * 8, cudaMemcpyDefault, s));
    CK(cudaStreamSynchronize(s));
    return ICMSLAM_OK;
}

__global__ void k_set_lsearch(DevState* st, int v) { st->lsearch = v; }

extern "C" int icmslam_calc_cambio(icmslam_handle* h, const double* map_new, int32_t L_new, int64_t ld_new, const double* map_old,
                                   int32_t L_old, int64_t ld_old, double* out3, int32_t memspace)
{
    if (!h || !map_new || !map_old || !out3 || L_new <= 0 || L_old <= 0 || L_new > h->Lcap || L_old > h->Lcap)
        return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    const int L = h->Lcap;
    cudaStream_t s = h->stream;
    CK(cudaMemcpy2DAsync(h->d_tmp_a, (size_t)L * 8, map_new, (size_t)ld_new * 8, (size_t)L_new * 8, 2, cudaMemcpyDefault, s));
    CK(cudaMemcpy2DAsync(h->d_tmp_b, (size_t)L * 8, map_old, (size_t)ld_old * 8, (size_t)L_old * 8, 2, cudaMemcpyDefault, s));
    k_set_lsearch<<<1, 1, 0, s>>>(h->d_st, L_old);
    CK(cudaGetLastError());
    LandmarkGrid& G = h->scratch_grid;
    int rc = build_fgrid(h, G, h->d_tmp_b, h->d_tmp_b + L, &h->d_st->lsearch, L_old);
    if (rc) return rc;
    double init[3] = {INFINITY, 0.0, 0.0};
    CK(cudaMemcpyAsync(h->d_acc, init, sizeof init, cudaMemcpyHostToDevice, s));
    k_cambio<<<nblk(L_new, 128), 128, 0, s>>>(h->d_tmp_a, h->d_tmp_a + L, L_new, h->d_tmp_b, h->d_tmp_b + L, L_old, G.geom, G.start, G.pts,
                                              h->dcfg.dist_thr, h->d_acc);
    CK(cudaGetLastError());
    double res[3];
    CK(cudaMemcpyAsync(res, h->d_acc, sizeof res, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    out3[0] = res[0]; out3[1] = res[1]; out3[2] = res[2] / (double)L_new;
    return ICMSLAM_OK;
}

// ---- Mapa.actualizar for one scan (ICM_SLAM.py:128-201) -------------------------------------------------------------------
// nearest landmark of one observation per block: cdist + argmin + gate, exactly (rooted distances, first index on ties)
__global__ void __launch_bounds__(128)
k_actualizar_nearest(const double* __restrict__ rx, const double* __restrict__ ry, int Ls, const double* __restrict__ ox,
                     const double* __restrict__ oy, double dist_thr, int* __restrict__ c)
{
    __shared__ double bd[4];
    __shared__ int bi[4];
    const int i = blockIdx.x;
    const double wx = ox[i], wy = oy[i];
    double best = INFINITY;
    int arg = 0x7fffffff;
    for (int l = threadIdx.x; l < Ls; l += blockDim.x) {
        const double d = dist_rn(rx[l] - wx, ry[l] - wy);
        if (d < best) { best = d; arg = l; }          // (ascending l within a thread: the first minimum stays)
    }
    for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(FULLMASK, best, o);
        const int oa = __shfl_xor_sync(FULLMASK, arg, o);
        if (ob < best || (ob == best && oa < arg)) { best = ob; arg = oa; }
    }
    if ((threadIdx.x & 31) == 0) { bd[threadIdx.x >> 5] = best; bi[threadIdx.x >> 5] = arg; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 4; ++w) if (bd[w] < best || (bd[w] == best && bi[w] < arg)) { best = bd[w]; arg = bi[w]; }
        c[i] = (Ls <= 0 || best > dist_thr) ? -1 : arg;          // amin > dist_thr -> far (ICM_SLAM.py:172)
    }
}

// labels of the far observations, then the running means and counts of every label present, in the reference's order
__global__ void __launch_bounds__(256)
k_actualizar_update(DevState* st, int Lcap, int n, const double* __restrict__ ox, const double* __restrict__ oy, int* __restrict__ c,
                    double* __restrict__ mapa, int cap, int64_t ld, double* __restrict__ cant)
{
    __shared__ int anyfar;
    if (threadIdx.x == 0) anyfar = 0;
    __syncthreads();
    const int lact = st->lact;
    for (int i = threadIdx.x; i < n; i += blockDim.x) if (c[i] < 0) anyfar = 1;
    __syncthreads();
    const int newl = lact + (anyfar ? 1 : 0);        // every far observation of the scan gets the ONE new label (:174-180)
    if (newl > Lcap || newl > cap) { if (threadIdx.x == 0) st->status |= ST_LABEL_CAP; return; }
    for (int i = threadIdx.x; i < n; i += blockDim.x) if (c[i] < 0) c[i] = lact;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int l = c[i];
        bool first = true;
        for (int j = 0; j < i; ++j) if (c[j] == l) { first = false; break; }
        if (!first) continue;
        double sx = 0.0, sy = 0.0;
        int k = 0;
        for (int j = i; j < n; ++j) if (c[j] == l) { sx = add_rn(sx, ox[j]); sy = add_rn(sy, oy[j]); ++k; }     // np.sum(obs[c==i], axis=0)
        const double cn = cant[l], tot = add_rn(cn, (double)k);
        mapa[l] = add_rn(sx / tot, mul_rn(mapa[l], cn) / tot);                                                   // :191-192
        mapa[ld + l] = add_rn(sy / tot, mul_rn(mapa[ld + l], cn) / tot);
        cant[l] = tot;
    }
    if (threadIdx.x == 0) st->lact = newl;
}

extern "C" int icmslam_associate(icmslam_handle* h, const double* map_ref, int32_t L_ref, int64_t ld_ref, const double* obs_x,
                                 const double* obs_y, int32_t n_obs, double* mapa, int32_t cap, int64_t ld_mapa, int32_t* c,
                                 int32_t memspace)
{
    if (!h || n_obs < 0 || !mapa || cap <= 0 || cap > h->Lcap || ld_mapa < cap || L_ref < 0 || L_ref > h->Lcap || (L_ref > 0 && (!map_ref || ld_ref < L_ref)))
        return ICMSLAM_ERR_INVALID;
    if (n_obs == 0) return ICMSLAM_OK;
    if (!obs_x || !obs_y || !c) return ICMSLAM_ERR_INVALID;
    CK(cudaSetDevice(h->cfg.device));
    const int L = h->Lcap;
    cudaStream_t s = h->stream;
    int rc = sync_state(h);
    if (rc) return rc;
    const int lact = h->h_st->lact;
    h->ch.grid_map = nullptr; h->ch.hint_map = nullptr; h->last_map_L = -1;      // (the Mapa state changes under any map chain in flight)
    if (lact == 0) {
        // Branch A (ICM_SLAM.py:160-165): clusters of the first scan, on the host like icmslam_pass0's first step
        std::vector<double> wx(n_obs), wy(n_obs);
        CK(cudaMemcpyAsync(wx.data(), obs_x, (size_t)n_obs * 8, cudaMemcpyDefault, s));
        CK(cudaMemcpyAsync(wy.data(), obs_y, (size_t)n_obs * 8, cudaMemcpyDefault, s));
        CK(cudaStreamSynchronize(s));
        std::vector<int> lab(n_obs);
        const int k0 = icm_fcluster::fcluster_inconsistent(wx.data(), wy.data(), n_obs, h->cfg.dist_thr, lab.data());
        if (k0 > L || k0 > cap) return ICMSLAM_ERR_LABEL_CAP;
        std::vector<double> mx(k0), my(k0), cn(k0);
        for (int i = 0; i < k0; ++i) {                                // np.mean(obs[c==i,:], axis=0)
            double sx = 0.0, sy = 0.0;
            int k = 0;
            for (int j = 0; j < n_obs; ++j) if (lab[j] == i) { sx += wx[j]; sy += wy[j]; ++k; }
            mx[i] = sx / (double)k; my[i] = sy / (double)k; cn[i] = (double)k;
        }
        CK(cudaMemcpyAsync(mapa, mx.data(), (size_t)k0 * 8, cudaMemcpyDefault, s));
        CK(cudaMemcpyAsync(mapa + ld_mapa, my.data(), (size_t)k0 * 8, cudaMemcpyDefault, s));
        CK(cudaMemcpyAsync(h->d_counts, cn.data(), (size_t)k0 * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(c, lab.data(), (size_t)n_obs * sizeof(int), cudaMemcpyDefault, s));
        k_set_lact<<<1, 1, 0, s>>>(h->d_st, k0);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(s));
        h->lact_host = k0; h->ch.lact_dirty = false;
        (void)memspace;
        return ICMSLAM_OK;
    }
    // Branch B: device copies of the reference map (d_tmp_a), the observations (d_kx / d_ky as scratch would clash with the
    // filter: d_ox / d_oy) and the map under construction (d_tmp_b)
    const int Ls = lact < L_ref ? lact : L_ref;
    if (n_obs > ASSOC_MAX_OBS) return ICMSLAM_ERR_UNSUPPORTED;
    if (Ls > 0) CK(cudaMemcpy2DAsync(h->d_tmp_a, (size_t)L * 8, map_ref, (size_t)ld_ref * 8, (size_t)Ls * 8, 2, cudaMemcpyDefault, s));
    double *aox = h->d_aobs, *aoy = h->d_aobs + ASSOC_MAX_OBS;
    CK(cudaMemcpyAsync(aox, obs_x, (size_t)n_obs * 8, cudaMemcpyDefault, s));
    CK(cudaMemcpyAsync(aoy, obs_y, (size_t)n_obs * 8, cudaMemcpyDefault, s));
    CK(cudaMemcpy2DAsync(h->d_tmp_b, (size_t)L * 8, mapa, (size_t)ld_mapa * 8, (size_t)cap * 8, 2, cudaMemcpyDefault, s));
    k_set_raw_l<<<1, 1, 0, s>>>(h->d_st, lact);                      // (clears the status word)
    CK(cudaGetLastError());
    k_actualizar_nearest<<<n_obs, 128, 0, s>>>(h->d_tmp_a, h->d_tmp_a + L, Ls, aox, aoy, h->dcfg.dist_thr, h->d_ac);
    CK(cudaGetLastError());
    k_actualizar_update<<<1, 256, 0, s>>>(h->d_st, L, n_obs, aox, aoy, h->d_ac, h->d_tmp_b, cap, L, h->d_counts);
    CK(cudaGetLastError());
    h->n_launch += 3;
    rc = sync_state(h);
    if (rc) return rc;
    if (h->h_st->status & ST_LABEL_CAP) return ICMSLAM_ERR_LABEL_CAP;
    CK(cudaMemcpy2DAsync(mapa, (size_t)ld_mapa * 8, h->d_tmp_b, (size_t)L * 8, (size_t)cap * 8, 2, cudaMemcpyDefault, s));
    CK(cudaMemcpyAsync(c, h->d_ac, (size_t)n_obs * sizeof(int), cudaMemcpyDefault, s));
    CK(cudaStreamSynchronize(s));
    return ICMSLAM_OK;
}

// ---- the driver loop with the convergence monitor (sensors.py:302-315) -------------------------------------------------
extern "C" int icmslam_iterate_until(icmslam_handle* h, const double* x0, int32_t max_sweeps, double tol_max_change,
                                     const icmslam_sweep_opts* opts, double* cambios, int32_t* n_done)
{
    if (!h || !x0 || max_sweeps < 0 || !n_done) return ICMSLAM_ERR_INVALID;
    *n_done = 0;
    const int L = h->Lcap;
    for (int k = 0; k < max_sweeps; ++k) {
        int rc = sync_state(h);
        if (rc) return rc;
        const int L_old = h->h_st->lact;
        rc = icmslam_iterate(h, nullptr, 0, x0, 1, opts, ICMSLAM_DEVICE);
        if (rc) return rc;
        rc = sync_state(h);
        if (rc) return rc;
        rc = status_from_state(h->h_st);
        if (rc) return rc;
        const DevState* st = h->h_st;
        double tri[3];
        if (h->ch.timed_fused && st->cambio_unres == 0 && st->new_l > 0) {
            tri[0] = st->cambio[0]; tri[1] = st->cambio[1]; tri[2] = st->cambio[2] / (double)st->new_l;
        } else {        // landmarks merged / appeared, or another sweep mode: the full search (new map = d_map_in, old = d_map_out)
            rc = icmslam_calc_cambio(h, h->d_map_in, st->new_l, L, h->d_map_out, L_old > 0 ? L_old : 1, L, tri, ICMSLAM_DEVICE);
            if (rc) return rc;
        }
        if (cambios) { cambios[k] = tri[0]; cambios[max_sweeps + k] = tri[1]; cambios[2 * max_sweeps + k] = tri[2]; }
        *n_done = k + 1;
        if (tol_max_change > 0.0 && tri[1] <= tol_max_change) break;
    }
    return ICMSLAM_OK;
}

// ---- the same driver loop for a batch handle, one monitor per trajectory -------------------------------------------------
// Each trajectory stops at its own first sweep whose largest landmark change is <= tol: from the next sweep on it is frozen on the
// device (Freeze: its scans commit nothing, its poses and landmarks pass through unchanged) while the others sweep on.
__global__ void k_fz_reset(const Freeze fz) { fz.reset_slots(blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x); }

static int batch_until_loop(icmslam_handle* h, int max_sweeps, double tol, const icmslam_sweep_opts& o, double* cambios, int32_t* n_done,
                            int32_t* n_run)
{
    const int K = h->traj_K, L = h->Lcap;
    cudaStream_t s = h->stream;
    double x0[3];
    for (int r = 0; r < 3; ++r) CK(cudaMemcpyAsync(x0 + r, h->d_x0s + (size_t)r * K, sizeof(double), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    std::vector<unsigned char> frozen((size_t)K, 0);
    std::vector<double> sl((size_t)FZ_SLOTS * K);
    int active = K;
    for (int it = 0; it < max_sweeps && active > 0; ++it) {
        int rc = sync_state(h);
        if (rc) return rc;
        const int L_old = h->h_st->lact;
        k_fz_reset<<<nblk(K, 256), 256, 0, s>>>(h->fz);
        CK(cudaGetLastError());
        rc = icmslam_iterate(h, nullptr, 0, x0, 1, &o, ICMSLAM_DEVICE);
        if (rc) return rc;
        rc = sync_state(h);
        if (rc) return rc;
        rc = status_from_state(h->h_st);
        if (rc) return rc;
        const int L_new = h->h_st->new_l;
        CK(cudaMemcpyAsync(sl.data(), h->d_fz_slots, sl.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        bool need = false;
        for (int k = 0; k < K; ++k) need = need || (!frozen[k] && sl[(size_t)4 * K + k] > 0.0);
        if (need && L_new > 0 && L_old > 0) {      // the full search for the trajectories the tail could not settle (new map = d_map_in)
            k_fz_regions<<<nblk(L_old, 256), 256, 0, s>>>(h->fz, h->d_map_out, h->d_map_out + L, L_old, h->d_fz_reg);
            CK(cudaGetLastError());
            k_fz_need<<<nblk(K, 256), 256, 0, s>>>(h->fz, h->d_fz_need);
            CK(cudaGetLastError());
            k_cambio_regions<<<nblk(L_new, 128), 128, 0, s>>>(h->fz, h->d_fz_need, h->d_map_in, h->d_map_in + L, L_new, h->d_map_out,
                                                              h->d_map_out + L, h->d_fz_reg, L_old);
            CK(cudaGetLastError());
            h->n_launch += 3;
            h->fz_fallbacks += 1;
            CK(cudaMemcpyAsync(sl.data(), h->d_fz_slots, sl.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
        }
        for (int k = 0; k < K; ++k) {
            if (frozen[k]) continue;
            const double tri[3] = {sl[k], sl[(size_t)K + k], sl[(size_t)2 * K + k] / sl[(size_t)3 * K + k]};
            if (cambios)
                for (int r = 0; r < 3; ++r) cambios[((size_t)r * K + k) * max_sweeps + it] = tri[r];
            n_done[k] = it + 1;
            if (tol > 0.0 && tri[1] <= tol) { frozen[k] = 1; --active; }
        }
        *n_run = it + 1;
        if (active > 0 && it + 1 < max_sweeps) CK(cudaMemcpyAsync(h->d_fz_mask, frozen.data(), (size_t)K, cudaMemcpyHostToDevice, s));
    }
    CK(cudaStreamSynchronize(s));      // (the staging vector of the last mask upload goes away)
    return ICMSLAM_OK;
}

extern "C" int icmslam_batch_iterate_until(icmslam_handle* h, int32_t max_sweeps, double tol_max_change, double region_pitch,
                                           int32_t region_cols, const icmslam_sweep_opts* opts, double* cambios, int32_t* n_done,
                                           int32_t* n_run)
{
    if (!h || !n_done || !n_run || max_sweeps < 0 || !(region_pitch > 0.0) || region_cols <= 0 || h->traj_K <= 0)
        return ICMSLAM_ERR_INVALID;
    icmslam_sweep_opts o;
    default_opts(o, opts);
    if (!fused_mode(h, o) || h->p2p.on || !h->seg_first || !h->seg_last)
        return ICMSLAM_ERR_UNSUPPORTED;
    CK(cudaSetDevice(h->cfg.device));
    const int K = h->traj_K, L = h->Lcap;
    cudaStream_t s = h->stream;
    *n_run = 0;
    for (int k = 0; k < K; ++k) n_done[k] = 0;
    {   // every landmark of the starting map belongs to one of the K regions
        int rc = sync_state(h);
        if (rc) return rc;
        const int L0 = h->h_st->lact;
        std::vector<double> m((size_t)2 * L0);
        if (L0 > 0) CK(cudaMemcpy2DAsync(m.data(), (size_t)L0 * 8, h->d_map_in, (size_t)L * 8, (size_t)L0 * 8, 2, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        for (int l = 0; l < L0; ++l) {
            const double k = rint(m[(size_t)L0 + l] / region_pitch) * (double)region_cols + rint(m[l] / region_pitch);
            if (!(k >= 0.0 && k < (double)K)) {
                snprintf(h->err, sizeof h->err, "landmark %d at (%g, %g) lies outside the %d trajectory regions", l, m[l], m[(size_t)L0 + l], K);
                return ICMSLAM_ERR_INVALID;
            }
        }
    }
    if (h->fz_K != K) {
        drop_graphs(h);      // (graphs of an earlier call hold the old buffers)
        h->fz_K = 0;
        CK(h->d_fz_mask.alloc((size_t)K)); CK(h->d_fz_need.alloc((size_t)K));
        CK(h->d_fz_slots.alloc((size_t)FZ_SLOTS * K)); CK(h->d_fz_reg.alloc((size_t)L));
        h->fz_K = K;
    }
    CK(cudaMemsetAsync(h->d_fz_mask, 0, (size_t)K, s));
    h->fz.frozen = h->d_fz_mask; h->fz.traj = h->d_traj_of; h->fz.K = K; h->fz.cols = region_cols; h->fz.pitch = region_pitch;
    h->fz.slots = h->d_fz_slots;
    h->fz_fallbacks = 0;
    const int rc = batch_until_loop(h, max_sweeps, tol_max_change, o, cambios, n_done, n_run);
    h->fz = Freeze{};      // every trajectory unfrozen: later sweeps run the plain batch path
    return rc;
}

extern "C" int icmslam_filtrar_obs(icmslam_handle* h, const double* obs, int32_t B, int32_t T, int64_t ld, double max_dist,
                                   int32_t cant_max, double* out, int64_t ld_out, int32_t memspace)
{
    if (!h || !obs || !out || B <= 0 || B > 1024 || T <= 0 || ld < T || ld_out < T) return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    cudaStream_t s = h->stream;
    DevBuf<double> d_in, d_out;
    DevBuf<int> d_a, d_keep, d_err;
    CK(d_in.alloc((size_t)B * T)); CK(d_out.alloc((size_t)B * T));
    CK(d_a.alloc((size_t)T)); CK(d_keep.alloc((size_t)T)); CK(d_err.alloc(1));
    CK(cudaMemcpy2DAsync(d_in, (size_t)T * 8, obs, (size_t)ld * 8, (size_t)T * 8, B, cudaMemcpyDefault, s));
    CK(cudaMemsetAsync(d_err, 0, sizeof(int), s));
    k_fo_count<<<nblk(T, 128), 128, 0, s>>>(d_in, B, T, T, max_dist, d_a);
    CK(cudaGetLastError());
    k_fo_interp<<<nblk(T, 128), 128, 0, s>>>(d_a, T, cant_max, d_keep, d_err);
    CK(cudaGetLastError());
    const size_t smem = (size_t)2 * B * (EX_TILE + 1) * sizeof(double);
    CK(cudaFuncSetAttribute(k_fo_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_fo_select<<<nblk(T, EX_TILE), 256, smem, s>>>(d_in, B, T, T, max_dist, d_keep, d_out, T);
    CK(cudaGetLastError());
    int err = 0;
    CK(cudaMemcpyAsync(&err, d_err, sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpy2DAsync(out, (size_t)ld_out * 8, d_out, (size_t)T * 8, (size_t)T * 8, B, cudaMemcpyDefault, s));
    CK(cudaStreamSynchronize(s));
    return err ? ICMSLAM_ERR_INVALID : ICMSLAM_OK;
}

// ---- pass 0: inicializar_online on the loaded log (sensors.py:51-123), as a walk that can stop and resume ---------------------
// begin: x0 and an empty walk.  advance: the steps of every loaded column the walk has not taken (Branch A / fcluster on the host
// at column 0, then k_pass0); the poses go to the resident pose buffer, the labels and running means to the per-observation
// arrays, the map under construction and its counts to the walk's own buffers, published as the handle's raw map.  finish:
// Mapa.filtrar of the map built so far (sensors.py:99-102).
// the walk's map under construction becomes the handle's raw map (d_raw, d_rawcnt, raw_l), as icmslam_pass0 leaves it
static int publish_walk(icmslam_handle* h)
{
    const int L = h->Lcap;
    CK(cudaMemcpyAsync(h->d_raw, h->walk.y, (size_t)2 * L * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    k_walk_publish<<<nblk(L, 256), 256, 0, h->stream>>>(h->walk.carry, h->walk.cant, L, h->d_rawcnt, h->d_st);
    CK(cudaGetLastError());
    h->n_launch += 1;
    h->ch.rawcnt_valid = true;
    h->ch.lact_dirty = true;
    return ICMSLAM_OK;
}

extern "C" int icmslam_pass0_begin(icmslam_handle* h, const double* x0)
{
    if (!h || !h->extracted || !x0) return ICMSLAM_ERR_INVALID;
    h->walk.on = false;
    if (h->first_empty) return ICMSLAM_EMPTY_FIRST_SCAN;        // (the reference would fail inside tras_rot_z / linkage)
    CK(cudaSetDevice(h->cfg.device));
    int rc = ensure_seen(h);
    if (rc) return rc;
    h->walk.on = true;
    h->walk.t = 0; h->walk.lact = 0;
    h->walk.x0[0] = x0[0]; h->walk.x0[1] = x0[1]; h->walk.x0[2] = x0[2];
    return ICMSLAM_OK;
}

extern "C" int icmslam_pass0_advance(icmslam_handle* h, int32_t* t_done)
{
    if (!h || !h->walk.on || !t_done) return ICMSLAM_ERR_INVALID;
    const int T = h->T, L = h->Lcap;
    int t_lo = h->walk.t;
    *t_done = t_lo;
    for (int t = t_lo; t < T; ++t)
        if (h->off_h[t + 1] - h->off_h[t] > 1024) return ICMSLAM_ERR_UNSUPPORTED;      // (k_pass0 stages one scan in shared memory)
    CK(cudaSetDevice(h->cfg.device));
    cudaStream_t s = h->stream;
    int rc = ensure_seen(h);
    if (rc) return rc;
    // the walk rewrites labels (the map chain's hints), the resident poses and the raw map
    h->ch.grid_map = nullptr; h->ch.hint_map = nullptr;
    rc = poses_home(h);
    if (rc) return rc;
    const double* x0 = h->walk.x0;
    int k0 = 0;
    if (t_lo == 0) {    // ---- step 0: Branch A of Mapa.actualizar on the first scan (ICM_SLAM.py:160-165), on the host ------------
        const int n0 = h->off_h[1] - h->off_h[0];
        DevBuf<double> d_w;
        CK(d_w.alloc((size_t)2 * n0));
        k_project_scan<<<nblk(n0, 128), 128, 0, s>>>(h->ex.d_off, 0, h->ex.d_bx, h->ex.d_by, x0[0], x0[1], x0[2], d_w, d_w + n0);
        CK(cudaGetLastError());
        std::vector<double> w((size_t)2 * n0);
        CK(cudaMemcpyAsync(w.data(), d_w, (size_t)2 * n0 * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        std::vector<int> lab0(n0);
        k0 = icm_fcluster::fcluster_inconsistent(w.data(), w.data() + n0, n0, h->cfg.dist_thr, lab0.data());
        if (k0 > L) { h->walk.on = false; return ICMSLAM_ERR_LABEL_CAP; }
        std::vector<double> y0((size_t)2 * L, 0.0), cant0((size_t)L, 0.0);
        for (int i = 0; i < k0; ++i) {                                // np.mean(obs[c==i,:], axis=0): row-order sum / count
            double sx = 0.0, sy = 0.0;
            int k = 0;
            for (int j = 0; j < n0; ++j) if (lab0[j] == i) { sx += w[j]; sy += w[n0 + j]; ++k; }
            y0[i] = sx / (double)k; y0[L + i] = sy / (double)k; cant0[i] = (double)k;
        }
        CK(cudaMemcpyAsync(h->walk.y, y0.data(), (size_t)2 * L * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(h->walk.cant, cant0.data(), (size_t)L * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(h->ex.d_c, lab0.data(), (size_t)n0 * sizeof(int), cudaMemcpyHostToDevice, s));
        CK(cudaMemsetAsync(&h->d_st->newton_iters, 0, sizeof(unsigned long long), s));
        t_lo = 1;
    }
    // ---- steps t_lo .. T-1 on the device ----------------------------------------------------------------------------------
    if (h->walk.t == 0 || t_lo < T) {      // (after step 0 even at T = 1: the launch starts the carry)
        Pass0Params P;
        P.t_lo = t_lo; P.t_hi = T; P.Lcap = L;
        P.off = h->ex.d_off; P.bx = h->ex.d_bx; P.by = h->ex.d_by; P.d = h->ex.d_d; P.beam = h->ex.d_beam; P.ang = h->ds.d_ang;
        P.odo = h->ds.d_odo; P.ldo = h->cap_T; P.u = h->ds.d_u; P.ldu = h->cap_T; P.cfg = h->dcfg;
        P.first = h->walk.t == 0 ? 1 : 0;
        P.x0[0] = x0[0]; P.x0[1] = x0[1]; P.x0[2] = x0[2]; P.lact0 = k0; P.carry = h->walk.carry;
        P.x = h->ds.d_x; P.ldx = h->cap_T; P.y = h->walk.y; P.cant = h->walk.cant;
        P.c = h->ex.d_c; P.seen_x = h->ex.d_seen_x; P.seen_y = h->ex.d_seen_y;
        P.st = h->d_st; P.nev = &h->d_st->newton_iters;
        const size_t smem = (size_t)2 * 1024 * 8 + 1024 * 4;
        k_pass0<<<1, 256, smem, s>>>(P);
        CK(cudaGetLastError());
        h->n_launch += 1;
        Pass0Carry c;
        CK(cudaMemcpyAsync(&c, h->walk.carry, sizeof c, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        h->walk.lact = c.lact;
        *t_done = c.t;
        if (c.t < T) {      // the label cap: the walk stops at the column that needed a label beyond L (begin it again)
            h->walk.on = false;
            h->ch.lact_dirty = true;
            return ICMSLAM_ERR_LABEL_CAP;
        }
    }
    h->walk.t = T;
    *t_done = T;
    return publish_walk(h);
}

extern "C" int icmslam_pass0_finish(icmslam_handle* h, double* x, int64_t ld_x, double* map_out, int32_t cap_out, int64_t ld_map_out,
                                    int32_t* L_out, int32_t memspace)
{
    if (!h || !h->walk.on || !x || ld_x < h->walk.t || !L_out) return ICMSLAM_ERR_INVALID;
    if (map_out && (cap_out <= 0 || ld_map_out < cap_out)) return ICMSLAM_ERR_INVALID;
    (void)memspace;
    CK(cudaSetDevice(h->cfg.device));
    const int L = h->Lcap, tw = h->walk.t, lact = h->walk.lact;
    cudaStream_t s = h->stream;
    int rc = ensure_layout(h);
    if (rc) return rc;
    rc = publish_walk(h);
    if (rc) return rc;
    // ---- Mapa.filtrar on the map that was built (sensors.py:99-100) ---------------------------------------------------------
    h->ch.grid_map = nullptr; h->ch.hint_map = nullptr;
    h->ch.stats_clean = false;
    k_counts_to_int<<<nblk(L, 256), 256, 0, s>>>(h->walk.cant, L, h->d_cnt);      // (get_raw_map reports integer counts)
    CK(cudaGetLastError());
    k_flags_from_counts<<<nblk(L, 256), 256, 0, s>>>(h->walk.cant, lact, h->dcfg.cota, h->d_kflag, L, h->d_blk_kept, h->grid.bb, h->d_ts);
    CK(cudaGetLastError());
    rc = filter_chain(h, h->d_raw, h->d_raw + L, nullptr, h->d_map_out, L, L, s, false);
    if (rc) return rc;
    rc = sync_state(h);
    if (rc) return rc;
    int status = status_from_state(h->h_st);
    if (status) return status;
    const int newL = h->h_st->new_l;
    *L_out = newL;
    if (tw > 0) CK(cudaMemcpy2DAsync(x, (size_t)ld_x * 8, h->ds.d_x, (size_t)h->cap_T * 8, (size_t)tw * 8, 3, cudaMemcpyDefault, s));
    const int wd = newL < cap_out ? newL : cap_out;
    if (map_out && wd > 0)
        CK(cudaMemcpy2DAsync(map_out, (size_t)ld_map_out * 8, h->d_map_out, (size_t)L * 8, (size_t)wd * 8, 2, cudaMemcpyDefault, s));
    CK(cudaStreamSynchronize(s));
    return ICMSLAM_OK;
}

// x (3 x T) receives the causal pose estimates (x[:,0] = x0), map_out the filtered map (`mapa_viejo`, sensors.py:99-102), *L_out
// its width; landmarks_actuales / cant_obs_i are left as the reference leaves them.  One walk over the whole log.
extern "C" int icmslam_pass0(icmslam_handle* h, const double* x0, double* x, int64_t ld_x, double* map_out, int32_t cap_out,
                             int64_t ld_map_out, int32_t* L_out, int32_t memspace)
{
    if (!h || !h->extracted || !x0 || !x || ld_x < h->T || !L_out) return ICMSLAM_ERR_INVALID;
    if (map_out && (cap_out <= 0 || ld_map_out < cap_out)) return ICMSLAM_ERR_INVALID;
    if (h->max_per_scan > 1024) return ICMSLAM_ERR_UNSUPPORTED;
    int rc = icmslam_pass0_begin(h, x0);
    if (rc) return rc;
    int32_t t_done = 0;
    rc = icmslam_pass0_advance(h, &t_done);
    if (rc) return rc;
    return icmslam_pass0_finish(h, x, ld_x, map_out, cap_out, ld_map_out, L_out, memspace);
}

// ---- pass 0 helpers ---------------------------------------------------------------------------------------------
// fcluster(linkage(pdist(obs)), t) - 1 as Mapa.actualizar calls it at t = 0 of pass 0 (ICM_SLAM.py:161): host code,
// no device needed.  obs = (px[i], py[i]), labels out; returns the number of clusters in *n_clusters.
extern "C" int icmslam_fcluster(const double* px, const double* py, int32_t n, double t, int32_t* labels, int32_t* n_clusters)
{
    if (n < 0 || (n > 0 && (!px || !py || !labels))) return ICMSLAM_ERR_INVALID;
    const int k = icm_fcluster::fcluster_inconsistent(px, py, n, t, labels);
    if (n_clusters) *n_clusters = k;
    return ICMSLAM_OK;
}
