/*
 * icmslam.h -- C ABI of libicmslam.so, the B200 (sm_100a) implementation of the ICM-SLAM
 * offline sweep path of Seba-san/icm-slam.
 *
 * The reference has no FFI: its hot path sits behind a Python class surface
 * (scripts/sensors.py:15-282 `ICM_ROS`, scripts/ICM_SLAM.py:104-265 `Mapa`,
 * scripts/ICM_SLAM.py:22-58 `filtrar_z`).  Each entry point below names the reference
 * interface it replaces; the ctypes binding a maintainer adds to the reference is shown in
 * INTEGRATION.md and implemented in icm_slam_b200/_lib.py.
 *
 * Conventions
 *  - plain C types only; all arrays are IEEE fp64 / int32 in numpy C order: a "3 x T" array is
 *    three rows, row r starts at base + r*ld (ld in ELEMENTS, ld >= T).
 *  - `memspace` says where caller buffers live: ICMSLAM_HOST (the library copies) or
 *    ICMSLAM_DEVICE (CUDA device pointers on the handle's device, used in place / copied D2D).
 *  - every call returns an int status (0 = ok, <0 = error below); nothing throws or exits.
 *    The reference's failure modes are mapped to status codes (see each code).
 *  - one handle per GPU, not thread-safe (the reference solver is not re-entrant either,
 *    sensors.py:214-220).  Work is enqueued on the handle's CUDA stream (its own, unless
 *    icmslam_set_stream is called); calls that return data to HOST buffers synchronise that
 *    stream before returning.  Callers passing DEVICE buffers produced on another stream order the
 *    two streams themselves (or share one through icmslam_set_stream).
 *  - there is NO CPU fallback: without a CUDA device icmslam_create fails with
 *    ICMSLAM_ERR_CUDA.
 */
#ifndef ICMSLAM_H_
#define ICMSLAM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ICMSLAM_ABI_VERSION 1

enum { ICMSLAM_HOST = 0, ICMSLAM_DEVICE = 1 };

/* status codes */
enum {
    ICMSLAM_OK = 0,
    ICMSLAM_EMPTY_FIRST_SCAN = 1,   /* not an error: scan 0 has no observation, the reference returns
                                       its inputs unchanged (sensors.py:137-139); outputs = inputs */
    ICMSLAM_ERR_INVALID = -1,       /* bad argument / call order */
    ICMSLAM_ERR_LABEL_CAP = -2,     /* a new label would exceed config.L: the reference raises
                                       IndexError at ICM_SLAM.py:191 */
    ICMSLAM_ERR_EMPTY_LAST = -3,    /* last scan has no observation: IndexError at sensors.py:148 */
    ICMSLAM_ERR_EMPTY_MAP = -4,     /* no landmark reaches `cota`: ValueError at ICM_SLAM.py:241-255 */
    ICMSLAM_ERR_ALLOC = -5,         /* device or host allocation failed */
    ICMSLAM_ERR_CUDA = -6,          /* CUDA runtime error; text via icmslam_last_error */
    ICMSLAM_ERR_UNSUPPORTED = -7
};

/* sweep mode switches.  (SEQUENTIAL, NM, RUNNING) is the reference's own semantics
 * (sensors.py:145-162, :221, ICM_SLAM.py:191-194); the others are the restated, parallel
 * variants described in DESIGN.md. */
enum { ICMSLAM_SCHED_SEQUENTIAL = 0, ICMSLAM_SCHED_REDBLACK = 1 };
enum { ICMSLAM_SOLVER_NM = 0, ICMSLAM_SOLVER_NEWTON = 1 };
enum { ICMSLAM_VIEW_RUNNING = 0, ICMSLAM_VIEW_FULL = 1, ICMSLAM_VIEW_PREV = 2 };

/* The live keys of ConfigICM (ICM_SLAM.py:72-99, config_default.yaml / config_ros.yaml). */
typedef struct icmslam_config {
    double deltat;          /* D['deltat'] */
    double q1, q2;          /* D['Q']  (diagonal observation weights) */
    double r1, r2, r3;      /* D['R']  (diagonal motion weights) */
    double cte_odom;        /* D['cte_odom'] */
    double cota;            /* D['cota'] */
    double dist_thr;        /* D['dist_thr'] */
    double rango_laser_max; /* D['rango_laser_max'] */
    double radio;           /* D['radio'] */
    int32_t L;              /* D['L']: label capacity */
    int32_t device;         /* CUDA device ordinal */
} icmslam_config;

typedef struct icmslam_sweep_opts {
    int32_t schedule;       /* ICMSLAM_SCHED_* */
    int32_t solver;         /* ICMSLAM_SOLVER_* */
    int32_t map_view;       /* ICMSLAM_VIEW_* */
    int32_t newton_maxit;   /* <=0: default 20 */
    double newton_tol;      /* Newton stops when |dtheta| <= tol; <=0: default 1e-7 (the remaining error is quadratic in it) */
    int32_t fused;          /* 1: allow the single-kernel path when (REDBLACK, NEWTON, PREV) */
    int32_t reserved;
} icmslam_sweep_opts;

typedef struct icmslam_handle icmslam_handle;

/* -- lifecycle.  Replaces ICM_ROS.__init__ / Mapa.__init__ (sensors.py:16-49, ICM_SLAM.py:109-117). */
int icmslam_create(const icmslam_config* cfg, icmslam_handle** out);
int icmslam_destroy(icmslam_handle* h);
int icmslam_abi_version(void);
const char* icmslam_strerror(int status);
const char* icmslam_last_error(const icmslam_handle* h);
/* cudaStream_t to enqueue on.  A handle is created with its own non-blocking stream; NULL switches
 * back to it.  (Steady-state sweeps replay as a CUDA graph, which the legacy default stream cannot
 * capture.) */
int icmslam_set_stream(icmslam_handle* h, void* cuda_stream);
int icmslam_synchronize(icmslam_handle* h);

/* -- data.  Replaces the ICM_ROS attributes `mediciones` (B x T), `odometria` (3 x T), `u` (2 x T)
 * (sensors.py:26-28, filled by ROS.principal_callback ICM_SLAM.py:332-339) and the legacy
 * ICM_method.load_data (ICM_SLAM_old.py:249-264).  `scans` are ranges ALREADY pre-conditioned
 * unless precondition != 0, in which case z = min(z + radio, rango_laser_max), NaN -> max is
 * applied on the device (sensors_definitions.py:21-22, IJAC2018_python.txt:43).
 * cos_tab / sin_tab (length B, host pointers, may be NULL) are cos/sin of the beam angles
 * (i*pi)/180 exactly as the caller's numpy computes them (ICM_SLAM.py:44,51-53); NULL -> libm. */
int icmslam_load(icmslam_handle* h, const double* scans, int32_t B, int32_t T, int64_t ld_scans,
                 const double* odometry, int64_t ld_odo, const double* controls, int64_t ld_u,
                 const double* cos_tab, const double* sin_tab, int32_t precondition, int32_t memspace);

/* -- filtrar_z for every scan (ICM_SLAM.py:22-58), once per dataset (the reference recomputes it
 * every sweep, sensors.py:134,146, although it does not depend on the poses).  Builds the CSR of
 * kept beams on the device. */
int icmslam_extract(icmslam_handle* h);
int icmslam_extraction_size(const icmslam_handle* h, int64_t* n_obs, int32_t* n_empty_scans,
                            int32_t* max_per_scan);
/* any pointer may be NULL.  off: T+1, the others: n_obs. */
int icmslam_get_extraction(icmslam_handle* h, int32_t* off, int32_t* beam, double* d, double* bx,
                           double* by, int32_t memspace);

/* -- Mapa state (ICM_SLAM.py:115, :119-126): landmarks_actuales and cant_obs_i. */
int icmslam_set_landmarks_actuales(icmslam_handle* h, int32_t lact);
int icmslam_get_landmarks_actuales(const icmslam_handle* h, int32_t* lact);
int icmslam_get_counts(icmslam_handle* h, double* cant_obs_i, int32_t n, int32_t memspace);
/* cant_obs_i[:n] = counts, the rest zero (n = 0: Mapa.clear_obs, ICM_SLAM.py:119-126) */
int icmslam_set_counts(icmslam_handle* h, const double* cant_obs_i, int32_t n, int32_t memspace);

/* -- one ICM sweep = ICM_ROS.iterations_process_offline(mapa_viejo, x) (sensors.py:125-168).
 * map_in: 2 x L_in (ld_map_in).  x: 3 x T (ld_x), updated IN PLACE like the reference.
 * x0: the pinned first pose `self.x0` (sensors.py:131), 3 doubles, always a HOST pointer.
 * map_out: 2 x cap_out (ld_map_out) receives `mapa_refinado`; *L_out its width (host int).
 * Association uses the first min(landmarks_actuales, L_in) columns of map_in; new labels start
 * at landmarks_actuales (ICM_SLAM.py:169-182).  On return landmarks_actuales = *L_out. */
int icmslam_sweep(icmslam_handle* h, const double* map_in, int32_t L_in, int64_t ld_map_in, double* x,
                  int64_t ld_x, const double* x0, double* map_out, int32_t cap_out, int64_t ld_map_out,
                  int32_t* L_out, const icmslam_sweep_opts* opts, int32_t memspace);

/* -- the driver loop `for i in range(config.N): mapa_refinado, x = iterations_process_offline(
 * mapa_viejo, x); mapa_viejo = mapa_refinado` (sensors.py:302-315, example.py:49-53) with the map
 * kept on the device between sweeps.  icmslam_set_map uploads `mapa_viejo` (2 x L_map) and sets
 * landmarks_actuales = L_map (sensors.py:102-103); icmslam_iterate runs n_sweeps sweeps, updating
 * x (3 x T) in place; icmslam_get_map returns the current `mapa_viejo` and its width. */
int icmslam_set_map(icmslam_handle* h, const double* map, int32_t L_map, int64_t ld, int32_t memspace);
int icmslam_get_map(icmslam_handle* h, double* map, int32_t cap, int64_t ld, int32_t* L_map, int32_t memspace);
int icmslam_iterate(icmslam_handle* h, double* x, int64_t ld_x, const double* x0, int32_t n_sweeps,
                    const icmslam_sweep_opts* opts, int32_t memspace);
/* `ICM.positions` resident on the device (sensors.py:104): icmslam_set_poses uploads x (3 x T);
 * icmslam_iterate with x == NULL then sweeps the resident poses without any copy;
 * icmslam_get_poses reads the current poses back. */
int icmslam_set_poses(icmslam_handle* h, const double* x, int64_t ld_x, int32_t memspace);
int icmslam_get_poses(icmslam_handle* h, double* x, int64_t ld_x, int32_t memspace);

/* -- a batch of INDEPENDENT trajectories in one handle (BASELINE.json configs[4]: Monte-Carlo multi-start; no reference
 * counterpart beyond running the reference once per trajectory).  The caller loads K trajectories of traj_T columns each laid
 * end to end (T = K * traj_T), each translated to its own region of the plane so that their landmarks are farther apart than
 * any gate (icm_slam_b200/batch.py does both); x0s (HOST, 3 x K) are their pinned first poses.  Every trajectory's first pose is
 * then pinned to its own x0, its last pose has no successor, and one sweep of the handle is one sweep of every trajectory: ONE
 * launch of each kernel for the whole batch.  Every sweep mode is valid on a batch handle (icmslam_iterate and icmslam_sweep; the
 * SEQUENTIAL schedule walks each trajectory with its own warp); new labels are numbered over the whole batch and the label cap L
 * applies to the batch.  The x0 argument of icmslam_iterate / icmslam_sweep is ignored.  traj_T <= 0 switches back to a single
 * trajectory. */
int icmslam_set_batch(icmslam_handle* h, int32_t traj_T, const double* x0s, int64_t ld_x0s, int32_t K);

/* -- time-segment partition over several GPUs (no reference counterpart: the reference sweep is strictly
 * sequential in time, sensors.py:145-162; only the restated (REDBLACK, NEWTON, PREV) sweep partitions).
 * One handle per GPU loads the columns [g_lo - 2, g_hi + 1) of the trajectory (two halo columns on the
 * left unless it holds the first pose, one on the right unless it holds the last) and owns the local
 * columns [t_lo, t_hi) (t_lo even).  A sweep is then
 *     icmslam_seg_begin    -> all-gather of every segment's ICMSLAM_PTR_SEG_REC record (16 doubles)
 *     icmslam_seg_exchange -> sum-reduction of ICMSLAM_PTR_STAT_X, _STAT_Y (int64), _STAT_N (int32) and
 *                             ICMSLAM_PTR_NEW_LABELS (fp64, disjoint non-zeros) over the segments; the four
 *                             live in one block, ICMSLAM_PTR_EXCHANGE, that may be reduced as int64 words
 *                             in ONE all-reduce (counts never carry out of 32 bits; a new label's mean is
 *                             non-zero on exactly one segment, so adding bit patterns reproduces it)
 *     icmslam_seg_finish
 * with the collectives issued by the caller (NCCL through torch.distributed in icm_slam_b200/multigpu.py)
 * on the handle's stream.  The landmark statistics are integers, so every segment computes bit-identical
 * maps for any number of GPUs.
 * With opts.reserved & 4 in icmslam_seg_begin the boundary poses travel on their own: the solve runs on the handle's
 * low-priority side stream (ICMSLAM_PTR_SIDE_STREAM: a cudaStream_t, not device memory), the caller all-gathers
 * ICMSLAM_PTR_SEG_REC_POSE on THAT stream (a second communicator) and hands the result to icmslam_seg_halo, while the
 * ICMSLAM_PTR_SEG_REC gather (now only the label counts), icmslam_seg_exchange, the reduction and icmslam_seg_finish proceed
 * on the handle's stream; icmslam_seg_finish joins the two. */
enum { ICMSLAM_PTR_SEG_REC = 0, ICMSLAM_PTR_STAT_X = 1, ICMSLAM_PTR_STAT_Y = 2, ICMSLAM_PTR_STAT_N = 3,
       ICMSLAM_PTR_NEW_LABELS = 4, ICMSLAM_PTR_POSES = 5, ICMSLAM_PTR_EXCHANGE = 6, ICMSLAM_PTR_SEG_REC_POSE = 7,
       ICMSLAM_PTR_SIDE_STREAM = 8 };
int icmslam_set_segment(icmslam_handle* h, int32_t t_lo, int32_t t_hi, int32_t is_first, int32_t is_last);
int icmslam_device_ptr(icmslam_handle* h, int32_t which, void** ptr, int64_t* count);
int icmslam_seg_begin(icmslam_handle* h, const double* x0, const icmslam_sweep_opts* opts);
int icmslam_seg_halo(icmslam_handle* h, const double* gathered, int32_t rank, int32_t world);
int icmslam_seg_exchange(icmslam_handle* h, const double* gathered, int32_t rank, int32_t world);
int icmslam_seg_finish(icmslam_handle* h);
/* The same exchange by the library's own kernels over peer memory (csrc/p2p.cuh; the ranks of ONE node): every rank exports three
 * CUDA IPC handles (3 x 64 bytes), the caller gathers them in rank order and hands the table to every rank.  From then on
 * icmslam_iterate(h, NULL, 0, x0, n, ...) on the segment handles -- called by every rank with the same n -- runs whole sweeps with
 * no collective from outside: far counts, statistics (reduce-scatter by remote loads, the gather folded into the landmark
 * update) and halo poses travel through NVLink stores / loads, flagged with the sweep number.  Results are bit-identical to the
 * collective path and to one GPU. */
int icmslam_p2p_export(icmslam_handle* h, void* handles, int64_t cap_bytes);
int icmslam_p2p_import(icmslam_handle* h, int32_t rank, int32_t world, const void* all_handles, int64_t bytes);

/* -- pass 0 (causal initialisation, sensors.py:51-123).  icmslam_fcluster is the one scipy call of its first
 * step: c = fcluster(linkage(pdist(obs)), dist_thr) - 1 (ICM_SLAM.py:161; single linkage, inconsistency
 * criterion, depth 2).  Host code: needs no device. */
int icmslam_fcluster(const double* px, const double* py, int32_t n, double t, int32_t* labels, int32_t* n_clusters);
/* icmslam_pass0 = ICM_ROS.inicializar_online replayed on the loaded log (= ICM_method.inicializar,
 * ICM_SLAM_old.py:266-333): x (3 x T) <- causal poses with x[:,0] = x0 (`positions`, sensors.py:104), map_out
 * (2 x cap_out) <- `mapa_viejo` = Mapa.filtrar of the map built on the way (sensors.py:99-102), *L_out its width.
 * Sequential by construction; the inner solver is the reference's Nelder-Mead on fun_x. */
int icmslam_pass0(icmslam_handle* h, const double* x0, double* x, int64_t ld_x, double* map_out, int32_t cap_out,
                  int64_t ld_map_out, int32_t* L_out, int32_t memspace);

/* -- the model functions the reference leaves to the user (sensors.py:170-282) for ONE pose, on the device: `op` selects
 * g(x_ant, u_ant) (:206-211), h(x, z) against the matched landmarks `seen` (:175-204), the energy fun_xn / fun_x at x (:224-282;
 * fun_x when x_pos is NULL), or its minimiser as minimizar_xn / minimizar_x find it (Nelder-Mead from the reference's start
 * point, :213-222 / :257-264) or exactly (Newton).  z = (range, beam angle) pairs, odo = 3 x 3 (columns t-1, t, t+1; 3 x 2 without
 * x_pos), all HOST pointers.  x: evaluation point in (ENERGY, H), result out (G, MIN_*); *f the energy there; *n_eval the
 * evaluations (NM) or iterations (Newton).  `model` names the motion / measurement model: ICMSLAM_MODEL_UNICYCLE_LASER2D is the
 * reference's (and the only one the sweep kernels implement); anything else returns ICMSLAM_ERR_UNSUPPORTED. */
enum { ICMSLAM_MODEL_UNICYCLE_LASER2D = 0 };
enum { ICMSLAM_POSE_ENERGY = 0, ICMSLAM_POSE_MIN_NM = 1, ICMSLAM_POSE_MIN_NEWTON = 2, ICMSLAM_POSE_G = 3, ICMSLAM_POSE_H = 4 };
int icmslam_pose_eval(icmslam_handle* h, int32_t model, int32_t op, int32_t n, const double* z_d, const double* z_ang,
                      const double* seen_x, const double* seen_y, const double* x_ant, const double* x_pos, const double* u_ant,
                      const double* u_act, const double* odo, int64_t ld_odo, double* x, double* f, int32_t* n_eval,
                      const icmslam_sweep_opts* opts);

/* -- instrumentation (no reference counterpart).  Kernel time of the last sweep run with
 * opts.reserved & 2, from CUDA events on the handle's stream: out2[0] = association (or the fused
 * sweep kernel), out2[1] = pose kernels (0 when fused), milliseconds.  Launch count = kernels of
 * this library enqueued since icmslam_create. */
int icmslam_get_kernel_ms(icmslam_handle* h, double* out2);
/* With ICMSLAM_TRACE=1 in the environment when the handle is created, the sweep's kernels leave %globaltimer marks (ns) in a ring
 * of the last 32 sweeps x 8 marks: entry of k_runs, k_assoc_tiles, k_tail_labels, k_p2p_reduce, k_tail_steady, k_solve_tile,
 * k_p2p_halo, and the end of k_tail_steady.  counters3 = (sweeps closed, p2p sweep number, halo sweep number). */
int icmslam_get_trace(icmslam_handle* h, uint64_t* out256, uint32_t* counters3);
int icmslam_get_launch_count(icmslam_handle* h, int64_t* n);
/* bytes icmslam_sweep has copied host->device / device->host so far for HOST-memspace callers (poses, maps, status words);
 * a map the caller feeds back unchanged is not re-uploaded (sensors.py:315, `mapa_viejo = mapa_refinado`). */
int icmslam_get_transfer_bytes(icmslam_handle* h, int64_t* h2d, int64_t* d2h);

/* -- results of the last sweep (all optional; mirror what Mapa / actualizar expose).
 * c: association label of every kept observation, CSR order (`c` of ICM_SLAM.py:201).
 * raw map / counts / Lact: the map before Mapa.filtrar (`y`, cant_obs_i, landmarks_actuales at
 * sensors.py:165). */
int icmslam_get_associations(icmslam_handle* h, int32_t* c, int32_t memspace);
int icmslam_get_raw_map(icmslam_handle* h, double* raw_map, int32_t cap, int64_t ld, double* raw_counts,
                        int32_t* raw_L, int32_t memspace);
/* device-side statistics of the last sweep: number of Newton iterations summed over poses etc. */
int icmslam_get_sweep_stats(icmslam_handle* h, int64_t* stats, int32_t n);

/* -- Mapa.filtrar on caller data (ICM_SLAM.py:204-265): prune counts < cota, merge neighbours
 * closer than dist_thr, count-weighted means.  In: 2 x L_in map + counts; out: 2 x cap map, counts. */
int icmslam_filter_map(icmslam_handle* h, const double* map_in, int64_t ld_in, const double* counts_in,
                       int32_t L_in, double* map_out, int32_t cap_out, int64_t ld_out, double* counts_out,
                       int32_t* L_out, int32_t memspace);

/* -- calc_cambio (ICM_SLAM.py:490-495): min / max / mean over the new landmarks of the distance to
 * the nearest old landmark.  out3 is a HOST pointer. */
int icmslam_calc_cambio(icmslam_handle* h, const double* map_new, int32_t L_new, int64_t ld_new,
                        const double* map_old, int32_t L_old, int64_t ld_old, double* out3, int32_t memspace);

/* -- Mapa.actualizar(mapa, mapa_referencia, obs) for ONE scan (ICM_SLAM.py:128-201): the step pass 0 and the sweep take per
 * scan, exposed for callers that drive the scan loop themselves.  obs_x / obs_y: the scan's n_obs projected observations
 * (world frame).  map_ref: 2 x L_ref reference map (searched over its first min(landmarks_actuales, L_ref) columns).
 * mapa: 2 x cap map under construction, updated in place (running means, ICM_SLAM.py:191-194).  c: n_obs labels out
 * (int32; the reference returns int64).  State read and updated: landmarks_actuales, cant_obs_i.  Branch A
 * (landmarks_actuales == 0: scipy's fcluster, ICM_SLAM.py:160-165) runs through icmslam_fcluster.
 * ICMSLAM_ERR_LABEL_CAP where the reference raises IndexError (:191). */
int icmslam_associate(icmslam_handle* h, const double* map_ref, int32_t L_ref, int64_t ld_ref, const double* obs_x,
                      const double* obs_y, int32_t n_obs, double* mapa, int32_t cap, int64_t ld_mapa, int32_t* c,
                      int32_t memspace);

/* -- the driver loop with the convergence monitor the reference only prints (sensors.py:302-315: calc_cambio of every
 * pass): at most max_sweeps sweeps of the resident poses / map (icmslam_set_poses, icmslam_set_map), stopping after the first
 * sweep whose largest landmark change (calc_cambio's maximum, ICM_SLAM.py:490-495) is <= tol_max_change (<= 0: never).
 * cambios (host, 3 x max_sweeps, row-major rows min / max / mean; may be NULL) receives every pass's triple; *n_done the
 * number of sweeps run.  The triple comes out of the sweep's own map filter (one 200-byte read-back per sweep); the
 * full search of icmslam_calc_cambio is only needed when landmarks merged or appeared in that sweep. */
int icmslam_iterate_until(icmslam_handle* h, const double* x0, int32_t max_sweeps, double tol_max_change,
                          const icmslam_sweep_opts* opts, double* cambios, int32_t* n_done);

/* -- the same driver loop on a batch handle (icmslam_set_batch), one convergence monitor per trajectory.  Trajectory k gets
 * exactly what icmslam_iterate_until gives it alone from the same poses and map: n_done[k] (HOST, K) sweeps, its calc_cambio
 * history in cambios (HOST, 3 x K x max_sweeps, element (r, k, s) at (r * K + k) * max_sweeps + s, rows min / max / mean; may be
 * NULL), its poses and landmarks.  After its first sweep whose own largest change is <= tol_max_change (<= 0: never) the
 * trajectory is FROZEN on the device: none of its scans is associated or contributes statistics or labels, none of its poses is
 * solved, and its poses, landmarks and landmark counts stay bit for bit as they were.  The call returns when every trajectory is
 * frozen or after max_sweeps sweeps (*n_run: sweeps the handle ran), with every trajectory unfrozen again: later sweeps continue
 * each one as its own handle would.
 * A landmark belongs to region k = rint(y / region_pitch) * region_cols + rint(x / region_pitch) (icm_slam_b200/batch.py lays the
 * trajectories out so); ICMSLAM_ERR_INVALID for a handle that is not a batch handle, region_pitch <= 0, region_cols <= 0,
 * max_sweeps < 0 or a landmark of the starting map outside regions 0 .. K-1.  (REDBLACK, NEWTON, PREV) sweeps on one GPU only
 * (ICMSLAM_ERR_UNSUPPORTED otherwise).  Element 16 of icmslam_get_sweep_stats: sweeps of the last call that needed the full
 * calc_cambio search for some trajectory (a landmark appeared, merged or left its proven radius). */
int icmslam_batch_iterate_until(icmslam_handle* h, int32_t max_sweeps, double tol_max_change, double region_pitch,
                                int32_t region_cols, const icmslam_sweep_opts* opts, double* cambios, int32_t* n_done,
                                int32_t* n_run);

/* -- filtrar_obs.m (scripts/filtrar_obs.m:6-50), the offline scan gate: keep the k(t) nearest
 * returns per scan.  obs / out: B x T. */
int icmslam_filtrar_obs(icmslam_handle* h, const double* obs, int32_t B, int32_t T, int64_t ld, double max_dist,
                        int32_t cant_max, double* out, int64_t ld_out, int32_t memspace);

#ifdef __cplusplus
}
#endif
#endif /* ICMSLAM_H_ */
