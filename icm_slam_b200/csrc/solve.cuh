// solve.cuh -- the red-black pose update of the (REDBLACK, NEWTON, PREV) sweep as ONE launch: k_solve_tile.
//
// For every pose t the exact conditional minimiser of fun_xn / fun_x (sensors.py:224-282) given its two neighbours, its
// odometry increments and controls, the static body-frame moments of its scan (k_body_moments) and the six landmark
// moments of its scan (runs.cuh: `dyn`, written by the run kernels).  Red-black Gauss-Seidel in time (the restated
// schedule of DESIGN.md section 2): odd poses from the OLD even neighbours, then even poses from the NEW odd ones.
//
// A block owns ST_OWN = 2 ST_SLOTS - 2 consecutive poses tb .. tb+ST_OWN-1 (tb even) and stages poses tb-2 .. tb+ST_OWN,
// their odometry increments, controls and heading sin/cos in shared memory.  Thread q (a slot) solves the whole odd pose
// tb-1+2q (q = 0: the halo tb-1, owned by the previous tile, which computes the identical value from the identical inputs),
// then, after a block barrier, the even pose tb+2q from the new odd poses in shared memory: every warp works in both colour
// phases.  Every input is read once; the new poses and their projection parameters (x, y, sin/cos of theta - pi/2: what
// tras_rot_z needs next sweep, ICM_SLAM.py:465-480) are written coalesced.
#pragma once
#include "common.cuh"

#define ST_SLOTS 64
#define ST_THREADS ST_SLOTS         // a thread per slot; a slot solves one odd and one even pose
#define ST_OWN (2 * ST_SLOTS - 2)
#define ST_XT (2 * ST_SLOTS + 4)    // pose-tile entries: poses tb-2 .. tb+ST_OWN (2*ST_SLOTS+1 used)
#define ST_MINB 8                   // resident blocks per SM k_solve_tile is compiled for (122 registers)

// odometry increments, sweep-invariant: D_t = Rota(o_t.theta) (o_{t+1}.xy - o_t.xy), dtheta_t
// (sensors.py:236-238, :250-253).  inc[:, t] for t < T-1; the last column is zero.
__global__ void k_odo_increments(const double* __restrict__ odo, int64_t ldo, int T, double* __restrict__ inc, int64_t ldi)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    double dx = 0.0, dy = 0.0, dth = 0.0;
    if (t + 1 < T) {
        double s, c;
        sincos(odo[2 * ldo + t], &s, &c);
        const double vx = odo[t + 1] - odo[t], vy = odo[ldo + t + 1] - odo[ldo + t];
        dx = c * vx + s * vy;
        dy = -s * vx + c * vy;
        dth = odo[2 * ldo + t + 1] - odo[2 * ldo + t];
    }
    inc[t] = dx; inc[ldi + t] = dy; inc[2 * ldi + t] = dth;
}

// body-frame moment sums of every scan's kept beams: sum bx, sum by, sum bx^2, sum by^2, sum bx*by and the beam count.
// They do not depend on the poses or the map, so they are formed once per dataset (one thread per scan, fixed order: the
// result does not depend on any tiling) and the solve only reads them (48 B per pose).
__global__ void __launch_bounds__(128)
k_body_moments(const int* __restrict__ off, const double2* __restrict__ bxy, int T, double* __restrict__ bm, int64_t ld)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    double Bx = 0.0, By = 0.0, Bxx = 0.0, Byy = 0.0, Bxy = 0.0;
    for (int i = off[t]; i < off[t + 1]; ++i) {
        const double2 b = bxy[i];
        Bx += b.x; By += b.y;
        Bxx = fma(b.x, b.x, Bxx); Byy = fma(b.y, b.y, Byy); Bxy = fma(b.x, b.y, Bxy);
    }
    bm[t] = Bx; bm[ld + t] = By; bm[2 * ld + t] = Bxx; bm[3 * ld + t] = Byy; bm[4 * ld + t] = Bxy;
    bm[5 * ld + t] = (double)(off[t + 1] - off[t]);
}

// interleaves the extraction's (bx, by) arrays into the double2 records the association kernel stages
__global__ void k_interleave(const double* __restrict__ bx, const double* __restrict__ by, int64_t n, double2* __restrict__ out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = make_double2(bx[i], by[i]);
}

// ppar of poses given from outside (set_poses, host sweeps, halo columns).  A pinned column is projected with its x0
// (sensors.py:131,141), not with x[:,t].
__global__ void k_ppar_init(const double* __restrict__ x, int64_t ld, int t_begin, int t_end, const TrajLayout L, double4* __restrict__ ppar)
{
    const int t = t_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= t_end) return;
    if (L.pinned(t)) ppar[t] = make_ppar(L.x0_of(t, 0), L.x0_of(t, 1), L.x0_of(t, 2));
    else ppar[t] = make_ppar(x[t], x[ld + t], x[2 * ld + t]);
}

__device__ __forceinline__ double entrepi_fast(double a)
{
    return (fabs(a) <= ICM_PI) ? a : entrepi(a);
}

// sin/cos of a small increment (|d| <= 0.125): Taylor to d^11 / d^10, error < 1e-18
__device__ __forceinline__ void sincos_small(double d, double& s, double& c)
{
    const double z = d * d;
    s = d * fma(z, fma(z, fma(z, fma(z, fma(z, -2.5052108385441719e-08, 2.7557319223985893e-06), -1.9841269841269841e-04),
                              8.3333333333333332e-03), -1.6666666666666666e-01), 1.0);
    c = fma(z, fma(z, fma(z, fma(z, fma(z, -2.7557319223985888e-07, 2.4801587301587302e-05), -1.3888888888888889e-03),
                          4.1666666666666664e-02), -0.5), 1.0);
}

struct Mom {   // moment sums of one pose's observations (landmark coordinates relative to the pose's input position)
    double n, Bx, By, Bxx, Byy, Bxy, Yx, Yy, Mxx, Mxy, Myx, Myy;
};

struct PoseIn {
    double ax, ay, ath, sa, ca;     // x_{t-1} and sin/cos of its heading
    double bx, by, bth;             // x_{t+1}
    double uav, uaw, ucv, ucw;      // u_{t-1}, u_t
    double D0x, D0y, dth0;          // odometry increment t-1 -> t
    double D1x, D1y, dth1;          // odometry increment t -> t+1
    int has_next;
};

// The reduced 1-D problem in closed form.  For fixed theta the energy is quadratic in (x, y) with diagonal weights
// (SURVEY.md App. A), so (x, y) are eliminated and phi(theta) remains.  With s = sin(theta), c = cos(theta),
//     phi'(theta)  = 2 (as s + ac c + au s c + av (c^2 - s^2)) + ang1(theta)
//     phi''(theta) = 2 (as c - ac s + au (c^2 - s^2) - 4 av s c) + ang2,
// ang1 the (piecewise linear) angular residuals.  The four coefficients depend on the pose's moments and neighbours but not
// on theta: they are formed ONCE, each the sum of an x-row share (role 0) and a y-row share (role 1; the y rows are the x
// rows rotated by -pi/2), and an iteration costs a dozen FMAs.  Same root as the oracle's newton_pose.
//
// row_coef forms one row's share, in the frame (a, b) = (c, s) for the x rows resp. (s, -c) for the y rows.  The caller
// passes the row's weights r, q, its coordinate of x_{t-1} and x_{t+1} relative to the pose's input position (a_, bp), hu
// (cos resp. sin of x_{t-1}'s heading: u_{t-1} along the row), e0i (the odometry increment t-1 -> t along the row) and the
// row's landmark moments Y, M1, M2.  Every product that meets a sum is written as the fma or the rounded product it is
// evaluated with: the two rows sit side by side in one thread and share sub-expressions, and the compiler must not be free
// to contract them differently from one row alone -- the result is the same to the last bit whichever way the rows are laid
// out.
struct RowCoef {
    double iS, KA, P1, P2;      // what the row's coordinate at the root needs
    double ba, bb, bab, bd;     // the row's share of the four coefficients
};

__device__ __forceinline__ RowCoef row_coef(const Mom& M, double r, double q, double k, double dt, double hn, double dv, double D1x,
                                            double D1y, double kD1x, double kD1y, double uav, double a_, double hu, double e0i,
                                            double bp, double Y, double M1, double M2)
{
    RowCoef R;
    const double ga = fma(mul_rn(hu, uav), dt, a_);                  // a_ + dt (hu u_{t-1}.v)
    const double e0 = add_rn(a_, e0i);
    const double rk = add_rn(r, k), rdv = mul_rn(r, dv);
    R.iS = 1.0 / fma(hn, rk, fma(M.n, q, rk));                       // 1 / (r + k + n q + hn (r + k))
    R.KA = fma(rk, bp, fma(q, Y, fma(ga, r, mul_rn(k, e0))));        // r ga + k e0 + q Y + (r + k) bp
    R.P1 = fma(q, M.By, add_rn(rdv, kD1x));                          // (r dv + k D1x) + q By
    R.P2 = fma(q, M.Bx, -kD1y);                                      // q Bx - k D1y
    const double iKA = mul_rn(R.iS, R.KA);
    R.ba = fma(iKA, R.P2, fma(mul_rn(k, bp), D1y, -mul_rn(q, M1)));
    R.bb = fma(-iKA, R.P1, fma(bp, fma(r, dv, kD1x), mul_rn(q, M2)));
    R.bab = fma(-R.iS, fma(R.P2, R.P2, -mul_rn(R.P1, R.P1)),
                fma(q, sub_rn(M.Bxx, M.Byy), -fma(rdv, dv, mul_rn(k, fma(D1x, D1x, -mul_rn(D1y, D1y))))));
    R.bd = fma(-mul_rn(R.iS, R.P1), R.P2, fma(q, M.Bxy, -mul_rn(kD1x, D1y)));
    return R;
}

// One pose in one thread: both rows' shares, one iteration loop, both coordinates and theta at the root.  A converged pose
// freezes, so its result does not depend on how long its warp-mates iterate.  Returns the iteration count.
__device__ __forceinline__ int newton_trig(const DevCfg& cfg, const PoseIn& P, const Mom& M, double ox, double oy, double& th,
                                           double s, double c, double tol, int maxit, double& x, double& y)
{
    const double dt = cfg.dt, k = cfg.kod;
    const double hn = P.has_next ? 1.0 : 0.0;
    const double D1x = mul_rn(hn, P.D1x), D1y = mul_rn(hn, P.D1y);
    const double dv = mul_rn(mul_rn(hn, dt), P.ucv);
    const double kD1x = mul_rn(k, D1x), kD1y = mul_rn(k, D1y);
    const RowCoef X = row_coef(M, cfg.r1, cfg.q1, k, dt, hn, dv, D1x, D1y, kD1x, kD1y, P.uav, sub_rn(P.ax, ox), P.ca,
                               fma(P.ca, P.D0x, -mul_rn(P.sa, P.D0y)), mul_rn(hn, sub_rn(P.bx, ox)), M.Yx, M.Mxx, M.Mxy);
    const RowCoef Y = row_coef(M, cfg.r2, cfg.q2, k, dt, hn, dv, D1x, D1y, kD1x, kD1y, P.uav, sub_rn(P.ay, oy), P.sa,
                               fma(P.ca, P.D0y, mul_rn(P.sa, P.D0x)), mul_rn(hn, sub_rn(P.by, oy)), M.Yy, M.Myx, M.Myy);
    const double as2 = 2.0 * add_rn(X.bb, Y.ba), ac2 = 2.0 * sub_rn(X.ba, Y.bb);
    const double au2 = 2.0 * sub_rn(X.bab, Y.bab), av2 = 2.0 * sub_rn(X.bd, Y.bd);
    const double av8 = 4.0 * av2;
    const double ang2 = (2.0 * cfg.r3 + 2.0 * k) * (1.0 + hn);
    const double r3_2 = 2.0 * cfg.r3, k_2 = 2.0 * k;
    const double th_ga = fma(dt, P.uaw, P.ath), c3 = add_rn(P.dth0, P.ath), c4 = sub_rn(P.dth1, P.bth), wb = fma(dt, P.ucw, -P.bth);
    int it = 0;
    bool done = false;
    for (;;) {
        const double u = s * c, v = fma(c, c, -s * s);
        double ang1 = fma(r3_2, entrepi_fast(th - th_ga), -k_2 * entrepi_fast(c3 - th));
        if (P.has_next) ang1 += fma(r3_2, entrepi_fast(th + wb), k_2 * entrepi_fast(c4 + th));
        const double p1 = fma(as2, s, fma(ac2, c, fma(au2, u, fma(av2, v, ang1))));
        double p2 = fma(as2, c, fma(-ac2, s, fma(au2, v, fma(-av8, u, ang2))));
        if (!(p2 > 0.0)) p2 = ang2;
        const double dth = mul_rn(-p1, (double)__frcp_rn((float)p2));   // quasi-Newton: 24-bit reciprocal of the curvature, same fixed point
        if (!done) {       // a converged pose is frozen: its result does not depend on how long its warp-mates iterate
            th = add_rn(th, dth);
            ++it;
            if (fabs(dth) <= 0.125) {
                double sd, cd;
                sincos_small(dth, sd, cd);
                const double s2 = fma(s, cd, c * sd);
                c = fma(c, cd, -s * sd);
                s = s2;
            } else {
                sincos(th, &s, &c);
            }
            done = fabs(dth) <= tol || it >= maxit;
        }
        if (__all_sync(FULLMASK, done)) break;
    }
    x = fma(fma(-s, X.P2, fma(-c, X.P1, X.KA)), X.iS, ox);       // (KA - c P1 - s P2) iS + ox
    y = fma(fma(c, Y.P2, fma(-s, Y.P1, Y.KA)), Y.iS, oy);        // (KA - s P1 + c P2) iS + oy
    return it;
}

struct SolveParams {
    int T;                                // columns of this handle's trajectory (a time segment incl. its halo columns)
    int t_lo, t_hi;                       // owned poses [t_lo, t_hi), t_lo even
    TrajLayout lay;                       // pinned first poses (self.x0) and trajectory ends
    const double* xin; int64_t ldin;      // 3 x T input poses
    double* xout; int64_t ldout;          // 3 x T output poses
    const double* inc; int64_t ldinc;     // 3 x T odometry increments
    const double* u; int64_t ldu;         // 2 x T controls
    const double* bm; int64_t ldbm;       // 6 x T static body-frame moments + beam count
    const double* dyn;                    // 6 doubles per pose: (Yx, Mxx, Mxy, Yy, Myx, Myy), written by the run kernels
    const double4* ppin; double4* ppout;  // projection parameters of the input / output poses
    DevCfg cfg;
    double tol; int maxit;
    unsigned long long* iters;
    int tile0;                            // first tile of this launch
    unsigned long long* trace_row;        // instrumentation: ring of %globaltimer marks (or null), indexed by *trace_seq
    const unsigned* trace_seq;
    Freeze fz;                            // a frozen trajectory's poses (and projection parameters) are copied through, not solved
};

struct __align__(16) SolveSmem {
    double xs[3][ST_XT];           // input poses tb-2 .. tb+ST_OWN, index li = t - (tb-2)
    double xn[3][ST_XT];           // new poses (same indexing)
    double inc[3][ST_XT];
    double u[2][ST_XT];
    double sn[ST_XT], cs[ST_XT];   // sin/cos of the input headings (after the odd phase: of the new odd headings)
};

// the pose a thread solves in one colour phase: everything it needs beyond the tile's shared arrays
struct SlotMom {
    Mom M;
    bool valid, pinned;
    int t, li;
};

template <bool FZ>
__device__ __forceinline__ SlotMom solve_slot_load(const SolveParams& p, int tb, int q, int phase)
{
    SlotMom s;
    s.t = phase == 0 ? tb - 1 + 2 * q : tb + 2 * q;
    s.li = s.t - (tb - 2);
    // (phase 0, slot 0 = the odd pose tb-1 left of the tile: re-solved here because the even pose tb needs its NEW value;
    //  phase 1, last slot = tb+ST_OWN: the next tile's)
    s.valid = s.t >= 0 && s.t < p.t_hi && (phase == 0 ? (q == 0 || s.t >= p.t_lo) : (q != ST_SLOTS - 1 && s.t >= p.t_lo));
    // (a frozen pose is handled like a pinned one: its input value passes through; the trajectory's first pose is pinned and its
    //  last has no successor, so no pose of another trajectory reads it)
    s.pinned = s.valid && (p.lay.pinned(s.t) || (FZ && p.fz.scan(s.t)));
    Mom& M = s.M;
    M.n = M.Bx = M.By = M.Bxx = M.Byy = M.Bxy = M.Yx = M.Yy = M.Mxx = M.Mxy = M.Myx = M.Myy = 0.0;
    if (s.valid && !s.pinned) {
        const double* bmq = p.bm + s.t;
        M.n = __ldg(bmq + 5 * p.ldbm);
        M.Bx = __ldg(bmq); M.By = __ldg(bmq + p.ldbm); M.Bxx = __ldg(bmq + 2 * p.ldbm);
        M.Byy = __ldg(bmq + 3 * p.ldbm); M.Bxy = __ldg(bmq + 4 * p.ldbm);
        // the six landmark moments, 48 B per pose (stale where the scan is empty: unused)
        const double2* d = reinterpret_cast<const double2*>(p.dyn + (size_t)s.t * 6);
        const double2 d0 = d[0], d1 = d[1], d2 = d[2];
        M.Yx = d0.x; M.Mxx = d0.y; M.Mxy = d1.x; M.Yy = d1.y; M.Myx = d2.x; M.Myy = d2.y;
    }
    return s;
}

// FZ: a batch with frozen trajectories (p.fz); the plain sweep launches the instance without the test
template <bool FZ>
__global__ void __launch_bounds__(ST_THREADS, ST_MINB)
k_solve_tile(const SolveParams p)
{
    __shared__ SolveSmem S;
    const int q = threadIdx.x;      // the slot
    if (p.trace_row && blockIdx.x == 0 && q == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); p.trace_row[((*p.trace_seq) & 31) * 8 + 5] = t; }
    const int tb = p.t_lo + (p.tile0 + blockIdx.x) * ST_OWN;      // t_lo is even: colours stay aligned with the global time index
    const int T = p.T;
    SlotMom cur = solve_slot_load<FZ>(p, tb, q, 0);      // (in flight while the tile is staged)
    for (int li = q; li < ST_XT; li += ST_THREADS) {
        const int t = tb - 2 + li;
        const bool ok = t >= 0 && t < T;
        double th = 0.0;
        for (int r = 0; r < 3; ++r) {
            const double v = ok ? p.xin[r * p.ldin + t] : 0.0;
            S.xs[r][li] = v; S.xn[r][li] = v;
            S.inc[r][li] = ok ? p.inc[r * p.ldinc + t] : 0.0;
            if (r == 2) th = v;
        }
        S.u[0][li] = ok ? p.u[t] : 0.0;
        S.u[1][li] = ok ? p.u[p.ldu + t] : 0.0;
        double sh = 0.0, ch = 1.0;
        if (ok) {
            if (p.lay.pinned(t)) sincos(th, &sh, &ch);       // (a pinned column's ppar belongs to its x0; x[:,t] is only a neighbour)
            else { const double4 pq = ldg_ppar(p.ppin + t); sh = pq.w; ch = -pq.z; }
        }
        S.sn[li] = sh; S.cs[li] = ch;
    }
    __syncthreads();
    int my_iters = 0;
    for (int phase = 0; phase < 2; ++phase) {
        // every thread solves one pose per colour phase: the odd pose tb-1+2q from the OLD even neighbours, then, after the
        // block barrier, the even pose tb+2q from the NEW odd ones
        const Mom& M = cur.M;
        const int t = cur.t, li = cur.li;
        const bool qvalid = cur.valid, pinned = cur.pinned;
        double rx = 0.0, ry = 0.0, th = 0.0;
        PoseIn P;
        P.ax = P.ay = P.ath = P.sa = 0.0; P.ca = 1.0; P.bx = P.by = P.bth = 0.0; P.uav = P.uaw = P.ucv = P.ucw = 0.0;
        P.D0x = P.D0y = P.dth0 = P.D1x = P.D1y = P.dth1 = 0.0; P.has_next = 0;
        bool solve = false;
        double ox = 0.0, oy = 0.0, th0 = 0.0, s0 = 0.0, c0 = 1.0;
        if (qvalid) {
            // neighbours: old poses for the odd phase, new (odd) poses for the even phase
            double (*X)[ST_XT] = phase == 0 ? S.xs : S.xn;
            const bool has_next = p.lay.has_next(t, T);
            solve = !pinned && M.n > 0.0;
            ox = S.xs[0][li]; oy = S.xs[1][li]; th0 = S.xs[2][li]; s0 = S.sn[li]; c0 = S.cs[li];
            th = th0;
            if (!pinned) {
                P.ax = X[0][li - 1]; P.ay = X[1][li - 1]; P.ath = X[2][li - 1];
                P.sa = S.sn[li - 1]; P.ca = S.cs[li - 1];
                if (has_next) { P.bx = X[0][li + 1]; P.by = X[1][li + 1]; P.bth = X[2][li + 1]; }
                P.uav = S.u[0][li - 1]; P.uaw = S.u[1][li - 1];
                P.ucv = S.u[0][li]; P.ucw = S.u[1][li];
                P.D0x = S.inc[0][li - 1]; P.D0y = S.inc[1][li - 1]; P.dth0 = S.inc[2][li - 1];
                P.D1x = S.inc[0][li]; P.D1y = S.inc[1][li]; P.dth1 = S.inc[2][li];
                P.has_next = has_next ? 1 : 0;
                if (!solve) {       // sensors.py:147-151: no observation, average of the neighbours
                    const bool t1 = p.lay.after_pinned(t);
                    rx = ((t1 ? p.lay.x0_of(t - 1, 0) : X[0][li - 1]) + X[0][li + 1]) / 2.0;
                    ry = ((t1 ? p.lay.x0_of(t - 1, 1) : X[1][li - 1]) + X[1][li + 1]) / 2.0;
                    th = ((t1 ? p.lay.x0_of(t - 1, 2) : X[2][li - 1]) + X[2][li + 1]) / 2.0;
                }
            }
        }
        {
            // (threads that do not solve still run the loop once with harmless values: its exit vote needs every lane)
            double x2 = 0.0, y2 = 0.0, th2 = th0;
            const int it = newton_trig(p.cfg, P, M, ox, oy, th2, s0, c0, p.tol, solve ? p.maxit : 1, x2, y2);
            if (solve) { rx = x2; ry = y2; th = th2; my_iters += it; }
        }
        SlotMom nxt = cur;
        if (phase == 0) nxt = solve_slot_load<FZ>(p, tb, q, 1);      // (the even pose's moments arrive during the barrier)
        if (qvalid && !pinned) {
            // the new heading's sin/cos exactly as next sweep's projection forms them (one sincos per pose per sweep)
            double st, ct;
            sincos(sub_rn(th, ICM_HALFPI), &st, &ct);
            S.xn[0][li] = rx; S.xn[1][li] = ry; S.xn[2][li] = th;
            S.sn[li] = ct; S.cs[li] = -st;      // (the old headings of this colour are no longer needed)
        }
        __syncthreads();
        cur = nxt;
    }
    if (p.iters) {
        my_iters = warp_sum_i(my_iters);
        if ((q & 31) == 0 && my_iters) atomicAdd(p.iters, (unsigned long long)my_iters);
    }
    // ---- outputs: the owned poses and their projection parameters ---------------------------------------------------
    const int n_own = min(ST_OWN, p.t_hi - tb);
    for (int r = 0; r < 3; ++r)
        for (int k = q; k < n_own; k += ST_THREADS) p.xout[r * p.ldout + tb + k] = S.xn[r][k + 2];
    for (int k = q; k < n_own; k += ST_THREADS) {
        const int tt = tb + k, l2 = k + 2;
        if (p.lay.pinned(tt)) p.ppout[tt] = make_ppar(p.lay.x0_of(tt, 0), p.lay.x0_of(tt, 1), p.lay.x0_of(tt, 2));
        else if (FZ && p.fz.scan(tt)) p.ppout[tt] = ldg_ppar(p.ppin + tt);
        else p.ppout[tt] = make_double4(S.xn[0][l2], S.xn[1][l2], -S.cs[l2], S.sn[l2]);
    }
}
