// pose.cuh -- the pose half of the ICM sweep (sensors.py:145-162, :213-282).
//
// Energies follow sensors.py:224-282 (fun_xn / fun_x).  Two inner solvers:
//   * NM      -- Nelder-Mead exactly as the reference runs scipy.optimize.fmin (xtol=1e-3,
//                ftol=1e-4, 600 evaluations), energy evaluated observation by observation;
//   * NEWTON  -- the exact conditional minimiser.  For a fixed heading the energy is quadratic in
//                (x, y) with a diagonal Hessian (Q, R diagonal, Rota orthonormal), so (x, y) is
//                eliminated in closed form and theta is found by Newton on the reduced function.
//                All observation terms enter through 11 moment sums accumulated in ONE pass over
//                the pose's observations, so the iterations cost O(1) per pose.
// Two schedules: REDBLACK (odd poses, then even poses; thread per pose) and SEQUENTIAL (the
// reference's forward Gauss-Seidel; one warp walks each trajectory).  Both keep to the batch
// rules of TrajLayout (common.cuh).
#pragma once
#include "common.cuh"
#include "assoc.cuh"

struct SeenSrc {
    int view;                       // ICMSLAM_VIEW_*
    const int* c;                   // labels per observation
    const double *seen_x, *seen_y;  // per observation (RUNNING)
    const double *raw_x, *raw_y;    // per label: this sweep's means (FULL; new labels in PREV)
    const double *min_x, *min_y;    // previous map rows (PREV)
    const int* lsearch_ptr;         // labels < *lsearch_ptr index the previous map (device value)
};

__device__ __forceinline__ void seen_of(const SeenSrc& S, int i, double& sx, double& sy)
{
    if (S.view == ICMSLAM_VIEW_RUNNING) { sx = S.seen_x[i]; sy = S.seen_y[i]; return; }
    int l = S.c[i];
    if (S.view == ICMSLAM_VIEW_PREV && l < __ldg(S.lsearch_ptr)) { sx = __ldg(S.min_x + l); sy = __ldg(S.min_y + l); }
    else { sx = S.raw_x[l]; sy = S.raw_y[l]; }
}

struct PoseProblem {
    double a[3], b[3];       // x_{t-1} (x_ant), x_{t+1} (x_pos)
    double ua[2], uc[2];     // u_{t-1}, u_t
    double o0[3], o1[3], o2[3];
    int has_next;            // fun_xn (1) or fun_x (0)
    int o, n;                // CSR slice of the pose's observations
};

struct ObsArrays {
    const double *bx, *by, *d;
    const int* beam;
    const double* ang;       // beam angle table (i*pi)/180
};

// g (sensors.py:206-211)
__device__ __forceinline__ void g_step(const double p[3], double v, double w, double dt, double out[3])
{
    double s, c;
    sincos(p[2], &s, &c);
    out[0] = p[0] + dt * (c * v);
    out[1] = p[1] + dt * (s * v);
    out[2] = p[2] + dt * w;
}

__device__ __forceinline__ void rota_mul(double phi, double vx, double vy, double& ox, double& oy)
{
    double s, c;
    sincos(phi, &s, &c);
    ox = c * vx + s * vy;
    oy = -s * vx + c * vy;
}

// ---- faithful energy (used by NM) ------------------------------------------------------------
// WARPED: called by all 32 lanes of a warp with the same arguments (k_pose_walk).  The lanes form the per-observation residuals
// side by side; every lane then adds them into h in observation order with the scalar loop's expressions, so the energy is the
// same to the last bit and the same on every lane.
template <bool WARPED = false>
__device__ double pose_energy(const DevCfg& cfg, const PoseProblem& P, const ObsArrays& O, const SeenSrc& S, const double x[3])
{
    double f = 0.0;
    double ox, oy, px, py;
    if (P.has_next) {   // sensors.py:233-240
        double gx[3];
        g_step(x, P.uc[0], P.uc[1], cfg.dt, gx);
        double g0 = gx[0] - P.b[0], g1 = gx[1] - P.b[1], g2 = entrepi(gx[2] - P.b[2]);
        rota_mul(P.o1[2], P.o2[0] - P.o1[0], P.o2[1] - P.o1[1], ox, oy);
        rota_mul(x[2], P.b[0] - x[0], P.b[1] - x[1], px, py);
        double e0 = ox - px, e1 = oy - py, e2 = entrepi(P.o2[2] - P.o1[2] - P.b[2] + x[2]);
        f = (g0 * cfg.r1 * g0 + g1 * cfg.r2 * g1 + g2 * cfg.r3 * g2) + cfg.kod * (e0 * e0 + e1 * e1 + e2 * e2);
    }
    double ga[3];
    g_step(P.a, P.ua[0], P.ua[1], cfg.dt, ga);   // sensors.py:247-255 / 273-281
    double g0 = x[0] - ga[0], g1 = x[1] - ga[1], g2 = entrepi(x[2] - ga[2]);
    double hh = 0.0;                              // h, sensors.py:194-204
    if constexpr (WARPED) {
        const int lane = threadIdx.x & (WARP - 1);
        for (int k0 = 0; k0 < P.n; k0 += WARP) {
            double dx = 0.0, dy = 0.0;
            if (k0 + lane < P.n) {
                int i = P.o + k0 + lane;
                double alfa = O.ang[O.beam[i]] + x[2] - ICM_HALFPI;
                double s, c, sx, sy;
                sincos(alfa, &s, &c);
                seen_of(S, i, sx, sy);
                dx = (x[0] + O.d[i] * c) - sx; dy = (x[1] + O.d[i] * s) - sy;
            }
            const int m = min(WARP, P.n - k0);
            for (int j = 0; j < m; ++j) {
                const double ex = __shfl_sync(FULLMASK, dx, j), ey = __shfl_sync(FULLMASK, dy, j);
                hh += ex * cfg.q1 * ex;
                hh += ey * cfg.q2 * ey;
            }
        }
    } else {
        for (int k = 0; k < P.n; ++k) {
            int i = P.o + k;
            double alfa = O.ang[O.beam[i]] + x[2] - ICM_HALFPI;
            double s, c, sx, sy;
            sincos(alfa, &s, &c);
            seen_of(S, i, sx, sy);
            double dx = (x[0] + O.d[i] * c) - sx, dy = (x[1] + O.d[i] * s) - sy;
            hh += dx * cfg.q1 * dx;
            hh += dy * cfg.q2 * dy;
        }
    }
    rota_mul(P.o0[2], P.o1[0] - P.o0[0], P.o1[1] - P.o0[1], ox, oy);
    rota_mul(P.a[2], x[0] - P.a[0], x[1] - P.a[1], px, py);
    double e0 = ox - px, e1 = oy - py, e2 = entrepi(P.o1[2] - P.o0[2] - x[2] + P.a[2]);
    f = f + (g0 * cfg.r1 * g0 + g1 * cfg.r2 * g1 + g2 * cfg.r3 * g2) + hh + cfg.kod * (e0 * e0 + e1 * e1 + e2 * e2);
    return f;
}

// ---- Nelder-Mead as scipy runs it for the reference (sensors.py:221,263) ---------------------
__device__ __forceinline__ void nm_sort4(double sim[4][3], double fs[4])
{
    for (int i = 1; i < 4; ++i) {
        double f = fs[i], v0 = sim[i][0], v1 = sim[i][1], v2 = sim[i][2];
        int j = i - 1;
        while (j >= 0 && fs[j] > f) {
            fs[j + 1] = fs[j];
            sim[j + 1][0] = sim[j][0]; sim[j + 1][1] = sim[j][1]; sim[j + 1][2] = sim[j][2];
            --j;
        }
        fs[j + 1] = f;
        sim[j + 1][0] = v0; sim[j + 1][1] = v1; sim[j + 1][2] = v2;
    }
}

template <bool WARPED = false>
__device__ int nelder_mead(const DevCfg& cfg, const PoseProblem& P, const ObsArrays& O, const SeenSrc& S,
                           const double start[3], double out[3])
{
    const double xtol = 1e-3, ftol = 1e-4;
    const int maxiter = 600, maxfun = 600;
    double sim[4][3], fs[4];
    int nev = 0;
    for (int j = 0; j < 3; ++j) sim[0][j] = start[j];
    for (int k = 0; k < 3; ++k) {
        for (int j = 0; j < 3; ++j) sim[k + 1][j] = start[j];
        if (sim[k + 1][k] != 0.0) sim[k + 1][k] = mul_rn(1 + 0.05, sim[k + 1][k]);
        else sim[k + 1][k] = 0.00025;
    }
    for (int k = 0; k < 4; ++k) { fs[k] = pose_energy<WARPED>(cfg, P, O, S, sim[k]); ++nev; }
    nm_sort4(sim, fs);
    int iterations = 1;
    while (nev < maxfun && iterations < maxiter) {
        double dxm = 0.0, dfm = 0.0;
        for (int k = 1; k < 4; ++k) {
            for (int j = 0; j < 3; ++j) dxm = fmax(dxm, fabs(sim[k][j] - sim[0][j]));
            dfm = fmax(dfm, fabs(fs[0] - fs[k]));
        }
        if (dxm <= xtol && dfm <= ftol) break;
        double xbar[3], xr[3], xe[3];
        for (int j = 0; j < 3; ++j) {
            xbar[j] = __ddiv_rn(add_rn(add_rn(sim[0][j], sim[1][j]), sim[2][j]), 3.0);
            xr[j] = sub_rn(mul_rn(2.0, xbar[j]), sim[3][j]);
        }
        double fxr = pose_energy<WARPED>(cfg, P, O, S, xr); ++nev;
        bool doshrink = false;
        if (fxr < fs[0]) {
            for (int j = 0; j < 3; ++j) xe[j] = sub_rn(mul_rn(3.0, xbar[j]), mul_rn(2.0, sim[3][j]));
            double fxe = pose_energy<WARPED>(cfg, P, O, S, xe); ++nev;
            if (fxe < fxr) { for (int j = 0; j < 3; ++j) sim[3][j] = xe[j]; fs[3] = fxe; }
            else { for (int j = 0; j < 3; ++j) sim[3][j] = xr[j]; fs[3] = fxr; }
        } else if (fxr < fs[2]) {
            for (int j = 0; j < 3; ++j) sim[3][j] = xr[j];
            fs[3] = fxr;
        } else {
            if (fxr < fs[3]) {
                for (int j = 0; j < 3; ++j) xe[j] = sub_rn(mul_rn(1.5, xbar[j]), mul_rn(0.5, sim[3][j]));
                double fxc = pose_energy<WARPED>(cfg, P, O, S, xe); ++nev;
                if (fxc <= fxr) { for (int j = 0; j < 3; ++j) sim[3][j] = xe[j]; fs[3] = fxc; }
                else doshrink = true;
            } else {
                for (int j = 0; j < 3; ++j) xe[j] = add_rn(mul_rn(0.5, xbar[j]), mul_rn(0.5, sim[3][j]));
                double fxcc = pose_energy<WARPED>(cfg, P, O, S, xe); ++nev;
                if (fxcc < fs[3]) { for (int j = 0; j < 3; ++j) sim[3][j] = xe[j]; fs[3] = fxcc; }
                else doshrink = true;
            }
            if (doshrink) {
                for (int k = 1; k < 4; ++k) {
                    for (int j = 0; j < 3; ++j) sim[k][j] = add_rn(sim[0][j], mul_rn(0.5, sub_rn(sim[k][j], sim[0][j])));
                    fs[k] = pose_energy<WARPED>(cfg, P, O, S, sim[k]); ++nev;
                }
            }
        }
        ++iterations;
        nm_sort4(sim, fs);
    }
    out[0] = sim[0][0]; out[1] = sim[0][1]; out[2] = sim[0][2];
    return nev;
}

// ---- exact solver: moments + Newton on the reduced 1-D function --------------------------------
// Moments of one pose's observations.  Body-frame sums are sweep-invariant; the seen-landmark
// sums use coordinates relative to (ox, oy) to keep the variance-like differences small.
struct Moments {
    double n, Bx, By, Bxx, Byy, Bxy;             // sum b, sum b b^T
    double Yx, Yy, Mxx, Mxy, Myx, Myy;           // sum yhat, sum yhat b^T
};

__device__ __forceinline__ void moments_zero(Moments& M)
{
    M.n = M.Bx = M.By = M.Bxx = M.Byy = M.Bxy = 0.0;
    M.Yx = M.Yy = M.Mxx = M.Mxy = M.Myx = M.Myy = 0.0;
}
__device__ __forceinline__ void moments_add(Moments& M, double bx, double by, double yx, double yy)
{
    M.n += 1.0;
    M.Bx += bx; M.By += by;
    M.Bxx = fma(bx, bx, M.Bxx); M.Byy = fma(by, by, M.Byy); M.Bxy = fma(bx, by, M.Bxy);
    M.Yx += yx; M.Yy += yy;
    M.Mxx = fma(yx, bx, M.Mxx); M.Mxy = fma(yx, by, M.Mxy);
    M.Myx = fma(yy, bx, M.Myx); M.Myy = fma(yy, by, M.Myy);
}

// Solves the pose problem given the moments.  (ox, oy) is the local origin the moments' yhat are
// relative to.  Returns the number of Newton iterations.
__device__ int newton_moments(const DevCfg& cfg, const PoseProblem& P, const Moments& M, double ox, double oy,
                              double th0, double tol, int maxit, double out[3])
{
    const double dt = cfg.dt, k = cfg.kod;
    double ga[3];
    g_step(P.a, P.ua[0], P.ua[1], dt, ga);
    double D0x, D0y, D1x = 0.0, D1y = 0.0;
    rota_mul(P.o0[2], P.o1[0] - P.o0[0], P.o1[1] - P.o0[1], D0x, D0y);
    double sa, ca;
    sincos(P.a[2], &sa, &ca);
    const double e0x = (P.a[0] - ox) + (ca * D0x - sa * D0y);     // a_xy + Rota(a_th)^T D0
    const double e0y = (P.a[1] - oy) + (sa * D0x + ca * D0y);
    const double gax = ga[0] - ox, gay = ga[1] - oy;
    double bxp = 0.0, byp = 0.0, v = 0.0, w_act = 0.0;
    double Sx = cfg.r1 + k + M.n * cfg.q1, Sy = cfg.r2 + k + M.n * cfg.q2;
    double KAx = cfg.r1 * gax + k * e0x + cfg.q1 * M.Yx;
    double KAy = cfg.r2 * gay + k * e0y + cfg.q2 * M.Yy;
    double ang2 = 2.0 * cfg.r3 + 2.0 * k;
    if (P.has_next) {
        rota_mul(P.o1[2], P.o2[0] - P.o1[0], P.o2[1] - P.o1[1], D1x, D1y);
        bxp = P.b[0] - ox; byp = P.b[1] - oy;
        v = P.uc[0]; w_act = P.uc[1];
        Sx += cfg.r1 + k; Sy += cfg.r2 + k;
        KAx += (cfg.r1 + k) * bxp;
        KAy += (cfg.r2 + k) * byp;
        ang2 += 2.0 * cfg.r3 + 2.0 * k;
    }
    const double hn = P.has_next ? 1.0 : 0.0;
    const double dv = dt * v;
    // A_x(th) = KAx - c*Pxc - s*Pxs ,  A_y(th) = KAy - s*Pys - c*Pyc
    const double Pxc = hn * (cfg.r1 * dv + k * D1x) + cfg.q1 * M.By;
    const double Pxs = cfg.q1 * M.Bx - hn * k * D1y;
    const double Pys = hn * (cfg.r2 * dv + k * D1x) + cfg.q2 * M.By;
    const double Pyc = hn * k * D1y - cfg.q2 * M.Bx;
    const double th_ga = ga[2];
    const double c3 = P.o1[2] - P.o0[2] + P.a[2];
    const double c4 = P.o2[2] - P.o1[2] - P.b[2];
    double th = th0;
    int it = 0;
    double s, c;
    for (; it < maxit;) {
        sincos(th, &s, &c);
        const double ss = s * s, cc = c * c, sc = s * c;
        const double Ax = KAx - c * Pxc - s * Pxs, Ax1 = s * Pxc - c * Pxs, Ax2 = KAx - Ax;
        const double Ay = KAy - s * Pys - c * Pyc, Ay1 = -c * Pys + s * Pyc, Ay2 = KAy - Ay;
        // sum W c c'  and  sum W (c'^2 + c c'')
        double Cx1 = 0.0, Cx2 = 0.0, Cy1 = 0.0, Cy2 = 0.0;
        if (P.has_next) {
            const double f2 = bxp - dv * c, f21 = dv * s, f22 = dv * c;
            const double f4 = bxp - (c * D1x - s * D1y), f41 = s * D1x + c * D1y, f42 = c * D1x - s * D1y;
            Cx1 = cfg.r1 * f2 * f21 + k * f4 * f41;
            Cx2 = cfg.r1 * (f21 * f21 + f2 * f22) + k * (f41 * f41 + f4 * f42);
            const double h2 = byp - dv * s, h21 = -dv * c, h22 = dv * s;
            const double h4 = byp - (s * D1x + c * D1y), h41 = -(c * D1x - s * D1y), h42 = s * D1x + c * D1y;
            Cy1 = cfg.r2 * h2 * h21 + k * h4 * h41;
            Cy2 = cfg.r2 * (h21 * h21 + h2 * h22) + k * (h41 * h41 + h4 * h42);
        }
        // observation sums with w = Rot(th - pi/2) b = (bx s + by c, -bx c + by s)
        const double Swxwy = sc * (M.Byy - M.Bxx) + (ss - cc) * M.Bxy;
        const double Swxx = ss * M.Bxx + 2.0 * sc * M.Bxy + cc * M.Byy;
        const double Swyy = cc * M.Bxx - 2.0 * sc * M.Bxy + ss * M.Byy;
        const double Yxwy = -c * M.Mxx + s * M.Mxy, Yxwx = s * M.Mxx + c * M.Mxy;
        const double Yywx = s * M.Myx + c * M.Myy, Yywy = -c * M.Myx + s * M.Myy;
        Cx1 += cfg.q1 * (Yxwy - Swxwy);                 // c = yx - wx, c' = wy, c'' = wx
        Cx2 += cfg.q1 * (Swyy + Yxwx - Swxx);
        Cy1 += cfg.q2 * (-Yywx + Swxwy);                // c = yy - wy, c' = -wx, c'' = wy
        Cy2 += cfg.q2 * (Swxx + Yywy - Swyy);
        const double w1 = entrepi(th - th_ga), w3 = entrepi(c3 - th);
        double ang1 = 2.0 * cfg.r3 * w1 - 2.0 * k * w3;
        if (P.has_next) {
            const double w2 = entrepi(th + dt * w_act - P.b[2]), w4 = entrepi(c4 + th);
            ang1 += 2.0 * cfg.r3 * w2 + 2.0 * k * w4;
        }
        const double p1 = 2.0 * Cx1 - 2.0 * Ax * Ax1 / Sx + 2.0 * Cy1 - 2.0 * Ay * Ay1 / Sy + ang1;
        double p2 = 2.0 * Cx2 - 2.0 * (Ax1 * Ax1 + Ax * Ax2) / Sx + 2.0 * Cy2 - 2.0 * (Ay1 * Ay1 + Ay * Ay2) / Sy + ang2;
        if (!(p2 > 0.0)) p2 = ang2;
        const double dth = -p1 / p2;
        th += dth;
        ++it;
        if (fabs(dth) <= tol) break;
    }
    sincos(th, &s, &c);
    out[0] = (KAx - c * Pxc - s * Pxs) / Sx + ox;
    out[1] = (KAy - s * Pys - c * Pyc) / Sy + oy;
    out[2] = th;
    return it;
}

// ---- one pose ------------------------------------------------------------------------------
struct PoseArrays {
    double* x; int64_t ldx;                 // 3 x T poses (in/out)
    const double* odo; int64_t ldo;         // 3 x T
    const double* u; int64_t ldu;           // 2 x T
    TrajLayout lay;                         // self.x0 (sensors.py:131) of the trajectory or of each trajectory of a batch
    const int* off;
    int T;
    // trajectories and columns per trajectory (one trajectory: 1 and T)
    __device__ __forceinline__ int traj_cols() const { return lay.traj_T > 0 ? lay.traj_T : T; }
};

// Pose t (never a pinned one).  WARPED: all 32 lanes of a warp call it for the same t (k_pose_walk) and compute the same
// result; lane 0 writes it.
template <bool WARPED = false>
__device__ __forceinline__ void update_pose(int t, const DevCfg& cfg, const PoseArrays& A, const ObsArrays& O,
                                            const SeenSrc& S, int solver, double tol, int maxit,
                                            unsigned long long* iters)
{
    const bool writer = !WARPED || (threadIdx.x & (WARP - 1)) == 0;
    const int o = A.off[t], n = A.off[t + 1] - o;
    double res[3];
    if (n == 0) {   // sensors.py:147-151: average of the previous result and the next (old) pose
        const bool t1 = A.lay.after_pinned(t);
        for (int j = 0; j < 3; ++j) {
            double prev = t1 ? A.lay.x0_of(t - 1, j) : A.x[j * A.ldx + t - 1];
            res[j] = (prev + A.x[j * A.ldx + t + 1]) / 2.0;
        }
    } else {
        PoseProblem P;
        P.has_next = A.lay.has_next(t, A.T) ? 1 : 0;
        P.o = o; P.n = n;
        for (int j = 0; j < 3; ++j) {
            P.a[j] = A.x[j * A.ldx + t - 1];
            P.o0[j] = A.odo[j * A.ldo + t - 1];
            P.o1[j] = A.odo[j * A.ldo + t];
            P.b[j] = 0.0; P.o2[j] = 0.0;
        }
        P.ua[0] = A.u[t - 1]; P.ua[1] = A.u[A.ldu + t - 1];
        P.uc[0] = P.uc[1] = 0.0;
        double start[3];
        if (P.has_next) {
            for (int j = 0; j < 3; ++j) {
                P.b[j] = A.x[j * A.ldx + t + 1];
                P.o2[j] = A.odo[j * A.ldo + t + 1];
                start[j] = (P.a[j] + P.b[j]) / 2.0;                      // sensors.py:221
            }
            P.uc[0] = A.u[t]; P.uc[1] = A.u[A.ldu + t];
        } else {
            g_step(P.a, P.ua[0], P.ua[1], cfg.dt, start);                // sensors.py:262
        }
        if (solver == ICMSLAM_SOLVER_NM) {
            int nev = nelder_mead<WARPED>(cfg, P, O, S, start, res);
            if (iters && writer) atomicAdd(iters, (unsigned long long)nev);
        } else {
            Moments M;
            moments_zero(M);
            for (int k = 0; k < n; ++k) {
                double sx, sy;
                seen_of(S, o + k, sx, sy);
                moments_add(M, O.bx[o + k], O.by[o + k], sx - start[0], sy - start[1]);
            }
            int it = newton_moments(cfg, P, M, start[0], start[1], start[2], tol, maxit, res);
            if (iters && writer) atomicAdd(iters, (unsigned long long)it);
        }
    }
    if (writer) { A.x[t] = res[0]; A.x[A.ldx + t] = res[1]; A.x[2 * A.ldx + t] = res[2]; }   // sensors.py:162
    if (WARPED) __syncwarp();      // (the next pose of the walk reads this one)
}

// red-black by trajectory-local time tl = t - k traj_T: parity 1 -> tl = 1,3,5,... ; parity 0 -> tl = 2,4,6,...  (so a
// trajectory of a batch is swept exactly as it is alone, whatever the parity of traj_T).  (traj_cols + 1) / 2 threads per
// trajectory.
__global__ void __launch_bounds__(128)
k_pose_colour(int parity, DevCfg cfg, PoseArrays A, ObsArrays O, SeenSrc S, int solver, double tol, int maxit,
              unsigned long long* iters)
{
    const int Tt = A.traj_cols(), per = (Tt + 1) / 2;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int k = idx / per, tl = 2 * (idx - k * per) + (parity ? 1 : 2);
    if (k >= A.T / Tt || tl >= Tt) return;
    update_pose(k * Tt + tl, cfg, A, O, S, solver, tol, maxit, iters);
}

// the reference's forward Gauss-Seidel (sensors.py:145): the warp of block k walks t = 1 .. traj_T-1 of trajectory k (one
// block of one warp per trajectory: trajectories take different Nelder-Mead branches).  Its lanes share each energy's
// observations (pose_energy<true>); everything else runs on every lane alike.
__global__ void __launch_bounds__(WARP)
k_pose_walk(DevCfg cfg, PoseArrays A, ObsArrays O, SeenSrc S, int solver, double tol, int maxit, unsigned long long* iters)
{
    const int Tt = A.traj_cols(), t0 = blockIdx.x * Tt;
    for (int t = t0 + 1; t < t0 + Tt; ++t) update_pose<true>(t, cfg, A, O, S, solver, tol, maxit, iters);
}
