// common.cuh -- shared device helpers for libicmslam (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/icmslam.h"

#define ICM_PI 3.141592653589793   // np.pi
#define ICM_TWOPI (2.0 * ICM_PI)
#define ICM_HALFPI (ICM_PI / 2.0)

#define WARP 32
#define FULLMASK 0xffffffffu

// Device-side copy of the configuration, passed by value to kernels.
struct DevCfg {
    double dt, q1, q2, r1, r2, r3, kod, cota, dist_thr, rmax, radio;
    int L;
};

// Per-trajectory freezing of a batch handle (icmslam_batch_iterate_until).  frozen == nullptr on every other path, where every
// test below is one uniform branch.  Landmark ownership is stateless: region k = rint(y / pitch) * cols + rint(x / pitch).
#define FZ_SLOTS 5     // per-trajectory results of a sweep: min, max, sum of the resolved changes, new landmarks, unresolved ones
struct Freeze {
    const unsigned char* frozen;   // K bytes: trajectory k is frozen
    int traj_T;                    // columns per trajectory: scan t belongs to trajectory t / traj_T
    int K, cols;
    double pitch;
    double* slots;                 // FZ_SLOTS x K (row r, trajectory k): calc_cambio of each trajectory's landmarks
    __device__ __forceinline__ int region(double x, double y) const
    {
        const double k = rint(y / pitch) * (double)cols + rint(x / pitch);
        return (k >= 0.0 && k < (double)K) ? (int)k : -1;
    }
    __device__ __forceinline__ bool scan(int t) const { return frozen != nullptr && frozen[t / traj_T] != 0; }
    __device__ __forceinline__ bool landmark(double x, double y) const
    {
        if (frozen == nullptr) return false;
        const int k = region(x, y);
        return k >= 0 && frozen[k] != 0;
    }
    // (grid-stride over the trajectories by thread i of n)
    __device__ __forceinline__ void reset_slots(int i, int n) const
    {
        for (int k = i; k < K; k += n) {
            slots[k] = INFINITY;
            for (int r = 1; r < FZ_SLOTS; ++r) slots[(size_t)r * K + k] = 0.0;
        }
    }
};

// Which columns are pinned first poses (sensors.py:131: x[:,0] is never updated, scan 0 is projected with self.x0): column 0
// of the trajectory's first segment, or -- a batch of independent trajectories of traj_T columns each laid end to end in one
// handle (BASELINE configs[4]) -- the first column of every trajectory, each with its own x0.  A trajectory's last pose has no
// successor.  The fused solve and the generic kernels both go by these rules.
struct TrajLayout {
    int first;                 // column 0 is the trajectory's first pose
    int traj_T;                // > 0: batch of trajectories of this many columns
    const double* x0s;         // batch: 3 x K first poses (row-major, leading dimension ldx0s)
    int64_t ldx0s;
    double x0[3];              // single trajectory: self.x0
    __device__ __forceinline__ bool pinned(int t) const { return traj_T > 0 ? (t % traj_T) == 0 : (t == 0 && first); }
    __device__ __forceinline__ bool after_pinned(int t) const { return traj_T > 0 ? (t % traj_T) == 1 : (t == 1 && first); }
    __device__ __forceinline__ bool has_next(int t, int T) const { return t + 1 < T && (traj_T == 0 || ((t + 1) % traj_T) != 0); }
    __device__ __forceinline__ double x0_of(int t, int r) const { return traj_T > 0 ? x0s[r * ldx0s + t / traj_T] : x0[r]; }
    // the pose scan t is projected with (sensors.py:141,153): its trajectory's x0 for a pinned column, else x[:, t]
    __device__ __forceinline__ void scan_pose(const double* x, int64_t ldx, int t, double& px, double& py, double& th) const
    {
        if (pinned(t)) { px = x0_of(t, 0); py = x0_of(t, 1); th = x0_of(t, 2); }
        else { px = x[t]; py = x[ldx + t]; th = x[2 * ldx + t]; }
    }
};

// Status word written by kernels (checked by the host after the sweep).
enum { ST_OK = 0, ST_LABEL_CAP = 1, /* 4: empty map */ ST_P2P_TIMEOUT = 8 };

// ---- exact (non-contracted) arithmetic: nvcc fuses a*b+c into DFMA by default; where a result
// must be bit-identical to numpy/scipy we spell out the roundings.
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dadd_rn(a, -b); }

// Euclidean distance exactly as scipy cdist/pdist: sqrt(dx*dx + dy*dy), each op rounded.
__device__ __forceinline__ double dist2_rn(double dx, double dy) { return add_rn(mul_rn(dx, dx), mul_rn(dy, dy)); }
__device__ __forceinline__ double dist_rn(double dx, double dy) { return __dsqrt_rn(dist2_rn(dx, dy)); }

// entrepi (ICM_SLAM.py:455-463): np.mod(a, 2*pi) (result in [0, 2*pi)), then -2*pi if > pi.
__device__ __forceinline__ double entrepi(double a)
{
    double m = fmod(a, ICM_TWOPI);
    if (m < 0.0) m += ICM_TWOPI;
    if (m > ICM_PI) m -= ICM_TWOPI;
    return m;
}

// tras_rot_z (ICM_SLAM.py:465-480).  numpy's matmul accumulates acc = a0*b0; acc = fma(a1,b1,acc)
// (verified bit-for-bit against the reference on the build host, tests/golden/units.npz).
struct Rot { double ct, st; };   // cos/sin of (theta - pi/2)
__device__ __forceinline__ Rot make_rot(double theta)
{
    Rot r;
    sincos(sub_rn(theta, ICM_HALFPI), &r.st, &r.ct);
    return r;
}
__device__ __forceinline__ void project(const Rot& r, double px, double py, double bx, double by, double& wx, double& wy)
{
    wx = add_rn(__fma_rn(by, -r.st, mul_rn(bx, r.ct)), px);
    wy = add_rn(__fma_rn(by, r.ct, mul_rn(bx, r.st)), py);
}

// Projection parameters of a pose: (x, y, sin(theta - pi/2), cos(theta - pi/2)) exactly as tras_rot_z forms them
// (ICM_SLAM.py:466-468; the subtraction rounded once, then libm-accurate sin/cos).  The sin/cos of the heading itself are
// (cos(theta - pi/2), -sin(theta - pi/2)).  One record per pose, rewritten by the solve for the poses it moves.
__device__ __forceinline__ double4 make_ppar(double x, double y, double th)
{
    double st, ct;
    sincos(sub_rn(th, ICM_HALFPI), &st, &ct);
    return make_double4(x, y, st, ct);
}

__device__ __forceinline__ double4 ldg_ppar(const double4* p)
{
    const double2 a = __ldg(reinterpret_cast<const double2*>(p)), b = __ldg(reinterpret_cast<const double2*>(p) + 1);
    return make_double4(a.x, a.y, b.x, b.y);
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULLMASK, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum_i(int v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULLMASK, v, o);
    return v;
}
__device__ __forceinline__ double warp_min(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULLMASK, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULLMASK, v, o));
    return v;
}

__device__ __forceinline__ void atomic_max_pos(double* addr, double v)   // v >= 0
{
    atomicMax((unsigned long long*)addr, (unsigned long long)__double_as_longlong(v));
}
__device__ __forceinline__ void atomic_min_pos(double* addr, double v)   // v >= 0
{
    atomicMin((unsigned long long*)addr, (unsigned long long)__double_as_longlong(v));
}
