// extract.cuh -- scan extraction kernels: filtrar_z (ICM_SLAM.py:22-58) for all T scans at once,
// range pre-conditioning (sensors_definitions.py:21-22) and filtrar_obs.m (scripts/filtrar_obs.m).
//
// Layout: `scans` is the reference's B x T array (row = beam, column = scan), so one scan is a
// strided column.  Every scan is filtered on its own, so the kernels take a window [t_lo, t_hi) of columns: the whole log, or
// the columns an append brought (the CSR offsets of the window continue those before it).  `masks` and `counts` are indexed
// from t_lo; `off`, `scan_of` and the observation arrays are global.  A block stages a [B][32 scans] tile through shared memory with coalesced row
// reads (32 consecutive scans = 256 B per beam row), then each warp owns whole scans.
#pragma once
#include "common.cuh"

#define EX_TILE 32      // scans per block
#define EX_WARPS 8
#define EX_THREADS (EX_WARPS * WARP)

__device__ __forceinline__ double precond(double z, double radio, double rmax)
{
    if (isnan(z)) z = rmax;                 // sensors_definitions.py:21
    z = z + radio;                          // :22
    return z < rmax ? z : rmax;             // np.minimum
}

__device__ __forceinline__ double median3(double a, double b, double c)
{
    double lo = fmin(a, b), hi = fmax(a, b);
    return c < lo ? lo : (c > hi ? hi : c);
}

// smem layout: tile[B][EX_TILE+1] | per warp: vpx[B], vpy[B], vb[B](int)
template <int PASS>
__global__ void __launch_bounds__(EX_THREADS)
k_extract(const double* __restrict__ scans, int B, int t_lo, int T, int64_t ld, const double* __restrict__ cosb,
          const double* __restrict__ sinb, DevCfg cfg, int precondition, int nwords,
          uint32_t* __restrict__ masks,      // (T - t_lo) * nwords keep bitmasks
          int* __restrict__ counts,          // PASS 1: kept beams per scan of the window
          const int* __restrict__ off,       // PASS 2: CSR offsets
          int* __restrict__ beam, double* __restrict__ d, double* __restrict__ bx, double* __restrict__ by,
          int* __restrict__ scan_of)
{
    extern __shared__ double smem[];
    double* tile = smem;                                   // B * (EX_TILE+1)
    const int TP = EX_TILE + 1;
    const int warp = threadIdx.x / WARP, lane = threadIdx.x % WARP;
    double* vpx = tile + (size_t)B * TP + (size_t)warp * 3 * B;
    double* vpy = vpx + B;
    int* vb = (int*)(vpy + B);
    const int t0 = t_lo + blockIdx.x * EX_TILE;
    // coalesced tile load: thread -> (beam row, scan column)
    for (int e = threadIdx.x; e < B * EX_TILE; e += EX_THREADS) {
        int b = e / EX_TILE, c = e % EX_TILE;
        double z = 0.0;
        if (t0 + c < T) {
            z = scans[(int64_t)b * ld + t0 + c];
            if (precondition) z = precond(z, cfg.radio, cfg.rmax);
        }
        tile[b * TP + c] = z;
    }
    __syncthreads();
    for (int c = warp; c < EX_TILE; c += EX_WARPS) {
        const int t = t0 + c;
        if (t >= T) break;
        if (PASS == 1) {
            // median filter (kernel 3, zero padded) + range gate, compact valid points
            int k = 0;
            for (int b0 = 0; b0 < B; b0 += WARP) {
                int b = b0 + lane;
                bool valid = false;
                double zf = 0.0;
                if (b < B) {
                    double a = b > 0 ? tile[(b - 1) * TP + c] : 0.0;
                    double m = tile[b * TP + c];
                    double n = b + 1 < B ? tile[(b + 1) * TP + c] : 0.0;
                    zf = median3(a, m, n);
                    valid = zf < cfg.rmax;                      // ICM_SLAM.py:41
                }
                unsigned bal = __ballot_sync(FULLMASK, valid);
                if (valid) {
                    int p = k + __popc(bal & ((1u << lane) - 1));
                    vpx[p] = mul_rn(__ldg(cosb + b), zf);       // :44-45
                    vpy[p] = mul_rn(__ldg(sinb + b), zf);
                    vb[p] = b;
                }
                k += __popc(bal);
            }
            __syncwarp();
            // zero the mask words of this scan
            for (int w = lane; w < nwords; w += WARP) masks[(int64_t)(t - t_lo) * nwords + w] = 0u;
            __syncwarp();
            int kept = 0;
            if (k > 1) {                                          // :42
                for (int j0 = 0; j0 < k; j0 += WARP) {
                    int j = j0 + lane;
                    bool keep = false;
                    if (j < k) {
                        double xj = vpx[j], yj = vpy[j];
                        double m2 = INFINITY;                   // min non-zero squared distance
                        for (int i = 0; i < k; ++i) {
                            double s = dist2_rn(vpx[i] - xj, vpy[i] - yj);
                            if (s != 0.0 && s < m2) m2 = s;    // zeros (diagonal, coincident) -> 100 (:48)
                        }
                        // sqrt is monotone and correctly rounded: min_i sqrt(s_i) == sqrt(min_i s_i)
                        double m = fmin(100.0, __dsqrt_rn(m2));
                        keep = m <= cfg.dist_thr;               // :50
                        if (keep) atomicOr(&masks[(int64_t)(t - t_lo) * nwords + (vb[j] >> 5)], 1u << (vb[j] & 31));
                    }
                    kept += __popc(__ballot_sync(FULLMASK, keep));
                }
            }
            if (lane == 0) counts[t - t_lo] = kept;
            __syncwarp();
        } else {
            int base = off[t];
            if (off[t + 1] == base) continue;
            for (int b0 = 0; b0 < B; b0 += WARP) {
                int b = b0 + lane;
                uint32_t word = masks[(int64_t)(t - t_lo) * nwords + (b0 >> 5)];
                bool keep = (b < B) && ((word >> lane) & 1u);
                if (keep) {
                    double a = b > 0 ? tile[(b - 1) * TP + c] : 0.0;
                    double m = tile[b * TP + c];
                    double n = b + 1 < B ? tile[(b + 1) * TP + c] : 0.0;
                    double zf = median3(a, m, n);
                    int p = base + __popc(word & ((1u << lane) - 1));
                    beam[p] = b;
                    d[p] = zf;                                  // :51 (median-filtered range)
                    bx[p] = mul_rn(zf, __ldg(cosb + b));        // :52-53
                    by[p] = mul_rn(zf, __ldg(sinb + b));
                    scan_of[p] = t;
                }
                base += __popc(word);
            }
        }
    }
}

static size_t extract_smem_bytes(int B) { return ((size_t)B * (EX_TILE + 1) + (size_t)EX_WARPS * 3 * B) * sizeof(double); }

// ---- filtrar_obs.m -------------------------------------------------------------------------
// pass A: a(t) = number of beams with range <= max_dist (scripts/filtrar_obs.m:8-17).
__global__ void k_fo_count(const double* __restrict__ obs, int B, int T, int64_t ld, double max_dist, int* __restrict__ a)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    int k = 0;
    for (int b = 0; b < B; ++b) {
        double v = obs[(int64_t)b * ld + t];      // coalesced across t
        k += (!(v > max_dist) && !isnan(v)) ? 1 : 0;
    }
    a[t] = k;
}

// pass B: counts above cant_max are replaced by the linear interpolation between the nearest
// kept neighbours (:23-27, a = fix(interp1(tt, a, t))); the sentinel a(T+1) = cant_max closes the
// right end.  Noisy runs are short, so each affected thread simply walks to its two knots.
__global__ void k_fo_interp(const int* __restrict__ a, int T, int cant_max, int* __restrict__ keep, int* __restrict__ err)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    int v = a[t];
    if (v > cant_max) {
        int p = t - 1, n = t + 1;
        while (p >= 0 && a[p] > cant_max) --p;
        while (n < T && a[n] > cant_max) ++n;       // n == T is the sentinel
        if (p < 0) { atomicExch(err, 1); keep[t] = 0; return; }   // interp1 gives NaN before the first knot
        double ap = (double)a[p], an = n >= T ? (double)cant_max : (double)a[n];
        double slope = __ddiv_rn(an - ap, (double)(n - p));
        double val = add_rn(mul_rn(slope, (double)(t - p)), ap);
        v = (int)trunc(val);
    }
    keep[t] = v;
}

// pass C: per scan keep the keep[t] smallest valid ranges (stable: ties -> lower beam), others and
// invalid -> max_dist (:33-50).  One warp per scan; rank by counting; coalesced tile in / out.
__global__ void k_fo_select(const double* __restrict__ obs, int B, int T, int64_t ld, double max_dist,
                            const int* __restrict__ keep, double* __restrict__ out, int64_t ldo)
{
    extern __shared__ double smem[];
    const int TP = EX_TILE + 1;
    double* tile = smem;
    double* res = smem + (size_t)B * TP;
    const int warp = threadIdx.x / WARP, lane = threadIdx.x % WARP;
    const int t0 = blockIdx.x * EX_TILE;
    for (int e = threadIdx.x; e < B * EX_TILE; e += blockDim.x) {
        int b = e / EX_TILE, c = e % EX_TILE;
        tile[b * TP + c] = (t0 + c < T) ? obs[(int64_t)b * ld + t0 + c] : max_dist;
    }
    __syncthreads();
    for (int c = warp; c < EX_TILE; c += blockDim.x / WARP) {
        int t = t0 + c;
        if (t >= T) break;
        int kk = keep[t];
        for (int b = lane; b < B; b += WARP) {
            double v = tile[b * TP + c];
            bool valid = !(v > max_dist) && !isnan(v);
            int rank = 0;
            if (valid)
                for (int i = 0; i < B; ++i) {
                    double w = tile[i * TP + c];
                    bool wv = !(w > max_dist) && !isnan(w);
                    rank += (wv && (w < v || (w == v && i < b))) ? 1 : 0;
                }
            res[b * TP + c] = (valid && rank < kk) ? v : max_dist;
        }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < B * EX_TILE; e += blockDim.x) {
        int b = e / EX_TILE, c = e % EX_TILE;
        if (t0 + c < T) out[(int64_t)b * ldo + t0 + c] = res[b * TP + c];
    }
}
