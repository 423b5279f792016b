// Noise level of a voxel as `deconv(lbda=None)` takes it (pybold/bold_signal.py:103):
//   sigma = mad(cD),  cD = level-1 db3 detail coefficients of y     (pybold/utils.py:16-25)
//   mad(x) = median(|x - median(x)|) / c                            (pybold/utils.py:10-13)
// One warp per voxel: the detail coefficients (doubles, whatever the storage type) live in shared
// memory, both medians are EXACT order statistics found by a bitwise radix selection on the ordered
// integer image of the doubles (64 counting passes per order statistic, no sort), so that the result
// equals NumPy's median to the last bit for a given cD.
//
// db3 analysis high-pass and PyWavelets' "symmetric" (half-sample) extension:
//   cD[o] = sum_j dec_hi[j] x_ext[2 o + 1 - j],  o < floor((T + 5) / 2),
//   x_ext[i] = x[-i - 1] (i < 0),  x[2 T - 1 - i] (i >= T).
// Series shorter than 10 scans have no level-1 decomposition (dwt_max_level = 0): the reference's
// `except ValueError` branch then takes `wavedec(level=0)`, i.e. the series itself.
#pragma once
#include <cstdint>
#include <math_constants.h>

#include "pb_device.cuh"
#include "pb_generic.cuh"

namespace pb {

__device__ __constant__ double kDb3DecHi[6] = {-0.3326705529509569, 0.8068915093133388,
                                               -0.4598775021193313, -0.13501102001039084,
                                               0.08544127388224149, 0.035226291882100656};

__host__ __device__ inline int noise_detail_len(int T) { return T < 10 ? T : (T + 5) / 2; }

// order-preserving map double -> uint64 (negative values flipped entirely, positive get the sign bit)
__device__ __forceinline__ unsigned long long ordered_key(double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_value(unsigned long long k) {
    const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

// k-th smallest (0-based) of d[0..n) -- every lane returns it
__device__ inline double warp_select(const double *d, int n, int k, int lane) {
    unsigned long long prefix = 0, mask = 0;
    for (int bit = 63; bit >= 0; --bit) {
        const unsigned long long b = 1ull << bit;
        int c = 0;
        for (int i = lane; i < n; i += 32) {
            const unsigned long long key = ordered_key(d[i]);
            c += ((key & mask) == prefix) && !(key & b);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(PB_FULL, c, o);
        if (k >= c) {
            k -= c;
            prefix |= b;
        }
        mask |= b;
    }
    return key_value(prefix);
}

// NumPy's median of a row holding a NaN is NaN, whatever the NaN's sign bit; ordered_key would rank it past +-inf
// instead, so the kernels test for one before they select
__device__ inline bool warp_any_nan(const double *d, int n, int lane) {
    bool nan = false;
    for (int i = lane; i < n; i += 32) nan = nan || isnan(d[i]);
    return __any_sync(PB_FULL, nan);
}

// NumPy's median: the middle order statistic, or the mean of the two middle ones
__device__ inline double warp_median(const double *d, int n, int lane) {
    const double lo = warp_select(d, n, (n - 1) / 2, lane);
    if (n & 1) return lo;
    const double hi = warp_select(d, n, n / 2, lane);
    return 0.5 * (lo + hi);
}

// MODE 0: mad of the rows of x[V, n].  MODE 1: mad of the db3 detail coefficients of y[V, T].
// Non-finite values: a row holding a NaN gives NaN.  So does a row whose median is +-inf: that median is one of the
// row's values, and its deviation inf - inf is NaN in NumPy too.  Otherwise every deviation is finite or +inf and
// both selections are exact.
template <typename real, int MODE>
__global__ void mad_rows_kernel(const real *x, double c, real *out, int64_t V, int T, int nmax) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    double *d = reinterpret_cast<double *>(smem) + (size_t)warp * nmax;
    const int n = MODE == 1 ? noise_detail_len(T) : T;
    for (int64_t v = (int64_t)blockIdx.x * nwarp + warp; v < V; v += (int64_t)gridDim.x * nwarp) {
        const real *row = x + v * T;
        if (MODE == 1 && T >= 10) {
            for (int o = lane; o < n; o += 32) {
                double acc = 0.0;
#pragma unroll
                for (int j = 0; j < 6; ++j) {
                    int i = 2 * o + 1 - j;
                    i = i < 0 ? -i - 1 : (i >= T ? 2 * T - 1 - i : i);
                    acc += kDb3DecHi[j] * (double)row[i];
                }
                d[o] = acc;
            }
        } else {
            for (int i = lane; i < n; i += 32) d[i] = (double)row[i];
        }
        __syncwarp();
        const double med = warp_any_nan(d, n, lane) ? CUDART_NAN : warp_median(d, n, lane);
        __syncwarp();
        if (!isfinite(med)) {
            if (lane == 0) out[v] = (real)CUDART_NAN;
            continue;
        }
        for (int i = lane; i < n; i += 32) d[i] = fabs(d[i] - med);
        __syncwarp();
        const double dev = warp_median(d, n, lane);
        if (lane == 0) out[v] = (real)(dev / c);
        __syncwarp();
    }
}

// pb_mad_daub_noise_est_censored: the db3 MAD over the level-1 detail coefficients that touch no censored scan (a
// coefficient reads six samples, after the symmetric extension; T < 10 takes the kept samples themselves).  The left-out
// coefficients are parked at +inf, above every kept one, so both medians are order statistics among the first n_kept.
// A voxel with no coefficient left gets NaN, and so does one with a NaN or an infinite median among its kept
// coefficients (as in mad_rows_kernel); a NaN at a censored scan reaches left-out coefficients only.
template <typename real>
__global__ void mad_daub_censored_kernel(const real *x, double c, real *out, int64_t V, int T, int nmax, Censor cz) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    double *d = reinterpret_cast<double *>(smem) + (size_t)warp * nmax;
    const int n = noise_detail_len(T);
    auto median_of_kept = [&](int nk) {
        const double lo = warp_select(d, n, (nk - 1) / 2, lane);
        return (nk & 1) ? lo : 0.5 * (lo + warp_select(d, n, nk / 2, lane));
    };
    for (int64_t v = (int64_t)blockIdx.x * nwarp + warp; v < V; v += (int64_t)gridDim.x * nwarp) {
        const real *row = x + v * T;
        const unsigned char *cm = cz.row(v);
        int nk = 0;
        for (int o = lane; o < n; o += 32) {
            double acc = 0.0;
            bool kept = true;
            if (T >= 10) {
#pragma unroll
                for (int j = 0; j < 6; ++j) {
                    int i = 2 * o + 1 - j;
                    i = i < 0 ? -i - 1 : (i >= T ? 2 * T - 1 - i : i);
                    kept = kept && cm[i] == 0;
                    acc += kDb3DecHi[j] * (double)row[i];
                }
            } else {
                kept = cm[o] == 0;
                acc = (double)row[o];
            }
            d[o] = kept ? acc : CUDART_INF;
            nk += kept;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) nk += __shfl_xor_sync(PB_FULL, nk, o);
        __syncwarp();
        const double med = nk == 0 || warp_any_nan(d, n, lane) ? CUDART_NAN : median_of_kept(nk);
        __syncwarp();
        if (!isfinite(med)) {
            if (lane == 0) out[v] = (real)CUDART_NAN;
            continue;
        }
        // a finite median: a kept +inf and a parked coefficient both deviate by +inf
        for (int i = lane; i < n; i += 32) d[i] = d[i] == CUDART_INF ? d[i] : fabs(d[i] - med);
        __syncwarp();
        const double dev = median_of_kept(nk);
        if (lane == 0) out[v] = (real)(dev / c);
        __syncwarp();
    }
}

// deconv(lbda=None) for a voxel whose noise level is NaN (a NaN among its kept samples, or a NaN sigma from the
// caller).  In the reference alpha and lambda turn NaN after the first pass, and its soft threshold then makes every
// later iterate NaN; the kernels' clamp fmin(fmax(u, -th), th) passes u through on a NaN th and would leave a finite,
// meaningless fit.  Launched after the solve on the same stream, this gives such a voxel the reference's outputs:
// x, z, diff_z NaN, and R, G NaN from the second outer iteration on.  J and lambda are NaN already, and the outer
// count is nb_outer, because the window test never passes on a NaN alpha.  Other voxels are not touched.
template <typename real>
__global__ void nan_sigma_rows_kernel(DeconvArgs<real> a) {
    const real nan = (real)CUDART_NAN;
    for (int64_t v = blockIdx.x; v < a.V; v += gridDim.x) {
        if (!isnan((double)a.sigma[a.voxel_of(v) * a.sigma_stride])) continue;
        for (int t = threadIdx.x; t < a.T; t += blockDim.x) {
            a.out_x[v * a.T + t] = nan;
            a.out_z[v * a.T + t] = nan;
            a.out_dz[v * a.T + t] = nan;
        }
        for (int j = 1 + threadIdx.x; j < a.nb_outer; j += blockDim.x) {
            if (a.out_R) a.out_R[v * a.nb_outer + j] = nan;
            if (a.out_G) a.out_G[v * a.nb_outer + j] = nan;
        }
    }
}

}  // namespace pb
