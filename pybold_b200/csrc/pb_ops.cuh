// Stand-alone operator kernels (A1, A2, A4, A5, A9, A10 of SURVEY.md section 8): the pieces of
// pybold/linear.py, pybold/convolution.py, pybold/hrf_model.py and pybold/utils.py that the
// solvers fuse, exposed one by one so that the reference's `op` / `adj` protocol and its
// operator tests have a device counterpart.  One warp per voxel row, row staged in shared
// memory (coalesced load / store, HBM bound).
#pragma once
#include "pb_generic.cuh"

namespace pb {

enum OpKind { OP_INTEG = 0, OP_INTEG_ADJ, OP_CONV, OP_CONV_ADJ, OP_HRFINTEG, OP_HRFINTEG_ADJ };

// Row operators on a zero-framed shared-memory copy of the row, four samples per lane and step:
//   scans: in-vector prefix + 5-step shuffle scan of the vector totals + running carry;
//   K-tap convolution / correlation: each lane makes 4 outputs from 16-byte window loads
//   (16 FMA per load) instead of K scalar loads per output.
template <typename real>
struct alignas(4 * sizeof(real) > 16 ? 16 : 4 * sizeof(real)) RowVec4 { real t[4]; };

struct OpLayout {
    int pad;     // zero frame before and after the row, >= K + 3, multiple of 4
    int tp;      // row length rounded up to 128 (zero filled)
    int hp;      // padded tap buffer: 3 + K rounded + 8
    __host__ __device__ static OpLayout make(int T, int K) {
        OpLayout l;
        l.pad = (K + 3 + 3) & ~3;
        l.tp = (T + 127) & ~127;
        l.hp = ((K + 3) & ~3) + 12;
        return l;
    }
    __host__ __device__ int row() const { return 2 * pad + tp; }
    __host__ __device__ size_t warp_bytes(size_t rs) const { return ((size_t)2 * row() + hp) * rs; }
};

template <typename real>
__device__ __forceinline__ void row_scan_fwd(real *a, int tp, int lane) {   // a = first sample
    real carry = 0;
    for (int base = 0; base < tp; base += 128) {
        RowVec4<real> v = *reinterpret_cast<RowVec4<real> *>(a + base + 4 * lane);
        v.t[1] += v.t[0];
        v.t[2] += v.t[1];
        v.t[3] += v.t[2];
        real inc = v.t[3];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const real t = __shfl_up_sync(PB_FULL, inc, d);
            if (lane >= d) inc += t;
        }
        real ex = __shfl_up_sync(PB_FULL, inc, 1);
        ex = (lane == 0 ? real(0) : ex) + carry;
#pragma unroll
        for (int e = 0; e < 4; ++e) v.t[e] += ex;
        *reinterpret_cast<RowVec4<real> *>(a + base + 4 * lane) = v;
        carry += __shfl_sync(PB_FULL, inc, 31);
    }
    __syncwarp();
}

template <typename real>
__device__ __forceinline__ void row_scan_rev(real *a, int tp, int lane) {
    real carry = 0;
    for (int base = tp - 128; base >= 0; base -= 128) {
        RowVec4<real> v = *reinterpret_cast<RowVec4<real> *>(a + base + 4 * lane);
        v.t[2] += v.t[3];
        v.t[1] += v.t[2];
        v.t[0] += v.t[1];
        real inc = v.t[0];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const real t = __shfl_down_sync(PB_FULL, inc, d);
            if (lane + d < 32) inc += t;
        }
        real ex = __shfl_down_sync(PB_FULL, inc, 1);
        ex = (lane == 31 ? real(0) : ex) + carry;
#pragma unroll
        for (int e = 0; e < 4; ++e) v.t[e] += ex;
        *reinterpret_cast<RowVec4<real> *>(a + base + 4 * lane) = v;
        carry += __shfl_sync(PB_FULL, inc, 0);
    }
    __syncwarp();
}

// out[i] = sum_j h[j] in[i - j] (ADJ = false) or sum_j h[j] in[i + j] (ADJ = true); hp[3 + j] = h[j]
template <typename real, bool ADJ>
__device__ __forceinline__ void row_conv(const real *in, real *out, const real *hp, int tp, int K,
                                         int lane) {
    const int nc = (K + 3 + 3) / 4;
    for (int base = 0; base < tp; base += 128) {
        const int i0 = base + 4 * lane;
        real acc[4] = {0, 0, 0, 0};
        for (int c = 0; c < nc; ++c) {
            const RowVec4<real> xv = *reinterpret_cast<const RowVec4<real> *>(in + (ADJ ? i0 + 4 * c : i0 - 4 * c));
            const RowVec4<real> h0 = *reinterpret_cast<const RowVec4<real> *>(hp + 4 * c);
            const RowVec4<real> h1 = *reinterpret_cast<const RowVec4<real> *>(hp + 4 * c + 4);
            real hh[8];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                hh[e] = h0.t[e];
                hh[4 + e] = h1.t[e];
            }
#pragma unroll
            for (int e = 0; e < 4; ++e)
#pragma unroll
                for (int t = 0; t < 4; ++t) acc[e] = fma(hh[3 + (ADJ ? t - e : e - t)], xv.t[t], acc[e]);
        }
        RowVec4<real> o;
#pragma unroll
        for (int e = 0; e < 4; ++e) o.t[e] = acc[e];
        *reinterpret_cast<RowVec4<real> *>(out + i0) = o;
    }
    __syncwarp();
}

template <typename real, int OP>
__global__ void op_kernel(const real *h, int64_t h_stride, const real *x, real *out, int64_t V,
                          int T, int K, OpLayout lay) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    real *bufA = reinterpret_cast<real *>(smem + (size_t)warp * lay.warp_bytes(sizeof(real)));
    real *bufB = bufA + lay.row();
    real *hp = bufB + lay.row();
    real *A = bufA + lay.pad, *B = bufB + lay.pad;
    for (int i = lane; i < 2 * lay.row() + lay.hp; i += 32) bufA[i] = real(0);   // zero frames
    __syncwarp();
    for (int64_t v = (int64_t)blockIdx.x * nwarp + warp; v < V; v += (int64_t)gridDim.x * nwarp) {
        for (int i = lane; i < T; i += 32) A[i] = x[v * T + i];
        if (OP == OP_HRFINTEG)      // a previous scan left the running total in the zero fill
            for (int i = T + lane; i < lay.tp; i += 32) A[i] = real(0);
        if (OP >= OP_CONV && (h_stride != 0 || v == (int64_t)blockIdx.x * nwarp + warp))
            for (int a = lane; a < K; a += 32) hp[3 + a] = h[v * h_stride + a];
        __syncwarp();
        real *res = A;
        if (OP == OP_INTEG) {
            row_scan_fwd(A, lay.tp, lane);
        } else if (OP == OP_INTEG_ADJ) {
            row_scan_rev(A, lay.tp, lane);
        } else if (OP == OP_CONV) {
            row_conv<real, false>(A, B, hp, lay.tp, K, lane);
            res = B;
        } else if (OP == OP_CONV_ADJ) {
            row_conv<real, true>(A, B, hp, lay.tp, K, lane);
            res = B;
        } else if (OP == OP_HRFINTEG) {
            row_scan_fwd(A, lay.tp, lane);
            row_conv<real, false>(A, B, hp, lay.tp, K, lane);
            res = B;
        } else {
            row_conv<real, true>(A, B, hp, lay.tp, K, lane);
            row_scan_rev(B, lay.tp, lane);
            res = B;
        }
        for (int i = lane; i < T; i += 32) out[v * T + i] = res[i];
        if (OP == OP_INTEG || OP == OP_INTEG_ADJ)   // restore the zero fill beyond T for the next row
            for (int i = T + lane; i < lay.tp; i += 32) A[i] = real(0);
        __syncwarp();
    }
}

// spm_hrf (pybold/hrf_model.py:12-39): taps at the kept samples; the optional normalisation
// divides by max(hrf + 1e-30) over the reference's full 1 ms grid (N = int(dur / dt) points).
template <typename real>
__global__ void spm_hrf_kernel(const real *theta, HrfGrid grid, int n_fine, int normalized,
                               real *out_h, int64_t V) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    for (int64_t v = (int64_t)blockIdx.x * nwarp + warp; v < V; v += (int64_t)gridDim.x * nwarp) {
        const double th = (double)theta[v];
        double scale = 1.0;
        if (normalized) {
            double mx = -1.0e300;
            for (int n = lane; n < n_fine; n += 32)
                mx = fmax(mx, hrf_value(th, (double)n * grid.t_step) + 1.0e-30);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(PB_FULL, mx, o));
            scale = mx;
        }
        for (int a = lane; a < grid.K; a += 32) {
            double hh, h1, h2;
            hrf_tap(th, grid.t(a), hh, h1, h2);
            out_h[v * grid.K + a] = (real)(normalized ? hh / scale : hh);
        }
    }
}

// spm_hrf with arbitrary shape parameters (pybold/hrf_model.py:12-14, :25-31): the default-parameter
// kernel above uses integer powers; here g(s; a, loc) = exp((a - 1) log x - x - lgamma(a)), x = s - loc.
struct HrfShape {
    double dt, a_peak, loc_peak, a_under, loc_under, ratio, t_shift;   // t_shift = onset / dt (:25)
};

__device__ __forceinline__ double gamma_pdf_general(double s, double a, double loc, double lg) {
    const double x = s - loc;
    if (x > 0.0) return exp((a - 1.0) * log(x) - x - lg);
    if (x == 0.0) return a > 1.0 ? 0.0 : (a == 1.0 ? 1.0 : INFINITY);
    return x == x ? 0.0 : x;
}

template <typename real>
__global__ void spm_hrf_ex_kernel(const real *theta, HrfGrid grid, HrfShape sh, int n_fine, int normalized,
                                  real *out_h, int64_t V) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const double lg_p = lgamma(sh.a_peak), lg_u = lgamma(sh.a_under);
    auto value = [&](double th, double t) {
        const double s = th * (t - sh.t_shift);
        return gamma_pdf_general(s, sh.a_peak, sh.loc_peak, lg_p) -
               sh.ratio * gamma_pdf_general(s, sh.a_under, sh.loc_under, lg_u);
    };
    for (int64_t v = (int64_t)blockIdx.x * nwarp + warp; v < V; v += (int64_t)gridDim.x * nwarp) {
        const double th = (double)theta[v];
        double scale = 1.0;
        if (normalized) {                                   // max over the FINE grid, hrf_model.py:33-34
            double mx = -1.0e300;
            for (int n = lane; n < n_fine; n += 32) mx = fmax(mx, value(th, (double)n * grid.t_step) + 1.0e-30);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(PB_FULL, mx, o));
            scale = mx;
        }
        for (int a = lane; a < grid.K; a += 32) {
            const double hh = value(th, grid.t(a));
            out_h[v * grid.K + a] = (real)(normalized ? hh / scale : hh);
        }
    }
}

// spectral_radius_est (pybold/utils.py:94-109) with the start vector supplied.  CENSOR: the power iteration of the
// censored operator A^T M A (M applied between op and adj), the mask of voxel v at cz.row(v).
template <typename real, bool CENSOR = false>
__global__ void lipschitz_power_kernel(const real *h, int64_t h_stride, const real *x0,
                                       int64_t x0_stride, int nb_iter, double tol, real *out_L,
                                       int64_t V, int T, int K, GenLayout lay, Censor cz) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    double *scratch;
    GenVoxel<real> g = gen_bind<real>(smem + (size_t)warp * lay.warp_bytes(sizeof(real)), lay, T, K,
                                      lane, scratch);
    for (int64_t v = (int64_t)blockIdx.x * nwarp + warp; v < V; v += (int64_t)gridDim.x * nwarp) {
        for (int i = lane; i < T; i += 32) g.ws[i] = x0[v * x0_stride + i];
        for (int a = lane; a < K; a += 32) g.hr[a] = h[v * h_stride + a];
        __syncwarp();
        double n_old = sqrt(g.sumsq(g.ws));
        double n_new = n_old;
        for (int it = 0; it < nb_iter; ++it) {
            for (int i = lane; i < T; i += 32) g.as[i] = g.ws[i];
            __syncwarp();
            g.scan_fwd(g.as);
            g.conv(g.as, nullptr, g.bs);
            if constexpr (CENSOR) {
                const unsigned char *cm = cz.row(v);
                for (int i = lane; i < T; i += 32)
                    if (cm[i]) g.bs[i] = real(0);
                __syncwarp();
            }
            g.adjoint();
            const real inv = (real)(1.0 / n_old);
            for (int i = lane; i < T; i += 32) g.as[i] *= inv;
            __syncwarp();
            n_new = sqrt(g.sumsq(g.as));
            if (fabs(n_new - n_old) < tol) break;
            for (int i = lane; i < T; i += 32) g.ws[i] = g.as[i];
            __syncwarp();
            n_old = n_new;
        }
        if (lane == 0) out_L[v] = (real)n_new;
        __syncwarp();
    }
}

template <typename real>
__global__ void lipschitz_frob_kernel(const real *h, int64_t h_stride, real *out_L, int64_t V,
                                      int T, int K, int kp) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    ThetaScratch sc;
    double *base = reinterpret_cast<double *>(smem) + (size_t)warp * 3 * kp;
    sc.hs = base;
    sc.cs = base + kp;
    sc.Ss = base + 2 * kp;
    for (int64_t v = (int64_t)blockIdx.x * nwarp + warp; v < V; v += (int64_t)gridDim.x * nwarp) {
        for (int a = lane; a < K; a += 32) sc.hs[a] = (double)h[v * h_stride + a];
        __syncwarp();
        const double Lc = frob_lipschitz_warp(sc, K, T, lane);
        if (lane == 0) out_L[v] = (real)Lc;
        __syncwarp();
    }
}

// Layout adapter (row N4 of SURVEY.md 8(f)): the ingest side of the reference pipeline holds voxel
// matrices time-major, [T, V] (NiftiMasker.fit_transform, examples/icassp_2019/validation.py:90-103,
// consumed as `voxels.T`); the solvers want [V, T].  32 x 32 tiles through padded shared memory:
// coalesced 128-byte rows on both sides, HBM bound (2 x 4 bytes per sample).
template <typename real>
__global__ void __launch_bounds__(256) transpose_kernel(const real *__restrict__ in, real *out, int64_t rows,
                                                         int64_t cols) {
    // 64 x 64 tiles: 256-byte runs on both sides and 16 independent loads per thread in flight
    __shared__ real tile[64][65];
    const int64_t c0 = (int64_t)blockIdx.x * 64, r0 = (int64_t)blockIdx.y * 64;
    const int tx = threadIdx.x, ty = threadIdx.y;      // 32 x 8 threads
    real v[16];
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
            const int64_t r = r0 + ty + 8 * k, c = c0 + tx + 32 * hf;
            v[2 * k + hf] = (r < rows && c < cols) ? in[r * cols + c] : real(0);
        }
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) tile[ty + 8 * k][tx + 32 * hf] = v[2 * k + hf];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
            const int64_t c = c0 + ty + 8 * k, r = r0 + tx + 32 * hf;
            if (r < rows && c < cols) out[c * rows + r] = tile[tx + 32 * hf][ty + 8 * k];
        }
}

// Dense Toeplitz matrix of k.conv(.) (pybold/convolution.py:105-132): K[i, c] = k[i - c] for
// 0 <= i - c < len(k), else 0; [dim_out, dim_in] row-major.  The solvers never form it (SURVEY.md 7.2);
// it exists for callers of the reference's convolution module.  Write-only, HBM bound.
template <typename real>
__global__ void toeplitz_kernel(const real *__restrict__ k, int klen, real *out, int64_t dim_out, int64_t dim_in) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t i = blockIdx.y; i < dim_out; i += gridDim.y) {
        if (c < dim_in) {
            const int64_t d = i - c;
            out[i * dim_in + c] = (d >= 0 && d < klen) ? k[d] : real(0);
        }
    }
}

// hrf_estim / the theta step alone (pybold/bold_signal.py:217-239, :329-334)
template <typename real>
__global__ void hrf_estim_kernel(const real *z, const real *y, HrfGrid grid, const real *theta0,
                                 int64_t theta0_stride, double lo, double hi, real *out_theta,
                                 real *out_h, real *out_cost, int64_t V, int T, GenLayout lay) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const int K = grid.K;
    double *scratch;
    GenVoxel<real> g = gen_bind<real>(smem + (size_t)warp * lay.warp_bytes(sizeof(real)), lay, T, K,
                                      lane, scratch);
    ThetaScratch sc;
    sc.bind(scratch, lay.kp);
    for (int64_t v = (int64_t)blockIdx.x * nwarp + warp; v < V; v += (int64_t)gridDim.x * nwarp) {
        for (int i = lane; i < T; i += 32) {
            g.as[i] = z[v * T + i];
            g.ys[i] = y[v * T + i];
        }
        __syncwarp();
        g.theta_moments(sc);
        gram_build_warp(sc, K, lane);
        const double th = theta_solve_warp((double)theta0[v * theta0_stride], lo, hi, grid, sc,
                                           lane, nullptr);
        hrf_eval_warp(th, grid, sc, lane);
        g.load_taps(sc);
        g.conv(g.as, g.ys, g.bs);
        const double cost = 0.5 * g.sumsq(g.bs);
        for (int a = lane; a < K; a += 32) out_h[v * K + a] = (real)sc.hs[a];
        if (lane == 0) {
            out_theta[v] = (real)th;
            out_cost[v] = (real)cost;
        }
        __syncwarp();
    }
}

}  // namespace pb
