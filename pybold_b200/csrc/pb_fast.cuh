// Register-tiled persistent solver kernels: ONE WARP PER VOXEL, the whole voxel on chip.
//
// Layout: lane q owns the R contiguous samples [q R, q R + R) of the voxel's time series in
// registers (32 R >= T).  Per prox-gradient iteration (SURVEY.md A3/A6, the recursion the
// reference actually executes, Q1):
//
//   v   = h * w                  K-tap causal convolution, R x KMAX FFMA per lane; the K-1
//                                samples owned by lower lanes arrive by warp shuffles
//   res = cumsum(v - dy)         = A w - y   (dy = first difference of y, so that the scan that
//                                integrates v also restores y: one add per sample saved);
//                                in-lane prefix + 5-step shuffle scan of the lane totals
//   c   = h^T res                anti-causal correlation, halo from higher lanes by shuffles
//   g   = reversed cumsum(c)     = A^T (A w - y)
//   u   = w - g / L;  cl = clamp(u, -lbda/L, lbda/L);  w <- u - (1 + beta_k) cl
//                                (== v + beta_k (v - u) with v = soft(u): the aliased recursion)
//
// HBM is touched only to load y and to store x, z, diff_z, h and the cost traces.  No tensor
// cores: the operator is a banded Toeplitz contraction with K <= 32 taps (FP32/FP64 FMA pipe).
//
// CIRC variant (T % R == 0 and at least ceil((KMAX-1)/R) idle lanes at the top of the warp):
// the idle lanes hold zeros and zero taps, so the shuffles may wrap around (lane 0 reads lane 31)
// and neither the halo nor the tail of the series needs a select: zero masking cost.
//
// Reference code replaced: pybold/bold_signal.py:49-97, :242-278, :281-382.
#pragma once
#include "pb_fast_registry.h"
#include "pb_generic.cuh"

#include "pb_tile.cuh"

// source order of the unrolled tile (pb_tile.cuh), picked with the register-file model on
// fast_deconv_kernel<float, 20, 20, circ> (cfg5: 1918 -> 1831 modelled cycles per iteration)
#ifndef PB_W_CONV_JDESC
#define PB_W_CONV_JDESC 1
#endif
#ifndef PB_W_CONV_RDESC
#define PB_W_CONV_RDESC 0
#endif
#ifndef PB_W_CONV_RB
#define PB_W_CONV_RB 10
#endif
#ifndef PB_W_CONV_DS
#define PB_W_CONV_DS 0
#endif
#ifndef PB_W_CORR_JDESC
#define PB_W_CORR_JDESC 1
#endif
#ifndef PB_W_CORR_RDESC
#define PB_W_CORR_RDESC 1
#endif
#ifndef PB_W_CORR_RB
#define PB_W_CORR_RB 10
#endif
#ifndef PB_W_CORR_DS
#define PB_W_CORR_DS 0
#endif

namespace pb {

template <int R, int KMAX>
__host__ __device__ constexpr int halo_lanes() { return (KMAX - 1 + R - 1) / R; }

template <typename real, int R, int KMAX, bool CIRC>
struct WarpVoxel {
    real w[R];      // iterate (the reference's diff_z)
    real dy[R];     // y[i] - y[i-1]
    real h[KMAX];   // taps, zero beyond K and on lanes that hold no sample
    real lanemask;  // CIRC: 1 on lanes that hold samples, else 0
    int nvalid;     // number of samples (< T) this lane holds, 0..R
    int lane;
    int srcu[halo_lanes<R, KMAX>() + 1];  // CIRC: (lane - d) & 31
    int srcd[halo_lanes<R, KMAX>() + 1];  // CIRC: (lane + d) & 31

    __device__ __forceinline__ void init(int lane_, int T) {
        lane = lane_;
        nvalid = max(0, min(R, T - lane * R));
        lanemask = nvalid > 0 ? real(1) : real(0);
#pragma unroll
        for (int d = 0; d <= halo_lanes<R, KMAX>(); ++d) {
            srcu[d] = (lane - d) & 31;
            srcd[d] = (lane + d) & 31;
        }
    }

    // halo[m-1] = a at voxel index (lane R - m), m = 1..KMAX-1 (zero before the series starts)
    template <bool WRAP>
    __device__ __forceinline__ void halo_up(const real (&a)[R], real (&halo)[KMAX - 1]) const {
#pragma unroll
        for (int m = 1; m < KMAX; ++m) {
            const int d = (m + R - 1) / R;
            const int rr = d * R - m;
            if (WRAP) {
                halo[m - 1] = __shfl_sync(PB_FULL, a[rr], srcu[d]);
            } else {
                const real t = __shfl_up_sync(PB_FULL, a[rr], d);
                halo[m - 1] = lane >= d ? t : real(0);
            }
        }
    }
    // halo[k] = a at voxel index (lane R + R + k), k = 0..KMAX-2 (zero past the last lane)
    template <bool WRAP>
    __device__ __forceinline__ void halo_down(const real (&a)[R], real (&halo)[KMAX - 1]) const {
#pragma unroll
        for (int k = 0; k < KMAX - 1; ++k) {
            const int d = (R + k) / R;
            const int rr = (R + k) - d * R;
            if (WRAP) {
                halo[k] = __shfl_sync(PB_FULL, a[rr], srcd[d]);
            } else {
                const real t = __shfl_down_sync(PB_FULL, a[rr], d);
                halo[k] = lane + d < 32 ? t : real(0);
            }
        }
    }
    // acc[r] += sum_j h[j] a(i - j)
    __device__ __forceinline__ void conv_acc(const real (&a)[R], const real (&halo)[KMAX - 1],
                                             real (&acc)[R]) const {
        tile_conv<real, R, KMAX, KMAX - 1, 0, PB_W_CONV_JDESC, PB_W_CONV_RDESC, PB_W_CONV_RB, PB_W_CONV_DS>(h, a, halo, acc);
    }
    // acc[r] += sum_j h[j] a(i + j)
    __device__ __forceinline__ void corr_acc(const real (&a)[R], const real (&halo)[KMAX - 1],
                                             real (&acc)[R]) const {
        tile_corr<real, R, KMAX, KMAX - 1, 0, PB_W_CORR_JDESC, PB_W_CORR_RDESC, PB_W_CORR_RB, PB_W_CORR_DS>(h, a, halo, acc);
    }
    // in-place inclusive prefix sum over the whole voxel
    __device__ __forceinline__ void scan_fwd(real (&a)[R]) const {
#pragma unroll
        for (int r = 1; r < R; ++r) a[r] += a[r - 1];
        const real carry = warp_excl_scan_up(a[R - 1], lane);
#pragma unroll
        for (int r = 0; r < R; ++r) a[r] += carry;
    }

    // res <- A w - y  (zero at and beyond T)
    __device__ __forceinline__ void forward(real (&res)[R]) const {
        real halo[KMAX - 1];
        halo_up<CIRC>(w, halo);
#pragma unroll
        for (int r = 0; r < R; ++r) res[r] = -dy[r];
        conv_acc(w, halo, res);
#pragma unroll
        for (int r = 1; r < R; ++r) res[r] += res[r - 1];
        const real carry = warp_excl_scan_up(res[R - 1], lane);
        if (CIRC) {
            const real cm = carry * lanemask;
#pragma unroll
            for (int r = 0; r < R; ++r) res[r] = fma(res[r], lanemask, cm);
        } else {
#pragma unroll
            for (int r = 0; r < R; ++r) res[r] = r < nvalid ? res[r] + carry : real(0);
        }
    }
    // g <- A^T res
    __device__ __forceinline__ void adjoint(const real (&res)[R], real (&g)[R]) const {
        real halo[KMAX - 1];
        halo_down<CIRC>(res, halo);
#pragma unroll
        for (int r = 0; r < R; ++r) g[r] = real(0);
        corr_acc(res, halo, g);
#pragma unroll
        for (int r = R - 2; r >= 0; --r) g[r] += g[r + 1];
        const real carry = warp_excl_scan_down(g[0], lane);
#pragma unroll
        for (int r = 0; r < R; ++r) g[r] += carry;
    }
    // u = w - step g; cl = clamp(u); w <- u - (1 + beta) cl.  Optionally keeps u and the
    // early-stop norms sum cl^2, sum w^2 (per-lane partials).
    template <bool KEEP_U, bool NORMS>
    __device__ __forceinline__ void update(const real (&g)[R], real step, real th, real beta,
                                           real (&u_out)[R], real &pc, real &pw) {
        const real ob = real(1) + beta;
        real lc = 0, lw = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const real u = fma(-step, g[r], w[r]);
            const real cl = fmin(fmax(u, -th), th);
            const real wn = fma(-ob, cl, u);
            w[r] = wn;
            if (KEEP_U) u_out[r] = u;
            if (NORMS) {
                lc = fma(cl, cl, lc);
                lw = fma(wn, wn, lw);
            }
        }
        pc = lc;
        pw = lw;
    }
    __device__ __forceinline__ real partial_sumsq(const real (&a)[R]) const {
        real s = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) s = fma(a[r], a[r], s);
        return s;
    }
    __device__ __forceinline__ real partial_sumabs(const real (&a)[R]) const {
        real s = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) s += fabs(a[r]);
        return s;
    }
    // taps from the double scratch (zero on idle lanes so that they produce exact zeros)
    __device__ __forceinline__ void load_taps(const double *hs, int K) {
#pragma unroll
        for (int j = 0; j < KMAX; ++j) h[j] = (j < K && nvalid > 0) ? (real)hs[j] : real(0);
    }
    // y (zero beyond T) and its first difference
    __device__ __forceinline__ void load_y(const real *yv, int T, real (&y)[R]) const {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = lane * R + r;
            y[r] = i < T ? yv[i] : real(0);
        }
    }
    __device__ __forceinline__ void set_dy(const real *yv, int T) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = lane * R + r;
            const real cur = i < T ? yv[i] : real(0);
            const real prv = (i > 0 && i - 1 < T) ? yv[i - 1] : real(0);
            dy[r] = i < T ? cur - prv : real(0);
        }
    }
    __device__ __forceinline__ void store(real *dst, const real (&a)[R], int T) const {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = lane * R + r;
            if (i < T) dst[i] = a[r];
        }
    }
    // inner loop of bd (_loops_deconv, pybold/bold_signal.py:259-276)
    __device__ __forceinline__ void inner_loop(const real *beta, int nb_iter, real step, real th,
                                               bool es, double tol) {
        real dummy[R];
        for (int j = 0; j < nb_iter; ++j) {
            real res[R], g[R];
            forward(res);
            adjoint(res, g);
            real pc, pw;
            if (es && j > 2) {
                update<false, true>(g, step, th, beta[j], dummy, pc, pw);
                const double sc2 = warp_sum((double)pc), sw2 = warp_sum((double)pw);
                const double num = (1.0 + (double)beta[j]) * sqrt(sc2);   // ||w_j - u_j||
                if (num / (sqrt(sw2) + 1.0e-10) < tol) break;
            } else {
                update<false, false>(g, step, th, beta[j], dummy, pc, pw);
            }
        }
    }
};

// ------------------------------------------------------------------------------------------------
// deconv, fixed lambda (pybold/bold_signal.py:49-97)
// ------------------------------------------------------------------------------------------------
// AUTO: deconv(lbda=None), one inner pass per outer iteration of the noise loop (pb_noise_loop.cuh), then the
// final pass; the window of alphas (wind doubles per warp) follows the rings in shared memory
template <typename real, int R, int KMAX, bool CIRC, int WARPS, int MINB, bool AUTO = false>
__global__ void __launch_bounds__(WARPS * 32, MINB)
fast_deconv_kernel(DeconvArgs<real> p, int ring_rows) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    real *beta = reinterpret_cast<real *>(smem);
    const size_t beta_bytes = ((size_t)p.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    fill_momentum_table(beta, p.nb_iter);
    // ring of past u's for the early stop (Q5): [slot][r][lane]
    real *ring = reinterpret_cast<real *>(smem + beta_bytes) + (size_t)warp * ring_rows * R * 32;
    const int T = p.T, K = p.K;
    const bool es = p.early_stopping && p.wind >= 2;
    const int sub = p.wind / 2, nring = p.wind - 1;

    WarpVoxel<real, R, KMAX, CIRC> vx;
    vx.init(lane, T);
    for (int64_t v = (int64_t)blockIdx.x * WARPS + warp; v < p.V; v += (int64_t)gridDim.x * WARPS) {
        if (!p.is_active(v)) continue;
        const real *yv = p.y_row(v);
        const real *hv = p.h_row(v);
        vx.set_dy(yv, T);
#pragma unroll
        for (int j = 0; j < KMAX; ++j) vx.h[j] = (j < K && vx.nvalid > 0) ? hv[j] : real(0);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = lane * R + r;
            vx.w[r] = (p.w0 && i < T) ? p.w0[v * T + i] : real(0);
        }
        const double Lc = p.L_of(v);
        NoiseLoop nl;
        if (AUTO) {
            const size_t ring_bytes = (size_t)WARPS * ring_rows * R * 32 * sizeof(real);
            nl.start(reinterpret_cast<double *>(smem + beta_bytes + ring_bytes) + (size_t)warp * p.wind);
        }
        double lam = AUTO ? nl.lbda : p.lam_of(v);
        const real step = (real)(1.0 / Lc);
        real th = (real)(lam / Lc);
        real *Jv = p.out_J + v * (int64_t)p.nb_iter;
        int n_done = 0, ring_pos = 0;
        real res[R];
        for (;;) {   // one pass (AUTO: one per outer iteration)
            n_done = 0;
            ring_pos = 0;
            for (int k = 0; k < p.nb_iter; ++k) {
                vx.forward(res);
                if (!AUTO && k > 0) {   // cost of the previous iterate: its residual has just been formed
                    const double J = 0.5 * warp_sum((double)vx.partial_sumsq(res)) +
                                     lam * warp_sum((double)vx.partial_sumabs(vx.w));
                    if (lane == 0 && p.out_J) Jv[k - 1] = (real)J;
                }
                real g[R], u[R], pc, pw;
                vx.adjoint(res, g);
                if (es) {
                    vx.template update<true, false>(g, step, th, beta[k], u, pc, pw);
                    real *slot = ring + (size_t)ring_pos * R * 32;         // ring_pos = k % nring
#pragma unroll
                    for (int r = 0; r < R; ++r) slot[r * 32 + lane] = u[r];
                } else {
                    vx.template update<false, false>(g, step, th, beta[k], u, pc, pw);
                }
                n_done = k + 1;
                if (es && k > p.wind) {
                    // xx = [u_{k-wind+2}, ..., u_k, w_k]; old = mean(first wind-sub), new = mean(last sub)
                    const real inv_old = real(1) / real(p.wind - sub), inv_new = real(1) / real(sub);
                    real so[R], sn[R];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        so[r] = 0;
                        sn[r] = vx.w[r];
                    }
                    int pos = ring_pos + 1 == nring ? 0 : ring_pos + 1;     // (k - wind + 2) % nring: oldest u
                    for (int m = 0; m < p.wind - 1; ++m) {
                        const real *slot = ring + (size_t)pos * R * 32;
                        pos = pos + 1 == nring ? 0 : pos + 1;
                        const bool is_old = m < p.wind - sub;
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const real uu = slot[r * 32 + lane];
                            if (is_old) so[r] += uu; else sn[r] += uu;
                        }
                    }
                    real qn = 0, qd = 0;                  // lane partials in `real`, warp sums in double
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const real mo = so[r] * inv_old, mn = sn[r] * inv_new;
                        qn = fma(mn - mo, mn - mo, qn);
                        qd = fma(mn, mn, qd);
                    }
                    const double pn = warp_sum((double)qn);
                    const double pd = warp_sum((double)qd);
                    if (sqrt(pn) / (sqrt(pd) + 1.0e-10) < p.tol) break;
                }
                if (es) ring_pos = ring_pos + 1 == nring ? 0 : ring_pos + 1;
            }
            vx.forward(res);
            if (AUTO) {
                const double rr = warp_sum((double)vx.partial_sumsq(res));
                const double gg = warp_sum((double)vx.partial_sumabs(vx.w));
                if (!nl.pass_done(p, v, rr, gg, lane == 0, lane, 32)) {
                    lam = nl.lbda;
                    th = (real)(lam / Lc);
                    continue;
                }
            } else if (n_done > 0) {
                const double rr = warp_sum((double)vx.partial_sumsq(res));
                const double gg = warp_sum((double)vx.partial_sumabs(vx.w));
                const double J = 0.5 * rr + lam * gg;
                if (lane == 0) {
                    if (p.out_J) Jv[n_done - 1] = (real)J;
                    if (p.out_r) p.out_r[v] = (real)rr;
                    if (p.out_g) p.out_g[v] = (real)gg;
                }
            }
            break;
        }
        real y[R], z[R];
        vx.load_y(yv, T, y);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            y[r] += res[r];      // x = (A w - y) + y
            z[r] = vx.w[r];
        }
        vx.scan_fwd(z);
        vx.store(p.out_x + v * T, y, T);
        vx.store(p.out_z + v * T, z, T);
        vx.store(p.out_dz + v * T, vx.w, T);
        if (lane == 0 && !AUTO) p.out_niter[v] = n_done;
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// bd (pybold/bold_signal.py:281-382)
// ------------------------------------------------------------------------------------------------
template <typename real, int R, int KMAX, bool CIRC, int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
fast_bd_kernel(BdArgs<real> p) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    real *beta = reinterpret_cast<real *>(smem);
    const size_t beta_bytes = ((size_t)p.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    fill_momentum_table(beta, p.nb_iter);
    ThetaScratch sc;
    sc.bind(reinterpret_cast<double *>(smem + beta_bytes) + (size_t)warp * pb_scratch_doubles(KMAX), KMAX);
    const int T = p.T, K = p.K, ntr = p.nb_iter + 2;
    const bool es = p.early_stopping != 0;
    const int sub = p.wind / 2;

    WarpVoxel<real, R, KMAX, CIRC> vx;
    vx.init(lane, T);
    for (int64_t v = (int64_t)blockIdx.x * WARPS + warp; v < p.V; v += (int64_t)gridDim.x * WARPS) {
        const real *yv = p.y + v * T;
        vx.set_dy(yv, T);
        const double lam = (double)p.lbda[v * p.lbda_stride];
        double theta = (double)p.theta0[v * p.theta0_stride];
        hrf_eval_warp(theta, p.grid, sc, lane);     // bold_signal.py:292 (theta_0 itself: Q9)
        vx.load_taps(sc.hs, K);
        double r0, g0;
        {
            real y[R];
            vx.load_y(yv, T, y);
            if (p.z0) {                                 // bold_signal.py:298-301
                const real *zv = p.z0 + v * T;
                real z[R], hal[KMAX - 1], xr[R];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int i = lane * R + r;
                    z[r] = i < T ? zv[i] : real(0);
                    vx.w[r] = (i > 0 && i < T) ? zv[i] - zv[i - 1] : real(0);
                    xr[r] = -y[r];
                }
                vx.template halo_up<false>(z, hal);
                vx.conv_acc(z, hal, xr);
#pragma unroll
                for (int r = 0; r < R; ++r) xr[r] = r < vx.nvalid ? xr[r] : real(0);
                r0 = warp_sum((double)vx.partial_sumsq(xr));
                g0 = warp_sum((double)vx.partial_sumabs(vx.w));
            } else {
#pragma unroll
                for (int r = 0; r < R; ++r) vx.w[r] = real(0);
                r0 = warp_sum((double)vx.partial_sumsq(y));
                g0 = 0.0;
            }
        }
        const double j0 = r0 + lam * g0;
        real *Jv = p.out_J + v * (int64_t)ntr, *rv = p.out_r + v * (int64_t)ntr,
             *gv = p.out_g + v * (int64_t)ntr;
        if (lane == 0) {
            Jv[0] = real(1);
            rv[0] = real(1);
            gv[0] = (real)g0;
        }
        int n = 1;
        double sumJ = 1.0;
        bool stopped = false;
        for (int idx = 0; idx <= p.nb_iter; ++idx) {
            const bool last = stopped || idx == p.nb_iter;    // final (long) deconvolution, :365-376
            const double Lc = frob_lipschitz_warp(sc, K, T, lane);
            vx.inner_loop(beta, p.nb_iter, (real)(1.0 / Lc), (real)(lam / Lc), es, p.tol);

            real z[R], hal[KMAX - 1], y[R];
#pragma unroll
            for (int r = 0; r < R; ++r) z[r] = vx.w[r];
            vx.scan_fwd(z);
            vx.template halo_up<false>(z, hal);
            vx.load_y(yv, T, y);
            if (!last) {
                // ---- theta step (bold_signal.py:329-334): b = Z^T y, Rz = autocorrelation of z ----
                real zm[R];
#pragma unroll
                for (int r = 0; r < R; ++r) zm[r] = r < vx.nvalid ? z[r] : real(0);
#pragma unroll
                for (int a = 0; a < KMAX; ++a) {
                    real pb_ = 0, pr = 0;
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const int id = r - a;
                        const real zz = id >= 0 ? z[id >= 0 ? id : 0] : hal[id >= 0 ? 0 : -id - 1];
                        pb_ = fma(y[r], zz, pb_);
                        pr = fma(zm[r], zz, pr);
                    }
                    pb_ = warp_sum(pb_);
                    pr = warp_sum(pr);
                    if (lane == 0 && a < K) {
                        sc.b[a] = (double)pb_;
                        sc.Rz[a] = (double)pr;
                    }
                }
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int pidx = T - 1 - (lane * R + r);
                    if (pidx >= 0 && pidx < K) sc.zend[pidx] = (double)z[r];
                }
                if (lane < K && lane >= T) sc.zend[lane] = 0.0;
                if (lane + 32 < K && lane + 32 >= T) sc.zend[lane + 32] = 0.0;
                __syncwarp();
                gram_build_warp(sc, K, lane);
                theta = theta_solve_warp(theta, p.theta_lo, p.theta_hi, p.grid, sc, lane, nullptr);
                hrf_eval_warp(theta, p.grid, sc, lane);
                vx.load_taps(sc.hs, K);
            }
            // ---- cost trace: x = h * z with the (new) taps ----
            real xr[R];
#pragma unroll
            for (int r = 0; r < R; ++r) xr[r] = -y[r];
            vx.conv_acc(z, hal, xr);
#pragma unroll
            for (int r = 0; r < R; ++r) xr[r] = r < vx.nvalid ? xr[r] : real(0);
            const double rr = warp_sum((double)vx.partial_sumsq(xr));
            const double gg = warp_sum((double)vx.partial_sumabs(vx.w));
            const double eps = last ? 0.0 : 1.0e-30;
            const double Jn = (rr + lam * gg) / j0 + eps;
            if (lane == 0) {
                Jv[n] = (real)Jn;
                rv[n] = (real)(rr / r0 + eps);
                gv[n] = (real)gg;
            }
            sumJ += (double)(real)Jn;
            ++n;
            if (last) {
#pragma unroll
                for (int r = 0; r < R; ++r) xr[r] += y[r];
                vx.store(p.out_x + v * T, xr, T);
                vx.store(p.out_z + v * T, z, T);
                vx.store(p.out_dz + v * T, vx.w, T);
                break;
            }
            __syncwarp();
            if (es && idx > p.wind) {                   // Q7
                int stop = 0;
                if (lane == 0) stop = bd_outer_stop(Jv, n, sumJ, sub, p.tol) ? 1 : 0;
                stopped = __shfl_sync(PB_FULL, stop, 0) != 0;
            }
        }
        for (int a = lane; a < K; a += 32) p.out_h[v * K + a] = (real)sc.hs[a];
        if (lane == 0) {
            p.out_theta[v] = (real)theta;
            p.out_ntrace[v] = n;
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// host-side launchers (one variant per translation unit, see gen_fast_instances.py)
// ------------------------------------------------------------------------------------------------
template <typename real, int R, int KMAX, bool CIRC>
bool fast_shape_ok(int T, int K) {
    if (K > KMAX || T > 32 * R) return false;
    if (CIRC) return T % R == 0 && T / R + halo_lanes<R, KMAX>() <= 32;
    return true;
}

// FAST_NO_MATCH when the ring does not fit: the generic kernel decides
template <typename real, int R, int KMAX, bool CIRC, int WARPS, int MINB, bool AUTO = false>
int fast_deconv_launch(const DeconvArgs<real> &a, cudaStream_t stream) {
    const bool es = a.early_stopping && a.wind >= 2;
    const int ring_rows = es ? a.wind - 1 : 0;
    const size_t beta_bytes = ((size_t)a.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    const size_t smem = beta_bytes + (size_t)WARPS * ring_rows * R * 32 * sizeof(real) +
                        (AUTO ? (size_t)WARPS * a.wind * sizeof(double) : 0);
    return launch_persistent(fast_deconv_kernel<real, R, KMAX, CIRC, WARPS, MINB, AUTO>, WARPS * 32, smem, WARPS,
                             a.V, nullptr, stream, a, ring_rows);
}

template <typename real, int R, int KMAX, bool CIRC, int WARPS, int MINB>
int fast_bd_launch(const BdArgs<real> &a, cudaStream_t stream) {
    const size_t beta_bytes = ((size_t)a.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    const size_t smem = beta_bytes + (size_t)WARPS * pb_scratch_doubles(KMAX) * sizeof(double);
    return launch_persistent(fast_bd_kernel<real, R, KMAX, CIRC, WARPS, MINB>, WARPS * 32, smem, WARPS, a.V,
                             nullptr, stream, a);
}

template <typename real, int R, int KMAX, bool CIRC, int WARPS, int MINB>
constexpr Variant<real> warp_variant() {
    return {TIER_WARP, 32, R, KMAX, 0, CIRC, fast_shape_ok<real, R, KMAX, CIRC>,
            fast_bd_launch<real, R, KMAX, CIRC, WARPS, MINB>, nullptr,
            fast_deconv_launch<real, R, KMAX, CIRC, WARPS, MINB>, nullptr,
            fast_deconv_launch<real, R, KMAX, CIRC, WARPS, MINB, true>};
}

}  // namespace pb
