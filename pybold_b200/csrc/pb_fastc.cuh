// Register-tiled persistent bd and deconv kernels, CTA variant: ONE CTA OF NW WARPS PER VOXEL, for long series
// (T = 1200 at cfg4) and many taps.  Thread t of the CTA owns the R contiguous samples [t R, t R + R) in
// registers (32 NW R >= T, R a multiple of 4).
//
// Why: with one warp per voxel a 1200-sample voxel needs R = 38-40 samples per lane, i.e. ~255
// registers, 8 resident warps per SM and a fully unrolled loop body of ~44 KB that no longer fits the
// instruction cache (measured IPC 0.52).  Two warps per voxel halve R: ~130 registers, 16 warps per
// SM and a 22 KB loop body.
//
// Differences from pb_fast.cuh / pb_fastg.cuh:
//  * the K-1 halo samples are exchanged through shared memory: every thread stores its R values as
//    float4 and loads the 28 preceding (or following) values as 7 float4.  Zero pads before and after
//    the voxel make the boundary handling free (no select), and this costs 12 instead of 54
//    instructions per convolution;
//  * the scans add a cross-warp carry (warp totals through shared memory);
//  * 4 __syncthreads per iteration (w visible, forward totals, residual visible, reverse totals);
//  * the Lipschitz constant and the theta solve are run by warp 0 with the code of pb_device.cuh.
// bd: tap 0 of the SPM HRF is identically zero.  ES = true runs the reference's early stopping (Q6 / Q7, below).
// deconv (fast_deconvc_kernel): every mode of fast_deconv_kernel, including the Q5 early stop and deconv(lbda=None),
// for the shapes no group or warp variant serves (pb_fast_registry.cu); the caller's taps start at tap 0.
//
// Reference code replaced: pybold/bold_signal.py:49-97, :99-214, :242-278, :281-382.
#pragma once
#include "pb_fast_registry.h"
#include "pb_generic.cuh"

#include "pb_tile.cuh"

// source order of the unrolled tile (pb_tile.cuh), picked with the register-file model on
// fast_bdc_kernel<float, 20, 28, 2, 6> (cfg4: 1587 -> 1423 modelled cycles per inner iteration; tools/order_search.py cta)
#ifndef PB_C_CONV_JDESC
#define PB_C_CONV_JDESC 1
#endif
#ifndef PB_C_CONV_RDESC
#define PB_C_CONV_RDESC 0
#endif
#ifndef PB_C_CONV_RB
#define PB_C_CONV_RB 5
#endif
#ifndef PB_C_CONV_DS
#define PB_C_CONV_DS 0
#endif
#ifndef PB_C_CORR_JDESC
#define PB_C_CORR_JDESC 1
#endif
#ifndef PB_C_CORR_RDESC
#define PB_C_CORR_RDESC 1
#endif
#ifndef PB_C_CORR_RB
#define PB_C_CORR_RB 5
#endif
#ifndef PB_C_CORR_DS
#define PB_C_CORR_DS 0
#endif

namespace pb {

template <typename real, int R, int KMAX, int NW>
struct CtaLayout {
    static constexpr int NT = NW * 32;
    static constexpr int SLOTS = NT * R;
    static constexpr int PAD = (KMAX + 3) & ~3;               // >= KMAX - 1, keeps float4 alignment
    // R = 8 / 16: the per-thread stride of R floats is a multiple of 8 banks and the 16-byte stores / loads
    // of a quarter warp would collide (round 1 measured R = 16 at 29 instead of 42 Tflop/s per slot and did
    // not build it).  SKEW inserts 4 unused floats after every 32 samples: sample i lives at
    // i + 4 (i >> 5), a thread's block and every aligned vector stay contiguous, and consecutive threads'
    // vectors fall into distinct banks again.  (i >> 5 is an arithmetic shift: the zero pad before the
    // series, i in [-PAD, -1], lands at i - 4.)
    static constexpr bool SKEW = R % 8 == 0;
    static constexpr int PADB = SKEW ? PAD + 8 : PAD;         // zero pad before sample 0
    __host__ __device__ static constexpr int pos(int i) { return SKEW ? i + ((i >> 5) << 2) : i; }
    static constexpr int BUF = PADB + pos(SLOTS + PAD) + 4;
    static constexpr int RED = NW * (2 * KMAX + 4);           // doubles for CTA-wide reductions
    __host__ __device__ static constexpr size_t bytes(int nb_iter) {
        return (((size_t)nb_iter * sizeof(real) + 15) & ~(size_t)15) +
               ((size_t)pb_scratch_doubles(KMAX) + RED + 2 * NW + 4) * sizeof(double) +
               (size_t)2 * BUF * sizeof(real);
    }
    // deconv (fast_deconvc_kernel): beta | doubles: totf [NW], totr [NW], red [NW][2], the window of nwin alphas |
    // the two buffers | the early-stopping ring of ring_rows past u's.  No theta scratch.
    __host__ __device__ static constexpr size_t beta_bytes(int nb_iter) {
        return ((size_t)nb_iter * sizeof(real) + 15) & ~(size_t)15;
    }
    __host__ __device__ static constexpr size_t deconv_dbl_bytes(int nwin) {
        return ((size_t)(4 * NW + nwin) * sizeof(double) + 15) & ~(size_t)15;
    }
    __host__ __device__ static constexpr size_t deconv_bytes(int nb_iter, int ring_rows, int nwin) {
        return beta_bytes(nb_iter) + deconv_dbl_bytes(nwin) + (size_t)2 * BUF * sizeof(real) +
               (size_t)ring_rows * SLOTS * sizeof(real);
    }
};

// Helpers over the register tiles of one CTA-resident deconv problem: the helpers of fast_bdc_kernel, except that
// the tiles start at tap 0 (the caller's HRF, not the SPM one whose tap 0 is zero) and that a CTA-wide sum uses two
// doubles per warp (red[2 w], red[2 w + 1]).  fast_bdc_kernel keeps its own copies as lambdas: routed through this
// struct, its register allocation changed (six SASS lines in the HRF evaluation).  Thread tid owns samples
// [i0, i0 + R).
template <typename real, int R, int KMAX, int NW>
struct CtaTile {
    static constexpr int JS = 0, RS = 2;
    using L = CtaLayout<real, R, KMAX, NW>;
    struct alignas(4 * sizeof(real)) V4 { real t[4]; };
    static constexpr int NH = (KMAX - 1 + 3) / 4;             // float4 per halo
    int tid, lane, warp, i0, nvalid;
    real *totf_r, *totr_r;                                    // [NW] forward / reverse warp totals
    double *red;

    __device__ __forceinline__ void put(real *dst, const real (&a)[R]) const {
#pragma unroll
        for (int r4 = 0; r4 < R / 4; ++r4) {
            V4 t;
#pragma unroll
            for (int e = 0; e < 4; ++e) t.t[e] = a[4 * r4 + e];
            reinterpret_cast<V4 *>(dst)[r4] = t;
        }
    }
    // hal[m-1] = value at index (i0 - m), m = 1..4 NH
    __device__ __forceinline__ void halo_before(const real *mine, real (&hal)[4 * NH]) const {
#pragma unroll
        for (int c = 0; c < NH; ++c) {
            const V4 t = L::SKEW ? *reinterpret_cast<const V4 *>(mine - L::pos(i0) + L::pos(i0 - 4 * (c + 1)))
                                 : reinterpret_cast<const V4 *>(mine)[-1 - c];
#pragma unroll
            for (int e = 0; e < 4; ++e) hal[4 * c + (3 - e)] = t.t[e];
        }
    }
    // hal[k] = value at index (i0 + R + k), k = 0..4 NH - 1
    __device__ __forceinline__ void halo_after(const real *mine, real (&hal)[4 * NH]) const {
#pragma unroll
        for (int c = 0; c < NH; ++c) {
            const V4 t = L::SKEW ? *reinterpret_cast<const V4 *>(mine - L::pos(i0) + L::pos(i0 + R + 4 * c))
                                 : reinterpret_cast<const V4 *>(mine + R)[c];
#pragma unroll
            for (int e = 0; e < 4; ++e) hal[4 * c + e] = t.t[e];
        }
    }
    __device__ __forceinline__ void conv_acc(const real (&h)[KMAX], const real (&a)[R], const real (&hal)[4 * NH],
                                             real (&acc)[R]) const {
        tile_conv<real, R, KMAX, 4 * NH, JS, PB_C_CONV_JDESC, PB_C_CONV_RDESC, PB_C_CONV_RB, PB_C_CONV_DS>(h, a, hal, acc);
    }
    __device__ __forceinline__ void corr_acc(const real (&h)[KMAX], const real (&a)[R], const real (&hal)[4 * NH],
                                             real (&acc)[R]) const {
        tile_corr<real, R, KMAX, 4 * NH, JS, PB_C_CORR_JDESC, PB_C_CORR_RDESC, PB_C_CORR_RB, PB_C_CORR_DS>(h, a, hal, acc);
    }
    __device__ __forceinline__ void mask_tail(real (&a)[R]) const {
#pragma unroll
        for (int r = 0; r < R; ++r) a[r] = r < nvalid ? a[r] : real(0);
    }
    // CTA-wide inclusive prefix of a register tile (one barrier inside)
    __device__ __forceinline__ void scan_fwd_cta(real (&a)[R]) const {
#pragma unroll
        for (int r = 1; r < R; ++r) a[r] += a[r - 1];
        real inc = a[R - 1];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const real t = __shfl_up_sync(PB_FULL, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) totf_r[warp] = inc;
        real carry = __shfl_up_sync(PB_FULL, inc, 1);
        if (lane == 0) carry = real(0);
        __syncthreads();
#pragma unroll
        for (int ww = 0; ww < NW - 1; ++ww)
            if (ww < warp) carry += totf_r[ww];
#pragma unroll
        for (int r = 0; r < R; ++r) a[r] += carry;
    }
    __device__ __forceinline__ void scan_rev_cta(real (&a)[R]) const {
#pragma unroll
        for (int r = R - 2; r >= 0; --r) a[r] += a[r + 1];
        real inc = a[0];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const real t = __shfl_down_sync(PB_FULL, inc, d);
            if (lane + d < 32) inc += t;
        }
        if (lane == 0) totr_r[warp] = inc;
        real carry = __shfl_down_sync(PB_FULL, inc, 1);
        if (lane == 31) carry = real(0);
        __syncthreads();
#pragma unroll
        for (int ww = 1; ww < NW; ++ww)
            if (ww > warp) carry += totr_r[ww];
#pragma unroll
        for (int r = 0; r < R; ++r) a[r] += carry;
    }
    // warp sums of a and b into this warp's slots of red (no barrier)
    __device__ __forceinline__ void publish2(double a, double b) const {
        a = warp_sum(a);
        b = warp_sum(b);
        if (lane == 0) {
            red[warp * RS] = a;
            red[warp * RS + 1] = b;
        }
    }
    // the CTA-wide sums of what publish2 wrote, warps added in a fixed order (call after a barrier)
    __device__ __forceinline__ void gather2(double &a, double &b) const {
        double sa = 0.0, sb = 0.0;
#pragma unroll
        for (int ww = 0; ww < NW; ++ww) {
            sa += red[ww * RS];
            sb += red[ww * RS + 1];
        }
        a = sa;
        b = sb;
    }
    // CTA-wide sums of two doubles (two barriers; result on every thread)
    __device__ __forceinline__ void cta_sum2(double &a, double &b) const {
        a = warp_sum(a);
        b = warp_sum(b);
        __syncthreads();
        if (lane == 0) {
            red[warp * RS] = a;
            red[warp * RS + 1] = b;
        }
        __syncthreads();
        gather2(a, b);
    }
};

// ES = true: bd(early_stopping=True).  Q6 -- the inner loop stops at iteration j > 2 once
// ||w_j - u_j|| / (||w_j|| + 1e-10) < tol, with ||w_j - u_j|| = (1 + beta_j) ||clamp(u_j)|| -- takes its two sums on
// the barriers already there: the warp sums of iteration j go to red[2], red[3] of the warp's row before B1 of
// iteration j + 1, and every thread reads them after it and takes the same break (iteration j + 1 has then only
// stored w).  Q7 -- the signed window test on J (bd_outer_stop) after pass idx > wind -- is run by thread 0, which
// wrote J, while warp 0 forms the Lipschitz constant of the next pass; the decision reaches every thread on the
// barrier after it and makes that pass the last one.  out_ntrace = idx + 3 for a stop after pass idx.  With
// ES = false none of this is compiled in.
template <typename real, int R, int KMAX, int NW, int MINB, bool ES = false>
__global__ void __launch_bounds__(NW * 32, MINB)
fast_bdc_kernel(BdArgs<real> p) {
    static_assert(R % 4 == 0, "R must be a multiple of 4 (vector halo exchange)");
    using L = CtaLayout<real, R, KMAX, NW>;
    struct alignas(4 * sizeof(real)) V4 { real t[4]; };
    constexpr int NH = (KMAX - 1 + 3) / 4;                    // float4 per halo
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    real *beta = reinterpret_cast<real *>(smem);
    const size_t beta_bytes = ((size_t)p.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    fill_momentum_table(beta, p.nb_iter);
    double *dbl = reinterpret_cast<double *>(smem + beta_bytes);
    ThetaScratch sc;
    sc.bind(dbl, KMAX);
    double *red = dbl + pb_scratch_doubles(KMAX);             // [NW][2 KMAX + 4]
    double *totf = red + L::RED;                              // [NW] forward warp totals
    double *totr = totf + NW;                                 // [NW] reverse warp totals
    double *bcast = totr + NW;                                // [4]  theta, Lipschitz, Q7 stop, -
    real *bufA = reinterpret_cast<real *>(bcast + 4);         // w / z with zero pads
    real *bufB = bufA + L::BUF;                               // residual with zero pads
    for (int i = tid; i < 2 * L::BUF; i += L::NT) bufA[i] = real(0);   // zero pads (and everything else once)
    real *const baseA = bufA + L::PADB, *const baseB = bufB + L::PADB;  // sample 0 of the two buffers
    real *myA = baseA + L::pos(tid * R), *myB = baseB + L::pos(tid * R);
    const int T = p.T, K = p.K, ntr = p.nb_iter + 2;
    const int i0 = tid * R;
    const int nvalid = max(0, min(R, T - i0));
    real *totf_r = reinterpret_cast<real *>(totf), *totr_r = reinterpret_cast<real *>(totr);
    __syncthreads();

    real w[R], dy[R], h[KMAX];

    // ---- small helpers over register tiles -------------------------------------------------
    auto put = [&](real *dst, const real (&a)[R]) {
#pragma unroll
        for (int r4 = 0; r4 < R / 4; ++r4) {
            V4 t;
#pragma unroll
            for (int e = 0; e < 4; ++e) t.t[e] = a[4 * r4 + e];
            reinterpret_cast<V4 *>(dst)[r4] = t;
        }
    };
    // hal[m-1] = value at voxel index (i0 - m), m = 1..4 NH
    auto halo_before = [&](const real *mine, real (&hal)[4 * NH]) {
#pragma unroll
        for (int c = 0; c < NH; ++c) {
            const V4 t = L::SKEW ? *reinterpret_cast<const V4 *>(mine - L::pos(i0) + L::pos(i0 - 4 * (c + 1)))
                                 : reinterpret_cast<const V4 *>(mine)[-1 - c];
#pragma unroll
            for (int e = 0; e < 4; ++e) hal[4 * c + (3 - e)] = t.t[e];
        }
    };
    // hal[k] = value at voxel index (i0 + R + k), k = 0..4 NH - 1
    auto halo_after = [&](const real *mine, real (&hal)[4 * NH]) {
#pragma unroll
        for (int c = 0; c < NH; ++c) {
            const V4 t = L::SKEW ? *reinterpret_cast<const V4 *>(mine - L::pos(i0) + L::pos(i0 + R + 4 * c))
                                 : reinterpret_cast<const V4 *>(mine + R)[c];
#pragma unroll
            for (int e = 0; e < 4; ++e) hal[4 * c + e] = t.t[e];
        }
    };
    auto conv_acc = [&](const real (&a)[R], const real (&hal)[4 * NH], real (&acc)[R]) {
        tile_conv<real, R, KMAX, 4 * NH, 1, PB_C_CONV_JDESC, PB_C_CONV_RDESC, PB_C_CONV_RB, PB_C_CONV_DS>(h, a, hal, acc);
    };
    auto corr_acc = [&](const real (&a)[R], const real (&hal)[4 * NH], real (&acc)[R]) {
        tile_corr<real, R, KMAX, 4 * NH, 1, PB_C_CORR_JDESC, PB_C_CORR_RDESC, PB_C_CORR_RB, PB_C_CORR_DS>(h, a, hal, acc);
    };
    auto mask_tail = [&](real (&a)[R]) {
#pragma unroll
        for (int r = 0; r < R; ++r) a[r] = r < nvalid ? a[r] : real(0);
    };
    // CTA-wide inclusive prefix of a register tile (one barrier inside)
    auto scan_fwd_cta = [&](real (&a)[R]) {
#pragma unroll
        for (int r = 1; r < R; ++r) a[r] += a[r - 1];
        real inc = a[R - 1];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const real t = __shfl_up_sync(PB_FULL, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) totf_r[warp] = inc;
        real carry = __shfl_up_sync(PB_FULL, inc, 1);
        if (lane == 0) carry = real(0);
        __syncthreads();
#pragma unroll
        for (int ww = 0; ww < NW - 1; ++ww)
            if (ww < warp) carry += totf_r[ww];
#pragma unroll
        for (int r = 0; r < R; ++r) a[r] += carry;
    };
    auto scan_rev_cta = [&](real (&a)[R]) {
#pragma unroll
        for (int r = R - 2; r >= 0; --r) a[r] += a[r + 1];
        real inc = a[0];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const real t = __shfl_down_sync(PB_FULL, inc, d);
            if (lane + d < 32) inc += t;
        }
        if (lane == 0) totr_r[warp] = inc;
        real carry = __shfl_down_sync(PB_FULL, inc, 1);
        if (lane == 31) carry = real(0);
        __syncthreads();
#pragma unroll
        for (int ww = 1; ww < NW; ++ww)
            if (ww > warp) carry += totr_r[ww];
#pragma unroll
        for (int r = 0; r < R; ++r) a[r] += carry;
    };
    // CTA-wide sums of two doubles (two barriers; result on every thread)
    auto cta_sum2 = [&](double &a, double &b) {
        a = warp_sum(a);
        b = warp_sum(b);
        __syncthreads();
        if (lane == 0) {
            red[warp * (2 * KMAX + 4)] = a;
            red[warp * (2 * KMAX + 4) + 1] = b;
        }
        __syncthreads();
        double sa = 0.0, sb = 0.0;
#pragma unroll
        for (int ww = 0; ww < NW; ++ww) {
            sa += red[ww * (2 * KMAX + 4)];
            sb += red[ww * (2 * KMAX + 4) + 1];
        }
        a = sa;
        b = sb;
    };
    auto load_taps = [&]() {
#pragma unroll
        for (int j = 0; j < KMAX; ++j) h[j] = j < K ? (real)sc.hs[j] : real(0);
    };

    // the first voxel of a CTA is static, the following ones come from the work queue when there is one
    __shared__ unsigned int next_task;
    for (int64_t v = blockIdx.x; v < p.V;) {
        const real *yv = p.y + v * T;
        real y[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = i0 + r;
            y[r] = i < T ? yv[i] : real(0);
            const real prv = (i > 0 && i - 1 < T) ? yv[i - 1] : real(0);
            dy[r] = i < T ? y[r] - prv : real(0);
        }
        const double lam = (double)p.lbda[v * p.lbda_stride];
        double theta = (double)p.theta0[v * p.theta0_stride];
        __syncthreads();
        if (warp == 0) hrf_eval_warp(theta, p.grid, sc, lane);   // bold_signal.py:292 (theta_0: Q9)
        __syncthreads();
        load_taps();
        double r0, g0 = 0.0;
        if (p.z0) {                                               // bold_signal.py:298-301
            const real *zv = p.z0 + v * T;
            real z[R], hal[4 * NH], xr[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int i = i0 + r;
                z[r] = i < T ? zv[i] : real(0);
                w[r] = (i > 0 && i < T) ? zv[i] - zv[i - 1] : real(0);
                xr[r] = -y[r];
            }
            put(myA, z);
            __syncthreads();
            halo_before(myA, hal);
            conv_acc(z, hal, xr);
            mask_tail(xr);
            real s2 = 0, s1 = 0;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                s2 = fma(xr[r], xr[r], s2);
                s1 += fabs(w[r]);
            }
            r0 = (double)s2;
            g0 = (double)s1;
            cta_sum2(r0, g0);
        } else {
            real s2 = 0;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                w[r] = real(0);
                s2 = fma(y[r], y[r], s2);
            }
            r0 = (double)s2;
            double zero = 0.0;
            cta_sum2(r0, zero);
        }
        const double j0 = r0 + lam * g0;
        real *Jv = p.out_J + v * (int64_t)ntr, *rv = p.out_r + v * (int64_t)ntr,
             *gv = p.out_g + v * (int64_t)ntr;
        if (tid == 0) {
            Jv[0] = real(1);
            rv[0] = real(1);
            gv[0] = (real)g0;
        }
        int n_tr = ntr;                                           // ES: trace entries written
        double sumJ = 1.0;                                        // ES: sum of the J entries (as stored)
        for (int idx = 0; idx <= p.nb_iter; ++idx) {
            bool last = idx == p.nb_iter;                         // final deconvolution, :365-376
            __syncthreads();
            if (warp == 0) {
                const double Lw = frob_lipschitz_warp(sc, K, T, lane);
                if (lane == 0) bcast[1] = Lw;
                if constexpr (ES)                                 // Q7 (:350-362) after pass idx - 1: J[0 .. idx]
                    if (lane == 0)
                        bcast[2] = idx - 1 > p.wind && bd_outer_stop(Jv, idx + 1, sumJ, p.wind / 2, p.tol) ? 1.0 : 0.0;
            }
            __syncthreads();
            if constexpr (ES) last = last || bcast[2] != 0.0;     // (:350-362: the pass after the stop is the last)
            const double Lc = bcast[1];
            const real step = (real)(1.0 / Lc), th = (real)(lam / Lc);
            for (int j = 0; j < p.nb_iter; ++j) {                 // _loops_deconv, :259-276
                real hal[4 * NH], res[R], g[R];
                put(myA, w);
                __syncthreads();                                  // B1: w visible
                if constexpr (ES) {
                    if (j > 3) {                                  // Q6 (:267-273) on iteration j - 1
                        double sc2 = 0.0, sw2 = 0.0;
#pragma unroll
                        for (int ww = 0; ww < NW; ++ww) {
                            sc2 += red[ww * (2 * KMAX + 4) + 2];
                            sw2 += red[ww * (2 * KMAX + 4) + 3];
                        }
                        const double num = (1.0 + (double)beta[j - 1]) * sqrt(sc2);   // ||w - u||
                        if (num / (sqrt(sw2) + 1.0e-10) < p.tol) break;
                    }
                }
                halo_before(myA, hal);
#pragma unroll
                for (int r = 0; r < R; ++r) res[r] = -dy[r];
                conv_acc(w, hal, res);
                scan_fwd_cta(res);                                // B2 inside
                mask_tail(res);
                put(myB, res);
                __syncthreads();                                  // B3: residual visible
                halo_after(myB, hal);
#pragma unroll
                for (int r = 0; r < R; ++r) g[r] = real(0);
                corr_acc(res, hal, g);
                scan_rev_cta(g);                                  // B4 inside
                const real ob = real(1) + beta[j];
                if constexpr (!ES) {
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const real u = fma(-step, g[r], w[r]);
                        const real cl = fmin(fmax(u, -th), th);
                        w[r] = fma(-ob, cl, u);
                    }
                } else {
                    real pc = 0, pw = 0;
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const real u = fma(-step, g[r], w[r]);
                        const real cl = fmin(fmax(u, -th), th);
                        w[r] = fma(-ob, cl, u);
                        pc = fma(cl, cl, pc);
                        pw = fma(w[r], w[r], pw);
                    }
                    if (j > 2) {                                  // read after the next B1
                        const double sc2 = warp_sum((double)pc), sw2 = warp_sum((double)pw);
                        if (lane == 0) {
                            red[warp * (2 * KMAX + 4) + 2] = sc2;
                            red[warp * (2 * KMAX + 4) + 3] = sw2;
                        }
                    }
                }
            }
            real z[R], hal[4 * NH];
#pragma unroll
            for (int r = 0; r < R; ++r) z[r] = w[r];
            scan_fwd_cta(z);
            put(myA, z);
            __syncthreads();
            halo_before(myA, hal);
            if (!last) {
                // ---- theta step (:329-334): b = Z^T y, Rz = autocorrelation of z ----
                real zm[R];
#pragma unroll
                for (int r = 0; r < R; ++r) zm[r] = z[r];
                mask_tail(zm);
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
                    if (lane == 0) {
                        red[warp * (2 * KMAX + 4) + 4 + a] = (double)pb_;
                        red[warp * (2 * KMAX + 4) + 4 + KMAX + a] = (double)pr;
                    }
                }
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int pidx = T - 1 - (i0 + r);
                    if (pidx >= 0 && pidx < K) sc.zend[pidx] = (double)z[r];
                }
                for (int a = tid; a < K; a += L::NT)
                    if (a >= T) sc.zend[a] = 0.0;
                __syncthreads();
                if (warp == 0) {
                    for (int a = lane; a < K; a += 32) {
                        double sb = 0.0, sr = 0.0;
#pragma unroll
                        for (int ww = 0; ww < NW; ++ww) {
                            sb += red[ww * (2 * KMAX + 4) + 4 + a];
                            sr += red[ww * (2 * KMAX + 4) + 4 + KMAX + a];
                        }
                        sc.b[a] = sb;
                        sc.Rz[a] = sr;
                    }
                    __syncwarp();
                    gram_build_warp(sc, K, lane);
                    const double th_n = theta_solve_warp(theta, p.theta_lo, p.theta_hi, p.grid, sc,
                                                         lane, nullptr);
                    hrf_eval_warp(th_n, p.grid, sc, lane);
                    if (lane == 0) bcast[0] = th_n;
                }
                __syncthreads();
                theta = bcast[0];
                load_taps();
            }
            // ---- cost trace: x = h * z with the (new) taps ----
            real xr[R];
#pragma unroll
            for (int r = 0; r < R; ++r) xr[r] = -y[r];
            conv_acc(z, hal, xr);
            mask_tail(xr);
            real s2 = 0, s1 = 0;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                s2 = fma(xr[r], xr[r], s2);
                s1 += fabs(w[r]);
            }
            double rr = (double)s2, gg = (double)s1;
            cta_sum2(rr, gg);
            const double eps = last ? 0.0 : 1.0e-30;
            if (tid == 0) {
                Jv[idx + 1] = (real)((rr + lam * gg) / j0 + eps);
                rv[idx + 1] = (real)(rr / r0 + eps);
                gv[idx + 1] = (real)gg;
            }
            if constexpr (ES) sumJ += (double)(real)((rr + lam * gg) / j0 + eps);
            if (last) {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int i = i0 + r;
                    if (i < T) {
                        p.out_x[v * T + i] = xr[r] + y[r];
                        p.out_z[v * T + i] = z[r];
                        p.out_dz[v * T + i] = w[r];
                    }
                }
                if constexpr (ES) {
                    n_tr = idx + 2;
                    break;
                }
            }
        }
        __syncthreads();
        for (int a = tid; a < K; a += L::NT) p.out_h[v * K + a] = (real)sc.hs[a];
        if (tid == 0) {
            p.out_theta[v] = (real)theta;
            p.out_ntrace[v] = n_tr;
            if (p.queue) next_task = atomicAdd(p.queue, 1u);
        }
        __syncthreads();
        v = p.queue ? (int64_t)gridDim.x + (int64_t)next_task : v + gridDim.x;
    }
}

// ------------------------------------------------------------------------------------------------
// deconv (pybold/bold_signal.py:49-97), one CTA per problem, with the semantics of fast_deconv_kernel
// (pb_fast.cuh) line for line: warm start w0, the problem's y row, taps, Lipschitz constant and lambda (the
// regularisation path's y_mod / lbda_div, per-voxel HRFs), the active mask, the cost trace, the Q5 early stop
// and the final cost terms.  AUTO: deconv(lbda=None), one inner pass per outer iteration of the noise loop
// (pb_noise_loop.cuh), each restarting from the iterate of the pass before, then the final pass.
// Barriers per iteration: the four of fast_bdc_kernel; the cost of the previous iterate rides on B3, the Q5
// test adds one CTA-wide pair of sums (two barriers), so every thread takes the same break.  With early stopping
// the problems come from the work queue after the first (their iteration counts differ).
// CENSOR: scan censoring (Censor, pb_generic.cuh).  A thread keeps the keep-bits of its R samples in one register;
// censored y entries are zeroed at load, a select masks the residual after forward() (before the adjoint and the cost
// sums), x = (A w - y) + y is formed from the unmasked final residual and the zeroed y, and the noise loop's target is
// n_kept sigma^2 with n_kept one CTA-wide sum at voxel start.
// ------------------------------------------------------------------------------------------------
template <typename real, int R, int KMAX, int NW, int MINB, bool AUTO = false, bool CENSOR = false>
__global__ void __launch_bounds__(NW * 32, MINB)
fast_deconvc_kernel(DeconvArgs<real> p, int ring_rows, Censor cz) {
    static_assert(R % 4 == 0, "R must be a multiple of 4 (vector halo exchange)");
    using L = CtaLayout<real, R, KMAX, NW>;
    using CT = CtaTile<real, R, KMAX, NW>;
    constexpr int NH = CT::NH;
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    real *beta = reinterpret_cast<real *>(smem);
    const size_t beta_bytes = L::beta_bytes(p.nb_iter);
    fill_momentum_table(beta, p.nb_iter);
    double *totf = reinterpret_cast<double *>(smem + beta_bytes);
    double *red = totf + 2 * NW;                              // [NW][2], after totf [NW] and totr [NW]
    double *win = red + 2 * NW;                               // AUTO: the window of alphas [wind]
    real *bufA = reinterpret_cast<real *>(smem + beta_bytes + L::deconv_dbl_bytes(AUTO ? p.wind : 0));
    real *bufB = bufA + L::BUF;
    // ring of the past u's for the early stop (Q5): [slot][r][thread]; a thread only touches its own column
    real *ring = bufB + L::BUF + tid;
    for (int i = tid; i < 2 * L::BUF; i += L::NT) bufA[i] = real(0);   // zero pads (and everything else once)
    real *const myA = bufA + L::PADB + L::pos(tid * R), *const myB = bufB + L::PADB + L::pos(tid * R);
    const int T = p.T, K = p.K;
    const int i0 = tid * R;
    const int nvalid = max(0, min(R, T - i0));
    const CT ct{tid, lane, warp, i0, nvalid, reinterpret_cast<real *>(totf), reinterpret_cast<real *>(totf + NW),
                red};
    const bool es = p.early_stopping && p.wind >= 2;
    const int sub = p.wind / 2, nring = p.wind - 1;
    __syncthreads();

    real w[R], dy[R], h[KMAX];
    auto sumsq = [&](const real (&a)[R]) {
        real s = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) s = fma(a[r], a[r], s);
        return (double)s;
    };
    auto sumabs = [&](const real (&a)[R]) {
        real s = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) s += fabs(a[r]);
        return (double)s;
    };
    // res <- A w - y, zero at and beyond T (B1, B2)
    auto forward = [&](real (&res)[R]) {
        real hal[4 * NH];
        ct.put(myA, w);
        __syncthreads();                                      // B1: w visible
        ct.halo_before(myA, hal);
#pragma unroll
        for (int r = 0; r < R; ++r) res[r] = -dy[r];
        ct.conv_acc(h, w, hal, res);
        ct.scan_fwd_cta(res);                                 // B2 inside
        ct.mask_tail(res);
    };
    // g <- A^T res (B3, B4)
    auto adjoint = [&](const real (&res)[R], real (&g)[R]) {
        real hal[4 * NH];
        ct.put(myB, res);
        __syncthreads();                                      // B3: residual visible
        ct.halo_after(myB, hal);
#pragma unroll
        for (int r = 0; r < R; ++r) g[r] = real(0);
        ct.corr_acc(h, res, hal, g);
        ct.scan_rev_cta(g);                                   // B4 inside
    };

    __shared__ unsigned int next_task;
    for (int64_t v = blockIdx.x; v < p.V;) {
        if (p.is_active(v)) {
            const real *yv = p.y_row(v);
            const real *hv = p.h_row(v);
            unsigned keep = 0;                                // CENSOR: bit r set when sample i0 + r is kept
            if constexpr (CENSOR) {
                const unsigned char *cm = cz.row(p.voxel_of(v));
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int i = i0 + r;
                    const bool kept = i < T && cm[i] == 0;
                    const real cur = kept ? yv[i] : real(0);
                    const real prv = (i > 0 && i - 1 < T && cm[i - 1] == 0) ? yv[i - 1] : real(0);
                    dy[r] = i < T ? cur - prv : real(0);
                    w[r] = (p.w0 && i < T) ? p.w0[v * T + i] : real(0);
                    keep |= (unsigned)kept << r;
                }
            } else {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int i = i0 + r;
                    const real cur = i < T ? yv[i] : real(0);
                    const real prv = (i > 0 && i - 1 < T) ? yv[i - 1] : real(0);
                    dy[r] = i < T ? cur - prv : real(0);
                    w[r] = (p.w0 && i < T) ? p.w0[v * T + i] : real(0);
                }
            }
            // res <- M res
            auto censor_res = [&](real (&res)[R]) {
#pragma unroll
                for (int r = 0; r < R; ++r) res[r] = (keep >> r) & 1u ? res[r] : real(0);
            };
            // ||M res||^2, res itself unchanged (the final residual gives x)
            auto sumsq_kept = [&](const real (&res)[R]) {
                real rm[R];
#pragma unroll
                for (int r = 0; r < R; ++r) rm[r] = res[r];
                censor_res(rm);
                return sumsq(rm);
            };
#pragma unroll
            for (int j = 0; j < KMAX; ++j) h[j] = j < K ? hv[j] : real(0);
            const double Lc = p.L_of(v);
            NoiseLoop nl;
            if (AUTO) nl.start(win);
            double n_kept = (double)T, zero = 0.0;
            if (AUTO && CENSOR) {
                n_kept = (double)__popc(keep);
                ct.cta_sum2(n_kept, zero);
            }
            double lam = AUTO ? nl.lbda : p.lam_of(v);
            const real step = (real)(1.0 / Lc);
            real th = (real)(lam / Lc);
            real *Jv = p.out_J + v * (int64_t)p.nb_iter;
            const bool trace = !AUTO && p.out_J;
            int n_done = 0, ring_pos = 0;
            real res[R];
            for (;;) {   // one pass (AUTO: one per outer iteration)
                n_done = 0;
                ring_pos = 0;
                for (int k = 0; k < p.nb_iter; ++k) {
                    forward(res);
                    if constexpr (CENSOR) censor_res(res);
                    // cost of the previous iterate: its residual has just been formed; the warp sums ride on B3
                    if (trace && k > 0) ct.publish2(sumsq(res), sumabs(w));
                    real g[R];
                    adjoint(res, g);
                    if (trace && k > 0 && tid == 0) {
                        double s2, s1;
                        ct.gather2(s2, s1);
                        Jv[k - 1] = (real)(0.5 * s2 + lam * s1);
                    }
                    const real ob = real(1) + beta[k];
                    real *slot = ring + (size_t)ring_pos * R * L::NT;    // ring_pos = k % nring
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const real u = fma(-step, g[r], w[r]);
                        const real cl = fmin(fmax(u, -th), th);
                        w[r] = fma(-ob, cl, u);
                        if (es) slot[r * L::NT] = u;
                    }
                    n_done = k + 1;
                    if (es && k > p.wind) {
                        // xx = [u_{k-wind+2}, ..., u_k, w_k]; old = mean(first wind-sub), new = mean(last sub)
                        const real inv_old = real(1) / real(p.wind - sub), inv_new = real(1) / real(sub);
                        real so[R], sn[R];
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            so[r] = 0;
                            sn[r] = w[r];
                        }
                        int pos = ring_pos + 1 == nring ? 0 : ring_pos + 1;   // (k - wind + 2) % nring: oldest u
                        for (int m = 0; m < p.wind - 1; ++m) {
                            const real *s = ring + (size_t)pos * R * L::NT;
                            pos = pos + 1 == nring ? 0 : pos + 1;
                            const bool is_old = m < p.wind - sub;
#pragma unroll
                            for (int r = 0; r < R; ++r) {
                                const real uu = s[r * L::NT];
                                if (is_old) so[r] += uu; else sn[r] += uu;
                            }
                        }
                        real qn = 0, qd = 0;              // thread partials in `real`, warp sums in double
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const real mo = so[r] * inv_old, mn = sn[r] * inv_new;
                            qn = fma(mn - mo, mn - mo, qn);
                            qd = fma(mn, mn, qd);
                        }
                        double pn = (double)qn, pd = (double)qd;
                        ct.cta_sum2(pn, pd);
                        if (sqrt(pn) / (sqrt(pd) + 1.0e-10) < p.tol) break;
                    }
                    if (es) ring_pos = ring_pos + 1 == nring ? 0 : ring_pos + 1;
                }
                forward(res);
                double rr = CENSOR ? sumsq_kept(res) : sumsq(res), gg = sumabs(w);
                ct.cta_sum2(rr, gg);
                if (AUTO) {
                    if (!nl.pass_done<CENSOR>(p, v, rr, gg, tid == 0, tid, L::NT, n_kept)) {
                        lam = nl.lbda;
                        th = (real)(lam / Lc);
                        continue;
                    }
                } else if (n_done > 0 && tid == 0) {
                    if (p.out_J) Jv[n_done - 1] = (real)(0.5 * rr + lam * gg);
                    if (p.out_r) p.out_r[v] = (real)rr;
                    if (p.out_g) p.out_g[v] = (real)gg;
                }
                break;
            }
            real z[R];
#pragma unroll
            for (int r = 0; r < R; ++r) z[r] = w[r];
            ct.scan_fwd_cta(z);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int i = i0 + r;
                if (i < T) {
                    if constexpr (CENSOR)                     // x = A w - y0 + y0, y0 = y zeroed on censored scans
                        p.out_x[v * T + i] = res[r] + ((keep >> r) & 1u ? yv[i] : real(0));
                    else
                        p.out_x[v * T + i] = res[r] + yv[i];  // x = (A w - y) + y
                    p.out_z[v * T + i] = z[r];
                    p.out_dz[v * T + i] = w[r];
                }
            }
            if (tid == 0 && !AUTO) p.out_niter[v] = n_done;
        }
        if (p.queue) {
            __syncthreads();
            if (tid == 0) next_task = atomicAdd(p.queue, 1u);
            __syncthreads();
            v = (int64_t)gridDim.x + (int64_t)next_task;
        } else {
            v += gridDim.x;
        }
    }
}

template <int R, int KMAX, int NW>
bool fastc_shape_ok(int T, int K) {
    // the last used thread may be partial, threads beyond it idle; up to half of the threads may idle
    // (the dispatcher picks the variant with the fewest slots among those that match)
    // (the smallest variants of the many-tap families, one warp of R = 4, also take everything shorter;
    // with K <= 32 short series are better served by the group / warp kernels)
    // the many-tap families (KMAX >= 40) only serve K > 28: with fewer taps the K <= 28 variants, the group
    // and the warp kernels are the better choice
    return K <= KMAX && (KMAX <= 32 || K > 28) && T <= NW * 32 * R &&
           (T > NW * 16 * R - R || (NW == 1 && R == 4)) && T >= 1;
}

// ES: bd(early_stopping=True), which needs no shared memory beyond the kernel without it
template <typename real, int R, int KMAX, int NW, int MINB, bool ES = false>
int fast_bdc_launch(const BdArgs<real> &a, cudaStream_t stream) {
    using L = CtaLayout<real, R, KMAX, NW>;
    return launch_persistent(fast_bdc_kernel<real, R, KMAX, NW, MINB, ES>, NW * 32, L::bytes(a.nb_iter), 1, a.V,
                             a.queue, stream, a);
}

template <typename real, int R, int KMAX, int NW, int MINB>
int fast_bdc_wave(int nb_iter) {
    using L = CtaLayout<real, R, KMAX, NW>;
    return wave_voxels(fast_bdc_kernel<real, R, KMAX, NW, MINB>, NW * 32, L::bytes(nb_iter), 1);
}

// FAST_NO_MATCH when the early-stopping ring does not fit: the generic kernel decides
template <typename real, int R, int KMAX, int NW, int MINB, bool AUTO = false, bool CENSOR = false>
int fast_deconvc_launch_c(const DeconvArgs<real> &a, const Censor &cz, cudaStream_t stream) {
    using L = CtaLayout<real, R, KMAX, NW>;
    const int ring_rows = a.early_stopping && a.wind >= 2 ? a.wind - 1 : 0;
    return launch_persistent(fast_deconvc_kernel<real, R, KMAX, NW, MINB, AUTO, CENSOR>, NW * 32,
                             L::deconv_bytes(a.nb_iter, ring_rows, AUTO ? a.wind : 0), 1, a.V, a.queue, stream, a,
                             ring_rows, cz);
}

template <typename real, int R, int KMAX, int NW, int MINB, bool AUTO = false>
int fast_deconvc_launch(const DeconvArgs<real> &a, cudaStream_t stream) {
    return fast_deconvc_launch_c<real, R, KMAX, NW, MINB, AUTO>(a, Censor{}, stream);
}

// censored calls run on the CTA rows only; below T = 181 no row of at most 32 taps serves a series, and the many-tap
// rows take K <= 28 there too, with zero-padded taps (pb_fast_registry.cu: pick_censored)
template <int R, int KMAX, int NW>
bool fastc_censored_ok(int T, int K) {
    return fastc_shape_ok<R, KMAX, NW>(T, K) || (KMAX > 32 && K <= 28 && T <= 180 && fastc_shape_ok<R, KMAX, NW>(T, 29));
}

template <typename real, int R, int KMAX, int NW, int MINB>
constexpr Variant<real> cta_variant() {
    return {TIER_GROUP_CTA, 32 * NW, R, KMAX, 0, false, fastc_shape_ok<R, KMAX, NW>,
            fast_bdc_launch<real, R, KMAX, NW, MINB>, fast_bdc_launch<real, R, KMAX, NW, MINB, true>,
            fast_deconvc_launch<real, R, KMAX, NW, MINB>,
            fast_bdc_wave<real, R, KMAX, NW, MINB>, fast_deconvc_launch<real, R, KMAX, NW, MINB, true>,
            fastc_censored_ok<R, KMAX, NW>, fast_deconvc_launch_c<real, R, KMAX, NW, MINB, false, true>,
            fast_deconvc_launch_c<real, R, KMAX, NW, MINB, true, true>};
}

}  // namespace pb
