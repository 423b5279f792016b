// Register-tiled persistent bd kernel, GROUP variant: a warp is split into 32/G groups of G lanes,
// one voxel per group (G = 32, 16 or 8), lane q of a group owns the R contiguous samples
// [q R, q R + R) of its voxel in registers (G R >= T).
//
// Why groups: the per-lane work of an iteration is 2 R K FFMA + ~9 R element-wise ops, while the
// halo exchange costs 2 (K-1) SHFL and the scans 2 log2(G) SHFL+FADD *per lane whatever R is*.
// A larger R per lane (fewer lanes per voxel) therefore amortises the non-FFMA instructions:
// T = 300, K = 20:  G = 32, R = 10  ->  624 issued instructions per voxel-iteration (measured)
//                   G = 16, R = 19  ->  ~530
// and no lane idles (16 x 19 = 304 slots for 300 samples instead of 320).
//
// Same recursion as pb_fast.cuh (see there); differences:
//  * shuffles / scans / reductions are segmented (width G);
//  * only the last TAIL slots of a lane can lie beyond T (dispatcher guarantees G R - T <= TAIL), so
//    the tail select costs TAIL instead of R instructions;
//  * tap 0 of the dilated SPM HRF is identically zero (s = -dt < 0, pybold/hrf_model.py:25-30), so
//    the bd kernel starts its tap loops at j = 1;
//  * the Lipschitz / theta phases (double, O(K^2)) run for all groups of the warp in lock step
//    (pb_theta_group.cuh): measured, running them group after group cost 14 % of the kernel.
// Early stopping (Q6/Q7) makes groups diverge: fast_bdg_kernel<..., ES = true> (below) lets a group that has
// stopped wait for its neighbour.
//
// Reference code replaced: pybold/bold_signal.py:242-278, :281-382.
#pragma once
#include "pb_fast_registry.h"
#include "pb_generic.cuh"
#include "pb_theta_group.cuh"
#include "pb_tile.cuh"

namespace pb {

// inc <- inc + (value of lane q-d if q >= d), segmented scan step without the ISETP/FSEL pair:
// shfl.up returns the lane's own value together with a false predicate when the source is out of
// the segment.
__device__ __forceinline__ float seg_scan_step_up(float inc, int d, int c) {
    float out;
    asm volatile(
        "{ .reg .f32 r0; .reg .pred p;\n"
        "  shfl.sync.up.b32 r0|p, %1, %2, %3, 0xffffffff;\n"
        "  @p add.f32 r0, r0, %1;\n"
        "  mov.f32 %0, r0; }\n"
        : "=f"(out) : "f"(inc), "r"(d), "r"(c));
    return out;
}
__device__ __forceinline__ float seg_scan_step_down(float inc, int d, int c) {
    float out;
    asm volatile(
        "{ .reg .f32 r0; .reg .pred p;\n"
        "  shfl.sync.down.b32 r0|p, %1, %2, %3, 0xffffffff;\n"
        "  @p add.f32 r0, r0, %1;\n"
        "  mov.f32 %0, r0; }\n"
        : "=f"(out) : "f"(inc), "r"(d), "r"(c));
    return out;
}

// source order of the unrolled tile (pb_tile.cuh), picked with the register-file model of
// profiles/r01_rf_bandwidth.txt on fast_bdg_kernel<float, 19, 20, 16, 8, 4, 3> and timed on a B200
#ifndef PB_CONV_JDESC
#define PB_CONV_JDESC 1
#endif
#ifndef PB_CONV_RDESC
#define PB_CONV_RDESC 0
#endif
#ifndef PB_CORR_JDESC
#define PB_CORR_JDESC 1
#endif
#ifndef PB_CORR_RDESC
#define PB_CORR_RDESC 1
#endif
#ifndef PB_CONV_DS
#define PB_CONV_DS 0
#endif
#ifndef PB_CORR_DS
#define PB_CORR_DS 0
#endif
#ifndef PB_CONV_RB
#define PB_CONV_RB 7
#endif
#ifndef PB_CORR_RB
#define PB_CORR_RB 7
#endif

// sqrt(x) for x >= 0 to double accuracy: float rsqrt estimate, one Newton step in double (6 FP64
// instructions instead of the ~35 of the IEEE sequence; relative error ~1e-14)
__device__ __forceinline__ double sqrt_refined(double x) {
    if (!(x > 1.0e-300)) return x > 0.0 ? sqrt(x) : 0.0;
    const float xf = (float)x;
    if (!(xf > 1.0e-30f) || !(xf < 1.0e30f)) return sqrt(x);
    const double r0 = (double)rsqrtf(xf);
    const double r1 = r0 * fma(-0.5 * x, r0 * r0, 1.5);
    const double r2 = r1 * fma(-0.5 * x, r1 * r1, 1.5);
    return x * r2;
}

template <typename real, int G>
struct Seg {
    static __device__ __forceinline__ real sum(real v) {
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(PB_FULL, v, o, G);
        return v;
    }
    // exclusive prefix over the lanes of the group
    static __device__ __forceinline__ real excl_up(real v, int q) {
        real inc = v;
#pragma unroll
        for (int d = 1; d < G; d <<= 1) {
            const real t = __shfl_up_sync(PB_FULL, inc, d, G);
            if (q >= d) inc += t;
        }
        const real ex = __shfl_up_sync(PB_FULL, inc, 1, G);
        return q == 0 ? real(0) : ex;
    }
    static __device__ __forceinline__ real excl_down(real v, int q) {
        real inc = v;
#pragma unroll
        for (int d = 1; d < G; d <<= 1) {
            const real t = __shfl_down_sync(PB_FULL, inc, d, G);
            if (q + d < G) inc += t;
        }
        const real ex = __shfl_down_sync(PB_FULL, inc, 1, G);
        return q == G - 1 ? real(0) : ex;
    }
};
template <int G>
struct Seg<float, G> {
    static __device__ __forceinline__ float sum(float v) {
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(PB_FULL, v, o, G);
        return v;
    }
    static __device__ __forceinline__ float excl_up(float v, int q) {
        float inc = v;
#pragma unroll
        for (int d = 1; d < G; d <<= 1) inc = seg_scan_step_up(inc, d, (32 - G) << 8);
        const float ex = __shfl_up_sync(PB_FULL, inc, 1, G);
        return q == 0 ? 0.f : ex;
    }
    static __device__ __forceinline__ float excl_down(float v, int q) {
        float inc = v;
#pragma unroll
        for (int d = 1; d < G; d <<= 1) inc = seg_scan_step_down(inc, d, ((32 - G) << 8) | 0x1f);
        const float ex = __shfl_down_sync(PB_FULL, inc, 1, G);
        return q == G - 1 ? 0.f : ex;
    }
};

// LEAN = true keeps only the iterate in registers: dy lives in shared memory ([r][lane], one
// conflict-free LDS per sample and iteration) and the taps are fetched four at a time (LDS.128,
// broadcast within the group) right before their R FFMA each.  ~40 registers less per thread, i.e.
// more resident warps to hide the scan / shuffle latencies, for ~3 % more instructions.
// SMH = true exchanges the K-1 halo samples through shared memory instead of shuffles: every lane
// stores its R values as 16-byte vectors into a per-voxel buffer framed by zero pads and loads the
// preceding / following samples as vectors (R % 4 == 0).  10 + 10 instead of 38 + 38 instructions
// per convolution pair at K = 20 and no boundary selects; measured +17 % at T = 600 (pb_fastc.cuh).
// SMH = 2 ("blocked") does the same for ANY R: every lane owns a 16-byte aligned block of RP >= R floats
// (RP / 4 odd, so that the 16-byte accesses of a quarter warp fall into distinct banks), stores its R
// values there (ceil(R / 4) STS.128) and reads the blocks of the lanes before / after it (LDS.128).  The
// lanes at the ends of a group read a block of zeros instead, picked once per kernel through a pointer:
// no boundary selects.  K = 20, R = 19: 5 + 5 instead of 19 SHFL + 19 FSEL per exchange.
#ifndef PB_HALO_PRED
#define PB_HALO_PRED 0
#endif
#ifdef PB_LEAN_KEEP_TAPS
constexpr bool kLeanTaps = false;   // experiment: LEAN moves only dy to shared memory
#else
constexpr bool kLeanTaps = true;
#endif
template <typename real, int R, int KMAX, int G, int TAIL, int J0, int LEAN = 0, int SMH = 0>
struct GroupVoxel {
    static constexpr bool LT = LEAN == 1 && kLeanTaps;   // LEAN = 2 keeps the taps in registers
    static_assert(SMH != 1 || R % 4 == 0, "SMH = 1 moves 16-byte vectors of a contiguous copy");
    static constexpr int NH = (KMAX - 1 + 3) / 4;   // vectors per halo
    struct alignas(4 * sizeof(real)) V4 { real t[4]; };
    real *myA;                     // SMH: this lane's R slots in the iterate buffer
    real *myB;                     // SMH: this lane's R slots in the residual buffer
    static constexpr int RP4 = ((R + 3) / 4) | 1;            // vectors per block (odd)
    static constexpr int RP = 4 * RP4;                       // SMH = 2: floats per lane block
    static constexpr int DUP = (KMAX - 1 + R - 1) / R;       // lanes a halo reaches into
    const real *upsrc[SMH == 2 ? DUP : 1];   // SMH = 2: block of lane q - d in the iterate buffer (or zeros)
    const real *dnsrc[SMH == 2 ? DUP : 1];   // SMH = 2: block of lane q + d in the residual buffer (or zeros)
    static_assert(G == 8 || G == 16 || G == 32, "group width");
    static_assert(TAIL >= 0 && TAIL <= R, "tail");
    static_assert(LEAN != 1 || KMAX % 4 == 0, "LEAN = 1 fetches taps as 16-byte vectors");
    real w[R];                     // iterate (the reference's diff_z)
    real dy[LEAN ? 1 : R];         // y[i] - y[i-1]            (registers unless LEAN)
    real h[LT ? 1 : KMAX];         // taps, zero beyond K       (registers unless LEAN)
    real *dy_s;                    // LEAN: dy[r] at dy_s[r * 32]  (pointer already offset by lane)
    const real *h_s;               // LEAN: this group's KMAX taps, 16-byte aligned
    int nvalid;                    // samples (< T) this lane holds
    int q;                         // lane within the group
    // PRED (PB_HALO_PRED): no select after the halo shuffles; the FFMA consuming a halo value of hop d is
    // predicated on the existence of lane q -+ d (pb_tile.cuh: fma_if)
    static constexpr bool PRED = PB_HALO_PRED != 0 && SMH == 0 && !LT && sizeof(real) == 4;
    unsigned ok_up[DUP], ok_dn[DUP];

    __device__ __forceinline__ void init(int lane, int T) {
        q = lane & (G - 1);
        nvalid = max(0, min(R, T - q * R));
#pragma unroll
        for (int d = 1; d <= DUP; ++d) {
            ok_up[d - 1] = q >= d ? 1u : 0u;
            ok_dn[d - 1] = q + d < G ? 1u : 0u;
        }
    }
    // SMH = 2: store the R values as ceil(R / 4) vectors (the pad of the last one is never used)
    __device__ __forceinline__ void put_block(real *dst, const real (&a)[R]) const {
#pragma unroll
        for (int c = 0; c < (R + 3) / 4; ++c) {
            V4 t;
#pragma unroll
            for (int e = 0; e < 4; ++e) t.t[e] = a[4 * c + e < R ? 4 * c + e : R - 1];
            reinterpret_cast<V4 *>(dst)[c] = t;
        }
    }
    __device__ __forceinline__ void put(real *dst, const real (&a)[R]) const {
#pragma unroll
        for (int r4 = 0; r4 < R / 4; ++r4) {
            V4 t;
#pragma unroll
            for (int e = 0; e < 4; ++e) t.t[e] = a[4 * r4 + e];
            reinterpret_cast<V4 *>(dst)[r4] = t;
        }
    }
    // halo[m-1] = a at voxel index (q R - m), zero before the series starts
    // (RAW: for the inner loop of a PRED build -- values of non-existent lanes are left in, see fma_if)
    template <bool RAW = false>
    __device__ __forceinline__ void halo_up(const real (&a)[R], real (&halo)[KMAX - 1]) const {
        if constexpr (SMH == 2) {
            put_block(myA, a);
            __syncwarp();
#pragma unroll
            for (int d = 1; d <= DUP; ++d) {
                // halo[m - 1], (d - 1) R < m <= min(d R, KMAX - 1), is element d R - m of lane q - d
                constexpr int dummy = 0;
                (void)dummy;
                const int m_hi = d * R < KMAX - 1 ? d * R : KMAX - 1;
                const int rr_lo = d * R - m_hi;
#pragma unroll
                for (int c = rr_lo / 4; c <= (R - 1) / 4; ++c) {
                    const V4 t = reinterpret_cast<const V4 *>(upsrc[d - 1])[c];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int rr = 4 * c + e;
                        const int m = d * R - rr;
                        if (rr >= rr_lo && rr < R) halo[m >= 1 && m <= KMAX - 1 ? m - 1 : 0] = t.t[e];
                    }
                }
            }
            return;
        }
        if constexpr (SMH == 1) {
            put(myA, a);
            __syncwarp();
#pragma unroll
            for (int c = 0; c < NH; ++c) {
                const V4 t = reinterpret_cast<const V4 *>(myA)[-1 - c];
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (4 * c + (3 - e) < KMAX - 1) halo[4 * c + (3 - e) < KMAX - 1 ? 4 * c + (3 - e) : 0] = t.t[e];
            }
            return;
        }
#pragma unroll
        for (int m = 1; m < KMAX; ++m) {
            const int d = (m + R - 1) / R;
            const int rr = d * R - m;
            const real t = __shfl_up_sync(PB_FULL, a[rr], d, G);
            halo[m - 1] = (RAW && PRED) ? t : (q >= d ? t : real(0));
        }
    }
    // halo[k] = a at voxel index (q R + R + k), zero past the last lane of the group
    template <bool RAW = false>
    __device__ __forceinline__ void halo_down(const real (&a)[R], real (&halo)[KMAX - 1]) const {
        if constexpr (SMH == 2) {
            put_block(myB, a);
            __syncwarp();
#pragma unroll
            for (int d = 1; d <= DUP; ++d) {
                // halo[k], (d - 1) R <= k < min(d R, KMAX - 1), is element k - (d - 1) R of lane q + d
                const int k_hi = d * R < KMAX - 1 ? d * R : KMAX - 1;
                const int n = k_hi - (d - 1) * R;
#pragma unroll
                for (int c = 0; c < (n + 3) / 4; ++c) {
                    const V4 t = reinterpret_cast<const V4 *>(dnsrc[d - 1])[c];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int rr = 4 * c + e;
                        const int k = (d - 1) * R + rr;
                        if (rr < n) halo[k < KMAX - 1 ? k : 0] = t.t[e];
                    }
                }
            }
            return;
        }
        if constexpr (SMH == 1) {
            put(myB, a);
            __syncwarp();
#pragma unroll
            for (int c = 0; c < NH; ++c) {
                const V4 t = reinterpret_cast<const V4 *>(myB + R)[c];
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (4 * c + e < KMAX - 1) halo[4 * c + e < KMAX - 1 ? 4 * c + e : 0] = t.t[e];
            }
            return;
        }
#pragma unroll
        for (int k = 0; k < KMAX - 1; ++k) {
            const int d = (R + k) / R;
            const int rr = (R + k) - d * R;
            const real t = __shfl_down_sync(PB_FULL, a[rr], d, G);
            halo[k] = (RAW && PRED) ? t : (q + d < G ? t : real(0));
        }
    }
    struct alignas(4 * sizeof(real)) Tap4 { real t[4]; };
    template <int JS>
    __device__ __forceinline__ void conv_acc(const real (&a)[R], const real (&halo)[KMAX - 1],
                                             real (&acc)[R]) const {
        if constexpr (LT) {
#pragma unroll
            for (int jj = 0; jj < KMAX / 4; ++jj) {
                const Tap4 t4 = reinterpret_cast<const Tap4 *>(h_s)[jj];
#pragma unroll
                for (int jx = 0; jx < 4; ++jx) {
                    const int j = 4 * jj + jx;
                    if (j < JS) continue;
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const int idx = r - j;
                        const real val = idx >= 0 ? a[idx >= 0 ? idx : 0] : halo[idx >= 0 ? 0 : -idx - 1];
                        acc[r] = fma(t4.t[jx], val, acc[r]);
                    }
                }
            }
        } else {
            tile_conv<real, R, KMAX, KMAX - 1, JS, PB_CONV_JDESC, PB_CONV_RDESC, PB_CONV_RB, PB_CONV_DS, PRED>(h, a, halo, acc, ok_up);
        }
    }
    template <int JS>
    __device__ __forceinline__ void corr_acc(const real (&a)[R], const real (&halo)[KMAX - 1],
                                             real (&acc)[R]) const {
        if constexpr (LT) {
#pragma unroll
            for (int jj = 0; jj < KMAX / 4; ++jj) {
                const Tap4 t4 = reinterpret_cast<const Tap4 *>(h_s)[jj];
#pragma unroll
                for (int jx = 0; jx < 4; ++jx) {
                    const int j = 4 * jj + jx;
                    if (j < JS) continue;
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const int idx = r + j;
                        const real val = idx < R ? a[idx < R ? idx : 0] : halo[idx < R ? 0 : idx - R];
                        acc[r] = fma(t4.t[jx], val, acc[r]);
                    }
                }
            }
        } else {
            tile_corr<real, R, KMAX, KMAX - 1, JS, PB_CORR_JDESC, PB_CORR_RDESC, PB_CORR_RB, PB_CORR_DS, PRED>(h, a, halo, acc, ok_dn);
        }
    }
    __device__ __forceinline__ void scan_fwd(real (&a)[R]) const {
#pragma unroll
        for (int r = 1; r < R; ++r) a[r] += a[r - 1];
        const real carry = Seg<real, G>::excl_up(a[R - 1], q);
#pragma unroll
        for (int r = 0; r < R; ++r) a[r] += carry;
    }
    // zero the slots at and beyond T (only the last TAIL slots of a lane can be)
    __device__ __forceinline__ void mask_tail(real (&a)[R]) const {
#pragma unroll
        for (int r = R - TAIL; r < R; ++r) a[r] = r < nvalid ? a[r] : real(0);
    }
    // res <- A w - y
    __device__ __forceinline__ void forward(real (&res)[R]) const {
        real halo[KMAX - 1];
        halo_up<true>(w, halo);
#pragma unroll
        for (int r = 0; r < R; ++r) res[r] = LEAN ? -dy_s[r * 32] : -dy[LEAN ? 0 : r];
        conv_acc<J0>(w, halo, res);
#pragma unroll
        for (int r = 1; r < R; ++r) res[r] += res[r - 1];
        const real carry = Seg<real, G>::excl_up(res[R - 1], q);
#pragma unroll
        for (int r = 0; r < R; ++r) res[r] += carry;
        mask_tail(res);
    }
    // g <- A^T res
    __device__ __forceinline__ void adjoint(const real (&res)[R], real (&g)[R]) const {
        real halo[KMAX - 1];
        halo_down<true>(res, halo);
#pragma unroll
        for (int r = 0; r < R; ++r) g[r] = real(0);
        corr_acc<J0>(res, halo, g);
#pragma unroll
        for (int r = R - 2; r >= 0; --r) g[r] += g[r + 1];
        const real carry = Seg<real, G>::excl_down(g[0], q);
#pragma unroll
        for (int r = 0; r < R; ++r) g[r] += carry;
    }
    __device__ __forceinline__ void update(const real (&g)[R], real step, real th, real beta) {
        const real ob = real(1) + beta;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const real u = fma(-step, g[r], w[r]);
            const real cl = fmin(fmax(u, -th), th);
            w[r] = fma(-ob, cl, u);
        }
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
    // taps of this group's voxel from the double scratch (call with the whole warp converged)
    __device__ __forceinline__ void load_taps(const double *hs, int K) {
        if constexpr (LT) {
            __syncwarp();
            for (int j = q; j < KMAX; j += G) const_cast<real *>(h_s)[j] = j < K ? (real)hs[j] : real(0);
            __syncwarp();
        } else {
#pragma unroll
            for (int j = 0; j < KMAX; ++j) h[LT ? 0 : j] = j < K ? (real)hs[j] : real(0);
        }
    }
    __device__ __forceinline__ void load_y(const real *yv, int T, real (&y)[R]) const {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = q * R + r;
            y[r] = i < T ? yv[i] : real(0);
        }
    }
    __device__ __forceinline__ void set_dy(const real *yv, int T) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = q * R + r;
            const real cur = i < T ? yv[i] : real(0);
            const real prv = (i > 0 && i - 1 < T) ? yv[i - 1] : real(0);
            const real d = i < T ? cur - prv : real(0);
            if (LEAN) dy_s[r * 32] = d; else dy[LEAN ? 0 : r] = d;
        }
    }
    __device__ __forceinline__ void store(real *dst, const real (&a)[R], int T, bool on) const {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = q * R + r;
            if (on && i < T) dst[i] = a[r];
        }
    }
};

template <int R, int KMAX, int G>
__host__ __device__ constexpr int fastg_halo_buf() { return 2 * ((KMAX + 3) & ~3) + G * R; }

template <int R>
__host__ __device__ constexpr int fastg_block_floats() { return 4 * (((R + 3) / 4) | 1); }

template <typename real, int R, int KMAX, int G, int LEAN, int SMH = 0>
__host__ __device__ constexpr size_t fastg_warp_bytes() {
    return (size_t)(32 / G) * pb_scratch_doubles(KMAX) * sizeof(double) +
           (LEAN ? ((size_t)R * 32 + (size_t)(32 / G) * KMAX) * sizeof(real) : 0) +
           (SMH == 1 ? (size_t)2 * (32 / G) * fastg_halo_buf<R, KMAX, G>() * sizeof(real) : 0) +
           (SMH == 2 ? (size_t)(2 * 32 + 1) * fastg_block_floats<R>() * sizeof(real) : 0);
}

// ES = true: the reference's `early_stopping=True` (non-default).  Q6 -- the inner loop of a voxel stops at
// iteration j > 2 once ||w_j - u_j|| / (||w_j|| + 1e-10) < tol -- and Q7 -- the outer loop stops on the signed
// change of the windowed means of J and runs one last pass -- are decided per GROUP; a group whose inner loop has
// stopped keeps its iterate (predicated update) until its neighbour's has, a group whose voxel is finished
// idles until its neighbour is (the double-precision phases stay in lock step for the warp), then the warp
// takes the next task.  With ES = false none of this is compiled in.
template <typename real, int R, int KMAX, int G, int TAIL, int WARPS, int MINB, int LEAN = 0,
          int SMH = 0, bool ES = false>
__global__ void __launch_bounds__(WARPS * 32, MINB)
fast_bdg_kernel(BdArgs<real> p) {
    constexpr int VPW = 32 / G;
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int grp = lane / G;
    real *beta = reinterpret_cast<real *>(smem);
    const size_t beta_bytes = ((size_t)p.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    fill_momentum_table(beta, p.nb_iter);
    unsigned char *wbase = smem + beta_bytes + (size_t)warp * fastg_warp_bytes<real, R, KMAX, G, LEAN, SMH>();
    ThetaScratch scs[VPW];
#pragma unroll
    for (int g = 0; g < VPW; ++g)
        scs[g].bind(reinterpret_cast<double *>(wbase) + (size_t)g * pb_scratch_doubles(KMAX), KMAX);
    ThetaScratch sc = scs[0];
#pragma unroll
    for (int g = 1; g < VPW; ++g)
        if (grp == g) sc = scs[g];
    const int T = p.T, K = p.K, ntr = p.nb_iter + 2;

    GroupVoxel<real, R, KMAX, G, TAIL, 1, LEAN, SMH> vx;
    vx.init(lane, T);
    if constexpr (SMH == 2) {
        using GV = GroupVoxel<real, R, KMAX, G, TAIL, 1, LEAN, SMH>;
        constexpr int RP = GV::RP;
        real *hb = reinterpret_cast<real *>(wbase + fastg_warp_bytes<real, R, KMAX, G, LEAN, 0>());
        for (int i = lane; i < (2 * 32 + 1) * RP; i += 32) hb[i] = real(0);
        real *bufA = hb, *bufB = hb + 32 * RP, *zeros = hb + 64 * RP;
        vx.myA = bufA + lane * RP;
        vx.myB = bufB + lane * RP;
#pragma unroll
        for (int d = 1; d <= GV::DUP; ++d) {
            vx.upsrc[d - 1] = vx.q >= d ? bufA + (lane - d) * RP : zeros;
            vx.dnsrc[d - 1] = vx.q + d < G ? bufB + (lane + d) * RP : zeros;
        }
        __syncwarp();
    }
    if constexpr (SMH == 1) {
        constexpr int PADH = (KMAX + 3) & ~3, BUFV = fastg_halo_buf<R, KMAX, G>();
        real *hb = reinterpret_cast<real *>(wbase + fastg_warp_bytes<real, R, KMAX, G, LEAN, false>());
        for (int i = lane; i < 2 * VPW * BUFV; i += 32) hb[i] = real(0);   // zero pads (and slots)
        vx.myA = hb + grp * BUFV + PADH + vx.q * R;
        vx.myB = hb + (VPW + grp) * BUFV + PADH + vx.q * R;
        __syncwarp();
    }
    if (LEAN) {
        real *lean = reinterpret_cast<real *>(wbase + (size_t)VPW * pb_scratch_doubles(KMAX) * sizeof(double));
        vx.h_s = lean + grp * KMAX;
        vx.dy_s = lean + VPW * KMAX + lane;
    }
    const int q = vx.q;
    // task = VPW consecutive voxels; the first task of a warp is static, the following ones come from the
    // work queue when there is one (tasks finish at different times as soon as anything else runs on the
    // GPU, e.g. the NCCL gather of the previous step), else from the usual grid stride
    const int64_t n_static = (int64_t)gridDim.x * WARPS;
    for (int64_t task = (int64_t)blockIdx.x * WARPS + warp; task * VPW < p.V;) {
        const int64_t v0 = task * VPW;
        if (p.queue) {
            unsigned int nxt = 0;
            if (lane == 0) nxt = atomicAdd(p.queue, 1u);
            task = n_static + (int64_t)__shfl_sync(PB_FULL, nxt, 0);
        } else {
            task += n_static;
        }
        const bool on = v0 + grp < p.V;                 // idle groups replay the last voxel
        const int64_t v = on ? v0 + grp : p.V - 1;
        const real *yv = p.y + v * T;
        vx.set_dy(yv, T);
        const double lam = (double)p.lbda[v * p.lbda_stride];
        double theta = (double)p.theta0[v * p.theta0_stride];
        hrf_eval_group<G>(theta, p.grid, sc, q);           // bold_signal.py:292 (theta_0 itself: Q9)
        vx.load_taps(sc.hs, K);
        double r0, g0;
        {
            real y[R];
            vx.load_y(yv, T, y);
            if (p.z0) {                                   // bold_signal.py:298-301
                const real *zv = p.z0 + v * T;
                real z[R], hal[KMAX - 1], xr[R];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int i = q * R + r;
                    z[r] = i < T ? zv[i] : real(0);
                    vx.w[r] = (i > 0 && i < T) ? zv[i] - zv[i - 1] : real(0);
                    xr[r] = -y[r];
                }
                vx.halo_up(z, hal);
                vx.template conv_acc<1>(z, hal, xr);
                vx.mask_tail(xr);
                r0 = (double)Seg<real, G>::sum(vx.partial_sumsq(xr));
                g0 = (double)Seg<real, G>::sum(vx.partial_sumabs(vx.w));
            } else {
#pragma unroll
                for (int r = 0; r < R; ++r) vx.w[r] = real(0);
                r0 = (double)Seg<real, G>::sum(vx.partial_sumsq(y));
                g0 = 0.0;
            }
        }
        const double j0 = r0 + lam * g0;
        real *Jv = p.out_J + v * (int64_t)ntr, *rv = p.out_r + v * (int64_t)ntr,
             *gv = p.out_g + v * (int64_t)ntr;
        const bool writer = on && q == 0;
#ifdef PB_DEBUG_EVALS
        int dbg_evals = 0;
#endif
        if (writer) {
            Jv[0] = real(1);
            rv[0] = real(1);
            gv[0] = (real)g0;
        }
        bool live = on, stopped = false;                  // ES: per-group progress
        int n_tr = 1;                                     // ES: trace entries written so far
        double sumJ = 1.0;
        for (int idx = 0; idx <= p.nb_iter; ++idx) {
            // final deconvolution, :365-376 (ES: also the pass after the outer stop fired, :350-362)
            const bool last = ES ? (stopped || idx == p.nb_iter) : idx == p.nb_iter;
            const double Lc = frob_lipschitz_group<G>(sc, K, T, q);
            const real step = (real)(1.0 / Lc), th = (real)(lam / Lc);
            if constexpr (!ES) {
                for (int j = 0; j < p.nb_iter; ++j) {     // _loops_deconv, :259-276
                    real res[R], gr[R];
                    vx.forward(res);
                    vx.adjoint(res, gr);
                    vx.update(gr, step, th, beta[j]);
                }
            } else {
                bool frozen = !live;
                for (int j = 0; j < p.nb_iter; ++j) {
                    real res[R], gr[R];
                    vx.forward(res);
                    vx.adjoint(res, gr);
                    const real ob = real(1) + beta[j];
                    real pc = 0, pw = 0;
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const real u = fma(-step, gr[r], vx.w[r]);
                        const real cl = fmin(fmax(u, -th), th);
                        const real wn = fma(-ob, cl, u);
                        pc = fma(cl, cl, pc);
                        pw = fma(wn, wn, pw);
                        vx.w[r] = frozen ? vx.w[r] : wn;
                    }
                    const double sc2 = (double)Seg<real, G>::sum(pc), sw2 = (double)Seg<real, G>::sum(pw);
                    // Q6 (:267-273): ||w_j - u_j|| = (1 + beta_j) ||clamp(u_j)||
                    const double num = (1.0 + (double)beta[j]) * sqrt_refined(sc2);
                    if (j > 2 && num < p.tol * (sqrt_refined(sw2) + 1.0e-10)) frozen = true;
                    if (__all_sync(PB_FULL, frozen)) break;
                }
            }
            real z[R], hal[KMAX - 1], y[R];
#pragma unroll
            for (int r = 0; r < R; ++r) z[r] = vx.w[r];
            vx.scan_fwd(z);
            vx.halo_up(z, hal);
            vx.load_y(yv, T, y);
            if (ES ? __any_sync(PB_FULL, !last) : !last) {
                // ---- theta step (:329-334): b = Z^T y, Rz = autocorrelation of z ----
                // (ES: in lock step for the warp; a group in its last pass keeps its theta and taps)
                real zm[R];
#pragma unroll
                for (int r = 0; r < R; ++r) zm[r] = z[r];
                vx.mask_tail(zm);
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
                    pb_ = Seg<real, G>::sum(pb_);
                    pr = Seg<real, G>::sum(pr);
                    if (q == 0 && a < K) {
                        sc.b[a] = (double)pb_;
                        sc.Rz[a] = (double)pr;
                    }
                }
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int pidx = T - 1 - (q * R + r);
                    if (pidx >= 0 && pidx < K) sc.zend[pidx] = (double)z[r];
                }
                for (int a = q; a < K; a += G)
                    if (a >= T) sc.zend[a] = 0.0;
                __syncwarp();
                gram_build_group<G>(sc, K, q);
#ifdef PB_DEBUG_EVALS
                int ne = 0;
                const double th_new = theta_solve_group<G>(theta, p.theta_lo, p.theta_hi, p.grid, sc, q, &ne);
                dbg_evals += ne;
#else
                const double th_new = theta_solve_group<G>(theta, p.theta_lo, p.theta_hi, p.grid, sc, q, nullptr);
#endif
                theta = (ES && last) ? theta : th_new;
                hrf_eval_group<G>(theta, p.grid, sc, q);
                vx.load_taps(sc.hs, K);
            }
            // ---- cost trace: x = h * z with the (new) taps ----
            real xr[R];
#pragma unroll
            for (int r = 0; r < R; ++r) xr[r] = -y[r];
            vx.template conv_acc<1>(z, hal, xr);
            vx.mask_tail(xr);
            const double rr = (double)Seg<real, G>::sum(vx.partial_sumsq(xr));
            const double gg = (double)Seg<real, G>::sum(vx.partial_sumabs(vx.w));
            const double eps = last ? 0.0 : 1.0e-30;
            if constexpr (!ES) {
                if (writer) {
                    Jv[idx + 1] = (real)((rr + lam * gg) / j0 + eps);
                    rv[idx + 1] = (real)(rr / r0 + eps);
                    gv[idx + 1] = (real)gg;
                }
                if (last) {
#pragma unroll
                    for (int r = 0; r < R; ++r) xr[r] += y[r];
                    vx.store(p.out_x + v * T, xr, T, on);
                    vx.store(p.out_z + v * T, z, T, on);
                    vx.store(p.out_dz + v * T, vx.w, T, on);
                }
            } else {
                const double Jn = (rr + lam * gg) / j0 + eps;
                if (writer && live) {
                    Jv[n_tr] = (real)Jn;
                    rv[n_tr] = (real)(rr / r0 + eps);
                    gv[n_tr] = (real)gg;
                }
                if (live) {
                    sumJ += (double)(real)Jn;
                    ++n_tr;
                }
                if (last && live) {                       // this voxel is done: everything it returns, now
#pragma unroll
                    for (int r = 0; r < R; ++r) xr[r] += y[r];
                    vx.store(p.out_x + v * T, xr, T, true);
                    vx.store(p.out_z + v * T, z, T, true);
                    vx.store(p.out_dz + v * T, vx.w, T, true);
                    for (int a = q; a < K; a += G) p.out_h[v * K + a] = (real)sc.hs[a];
                    if (q == 0) {
                        p.out_theta[v] = (real)theta;
                        p.out_ntrace[v] = n_tr;
                    }
                    live = false;
                }
                __syncwarp();
                if (idx > p.wind) {                       // Q7 (:350-362); warp-uniform condition
                    int stop = 0;
                    if (live && q == 0) stop = bd_outer_stop(Jv, n_tr, sumJ, p.wind / 2, p.tol) ? 1 : 0;
                    stop = __shfl_sync(PB_FULL, stop, 0, G);
                    if (live) stopped = stop != 0;
                }
                if (!__any_sync(PB_FULL, live)) break;
            }
            __syncwarp();
        }
        if constexpr (!ES) {
            if (on)
                for (int a = q; a < K; a += G) p.out_h[v * K + a] = (real)sc.hs[a];
            if (writer) {
                p.out_theta[v] = (real)theta;
#ifdef PB_DEBUG_EVALS
                p.out_ntrace[v] = dbg_evals;
#else
                p.out_ntrace[v] = ntr;
#endif
            }
        }
        __syncwarp();
    }
}

template <typename real, int R, int KMAX, int G, int TAIL, int WARPS, int MINB, int LEAN = 0,
          int SMH = 0>
int fast_bdg_wave(int nb_iter) {
    const size_t beta_bytes = ((size_t)nb_iter * sizeof(real) + 15) & ~(size_t)15;
    const size_t smem = beta_bytes + (size_t)WARPS * fastg_warp_bytes<real, R, KMAX, G, LEAN, SMH>();
    return wave_voxels(fast_bdg_kernel<real, R, KMAX, G, TAIL, WARPS, MINB, LEAN, SMH>, WARPS * 32, smem,
                       WARPS * (32 / G));
}

// ------------------------------------------------------------------------------------------------
// deconv, fixed lambda, no early stopping (pybold/bold_signal.py:49-97), group layout.
// Taps are the caller's (tap 0 is not assumed zero); J_k is taken from the residual that iteration
// k+1 forms anyway (two segmented sums per iteration).
// ------------------------------------------------------------------------------------------------
template <typename real, int R, int KMAX, int G, int TAIL, int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
fast_deconvg_kernel(DeconvArgs<real> p) {
    constexpr int VPW = 32 / G;
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int grp = lane / G;
    real *beta = reinterpret_cast<real *>(smem);
    fill_momentum_table(beta, p.nb_iter);
    const int T = p.T, K = p.K;
    GroupVoxel<real, R, KMAX, G, TAIL, 0> vx;
    vx.init(lane, T);
    const int q = vx.q;
    for (int64_t v0 = ((int64_t)blockIdx.x * WARPS + warp) * VPW; v0 < p.V;
         v0 += (int64_t)gridDim.x * WARPS * VPW) {
        const bool on = v0 + grp < p.V && p.is_active(v0 + grp < p.V ? v0 + grp : p.V - 1);
        if (!__any_sync(PB_FULL, on)) continue;
        const int64_t v = on ? v0 + grp : p.V - 1;
        const real *yv = p.y_row(v);
        const real *hv = p.h_row(v);
        vx.set_dy(yv, T);
#pragma unroll
        for (int j = 0; j < KMAX; ++j) vx.h[j] = j < K ? hv[j] : real(0);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = q * R + r;
            vx.w[r] = (p.w0 && i < T) ? p.w0[v * T + i] : real(0);
        }
        const double Lc = p.L_of(v);
        const double lam = p.lam_of(v);
        const real step = (real)(1.0 / Lc), th = (real)(lam / Lc);
        real *Jv = p.out_J + v * (int64_t)p.nb_iter;
        const bool writer = on && q == 0;
        const bool tracer = writer && p.out_J;
        real res[R];
        for (int k = 0; k < p.nb_iter; ++k) {
            vx.forward(res);
            if (k > 0) {
                const double J = 0.5 * (double)Seg<real, G>::sum(vx.partial_sumsq(res)) +
                                 lam * (double)Seg<real, G>::sum(vx.partial_sumabs(vx.w));
                if (tracer) Jv[k - 1] = (real)J;
            }
            real g[R];
            vx.adjoint(res, g);
            vx.update(g, step, th, beta[k]);
        }
        vx.forward(res);
        {
            const double rr = (double)Seg<real, G>::sum(vx.partial_sumsq(res));
            const double gg = (double)Seg<real, G>::sum(vx.partial_sumabs(vx.w));
            const double J = 0.5 * rr + lam * gg;
            if (tracer) Jv[p.nb_iter - 1] = (real)J;
            if (writer && p.out_r) p.out_r[v] = (real)rr;
            if (writer && p.out_g) p.out_g[v] = (real)gg;
        }
        real y[R], z[R];
        vx.load_y(yv, T, y);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            y[r] += res[r];
            z[r] = vx.w[r];
        }
        vx.scan_fwd(z);
        vx.store(p.out_x + v * T, y, T, on);
        vx.store(p.out_z + v * T, z, T, on);
        vx.store(p.out_dz + v * T, vx.w, T, on);
        if (writer) p.out_niter[v] = p.nb_iter;
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// deconv with EARLY STOPPING (the reference's default call, pybold/bold_signal.py:13, :82-95; Q5), group
// layout.  Iteration counts differ from voxel to voxel, so
//  * every group of a warp runs its own voxel at its own iteration k (own momentum weight, own ring
//    position, own stop test); a group whose voxel stops -- or reaches nb_iter -- stores it and
//  * pulls the next voxel from an atomic work queue (p.queue) while its neighbour group carries on.
// The warp executes one common instruction stream (the iteration body); only the per-voxel prologue /
// epilogue is predicated.  Results cannot depend on which group solves a voxel: the arithmetic of a
// voxel only involves its own G lanes, in the same lane order.
// Ring of the past u's (Q5 window): [slot][lane][RP] in shared memory, every lane reads and writes its
// own 16-byte aligned block with vector accesses (RP / 4 odd: conflict free).
// AUTO: deconv(lbda=None).  A group keeps its voxel through every outer iteration of the noise loop
// (pb_noise_loop.cuh): where an inner pass ends, it updates lambda and starts the next pass in the same turn
// from the residual just formed, so only the final pass of a voxel costs the neighbour group a turn.  The
// windows of alphas (wind doubles per group) follow the rings in shared memory.
// ------------------------------------------------------------------------------------------------
template <typename real, int R, int KMAX, int G, int TAIL, int WARPS, int MINB, bool AUTO = false>
__global__ void __launch_bounds__(WARPS * 32, MINB)
fast_deconvg_es_kernel(DeconvArgs<real> p, int ring_rows) {
    using GV = GroupVoxel<real, R, KMAX, G, TAIL, 0>;
    using V4 = typename GV::V4;
    constexpr int RP = GV::RP, NV = (R + 3) / 4;
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    real *beta = reinterpret_cast<real *>(smem);
    const size_t beta_bytes = ((size_t)p.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    fill_momentum_table(beta, p.nb_iter);
    real *ring = reinterpret_cast<real *>(smem + beta_bytes) + ((size_t)warp * ring_rows * 32 + lane) * RP;
    const int T = p.T, K = p.K;
    const int sub = p.wind / 2, nring = p.wind - 1;
    const real inv_old = real(1) / real(p.wind - sub), inv_new = real(1) / real(sub);
    const bool even_wind = p.wind - sub == sub;
    const bool es_on = p.early_stopping != 0;
    GV vx;
    vx.init(lane, T);
    const int q = vx.q;
#pragma unroll
    for (int r = 0; r < R; ++r) vx.w[r] = vx.dy[r] = real(0);
#pragma unroll
    for (int j = 0; j < KMAX; ++j) vx.h[j] = real(0);
    // per-group state (identical in the G lanes of a group)
    int64_t v = 0;
    int k = 0, ring_pos = 0;
    bool active = false, want = true;
    double lam = 0.0;
    real step = 0, th = 0;
    NoiseLoop nl;
    for (;;) {
        if (__any_sync(PB_FULL, want)) {
            unsigned int idx = 0xffffffffu;
            if (want && q == 0) {
                do {                                    // skip the problems masked out by p.active
                    idx = atomicAdd(p.queue, 1u);
                } while ((int64_t)idx < p.V && !p.is_active(idx));
            }
            idx = __shfl_sync(PB_FULL, idx, 0, G);
            if (want) {
                want = false;
                active = (int64_t)idx < p.V;
                if (active) {
                    v = idx;
                    const real *hv = p.h_row(v);
                    vx.set_dy(p.y_row(v), T);
#pragma unroll
                    for (int j = 0; j < KMAX; ++j) vx.h[j] = j < K ? hv[j] : real(0);
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const int i = q * R + r;
                        vx.w[r] = (p.w0 && i < T) ? p.w0[v * T + i] : real(0);
                    }
                    const double Lc = p.L_of(v);
                    if constexpr (AUTO) {
                        nl.start(reinterpret_cast<double *>(smem + beta_bytes + (size_t)WARPS * ring_rows * 32 * RP *
                                                                                    sizeof(real)) +
                                 (size_t)(warp * (32 / G) + lane / G) * p.wind);
                        lam = nl.lbda;
                    } else {
                        lam = p.lam_of(v);
                    }
                    step = (real)(1.0 / Lc);
                    th = (real)(lam / Lc);
                    k = 0;
                    ring_pos = 0;
                }
            }
        }
        if (!__any_sync(PB_FULL, active)) break;
        real *Jv = p.out_J + v * (int64_t)p.nb_iter;
        // ---- stop test of the iteration just done (reference iteration k - 1; Q5), evaluated at the START of
        // the next turn: xx = [u_{k-wind+1}, ..., u_{k-1}, w_k] with w_k the iterate in registers.  Its long
        // dependent tail (window sums -> norms -> segmented sums -> one square root -> vote) sits in the same
        // basic block as the forward pass below and overlaps with its FFMA.  Always computed (the first turns
        // read an unfilled ring and are ignored).
        real qn[4] = {0, 0, 0, 0}, qd[4] = {0, 0, 0, 0};
        {
            real so[R], sn[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                so[r] = 0;
                sn[r] = vx.w[r];
            }
            int pos = ring_pos;                                        // oldest u of this group's window
            auto add_slot = [&](real (&acc)[R]) {
                const real *slot = ring + (size_t)pos * 32 * RP;
                pos = pos + 1 == nring ? 0 : pos + 1;
#pragma unroll
                for (int c = 0; c < NV; ++c) {
                    const V4 t = reinterpret_cast<const V4 *>(slot)[c];
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        if (4 * c + e < R) acc[4 * c + e < R ? 4 * c + e : 0] += t.t[e];
                }
            };
            for (int m = 0; m < p.wind - sub; ++m) add_slot(so);
            for (int m = p.wind - sub; m < p.wind - 1; ++m) add_slot(sn);
            if (even_wind) {
                // both means are over wind / 2 entries: the common factor 1 / sub is applied to the norms
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const real df = sn[r] - so[r];
                    qn[r & 3] = fma(df, df, qn[r & 3]);
                    qd[r & 3] = fma(sn[r], sn[r], qd[r & 3]);
                }
            } else {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const real mo = so[r] * inv_old, mn = sn[r] * inv_new;
                    qn[r & 3] = fma(mn - mo, mn - mo, qn[r & 3]);
                    qd[r & 3] = fma(mn, mn, qd[r & 3]);
                }
            }
        }
        real res[R];
        vx.forward(res);
        bool stop;
        {
            const double scale = even_wind ? (double)inv_new * (double)inv_new : 1.0;
            const double pn = scale * (double)Seg<real, G>::sum((qn[0] + qn[1]) + (qn[2] + qn[3]));
            const double pd = scale * (double)Seg<real, G>::sum((qd[0] + qd[1]) + (qd[2] + qd[3]));
            // ||new - old|| / (||new|| + 1e-10) < tol  <=>  pn < (tol (sqrt(pd) + 1e-10))^2, with the one
            // square root from a float estimate refined in double (no FP64 sqrt / division sequences)
            const double rhs = p.tol * (sqrt_refined(pd) + 1.0e-10);
            stop = es_on && k - 1 > p.wind && pn < rhs * rhs;
        }
        if constexpr (!AUTO) {   // cost of the previous iterate: its residual has just been formed.  For a
                                 // closing voxel k is the number of iterations done and this is its last cost.
            const double J = 0.5 * (double)Seg<real, G>::sum(vx.partial_sumsq(res)) +
                             lam * (double)Seg<real, G>::sum(vx.partial_sumabs(vx.w));
            if (active && q == 0 && k > 0 && p.out_J) Jv[k - 1] = (real)J;
        }
        bool closing = active && k > 0 && (stop || k == p.nb_iter);
        if constexpr (AUTO) if (__any_sync(PB_FULL, closing)) {
            // an inner pass has ended; unless it was the voxel's final pass, the next one starts here: the
            // residual just formed is that of its starting iterate (iteration 0 below)
            const double rr = (double)Seg<real, G>::sum(vx.partial_sumsq(res));
            const double gg = (double)Seg<real, G>::sum(vx.partial_sumabs(vx.w));
            if (closing && !nl.pass_done(p, v, rr, gg, q == 0, q, G)) {
                closing = false;
                lam = nl.lbda;
                th = (real)(lam / p.L_of(v));
                k = 0;
                ring_pos = 0;
            }
        }
        if (__any_sync(PB_FULL, closing)) {
            // The iterate in registers is final for this voxel and the residual just formed is its own: store
            // it and hand the group back to the queue; the neighbour group loses this turn's forward pass
            // (its iterate is untouched), once per voxel.
            real z[R];
#pragma unroll
            for (int r = 0; r < R; ++r) z[r] = vx.w[r];
            vx.scan_fwd(z);
            // the two terms of the last cost, summed again like above (same values) rather than carried
            // through every turn in registers
            double rr = 0.0, gg = 0.0;
            if (p.out_r || p.out_g) {
                rr = (double)Seg<real, G>::sum(vx.partial_sumsq(res));
                gg = (double)Seg<real, G>::sum(vx.partial_sumabs(vx.w));
            }
            if (closing) {
                if constexpr (!AUTO) if (q == 0) p.out_niter[v] = k;
                if (q == 0 && p.out_r) p.out_r[v] = (real)rr;
                if (q == 0 && p.out_g) p.out_g[v] = (real)gg;
                real y[R];
                vx.load_y(p.y_row(v), T, y);
#pragma unroll
                for (int r = 0; r < R; ++r) y[r] += res[r];          // x = (A w - y) + y
                vx.store(p.out_x + v * T, y, T, true);
                vx.store(p.out_z + v * T, z, T, true);
                vx.store(p.out_dz + v * T, vx.w, T, true);
                active = false;
                want = true;
            }
            continue;
        }
        real g[R], u[R];
        vx.adjoint(res, g);
        {
            const real ob = real(1) + beta[k < p.nb_iter ? k : p.nb_iter - 1];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                u[r] = fma(-step, g[r], vx.w[r]);
                const real cl = fmin(fmax(u[r], -th), th);
                vx.w[r] = fma(-ob, cl, u[r]);
            }
        }
        {   // u_k into the ring slot k % nring; afterwards ring_pos points at the oldest entry again
            real *slot = ring + (size_t)ring_pos * 32 * RP;
#pragma unroll
            for (int c = 0; c < NV; ++c) {
                V4 t;
#pragma unroll
                for (int e = 0; e < 4; ++e) t.t[e] = u[4 * c + e < R ? 4 * c + e : R - 1];
                reinterpret_cast<V4 *>(slot)[c] = t;
            }
        }
        // k = iterations done; groups without a voxel iterate on stale registers, keep their indices in range
        k = k < p.nb_iter ? k + 1 : k;
        ring_pos = ring_pos + 1 == nring ? 0 : ring_pos + 1;
    }
}

// AUTO (deconv(lbda=None)) always runs the early-stopping kernel: its launcher sets wind >= 2
template <typename real, int R, int KMAX, int G, int TAIL, int WARPS, int MINB, bool AUTO = false>
int fast_deconvg_launch(const DeconvArgs<real> &a, cudaStream_t stream) {
    constexpr int VPW = 32 / G;
    const size_t beta_bytes = ((size_t)a.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    if (AUTO || (a.early_stopping && a.wind >= 2)) {
        if (!a.queue) return FAST_NO_MATCH;
        const int ring_rows = a.wind - 1;
        const size_t smem = beta_bytes + (size_t)WARPS * ring_rows * 32 * fastg_block_floats<R>() * sizeof(real) +
                            (AUTO ? (size_t)WARPS * VPW * a.wind * sizeof(double) : 0);
        return launch_persistent(fast_deconvg_es_kernel<real, R, KMAX, G, TAIL, WARPS, MINB, AUTO>, WARPS * 32,
                                 smem, WARPS * VPW, a.V, a.queue, stream, a, ring_rows);
    }
    return launch_persistent(fast_deconvg_kernel<real, R, KMAX, G, TAIL, WARPS, MINB>, WARPS * 32, beta_bytes,
                             WARPS * VPW, a.V, nullptr, stream, a);
}

template <int R, int KMAX, int G, int TAIL>
bool fastg_shape_ok(int T, int K) {
    // short-series variants (G = 8, or G = 16 with R <= 12; TAIL = R: every slot maskable) serve T down to half
    // their slots; the others tolerate at most TAIL dead slots, all in the last lane
    const bool short_series = TAIL == R && (G == 8 || (G == 16 && R <= 12));
    return K <= KMAX && T <= G * R && (short_series ? 2 * T > G * R : G * R - T <= TAIL) && T >= 1;
}

template <typename real, int R, int KMAX, int G, int TAIL, int WARPS, int MINB, int LEAN = 0,
          int SMH = 0, bool ES = false>
int fast_bdg_launch(const BdArgs<real> &a, cudaStream_t stream) {
    const size_t beta_bytes = ((size_t)a.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    const size_t smem = beta_bytes + (size_t)WARPS * fastg_warp_bytes<real, R, KMAX, G, LEAN, SMH>();
    return launch_persistent(fast_bdg_kernel<real, R, KMAX, G, TAIL, WARPS, MINB, LEAN, SMH, ES>, WARPS * 32, smem,
                             WARPS * (32 / G), a.V, a.queue, stream, a);
}

template <typename real, int R, int KMAX, int G, int TAIL, int WARPS, int MINB>
constexpr Variant<real> group_variant() {
    return {TIER_GROUP_CTA, G, R, KMAX, TAIL, false, fastg_shape_ok<R, KMAX, G, TAIL>,
            fast_bdg_launch<real, R, KMAX, G, TAIL, WARPS, MINB>,
            fast_bdg_launch<real, R, KMAX, G, TAIL, WARPS, MINB, 0, 0, true>,
            fast_deconvg_launch<real, R, KMAX, G, TAIL, WARPS, MINB>,
            fast_bdg_wave<real, R, KMAX, G, TAIL, WARPS, MINB>,
            fast_deconvg_launch<real, R, KMAX, G, TAIL, WARPS, MINB, true>};
}

}  // namespace pb
