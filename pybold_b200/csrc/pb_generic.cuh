// Generic solver kernels: one warp per voxel, the voxel's arrays resident in shared memory,
// run-time T and K.  This is the any-shape path (T <= PB_MAX_T, K <= PB_MAX_K, float or double)
// used when no register-tiled instantiation (pb_fast.cuh) matches; it executes the same
// recursion, Lipschitz formula and theta step, so it doubles as an independent implementation
// the fast kernels are tested against.
//
// Reference code replaced: pybold/bold_signal.py:49-97 (deconv), :242-278 (_loops_deconv),
// :281-382 (bd); quirks Q1-Q9 of SURVEY.md section 8 are reproduced on purpose.
#pragma once
#include "pb_device.cuh"
#include "pb_noise_loop.cuh"

namespace pb {

template <typename real>
struct GenVoxel {
    real *ws;    // iterate w (the reference's diff_z)
    real *ys;    // observed signal
    real *as;    // scratch: z = cumsum(w), then c / gradient
    real *bs;    // scratch: residual A w - y
    real *hr;    // taps in signal precision
    real *ring;  // (wind-1) x T history of u for deconv's early stop (Q5); may be null
    int T, K, lane;

    // in-place inclusive prefix sum over a[0..T)
    __device__ __forceinline__ void scan_fwd(real *a) const {
        const int ch = (T + 31) >> 5;
        const int i0 = min(lane * ch, T), i1 = min(i0 + ch, T);
        real s = 0;
        for (int i = i0; i < i1; ++i) {
            s += a[i];
            a[i] = s;
        }
        const real carry = warp_excl_scan_up(s, lane);
        for (int i = i0; i < i1; ++i) a[i] += carry;
        __syncwarp();
    }
    // in-place inclusive suffix sum
    __device__ __forceinline__ void scan_rev(real *a) const {
        const int ch = (T + 31) >> 5;
        const int i0 = min(lane * ch, T), i1 = min(i0 + ch, T);
        real s = 0;
        for (int i = i1 - 1; i >= i0; --i) {
            s += a[i];
            a[i] = s;
        }
        const real carry = warp_excl_scan_down(s, lane);
        for (int i = i0; i < i1; ++i) a[i] += carry;
        __syncwarp();
    }
    // out[i] = sum_j h[j] in[i-j]  (- sub[i] when sub != null)
    __device__ __forceinline__ void conv(const real *in, const real *sub, real *out) const {
        for (int i = lane; i < T; i += 32) {
            real acc = sub ? -sub[i] : real(0);
            const int jm = min(K - 1, i);
            for (int j = 0; j <= jm; ++j) acc = fma(hr[j], in[i - j], acc);
            out[i] = acc;
        }
        __syncwarp();
    }
    // out[i] = sum_j h[j] in[i+j]
    __device__ __forceinline__ void corr(const real *in, real *out) const {
        for (int i = lane; i < T; i += 32) {
            real acc = 0;
            const int jm = min(K - 1, T - 1 - i);
            for (int j = 0; j <= jm; ++j) acc = fma(hr[j], in[i + j], acc);
            out[i] = acc;
        }
        __syncwarp();
    }
    // as <- z = cumsum(w);  bs <- A w - y
    __device__ __forceinline__ void forward() const {
        for (int i = lane; i < T; i += 32) as[i] = ws[i];
        __syncwarp();
        scan_fwd(as);
        conv(as, ys, bs);
    }
    // as <- A^T bs
    __device__ __forceinline__ void adjoint() const {
        corr(bs, as);
        scan_rev(as);
    }
    // u = w - step g; c = clamp(u, -th, th); w <- u - (1 + beta) c   (== v + beta (v - u), v = u - c)
    // Returns (sum c^2, sum w^2) partials when `norms` (bd's inner early stop, Q6).
    __device__ __forceinline__ void update(real step, real th, real beta, real *u_out,
                                           bool norms, double &sc2, double &sw2) const {
        double pc = 0.0, pw = 0.0;
        const real ob = real(1) + beta;
        for (int i = lane; i < T; i += 32) {
            const real u = fma(-step, as[i], ws[i]);
            const real c = fmin(fmax(u, -th), th);
            const real w = fma(-ob, c, u);
            ws[i] = w;
            if (u_out) u_out[i] = u;
            if (norms) {
                pc += (double)c * (double)c;
                pw += (double)w * (double)w;
            }
        }
        if (norms) {
            sc2 = warp_sum(pc);
            sw2 = warp_sum(pw);
        }
        __syncwarp();
    }
    __device__ __forceinline__ double sumsq(const real *a) const {
        double p = 0.0;
        for (int i = lane; i < T; i += 32) p += (double)a[i] * (double)a[i];
        return warp_sum(p);
    }
    __device__ __forceinline__ double sumabs(const real *a) const {
        double p = 0.0;
        for (int i = lane; i < T; i += 32) p += fabs((double)a[i]);
        return warp_sum(p);
    }
    // inner loop of bd (_loops_deconv, bold_signal.py:259-276)
    __device__ __forceinline__ void inner_loop(const real *beta, int nb_iter, real step, real th,
                                               bool es, double tol) const {
        for (int j = 0; j < nb_iter; ++j) {
            forward();
            adjoint();
            double sc2 = 0.0, sw2 = 0.0;
            const bool chk = es && j > 2;
            update(step, th, beta[j], nullptr, chk, sc2, sw2);
            if (chk) {
                // ||w_j - u_j|| = (1 + beta_j) ||c||
                const double num = (1.0 + (double)beta[j]) * sqrt(sc2);
                if (num / (sqrt(sw2) + 1.0e-10) < tol) break;
            }
        }
    }
    __device__ __forceinline__ void load_taps(const ThetaScratch &sc) const {
        for (int a = lane; a < K; a += 32) hr[a] = (real)sc.hs[a];
        __syncwarp();
    }
    // b = Z^T y, Rz = autocorrelation of z, zend = reversed tail of z  (z in `as`)
    __device__ __forceinline__ void theta_moments(ThetaScratch &sc) const {
        for (int a = 0; a < K; ++a) {
            double pb_ = 0.0, pr = 0.0;
            for (int i = a + lane; i < T; i += 32) {
                const double zz = (double)as[i - a];
                pb_ = fma((double)ys[i], zz, pb_);
                pr = fma((double)as[i], zz, pr);
            }
            pb_ = warp_sum(pb_);
            pr = warp_sum(pr);
            if (lane == 0) {
                sc.b[a] = pb_;
                sc.Rz[a] = pr;
            }
        }
        for (int p = lane; p < K; p += 32) sc.zend[p] = (T - 1 - p >= 0) ? (double)as[T - 1 - p] : 0.0;
        __syncwarp();
    }
};

struct GenLayout {
    int tp;           // padded T (multiple of 4)
    int kp;           // padded K (multiple of 4)
    int ring_rows;    // wind - 1 for deconv with early stopping, else 0
    int ring_smem;    // how many of them live in shared memory; up to three of the rest use the voxel's own
                      // output rows (out_x, out_z, out_dz: free until the final store) as scratch
    size_t doubles;   // per-warp scratch doubles
    size_t reals;     // per-warp reals
    __host__ __device__ static GenLayout make(int T, int K, int ring_rows, bool with_theta) {
        GenLayout l;
        l.tp = (T + 3) & ~3;
        l.kp = (K + 3) & ~3;
        l.ring_rows = ring_rows;
        l.ring_smem = ring_rows;
        l.doubles = with_theta ? (size_t)pb_scratch_doubles(l.kp) : (size_t)(3 * l.kp);
        l.reals = (size_t)4 * l.tp + l.kp + (size_t)ring_rows * l.tp;
        return l;
    }
    // move one more ring row out of shared memory; false when no output row is left to take it
    __host__ bool spill_ring_row() {
        if (ring_smem == 0 || ring_rows - ring_smem >= 3) return false;
        --ring_smem;
        reals -= (size_t)tp;
        return true;
    }
    __host__ __device__ size_t warp_bytes(size_t real_size) const {
        return doubles * sizeof(double) + ((reals * real_size + 7) & ~(size_t)7);
    }
};

template <typename real>
__device__ __forceinline__ GenVoxel<real> gen_bind(unsigned char *warp_base, const GenLayout &l,
                                                   int T, int K, int lane, double *&scratch) {
    scratch = reinterpret_cast<double *>(warp_base);
    real *r = reinterpret_cast<real *>(warp_base + l.doubles * sizeof(double));
    GenVoxel<real> g;
    g.ws = r;
    g.ys = r + l.tp;
    g.as = r + 2 * l.tp;
    g.bs = r + 3 * l.tp;
    g.hr = r + 4 * l.tp;
    g.ring = l.ring_rows ? r + 4 * l.tp + l.kp : nullptr;
    g.T = T;
    g.K = K;
    g.lane = lane;
    return g;
}

// ------------------------------------------------------------------------------------------------
// deconv, fixed lambda
// ------------------------------------------------------------------------------------------------
template <typename real>
struct DeconvArgs {
    const real *y, *h;
    int64_t h_stride;
    const real *L;
    int64_t L_stride;
    const real *lbda;
    int64_t lbda_stride;
    const real *w0;
    int nb_iter, early_stopping, wind;
    double tol;
    real *out_x, *out_z, *out_dz, *out_J;
    int32_t *out_niter;
    int64_t V;
    int T, K;
    // optional [V] terms of the final cost J = 0.5 R + lambda G of the returned iterate w (null: not written):
    // R = ||x - y||^2 = ||A w - y||^2, G = ||w||_1
    real *out_r = nullptr, *out_g = nullptr;
    // regularisation path (cfg5): problem p = l * y_mod + v solves voxel v with lambda l.  y_mod > 0 makes
    // the problems share the voxel's y row, taps row and Lipschitz constant (voxel p % y_mod) instead of a
    // replicated copy, lbda_div > 0 takes lbda[p / lbda_div].  Both 0: one voxel and one lbda (element
    // stride lbda_stride) per problem.
    int64_t y_mod = 0, lbda_div = 0;
    // early-stopping group kernel: device counter (zeroed on the launch stream) the groups pull voxels from
    unsigned int *queue = nullptr;
    // optional mask: problems with active[v] == 0 are skipped, their outputs stay untouched (the outer loop
    // of deconv(lbda=None) keeps calling with fewer and fewer live voxels); out_J may be null (no cost trace)
    const unsigned char *active = nullptr;
    // deconv(lbda=None) (nb_outer > 0, kernels instantiated with AUTO): lambda follows the noise level
    // sigma[v * sigma_stride] through at most nb_outer outer iterations (pb_noise_loop.cuh) instead of coming from
    // lbda; nb_iter stays the inner count.  out_J, out_R, out_G are [V, nb_outer] (NaN past the voxel's outer
    // count), out_lbda [V] the last lambda, out_nouter [V] the outer count; each may be null.
    const real *sigma = nullptr;
    int64_t sigma_stride = 0;
    int nb_outer = 0;
    real *out_R = nullptr, *out_G = nullptr, *out_lbda = nullptr;
    int32_t *out_nouter = nullptr;
    __device__ __forceinline__ bool is_active(int64_t v) const { return !active || active[v] != 0; }
    __device__ __forceinline__ int64_t voxel_of(int64_t v) const { return y_mod ? v % y_mod : v; }
    __device__ __forceinline__ const real *y_row(int64_t v) const { return y + voxel_of(v) * T; }
    // taps row and Lipschitz constant of the problem's voxel (h_stride / L_stride 0: shared)
    __device__ __forceinline__ const real *h_row(int64_t v) const { return h + voxel_of(v) * h_stride; }
    __device__ __forceinline__ double L_of(int64_t v) const { return (double)L[voxel_of(v) * L_stride]; }
    __device__ __forceinline__ double lam_of(int64_t v) const {
        return (double)lbda[lbda_div ? v / lbda_div : v * lbda_stride];
    }
};

// Scan censoring (pb_deconv_censored_*): m[voxel * stride + i] != 0 leaves scan i of the voxel out of the data term,
// min 1/2 ||M (A w - y)||^2 + lbda ||w||_1 with M = diag(1 - censor).  y reads as 0 on censored scans (NaN there is
// ignored); x = A w is still written on every scan.  Kernels take it as their last parameter and read it only in
// their CENSOR instances.
struct Censor {
    const unsigned char *m = nullptr;
    int64_t stride = 0;       // 0: one mask shared by the batch
    __device__ __forceinline__ const unsigned char *row(int64_t voxel) const { return m + voxel * stride; }
};

// AUTO: deconv(lbda=None), one inner pass per outer iteration of the noise loop, then the final pass; the
// window of alphas lives in the warp's scratch doubles.  CENSOR: the residual is masked with cz before the adjoint
// and the cost terms, and the noise target is n_kept sigma^2.
template <typename real, bool AUTO = false, bool CENSOR = false>
__global__ void generic_deconv_kernel(DeconvArgs<real> p, GenLayout lay, Censor cz) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    real *beta = reinterpret_cast<real *>(smem);
    const size_t beta_bytes = ((size_t)p.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    fill_momentum_table(beta, p.nb_iter);
    unsigned char *base = smem + beta_bytes + (size_t)warp * lay.warp_bytes(sizeof(real));
    double *scratch;
    GenVoxel<real> g = gen_bind<real>(base, lay, p.T, p.K, lane, scratch);
    const int T = p.T, K = p.K;
    const bool es = p.early_stopping && p.wind >= 2;
    const int sub = p.wind / 2, nring = p.wind - 1;

    for (int64_t v = (int64_t)blockIdx.x * nwarp + warp; v < p.V; v += (int64_t)gridDim.x * nwarp) {
        if (!p.is_active(v)) continue;
        const real *yv = p.y_row(v);
        const real *hv = p.h_row(v);
        const unsigned char *cm = CENSOR ? cz.row(p.voxel_of(v)) : nullptr;
        double n_kept = (double)T;
        if constexpr (CENSOR) {
            int nk = 0;
            for (int i = lane; i < T; i += 32) {
                const bool kept = cm[i] == 0;
                g.ys[i] = kept ? yv[i] : real(0);
                g.ws[i] = p.w0 ? p.w0[v * T + i] : real(0);
                nk += kept;
            }
            n_kept = warp_sum((double)nk);
        } else {
            for (int i = lane; i < T; i += 32) {
                g.ys[i] = yv[i];
                g.ws[i] = p.w0 ? p.w0[v * T + i] : real(0);
            }
        }
        // bs <- M bs (CENSOR), after forward() and before the adjoint and the cost sums
        auto censor_res = [&]() {
            if constexpr (CENSOR) {
                for (int i = lane; i < T; i += 32)
                    if (cm[i]) g.bs[i] = real(0);
                __syncwarp();
            }
        };
        for (int a = lane; a < K; a += 32) g.hr[a] = hv[a];
        __syncwarp();
        const double Lc = p.L_of(v);
        NoiseLoop nl;
        if (AUTO) nl.start(scratch);
        double lam = AUTO ? nl.lbda : p.lam_of(v);
        const real step = (real)(1.0 / Lc);
        real th = (real)(lam / Lc);
        real *Jv = p.out_J + v * (int64_t)p.nb_iter;
        // ring row r: shared memory, or (long series in double) this voxel's output rows until the final store;
        // a lane only ever reads back the elements it wrote itself
        auto ring_row = [&](int r) -> real * {
            if (r < lay.ring_smem) return g.ring + (size_t)r * lay.tp;
            const int o = r - lay.ring_smem;
            return (o == 0 ? p.out_x : (o == 1 ? p.out_z : p.out_dz)) + v * T;
        };
        int n_done = 0;
        for (;;) {   // one pass (AUTO: one per outer iteration)
            n_done = 0;
            for (int k = 0; k < p.nb_iter; ++k) {
                g.forward();
                censor_res();
                if (!AUTO && k > 0) {
                    const double J = 0.5 * g.sumsq(g.bs) + lam * g.sumabs(g.ws);
                    if (lane == 0 && p.out_J) Jv[k - 1] = (real)J;
                }
                g.adjoint();
                double d0, d1;
                real *uslot = es ? ring_row(k % nring) : nullptr;
                g.update(step, th, beta[k], uslot, false, d0, d1);
                n_done = k + 1;
                if (es && k > p.wind) {
                    // xx = [u_{k-wind+2}, ..., u_k, w_k]; old = mean(first wind-sub), new = mean(last sub)
                    double pn = 0.0, pd = 0.0;
                    const real inv_old = real(1) / real(p.wind - sub), inv_new = real(1) / real(sub);
                    for (int i = lane; i < T; i += 32) {
                        real so = 0, sn = 0;
                        for (int m = 0; m < p.wind - 1; ++m) {
                            const int j = k - p.wind + 2 + m;
                            const real u = ring_row(j % nring)[i];
                            if (m < p.wind - sub) so += u; else sn += u;
                        }
                        sn += g.ws[i];
                        const real mo = so * inv_old, mn = sn * inv_new;
                        pn += (double)(mn - mo) * (double)(mn - mo);
                        pd += (double)mn * (double)mn;
                    }
                    pn = warp_sum(pn);
                    pd = warp_sum(pd);
                    if (sqrt(pn) / (sqrt(pd) + 1.0e-10) < p.tol) break;
                }
            }
            g.forward();
            // the final residual stays unmasked in bs: x = bs + ys = A w on every scan
            auto res_sumsq = [&]() -> double {
                if constexpr (CENSOR) {
                    double q = 0.0;
                    for (int i = lane; i < T; i += 32)
                        if (!cm[i]) q += (double)g.bs[i] * (double)g.bs[i];
                    return warp_sum(q);
                } else {
                    return g.sumsq(g.bs);
                }
            };
            if (AUTO) {
                if (!nl.pass_done<CENSOR>(p, v, res_sumsq(), g.sumabs(g.ws), lane == 0, lane, 32, n_kept)) {
                    lam = nl.lbda;
                    th = (real)(lam / Lc);
                    continue;
                }
            } else if (n_done > 0) {
                const double rr = res_sumsq(), gg = g.sumabs(g.ws);
                const double J = 0.5 * rr + lam * gg;
                if (lane == 0) {
                    if (p.out_J) Jv[n_done - 1] = (real)J;
                    if (p.out_r) p.out_r[v] = (real)rr;
                    if (p.out_g) p.out_g[v] = (real)gg;
                }
            }
            break;
        }
        for (int i = lane; i < T; i += 32) {
            p.out_x[v * T + i] = g.bs[i] + g.ys[i];
            p.out_z[v * T + i] = g.as[i];
            p.out_dz[v * T + i] = g.ws[i];
        }
        if (lane == 0 && !AUTO) p.out_niter[v] = n_done;
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// bd
// ------------------------------------------------------------------------------------------------
template <typename real>
struct BdArgs {
    const real *y;
    HrfGrid grid;
    const real *lbda;
    int64_t lbda_stride;
    const real *theta0;
    int64_t theta0_stride;
    const real *z0;
    double theta_lo, theta_hi;
    int nb_iter, early_stopping, wind;
    double tol;
    real *out_x, *out_z, *out_dz, *out_h, *out_theta, *out_J, *out_r, *out_g;
    int32_t *out_ntrace;
    int64_t V;
    int T, K;
    // optional work-queue counter (zeroed on the launch stream): after its first, statically assigned task a
    // warp / CTA pulls the next one from it instead of striding through the batch.  Same results either way.
    unsigned int *queue = nullptr;
};

// Q7: outer early stop of bd on the (signed) relative change of windowed means of J.
template <typename real>
__device__ __forceinline__ bool bd_outer_stop(const real *Jv, int n, double sum_all, int sub,
                                              double tol) {
    // old_j = mean(J[:-sub]), new_j = mean(J[-sub:]) over the n entries stored so far
    if (sub <= 0 || n - sub <= 0) return false;
    double tail = 0.0;
    for (int m = n - sub; m < n; ++m) tail += (double)Jv[m];
    const double old_j = (sum_all - tail) / (double)(n - sub);
    const double new_j = tail / (double)sub;
    return (new_j - old_j) / new_j < tol;
}

template <typename real>
__global__ void generic_bd_kernel(BdArgs<real> p, GenLayout lay) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    real *beta = reinterpret_cast<real *>(smem);
    const size_t beta_bytes = ((size_t)p.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    fill_momentum_table(beta, p.nb_iter);
    unsigned char *base = smem + beta_bytes + (size_t)warp * lay.warp_bytes(sizeof(real));
    double *scratch;
    GenVoxel<real> g = gen_bind<real>(base, lay, p.T, p.K, lane, scratch);
    ThetaScratch sc;
    sc.bind(scratch, lay.kp);
    const int T = p.T, K = p.K, ntr = p.nb_iter + 2;
    const bool es = p.early_stopping != 0;
    const int sub = p.wind / 2;

    for (int64_t v = (int64_t)blockIdx.x * nwarp + warp; v < p.V; v += (int64_t)gridDim.x * nwarp) {
        const real *yv = p.y + v * T;
        for (int i = lane; i < T; i += 32) g.ys[i] = yv[i];
        const double lam = (double)p.lbda[v * p.lbda_stride];
        double theta = (double)p.theta0[v * p.theta0_stride];
        hrf_eval_warp(theta, p.grid, sc, lane);   // bold_signal.py:292 (theta_0 itself, not clipped: Q9)
        g.load_taps(sc);
        double r0, g0;
        if (p.z0) {                               // bold_signal.py:298-301
            const real *zv = p.z0 + v * T;
            for (int i = lane; i < T; i += 32) {
                g.as[i] = zv[i];
                g.ws[i] = i == 0 ? real(0) : zv[i] - zv[i - 1];
            }
            __syncwarp();
            g.conv(g.as, g.ys, g.bs);
            r0 = g.sumsq(g.bs);
            g0 = g.sumabs(g.ws);
        } else {
            for (int i = lane; i < T; i += 32) g.ws[i] = real(0);
            __syncwarp();
            r0 = g.sumsq(g.ys);
            g0 = 0.0;
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
        for (int idx = 0; idx < p.nb_iter; ++idx) {
            const double Lc = frob_lipschitz_warp(sc, K, T, lane);
            g.inner_loop(beta, p.nb_iter, (real)(1.0 / Lc), (real)(lam / Lc), es, p.tol);
            for (int i = lane; i < T; i += 32) g.as[i] = g.ws[i];
            __syncwarp();
            g.scan_fwd(g.as);
            g.theta_moments(sc);
            gram_build_warp(sc, K, lane);
            theta = theta_solve_warp(theta, p.theta_lo, p.theta_hi, p.grid, sc, lane, nullptr);
            hrf_eval_warp(theta, p.grid, sc, lane);
            g.load_taps(sc);
            g.conv(g.as, g.ys, g.bs);
            const double r = g.sumsq(g.bs), gg = g.sumabs(g.ws);
            const double Jn = (r + lam * gg) / j0 + 1.0e-30;
            if (lane == 0) {
                Jv[n] = (real)Jn;
                rv[n] = (real)(r / r0 + 1.0e-30);
                gv[n] = (real)gg;
            }
            sumJ += (double)(real)Jn;
            ++n;
            __syncwarp();
            if (es && idx > p.wind) {
                int stop = 0;
                if (lane == 0) stop = bd_outer_stop(Jv, n, sumJ, sub, p.tol) ? 1 : 0;
                stop = __shfl_sync(PB_FULL, stop, 0);
                if (stop) break;
            }
        }
        {
            const double Lc = frob_lipschitz_warp(sc, K, T, lane);
            g.inner_loop(beta, p.nb_iter, (real)(1.0 / Lc), (real)(lam / Lc), es, p.tol);
            g.forward();
            const double r = g.sumsq(g.bs), gg = g.sumabs(g.ws);
            if (lane == 0) {
                Jv[n] = (real)((r + lam * gg) / j0);
                rv[n] = (real)(r / r0);
                gv[n] = (real)gg;
            }
            ++n;
        }
        for (int i = lane; i < T; i += 32) {
            p.out_x[v * T + i] = g.bs[i] + g.ys[i];
            p.out_z[v * T + i] = g.as[i];
            p.out_dz[v * T + i] = g.ws[i];
        }
        for (int a = lane; a < K; a += 32) p.out_h[v * K + a] = (real)sc.hs[a];
        if (lane == 0) {
            p.out_theta[v] = (real)theta;
            p.out_ntrace[v] = n;
        }
        __syncwarp();
    }
}

}  // namespace pb
