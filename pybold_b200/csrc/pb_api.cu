// extern "C" boundary of libpybold_b200.so (declared in include/pybold_b200.h).
// Host-side argument checks, shared-memory sizing, persistent-grid sizing and dispatch between
// the register-tiled warp kernels (pb_fast.cuh) and the generic kernels (pb_generic.cuh).
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>

#include "../../include/pybold_b200.h"
#include "pb_fast_registry.h"
#include "pb_ops.cuh"
#include "pb_ops_rows.cuh"
#include "pb_noise.cuh"
#include "pb_synth.cuh"
#include "pb_transpose_tma.cuh"

#define PB_VERSION 100   /* 0.1.0 */
#define PB_MAX_T 4096
#define PB_MAX_K 64
#define PB_MAX_ITER 8192
#define PB_MAX_OP_K 1024

namespace {

struct DeviceInfo {
    int sm_count = 0;
    int max_smem_optin = 0;
    int err = 0;
};

DeviceInfo device_info() {
    DeviceInfo d;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        d.err = (int)e;
        return d;
    }
    cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&d.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    return d;
}

// Pick warps per CTA so that the CTA's dynamic shared memory fits, then a persistent grid of
// `ctas_per_sm * sm_count` CTAs (or fewer when the batch is small).
struct LaunchPlan {
    int warps = 0;
    int grid = 0;
    size_t smem = 0;
};

LaunchPlan plan_launch(const DeviceInfo &d, size_t fixed_bytes, size_t warp_bytes, int64_t V,
                       int max_warps) {
    LaunchPlan p;
    const size_t budget = (size_t)d.max_smem_optin;
    if (fixed_bytes + warp_bytes > budget) return p;  // warps == 0 => unsupported
    // aim for two CTAs per SM so that one CTA's tail does not idle the SM
    size_t per_cta = budget / 2;
    int w = (int)((per_cta > fixed_bytes ? per_cta - fixed_bytes : 0) / warp_bytes);
    if (w < 1) w = (int)((budget - fixed_bytes) / warp_bytes);
    if (w > max_warps) w = max_warps;
    if (w < 1) w = 1;
    p.warps = w;
    p.smem = fixed_bytes + (size_t)w * warp_bytes;
    const int ctas_per_sm = (int)(budget / p.smem) > 0 ? (int)(budget / p.smem) : 1;
    int64_t need = (V + w - 1) / w;
    int64_t cap = (int64_t)d.sm_count * (ctas_per_sm > 4 ? 4 : ctas_per_sm);
    p.grid = (int)(need < cap ? need : cap);
    if (p.grid < 1) p.grid = 1;
    return p;
}

template <typename K>
int set_smem(K kernel, size_t bytes) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    return (int)e;
}

// Work-queue counters of the early-stopping kernels: the library owns no memory (SURVEY.md 8(b)), so the
// counters live in a small static device array; every launch takes the next slot round-robin and zeroes it
// on its own stream, which keeps up to 4096 launches in flight (on different streams) independent of each
// other; launches on one stream are ordered anyway.
__device__ unsigned int pb_queue_pool[4096];

unsigned int *queue_slot() {
    static std::atomic<unsigned int> next{0};
    static std::atomic<unsigned int *> base_of[64];     // address of the pool on every device, looked up once
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) {
        cudaGetLastError();
        return nullptr;
    }
    unsigned int *base = base_of[dev].load(std::memory_order_acquire);
    if (!base) {
        if (cudaGetSymbolAddress(reinterpret_cast<void **>(&base), pb_queue_pool) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        base_of[dev].store(base, std::memory_order_release);
    }
    return base + (next.fetch_add(1u) & 4095u);
}

int last_error() {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? PB_OK : (int)e;
}

pb::HrfGrid make_grid(double t_r, double dur, int *n_fine, double dt = 0.001) {
    pb::HrfGrid g;
    const int N = (int)(dur / dt);           // int(float(dur) / dt), hrf_model.py:25
    const int stride = (int)(t_r / dt);      // int(t_r / dt),       hrf_model.py:36
    g.t_step = dur / (double)(N - 1);
    g.stride = stride;
    g.K = stride > 0 ? (N + stride - 1) / stride : 0;
    if (n_fine) *n_fine = N;
    return g;
}

// Register-resident row kernels (pb_ops_rows.cuh) for the shapes they cover; NO_FAST_OP otherwise.
constexpr int NO_FAST_OP = -1000;

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <typename real, bool REV, int NCH>
int launch_rows_scan(const DeviceInfo &d, const real *x, real *out, int64_t V, int T, pb_stream_t stream) {
    const int64_t need = (V + 7) / 8;
    const int64_t cap = (int64_t)d.sm_count * 8;
    pb::rows_scan_kernel<real, REV, NCH><<<(int)(need < cap ? need : cap), 256, 0, (cudaStream_t)stream>>>(
        x, out, V, T);
    return last_error();
}

template <typename real, bool REV>
int run_rows_scan(const real *x, real *out, int64_t V, int T, pb_stream_t stream) {
    constexpr int VEC = pb::Vec16<real>::N;
    if (T % VEC != 0 || !aligned16(x) || !aligned16(out) || T > 32 * VEC * 10) return NO_FAST_OP;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const int nch = (T + 32 * VEC - 1) / (32 * VEC);
    if (nch <= 3) return launch_rows_scan<real, REV, 3>(d, x, out, V, T, stream);
    if (nch <= 5) return launch_rows_scan<real, REV, 5>(d, x, out, V, T, stream);
    return launch_rows_scan<real, REV, 10>(d, x, out, V, T, stream);
}

template <int OP, int KMAX, int NCH>
int launch_rows_conv(const DeviceInfo &d, const float *h, int64_t h_stride, const float *x, float *out,
                     int64_t V, int T, int K, pb_stream_t stream) {
    using L = pb::RowsConvLayout<float, KMAX, NCH>;
    const int warps = 8;
    const size_t smem = (size_t)warps * L::WARP_BYTES;
    auto kern = pb::rows_conv_kernel<float, OP, KMAX, NCH>;
    int e = set_smem(kern, smem);
    if (e) return e;
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, warps * 32, smem) != cudaSuccess || occ < 1) {
        cudaGetLastError();
        return NO_FAST_OP;
    }
    const int64_t need = (V + warps - 1) / warps;
    const int64_t cap = (int64_t)d.sm_count * occ;
    kern<<<(int)(need < cap ? need : cap), warps * 32, smem, (cudaStream_t)stream>>>(h, h_stride, x, out, V, T, K);
    return last_error();
}

template <int OP, int KMAX>
int pick_rows_conv_nch(const DeviceInfo &d, const float *h, int64_t h_stride, const float *x, float *out,
                       int64_t V, int T, int K, pb_stream_t stream) {
    const int nch = (T + 127) / 128;
    if (nch <= 3) return launch_rows_conv<OP, KMAX, 3>(d, h, h_stride, x, out, V, T, K, stream);
    if (nch <= 5) return launch_rows_conv<OP, KMAX, 5>(d, h, h_stride, x, out, V, T, K, stream);
    return launch_rows_conv<OP, KMAX, 10>(d, h, h_stride, x, out, V, T, K, stream);
}

template <int OP, int KMAX, int NCH>
int launch_rows_conv8(const DeviceInfo &d, const float *h, int64_t h_stride, const float *x, float *out,
                      int64_t V, int T, int K, pb_stream_t stream) {
    using L = pb::RowsConv8Layout<KMAX, NCH>;
    const int warps = 8;
    const size_t smem = (size_t)warps * L::WARP_BYTES;
    auto kern = pb::rows_conv8_kernel<OP, KMAX, NCH>;
    int e = set_smem(kern, smem);
    if (e) return e;
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, warps * 32, smem) != cudaSuccess || occ < 1) {
        cudaGetLastError();
        return NO_FAST_OP;
    }
    const int64_t need = (V + warps - 1) / warps;
    const int64_t cap = (int64_t)d.sm_count * occ;
    kern<<<(int)(need < cap ? need : cap), warps * 32, smem, (cudaStream_t)stream>>>(h, h_stride, x, out, V, T, K);
    return last_error();
}

template <int OP, int KMAX>
int pick_rows_conv8_nch(const DeviceInfo &d, const float *h, int64_t h_stride, const float *x, float *out,
                        int64_t V, int T, int K, pb_stream_t stream) {
    if (T <= 512) return launch_rows_conv8<OP, KMAX, 2>(d, h, h_stride, x, out, V, T, K, stream);
    return launch_rows_conv8<OP, KMAX, 5>(d, h, h_stride, x, out, V, T, K, stream);
}

inline bool aligned32(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 31) == 0; }

template <int OP>
int run_rows_conv(const float *h, int64_t h_stride, const float *x, float *out, int64_t V, int T, int K,
                  pb_stream_t stream) {
    if (T % 4 != 0 || !aligned16(x) || !aligned16(out) || T > 1280 || K > 32) return NO_FAST_OP;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    // 32-byte rows: eight samples per lane (half the shared-memory window traffic); PB_ROWS_CONV4=1 keeps
    // the four-sample kernel for A/B timing
    static const bool conv4 = getenv("PB_ROWS_CONV4") != nullptr;
    if (!conv4 && T % 8 == 0 && aligned32(x) && aligned32(out)) {
        if (K <= 20) return pick_rows_conv8_nch<OP, 20>(d, h, h_stride, x, out, V, T, K, stream);
        if (K <= 28) return pick_rows_conv8_nch<OP, 28>(d, h, h_stride, x, out, V, T, K, stream);
        return pick_rows_conv8_nch<OP, 32>(d, h, h_stride, x, out, V, T, K, stream);
    }
    if (K <= 20) return pick_rows_conv_nch<OP, 20>(d, h, h_stride, x, out, V, T, K, stream);
    if (K <= 28) return pick_rows_conv_nch<OP, 28>(d, h, h_stride, x, out, V, T, K, stream);
    return pick_rows_conv_nch<OP, 32>(d, h, h_stride, x, out, V, T, K, stream);
}
template <int OP>
int run_rows_conv(const double *, int64_t, const double *, double *, int64_t, int, int, pb_stream_t) {
    return NO_FAST_OP;      // the double build uses op_kernel
}

template <typename real, int OP>
int run_op(const real *h, int64_t h_stride, const real *x, real *out, int64_t V, int T, int K,
           pb_stream_t stream) {
    if (V == 0) return PB_OK;
    if (!x || !out || V < 0 || T <= 0) return PB_ERR_INVALID_ARG;
    if (OP >= pb::OP_CONV && (!h || K <= 0)) return PB_ERR_INVALID_ARG;
    if (T > PB_MAX_T || K > PB_MAX_OP_K) return PB_ERR_UNSUPPORTED;
    {
        int rc = NO_FAST_OP;
        if constexpr (OP == pb::OP_INTEG) rc = run_rows_scan<real, false>(x, out, V, T, stream);
        else if constexpr (OP == pb::OP_INTEG_ADJ) rc = run_rows_scan<real, true>(x, out, V, T, stream);
        else rc = run_rows_conv<OP>(h, h_stride, x, out, V, T, K, stream);
        if (rc != NO_FAST_OP) return rc;
    }
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    pb::OpLayout lay = pb::OpLayout::make(T, OP >= pb::OP_CONV ? K : 1);
    LaunchPlan p = plan_launch(d, 0, lay.warp_bytes(sizeof(real)), V, 8);
    if (!p.warps) return PB_ERR_UNSUPPORTED;
    auto kern = pb::op_kernel<real, OP>;
    int e = set_smem(kern, p.smem);
    if (e) return e;
    kern<<<p.grid, p.warps * 32, p.smem, (cudaStream_t)stream>>>(h, h_stride, x, out, V, T, K, lay);
    return last_error();
}

template <typename real>
int run_spm_hrf(const real *theta, double t_r, double dur, int normalized, real *out_h, int64_t V,
                int K, pb_stream_t stream) {
    if (V == 0) return PB_OK;
    if (!theta || !out_h || V < 0 || !(t_r >= 0.001) || !(dur > 0.002)) return PB_ERR_INVALID_ARG;
    int n_fine = 0;
    pb::HrfGrid g = make_grid(t_r, dur, &n_fine);
    if (K != g.K) return PB_ERR_INVALID_ARG;
    if (V == 0) return PB_OK;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const int warps = 4;
    int64_t need = (V + warps - 1) / warps;
    int grid = (int)(need < (int64_t)d.sm_count * 8 ? need : (int64_t)d.sm_count * 8);
    pb::spm_hrf_kernel<real><<<grid, warps * 32, 0, (cudaStream_t)stream>>>(theta, g, n_fine,
                                                                            normalized, out_h, V);
    return last_error();
}

template <typename real>
int run_spm_hrf_ex(const real *theta, double t_r, double dur, int normalized, const double *shape7,
                   real *out_h, int64_t V, int K, pb_stream_t stream) {
    if (V == 0) return PB_OK;
    if (!theta || !out_h || !shape7 || V < 0) return PB_ERR_INVALID_ARG;
    const double dt = shape7[0], p_delay = shape7[1], undershoot = shape7[2], p_disp = shape7[3],
                 u_disp = shape7[4], ratio = shape7[5], onset = shape7[6];
    if (!(dt > 0.0) || !(t_r >= dt) || !(dur > 2.0 * dt) || !(p_disp > 0.0) || !(u_disp > 0.0) ||
        !(p_delay > 0.0) || !(undershoot > 0.0))
        return PB_ERR_INVALID_ARG;
    int n_fine = 0;
    pb::HrfGrid g = make_grid(t_r, dur, &n_fine, dt);
    if (K != g.K) return PB_ERR_INVALID_ARG;
    pb::HrfShape sh;
    sh.dt = dt;
    sh.a_peak = p_delay / p_disp;
    sh.loc_peak = dt / p_disp;
    sh.a_under = undershoot / u_disp;
    sh.loc_under = dt / u_disp;
    sh.ratio = ratio;
    sh.t_shift = onset / dt;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const int warps = 4;
    int64_t need = (V + warps - 1) / warps;
    int grid = (int)(need < (int64_t)d.sm_count * 8 ? need : (int64_t)d.sm_count * 8);
    pb::spm_hrf_ex_kernel<real><<<grid, warps * 32, 0, (cudaStream_t)stream>>>(theta, g, sh, n_fine,
                                                                               normalized, out_h, V);
    return last_error();
}

// censor != null: the power iteration of the censored operator A^T M A (censor_stride 0: one mask for the batch)
template <typename real>
int run_lipschitz_power(const real *h, int64_t h_stride, const real *x0, int64_t x0_stride,
                        int nb_iter, double tol, real *out_L, int64_t V, int T, int K,
                        pb_stream_t stream, const unsigned char *censor = nullptr, int64_t censor_stride = 0) {
    if (V == 0) return PB_OK;
    if (!h || !x0 || !out_L || V < 0 || T <= 0 || K <= 0 || nb_iter < 1 || censor_stride < 0)
        return PB_ERR_INVALID_ARG;
    if (T > PB_MAX_T || K > PB_MAX_OP_K) return PB_ERR_UNSUPPORTED;
    if (V == 0) return PB_OK;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    pb::GenLayout lay = pb::GenLayout::make(T, K, 0, false);
    LaunchPlan p = plan_launch(d, 0, lay.warp_bytes(sizeof(real)), V, 8);
    if (!p.warps) return PB_ERR_UNSUPPORTED;
    auto go = [&](auto kern) {
        int e = set_smem(kern, p.smem);
        if (e) return e;
        kern<<<p.grid, p.warps * 32, p.smem, (cudaStream_t)stream>>>(h, h_stride, x0, x0_stride, nb_iter,
                                                                     tol, out_L, V, T, K, lay,
                                                                     pb::Censor{censor, censor_stride});
        return last_error();
    };
    return censor ? go(pb::lipschitz_power_kernel<real, true>) : go(pb::lipschitz_power_kernel<real, false>);
}

template <typename real>
int run_lipschitz_frob(const real *h, int64_t h_stride, real *out_L, int64_t V, int T, int K,
                       pb_stream_t stream) {
    if (V == 0) return PB_OK;
    if (!h || !out_L || V < 0 || T <= 0 || K <= 0) return PB_ERR_INVALID_ARG;
    if (T > (1 << 20) || K > PB_MAX_OP_K) return PB_ERR_UNSUPPORTED;
    if (V == 0) return PB_OK;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const int kp = (K + 3) & ~3;
    const int warps = 4;
    const size_t smem = (size_t)warps * 3 * kp * sizeof(double);
    auto kern = pb::lipschitz_frob_kernel<real>;
    int e = set_smem(kern, smem);
    if (e) return e;
    int64_t need = (V + warps - 1) / warps;
    int grid = (int)(need < (int64_t)d.sm_count * 8 ? need : (int64_t)d.sm_count * 8);
    kern<<<grid, warps * 32, smem, (cudaStream_t)stream>>>(h, h_stride, out_L, V, T, K, kp);
    return last_error();
}

template <typename real>
int run_transpose(const real *in, real *out, int64_t rows, int64_t cols, pb_stream_t stream) {
    if (rows == 0 || cols == 0) return PB_OK;
    if (!in || !out || rows < 0 || cols < 0 || in == out) return PB_ERR_INVALID_ARG;
    // TMA tile mover when pointers and row pitches are 16-byte aligned (pb_transpose_tma.cuh);
    // PB_TRANSPOSE_NO_TMA=1 keeps the plain-load kernel for A/B timing
    static const bool no_tma = getenv("PB_TRANSPOSE_NO_TMA") != nullptr;
    if (!no_tma) {
        DeviceInfo d = device_info();
        if (d.err) return d.err;
        const int rc = pb::transpose_tma_launch<real>(in, out, rows, cols, d.sm_count, (cudaStream_t)stream);
        if (rc != -1000) return rc == 0 ? PB_OK : rc;
    }
    const int64_t gx = (cols + 63) / 64, gy = (rows + 63) / 64;
    if (gy > 65535 || gx > 2147483647LL) return PB_ERR_UNSUPPORTED;
    pb::transpose_kernel<real><<<dim3((unsigned)gx, (unsigned)gy), dim3(32, 8), 0, (cudaStream_t)stream>>>(
        in, out, rows, cols);
    return last_error();
}

template <typename real>
int run_toeplitz(const real *k, int klen, real *out, int64_t dim_out, int64_t dim_in, pb_stream_t stream) {
    if (dim_out == 0 || dim_in == 0) return PB_OK;
    if (!k || !out || klen <= 0 || dim_out < 0 || dim_in < 0) return PB_ERR_INVALID_ARG;
    const int64_t gx = (dim_in + 255) / 256;
    if (gx > 2147483647LL) return PB_ERR_UNSUPPORTED;
    const unsigned gy = (unsigned)(dim_out < 65535 ? dim_out : 65535);
    pb::toeplitz_kernel<real><<<dim3((unsigned)gx, gy), 256, 0, (cudaStream_t)stream>>>(k, klen, out, dim_out, dim_in);
    return last_error();
}

// the register-tiled variant the dispatch chooses (pb_fast_registry.cu), else the generic kernel; a.nb_outer > 0
// selects the deconv(lbda=None) instances, cz (scan censoring) the censored ones.  V == 0 launches nothing: *id /
// *family report the kernel a launch would run (pb_deconv_variant, pb_deconv_censored_variant).
template <typename real>
int launch_deconv(const pb::DeconvArgs<real> &a, pb_stream_t stream, int *id = nullptr, int *family = nullptr,
                  const pb::Censor *cz = nullptr) {
    int rc = cz ? pb::fast_deconv_censored_dispatch(a, *cz, (cudaStream_t)stream, id, family)
                : pb::fast_deconv_dispatch(a, (cudaStream_t)stream, id, family);
    if (rc != pb::FAST_NO_MATCH) return rc;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const bool es = a.early_stopping && a.wind >= 2;
    pb::GenLayout lay = pb::GenLayout::make(a.T, a.K, es ? a.wind - 1 : 0, false);
    if (a.nb_outer > 0 && lay.doubles < (size_t)a.wind) lay.doubles = (size_t)a.wind;   // the window of alphas
    const size_t beta_bytes = ((size_t)a.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    // long series in double with the early-stopping ring: rows that do not fit move to the output rows
    while (beta_bytes + lay.warp_bytes(sizeof(real)) > (size_t)d.max_smem_optin && lay.spill_ring_row()) {
    }
    LaunchPlan p = plan_launch(d, beta_bytes, lay.warp_bytes(sizeof(real)), a.V, 8);
    if (!p.warps) return PB_ERR_UNSUPPORTED;
    if (a.V == 0) return PB_OK;
    auto go = [&](auto kern) {
        int e = set_smem(kern, p.smem);
        if (e) return e;
        kern<<<p.grid, p.warps * 32, p.smem, (cudaStream_t)stream>>>(a, lay, cz ? *cz : pb::Censor{});
        return last_error();
    };
    if (cz)
        return a.nb_outer > 0 ? go(pb::generic_deconv_kernel<real, true, true>)
                              : go(pb::generic_deconv_kernel<real, false, true>);
    return a.nb_outer > 0 ? go(pb::generic_deconv_kernel<real, true>) : go(pb::generic_deconv_kernel<real, false>);
}

// What the deconv entry points set before the dispatch: for deconv(lbda=None) without early stopping (or with
// wind < 2, which has no window) wind = 2 -- the window length does not matter then, and 2 keeps the group kernel's
// ring of u's one row long -- and the work-queue counter of the early-stopping and deconv(lbda=None) kernels, taken
// from `queue` (queue_slot for a launch).
template <typename real>
void set_routing(pb::DeconvArgs<real> &a, unsigned int *(*queue)()) {
    if (a.nb_outer > 0 && !(a.early_stopping && a.wind >= 2)) {
        a.early_stopping = 0;
        a.wind = 2;
    }
    if (a.nb_outer > 0 || (a.early_stopping && a.wind >= 2)) a.queue = queue();
}

template <typename real>
int run_deconv(pb::DeconvArgs<real> a, pb_stream_t stream, const pb::Censor *cz = nullptr) {
    if (a.V == 0) return PB_OK;
    if (cz && (!cz->m || cz->stride < 0)) return PB_ERR_INVALID_ARG;
    if (!a.y || !a.h || !a.L || !a.lbda || !a.out_x || !a.out_z || !a.out_dz ||
        !a.out_niter || a.V < 0 || a.T <= 0 || a.K <= 0 || a.nb_iter < 1 || a.wind < 0)
        return PB_ERR_INVALID_ARG;
    if (a.T > PB_MAX_T || a.K > PB_MAX_K || a.nb_iter > PB_MAX_ITER) return PB_ERR_UNSUPPORTED;
    if (a.V == 0) return PB_OK;
    set_routing(a, queue_slot);
    return launch_deconv(a, stream, nullptr, nullptr, cz);
}

// deconv(lbda=None): the noise loop runs inside the kernel, nb_outer outer iterations at most, nb_iter inner
// ones per pass; then the voxels with a NaN sigma get the reference's NaN outputs (pb_noise.cuh)
template <typename real>
int run_deconv_auto(pb::DeconvArgs<real> a, pb_stream_t stream, const pb::Censor *cz = nullptr) {
    if (a.V == 0) return PB_OK;
    if (cz && (!cz->m || cz->stride < 0)) return PB_ERR_INVALID_ARG;
    if (!a.y || !a.h || !a.L || !a.sigma || !a.out_x || !a.out_z || !a.out_dz || a.V < 0 || a.T <= 0 ||
        a.K <= 0 || a.nb_iter < 1 || a.nb_outer < 1 || a.wind < 0 || a.h_stride < 0 || a.L_stride < 0 ||
        a.sigma_stride < 0)
        return PB_ERR_INVALID_ARG;
    if (a.T > PB_MAX_T || a.K > PB_MAX_K || a.nb_iter > PB_MAX_ITER) return PB_ERR_UNSUPPORTED;
    set_routing(a, queue_slot);
    const int rc = launch_deconv(a, stream, nullptr, nullptr, cz);
    if (rc) return rc;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const int64_t cap = (int64_t)d.sm_count * 8;
    pb::nan_sigma_rows_kernel<real><<<(int)(a.V < cap ? a.V : cap), 128, 0, (cudaStream_t)stream>>>(a);
    return last_error();
}

// pb_deconv_variant / pb_deconv_censored_variant: the routing of a deconv call with V = 0 (nothing is launched)
template <typename real>
int deconv_variant(int T, int K, int nb_iter, int early_stopping, int wind, int is_auto, int *family,
                   bool censored = false) {
    if (!family || T <= 0 || K <= 0 || nb_iter < 1 || wind < 0) return PB_ERR_INVALID_ARG;
    if (T > PB_MAX_T || K > PB_MAX_K || nb_iter > PB_MAX_ITER) return PB_ERR_UNSUPPORTED;
    pb::DeconvArgs<real> a{};
    a.T = T;
    a.K = K;
    a.nb_iter = nb_iter;
    a.early_stopping = early_stopping;
    a.wind = wind;
    a.nb_outer = is_auto ? 1 : 0;
    a.V = 0;
    // a placeholder counter: the routing sees a work queue exactly when a call would, and a launch with V = 0
    // neither zeroes nor reads it, so the query takes no slot of the pool
    set_routing(a, +[]() -> unsigned int * {
        static unsigned int placeholder;
        return &placeholder;
    });
    int id = 0;
    static const unsigned char placeholder_mask = 0;
    const pb::Censor cz{&placeholder_mask, 0};
    const int rc = launch_deconv(a, nullptr, &id, family, censored ? &cz : nullptr);
    if (rc > 0) {               // a CUDA error
        cudaGetLastError();
        return PB_ERR_NO_DEVICE;
    }
    return rc < 0 ? rc : id;
}

// the register-tiled variant bd_dispatch chooses (pb_fast_registry.cu), else the generic kernel.  V == 0 launches
// nothing: *id / *family report the kernel a launch would run (pb_bd_variant).
template <typename real>
int launch_bd(const pb::BdArgs<real> &a, pb_stream_t stream, int *id = nullptr, int *family = nullptr) {
    int rc = pb::fast_bd_dispatch(a, (cudaStream_t)stream, id, family);
    if (rc != pb::FAST_NO_MATCH) return rc;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    pb::GenLayout lay = pb::GenLayout::make(a.T, a.K, 0, true);
    const size_t beta_bytes = ((size_t)a.nb_iter * sizeof(real) + 15) & ~(size_t)15;
    LaunchPlan p = plan_launch(d, beta_bytes, lay.warp_bytes(sizeof(real)), a.V, 8);
    if (!p.warps) return PB_ERR_UNSUPPORTED;
    if (a.V == 0) return PB_OK;
    auto kern = pb::generic_bd_kernel<real>;
    int e = set_smem(kern, p.smem);
    if (e) return e;
    kern<<<p.grid, p.warps * 32, p.smem, (cudaStream_t)stream>>>(a, lay);
    return last_error();
}

template <typename real>
int run_bd(pb::BdArgs<real> a, double t_r, double hrf_dur, pb_stream_t stream) {
    if (a.V == 0) return PB_OK;
    if (!a.y || !a.lbda || !a.theta0 || !a.out_x || !a.out_z || !a.out_dz || !a.out_h ||
        !a.out_theta || !a.out_J || !a.out_r || !a.out_g || !a.out_ntrace || a.V < 0 || a.T <= 0 ||
        a.nb_iter < 1 || a.wind < 0 || !(a.theta_lo <= a.theta_hi) || !(t_r >= 0.001) ||
        !(hrf_dur > 0.002))
        return PB_ERR_INVALID_ARG;
    a.grid = make_grid(t_r, hrf_dur, nullptr);
    if (a.K != a.grid.K) return PB_ERR_INVALID_ARG;
    if (a.T > PB_MAX_T || a.K > PB_MAX_K || a.nb_iter > PB_MAX_ITER) return PB_ERR_UNSUPPORTED;
    if (a.V == 0) return PB_OK;
    // group / CTA kernels pull their tasks from it (static stride if null; PB_NO_QUEUE=1: developer A/B switch)
    static const bool no_queue = getenv("PB_NO_QUEUE") != nullptr;
    a.queue = no_queue ? nullptr : queue_slot();
    return launch_bd(a, stream);
}

// pb_bd_variant: the routing of a bd call with V = 0 (nothing is launched; the work-queue counter plays no part in
// the choice)
template <typename real>
int bd_variant(int T, int K, int nb_iter, int early_stopping, int wind, int *family) {
    if (!family || T <= 0 || K <= 0 || nb_iter < 1 || wind < 0) return PB_ERR_INVALID_ARG;
    if (T > PB_MAX_T || K > PB_MAX_K || nb_iter > PB_MAX_ITER) return PB_ERR_UNSUPPORTED;
    pb::BdArgs<real> a{};
    a.T = T;
    a.K = K;
    a.nb_iter = nb_iter;
    a.early_stopping = early_stopping;
    a.wind = wind;
    a.V = 0;
    int id = 0;
    const int rc = launch_bd(a, nullptr, &id, family);
    if (rc > 0) {               // a CUDA error
        cudaGetLastError();
        return PB_ERR_NO_DEVICE;
    }
    return rc < 0 ? rc : id;
}

template <typename real>
int run_hrf_estim(const real *z, const real *y, double t_r, double hrf_dur, const real *theta0,
                  int64_t theta0_stride, double lo, double hi, real *out_theta, real *out_h,
                  real *out_cost, int64_t V, int T, int K, pb_stream_t stream) {
    if (V == 0) return PB_OK;
    if (!z || !y || !theta0 || !out_theta || !out_h || !out_cost || V < 0 || T <= 0 || !(lo <= hi) ||
        !(t_r >= 0.001) || !(hrf_dur > 0.002))
        return PB_ERR_INVALID_ARG;
    pb::HrfGrid g = make_grid(t_r, hrf_dur, nullptr);
    if (K != g.K) return PB_ERR_INVALID_ARG;
    if (T > PB_MAX_T || K > PB_MAX_K) return PB_ERR_UNSUPPORTED;
    if (V == 0) return PB_OK;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    pb::GenLayout lay = pb::GenLayout::make(T, K, 0, true);
    LaunchPlan p = plan_launch(d, 0, lay.warp_bytes(sizeof(real)), V, 8);
    if (!p.warps) return PB_ERR_UNSUPPORTED;
    auto kern = pb::hrf_estim_kernel<real>;
    int e = set_smem(kern, p.smem);
    if (e) return e;
    kern<<<p.grid, p.warps * 32, p.smem, (cudaStream_t)stream>>>(z, y, g, theta0, theta0_stride, lo, hi,
                                                                 out_theta, out_h, out_cost, V, T, lay);
    return last_error();
}

template <typename real>
int run_synth(uint64_t seed, int64_t first_voxel, double t_r, double hrf_dur, double snr_db, int nb_events,
              int blk, double delta_lo, double delta_hi, real *out_y, real *out_z, real *out_delta, int64_t V,
              int T, pb_stream_t stream) {
    if (V == 0) return PB_OK;
    if (!out_y || V < 0 || T <= 0 || first_voxel < 0 || nb_events < 0 || blk < 1 || !(t_r >= 0.001) ||
        !(hrf_dur > 0.002) || !(delta_lo <= delta_hi) || !(delta_lo >= 0.5) || !(delta_hi <= 2.0))
        return PB_ERR_INVALID_ARG;
    if (T > PB_MAX_T || nb_events > pb::PB_SYNTH_MAX_EVENTS) return PB_ERR_UNSUPPORTED;
    pb::SynthArgs a;
    a.seed = seed; a.first_voxel = first_voxel; a.grid = make_grid(t_r, hrf_dur, nullptr);
    a.delta_lo = delta_lo; a.delta_hi = delta_hi; a.snr_db = snr_db; a.nb_events = nb_events; a.blk = blk;
    a.V = V; a.T = T;
    if (a.grid.K < 1 || a.grid.K > PB_MAX_OP_K) return PB_ERR_UNSUPPORTED;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const int warps = 4;
    const size_t smem = (size_t)warps * ((((size_t)T * sizeof(float) + 15) & ~(size_t)15) +
                                         (size_t)a.grid.K * sizeof(double));
    auto kern = pb::synth_voxels_kernel<real>;
    int e = set_smem(kern, smem);
    if (e) return e;
    const int64_t need = (V + warps - 1) / warps;
    const int64_t cap = (int64_t)d.sm_count * 8;
    kern<<<(int)(need < cap ? need : cap), warps * 32, smem, (cudaStream_t)stream>>>(a, out_y, out_z, out_delta);
    return last_error();
}

template <typename real>
int run_inf_norm(const real *x, real *out, int64_t V, int T, pb_stream_t stream) {
    if (V == 0) return PB_OK;
    if (!x || !out || V < 0 || T <= 0) return PB_ERR_INVALID_ARG;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const int64_t need = (V + 7) / 8, cap = (int64_t)d.sm_count * 8;
    pb::inf_norm_kernel<real><<<(int)(need < cap ? need : cap), 256, 0, (cudaStream_t)stream>>>(x, out, V, T);
    return last_error();
}

template <typename real>
int run_rel_l2_err(const real *est, const real *ref, int64_t ref_stride, real *out_err, int64_t V, int T,
                   pb_stream_t stream) {
    if (V == 0) return PB_OK;
    if (!est || !ref || !out_err || V < 0 || T <= 0 || ref_stride < 0) return PB_ERR_INVALID_ARG;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const int64_t need = (V + 7) / 8, cap = (int64_t)d.sm_count * 8;
    pb::rel_l2_err_kernel<real><<<(int)(need < cap ? need : cap), 256, 0, (cudaStream_t)stream>>>(
        est, ref, ref_stride, out_err, V, T);
    return last_error();
}

template <typename real>
int run_noise_step(const real *xn, const real *zn, const real *wn, const real *y, const real *sigma,
                   const unsigned char *active, double mu, real *x, real *z, real *w, real *alpha, real *lbda,
                   real *out_r, real *out_g, int64_t V, int T, pb_stream_t stream) {
    if (V == 0) return PB_OK;
    if (!xn || !zn || !wn || !y || !sigma || !active || !x || !z || !w || !alpha || !lbda || !out_r || !out_g ||
        V < 0 || T <= 0)
        return PB_ERR_INVALID_ARG;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const int64_t need = (V + 7) / 8, cap = (int64_t)d.sm_count * 8;
    pb::noise_step_kernel<real><<<(int)(need < cap ? need : cap), 256, 0, (cudaStream_t)stream>>>(
        xn, zn, wn, y, sigma, active, mu, x, z, w, alpha, lbda, out_r, out_g, V, T);
    return last_error();
}

template <typename real, int MODE>
int run_mad(const real *x, double c, real *out, int64_t V, int T, pb_stream_t stream) {
    if (V == 0) return PB_OK;
    if (!x || !out || V < 0 || T <= 0 || !(c > 0.0)) return PB_ERR_INVALID_ARG;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const int nmax = MODE == 1 ? pb::noise_detail_len(T) : T;
    const size_t warp_bytes = (size_t)nmax * sizeof(double);
    if (warp_bytes > (size_t)d.max_smem_optin) return PB_ERR_UNSUPPORTED;
    int warps = (int)((size_t)d.max_smem_optin / 2 / warp_bytes);
    warps = warps < 1 ? 1 : (warps > 8 ? 8 : warps);
    const size_t smem = (size_t)warps * warp_bytes;
    auto kern = pb::mad_rows_kernel<real, MODE>;
    int e = set_smem(kern, smem);
    if (e) return e;
    const int64_t need = (V + warps - 1) / warps, cap = (int64_t)d.sm_count * 2;
    kern<<<(int)(need < cap ? need : cap), warps * 32, smem, (cudaStream_t)stream>>>(x, c, out, V, T, nmax);
    return last_error();
}

template <typename real>
int run_mad_censored(const real *y, const unsigned char *censor, int64_t censor_stride, double c, real *out,
                     int64_t V, int T, pb_stream_t stream) {
    if (V == 0) return PB_OK;
    if (!y || !censor || !out || V < 0 || T <= 0 || censor_stride < 0 || !(c > 0.0)) return PB_ERR_INVALID_ARG;
    DeviceInfo d = device_info();
    if (d.err) return d.err;
    const int nmax = pb::noise_detail_len(T);
    const size_t warp_bytes = (size_t)nmax * sizeof(double);
    if (warp_bytes > (size_t)d.max_smem_optin) return PB_ERR_UNSUPPORTED;
    int warps = (int)((size_t)d.max_smem_optin / 2 / warp_bytes);
    warps = warps < 1 ? 1 : (warps > 8 ? 8 : warps);
    const size_t smem = (size_t)warps * warp_bytes;
    auto kern = pb::mad_daub_censored_kernel<real>;
    int e = set_smem(kern, smem);
    if (e) return e;
    const int64_t need = (V + warps - 1) / warps, cap = (int64_t)d.sm_count * 2;
    kern<<<(int)(need < cap ? need : cap), warps * 32, smem, (cudaStream_t)stream>>>(
        y, c, out, V, T, nmax, pb::Censor{censor, censor_stride});
    return last_error();
}

// FP32 FMA-pipe ceiling: 16 independent chains a = a * m + c per thread (one register read per FFMA, the
// multiplier and the addend sit in the operand-reuse cache); launch with 4 CTAs of 256 threads per SM.
// Best of the variants in tools/exp_fma.cu (profiles/r01_fma_microbench.txt: 70.7 Tflop/s of 74.4 nominal).
__global__ void __launch_bounds__(256) fma_peak_kernel(float *sink, int iters) {
    float a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = threadIdx.x * 1e-9f + 0.5f * i;
    const float m0 = 0.999f + blockIdx.x * 1e-9f, m1 = 0.998f, c0 = 1e-3f, c1 = 2e-3f;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
            a[i] = fmaf(a[i], m0, c0);
            a[i + 1] = fmaf(a[i + 1], m1, c1);
        }
    }
    float r = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) r += a[i];
    sink[blockIdx.x * blockDim.x + threadIdx.x] = r;
}

}  // namespace

extern "C" {

int pb_bench_fma_f32(float *sink, int blocks, int iters, pb_stream_t stream) {
    if (!sink || blocks < 1 || iters < 1) return PB_ERR_INVALID_ARG;
    fma_peak_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(sink, iters);
    return last_error();
}


int pb_copy_async(void *dst, const void *src, size_t bytes, pb_stream_t stream) {
    if (bytes == 0) return PB_OK;
    if (!dst || !src) return PB_ERR_INVALID_ARG;
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)stream);
    return e == cudaSuccess ? PB_OK : (int)e;
}

int pb_version(void) { return PB_VERSION; }
int pb_max_T(void) { return PB_MAX_T; }
int pb_max_K(void) { return PB_MAX_K; }
int pb_max_iter(void) { return PB_MAX_ITER; }

const char *pb_error_string(int code) {
    switch (code) {
        case PB_OK: return "ok";
        case PB_ERR_INVALID_ARG: return "invalid argument";
        case PB_ERR_UNSUPPORTED: return "unsupported shape (T, K, nb_iter or wind above the compiled limits)";
        case PB_ERR_NO_DEVICE: return "no usable CUDA device";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
    }
}

int pb_solver_variant(int T, int K, int is_f64) { return pb::fast_variant_id(T, K, is_f64 != 0); }

int pb_deconv_variant(int T, int K, int is_f64, int nb_iter, int early_stopping, int wind, int is_auto,
                      int *family) {
    return is_f64 ? deconv_variant<double>(T, K, nb_iter, early_stopping, wind, is_auto, family)
                  : deconv_variant<float>(T, K, nb_iter, early_stopping, wind, is_auto, family);
}

int pb_deconv_censored_variant(int T, int K, int is_f64, int nb_iter, int early_stopping, int wind, int is_auto,
                               int *family) {
    return is_f64 ? deconv_variant<double>(T, K, nb_iter, early_stopping, wind, is_auto, family, true)
                  : deconv_variant<float>(T, K, nb_iter, early_stopping, wind, is_auto, family, true);
}

int pb_bd_variant(int T, int K, int is_f64, int nb_iter, int early_stopping, int wind, int *family) {
    return is_f64 ? bd_variant<double>(T, K, nb_iter, early_stopping, wind, family)
                  : bd_variant<float>(T, K, nb_iter, early_stopping, wind, family);
}

int pb_bd_wave_voxels(int T, int K, int is_f64, int nb_iter) {
    if (T <= 0 || K <= 0 || nb_iter < 1) return 0;
    return pb::fast_bd_wave_voxels(T, K, is_f64 != 0, nb_iter);
}

int pb_hrf_len(double t_r, double dur) {
    if (!(t_r >= 0.001) || !(dur > 0.002)) return PB_ERR_INVALID_ARG;
    return make_grid(t_r, dur, nullptr).K;
}

int pb_hrf_len_ex(double t_r, double dur, double dt) {
    if (!(dt > 0.0) || !(t_r >= dt) || !(dur > 2.0 * dt)) return PB_ERR_INVALID_ARG;
    return make_grid(t_r, dur, nullptr, dt).K;
}

#define PB_DEFINE_OPS(SUF, REAL)                                                                       \
    int pb_integ_op_##SUF(const REAL *x, REAL *out, int64_t V, int T, pb_stream_t s) {                 \
        return run_op<REAL, pb::OP_INTEG>(nullptr, 0, x, out, V, T, 0, s);                             \
    }                                                                                                  \
    int pb_integ_adj_##SUF(const REAL *x, REAL *out, int64_t V, int T, pb_stream_t s) {                \
        return run_op<REAL, pb::OP_INTEG_ADJ>(nullptr, 0, x, out, V, T, 0, s);                         \
    }                                                                                                  \
    int pb_conv_op_##SUF(const REAL *h, int64_t hs, const REAL *x, REAL *out, int64_t V, int T, int K, \
                         pb_stream_t s) {                                                              \
        return run_op<REAL, pb::OP_CONV>(h, hs, x, out, V, T, K, s);                                   \
    }                                                                                                  \
    int pb_conv_adj_##SUF(const REAL *h, int64_t hs, const REAL *x, REAL *out, int64_t V, int T,       \
                          int K, pb_stream_t s) {                                                      \
        return run_op<REAL, pb::OP_CONV_ADJ>(h, hs, x, out, V, T, K, s);                               \
    }                                                                                                  \
    int pb_hrfinteg_op_##SUF(const REAL *h, int64_t hs, const REAL *x, REAL *out, int64_t V, int T,    \
                             int K, pb_stream_t s) {                                                   \
        return run_op<REAL, pb::OP_HRFINTEG>(h, hs, x, out, V, T, K, s);                               \
    }                                                                                                  \
    int pb_hrfinteg_adj_##SUF(const REAL *h, int64_t hs, const REAL *x, REAL *out, int64_t V, int T,   \
                              int K, pb_stream_t s) {                                                  \
        return run_op<REAL, pb::OP_HRFINTEG_ADJ>(h, hs, x, out, V, T, K, s);                           \
    }                                                                                                  \
    int pb_spm_hrf_##SUF(const REAL *theta, double t_r, double dur, int normalized, REAL *out_h,       \
                         int64_t V, int K, pb_stream_t s) {                                            \
        return run_spm_hrf<REAL>(theta, t_r, dur, normalized, out_h, V, K, s);                         \
    }                                                                                                  \
    int pb_spm_hrf_ex_##SUF(const REAL *theta, double t_r, double dur, int normalized,                 \
                            const double *shape7, REAL *out_h, int64_t V, int K, pb_stream_t s) {      \
        return run_spm_hrf_ex<REAL>(theta, t_r, dur, normalized, shape7, out_h, V, K, s);              \
    }                                                                                                  \
    int pb_lipschitz_power_##SUF(const REAL *h, int64_t hs, const REAL *x0, int64_t xs, int nb_iter,   \
                                 double tol, REAL *out_L, int64_t V, int T, int K, pb_stream_t s) {    \
        return run_lipschitz_power<REAL>(h, hs, x0, xs, nb_iter, tol, out_L, V, T, K, s);              \
    }                                                                                                  \
    int pb_lipschitz_power_censored_##SUF(const REAL *h, int64_t hs, const REAL *x0, int64_t xs,       \
                                          const unsigned char *censor, int64_t censor_stride,          \
                                          int nb_iter, double tol, REAL *out_L, int64_t V, int T,      \
                                          int K, pb_stream_t s) {                                      \
        if (!censor && V != 0) return PB_ERR_INVALID_ARG;                                              \
        return run_lipschitz_power<REAL>(h, hs, x0, xs, nb_iter, tol, out_L, V, T, K, s, censor,       \
                                         censor_stride);                                               \
    }                                                                                                  \
    int pb_lipschitz_frob_##SUF(const REAL *h, int64_t hs, REAL *out_L, int64_t V, int T, int K,       \
                                pb_stream_t s) {                                                       \
        return run_lipschitz_frob<REAL>(h, hs, out_L, V, T, K, s);                                     \
    }                                                                                                  \
    int pb_deconv_##SUF(const REAL *y, const REAL *h, int64_t h_stride, const REAL *L,                 \
                        int64_t L_stride, const REAL *lbda, int64_t lbda_stride, const REAL *w0,       \
                        int nb_iter, int early_stopping, int wind, double tol, REAL *out_x,            \
                        REAL *out_z, REAL *out_dz, REAL *out_J, int32_t *out_niter, int64_t V, int T,  \
                        int K, pb_stream_t s) {                                                        \
        pb::DeconvArgs<REAL> a;                                                                        \
        a.y = y; a.h = h; a.h_stride = h_stride; a.L = L; a.L_stride = L_stride; a.lbda = lbda;        \
        a.lbda_stride = lbda_stride; a.w0 = w0; a.nb_iter = nb_iter;                                   \
        a.early_stopping = early_stopping; a.wind = wind; a.tol = tol; a.out_x = out_x;                \
        a.out_z = out_z; a.out_dz = out_dz; a.out_J = out_J; a.out_niter = out_niter; a.V = V;         \
        a.T = T; a.K = K;                                                                              \
        if (!out_J && V != 0) return PB_ERR_INVALID_ARG;                                               \
        return run_deconv<REAL>(a, s);                                                                 \
    }                                                                                                  \
    int pb_deconv_censored_##SUF(const REAL *y, const REAL *h, int64_t h_stride, const REAL *L,        \
                                 int64_t L_stride, const REAL *lbda, int64_t lbda_stride, const REAL *w0,\
                                 const unsigned char *censor, int64_t censor_stride, int nb_iter,      \
                                 int early_stopping, int wind, double tol, REAL *out_x, REAL *out_z,   \
                                 REAL *out_dz, REAL *out_J, int32_t *out_niter, int64_t V, int T,      \
                                 int K, pb_stream_t s) {                                               \
        pb::DeconvArgs<REAL> a;                                                                        \
        a.y = y; a.h = h; a.h_stride = h_stride; a.L = L; a.L_stride = L_stride; a.lbda = lbda;        \
        a.lbda_stride = lbda_stride; a.w0 = w0; a.nb_iter = nb_iter;                                   \
        a.early_stopping = early_stopping; a.wind = wind; a.tol = tol; a.out_x = out_x;                \
        a.out_z = out_z; a.out_dz = out_dz; a.out_J = out_J; a.out_niter = out_niter; a.V = V;         \
        a.T = T; a.K = K;                                                                              \
        if (!out_J && V != 0) return PB_ERR_INVALID_ARG;                                               \
        const pb::Censor cz{censor, censor_stride};                                                    \
        return run_deconv<REAL>(a, s, &cz);                                                            \
    }                                                                                                  \
    int pb_deconv_masked_##SUF(const REAL *y, const REAL *h, int64_t h_stride, const REAL *L,          \
                               int64_t L_stride, const REAL *lbda, int64_t lbda_stride, const REAL *w0, \
                               const unsigned char *active, int nb_iter, int early_stopping, int wind,  \
                               double tol, REAL *out_x, REAL *out_z, REAL *out_dz, REAL *out_J,         \
                               int32_t *out_niter, int64_t V, int T, int K, pb_stream_t s) {            \
        pb::DeconvArgs<REAL> a;                                                                        \
        a.y = y; a.h = h; a.h_stride = h_stride; a.L = L; a.L_stride = L_stride; a.lbda = lbda;        \
        a.lbda_stride = lbda_stride; a.w0 = w0; a.nb_iter = nb_iter;                                   \
        a.early_stopping = early_stopping; a.wind = wind; a.tol = tol; a.out_x = out_x;                \
        a.out_z = out_z; a.out_dz = out_dz; a.out_J = out_J; a.out_niter = out_niter; a.V = V;         \
        a.T = T; a.K = K; a.active = active;                                                           \
        return run_deconv<REAL>(a, s);                                                                 \
    }                                                                                                  \
    int pb_deconv_auto_##SUF(const REAL *y, const REAL *h, int64_t h_stride, const REAL *L,            \
                             int64_t L_stride, const REAL *sigma, int64_t sigma_stride, int nb_iter,     \
                             int nb_sub_iter, int early_stopping, int wind, double tol, REAL *out_x,     \
                             REAL *out_z, REAL *out_dz, REAL *out_J, REAL *out_R, REAL *out_G,           \
                             REAL *out_lbda, int32_t *out_nouter, int64_t V, int T, int K,               \
                             pb_stream_t s) {                                                            \
        pb::DeconvArgs<REAL> a;                                                                        \
        a.y = y; a.h = h; a.h_stride = h_stride; a.L = L; a.L_stride = L_stride; a.lbda = nullptr;     \
        a.lbda_stride = 0; a.w0 = nullptr; a.nb_iter = nb_sub_iter; a.early_stopping = early_stopping; \
        a.wind = wind; a.tol = tol; a.out_x = out_x; a.out_z = out_z; a.out_dz = out_dz;               \
        a.out_J = out_J; a.out_niter = nullptr; a.V = V; a.T = T; a.K = K;                             \
        a.sigma = sigma; a.sigma_stride = sigma_stride; a.nb_outer = nb_iter; a.out_R = out_R;         \
        a.out_G = out_G; a.out_lbda = out_lbda; a.out_nouter = out_nouter;                             \
        return run_deconv_auto<REAL>(a, s);                                                            \
    }                                                                                                  \
    int pb_deconv_auto_censored_##SUF(const REAL *y, const REAL *h, int64_t h_stride, const REAL *L,   \
                                      int64_t L_stride, const REAL *sigma, int64_t sigma_stride,       \
                                      const unsigned char *censor, int64_t censor_stride, int nb_iter, \
                                      int nb_sub_iter, int early_stopping, int wind, double tol,       \
                                      REAL *out_x, REAL *out_z, REAL *out_dz, REAL *out_J,             \
                                      REAL *out_R, REAL *out_G, REAL *out_lbda, int32_t *out_nouter,   \
                                      int64_t V, int T, int K, pb_stream_t s) {                        \
        pb::DeconvArgs<REAL> a;                                                                        \
        a.y = y; a.h = h; a.h_stride = h_stride; a.L = L; a.L_stride = L_stride; a.lbda = nullptr;     \
        a.lbda_stride = 0; a.w0 = nullptr; a.nb_iter = nb_sub_iter; a.early_stopping = early_stopping; \
        a.wind = wind; a.tol = tol; a.out_x = out_x; a.out_z = out_z; a.out_dz = out_dz;               \
        a.out_J = out_J; a.out_niter = nullptr; a.V = V; a.T = T; a.K = K;                             \
        a.sigma = sigma; a.sigma_stride = sigma_stride; a.nb_outer = nb_iter; a.out_R = out_R;         \
        a.out_G = out_G; a.out_lbda = out_lbda; a.out_nouter = out_nouter;                             \
        const pb::Censor cz{censor, censor_stride};                                                    \
        return run_deconv_auto<REAL>(a, s, &cz);                                                       \
    }                                                                                                  \
    int pb_deconv_lbda_path_censored_##SUF(const REAL *y, const REAL *h, int64_t h_stride,             \
                                           const REAL *L, int64_t L_stride, const REAL *lbdas,         \
                                           int n_lbda, const unsigned char *censor,                    \
                                           int64_t censor_stride, int nb_iter, int early_stopping,     \
                                           int wind, double tol, REAL *out_x, REAL *out_z,             \
                                           REAL *out_dz, REAL *out_J, REAL *out_r, REAL *out_g,        \
                                           int32_t *out_niter, int64_t V, int T, int K,                \
                                           pb_stream_t s) {                                            \
        if (n_lbda < 0 || V < 0 || h_stride < 0 || L_stride < 0) return PB_ERR_INVALID_ARG;          \
        pb::DeconvArgs<REAL> a;                                                                        \
        a.y = y; a.h = h; a.h_stride = h_stride; a.L = L; a.L_stride = L_stride; a.lbda = lbdas;       \
        a.lbda_stride = 0; a.w0 = nullptr; a.nb_iter = nb_iter; a.early_stopping = early_stopping;     \
        a.wind = wind; a.tol = tol; a.out_x = out_x; a.out_z = out_z; a.out_dz = out_dz;               \
        a.out_J = out_J; a.out_r = out_r; a.out_g = out_g; a.out_niter = out_niter;                    \
        a.V = (int64_t)n_lbda * V; a.T = T; a.K = K;                                                   \
        a.y_mod = V; a.lbda_div = V;                                                                   \
        const pb::Censor cz{censor, censor_stride};                                                    \
        return run_deconv<REAL>(a, s, &cz);                                                            \
    }                                                                                                  \
    int pb_deconv_lbda_path_ex_##SUF(const REAL *y, const REAL *h, int64_t h_stride, const REAL *L,    \
                                     int64_t L_stride, const REAL *lbdas, int n_lbda, int nb_iter,     \
                                     int early_stopping, int wind, double tol, REAL *out_x,            \
                                     REAL *out_z, REAL *out_dz, REAL *out_J, REAL *out_r,              \
                                     REAL *out_g, int32_t *out_niter, int64_t V, int T, int K,         \
                                     pb_stream_t s) {                                                  \
        if (n_lbda < 0 || V < 0 || h_stride < 0 || L_stride < 0) return PB_ERR_INVALID_ARG;          \
        pb::DeconvArgs<REAL> a;                                                                        \
        a.y = y; a.h = h; a.h_stride = h_stride; a.L = L; a.L_stride = L_stride; a.lbda = lbdas;       \
        a.lbda_stride = 0; a.w0 = nullptr; a.nb_iter = nb_iter; a.early_stopping = early_stopping;     \
        a.wind = wind; a.tol = tol; a.out_x = out_x; a.out_z = out_z; a.out_dz = out_dz;               \
        a.out_J = out_J; a.out_r = out_r; a.out_g = out_g; a.out_niter = out_niter;                    \
        a.V = (int64_t)n_lbda * V; a.T = T; a.K = K;                                                   \
        a.y_mod = V; a.lbda_div = V;                                                                   \
        return run_deconv<REAL>(a, s);                                                                 \
    }                                                                                                  \
    int pb_deconv_lbda_path_##SUF(const REAL *y, const REAL *h, const REAL *L, const REAL *lbdas,      \
                                  int n_lbda, int nb_iter, REAL *out_x, REAL *out_z, REAL *out_dz,     \
                                  REAL *out_J, int32_t *out_niter, int64_t V, int T, int K,            \
                                  pb_stream_t s) {                                                     \
        return pb_deconv_lbda_path_ex_##SUF(y, h, 0, L, 0, lbdas, n_lbda, nb_iter, 0, 0, 0.0, out_x,   \
                                            out_z, out_dz, out_J, nullptr, nullptr, out_niter, V, T,   \
                                            K, s);                                                     \
    }                                                                                                  \
    int pb_bd_##SUF(const REAL *y, double t_r, double hrf_dur, const REAL *lbda, int64_t lbda_stride,  \
                    const REAL *theta0, int64_t theta0_stride, const REAL *z0, double theta_lo,        \
                    double theta_hi, int nb_iter, int early_stopping, int wind, double tol,            \
                    REAL *out_x, REAL *out_z, REAL *out_dz, REAL *out_h, REAL *out_theta, REAL *out_J, \
                    REAL *out_r, REAL *out_g, int32_t *out_ntrace, int64_t V, int T, int K,            \
                    pb_stream_t s) {                                                                   \
        pb::BdArgs<REAL> a;                                                                            \
        a.y = y; a.lbda = lbda; a.lbda_stride = lbda_stride; a.theta0 = theta0;                        \
        a.theta0_stride = theta0_stride; a.z0 = z0; a.theta_lo = theta_lo; a.theta_hi = theta_hi;      \
        a.nb_iter = nb_iter; a.early_stopping = early_stopping; a.wind = wind; a.tol = tol;            \
        a.out_x = out_x; a.out_z = out_z; a.out_dz = out_dz; a.out_h = out_h;                          \
        a.out_theta = out_theta; a.out_J = out_J; a.out_r = out_r; a.out_g = out_g;                    \
        a.out_ntrace = out_ntrace; a.V = V; a.T = T; a.K = K;                                          \
        return run_bd<REAL>(a, t_r, hrf_dur, s);                                                       \
    }                                                                                                  \
    int pb_transpose_##SUF(const REAL *in, REAL *out, int64_t rows, int64_t cols, pb_stream_t s) {    \
        return run_transpose<REAL>(in, out, rows, cols, s);                                            \
    }                                                                                                  \
    int pb_synth_voxels_##SUF(uint64_t seed, int64_t first_voxel, double t_r, double hrf_dur,         \
                              double snr_db, int nb_events, int blk, double delta_lo, double delta_hi, \
                              REAL *out_y, REAL *out_z, REAL *out_delta, int64_t V, int T,             \
                              pb_stream_t s) {                                                         \
        return run_synth<REAL>(seed, first_voxel, t_r, hrf_dur, snr_db, nb_events, blk, delta_lo,      \
                               delta_hi, out_y, out_z, out_delta, V, T, s);                            \
    }                                                                                                  \
    int pb_inf_norm_##SUF(const REAL *x, REAL *out, int64_t V, int T, pb_stream_t s) {                 \
        return run_inf_norm<REAL>(x, out, V, T, s);                                                    \
    }                                                                                                  \
    int pb_rel_l2_err_##SUF(const REAL *est, const REAL *ref, int64_t ref_stride, REAL *out_err,       \
                            int64_t V, int T, pb_stream_t s) {                                         \
        return run_rel_l2_err<REAL>(est, ref, ref_stride, out_err, V, T, s);                           \
    }                                                                                                  \
    int pb_toeplitz_##SUF(const REAL *k, int klen, REAL *out, int64_t dim_out, int64_t dim_in,         \
                          pb_stream_t s) {                                                             \
        return run_toeplitz<REAL>(k, klen, out, dim_out, dim_in, s);                                   \
    }                                                                                                  \
    int pb_noise_step_##SUF(const REAL *xn, const REAL *zn, const REAL *wn, const REAL *y,             \
                            const REAL *sigma, const unsigned char *active, double mu, REAL *x, REAL *z, \
                            REAL *w, REAL *alpha, REAL *lbda, REAL *out_r, REAL *out_g, int64_t V,     \
                            int T, pb_stream_t s) {                                                    \
        return run_noise_step<REAL>(xn, zn, wn, y, sigma, active, mu, x, z, w, alpha, lbda, out_r,     \
                                    out_g, V, T, s);                                                   \
    }                                                                                                  \
    int pb_mad_##SUF(const REAL *x, double c, REAL *out, int64_t V, int n, pb_stream_t s) {            \
        return run_mad<REAL, 0>(x, c, out, V, n, s);                                                   \
    }                                                                                                  \
    int pb_mad_daub_noise_est_##SUF(const REAL *y, double c, REAL *out_sigma, int64_t V, int T,        \
                                    pb_stream_t s) {                                                   \
        return run_mad<REAL, 1>(y, c, out_sigma, V, T, s);                                             \
    }                                                                                                  \
    int pb_mad_daub_noise_est_censored_##SUF(const REAL *y, const unsigned char *censor,              \
                                             int64_t censor_stride, double c, REAL *out_sigma,         \
                                             int64_t V, int T, pb_stream_t s) {                        \
        return run_mad_censored<REAL>(y, censor, censor_stride, c, out_sigma, V, T, s);                \
    }                                                                                                  \
    int pb_hrf_estim_##SUF(const REAL *z, const REAL *y, double t_r, double hrf_dur,                   \
                           const REAL *theta0, int64_t theta0_stride, double lo, double hi,            \
                           REAL *out_theta, REAL *out_h, REAL *out_cost, int64_t V, int T, int K,      \
                           pb_stream_t s) {                                                            \
        return run_hrf_estim<REAL>(z, y, t_r, hrf_dur, theta0, theta0_stride, lo, hi, out_theta,       \
                                   out_h, out_cost, V, T, K, s);                                       \
    }

PB_DEFINE_OPS(f32, float)
PB_DEFINE_OPS(f64, double)

}  // extern "C"
