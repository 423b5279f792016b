/*
 * pybold_b200 -- C ABI of the B200-native batched solver for pyBOLD's hot path.
 *
 * The reference (hcherkaoui/pybold) is pure Python and has no FFI layer; its boundary for
 * this path is the Python signature of `deconv` / `bd` and the duck-typed `op` / `adj`
 * protocol of `pybold/linear.py` (SURVEY.md 8(b)).  Each entry point below names the
 * reference code (file:line, relative to the reference root) whose per-voxel work it
 * replaces for a whole batch of voxels.  `pybold_b200/_lib.py` binds them with ctypes;
 * INTEGRATION.md shows the stub a pyBOLD maintainer would add.
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer.  Arrays are row-major `[V, T]` (T fastest),
 *    `[V, K]` for HRF taps, `[V, n_trace]` for cost traces.
 *  - `*_stride` arguments are ELEMENT strides between voxels for per-voxel parameters;
 *    0 means "one value (or one row) shared by every voxel".
 *  - `_f32` / `_f64` suffix = storage and arithmetic type of the signal arrays.  The HRF
 *    evaluation, the Lipschitz constant and the theta step always run in double.
 *  - All functions are asynchronous on `stream` (a `cudaStream_t` passed as `void*`),
 *    re-entrant, keep no global mutable state and own no memory.
 *  - Return value: 0 on success, a negative `PB_ERR_*` code, or a positive CUDA error
 *    code (`cudaError_t`) passed through.  No exceptions cross the boundary.
 */
#ifndef PYBOLD_B200_H
#define PYBOLD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB_OK 0
#define PB_ERR_INVALID_ARG (-1)  /* null pointer, non-positive size, bad bounds           */
#define PB_ERR_UNSUPPORTED (-2)  /* T, K, nb_iter or wind above the compiled limits        */
#define PB_ERR_NO_DEVICE (-3)    /* no sm_100 kernel image can run on the current device   */

typedef void *pb_stream_t;

/* Library identification / limits. */
int pb_version(void);               /* major*10000 + minor*100 + patch                     */
int pb_max_T(void);                 /* largest number of scans per voxel                   */
int pb_max_K(void);                 /* largest number of HRF taps for the solvers          */
int pb_max_iter(void);              /* largest nb_iter (momentum table lives on chip)      */
const char *pb_error_string(int code);
/* Which kernel a bd call (no early stopping) with this shape dispatches to: 0 = generic
 * shared-memory kernel, otherwise G*1000000 + R*1000 + KMAX of the register-tiled kernel
 * (G lanes per voxel, R samples per lane, KMAX unrolled taps; see DESIGN.md). */
int pb_solver_variant(int T, int K, int is_f64);
/* Voxels that one full wave of the persistent bd grid holds on the current device (0 when the
 * shape runs on a kernel without that notion).  Hosts that stream a large batch in chunks should
 * cut it at multiples of this number. */
int pb_bd_wave_voxels(int T, int K, int is_f64, int nb_iter);
/* Which kernel a deconvolution with this shape runs on the current device: pb_deconv / pb_deconv_masked /
 * pb_deconv_lbda_path(_ex) with (nb_iter, early_stopping, wind), or pb_deconv_auto (is_auto != 0, nb_iter the
 * inner count nb_sub_iter).  Returns the variant in the encoding of pb_solver_variant (0 = generic kernel) and
 * the family in *family: 0 generic, 1 group, 2 warp per voxel, 3 CTA per voxel (a one-warp CTA and a warp
 * variant can share an id).  The choice is the launch's own, shared-memory and occupancy checks included.
 * Negative PB_ERR_* on bad arguments, shapes beyond the limits, or PB_ERR_NO_DEVICE. */
int pb_deconv_variant(int T, int K, int is_f64, int nb_iter, int early_stopping, int wind, int is_auto,
                      int *family);
/* Which kernel a pb_bd_f32 / pb_bd_f64 call with this shape and (nb_iter, early_stopping, wind) runs on the current
 * device, in the encoding and with the family codes and errors of pb_deconv_variant.  The choice is the launch's
 * own, shared-memory and occupancy checks included.  With early_stopping = 0 the id is pb_solver_variant's. */
int pb_bd_variant(int T, int K, int is_f64, int nb_iter, int early_stopping, int wind, int *family);

/* ---- A1: DiscretInteg.op / .adj (pybold/linear.py:15-28, :30-43) -------------------- */
int pb_integ_op_f32(const float *x, float *out, int64_t V, int T, pb_stream_t stream);
int pb_integ_op_f64(const double *x, double *out, int64_t V, int T, pb_stream_t stream);
int pb_integ_adj_f32(const float *x, float *out, int64_t V, int T, pb_stream_t stream);
int pb_integ_adj_f64(const double *x, double *out, int64_t V, int T, pb_stream_t stream);

/* ---- A5: simple_convolve / spectral_convolve and their retro (adjoint) versions ------
 * out[v,i] = sum_j h[j] x[v,i-j]   (pybold/convolution.py:9-30, :135-164; K.dot, linear.py:91)
 * out[v,i] = sum_j h[j] x[v,i+j]   (pybold/convolution.py:33-54, :167-196; K.T.dot, linear.py:111) */
int pb_conv_op_f32(const float *h, int64_t h_stride, const float *x, float *out,
                   int64_t V, int T, int K, pb_stream_t stream);
int pb_conv_op_f64(const double *h, int64_t h_stride, const double *x, double *out,
                   int64_t V, int T, int K, pb_stream_t stream);
int pb_conv_adj_f32(const float *h, int64_t h_stride, const float *x, float *out,
                    int64_t V, int T, int K, pb_stream_t stream);
int pb_conv_adj_f64(const double *h, int64_t h_stride, const double *x, double *out,
                    int64_t V, int T, int K, pb_stream_t stream);

/* ---- A2: ConvAndLinear(DiscretInteg(), h).op / .adj (pybold/linear.py:73-113) --------
 * op: conv(h, cumsum(x));  adj: reversed-cumsum(corr(h, x)). */
int pb_hrfinteg_op_f32(const float *h, int64_t h_stride, const float *x, float *out,
                       int64_t V, int T, int K, pb_stream_t stream);
int pb_hrfinteg_op_f64(const double *h, int64_t h_stride, const double *x, double *out,
                       int64_t V, int T, int K, pb_stream_t stream);
int pb_hrfinteg_adj_f32(const float *h, int64_t h_stride, const float *x, float *out,
                        int64_t V, int T, int K, pb_stream_t stream);
int pb_hrfinteg_adj_f64(const double *h, int64_t h_stride, const double *x, double *out,
                        int64_t V, int T, int K, pb_stream_t stream);

/* ---- A9: spm_hrf (pybold/hrf_model.py:12-39) ------------------------------------------
 * out_h[v, m] for m < K, K = pb_hrf_len(t_r, dur).  `normalized` != 0 divides by the
 * maximum over the reference's 1 ms grid (hrf_model.py:33-34).  theta outside [0.5, 2]
 * is the caller's error to raise (hrf_model.py:17-21); the kernel writes NaN taps. */
int pb_hrf_len(double t_r, double dur);
int pb_spm_hrf_f32(const float *theta, double t_r, double dur, int normalized,
                   float *out_h, int64_t V, int K, pb_stream_t stream);
int pb_spm_hrf_f64(const double *theta, double t_r, double dur, int normalized,
                   double *out_h, int64_t V, int K, pb_stream_t stream);
/* Same with the shape parameters of the reference's signature (hrf_model.py:12-14):
 * shape7 (HOST pointer, read during the call) = {dt, p_delay, undershoot, p_disp, u_disp,
 * p_u_ratio, onset}; K = pb_hrf_len_ex(t_r, dur, dt).  Like the reference, the time axis is
 * shifted by onset / dt (hrf_model.py:25). */
int pb_hrf_len_ex(double t_r, double dur, double dt);
int pb_spm_hrf_ex_f32(const float *theta, double t_r, double dur, int normalized,
                      const double *shape7, float *out_h, int64_t V, int K, pb_stream_t stream);
int pb_spm_hrf_ex_f64(const double *theta, double t_r, double dur, int normalized,
                      const double *shape7, double *out_h, int64_t V, int K, pb_stream_t stream);

/* ---- A4: spectral_radius_est (pybold/utils.py:94-109) ---------------------------------
 * Power iteration on A^T A, A = conv(h) o cumsum, from the supplied start x0 (the reference
 * draws it from the global NumPy RNG).  out_L[v] = ||x_new|| (NOT multiplied by 0.9). */
int pb_lipschitz_power_f32(const float *h, int64_t h_stride, const float *x0, int64_t x0_stride,
                           int nb_iter, double tol, float *out_L,
                           int64_t V, int T, int K, pb_stream_t stream);
int pb_lipschitz_power_f64(const double *h, int64_t h_stride, const double *x0, int64_t x0_stride,
                           int nb_iter, double tol, double *out_L,
                           int64_t V, int T, int K, pb_stream_t stream);

/* ---- A6 (setup): ||A^T A||_F of _loops_deconv (pybold/bold_signal.py:249-253) -------- */
int pb_lipschitz_frob_f32(const float *h, int64_t h_stride, float *out_L,
                          int64_t V, int T, int K, pb_stream_t stream);
int pb_lipschitz_frob_f64(const double *h, int64_t h_stride, double *out_L,
                          int64_t V, int T, int K, pb_stream_t stream);

/* ---- A3: deconv, fixed lambda (pybold/bold_signal.py:49-97) ---------------------------
 * One persistent kernel: all `nb_iter` iterations of the (aliased, SURVEY.md Q1) recursion
 * with the voxel resident on chip.
 *   L[v*L_stride]       gradient Lipschitz constant actually used (0.9 * power estimate)
 *   lbda[v*lbda_stride] regularisation
 *   w0                  optional warm start [V,T] (NULL = zeros, the reference's start)
 *   out_J [V, nb_iter]  J_k = 0.5||x_k-y||^2 + lbda||w_k||_1, UN-normalised; entries at and
 *                       after out_niter[v] are left untouched
 *   out_niter [V]       iterations executed (early stop, Q5)
 * out_x / out_z / out_dz = x, z, diff_z of the reference's return tuple. */
int pb_deconv_f32(const float *y, const float *h, int64_t h_stride,
                  const float *L, int64_t L_stride, const float *lbda, int64_t lbda_stride,
                  const float *w0, int nb_iter, int early_stopping, int wind, double tol,
                  float *out_x, float *out_z, float *out_dz, float *out_J, int32_t *out_niter,
                  int64_t V, int T, int K, pb_stream_t stream);
int pb_deconv_f64(const double *y, const double *h, int64_t h_stride,
                  const double *L, int64_t L_stride, const double *lbda, int64_t lbda_stride,
                  const double *w0, int nb_iter, int early_stopping, int wind, double tol,
                  double *out_x, double *out_z, double *out_dz, double *out_J, int32_t *out_niter,
                  int64_t V, int T, int K, pb_stream_t stream);

/* ---- A7 (+A6, A9, A10): bd, semi-blind deconvolution (pybold/bold_signal.py:281-382) --
 * One persistent kernel per batch: outer loop of { Frobenius Lipschitz, nb_iter inner
 * prox-gradient iterations (the outer count is forwarded, Q3), bounded theta step on
 * 0.5||y - h(theta)*z||^2, cost trace }, then the final inner loop.
 *   theta0[v*theta0_stride]  start dilation (reference default MAX_DELTA = 2.0)
 *   z0                       optional warm start [V,T] (NULL = zeros)
 *   theta_lo / theta_hi      bounds of the theta step (reference default 0.6 / 1.9)
 *   out_h [V,K] non-normalised taps; out_theta [V];
 *   out_J / out_r / out_g [V, nb_iter+2] as d['J'], d['r'], d['g']; out_ntrace [V] = number
 *   of valid trace entries (nb_iter+2 unless the outer early stop fired, Q7). */
int pb_bd_f32(const float *y, double t_r, double hrf_dur,
              const float *lbda, int64_t lbda_stride, const float *theta0, int64_t theta0_stride,
              const float *z0, double theta_lo, double theta_hi,
              int nb_iter, int early_stopping, int wind, double tol,
              float *out_x, float *out_z, float *out_dz, float *out_h, float *out_theta,
              float *out_J, float *out_r, float *out_g, int32_t *out_ntrace,
              int64_t V, int T, int K, pb_stream_t stream);
int pb_bd_f64(const double *y, double t_r, double hrf_dur,
              const double *lbda, int64_t lbda_stride, const double *theta0, int64_t theta0_stride,
              const double *z0, double theta_lo, double theta_hi,
              int nb_iter, int early_stopping, int wind, double tol,
              double *out_x, double *out_z, double *out_dz, double *out_h, double *out_theta,
              double *out_J, double *out_r, double *out_g, int32_t *out_ntrace,
              int64_t V, int T, int K, pb_stream_t stream);

/* Same solve for a SUBSET of the batch: voxels with active[v] == 0 are skipped and their output rows stay
 * untouched; out_J may be NULL (no cost trace).  This is the inner loop of `deconv(lbda=None)`
 * (pybold/bold_signal.py:114-138), which the outer lambda loop calls again and again, warm-started through
 * w0, while more and more voxels have met their stopping rule. */
int pb_deconv_masked_f32(const float *y, const float *h, int64_t h_stride, const float *L, int64_t L_stride,
                         const float *lbda, int64_t lbda_stride, const float *w0, const unsigned char *active,
                         int nb_iter, int early_stopping, int wind, double tol, float *out_x, float *out_z,
                         float *out_dz, float *out_J, int32_t *out_niter, int64_t V, int T, int K,
                         pb_stream_t stream);
int pb_deconv_masked_f64(const double *y, const double *h, int64_t h_stride, const double *L, int64_t L_stride,
                         const double *lbda, int64_t lbda_stride, const double *w0, const unsigned char *active,
                         int nb_iter, int early_stopping, int wind, double tol, double *out_x, double *out_z,
                         double *out_dz, double *out_J, int32_t *out_niter, int64_t V, int T, int K,
                         pb_stream_t stream);

/* ---- N1: `deconv(lbda=None)`, the noise-constrained lambda (pybold/bold_signal.py:99-214), in ONE launch: every
 * voxel runs its outer loop inside the deconv kernel -- alpha = 1, lbda = 1 / (2 alpha); per outer iteration an
 * inner pass of at most nb_sub_iter prox-gradient iterations (warm start, Q5 early stop), then
 * alpha += 1e-4 (||x - y||^2 - T sigma^2), lbda = 1 / (2 alpha) and the alpha-window stop (`early_stopping`, `wind`,
 * `tol`); then one final inner pass with the last lambda.  Asynchronous on `stream`.
 *   h[v*h_stride + k], L[v*L_stride], sigma[v*sigma_stride]   taps, Lipschitz constant, noise level (strides 0: shared)
 *   nb_iter >= 1            outer iterations at most; nb_sub_iter <= pb_max_iter() inner iterations per pass
 *   out_x, out_z, out_dz    [V,T] from the final pass
 *   out_J, out_R, out_G     [V, nb_iter]: 0.5 R + lbda G (with the updated lbda), ||x - y||^2, ||diff_z||_1 of every
 *                           outer iteration, NaN past the voxel's outer count
 *   out_lbda [V]            the lambda of the final pass;  out_nouter [V]  outer iterations done
 * out_J, out_R, out_G, out_lbda and out_nouter may be NULL (not written).
 * A voxel whose sigma is NaN gets the reference's result: out_x, out_z, out_dz, out_J and out_lbda NaN, out_R and
 * out_G NaN from the second outer iteration on, out_nouter = nb_iter.  Other voxels are not affected.  The censored
 * entry points below do the same. */
int pb_deconv_auto_f32(const float *y, const float *h, int64_t h_stride, const float *L, int64_t L_stride,
                       const float *sigma, int64_t sigma_stride, int nb_iter, int nb_sub_iter, int early_stopping,
                       int wind, double tol, float *out_x, float *out_z, float *out_dz, float *out_J, float *out_R,
                       float *out_G, float *out_lbda, int32_t *out_nouter, int64_t V, int T, int K,
                       pb_stream_t stream);
int pb_deconv_auto_f64(const double *y, const double *h, int64_t h_stride, const double *L, int64_t L_stride,
                       const double *sigma, int64_t sigma_stride, int nb_iter, int nb_sub_iter, int early_stopping,
                       int wind, double tol, double *out_x, double *out_z, double *out_dz, double *out_J,
                       double *out_R, double *out_G, double *out_lbda, int32_t *out_nouter, int64_t V, int T,
                       int K, pb_stream_t stream);

/* ---- cfg5: regularisation path, `deconv` (fixed lambda, no early stopping, pybold/bold_signal.py:49-97)
 * for every lambda of lbdas[n_lbda] and every voxel of y[V,T] in one launch -- the lambda grid search of
 * examples/icassp_2019/validation.py batched over (lambda, voxel).  Problem (l, v) reads row v of y (the
 * rows are NOT replicated per lambda) and lbdas[l]; h[K] and L[1] are shared.  Outputs are lambda-major:
 * out_x, out_z, out_dz [n_lbda, V, T], out_J [n_lbda, V, nb_iter] (raw costs), out_niter [n_lbda * V]. */
int pb_deconv_lbda_path_f32(const float *y, const float *h, const float *L, const float *lbdas, int n_lbda,
                            int nb_iter, float *out_x, float *out_z, float *out_dz, float *out_J,
                            int32_t *out_niter, int64_t V, int T, int K, pb_stream_t stream);
int pb_deconv_lbda_path_f64(const double *y, const double *h, const double *L, const double *lbdas,
                            int n_lbda, int nb_iter, double *out_x, double *out_z, double *out_dz,
                            double *out_J, int32_t *out_niter, int64_t V, int T, int K, pb_stream_t stream);

/* Same path with per-voxel HRFs, the reference's early stop and the cost terms of every problem -- a loop of
 * `deconv(y, t_r, h, lbda=l, early_stopping=..., tol=..., wind=...)` over lbdas, in one launch.
 *   h[v*h_stride + k], L[v*L_stride]   taps and Lipschitz constant of voxel v (strides 0: shared)
 *   early_stopping, wind, tol          as in pb_deconv_*: out_niter[l*V + v] = iterations done, out_J rows are
 *                                      written up to it (the caller fills the tail, e.g. with NaN)
 *   out_r, out_g [n_lbda * V]          terms of the final cost J = 0.5 R + lambda G of each problem:
 *                                      R = ||x - y||^2, G = ||diff_z||_1, in the working precision
 * out_J, out_r and out_g may be NULL (not written).  out_x, out_z, out_dz are always written; a caller that
 * only wants the cost terms cuts V into ranges and reuses the same solution buffers range after range. */
int pb_deconv_lbda_path_ex_f32(const float *y, const float *h, int64_t h_stride, const float *L, int64_t L_stride,
                               const float *lbdas, int n_lbda, int nb_iter, int early_stopping, int wind,
                               double tol, float *out_x, float *out_z, float *out_dz, float *out_J, float *out_r,
                               float *out_g, int32_t *out_niter, int64_t V, int T, int K, pb_stream_t stream);
int pb_deconv_lbda_path_ex_f64(const double *y, const double *h, int64_t h_stride, const double *L,
                               int64_t L_stride, const double *lbdas, int n_lbda, int nb_iter, int early_stopping,
                               int wind, double tol, double *out_x, double *out_z, double *out_dz, double *out_J,
                               double *out_r, double *out_g, int32_t *out_niter, int64_t V, int T, int K,
                               pb_stream_t stream);

/* ---- Scan censoring for deconv, deconv(lbda=None) and the lambda path (no reference counterpart).
 * Volumes flagged for head motion ("scrubbing") stay on the model's time grid and leave the data term:
 *   min_w 1/2 ||M (A w - y)||^2 + lbda ||w||_1,   M = diag(1 - censor)
 *   censor[v*censor_stride + i] != 0   scan i of voxel v is left out (uint8; censor_stride 0: one [T] mask for the
 *                                      batch, T: one row per voxel; for the path, per voxel of y, not per problem)
 *   y                                  read as 0 on censored scans: NaN or Inf there are ignored
 *   out_x                              A w on EVERY scan (the model's prediction at the gaps); z, diff_z likewise
 *   out_J, out_r / out_R               with the masked residual M (A w - y)
 *   L                                  the caller's Lipschitz constant; the censored operator's is 0.9 x
 *                                      pb_lipschitz_power_censored_* from the same start
 *   deconv(lbda=None)                  alpha += 1e-4 (||M (x - y)||^2 - n_kept sigma^2), n_kept = the voxel's kept scans
 * Precondition: every voxel keeps at least one scan (an all-censored voxel has a zero operator and no Lipschitz
 * constant).  Otherwise each entry point takes the arguments of its uncensored twin and behaves like it; calls run
 * on the register-tiled CTA kernels wherever one fits (pb_deconv_censored_variant), else on the generic kernel. */
int pb_deconv_censored_f32(const float *y, const float *h, int64_t h_stride, const float *L, int64_t L_stride,
                           const float *lbda, int64_t lbda_stride, const float *w0, const unsigned char *censor,
                           int64_t censor_stride, int nb_iter, int early_stopping, int wind, double tol, float *out_x,
                           float *out_z, float *out_dz, float *out_J, int32_t *out_niter, int64_t V, int T, int K,
                           pb_stream_t stream);
int pb_deconv_censored_f64(const double *y, const double *h, int64_t h_stride, const double *L, int64_t L_stride,
                           const double *lbda, int64_t lbda_stride, const double *w0, const unsigned char *censor,
                           int64_t censor_stride, int nb_iter, int early_stopping, int wind, double tol,
                           double *out_x, double *out_z, double *out_dz, double *out_J, int32_t *out_niter,
                           int64_t V, int T, int K, pb_stream_t stream);
int pb_deconv_auto_censored_f32(const float *y, const float *h, int64_t h_stride, const float *L, int64_t L_stride,
                                const float *sigma, int64_t sigma_stride, const unsigned char *censor,
                                int64_t censor_stride, int nb_iter, int nb_sub_iter, int early_stopping, int wind,
                                double tol, float *out_x, float *out_z, float *out_dz, float *out_J, float *out_R,
                                float *out_G, float *out_lbda, int32_t *out_nouter, int64_t V, int T, int K,
                                pb_stream_t stream);
int pb_deconv_auto_censored_f64(const double *y, const double *h, int64_t h_stride, const double *L,
                                int64_t L_stride, const double *sigma, int64_t sigma_stride,
                                const unsigned char *censor, int64_t censor_stride, int nb_iter, int nb_sub_iter,
                                int early_stopping, int wind, double tol, double *out_x, double *out_z,
                                double *out_dz, double *out_J, double *out_R, double *out_G, double *out_lbda,
                                int32_t *out_nouter, int64_t V, int T, int K, pb_stream_t stream);
int pb_deconv_lbda_path_censored_f32(const float *y, const float *h, int64_t h_stride, const float *L,
                                     int64_t L_stride, const float *lbdas, int n_lbda, const unsigned char *censor,
                                     int64_t censor_stride, int nb_iter, int early_stopping, int wind, double tol,
                                     float *out_x, float *out_z, float *out_dz, float *out_J, float *out_r,
                                     float *out_g, int32_t *out_niter, int64_t V, int T, int K, pb_stream_t stream);
int pb_deconv_lbda_path_censored_f64(const double *y, const double *h, int64_t h_stride, const double *L,
                                     int64_t L_stride, const double *lbdas, int n_lbda, const unsigned char *censor,
                                     int64_t censor_stride, int nb_iter, int early_stopping, int wind, double tol,
                                     double *out_x, double *out_z, double *out_dz, double *out_J, double *out_r,
                                     double *out_g, int32_t *out_niter, int64_t V, int T, int K, pb_stream_t stream);
/* Power iteration on A^T M A, M applied between op and adj (arguments of pb_lipschitz_power_*, mask as above). */
int pb_lipschitz_power_censored_f32(const float *h, int64_t h_stride, const float *x0, int64_t x0_stride,
                                    const unsigned char *censor, int64_t censor_stride, int nb_iter, double tol,
                                    float *out_L, int64_t V, int T, int K, pb_stream_t stream);
int pb_lipschitz_power_censored_f64(const double *h, int64_t h_stride, const double *x0, int64_t x0_stride,
                                    const unsigned char *censor, int64_t censor_stride, int nb_iter, double tol,
                                    double *out_L, int64_t V, int T, int K, pb_stream_t stream);
/* pb_mad_daub_noise_est over the level-1 db3 detail coefficients that touch no censored scan (a coefficient reads
 * six samples, after the symmetric extension; T < 10: the kept samples).  NaN for a voxel with none left, and, as for
 * pb_mad_daub_noise_est, for one with a NaN or an infinite median among its kept coefficients. */
int pb_mad_daub_noise_est_censored_f32(const float *y, const unsigned char *censor, int64_t censor_stride, double c,
                                       float *out_sigma, int64_t V, int T, pb_stream_t stream);
int pb_mad_daub_noise_est_censored_f64(const double *y, const unsigned char *censor, int64_t censor_stride,
                                       double c, double *out_sigma, int64_t V, int T, pb_stream_t stream);
/* The kernel a censored deconv call of this shape runs on, in the encoding, family codes and V = 0 routing of
 * pb_deconv_variant (3 = CTA, 0 = generic). */
int pb_deconv_censored_variant(int T, int K, int is_f64, int nb_iter, int early_stopping, int wind, int is_auto,
                               int *family);

/* ---- A10: the theta step alone / hrf_estim (pybold/bold_signal.py:217-239, :329-334) --
 * theta[v] <- bounded local minimiser of 0.5||y_v - h(theta)*z_v||^2 from theta0;
 * out_h [V,K] = non-normalised taps at the minimiser; out_cost [V] = the cost there. */
int pb_hrf_estim_f32(const float *z, const float *y, double t_r, double hrf_dur,
                     const float *theta0, int64_t theta0_stride, double theta_lo, double theta_hi,
                     float *out_theta, float *out_h, float *out_cost,
                     int64_t V, int T, int K, pb_stream_t stream);
int pb_hrf_estim_f64(const double *z, const double *y, double t_r, double hrf_dur,
                     const double *theta0, int64_t theta0_stride, double theta_lo, double theta_hi,
                     double *out_theta, double *out_h, double *out_cost,
                     int64_t V, int T, int K, pb_stream_t stream);

/* Dense Toeplitz matrix of k.conv(.): out[i, c] = k[i - c] for 0 <= i - c < klen, else 0; out is
 * [dim_out, dim_in] row-major.  pybold/convolution.py:105-132 (`toeplitz_from_kernel`).  The solvers never
 * form this matrix; it serves callers of the reference's convolution module. */
int pb_toeplitz_f32(const float *k, int klen, float *out, int64_t dim_out, int64_t dim_in, pb_stream_t stream);
int pb_toeplitz_f64(const double *k, int klen, double *out, int64_t dim_out, int64_t dim_in, pb_stream_t stream);

/* ---- N3: on-device synthetic voxels and the post-processing of the ICASSP-2019 simulation.
 * pb_synth_voxels: the batch that `examples/icassp_2019/simulation.py:27-48` builds one voxel at a time
 * with `gen_rnd_bloc_bold` (pybold/data.py:243-400): `nb_events` unit boxcars of `blk` samples, the
 * normalised SPM HRF at a per-voxel dilation in [delta_lo, delta_hi], Gaussian noise at `snr_db`
 * (scaling rule of pybold/data.py:439-444).  Own counter-based generator ("philox-v1", csrc/pb_synth.cuh;
 * NumPy restatement in pybold_b200/synth.py): voxel `first_voxel + v` gets the same numbers on every
 * rank and for every batch split.  out_z (block signal) and out_delta may be null.  nb_events <= 31.
 * pb_inf_norm: out[v,:] = x[v,:] / (max|x[v,:]| + 1e-12)  (pybold/utils.py:112-138, 2-D input, axis=1).
 * pb_rel_l2_err: err[v] = ||est[v,:] - ref[v,:]|| / ||ref[v,:]||  (simulation.py:143-147); ref_stride = 0
 * compares every voxel with one reference row. */
int pb_synth_voxels_f32(uint64_t seed, int64_t first_voxel, double t_r, double hrf_dur, double snr_db,
                        int nb_events, int blk, double delta_lo, double delta_hi, float *out_y,
                        float *out_z, float *out_delta, int64_t V, int T, pb_stream_t stream);
int pb_synth_voxels_f64(uint64_t seed, int64_t first_voxel, double t_r, double hrf_dur, double snr_db,
                        int nb_events, int blk, double delta_lo, double delta_hi, double *out_y,
                        double *out_z, double *out_delta, int64_t V, int T, pb_stream_t stream);
int pb_inf_norm_f32(const float *x, float *out, int64_t V, int T, pb_stream_t stream);
int pb_inf_norm_f64(const double *x, double *out, int64_t V, int T, pb_stream_t stream);
int pb_rel_l2_err_f32(const float *est, const float *ref, int64_t ref_stride, float *out_err,
                      int64_t V, int T, pb_stream_t stream);
int pb_rel_l2_err_f64(const double *est, const double *ref, int64_t ref_stride, double *out_err,
                      int64_t V, int T, pb_stream_t stream);

/* ---- A8 / N1: noise level of `deconv(lbda=None)` (pybold/utils.py:10-25, called at
 * pybold/bold_signal.py:103).  pb_mad: out[v] = median(|x_v - median(x_v)|) / c for the rows of
 * x[V, n] (`mad`, utils.py:10-13).  pb_mad_daub_noise_est: the same statistic of the level-1 db3
 * detail coefficients of y[V, T] (PyWavelets "symmetric" extension, floor((T + 5) / 2)
 * coefficients; T < 10 has no level-1 decomposition and takes the series itself, the reference's
 * `except ValueError` branch, utils.py:23-24).  Medians are exact order statistics.  A row holding a NaN gives NaN,
 * like NumPy's median, and so does a row whose median is +-inf (its deviation there is inf - inf). */
int pb_mad_f32(const float *x, double c, float *out, int64_t V, int n, pb_stream_t stream);
int pb_mad_f64(const double *x, double c, double *out, int64_t V, int n, pb_stream_t stream);
int pb_mad_daub_noise_est_f32(const float *y, double c, float *out_sigma, int64_t V, int T,
                              pb_stream_t stream);
int pb_mad_daub_noise_est_f64(const double *y, double c, double *out_sigma, int64_t V, int T,
                              pb_stream_t stream);

/* ---- N1: one outer iteration of the noise-constrained lambda loop of `deconv(lbda=None)`
 * (pybold/bold_signal.py:139-162) for the whole batch: voxels with active[v] != 0 take the new inner-loop
 * result (x, z, w <- xn, zn, wn), then r[v] = ||x - y||^2, g[v] = ||w||_1,
 * alpha[v] += mu (r[v] - T sigma[v]^2) (active voxels only) and lbda[v] = 1 / (2 alpha[v]). */
int pb_noise_step_f32(const float *xn, const float *zn, const float *wn, const float *y, const float *sigma,
                      const unsigned char *active, double mu, float *x, float *z, float *w, float *alpha,
                      float *lbda, float *out_r, float *out_g, int64_t V, int T, pb_stream_t stream);
int pb_noise_step_f64(const double *xn, const double *zn, const double *wn, const double *y,
                      const double *sigma, const unsigned char *active, double mu, double *x, double *z,
                      double *w, double *alpha, double *lbda, double *out_r, double *out_g, int64_t V, int T,
                      pb_stream_t stream);

/* ---- N4: layout adapter between the reference pipeline's time-major voxel matrices [T, V]
 * (`NiftiMasker.fit_transform`, consumed as `voxels.T`, examples/icassp_2019/validation.py:90-103)
 * and the solvers' [V, T]: out[c, r] = in[r, c] for an in[rows, cols] row-major matrix.  Out of place
 * (in != out); rows <= 2 097 120. */
int pb_transpose_f32(const float *in, float *out, int64_t rows, int64_t cols, pb_stream_t stream);
int pb_transpose_f64(const double *in, double *out, int64_t rows, int64_t cols, pb_stream_t stream);

/* ---- 8(e): one asynchronous copy between device buffers of this or of a PEER GPU (unified addressing:
 * `dst` may be a CUDA-IPC mapping of another rank's result tensor).  A plain cudaMemcpyAsync on `stream`:
 * the copy engines move the slab over NVLink while the SMs keep solving.  Used by the peer gather of
 * pybold_b200/sharding.py; the reference gathers its per-voxel results by pickling them back from the
 * joblib workers (examples/icassp_2019/validation.py:43-47). */
int pb_copy_async(void *dst, const void *src, size_t bytes, pb_stream_t stream);

/* ---- measurement utility (not part of the reference API) --------------------------------
 * FP32 FMA-pipe microbenchmark reported beside the nominal roofline (SURVEY.md 8(d)): launches
 * `blocks` CTAs of 256 threads (use 4 per SM), each thread running 16 independent chains of
 * `iters` FFMA.  Executed flops = blocks * 256 * 16 * iters * 2.  `sink` holds blocks*256 floats. */
int pb_bench_fma_f32(float *sink, int blocks, int iters, pb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PYBOLD_B200_H */
