// Outer loop of deconv(lbda=None), the noise-constrained lambda (pybold/bold_signal.py:99-214), for one
// voxel inside a persistent deconv kernel:
//
//   alpha = 1, lbda = 1 / (2 alpha), w = 0
//   for i < nb_outer:   inner pass with lbda (momentum from beta_0, empty Q5 window, w warm in registers)
//                       r = ||A w - y||^2, g = ||w||_1
//                       alpha += 1e-4 (r - T sigma^2), lbda = 1 / (2 alpha)   (censored: n_kept, not T)
//                       J[i] = 0.5 r + lbda g, R[i] = r, G[i] = g
//                       early stop: i > wind, |mean(new) - mean(old)| / |mean(new)| < tol over the last
//                       wind alphas (old: the first wind - wind/2, new: the last wind/2)
//   final inner pass with the last lbda: x, z, diff_z
//
// Every kernel family calls pass_done() where an inner pass has ended (the iterate is final for that pass
// and its residual has just been formed) and gets back "next pass with lbda" or "that was the final pass".
// Every lane of the voxel runs the same scalar code on the same (butterfly-reduced, bit-identical) r and g,
// so no broadcast is needed.  alpha, lbda and the window are doubles in both builds; the window is a ring
// of `wind` doubles in shared memory that all lanes of the voxel write with the same value.
#pragma once
#include <math_constants.h>

#include "pb_device.cuh"

namespace pb {

template <typename real>
struct DeconvArgs;

struct NoiseLoop {
    double alpha, lbda;
    double *win;   // ring of the last wind alphas (alpha_i in slot i % wind), used with early stopping
    int i;         // outer iterations done
    bool last;     // the pass under way is the final one

    __device__ __forceinline__ void start(double *win_) {
        alpha = 1.0;                        // bold_signal.py:104
        lbda = 1.0 / (2.0 * alpha);
        win = win_;
        i = 0;
        last = false;
    }

    // An inner pass with `lbda` has ended with r = ||A w - y||^2, g = ||w||_1.  Returns true when it was the
    // final pass (the caller stores x, z, diff_z), else the next pass runs with the updated `lbda`.
    // `writer`: the one lane that stores the scalars; lane q of the nq lanes of the voxel fills the row tails.
    // KEPT (scan censoring): n_kept scans in the data term, r = ||M (A w - y)||^2 is steered toward n_kept sigma^2.
    template <bool KEPT = false, typename real>
    __device__ __forceinline__ bool pass_done(const DeconvArgs<real> &p, int64_t v, double r, double g,
                                              bool writer, int q, int nq, double n_kept = 0.0) {
        const int64_t row = v * (int64_t)p.nb_outer;
        if (last) {
            // complete rows for a C caller: NaN past the voxel's outer count
            const real nan = (real)CUDART_NAN;
            for (int j = i + q; j < p.nb_outer; j += nq) {
                if (p.out_J) p.out_J[row + j] = nan;
                if (p.out_R) p.out_R[row + j] = nan;
                if (p.out_G) p.out_G[row + j] = nan;
            }
            if (writer && p.out_lbda) p.out_lbda[v] = (real)lbda;
            if (writer && p.out_nouter) p.out_nouter[v] = i;
            return true;
        }
        const double s = (double)p.sigma[p.voxel_of(v) * p.sigma_stride];
        if constexpr (KEPT)
            alpha += 1.0e-4 * (r - n_kept * (s * s));
        else
            alpha += 1.0e-4 * (r - (double)p.T * (s * s));     // bold_signal.py:139-145
        lbda = 1.0 / (2.0 * alpha);
        if (writer) {
            if (p.out_J) p.out_J[row + i] = (real)(0.5 * r + lbda * g);
            if (p.out_R) p.out_R[row + i] = (real)r;
            if (p.out_G) p.out_G[row + i] = (real)g;
        }
        bool stop = false;
        if (p.early_stopping) {            // the launcher clears it when wind < 2 (no window, wind / 2 = 0)
            const int wind = p.wind, sub = wind / 2;
            win[i % wind] = alpha;
            if (i > wind) {                // bold_signal.py:164-178; the oldest alpha is in slot (i + 1) % wind
                double so = 0.0, sn = 0.0;
                for (int m = 0, s_ = (i + 1) % wind; m < wind; ++m, s_ = s_ + 1 == wind ? 0 : s_ + 1) {
                    if (m < wind - sub) so += win[s_];
                    else sn += win[s_];
                }
                const double mo = so / (double)(wind - sub), mn = sn / (double)sub;
                stop = fabs(mn - mo) / fabs(mn) < p.tol;
            }
        }
        ++i;
        last = stop || i == p.nb_outer;
        return false;
    }
};

}  // namespace pb
