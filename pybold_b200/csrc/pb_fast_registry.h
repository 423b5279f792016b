// Register-tiled solver variants (pb_fast.cuh, pb_fastg.cuh, pb_fastc.cuh) and their dispatch.
// gen_fast_instances.py writes one translation unit per variant into build/gen/ at build time, so
// that they compile in parallel, each defining one Variant, plus the table pb_fast_registry.cu
// picks from by (T, K, dtype).
#pragma once
#include <cuda_runtime.h>

#include "pb_generic.cuh"

namespace pb {

constexpr int FAST_NO_MATCH = -1000;

// the variant that ran (id as fast_variant_id, family a VariantFamily) go to *id / *family when given; the
// generic kernel is the caller's step after FAST_NO_MATCH.  V == 0: nothing is launched, the result and the
// variant are those a launch would have
int fast_deconv_dispatch(const DeconvArgs<float> &a, cudaStream_t stream, int *id = nullptr, int *family = nullptr);
int fast_deconv_dispatch(const DeconvArgs<double> &a, cudaStream_t stream, int *id = nullptr, int *family = nullptr);
// censored deconv (Censor, pb_generic.cuh): the cheapest CTA row with a censored entry point that serves (T, K); the
// generic kernel is the caller's step after FAST_NO_MATCH
int fast_deconv_censored_dispatch(const DeconvArgs<float> &a, const Censor &cz, cudaStream_t stream, int *id = nullptr,
                                  int *family = nullptr);
int fast_deconv_censored_dispatch(const DeconvArgs<double> &a, const Censor &cz, cudaStream_t stream, int *id = nullptr,
                                  int *family = nullptr);
int fast_bd_dispatch(const BdArgs<float> &a, cudaStream_t stream, int *id = nullptr, int *family = nullptr);
int fast_bd_dispatch(const BdArgs<double> &a, cudaStream_t stream, int *id = nullptr, int *family = nullptr);
// 0 = generic kernel, else lanes per voxel * 1000000 + R * 1000 + KMAX
int fast_variant_id(int T, int K, bool is_f64);
// voxels per full wave of the persistent bd grid (0 when unknown): batch sizes that are multiples
// of it waste no tail
int fast_bd_wave_voxels(int T, int K, bool is_f64, int nb_iter);

// bd runs the cheapest matching variant of tier 0 (group and CTA variants) and falls back to the cheapest
// warp-per-voxel variant only when that launch returns FAST_NO_MATCH (bd_dispatch).  deconv goes through the
// families in the order group, warp, CTA, then the generic kernel (deconv_dispatch, pb_fast_registry.cu).
enum VariantTier { TIER_GROUP_CTA = 0, TIER_WARP = 1 };
// the kernel family a call ran on (the *family of pb_deconv_variant and pb_bd_variant)
enum VariantFamily { FAMILY_GENERIC = 0, FAMILY_GROUP = 1, FAMILY_WARP = 2, FAMILY_CTA = 3 };

template <typename real>
struct Variant {
    int tier;
    int lanes;          // lanes per voxel: G (group), 32 NW (CTA), 32 (warp)
    int R, KMAX, TAIL;  // samples per lane, unrolled taps, maskable tail slots (group)
    bool circ;          // wrap-around warp variant
    // entry points; null: the variant has none
    bool (*ok)(int T, int K);
    int (*bd)(const BdArgs<real> &, cudaStream_t);
    int (*bd_es)(const BdArgs<real> &, cudaStream_t);  // bd with early stopping (Q6 / Q7)
    int (*deconv)(const DeconvArgs<real> &, cudaStream_t);
    int (*wave)(int nb_iter);
    // deconv(lbda=None): DeconvArgs::nb_outer > 0, the noise loop inside the kernel (pb_noise_loop.cuh)
    int (*deconv_auto)(const DeconvArgs<real> &, cudaStream_t);
    // scan censoring (CTA rows only): the shapes a censored call may take, deconv and deconv(lbda=None)
    bool (*ok_censored)(int T, int K);
    int (*deconv_censored)(const DeconvArgs<real> &, const Censor &, cudaStream_t);
    int (*deconv_auto_censored)(const DeconvArgs<real> &, const Censor &, cudaStream_t);
};

// Whether a kernel of `threads` threads and `smem` bytes of dynamic shared memory per CTA can run:
// FAST_NO_MATCH when it does not fit (shared memory beyond the opt-in limit, or no resident CTA), else 0 with
// the resident CTAs per SM in *occ and the SM count in *sms, or the CUDA error.
template <typename Kern>
int persistent_fit(Kern kern, int threads, size_t smem, int *occ, int *sms) {
    int dev = 0, max_smem = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (smem > (size_t)max_smem) return FAST_NO_MATCH;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, kern, threads, smem);
    if (e != cudaSuccess) return (int)e;
    return *occ < 1 ? FAST_NO_MATCH : 0;
}

// Launches a persistent kernel of `threads` threads and `smem` bytes of dynamic shared memory per
// CTA: as many CTAs as fit on the device at once, at most one per `voxels_per_cta` voxels.  Returns
// persistent_fit's FAST_NO_MATCH or CUDA error, else 0 or the CUDA error of the launch.  A work-queue counter,
// when given, is zeroed on the stream first.  V == 0 launches nothing: only the fit is checked.
template <typename Kern, typename... Args>
int launch_persistent(Kern kern, int threads, size_t smem, int voxels_per_cta, int64_t V,
                      unsigned int *queue, cudaStream_t stream, const Args &...args) {
    int sms = 0, occ = 0;
    const int fit = persistent_fit(kern, threads, smem, &occ, &sms);
    if (fit != 0 || V == 0) return fit;
    if (queue) {
        const cudaError_t e = cudaMemsetAsync(queue, 0, sizeof(unsigned int), stream);
        if (e != cudaSuccess) return (int)e;
    }
    const int64_t need = (V + voxels_per_cta - 1) / voxels_per_cta;
    const int64_t cap = (int64_t)sms * occ;
    kern<<<(int)(need < cap ? need : cap), threads, smem, stream>>>(args...);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

// voxels one full wave of the persistent grid holds (SMs x resident CTAs x voxels per CTA); 0 on
// any failure, with the error cleared
template <typename Kern>
int wave_voxels(Kern kern, int threads, size_t smem, int voxels_per_cta) {
    int dev = 0, sms = 0, occ = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return sms * occ * voxels_per_cta;
}

}  // namespace pb
