// Dispatch over the register-tiled variants listed in the generated pb_fast_table.inc.
#include <cstdlib>

#include "pb_fast_registry.h"

namespace pb {

// variants_f32[], variants_f64[]: CTA rows, then group rows, then warp rows
#include "pb_fast_table.inc"

static const auto &variants(float) { return variants_f32; }
static const auto &variants(double) { return variants_f64; }

template <typename real>
static long cost(const Variant<real> &v) {
    // warp tier: unrolled work per iteration ~ R * KMAX (the CIRC variants skip the halo / tail selects,
    // hence the small bonus)
    if (v.tier == TIER_WARP) return (long)v.R * v.KMAX * (v.circ ? 19 : 20);
    // tier 0: slots per voxel (lanes x samples per lane) x unrolled taps, ties broken by the tail-select count
    long c = (long)v.R * v.KMAX * v.lanes * 64 + v.TAIL;
    // one warp per voxel with 64 taps runs four warps per SM (shared-memory scratch), two warps per
    // voxel run eight: prefer the latter up to 1.3 x the slots (measured: T = 405..512 2.5 x faster on two
    // warps of R = 8 than on one of R = 16; T = 300 5 % slower than on one warp of R = 12)
    if (v.KMAX == 64 && v.lanes == 32) c += c * 3 / 10;
    return c;
}

// the family of a row: warp tier, or tier 0 with fewer lanes than a warp (group) or a whole number of warps (CTA)
template <typename real>
static int family(const Variant<real> &v) {
    return v.tier == TIER_WARP ? FAMILY_WARP : (v.lanes < 32 ? FAMILY_GROUP : FAMILY_CTA);
}

constexpr unsigned bit(int family) { return 1u << family; }
constexpr unsigned TIER0 = bit(FAMILY_GROUP) | bit(FAMILY_CTA);

// cheapest variant of the families in the mask `families` that serves (T, K) and has the entry point `need`;
// ties go to the first row (strict <), so CTA rows win ties against group rows
template <typename real, typename Fn>
static const Variant<real> *pick(unsigned families, int T, int K, Fn Variant<real>::*need) {
    const Variant<real> *best = nullptr;
    long best_cost = 0;
    for (const Variant<real> *v : variants(real())) {
        if (!(families & bit(family(*v))) || !(v->*need) || !v->ok(T, K)) continue;
        const long c = cost(*v);
        if (!best || c < best_cost) {
            best = v;
            best_cost = c;
        }
    }
    return best;
}

// PB_DISABLE_GROUP=1: developer switch for A/B timing of tier 0 against the warp-per-voxel kernels
static bool tier0_disabled() {
    static const bool disabled = getenv("PB_DISABLE_GROUP") != nullptr;
    return disabled;
}

template <typename real>
static int encode(const Variant<real> &v) { return v.lanes * 1000000 + v.R * 1000 + v.KMAX; }

// The warp tier runs only when the one tier-0 candidate returns FAST_NO_MATCH (its shared memory
// does not fit); no second tier-0 candidate is tried.  Every tier-0 row (group and CTA) has both bd entry points, so
// with and without early stopping a call runs on the same row.  V == 0 launches nothing and reports the same choice.
template <typename real>
static int bd_dispatch(const BdArgs<real> &a, cudaStream_t s, int *id, int *fam_out) {
    const auto need = a.early_stopping ? &Variant<real>::bd_es : &Variant<real>::bd;
    auto ran = [&](const Variant<real> &v, int rc) {
        if (id) *id = encode(v);
        if (fam_out) *fam_out = family(v);
        return rc;
    };
    if (!tier0_disabled())
        if (const Variant<real> *v = pick<real>(TIER0, a.T, a.K, need)) {
            const int rc = (v->*need)(a, s);
            if (rc != FAST_NO_MATCH) return ran(*v, rc);
        }
    if (const Variant<real> *v = pick<real>(bit(FAMILY_WARP), a.T, a.K, &Variant<real>::bd)) {
        const int rc = v->bd(a, s);
        if (rc != FAST_NO_MATCH) return ran(*v, rc);
    }
    if (id) *id = 0;
    if (fam_out) *fam_out = FAMILY_GENERIC;
    return FAST_NO_MATCH;
}

// Routing of every deconv call (fixed lambda, early stopping, lbda=None, path, masked): group rows, then warp rows,
// then CTA rows, then (launch_deconv) the generic kernel.  A step is taken when the one before has no variant for
// (T, K) or its launch returns FAST_NO_MATCH (shared memory or occupancy).  The group rows run early stopping only
// with a work-queue counter (a.queue).  V == 0 launches nothing and reports the same choice.
template <typename real>
static int deconv_dispatch(const DeconvArgs<real> &a, cudaStream_t s, int *id, int *fam_out) {
    // deconv(lbda=None) (nb_outer > 0) takes the same rows through their deconv_auto entry points
    const auto need = a.nb_outer > 0 ? &Variant<real>::deconv_auto : &Variant<real>::deconv;
    const bool group_ok = (!(a.early_stopping && a.wind >= 2) || a.queue) && !tier0_disabled();
    for (const int fam : {FAMILY_GROUP, FAMILY_WARP, FAMILY_CTA}) {
        if (fam == FAMILY_GROUP && !group_ok) continue;
        if (const Variant<real> *v = pick<real>(bit(fam), a.T, a.K, need)) {
            const int rc = (v->*need)(a, s);
            if (rc != FAST_NO_MATCH) {
                if (id) *id = encode(*v);
                if (fam_out) *fam_out = fam;
                return rc;
            }
        }
    }
    if (id) *id = 0;
    if (fam_out) *fam_out = FAMILY_GENERIC;
    return FAST_NO_MATCH;
}

// Routing of a censored deconv call: the cheapest CTA row whose ok_censored takes (T, K), then (launch_deconv) the
// generic kernel.  The group and warp kernels have no censored mode.
template <typename real>
static int deconv_censored_dispatch(const DeconvArgs<real> &a, const Censor &cz, cudaStream_t s, int *id, int *fam_out) {
    const auto need = a.nb_outer > 0 ? &Variant<real>::deconv_auto_censored : &Variant<real>::deconv_censored;
    const Variant<real> *best = nullptr;
    long best_cost = 0;
    for (const Variant<real> *v : variants(real())) {
        if (!(v->*need) || !v->ok_censored(a.T, a.K)) continue;
        const long c = cost(*v);
        if (!best || c < best_cost) {
            best = v;
            best_cost = c;
        }
    }
    if (best) {
        const int rc = (best->*need)(a, cz, s);
        if (rc != FAST_NO_MATCH) {
            if (id) *id = encode(*best);
            if (fam_out) *fam_out = family(*best);
            return rc;
        }
    }
    if (id) *id = 0;
    if (fam_out) *fam_out = FAMILY_GENERIC;
    return FAST_NO_MATCH;
}

// the queries describe bd without early stopping and ignore PB_DISABLE_GROUP
template <typename real>
static int variant_id(int T, int K) {
    const Variant<real> *v = pick<real>(TIER0, T, K, &Variant<real>::bd);
    if (!v) v = pick<real>(bit(FAMILY_WARP), T, K, &Variant<real>::bd);
    return v ? encode(*v) : 0;
}

template <typename real>
static int bd_wave_voxels(int T, int K, int nb_iter) {
    const Variant<real> *v = pick<real>(TIER0, T, K, &Variant<real>::wave);
    return v ? v->wave(nb_iter) : 0;
}

int fast_deconv_dispatch(const DeconvArgs<float> &a, cudaStream_t s, int *id, int *fam) {
    return deconv_dispatch<float>(a, s, id, fam);
}
int fast_deconv_dispatch(const DeconvArgs<double> &a, cudaStream_t s, int *id, int *fam) {
    return deconv_dispatch<double>(a, s, id, fam);
}
int fast_deconv_censored_dispatch(const DeconvArgs<float> &a, const Censor &cz, cudaStream_t s, int *id, int *fam) {
    return deconv_censored_dispatch<float>(a, cz, s, id, fam);
}
int fast_deconv_censored_dispatch(const DeconvArgs<double> &a, const Censor &cz, cudaStream_t s, int *id, int *fam) {
    return deconv_censored_dispatch<double>(a, cz, s, id, fam);
}
int fast_bd_dispatch(const BdArgs<float> &a, cudaStream_t s, int *id, int *fam) {
    return bd_dispatch<float>(a, s, id, fam);
}
int fast_bd_dispatch(const BdArgs<double> &a, cudaStream_t s, int *id, int *fam) {
    return bd_dispatch<double>(a, s, id, fam);
}

int fast_bd_wave_voxels(int T, int K, bool is_f64, int nb_iter) {
    return is_f64 ? bd_wave_voxels<double>(T, K, nb_iter) : bd_wave_voxels<float>(T, K, nb_iter);
}

int fast_variant_id(int T, int K, bool is_f64) {
    return is_f64 ? variant_id<double>(T, K) : variant_id<float>(T, K);
}

}  // namespace pb
