// bn_cohort_kernel.cu -- the Bayesian-network method for a cohort ped file: every family, looped ones included, enumerated
// on its own with the plan fs_create would build for the family's rows alone.
//
// The reference enumerates the whole file as one pedigree: its joint is 1e7 * the product of every member's factor, and a
// factor depends only on members of the same family, so the joint factorises by family and each member's normalised
// marginal is that of its own family's joint.  The per-family run returns the reference's answer up to rounding; it
// differs only where the whole-file product leaves the double range and no family's product does.  The LRC gate and the
// failure rule stay whole-row.  A call is 2 + (launch classes) launches, whatever the number of families or plans:
//   1. es_cohort_head_kernel with no nuclear families: individual-only posteriors, FPP := GPP where the gate keeps the
//      pedigree out, status := failed | needed << 1;
//   2. bn_cohort_kernel<U, INDEP, FACTOR>, once per launch class: one block per (tile of 256 / group variants, family of
//      the class) running bn_kernel's body (bn_body.cuh) on the variants with status 2;
//   3. es_cohort_finish_kernel: NA rows over every column of a failed variant, and status := failed.
#include <algorithm>

#include "bn_body.cuh"

namespace famseq {

namespace {

constexpr int BN_COHORT_BLOCK = 256; // the plan's block size: vpb * group rounds up to 256 for every group 3^h, h = 0..5

template <int U, bool INDEP, bool FACTOR>
__global__ void __launch_bounds__(BN_COHORT_BLOCK, 2) bn_cohort_kernel(const __grid_constant__ BnCohortLaunch P, const BatchPtrs B, int n_tiles) {
    bn_body<U, INDEP, FACTOR, true>(P, B, n_tiles);
}

template <int U, bool INDEP, bool FACTOR = false>
cudaError_t launch_class(const BnCohortLaunch &L, const BnCohortClass &k, const BatchPtrs &B, cudaStream_t stream) {
    cudaError_t rc = cudaFuncSetAttribute(bn_cohort_kernel<U, INDEP, FACTOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem);
    if (rc != cudaSuccess) return rc;
    const int64_t n_tiles = (B.V + BN_COHORT_BLOCK / k.group - 1) / (BN_COHORT_BLOCK / k.group);
    if (n_tiles > 0x7fffffff) return cudaErrorInvalidValue;
    const unsigned fy = (unsigned)std::min(L.n_fam, 65535), fz = (unsigned)((L.n_fam + 65534) / 65535);
    bn_cohort_kernel<U, INDEP, FACTOR><<<dim3((unsigned)n_tiles, fy, fz), BN_COHORT_BLOCK, k.smem, stream>>>(L, B, (int)n_tiles);
    return cudaGetLastError();
}

cudaError_t launch_class_u(const BnCohortLaunch &L, const BnCohortClass &k, const BatchPtrs &B, cudaStream_t stream) {
    const bool indep = k.independent != 0;
    if (indep && k.factor_leaves) {
        switch (k.u) {
        case 2: return launch_class<2, true, true>(L, k, B, stream);
        case 3: return launch_class<3, true, true>(L, k, B, stream);
        case 4: return launch_class<4, true, true>(L, k, B, stream);
        case 5: return launch_class<5, true, true>(L, k, B, stream);
        default: break;
        }
    }
    switch (k.u) {
    case 1: return launch_class<1, false>(L, k, B, stream);
    case 2: return indep ? launch_class<2, true>(L, k, B, stream) : launch_class<2, false>(L, k, B, stream);
    case 3: return indep ? launch_class<3, true>(L, k, B, stream) : launch_class<3, false>(L, k, B, stream);
    case 4: return indep ? launch_class<4, true>(L, k, B, stream) : launch_class<4, false>(L, k, B, stream);
    case 5: return indep ? launch_class<5, true>(L, k, B, stream) : launch_class<5, false>(L, k, B, stream);
    default: return cudaErrorInvalidValue;
    }
}

} // namespace

size_t bn_cohort_smem_bytes(const BnPlan &pl) { // bn_smem_bytes without the per-column state (C.s = 0)
    const size_t d = (size_t)pl.vpb * pl.table_doubles + (size_t)pl.vpb * pl.n_levels * 3 + (size_t)pl.r * 5 * BN_COHORT_BLOCK +
                     (size_t)(3 * pl.u + 1) * BN_COHORT_BLOCK;
    return ((d * sizeof(double) + (size_t)pl.vpb * sizeof(int)) + 15) & ~(size_t)15;
}

cudaError_t launch_bn_cohort(const BnCohortParams &P, const BatchPtrs &B, cudaStream_t stream) {
    if (B.V <= 0) return cudaSuccess;
    cudaError_t rc = launch_es_cohort_head(P.head, B, stream);
    if (rc != cudaSuccess) return rc;
    BnCohortLaunch L;
    L.C = P.head.C;
    L.C.s = 0;
    L.s_row = P.head.C.s;
    L.plans = P.plans;
    L.fam_plan = P.fam_plan;
    L.fam_col_off = P.fam_col_off;
    L.cols = P.cols;
    for (const BnCohortClass &k : P.classes) {
        L.begin = k.begin;
        L.n_fam = k.end - k.begin;
        rc = launch_class_u(L, k, B, stream);
        if (rc != cudaSuccess) return rc;
    }
    return launch_es_cohort_finish(B, P.head.C.s, stream);
}

} // namespace famseq
