// bn_kernel.cu -- Bayesian-network method: exhaustive enumeration of all 3^N joint genotype
// configurations, for sm_100a.  Replaces family::calPostProbBN (src/family.cpp:750-1124) and the
// reference's own GPU kernels calPostProb / calPostProbX (src/family.cu:769-800, :929-971).
//
// Every configuration's joint probability  1e7 * prod_j f_j(g_j | g_mother, g_father)  is formed and
// added to the marginal bins of all N members, as in the reference.  What differs is the bookkeeping:
//   * the per-variant factors f_j = (prior | transmission) * likelihood are tabulated ONCE per variant
//     in shared memory (the reference re-derives all N of them for every configuration);
//   * members are enumerated parents-before-children (host/bn_plan.cpp), so the joint is carried as a
//     prefix product down the loop nest and only the factors of the digits that changed are touched;
//   * a group of 3^h threads splits the outermost h digits, every thread runs an odometer over the
//     middle digits and a fully unrolled block over the innermost u digits, with the marginal bins of
//     the unrolled digits in registers;
//   * no per-configuration division/modulo, no local-memory arrays, no global traffic in the loop.
// Threads of one variant walk the inner digits in lock step, so their shared-memory table reads are
// broadcasts.  The group's partial bins are summed in a fixed order (deterministic results).
// Summation order differs from the reference's single odometer; all terms are non-negative, so the
// marginals agree to ~1e-13 relative (tests/test_parity_gpu.py asserts 1e-9).
#include "bn_body.cuh"

namespace famseq {

namespace {

template <int U, bool INDEP, bool FACTOR = false>
__global__ void __launch_bounds__(256, 2) bn_kernel(const __grid_constant__ BnParams P, const BatchPtrs B, int n_tiles) {
    bn_body<U, INDEP, FACTOR, false>(P, B, n_tiles);
}

} // namespace

size_t bn_smem_bytes(const BnParams &P) {
    const BnPlan &pl = P.plan;
    size_t d = (size_t)pl.vpb * pl.table_doubles + (size_t)pl.vpb * pl.n_levels * 3 + (size_t)pl.r * 5 * pl.threads +
               (size_t)(3 * pl.u + 1) * pl.threads + (size_t)pl.vpb * P.C.s * 3;
    return ((d * sizeof(double) + (size_t)pl.vpb * sizeof(int)) + 15) & ~(size_t)15;
}

template <int U, bool INDEP, bool FACTOR = false>
static cudaError_t launch_bn_u(const BnParams &P, const BatchPtrs &B, int sm_count, cudaStream_t stream) {
    const size_t smem = bn_smem_bytes(P);
    cudaError_t rc = cudaFuncSetAttribute(bn_kernel<U, INDEP, FACTOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc != cudaSuccess) return rc;
    int per_sm = 0;
    rc = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bn_kernel<U, INDEP, FACTOR>, P.plan.threads, smem);
    if (rc != cudaSuccess) return rc;
    if (per_sm < 1) return cudaErrorInvalidConfiguration;
    const int64_t n_tiles = (B.V + P.plan.vpb - 1) / P.plan.vpb;
    if (n_tiles > 0x7fffffff) return cudaErrorInvalidValue;
    const int grid = (int)std::min<int64_t>(n_tiles, (int64_t)sm_count * per_sm);
    bn_kernel<U, INDEP, FACTOR><<<grid, P.plan.threads, smem, stream>>>(P, B, (int)n_tiles);
    return cudaGetLastError();
}

cudaError_t launch_bn(const BnParams &P, const BatchPtrs &B, int sm_count, cudaStream_t stream) {
    if (B.V <= 0) return cudaSuccess;
    const bool indep = P.plan.independent != 0;
    if (indep && P.plan.factor_leaves) {
        switch (P.plan.u) {
        case 2: return launch_bn_u<2, true, true>(P, B, sm_count, stream);
        case 3: return launch_bn_u<3, true, true>(P, B, sm_count, stream);
        case 4: return launch_bn_u<4, true, true>(P, B, sm_count, stream);
        case 5: return launch_bn_u<5, true, true>(P, B, sm_count, stream);
        default: break;
        }
    }
    switch (P.plan.u) {
    case 1: return launch_bn_u<1, false>(P, B, sm_count, stream);
    case 2: return indep ? launch_bn_u<2, true>(P, B, sm_count, stream) : launch_bn_u<2, false>(P, B, sm_count, stream);
    case 3: return indep ? launch_bn_u<3, true>(P, B, sm_count, stream) : launch_bn_u<3, false>(P, B, sm_count, stream);
    case 4: return indep ? launch_bn_u<4, true>(P, B, sm_count, stream) : launch_bn_u<4, false>(P, B, sm_count, stream);
    case 5: return indep ? launch_bn_u<5, true>(P, B, sm_count, stream) : launch_bn_u<5, false>(P, B, sm_count, stream);
    default: return cudaErrorInvalidValue;
    }
}

} // namespace famseq
