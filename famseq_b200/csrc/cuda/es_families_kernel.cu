// es_families_kernel.cu -- Elston-Stewart for a ped file of many unrelated families (a cohort): nuclear families (two
// founders, 1..5 childless children) and lone individuals, any number of members.
//
// The reference peels the whole ped file as one family (family.cpp:1126-1403).  Each member's marginal depends only on
// its own family, so the families are peeled independently -- with the nuclear-family kernel's arithmetic (peel<NC, X>,
// es_nuclear_kernel.cuh), which returns the interpreter's doubles -- and two rules stay whole-file, per variant:
//   * the LRC gate (family.cpp:1140-1162): the pedigree is used for every sample as soon as one sequenced sample anywhere
//     in the row asks for it;
//   * failure: every sample is reported NA when any family fails, any sample's individual-only row sum is <= 0, or an
//     unsequenced member's prior row does (unseq_fail).
// A group of threads shares one variant row: it strides over the columns for the individual-only posteriors and the two
// flags, reduces the flags, then strides over the families, one family per thread.  Families are ordered by class, so
// the threads of a warp mostly peel the same shape.  The row is read from HBM once; the family pass re-reads it from
// L1/L2.  Every division is an IEEE division (the complete pass of the nuclear kernel, Divider<false, X>).
#include "es_families_body.cuh"

namespace famseq {

namespace {

// NCMAX: largest sibship of the cohort (the register budget is that of the largest family shape instantiated).
template <int NCMAX, bool PL, bool SINGLE>
__global__ void __launch_bounds__(ES_FAMILIES_BLOCK) es_families_kernel(const __grid_constant__ FamiliesParams P, const BatchPtrs B) {
    es_families_row<NCMAX, PL, SINGLE, false>(P, B);
}

template <int NCMAX, bool PL, bool SINGLE> cudaError_t launch_fam(const FamiliesParams &P, const BatchPtrs &B, cudaStream_t stream) {
    const int64_t per_block = ES_FAMILIES_BLOCK / P.group;
    const unsigned grid = (unsigned)((B.V + per_block - 1) / per_block);
    es_families_kernel<NCMAX, PL, SINGLE><<<grid, ES_FAMILIES_BLOCK, 0, stream>>>(P, B);
    return cudaGetLastError();
}

template <int NCMAX> cudaError_t launch_nc_max(const FamiliesParams &P, const BatchPtrs &B, cudaStream_t stream) {
    if (B.pl) return B.single ? launch_fam<NCMAX, true, true>(P, B, stream) : launch_fam<NCMAX, true, false>(P, B, stream);
    return B.single ? launch_fam<NCMAX, false, true>(P, B, stream) : launch_fam<NCMAX, false, false>(P, B, stream);
}

} // namespace

// A warp or less for narrow rows, several variants per block; the whole block for wide ones.  About three columns per
// thread in the column pass: a family of a cohort has about three members.
int es_families_group(int S) {
    if (S >= 384) return ES_FAMILIES_BLOCK;
    int g = 4;
    while (g < 32 && 3 * g < S) g *= 2;
    return g;
}

cudaError_t launch_es_families(const FamiliesParams &P, const BatchPtrs &B, cudaStream_t stream) {
    if (B.V <= 0) return cudaSuccess;
    switch (P.nc_max) {
    case 0: return launch_nc_max<0>(P, B, stream);
    case 1: return launch_nc_max<1>(P, B, stream);
    case 2: return launch_nc_max<2>(P, B, stream);
    case 3: return launch_nc_max<3>(P, B, stream);
    case 4: return launch_nc_max<4>(P, B, stream);
    case 5: return launch_nc_max<5>(P, B, stream);
    default: return cudaErrorInvalidValue;
    }
}

} // namespace famseq
