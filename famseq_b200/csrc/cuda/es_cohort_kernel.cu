// es_cohort_kernel.cu -- Elston-Stewart for a cohort ped file whose families may have any loop-free shape: three
// generations, half-sibs, several spouses, sibships of six or more, next to the nuclear families and lone individuals of
// es_families_kernel.cu.
//
// The reference peels the whole file as one family; each member's marginal depends only on its own family, and the LRC
// gate and the failure rule stay whole-row (es_families_kernel.cu).  A call is three launches, whatever the number of
// families:
//   1. es_cohort_head_kernel: what es_families_kernel does -- the column pass (individual-only posteriors, the gate, the
//      failure flag), the nuclear families and lone individuals when the gate asks for the pedigree, post := single when it
//      does not -- but it records status = failed | needed << 1 instead of writing the NA rows and the final status;
//   2. es_cohort_kernel<TB>: one block per (tile of TB variants, program family).  The family's likelihood rows are
//      gathered from the row through its column map (PL input is decoded through the table on the way) into the vector
//      file in shared memory, and es_interpret runs the family's message program, one variant per thread in lock step.
//      FIN writes post / gt at the global column.  A zero row sum fails the variant: status := 3 (a plain store of a
//      constant, so the blocks of the other families that share the variant cannot lose it);
//   3. es_cohort_finish_kernel: NA rows over every column of a failed variant, and status := failed.
// Compiled with -fmad=false like es_kernel.cu: the programs return the interpreter's doubles.
#include <algorithm>

#include "es_families_body.cuh"
#include "es_interpret.cuh"

namespace famseq {

namespace {

template <int NCMAX, bool PL, bool SINGLE>
__global__ void __launch_bounds__(ES_FAMILIES_BLOCK) es_cohort_head_kernel(const __grid_constant__ FamiliesParams P, const BatchPtrs B) {
    es_families_row<NCMAX, PL, SINGLE, true>(P, B);
}

// One family's program: its words and its local -> global column map, both in global memory.
struct CohortProgram {
    const uint32_t *words;
    const int32_t *cols;
    __device__ __forceinline__ uint32_t word(int pc) const { return __ldg(words + pc); }
    __device__ __forceinline__ int col(int c) const { return __ldg(cols + c); }
};

template <int TB, bool PL>
__global__ void __launch_bounds__(TB) es_cohort_kernel(const __grid_constant__ CohortParams P, const BatchPtrs B) {
    extern __shared__ __align__(16) unsigned char cohort_smem[];
    const RunConstants &C = P.fam.C;
    const int S = C.s;
    const int64_t S3 = 3 * (int64_t)S;
    double *s_vec = reinterpret_cast<double *>(cohort_smem); // [(max_vectors + 3) * 3][TB + 1] vector file

    const int tid = threadIdx.x;
    const int64_t v0 = (int64_t)blockIdx.x * TB;
    const int nv = (int)min((int64_t)TB, B.V - v0);
    const int64_t v = v0 + tid;
    // status 2: the gate asks for the pedigree and nothing has failed (yet)
    const bool mine = tid < nv && B.status[v] == 2;
    if (!__syncthreads_or(mine)) return;
    const unsigned flag = (mine && B.flags) ? B.flags[v] : 0u;
    for (int pf = blockIdx.y; pf < P.n_pf; pf += gridDim.y) {
        const int q = __ldg(P.pf_prog + pf);
        const int n_cols = __ldg(P.prog_cols + q), K = 3 * n_cols;
        const CohortProgram prog{P.words + __ldg(P.prog_off + q), P.cols + __ldg(P.pf_col_off + pf)};
        // the family's likelihood rows of the block's variants, gathered into rows [0, 3 n_cols) of the vector file
        for (int e = tid; e < nv * K; e += TB) {
            const int tt = e / K, k = e - tt * K;
            const int c = k / 3;
            const int64_t at = (v0 + tt) * S3 + (int64_t)prog.col(c) * 3 + (k - 3 * c);
            s_vec[k * (TB + 1) + tt] = PL ? __ldg(B.lut + B.pl[at]) : __ldg(B.lk + at);
        }
        __syncthreads();
        if (mine) {
            EsThread<TB> t;
            t.vec = s_vec + tid;
            t.pr = select_priors(C, flag);
            // the three special vectors behind the scratch: prior (non-male), prior (male), ones
            const uint32_t special = (uint32_t)(n_cols + __ldg(P.prog_slots + q));
            const double one[3] = {1.0, 1.0, 1.0};
            t.store(special, t.pr.a);
            t.store(special + 1, t.pr.m);
            t.store(special + 2, one);
            double *post_row = B.post + v * S3;
            uint8_t *gt_row = B.gt + v * S;
            const bool failed = ((flag >> 1) & 1u) ? es_interpret<true, TB>(C, prog, t, post_row, gt_row)
                                                   : es_interpret<false, TB>(C, prog, t, post_row, gt_row);
            if (failed) B.status[v] = 3;
        }
        __syncthreads(); // the next family's gather overwrites the vector file
    }
}

// NA rows of every failed variant, then status := failed.  One thread per (variant, column); the thread of column 0 clears
// bit 1 of the status, which leaves bit 0 -- all the other threads of the variant read -- as it is.
template <bool SINGLE> __global__ void __launch_bounds__(256) es_cohort_finish_kernel(const BatchPtrs B, int S) {
    const int64_t n = B.V * (int64_t)S, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int64_t v = i / S;
        const int c = (int)(i - v * S);
        const uint8_t st = B.status[v];
        if (st & 1u) {
            double *p = B.post + i * 3;
            p[0] = p[1] = p[2] = 0.0;
            if (SINGLE) {
                double *s = B.single + i * 3;
                s[0] = s[1] = s[2] = 0.0;
            }
            B.gt[i] = 255;
        }
        if (c == 0) B.status[v] = st & 1u;
    }
}

template <int NCMAX, bool PL, bool SINGLE> void launch_head(const FamiliesParams &P, const BatchPtrs &B, cudaStream_t stream) {
    const int64_t per_block = ES_FAMILIES_BLOCK / P.group;
    const unsigned grid = (unsigned)((B.V + per_block - 1) / per_block);
    es_cohort_head_kernel<NCMAX, PL, SINGLE><<<grid, ES_FAMILIES_BLOCK, 0, stream>>>(P, B);
}

template <int NCMAX> void launch_head_nc(const FamiliesParams &P, const BatchPtrs &B, cudaStream_t stream) {
    if (B.pl) return B.single ? launch_head<NCMAX, true, true>(P, B, stream) : launch_head<NCMAX, true, false>(P, B, stream);
    return B.single ? launch_head<NCMAX, false, true>(P, B, stream) : launch_head<NCMAX, false, false>(P, B, stream);
}

template <int TB, bool PL> cudaError_t launch_programs(const CohortParams &P, const BatchPtrs &B, cudaStream_t stream) {
    const size_t smem = es_cohort_smem_bytes(P.max_vectors, TB);
    const cudaError_t rc = cudaFuncSetAttribute(es_cohort_kernel<TB, PL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc != cudaSuccess) return rc;
    const dim3 grid((unsigned)((B.V + TB - 1) / TB), (unsigned)std::min(P.n_pf, 65535));
    es_cohort_kernel<TB, PL><<<grid, TB, smem, stream>>>(P, B);
    return cudaSuccess;
}

template <int TB> cudaError_t launch_programs_tb(const CohortParams &P, const BatchPtrs &B, cudaStream_t stream) {
    return B.pl ? launch_programs<TB, true>(P, B, stream) : launch_programs<TB, false>(P, B, stream);
}

} // namespace

size_t es_cohort_smem_bytes(int max_vectors, int tb) {
    const size_t bytes = (size_t)(max_vectors + 3) * 3 * (tb + 1) * sizeof(double); // the vector file
    return (bytes + 15) & ~(size_t)15;
}

cudaError_t launch_es_cohort_head(const FamiliesParams &P, const BatchPtrs &B, cudaStream_t stream) {
    switch (P.nc_max) {
    case 0: launch_head_nc<0>(P, B, stream); break;
    case 1: launch_head_nc<1>(P, B, stream); break;
    case 2: launch_head_nc<2>(P, B, stream); break;
    case 3: launch_head_nc<3>(P, B, stream); break;
    case 4: launch_head_nc<4>(P, B, stream); break;
    case 5: launch_head_nc<5>(P, B, stream); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t launch_es_cohort_finish(const BatchPtrs &B, int S, cudaStream_t stream) {
    const int64_t n = B.V * (int64_t)S;
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, 148 * 16));
    if (B.single)
        es_cohort_finish_kernel<true><<<grid, 256, 0, stream>>>(B, S);
    else
        es_cohort_finish_kernel<false><<<grid, 256, 0, stream>>>(B, S);
    return cudaGetLastError();
}

cudaError_t launch_es_cohort(const CohortParams &P, const BatchPtrs &B, cudaStream_t stream) {
    if (B.V <= 0) return cudaSuccess;
    cudaError_t rc = launch_es_cohort_head(P.fam, B, stream);
    if (rc != cudaSuccess) return rc;
    switch (P.tb) {
    case 128: rc = launch_programs_tb<128>(P, B, stream); break;
    case 64: rc = launch_programs_tb<64>(P, B, stream); break;
    case 32: rc = launch_programs_tb<32>(P, B, stream); break;
    default: return cudaErrorInvalidValue;
    }
    if (rc == cudaSuccess) rc = cudaGetLastError();
    if (rc != cudaSuccess) return rc;
    return launch_es_cohort_finish(B, P.fam.C.s, stream);
}

} // namespace famseq
