// es_kernel.cu -- Elston-Stewart peeling, one variant per thread, for sm_100a.
//
// Replaces family::calPostProbPeeling + calAntProb[X] + calPosProb[X] (src/family.cpp:1126-1403,
// :1501-1930).  The reference walks a memoised recursion per variant with heap-allocated matrices;
// here the recursion is compiled once on the host into a message program (host/es_program.cpp) that
// every thread interprets in lock step for its own variant, so there is no divergence and no
// per-variant allocation.
//
// This is the path of multi-generation pedigrees (nuclear families take es_nuclear_kernel.cu): the work per
// variant (one 27-term contraction per message) dominates its 73*S+2 bytes, so
//   * every operand of the program -- likelihood rows, message scratch (liveness-compacted by the host compiler),
//     the founder priors, the vector of ones -- lives in one per-variant "vector file" in shared memory and is
//     addressed by a plain index, so the interpreter fetches an operand with three loads and no case distinction;
//   * the block's likelihood tile ([TB][S][3], contiguous in HBM) is copied once, coalesced, into that file in
//     transposed form (row stride TB+1: conflict-free for the copy and for the per-thread accesses);
//   * post / single / gt rows are written directly (write-only, never read back); the block size is the one that
//     keeps the most variants resident per SM.
// Arithmetic: this file is compiled with -fmad=false and every product is formed in the reference's
// association order, so the FP64 results are bit-identical to the reference CPU build.
#include <algorithm>

#include "common.cuh"
#include "es_interpret.cuh"
#include "kernels.hpp"

namespace famseq {

namespace {

// The program of fs_create's pedigree: words in the kernel parameters, input column = output column.
struct EsParamProgram {
    const EsParams &P;
    __device__ __forceinline__ uint32_t word(int pc) const { return P.prog.words[pc]; }
    __device__ __forceinline__ int col(int c) const { return c; }
};

template <int TB> __global__ void __launch_bounds__(TB) es_kernel(const __grid_constant__ EsParams P, const BatchPtrs B) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const RunConstants &C = P.C;
    const int S = C.s, S3 = 3 * S;
    double *s_vec = reinterpret_cast<double *>(smem_raw); // [(S + n_slots + 3) * 3][TB + 1] vector file

    const int tid = threadIdx.x;
    const int64_t v0 = (int64_t)blockIdx.x * TB;
    const int nv = (int)min((int64_t)TB, B.V - v0);
    {   // coalesced copy of the block's contiguous [nv][S][3] likelihood tile into rows [0, 3S) of the vector file
        const double *gin = B.lk + v0 * S3;
        for (int e = tid; e < nv * S3; e += TB) {
            const int tt = e / S3, k = e - tt * S3;
            s_vec[k * (TB + 1) + tt] = __ldcs(gin + e);
        }
    }
    __syncthreads();
    const int64_t v = v0 + tid;
    if (tid >= nv) return;
    const unsigned flag = B.flags ? B.flags[v] : 0u;
    EsThread<TB> t;
    t.vec = s_vec + tid;
    t.pr = select_priors(C, flag);
    {   // the three special vectors behind the scratch: prior (non-male), prior (male), ones
        const uint32_t special = (uint32_t)(S + P.prog.n_slots);
        const double one[3] = {1.0, 1.0, 1.0};
        t.store(special, t.pr.a);
        t.store(special + 1, t.pr.m);
        t.store(special + 2, one);
    }
    double *post_row = B.post + v * S3;
    double *single_row = B.single + v * S3;
    uint8_t *gt_row = B.gt + v * S;

    // individual-only posterior (family.cpp:1405-1499) and LRC gate (family.cpp:1140-1162)
    bool failed = C.unseq_fail[flag & 3u] != 0;
    bool pedigree_needed = false;
    for (int c = 0; c < S; c++) {
        const double l0 = t.vec[(c * 3) * (TB + 1)], l1 = t.vec[(c * 3 + 1) * (TB + 1)], l2 = t.vec[(c * 3 + 2) * (TB + 1)];
        const bool male = C.col_male[c] != 0;
        const double r0 = l0 * (male ? t.pr.m[0] : t.pr.a[0]);
        const double r1 = l1 * (male ? t.pr.m[1] : t.pr.a[1]);
        const double r2 = l2 * (male ? t.pr.m[2] : t.pr.a[2]);
        const double rs = (r0 + r1) + r2;
        if (rs <= 0.0) failed = true;
        double q0, q1, q2;
        div3(r0, r1, r2, rs, q0, q1, q2);
        single_row[c * 3] = q0;
        single_row[c * 3 + 1] = q1;
        single_row[c * 3 + 2] = q2;
        gt_row[c] = call_genotype(q0, q1, q2); // stands when the gate keeps the pedigree out; FIN overwrites it otherwise
        double big = 0.0;
        if (big < l0) big = l0;
        if (big < l1) big = l1;
        if (big < l2) big = l2;
        const double ls = (l0 + l1) + l2;
        if (lrc_wants_pedigree(C.lrc, l0, l1, l2, big, ls)) pedigree_needed = true;
    }
    if (!failed) {
        if (!pedigree_needed) { // family.cpp:1164-1253: FPP := individual-only posterior
            for (int k = 0; k < S3; k++) post_row[k] = single_row[k];
        } else if ((flag >> 1) & 1u) {
            failed = es_interpret<true, TB>(C, EsParamProgram{P}, t, post_row, gt_row);
        } else {
            failed = es_interpret<false, TB>(C, EsParamProgram{P}, t, post_row, gt_row);
        }
    }
    if (failed) {
        for (int k = 0; k < S3; k++) {
            post_row[k] = 0.0;
            single_row[k] = 0.0;
        }
        for (int c = 0; c < S; c++) gt_row[c] = 255;
    }
    B.status[v] = failed ? 1 : 0;
}

} // namespace

size_t es_smem_bytes(const EsParams &P, int tb) {
    const size_t bytes = (size_t)(P.C.s + P.prog.n_slots + 3) * 3 * (tb + 1) * sizeof(double); // the vector file
    return (bytes + 15) & ~(size_t)15;
}

// Picks the largest block the scratch fits in (more threads per SM hide FP64 and LDS latency).
int es_pick_block(const EsParams &P, size_t smem_limit) {
    // the block size that keeps the most variants resident per SM (registers allow 512 threads)
    const int candidates[] = {128, 64, 32};
    int best = 0, best_threads = 0;
    for (int tb : candidates) {
        const size_t need = es_smem_bytes(P, tb) + 1024;
        if (need > smem_limit + 1024) continue;
        const int threads = (int)std::min<size_t>(512, (smem_limit + 1024) / need * tb);
        if (threads > best_threads) {
            best_threads = threads;
            best = tb;
        }
    }
    return best;
}

cudaError_t launch_es(const EsParams &P, const BatchPtrs &B, int tb, cudaStream_t stream) {
    if (B.V <= 0) return cudaSuccess;
    const size_t smem = es_smem_bytes(P, tb);
    const unsigned grid = (unsigned)((B.V + tb - 1) / tb);
    cudaError_t rc;
    switch (tb) {
    case 128:
        rc = cudaFuncSetAttribute(es_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (rc != cudaSuccess) return rc;
        es_kernel<128><<<grid, 128, smem, stream>>>(P, B);
        break;
    case 64:
        rc = cudaFuncSetAttribute(es_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (rc != cudaSuccess) return rc;
        es_kernel<64><<<grid, 64, smem, stream>>>(P, B);
        break;
    case 32:
        rc = cudaFuncSetAttribute(es_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (rc != cudaSuccess) return rc;
        es_kernel<32><<<grid, 32, smem, stream>>>(P, B);
        break;
    default:
        return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

} // namespace famseq
