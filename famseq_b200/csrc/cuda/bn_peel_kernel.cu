// bn_peel_kernel.cu -- exact BN posteriors by conditioned Elston-Stewart peeling (host/bn_peel.hpp), one variant per thread.
//
// Shaped like es_kernel: the block's likelihood tile is copied into the per-variant vector file in shared memory, the
// individual-only posterior and the LRC gate are es_kernel's, and the pedigree goes through the message-program interpreter
// (es_interpret.cuh).  When the pedigree is needed, the conditioned program runs once per clamp c = 0 .. 3^K - 1 (the same
// for the whole block, so there is no divergence): the K breakers' clamped likelihoods and indicators are written from the
// digits of c, and every member's ES_OP_ACC stores (c = 0) or adds its unnormalised marginal into its accumulator.  Then each
// accumulator is normalised; the variant fails when any member's accumulated row sum is <= 0, the Bayesian network's rule.
// With K = 0 (a loop-free pedigree) there is one peel and every accumulator holds FIN's vector, so the outputs are es_kernel's
// bytes.  Compiled with -fmad=false like the other Elston-Stewart kernels.
#include <algorithm>
#include <memory>

#include "common.cuh"
#include "es_interpret.cuh"
#include "kernels.hpp"

namespace famseq {

namespace {

struct PeelParamProgram {
    const BnPeelParams &P;
    __device__ __forceinline__ uint32_t word(int pc) const { return P.peel.prog.words[pc]; }
    __device__ __forceinline__ int col(int c) const { return c; }
};

template <bool X, int TB> __device__ __forceinline__ void peel_all(const BnPeelParams &P, const EsThread<TB> &t) {
    const RunConstants &C = P.C;
    const int K = P.peel.n_breakers;
    int n_clamps = 1;
    for (int j = 0; j < K; j++) n_clamps *= 3;
    for (int c = 0; c < n_clamps; c++) {
        for (int j = 0, rest = c; j < K; j++, rest /= 3) {
            const int d = rest % 3, col = P.peel.breaker_col[j];
            double e[3], l[3];
#pragma unroll
            for (int g = 0; g < 3; g++) e[g] = g == d ? 1.0 : 0.0;
            if (col >= 0) {
                t.load((uint32_t)col, l);
#pragma unroll
                for (int g = 0; g < 3; g++) l[g] = g == d ? l[g] : 0.0;
            } else {
#pragma unroll
                for (int g = 0; g < 3; g++) l[g] = e[g];
            }
            t.store((uint32_t)(P.peel.clamp_base + j), l);
            t.store((uint32_t)(P.peel.clamp_base + K + j), e);
        }
        es_interpret<X, TB, PeelParamProgram, true>(C, PeelParamProgram{P}, t, nullptr, nullptr, c == 0);
    }
}

template <int TB> __global__ void __launch_bounds__(TB) bn_peel_kernel(const __grid_constant__ BnPeelParams P, const BatchPtrs B) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const RunConstants &C = P.C;
    const int S = C.s, S3 = 3 * S;
    double *s_vec = reinterpret_cast<double *>(smem_raw); // [n_vectors * 3][TB + 1] vector file

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
        const uint32_t special = (uint32_t)(S + P.peel.prog.n_slots);
        const double one[3] = {1.0, 1.0, 1.0};
        t.store(special, t.pr.a);
        t.store(special + 1, t.pr.m);
        t.store(special + 2, one);
    }
    double *post_row = B.post + v * S3;
    double *single_row = B.single + v * S3;
    uint8_t *gt_row = B.gt + v * S;

    // individual-only posterior (family.cpp:1405-1499) and LRC gate (family.cpp:1140-1162), as es_kernel
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
        gt_row[c] = call_genotype(q0, q1, q2);
        double big = 0.0;
        if (big < l0) big = l0;
        if (big < l1) big = l1;
        if (big < l2) big = l2;
        const double ls = (l0 + l1) + l2;
        if (lrc_wants_pedigree(C.lrc, l0, l1, l2, big, ls)) pedigree_needed = true;
    }
    if (!failed) {
        if (!pedigree_needed) {
            for (int k = 0; k < S3; k++) post_row[k] = single_row[k];
        } else {
            if ((flag >> 1) & 1u)
                peel_all<true, TB>(P, t);
            else
                peel_all<false, TB>(P, t);
            // every member's marginal: the failure rule covers all of them, the sequenced ones (k < S) are written
            for (int k = 0; k < P.peel.n_acc; k++) {
                double a[3];
                t.load((uint32_t)(P.peel.acc_base + k), a);
                const double sum = (a[0] + a[1]) + a[2];
                if (sum <= 0.0) failed = true;
                if (k < S) {
                    double q0, q1, q2;
                    div3(a[0], a[1], a[2], sum, q0, q1, q2);
                    post_row[k * 3] = q0;
                    post_row[k * 3 + 1] = q1;
                    post_row[k * 3 + 2] = q2;
                    gt_row[k] = call_genotype(q0, q1, q2);
                }
            }
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

template <int TB> cudaError_t launch_tb(const BnPeelParams &P, const BatchPtrs &B, size_t smem, cudaStream_t stream) {
    const cudaError_t rc = cudaFuncSetAttribute(bn_peel_kernel<TB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc != cudaSuccess) return rc;
    bn_peel_kernel<TB><<<(unsigned)((B.V + TB - 1) / TB), TB, smem, stream>>>(P, B);
    return cudaGetLastError();
}

} // namespace

int bn_peel_pick_block(const BnPeelParams &P, size_t smem_limit) {
    auto proxy = std::make_unique<EsParams>(); // es_pick_block sizes a file of C.s + n_slots + 3 vectors
    proxy->C.s = P.peel.n_vectors - 3;
    proxy->prog.n_slots = 0;
    return es_pick_block(*proxy, smem_limit);
}

cudaError_t launch_bn_peel(const BnPeelParams &P, const BatchPtrs &B, int tb, cudaStream_t stream) {
    if (B.V <= 0) return cudaSuccess;
    const size_t smem = ((size_t)P.peel.n_vectors * 3 * (tb + 1) * sizeof(double) + 15) & ~(size_t)15;
    switch (tb) {
    case 128: return launch_tb<128>(P, B, smem, stream);
    case 64: return launch_tb<64>(P, B, smem, stream);
    case 32: return launch_tb<32>(P, B, smem, stream);
    default: return cudaErrorInvalidValue;
    }
}

} // namespace famseq
