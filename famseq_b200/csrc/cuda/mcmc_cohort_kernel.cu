// mcmc_cohort_kernel.cu -- the Gibbs sampler for a cohort ped file: every family's chain runs on its own, and it is the
// chain of the whole file restricted to that family.
//
// The whole-file sampler (mcmc_kernel.cu) visits the members in ped order, and a member's full conditional reads only the
// current genotypes of its own family.  Its random word depends only on (seed, global site, sweep, ped row).  So a family's
// chain, with its members swept in increasing ped row and each word drawn with the member's global ped row as the Philox
// counter, is bit for bit the family's part of the whole-file chain: the step (mcmc_step.cuh) is the same arithmetic in
// the same order.  The LRC gate and the failure rule stay whole-row.  A call is 2 + (launch classes) launches, whatever the
// number of families or plans:
//   1. es_cohort_head_kernel with no nuclear families: individual-only posteriors, FPP := GPP where the gate keeps the
//      pedigree out, status := failed | needed << 1;
//   2. mcmc_cohort_kernel<GW>, once per launch class (genotype-vector width): one block per (tile of TB variants, family of
//      the class), one chain per thread, on the variants with status 2.  All lanes work on the same family, so member and
//      link descriptors and ped rows are warp-uniform.  The block stages its family's plan and row / column maps in shared
//      memory; own factors and Rao-Blackwell accumulators live there too, [member][g][thread], thread-private.  A member
//      row whose posterior sums to <= 0 fails the variant: status := 3 (a plain store of a constant, so the blocks of the
//      other families that share the variant cannot lose it);
//   3. es_cohort_finish_kernel: NA rows over every column of a failed variant, and status := failed.
// Compiled with mcmc_kernel.cu's flags (FMA contraction on): the step's sums and the accumulation are written with explicit
// roundings where a contraction could otherwise differ between the two kernels.
#include <algorithm>

#include "kernels.hpp"
#include "mcmc_step.cuh"

namespace famseq {

namespace {

constexpr int MCMC_COHORT_MAX_BLOCK = 256;
constexpr size_t MCMC_COHORT_STATIC_SMEM = sizeof(McmcPlan) + 2 * MCMC_MAX_MEMBERS * sizeof(int32_t);

// mcmc_cohort_kernel's parameters: one launch class.  C.s is unused; s_row is the input row's column count.
struct McmcCohortLaunch {
    RunConstants C;
    const McmcPlan *plans;
    const int32_t *fam_plan, *fam_col_off, *fam_row_off, *cols, *rows;
    int32_t begin, n_fam; // the class's families: device order [begin, begin + n_fam)
    int32_t s_row;
    int32_t burn, rep;
    uint64_t seed;
    int64_t v_offset;
};

template <int GW>
__global__ void __launch_bounds__(MCMC_COHORT_MAX_BLOCK) mcmc_cohort_kernel(const __grid_constant__ McmcCohortLaunch P, const BatchPtrs B) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint32_t s_plan_raw[sizeof(McmcPlan) / sizeof(uint32_t)]; // raw words: McmcPlan's member initialisers have no place in shared memory
    __shared__ int32_t s_row[MCMC_MAX_MEMBERS], s_col[MCMC_MAX_MEMBERS];   // global ped row, global input column (-1) of each member
    const int TB = blockDim.x, tid = threadIdx.x, lane = tid & 31;
    const int fam = (int)(blockIdx.y + gridDim.y * blockIdx.z);
    if (fam >= P.n_fam) return;
    const int64_t v = (int64_t)blockIdx.x * TB + tid;
    const bool mine = v < B.V && B.status[v] == 2; // the gate asks for the pedigree and nothing has failed (yet)
    if (!__syncthreads_or(mine)) return;

    const int f = P.begin + fam;
    const uint32_t *src = reinterpret_cast<const uint32_t *>(P.plans + __ldg(P.fam_plan + f));
    for (int k = tid; k < (int)(sizeof(McmcPlan) / sizeof(uint32_t)); k += TB) s_plan_raw[k] = __ldg(src + k);
    double *s_tab = reinterpret_cast<double *>(smem_raw); // [108][16]
    for (int e = tid; e < kEntries * kCopies; e += TB) {
        const int entry = e / kCopies;
        s_tab[e] = entry < 81 ? P.C.tab[entry / 27][entry % 27] : 1.0;
    }
    __syncthreads();
    const McmcPlan &pl = *reinterpret_cast<const McmcPlan *>(s_plan_raw);
    const int N = pl.n;
    {
        const int32_t *rmap = P.rows + __ldg(P.fam_row_off + f), *cmap = P.cols + __ldg(P.fam_col_off + f);
        for (int i = tid; i < N; i += TB) {
            s_row[i] = __ldg(rmap + i);
            s_col[i] = pl.col[i] >= 0 ? __ldg(cmap + pl.col[i]) : -1;
        }
    }
    __syncthreads();
    if (!mine) return;

    const uint32_t tab_addr = (uint32_t)__cvta_generic_to_shared(s_tab) + (uint32_t)(lane & (kCopies - 1)) * 8u;
    double *w = s_tab + kEntries * kCopies + tid; // [N][3][TB] own factors: (1e6*prior)*lk or 1e6*lk
    double *acc = w + (size_t)N * 3 * TB;         // [N][3][TB] Rao-Blackwell accumulators
    const uint32_t w_addr = (uint32_t)__cvta_generic_to_shared(w);
    const unsigned flag = B.flags ? B.flags[v] : 0u;
    const bool chrx = (flag >> 1) & 1u;
    const VariantPriors pr = select_priors(P.C, flag);
    const int64_t row0 = v * 3 * (int64_t)P.s_row;
    for (int i = 0; i < N; i++) {
        const uint32_t d = pl.member[i];
        const int col = s_col[i];
#pragma unroll
        for (int g = 0; g < 3; g++) {
            const int64_t at = row0 + (int64_t)col * 3 + g;
            const double lk = col < 0 ? 1.0 : (B.pl ? __ldg(B.lut + B.pl[at]) : __ldg(B.lk + at));
            w[(i * 3 + g) * TB] = gibbs_own_factor(d, pr, g, lk);
            acc[(i * 3 + g) * TB] = 0.0;
        }
    }
    const uint64_t gv = (uint64_t)(P.v_offset + v);
    const uint32_t gv_lo = (uint32_t)gv, gv_hi = (uint32_t)(gv >> 32);
    const uint32_t k0 = (uint32_t)P.seed, k1 = (uint32_t)(P.seed >> 32);
    // the word of ped row r in sweep s is word r % 4 of Philox(s, r / 4, gv); rows increase within a family, so a block of
    // four words is generated once per sweep for all the family's rows it covers (a warp-uniform branch)
    uint32_t r0 = 0, r1 = 0, r2 = 0, r3 = 0, blk = ~0u;
    auto word = [&](uint32_t sweep, int i) {
        const uint32_t r = (uint32_t)s_row[i];
        if ((r >> 2) != blk) {
            blk = r >> 2;
            philox4x32_10(sweep, blk, gv_lo, gv_hi, k0, k1, r0, r1, r2, r3);
        }
        const uint32_t q = r & 3u;
        return q == 0 ? r0 : (q == 1 ? r1 : (q == 2 ? r2 : r3));
    };
    Genotypes<GW> cur;
#pragma unroll
    for (int k = 0; k < GW; k++) cur.w[k] = 0;
    for (int i = 0; i < N; i++) cur.set(i, (int)(word(0u, i) % 3u)); // family.cpp:2063-2067

    const int total_sweeps = P.burn + P.rep;
    for (int sweep = 1; sweep <= total_sweeps; sweep++) {
        const bool sampling = sweep > P.burn;
        blk = ~0u;
        for (int i = 0; i < N; i++) {
            const uint32_t d = pl.member[i];
            const uint32_t wa = w_addr + (uint32_t)i * (3u * TB * 8u);
            double w0 = lds64(wa), w1 = lds64(wa + TB * 8), w2 = lds64(wa + 2 * TB * 8);
            const double sum = gibbs_weights(d, pl.link, cur, chrx, tab_addr, w0, w1, w2);
            cur.set(i, gibbs_draw(word((uint32_t)sweep, i), sum, w0, w2));
            if (sampling) { // family.cpp:2175-2178, Rao-Blackwellised; the products rounded before the sum, as red.add of mcmc_kernel
                const double inv = gibbs_inv(sum);
                double *a = acc + (i * 3) * TB;
                a[0] = __dadd_rn(a[0], __dmul_rn(w0, inv));
                a[TB] = __dadd_rn(a[TB], __dmul_rn(w1, inv));
                a[2 * TB] = __dadd_rn(a[2 * TB], __dmul_rn(w2, inv));
            }
        }
    }

    // ---- postProb = genoFry / numRep, not renormalised; a row summing to <= 0 fails (family.cpp:2082-2092) ----
    const double nrep = (double)P.rep;
    bool failed = false;
    double *post_row = B.post + row0;
    uint8_t *gt_row = B.gt + v * (int64_t)P.s_row;
    for (int i = 0; i < N; i++) {
        const double *a = acc + (i * 3) * TB;
        const double p0 = a[0] / nrep, p1 = a[TB] / nrep, p2 = a[2 * TB] / nrep;
        if (__dadd_rn(__dadd_rn(p0, p1), p2) <= 0.0) failed = true;
        const int c = s_col[i];
        if (c >= 0) {
            post_row[c * 3] = p0;
            post_row[c * 3 + 1] = p1;
            post_row[c * 3 + 2] = p2;
            gt_row[c] = call_genotype(p0, p1, p2);
        }
    }
    if (failed) B.status[v] = 3;
}

template <int GW> cudaError_t launch_class(const McmcCohortLaunch &L, const McmcCohortClass &k, const BatchPtrs &B, cudaStream_t stream) {
    const size_t smem = mcmc_cohort_smem_bytes(k.n_max, k.tb);
    const cudaError_t rc = cudaFuncSetAttribute(mcmc_cohort_kernel<GW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc != cudaSuccess) return rc;
    const int64_t n_tiles = (B.V + k.tb - 1) / k.tb;
    if (n_tiles > 0x7fffffff) return cudaErrorInvalidValue;
    const unsigned fy = (unsigned)std::min(L.n_fam, 65535), fz = (unsigned)((L.n_fam + 65534) / 65535);
    mcmc_cohort_kernel<GW><<<dim3((unsigned)n_tiles, fy, fz), k.tb, smem, stream>>>(L, B);
    return cudaGetLastError();
}

} // namespace

size_t mcmc_cohort_smem_bytes(int n, int tb) { return (size_t)(kEntries * kCopies + 2 * n * 3 * tb) * sizeof(double); }

int mcmc_cohort_pick_block(int n, size_t smem_limit, size_t smem_per_sm) {
    int best = 0, best_threads = 0;
    for (int tb = MCMC_COHORT_MAX_BLOCK; tb >= 32; tb -= 32) {
        const size_t need = mcmc_cohort_smem_bytes(n, tb) + MCMC_COHORT_STATIC_SMEM + 1024; // 1 KB per-block reservation
        if (need > smem_limit + 1024) continue;
        const int blocks = (int)std::min<size_t>(32, smem_per_sm / need);
        const int threads = std::min(2048, blocks * tb);
        if (threads > best_threads) {
            best_threads = threads;
            best = tb;
        }
    }
    return best;
}

cudaError_t launch_mcmc_cohort(const McmcCohortParams &P, const BatchPtrs &B, int burn, int rep, uint64_t seed, int64_t v_offset,
                               cudaStream_t stream) {
    if (B.V <= 0) return cudaSuccess;
    cudaError_t rc = launch_es_cohort_head(P.head, B, stream);
    if (rc != cudaSuccess) return rc;
    McmcCohortLaunch L;
    L.C = P.head.C;
    L.s_row = P.head.C.s;
    L.plans = P.plans;
    L.fam_plan = P.fam_plan;
    L.fam_col_off = P.fam_col_off;
    L.fam_row_off = P.fam_row_off;
    L.cols = P.cols;
    L.rows = P.rows;
    L.burn = burn;
    L.rep = rep;
    L.seed = seed;
    L.v_offset = v_offset;
    for (const McmcCohortClass &k : P.classes) {
        L.begin = k.begin;
        L.n_fam = k.end - k.begin;
        switch (k.gw) {
        case 1: rc = launch_class<1>(L, k, B, stream); break;
        case 2: rc = launch_class<2>(L, k, B, stream); break;
        case 4: rc = launch_class<4>(L, k, B, stream); break;
        default: return cudaErrorInvalidValue;
        }
        if (rc != cudaSuccess) return rc;
    }
    return launch_es_cohort_finish(B, P.head.C.s, stream);
}

} // namespace famseq
