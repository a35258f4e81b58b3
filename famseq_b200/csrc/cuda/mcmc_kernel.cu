// mcmc_kernel.cu -- single-site Gibbs sampler with Rao-Blackwellised marginals, one chain (= one variant)
// per thread, for sm_100a.  Replaces family::calPostProbMCMC + estGenoProb (src/family.cpp:1932-2096,
// :2098-2299).
//
// What follows the reference: the ped-order scan, the full conditionals, the 1e6 pre-scale, the
// `rd < w0` / `rd > 1 - w2` draw rule, accumulation of the normalised weights (not of indicator counts),
// `postProb = sum / numRep` without renormalisation, and the chrX quirk (females get no children factor,
// family.cpp:2230-2257).
// What does not: libc rand() (one global, never seeded stream) is replaced by counter-based Philox4x32-10.
// The random word of member i in sweep s of site v is word i%4 of Philox(counter = (s, i/4, v_lo, v_hi),
// key = seed); s = 0 initialises the genotypes (word % 3), s >= 1 are the sweeps, whose uniform is
// rd = ((word >> 1) + 0.5) * 2^-31 (31 bits like rand() / RAND_MAX; it lets the generated kernel of gibbs_jit.cu decide a
// draw by integer comparisons that are exactly equivalent to rd < w0, rd > 1 - w2).  A value depends on
// (seed, global site, sweep, member) only: any batch split or GPU count gives the same bytes.
//
// A chain is strictly sequential, so the kernel is bound by instruction issue of the few warps whose chain
// state fits on an SM, not by FP64 throughput or HBM (profiles/*mcmc*): the design minimises instructions per
// Gibbs step and on-chip bytes per chain.
//   * all threads of a warp work on the same member: control flow is uniform, pedigree metadata are one
//     uniform constant-bank word per member and per parent-child link (host/mcmc_plan.cpp);
//   * the 3N accumulators live in a global scratch ([block][member][g][thread], thread-private, coalesced) and
//     are updated with fire-and-forget red.global.add.f64 -- three instructions per step, off the dependency
//     chain; the 3N own factors live in shared memory as [member][g][thread] when a full SM's worth of chains
//     fits (small pedigrees), otherwise in the same scratch, fetched one member ahead through L2, so that the
//     number of chains in flight is set by registers (24 warps/SM) and not by shared memory (7 warps/SM for 40
//     members);
//   * the draw is decided on un-normalised weights (rd*sum < w0, rd*sum > sum - w2), so the reciprocal
//     (MUFU seed + two Newton steps) is off the critical path;
//   * the transmission tables are replicated 16 times in shared memory so that the data-dependent look-ups
//     of a half-warp hit 16 different bank pairs;
//   * persistent blocks loop over tiles of TB variants.
#include <algorithm>

#include "kernels.hpp"
#include "mcmc_step.cuh"

namespace famseq {

namespace {

// WGLOBAL = false: own factors in shared memory (small pedigrees: every chain of a full SM fits).
// WGLOBAL = true : own factors in the global scratch next to the accumulators, read one member ahead through L2;
//                  shared memory then only holds the tables and the number of chains per SM is set by registers.
template <int TB, bool WGLOBAL, int GW>
__global__ void __launch_bounds__(TB) mcmc_kernel(const __grid_constant__ McmcParams P, const BatchPtrs B, int burn, int rep,
                                                  uint64_t seed, int64_t v_offset, double *__restrict__ scratch, int n_tiles, int fixup,
                                                  unsigned long long *fixup_count) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const RunConstants &C = P.C;
    const McmcPlan &pl = P.plan;
    const int N = pl.n, S = C.s;
    double *s_tab = reinterpret_cast<double *>(smem_raw); // [108][16]
    double *s_w = s_tab + kEntries * kCopies;              // [N][3][TB] own factor: (1e6*prior)*lk or 1e6*lk

    const int tid = threadIdx.x, lane = tid & 31;
    for (int e = tid; e < kEntries * kCopies; e += TB) {
        const int entry = e / kCopies;
        s_tab[e] = entry < 81 ? C.tab[entry / 27][entry % 27] : 1.0;
    }
    __syncthreads();
    const uint32_t tab_addr = (uint32_t)__cvta_generic_to_shared(s_tab) + (uint32_t)(lane & (kCopies - 1)) * 8u;
    const uint32_t w_addr = (uint32_t)__cvta_generic_to_shared(s_w) + (uint32_t)tid * 8u;
    double *acc = scratch + (size_t)blockIdx.x * ((size_t)N * 3 * TB * (WGLOBAL ? 2 : 1)) + tid; // [member][g][TB], thread-private
    double *wg = acc + (size_t)N * 3 * TB;                                                       // WGLOBAL: own factors
    double *w = WGLOBAL ? wg : s_w + tid;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);

    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t v = (int64_t)tile * TB + tid;
        if (v >= B.V) continue;
        if (fixup) { // second pass after the specialised kernel: only what it left (status 2)
            if (B.status[v] != 2) continue;
            if (fixup_count) atomicAdd(fixup_count, 1ull);
        }
        const unsigned flag = B.flags ? B.flags[v] : 0u;
        const bool chrx = (flag >> 1) & 1u;
        const VariantPriors pr = select_priors(C, flag);
        const double *lkv = B.lk + v * S * 3;
        double *gp = B.post + v * S * 3, *gs = B.single + v * S * 3;
        uint8_t *gg = B.gt + v * S;

        // ---- individual-only posterior + LRC gate (family.cpp:1940-1971) ----------------------------------------
        bool failed = C.unseq_fail[flag & 3u] != 0;
        bool pedigree_needed = false;
        for (int c = 0; c < S; c++) {
            const double l0 = lkv[c * 3], l1 = lkv[c * 3 + 1], l2 = lkv[c * 3 + 2];
            const bool male = C.col_male[c] != 0;
            const double r0 = l0 * (male ? pr.m[0] : pr.a[0]);
            const double r1 = l1 * (male ? pr.m[1] : pr.a[1]);
            const double r2 = l2 * (male ? pr.m[2] : pr.a[2]);
            const double rs = __dadd_rn(__dadd_rn(r0, r1), r2);
            if (rs <= 0.0) failed = true;
            gs[c * 3] = r0 / rs;
            gs[c * 3 + 1] = r1 / rs;
            gs[c * 3 + 2] = r2 / rs;
            double big = 0.0;
            if (big < l0) big = l0;
            if (big < l1) big = l1;
            if (big < l2) big = l2;
            const double ls = __dadd_rn(__dadd_rn(l0, l1), l2);
            if (big / ls < C.lrc) pedigree_needed = true;
        }
        if (failed) {
            for (int k = 0; k < S * 3; k++) gp[k] = gs[k] = 0.0;
            for (int c = 0; c < S; c++) gg[c] = 255;
            B.status[v] = 1;
            continue;
        }
        if (!pedigree_needed) { // family.cpp:1973-2058: FPP := individual-only posterior
            for (int c = 0; c < S; c++) {
                const double p0 = gs[c * 3], p1 = gs[c * 3 + 1], p2 = gs[c * 3 + 2];
                gp[c * 3] = p0;
                gp[c * 3 + 1] = p1;
                gp[c * 3 + 2] = p2;
                gg[c] = call_genotype(p0, p1, p2);
            }
            B.status[v] = 0;
            continue;
        }

        // ---- chain state: own factors ((1e6 * prior) * lk for founders, 1e6 * lk otherwise, family.cpp:2115-2126)
        for (int i = 0; i < N; i++) {
            const uint32_t d = pl.member[i];
            const int col = pl.col[i];
#pragma unroll
            for (int g = 0; g < 3; g++) {
                w[(i * 3 + g) * TB] = gibbs_own_factor(d, pr, g, col >= 0 ? lkv[col * 3 + g] : 1.0);
                acc[(size_t)((i * 3 + g) * TB)] = 0.0;
            }
        }
        const uint64_t gv = (uint64_t)(v_offset + v);
        const uint32_t gv_lo = (uint32_t)gv, gv_hi = (uint32_t)(gv >> 32);
        uint32_t r0 = 0, r1 = 0, r2 = 0, r3 = 0;
        Genotypes<GW> cur;
#pragma unroll
        for (int k = 0; k < GW; k++) cur.w[k] = 0;
        for (int i = 0; i < N; i++) { // family.cpp:2063-2067
            if ((i & 3) == 0) philox4x32_10(0u, (uint32_t)(i >> 2), gv_lo, gv_hi, k0, k1, r0, r1, r2, r3);
            const int q = i & 3;
            const uint32_t u = q == 0 ? r0 : (q == 1 ? r1 : (q == 2 ? r2 : r3));
            cur.set(i, (int)(u % 3u));
        }

        // ---- sweeps (the step: mcmc_step.cuh) ---------------------------------------------------------------------
        asm volatile("" ::: "memory");
        double nw0 = 0.0, nw1 = 0.0, nw2 = 0.0; // WGLOBAL: own factors of the next member, fetched one step ahead
        if constexpr (WGLOBAL) {
            nw0 = __ldcg(wg);
            nw1 = __ldcg(wg + TB);
            nw2 = __ldcg(wg + 2 * TB);
        }
        const int total_sweeps = burn + rep;
        for (int sweep = 1; sweep <= total_sweeps; sweep++) {
            const bool sampling = sweep > burn;
            for (int i = 0; i < N; i++) {
                const uint32_t d = pl.member[i];
                double w0, w1, w2;
                if constexpr (WGLOBAL) {
                    w0 = nw0;
                    w1 = nw1;
                    w2 = nw2;
                    const double *nx = wg + (size_t)(((i + 1 < N) ? i + 1 : 0) * 3 * TB);
                    nw0 = __ldcg(nx);
                    nw1 = __ldcg(nx + TB);
                    nw2 = __ldcg(nx + 2 * TB);
                } else {
                    const uint32_t wa = w_addr + (uint32_t)i * (3u * TB * 8u);
                    w0 = lds64(wa);
                    w1 = lds64(wa + TB * 8);
                    w2 = lds64(wa + 2 * TB * 8);
                }
                const double sum = gibbs_weights(d, pl.link, cur, chrx, tab_addr, w0, w1, w2);
                if ((i & 3) == 0) philox4x32_10((uint32_t)sweep, (uint32_t)(i >> 2), gv_lo, gv_hi, k0, k1, r0, r1, r2, r3);
                const uint32_t u = r0; // words are consumed in order: rotate the block
                r0 = r1;
                r1 = r2;
                r2 = r3;
                cur.set(i, gibbs_draw(u, sum, w0, w2));
                if (sampling) { // family.cpp:2175-2178, Rao-Blackwellised
                    const double inv = gibbs_inv(sum);
                    double *a = acc + (size_t)((i * 3) * TB);
                    atomicAdd(a, w0 * inv);
                    atomicAdd(a + TB, w1 * inv);
                    atomicAdd(a + 2 * TB, w2 * inv);
                }
            }
        }

        // ---- postProb = genoFry / numRep, not renormalised; a row summing to <= 0 fails (family.cpp:2082-2092) ----
        const double nrep = (double)rep;
        for (int i = 0; i < N; i++) {
            const double *a = acc + (size_t)((i * 3) * TB);
            const double p0 = __ldcg(a) / nrep, p1 = __ldcg(a + TB) / nrep, p2 = __ldcg(a + 2 * TB) / nrep;
            if (__dadd_rn(__dadd_rn(p0, p1), p2) <= 0.0) failed = true;
            const int c = pl.col[i];
            if (c >= 0) {
                gp[c * 3] = p0;
                gp[c * 3 + 1] = p1;
                gp[c * 3 + 2] = p2;
                gg[c] = call_genotype(p0, p1, p2);
            }
        }
        if (failed) {
            for (int k = 0; k < S * 3; k++) gp[k] = gs[k] = 0.0;
            for (int c = 0; c < S; c++) gg[c] = 255;
        }
        B.status[v] = failed ? 1 : 0;
    }
}

template <int TB, bool WGLOBAL, int GW = 2>
cudaError_t launch_tb(const McmcParams &P, const BatchPtrs &B, int burn, int rep, uint64_t seed, int64_t v_offset, int sm_count,
                      cudaStream_t stream, int blocks_cap, bool fixup, unsigned long long *fixup_count) {
    const size_t smem = WGLOBAL ? (size_t)kEntries * kCopies * sizeof(double) : mcmc_smem_bytes(P, TB);
    cudaError_t rc = cudaFuncSetAttribute(mcmc_kernel<TB, WGLOBAL, GW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc != cudaSuccess) return rc;
    int per_sm = 0;
    rc = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mcmc_kernel<TB, WGLOBAL, GW>, TB, smem);
    if (rc != cudaSuccess) return rc;
    if (per_sm < 1) return cudaErrorInvalidConfiguration;
    if (WGLOBAL) { // resident blocks per SM (measured on ped40: 1 -> 1.60e5, 2 -> 1.63e5, 3 -> 1.79e5 variants/s)
        per_sm = std::min(per_sm, std::max(1, blocks_cap));
    }
    const int64_t n_tiles = (B.V + TB - 1) / TB;
    if (n_tiles > 0x7fffffff) return cudaErrorInvalidValue;
    const int grid = (int)std::min<int64_t>(n_tiles, (int64_t)sm_count * per_sm);
    // thread-private chain state: [grid][N][3][TB] accumulators (+ as many own factors when WGLOBAL), stream-ordered
    double *scratch = nullptr;
    rc = cudaMallocAsync(&scratch, (size_t)grid * P.plan.n * 3 * TB * sizeof(double) * (WGLOBAL ? 2 : 1), stream);
    if (rc != cudaSuccess) return rc;
    mcmc_kernel<TB, WGLOBAL, GW><<<grid, TB, smem, stream>>>(P, B, burn, rep, seed, v_offset, scratch, (int)n_tiles, fixup ? 1 : 0,
                                                           fixup_count);
    rc = cudaGetLastError();
    const cudaError_t rc2 = cudaFreeAsync(scratch, stream);
    return rc != cudaSuccess ? rc : rc2;
}

} // namespace

size_t mcmc_smem_bytes(const McmcParams &P, int tb) { return (size_t)(kEntries * kCopies + P.plan.n * 3 * tb) * sizeof(double); }

// Block size that keeps the most chains resident per SM.
int mcmc_pick_block(const McmcParams &P, size_t smem_limit, size_t smem_per_sm) {
    int best = 0, best_threads = 0;
    for (int tb = 256; tb >= 32; tb -= 32) {
        const size_t need = mcmc_smem_bytes(P, tb) + 1024; // 1 KB per-block reservation
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

cudaError_t launch_mcmc(const McmcParams &P, const BatchPtrs &B, int tb, int burn, int rep, uint64_t seed, int64_t v_offset,
                        int sm_count, cudaStream_t stream, const McmcTuning &tune, bool fixup, unsigned long long *fixup_count) {
    if (B.V <= 0) return cudaSuccess;
    // Large pedigrees: the own factors of fewer than 512 chains fit in an SM's shared memory -> keep them in L2 instead.
    const bool wglobal = tune.wglobal < 0 ? tb < 256 : tune.wglobal != 0;
    if (P.plan.n > 64) return launch_tb<256, true, 4>(P, B, burn, rep, seed, v_offset, sm_count, stream, tune.blocks_cap, fixup, fixup_count); // wide genotype vector
    if (wglobal) return launch_tb<256, true>(P, B, burn, rep, seed, v_offset, sm_count, stream, tune.blocks_cap, fixup, fixup_count);
    switch (tb) {
    case 256: return launch_tb<256, false>(P, B, burn, rep, seed, v_offset, sm_count, stream, tune.blocks_cap, fixup, fixup_count);
    case 224: return launch_tb<224, false>(P, B, burn, rep, seed, v_offset, sm_count, stream, tune.blocks_cap, fixup, fixup_count);
    case 192: return launch_tb<192, false>(P, B, burn, rep, seed, v_offset, sm_count, stream, tune.blocks_cap, fixup, fixup_count);
    case 160: return launch_tb<160, false>(P, B, burn, rep, seed, v_offset, sm_count, stream, tune.blocks_cap, fixup, fixup_count);
    case 128: return launch_tb<128, false>(P, B, burn, rep, seed, v_offset, sm_count, stream, tune.blocks_cap, fixup, fixup_count);
    case 96: return launch_tb<96, false>(P, B, burn, rep, seed, v_offset, sm_count, stream, tune.blocks_cap, fixup, fixup_count);
    case 64: return launch_tb<64, false>(P, B, burn, rep, seed, v_offset, sm_count, stream, tune.blocks_cap, fixup, fixup_count);
    case 32: return launch_tb<32, false>(P, B, burn, rep, seed, v_offset, sm_count, stream, tune.blocks_cap, fixup, fixup_count);
    default: return cudaErrorInvalidValue;
    }
}

} // namespace famseq
