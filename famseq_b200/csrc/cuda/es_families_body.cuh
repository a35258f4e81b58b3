// es_families_body.cuh -- the per-variant work of the cohort kernel (es_families_kernel.cu): individual-only posteriors,
// the whole-row LRC gate and failure flag, the nuclear families and lone individuals.  Shared with es_cohort_head_kernel
// (es_cohort_kernel.cu), which runs it for cohorts that also hold families peeled by message programs.
#pragma once

#include "es_nuclear_kernel.cuh"

namespace famseq {

namespace {


// OR of `x` over the group that shares the variant.  Also orders the group's global-memory writes before what follows
// (the failure path overwrites rows other threads of the group wrote).
__device__ __forceinline__ bool group_any(bool x, int G) {
    if (G > 32) return __syncthreads_or(x); // the group is the whole block
    const unsigned votes = __ballot_sync(0xffffffffu, x);
    const unsigned base = (threadIdx.x & 31u) & ~(unsigned)(G - 1);
    const unsigned mine = G == 32 ? 0xffffffffu : ((1u << G) - 1u) << base;
    __syncwarp();
    return (votes & mine) != 0;
}

struct SexBits {
    unsigned bits;
    __device__ __forceinline__ unsigned operator[](int c) const { return (bits >> c) & 1u; }
};

// Family f (class NC >= 1) of this variant; true when the reference would fail the variant.
template <int NC, bool X, bool PL>
__device__ __forceinline__ bool peel_family(const FamiliesParams &P, int f, const VariantPriors &pr, const void *in_row,
                                            const double *__restrict__ lut, const OutRows &out) {
    const int F = P.n_families;
    int col[NC + 2];
    Row3 L[NC + 2];
#pragma unroll
    for (int r = 0; r < NC + 2; r++) {
        col[r] = P.fam_col[r * F + f];
        L[r] = load_lk<PL>(in_row, lut, col[r]);
    }
    const SexBits male{P.fam_male[f]};
    Row3 wf, wm; // lk * prior of the founders: the father is male, the mother is not
#pragma unroll
    for (int g = 0; g < 3; g++) {
        wf.v[g] = L[0].v[g] * pr.m[g];
        wm.v[g] = L[1].v[g] * pr.a[g];
    }
    Divider<false, X> div;
    return peel<NC, X>(P.C, male, pr, L, wf, wm, col, out, div);
}

// A lone individual: (1 * lk) * prior over its sum, the message program's FIN with an empty spouse product
// (es_program.cpp:48-57); 1 * lk == lk bit for bit.
template <bool X, bool PL>
__device__ __forceinline__ bool peel_lone(const FamiliesParams &P, int f, const VariantPriors &pr, const void *in_row,
                                          const double *__restrict__ lut, const OutRows &out) {
    const int col = P.fam_col[f];
    const Row3 L = load_lk<PL>(in_row, lut, col);
    const bool male = P.fam_male[f] & 1u;
    Row3 a;
#pragma unroll
    for (int g = 0; g < 3; g++) a.v[g] = male ? pr.m[g] : pr.a[g];
    Divider<false, X> div;
    return finish(div, L, a, out, col);
}

template <int NCMAX, bool X, bool PL>
__device__ __forceinline__ bool peel_any(const FamiliesParams &P, int f, const VariantPriors &pr, const void *in_row,
                                         const double *__restrict__ lut, const OutRows &out) {
    int k = 0; // children of family f
#pragma unroll
    for (int c = 0; c < NCMAX; c++) k += f >= P.class_end[c];
    if (k == 0) return peel_lone<X, PL>(P, f, pr, in_row, lut, out);
    if constexpr (NCMAX >= 1) if (k == 1) return peel_family<1, X, PL>(P, f, pr, in_row, lut, out);
    if constexpr (NCMAX >= 2) if (k == 2) return peel_family<2, X, PL>(P, f, pr, in_row, lut, out);
    if constexpr (NCMAX >= 3) if (k == 3) return peel_family<3, X, PL>(P, f, pr, in_row, lut, out);
    if constexpr (NCMAX >= 4) if (k == 4) return peel_family<4, X, PL>(P, f, pr, in_row, lut, out);
    if constexpr (NCMAX >= 5) return peel_family<5, X, PL>(P, f, pr, in_row, lut, out);
    return false;
}

// The work of es_families_kernel for the variant of this thread's group.  NCMAX: largest sibship of the cohort (the register
// budget is that of the largest family shape instantiated).  DEFER (es_cohort_head_kernel): the families peeled by message
// programs are still to come, so instead of the NA rows and `status` the group records status = failed | needed << 1 for
// the program kernel and the finish pass (es_cohort_kernel.cu).
template <int NCMAX, bool PL, bool SINGLE, bool DEFER>
__device__ __forceinline__ void es_families_row(const FamiliesParams &P, const BatchPtrs B) {
    const RunConstants &C = P.C;
    const int S = C.s, S3 = 3 * S, G = P.group;
    const int lane = threadIdx.x & (G - 1);
    const int64_t v = (int64_t)blockIdx.x * (ES_FAMILIES_BLOCK / G) + threadIdx.x / G;
    const bool live = v < B.V; // every thread takes part in the group reductions
    const int64_t row = live ? v : 0;
    const unsigned flag = (live && B.flags) ? B.flags[row] : 0u;
    const VariantPriors pr = select_priors(C, flag);
    const void *in_row = PL ? static_cast<const void *>(B.pl + row * S3) : static_cast<const void *>(B.lk + row * S3);
    double *post_row = B.post + row * S3;
    uint8_t *gt_row = B.gt + row * S;

    // individual-only posterior of column c (family.cpp:1405-1499)
    auto single_of = [&](int c, const Row3 &l, double &q0, double &q1, double &q2) {
        const bool male = P.col_male[c] != 0;
        const double r0 = l.v[0] * (male ? pr.m[0] : pr.a[0]);
        const double r1 = l.v[1] * (male ? pr.m[1] : pr.a[1]);
        const double r2 = l.v[2] * (male ? pr.m[2] : pr.a[2]);
        const double rs = (r0 + r1) + r2;
        q0 = r0 / rs;
        q1 = r1 / rs;
        q2 = r2 / rs;
        return rs;
    };

    // 1. individual-only posteriors, failure and LRC gate (family.cpp:1140-1162) over the whole row
    bool failed = false, needed = false;
    if (live) {
        failed = C.unseq_fail[flag & 3u] != 0;
        for (int c = lane; c < S; c += G) {
            const Row3 l = load_lk<PL>(in_row, B.lut, c);
            double q0, q1, q2;
            if (single_of(c, l, q0, q1, q2) <= 0.0) failed = true;
            if (SINGLE) {
                double *s = B.single + row * S3 + c * 3;
                s[0] = q0, s[1] = q1, s[2] = q2;
            }
            double big = 0.0;
            if (big < l.v[0]) big = l.v[0];
            if (big < l.v[1]) big = l.v[1];
            if (big < l.v[2]) big = l.v[2];
            const double ls = (l.v[0] + l.v[1]) + l.v[2];
            if (lrc_wants_pedigree(C.lrc, l.v[0], l.v[1], l.v[2], big, ls)) needed = true;
        }
    }
    failed = group_any(failed, G);
    needed = group_any(needed, G);

    // 2. the pedigree, one family per thread; or, when no sample asks for it, FPP := GPP (family.cpp:1164-1249)
    if (live && !failed) {
        if (needed) {
            const OutRows out{post_row, gt_row};
            const bool x = (flag >> 1) & 1u;
            for (int f = lane; f < P.n_families; f += G)
                failed |= x ? peel_any<NCMAX, true, PL>(P, f, pr, in_row, B.lut, out) : peel_any<NCMAX, false, PL>(P, f, pr, in_row, B.lut, out);
        } else {
            for (int c = lane; c < S; c += G) {
                double q0, q1, q2;
                single_of(c, load_lk<PL>(in_row, B.lut, c), q0, q1, q2);
                post_row[c * 3] = q0, post_row[c * 3 + 1] = q1, post_row[c * 3 + 2] = q2;
                gt_row[c] = call_genotype(q0, q1, q2);
            }
        }
    }
    failed = group_any(failed, G);

    if constexpr (DEFER) {
        if (live && lane == 0) B.status[row] = (failed ? 1 : 0) | (needed ? 2 : 0);
        return;
    }
    // 3. a failing variant reports every sample as NA
    if (live) {
        if (failed)
            for (int c = lane; c < S; c += G) {
                post_row[c * 3] = post_row[c * 3 + 1] = post_row[c * 3 + 2] = 0.0;
                if (SINGLE) {
                    double *s = B.single + row * S3 + c * 3;
                    s[0] = s[1] = s[2] = 0.0;
                }
                gt_row[c] = 255;
            }
        if (lane == 0) B.status[row] = failed ? 1 : 0;
    }
}

} // namespace

} // namespace famseq
