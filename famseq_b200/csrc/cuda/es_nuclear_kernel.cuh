// es_nuclear_kernel.cuh -- Elston-Stewart peeling for NUCLEAR FAMILIES (two founders and their C <= 5
// childless children: trios, quads, ...), the pedigree shape of almost every real FamSeq run and of the
// headline benchmark (BASELINE.json: 10 M-variant trio).  One variant per thread, everything in registers.
//
// It computes exactly what the message program of es_kernel.cu computes for such a pedigree -- the same
// products in the same association order as the reference (family.cpp:1501-1649, :1783-1845, :1292-1314;
// compiled with -fmad=false) -- so the doubles are bit-identical to the reference CPU build; the general
// interpreter remains the path for every other loop-free pedigree.  What the specialisation buys:
//   * no interpreter, no scratch in shared memory: ~3x fewer instructions per variant;
//   * the per-child vectors  K_c[a][b] = sum_l T_c[l][a][b] * lk_c[l]  are formed once and shared by the two
//     posterior messages and by the sibs' anterior messages (the recursion re-derives them each time);
//   * x/s for the three genotypes of a row shares one correctly rounded reciprocal (one Markstein
//     correction step per quotient); a variant with an operand outside the safe exponent range, a failing row
//     or an LRC gate that keeps the pedigree out is redone by the complete pass with plain IEEE divisions;
//     tests/test_parity_gpu.py::test_nuclear_fast_path_is_bit_identical checks the result bit for bit;
//   * the block's input tile ([TB][S][3] FP64, contiguous in HBM) arrives through one TMA bulk copy
//     (cp.async.bulk + mbarrier) and the post / single / gt / status tiles leave through TMA bulk stores, so
//     global traffic is fully coalesced 16-byte-granular and costs no LSU wavefronts.
// HBM-bound: 73*S+2 algorithmic bytes per variant (221 B for a trio).
#include <algorithm>
#include <type_traits>

#pragma once

#include "common.cuh"
#include "kernels.hpp"

namespace famseq {

namespace {

// ---- TMA bulk copy helpers (sm_90+ PTX, SASS: UBLKCP) -------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_load(void *smem_dst, const void *gmem_src, unsigned bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_store(void *gmem_dst, const void *smem_src, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit_and_wait_read() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <bool X> __device__ __forceinline__ double trans(const RunConstants &C, int sel, int g, int a, int b) {
    return X ? C.tab[sel][g * 9 + a * 3 + b] : C.tab[0][g * 9 + a * 3 + b];
}

struct Row3 {
    double v[3];
};

// Likelihood row of input column `col` of this thread's variant: FP64 as it stands, or (compact input, fs_run_pl)
// integer Phred-scaled likelihoods decoded through the host-built table lut[pl] = pow(10, -pl/10) (file.cpp:588-590).
template <bool PL> __device__ __forceinline__ Row3 load_lk(const void *in_row, const double *__restrict__ lut, int col) {
    Row3 r;
    if (col < 0) {
        r.v[0] = r.v[1] = r.v[2] = 1.0; // unsequenced member (file.cpp:565)
    } else if (PL) {
        const uint16_t *q = static_cast<const uint16_t *>(in_row) + col * 3;
        r.v[0] = __ldg(lut + q[0]);
        r.v[1] = __ldg(lut + q[1]);
        r.v[2] = __ldg(lut + q[2]);
    } else {
        const double *q = static_cast<const double *>(in_row) + col * 3;
        r.v[0] = q[0];
        r.v[1] = q[1];
        r.v[2] = q[2];
    }
    return r;
}

// Where a thread's results go: its rows of the post / gt tiles in shared memory.
struct OutRows {
    double *post;
    uint8_t *gt;
    __device__ __forceinline__ void put(int col, double p0, double p1, double p2) const {
        if (col < 0) return; // unsequenced member: nothing is reported for it
        post[col * 3] = p0;
        post[col * 3 + 1] = p1;
        post[col * 3 + 2] = p2;
        gt[col] = call_genotype(p0, p1, p2);
    }
};

// ---- x[0..2] / s for the rows of one variant ------------------------------------------------------------------
// Every row this kernel normalises has the form x0, x1, x2 >= 0, s = (x0 + x1) + x2, so x_i <= s.
//   FAST = false: IEEE divisions.  Used by the complete ("exact") pass, which also evaluates every failure rule.
//   FAST = true : one correctly rounded reciprocal per row and one Markstein correction per quotient (common.cuh,
//                 div3), which IS the IEEE quotient when s and the x_i are normal numbers in [2^-900, 2^900] (ZEROS: or
//                 exact zeros -- the chrX priors contain structural zeros).  Instead of guarding every division, the
//                 fast pass only RECORDS (in `bad`) whether an operand ever left that range: two integer min/max on the
//                 high words per row (non-negative doubles order like their high words; a negative, NaN or infinite
//                 operand lands outside as well).  A variant with bad == true is redone by the exact pass, so nothing is
//                 approximated; in range, both passes produce the same bytes (tests/test_parity_gpu.py,
//                 test_nuclear_fast_path_is_bit_identical runs wide-exponent inputs through both).
constexpr int kHiLo = (1023 - 900) << 20, kHiHi = (1023 + 900) << 20;
template <bool FAST, bool ZEROS> struct Divider {
    static constexpr bool fast = FAST;
    bool bad = false;
    __device__ __forceinline__ static int key(double x) {
        const int h = __double2hiint(x);
        if (!ZEROS) return h;
        return (h | __double2loint(x)) == 0 ? kHiLo : h; // an exact zero divides exactly
    }
    __device__ __forceinline__ void check(double x0, double x1, double x2, double s) {
        // x_i <= s, so the x_i need the lower bound only; s needs both (ZEROS: every x_i may be an exact zero, and so s)
        bad |= (min(min(key(x0), key(x1)), key(x2)) < kHiLo) | ((unsigned)(__double2hiint(s) - kHiLo) > (unsigned)(kHiHi - kHiLo));
    }
    __device__ __forceinline__ void operator()(double x0, double x1, double x2, double s, double &q0, double &q1, double &q2) {
        if (FAST) {
            check(x0, x1, x2, s);
            const double r = __drcp_rn(s);
            const double a = __dmul_rn(x0, r), b = __dmul_rn(x1, r), c = __dmul_rn(x2, r);
            q0 = __fma_rn(__fma_rn(-s, a, x0), r, a);
            q1 = __fma_rn(__fma_rn(-s, b, x1), r, b);
            q2 = __fma_rn(__fma_rn(-s, c, x2), r, c);
        } else {
            q0 = x0 / s;
            q1 = x1 / s;
            q2 = x2 / s;
        }
    }
};

// marginal of one member: v = (m * l) * a, row sum == 0 fails the variant (family.cpp:1296-1314).  In the fast pass a zero
// (or any out-of-range) sum is caught by the divider instead.
template <class Div> __device__ __forceinline__ bool finish(Div &div, const Row3 &ml, const Row3 &a, const OutRows &out, int col) {
    const double v0 = ml.v[0] * a.v[0], v1 = ml.v[1] * a.v[1], v2 = ml.v[2] * a.v[2];
    const double sum = (v0 + v1) + v2;
    double p0, p1, p2;
    div(v0, v1, v2, sum, p0, p1, p2);
    out.put(col, p0, p1, p2);
    return sum == 0.0;
}

// The peeling of a nuclear family; returns true when the reference would return false.  Rows are indexed by ROLE:
// 0 father, 1 mother, 2.. children in ped order.  wf / wm = prior * lk of the founders (the numerators of their
// individual-only posteriors: the same products, formed once).  male_child[c] != 0: child c is male.  Shared with the
// cohort kernel (es_families_kernel.cu), which peels many such families per variant.
template <int NC, bool X, class Div, class Male>
__device__ __forceinline__ bool peel(const RunConstants &C, const Male &male_child, const VariantPriors &pr, const Row3 (&L)[NC + 2],
                                     const Row3 &wf, const Row3 &wm, const int (&col)[NC + 2], const OutRows &out, Div &div) {
    // K[c][a][b] = sum_l (T_c[l][a][b] * lk_c[l])
    double K[NC][3][3];
#pragma unroll
    for (int c = 0; c < NC; c++) {
        const Row3 &lc = L[2 + c];
        const int sel = male_child[c] ? K_TAB_XM : K_TAB_XF;
#pragma unroll
        for (int a = 0; a < 3; a++)
#pragma unroll
            for (int b = 0; b < 3; b++) {
                double sc = trans<X>(C, sel, 0, a, b) * lc.v[0];
                sc = sc + trans<X>(C, sel, 1, a, b) * lc.v[1];
                sc = sc + trans<X>(C, sel, 2, a, b) * lc.v[2];
                K[c][a][b] = sc;
            }
    }
    // product over all children, in ped order (the posterior messages of both parents use it)
    double kids[3][3];
#pragma unroll
    for (int a = 0; a < 3; a++)
#pragma unroll
        for (int b = 0; b < 3; b++) {
            double p = K[0][a][b];
#pragma unroll
            for (int c = 1; c < NC; c++) p = p * K[c][a][b];
            kids[a][b] = p;
        }
    // posterior messages.  Autosome: the table index is (own genotype, spouse genotype) for both parents
    // (family.cpp:1836); chrX: (mother, father) (family.cpp:1900-1921).
    Row3 pl_f, pl_m; // (posterior message * lk) of the founders
#pragma unroll
    for (int g = 0; g < 3; g++) {
        double a = wf.v[0] * kids[g][0]; // mother g, father b
        a = a + wf.v[1] * kids[g][1];
        a = a + wf.v[2] * kids[g][2];
        pl_m.v[g] = a * L[1].v[g];
        double f = wm.v[0] * (X ? kids[0][g] : kids[g][0]);
        f = f + wm.v[1] * (X ? kids[1][g] : kids[g][1]);
        f = f + wm.v[2] * (X ? kids[2][g] : kids[g][2]);
        pl_f.v[g] = f * L[0].v[g];
    }
    Row3 prior_f, prior_m;
#pragma unroll
    for (int g = 0; g < 3; g++) {
        prior_f.v[g] = pr.m[g]; // the father is male: chrX male prior on X (family.cpp:1281-1290 / :1337-1358)
        prior_m.v[g] = pr.a[g];
    }
    bool failed = false;
    // every member's row sum is checked (the order of the members does not matter for the values)
    failed |= finish(div, pl_f, prior_f, out, col[0]);
    failed |= finish(div, pl_m, prior_m, out, col[1]);
#pragma unroll
    for (int c = 0; c < NC; c++) {
        const int sel = male_child[c] ? K_TAB_XM : K_TAB_XF;
        Row3 ant;
#pragma unroll
        for (int g = 0; g < 3; g++) {
            // the reference starts both sums from 0.0; 0.0 + t == t bit for bit unless t is -0.0, which needs a negative
            // likelihood -- and those variants belong to the complete pass, so the fast pass skips the two additions
            double over_m = 0.0;
#pragma unroll
            for (int a = 0; a < 3; a++) {
                double over_f = 0.0;
#pragma unroll
                for (int b = 0; b < 3; b++) {
                    double term = wf.v[b] * trans<X>(C, sel, g, a, b);
                    if (NC > 1) { // full sibs in the mother's child order (family.cpp:1576-1587, :1616-1631)
                        double sibs = 1.0;
                        bool first = true;
#pragma unroll
                        for (int k = 0; k < NC; k++) {
                            if (k == c) continue;
                            sibs = first ? K[k][a][b] : sibs * K[k][a][b];
                            first = false;
                        }
                        term = term * sibs;
                    }
                    over_f = (Div::fast && b == 0) ? term : over_f + term;
                }
                over_m = (Div::fast && a == 0) ? wm.v[a] * over_f : over_m + wm.v[a] * over_f;
            }
            ant.v[g] = over_m;
        }
        failed |= finish(div, L[2 + c], ant, out, col[2 + c]); // the posterior message of a childless member is (1, 1, 1): 1 * lk = lk
    }
    return failed;
}

// One variant: individual-only posterior, LRC gate, peeling, genotype calls -- from the thread's row of the input tile
// into its rows of the output tiles (all in shared memory).  Everything in between lives in registers, indexed by role.
//
// FAST = false is the complete computation (every rule of the reference: failing rows, any -LRC value, the LRC gate
// keeping the pedigree out).  FAST = true is the same arithmetic for the case that is nearly every variant -- default
// -LRC 1, pedigree needed, nothing fails, every division in the divider's range -- without the tests for the others; it
// returns true when the variant was not such a case, and the caller then runs the complete computation over it.
template <int NC, bool PL, bool SINGLE, bool X, bool FAST, bool IDENT>
__device__ __forceinline__ bool variant_body(const NuclearParams &P, unsigned flag, const void *in_row, const double *__restrict__ lut,
                                             double *post_row, double *single_row, uint8_t *gt_row, uint8_t *status) {
    constexpr int NR = NC + 2;
    const RunConstants &C = P.C;
    VariantPriors pr;
    {   // prior[known] for females and autosomes, prior[2 + known] for males on chrX: per-thread constant-bank look-ups
        const int known = flag & 1u;
#pragma unroll
        for (int g = 0; g < 3; g++) {
            pr.a[g] = C.prior[known][g];
            pr.m[g] = X ? C.prior[2 + known][g] : pr.a[g];
        }
    }
    int col[NR];
    bool male[NR];
    // IDENT: every member sequenced, input columns in role order (father, mother, children) -- the column of a role is a
    // literal and the address arithmetic of the row accesses folds away
    col[0] = IDENT ? 0 : P.col_father;
    col[1] = IDENT ? 1 : P.col_mother;
    male[0] = true;
    male[1] = false;
#pragma unroll
    for (int c = 0; c < NC; c++) {
        col[2 + c] = IDENT ? 2 + c : P.col_child[c];
        male[2 + c] = P.male_child[c] != 0;
    }
    // individual-only posterior (family.cpp:1405-1499) and LRC gate (family.cpp:1140-1162)
    const OutRows out{post_row, gt_row};
    Divider<FAST, X> div;
    Row3 L[NR], W[2]; // lk of every role; lk * prior of the founders (also their "anterior * lk" in the peeling)
    bool failed = C.unseq_fail[flag & 3u] != 0;
    bool pedigree_needed = false;
#pragma unroll
    for (int r = 0; r < NR; r++) {
        L[r] = load_lk<PL>(in_row, lut, col[r]);
        const double w0 = L[r].v[0] * (male[r] ? pr.m[0] : pr.a[0]);
        const double w1 = L[r].v[1] * (male[r] ? pr.m[1] : pr.a[1]);
        const double w2 = L[r].v[2] * (male[r] ? pr.m[2] : pr.a[2]);
        if (r < 2) W[r].v[0] = w0, W[r].v[1] = w1, W[r].v[2] = w2;
        if (col[r] >= 0) {
            const double rs = (w0 + w1) + w2;
            if (!FAST && rs <= 0.0) failed = true;
            if (SINGLE) {
                const int k = col[r] * 3;
                div(w0, w1, w2, rs, single_row[k], single_row[k + 1], single_row[k + 2]);
            } else if (FAST) {
                div.check(w0, w1, w2, rs); // a row sum <= 0 (or NaN) must not go unnoticed
            }
            const double ls = (L[r].v[0] + L[r].v[1]) + L[r].v[2];
            if (FAST) {
                // -LRC 1 and non-negative likelihoods (anything else is left to the complete pass): big / ls < 1 <=> big < ls,
                // and since ls >= big, the sample is certain exactly when ls equals one of its three likelihoods
                if (!((ls == L[r].v[0]) | (ls == L[r].v[1]) | (ls == L[r].v[2]))) pedigree_needed = true;
            } else {
                double big = 0.0;
                if (big < L[r].v[0]) big = L[r].v[0];
                if (big < L[r].v[1]) big = L[r].v[1];
                if (big < L[r].v[2]) big = L[r].v[2];
                if (lrc_wants_pedigree(C.lrc, L[r].v[0], L[r].v[1], L[r].v[2], big, ls)) pedigree_needed = true;
            }
        }
    }
    if (FAST) {
        peel<NC, X>(C, P.male_child, pr, L, W[0], W[1], col, out, div);
        *status = 0;
        // not this pass's case: an individual-only failure, a likelihood that is negative, NaN or out of the divider's range
        // (the products inherit it), the LRC gate keeping the pedigree out, another -LRC value
        return failed | div.bad | !pedigree_needed | (C.lrc != 1.0);
    }
    if (!failed) {
        if (!pedigree_needed) { // FPP := GPP (family.cpp:1164-1249); rare with the default -LRC 1
#pragma unroll
            for (int r = 0; r < NR; r++) {
                if (col[r] < 0) continue;
                double p0, p1, p2;
                if (SINGLE) {
                    p0 = single_row[col[r] * 3], p1 = single_row[col[r] * 3 + 1], p2 = single_row[col[r] * 3 + 2];
                } else {
                    const double w0 = L[r].v[0] * (male[r] ? pr.m[0] : pr.a[0]);
                    const double w1 = L[r].v[1] * (male[r] ? pr.m[1] : pr.a[1]);
                    const double w2 = L[r].v[2] * (male[r] ? pr.m[2] : pr.a[2]);
                    div(w0, w1, w2, (w0 + w1) + w2, p0, p1, p2);
                }
                out.put(col[r], p0, p1, p2);
            }
        } else {
            failed = peel<NC, X>(C, P.male_child, pr, L, W[0], W[1], col, out, div);
        }
    }
    if (failed) { // the reference returns false: every sample of the variant is reported as NA
        const int S = IDENT ? NR : C.s;
        for (int k = 0; k < 3 * S; k++) {
            post_row[k] = 0.0;
            if (SINGLE) single_row[k] = 0.0;
        }
        for (int c = 0; c < S; c++) gt_row[c] = 255;
    }
    *status = failed ? 1 : 0;
    return false;
}

// The complete computation, kept out of line: it runs for the few variants the fast pass hands over.
template <int NC, bool PL, bool SINGLE, bool IDENT>
__device__ __noinline__ void variant_exact(const NuclearParams &P, unsigned flag, const void *in_row, const double *__restrict__ lut, double *post_row,
                                           double *single_row, uint8_t *gt_row, uint8_t *status) {
    if ((flag >> 1) & 1u)
        variant_body<NC, PL, SINGLE, true, false, IDENT>(P, flag, in_row, lut, post_row, single_row, gt_row, status);
    else
        variant_body<NC, PL, SINGLE, false, false, IDENT>(P, flag, in_row, lut, post_row, single_row, gt_row, status);
}

template <int NC, bool PL, bool SINGLE, bool IDENT>
__device__ __forceinline__ void variant_thread(const NuclearParams &P, unsigned flag, const void *in_row, const double *__restrict__ lut,
                                               double *post_row, double *single_row, uint8_t *gt_row, uint8_t *status) {
    const bool redo = ((flag >> 1) & 1u) ? variant_body<NC, PL, SINGLE, true, true, IDENT>(P, flag, in_row, lut, post_row, single_row, gt_row, status)
                                         : variant_body<NC, PL, SINGLE, false, true, IDENT>(P, flag, in_row, lut, post_row, single_row, gt_row, status);
    if (redo) variant_exact<NC, PL, SINGLE, IDENT>(P, flag, in_row, lut, post_row, single_row, gt_row, status);
}

// PL = compact input (uint16 Phred-scaled likelihoods + decode table), SINGLE = the caller wants the individual-only
// posteriors too (B.single != nullptr).
// MINB: resident blocks per SM the register allocation must allow (0: the compiler's choice).
template <int NC, int TB, bool PL, bool SINGLE, bool IDENT, int MINB>
__global__ void __launch_bounds__(TB, MINB > 0 ? MINB : 1) es_nuclear_kernel(const __grid_constant__ NuclearParams P, const BatchPtrs B) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    using In = typename std::conditional<PL, uint16_t, double>::type;
    const RunConstants &C = P.C;
    const int S = IDENT ? NC + 2 : C.s, S3 = 3 * S;
    const unsigned out_bytes = (unsigned)(TB * S3 * sizeof(double));
    const unsigned in_bytes = (unsigned)(TB * S3 * sizeof(In)); // 192 S (PL) or 768 S bytes per 32 variants: a multiple of 16
    double *s_post = reinterpret_cast<double *>(smem_raw); // [TB][S][3]
    double *s_single = s_post + (SINGLE ? TB * S3 : 0);
    In *s_in = reinterpret_cast<In *>(s_single + TB * S3);                           // [TB][S][3]
    uint8_t *s_gt = reinterpret_cast<uint8_t *>(s_in) + ((in_bytes + 15u) & ~15u); // [TB][S]
    uint8_t *s_status = s_gt + ((TB * S + 15) & ~15);                              // [TB]
    __shared__ uint64_t bar;

    const int tid = threadIdx.x;
    const int64_t v0 = (int64_t)blockIdx.x * TB;
    const int nv = (int)min((int64_t)TB, B.V - v0);
    const bool full = nv == TB; // full tiles go through TMA; the ragged last tile uses plain loads/stores
    const In *g_in = (PL ? reinterpret_cast<const In *>(B.pl) : reinterpret_cast<const In *>(B.lk)) + v0 * S3;

    auto block_sync = [] { // a one-warp block needs no CTA barrier
        if (TB == 32)
            __syncwarp();
        else
            __syncthreads();
    };
    if (full) {
        if (tid == 0) mbar_init(&bar, 1);
        block_sync();
        if (tid == 0) {
            mbar_expect_tx(&bar, in_bytes);
            bulk_load(s_in, g_in, in_bytes, &bar);
        }
    } else {
        for (int k = tid; k < nv * S3; k += TB) s_in[k] = g_in[k];
    }
    unsigned flag = 0;
    if (tid < nv && B.flags) flag = B.flags[v0 + tid];
    if (full)
        mbar_wait(&bar, 0);
    else
        block_sync();

    if (tid < nv)
        variant_thread<NC, PL, SINGLE, IDENT>(P, flag, s_in + tid * S3, B.lut, s_post + tid * S3, s_single + tid * S3, s_gt + tid * S, s_status + tid);

    if (full) {
        fence_async_smem(); // make this thread's shared-memory writes visible to the TMA engine
        block_sync();
        if (tid == 0) {
            bulk_store(B.post + v0 * S3, s_post, out_bytes);
            if (SINGLE) bulk_store(B.single + v0 * S3, s_single, out_bytes);
            bulk_store(B.gt + v0 * S, s_gt, (unsigned)(TB * S));
            bulk_store(B.status + v0, s_status, (unsigned)TB);
            bulk_commit_and_wait_read(); // shared memory must stay alive until the engine has read it
        }
    } else {
        block_sync();
        for (int k = tid; k < nv * S3; k += TB) {
            B.post[v0 * S3 + k] = s_post[k];
            if (SINGLE) B.single[v0 * S3 + k] = s_single[k];
        }
        for (int k = tid; k < nv * S; k += TB) B.gt[v0 * S + k] = s_gt[k];
        if (tid < nv) B.status[v0 + tid] = s_status[tid];
    }
}

// The same computation for compact input as a tile pipeline: a block walks a short list of consecutive tiles.  The compact tile
// is small (192 S bytes + 32 flags), so it is double-buffered: tile k+1's TMA copy is issued when tile k starts and lands under
// its arithmetic; the stores of tile k are committed and left alone, and only waited for (the copy engine's READ of shared
// memory) right before tile k+1 writes the same rows.  With compact input the kernel is bound by instruction issue and
// latencies, not HBM: with one tile per block a warp spent 20 % of its life waiting for its 576 bytes to arrive
// (profiles/r2i_es_l3_sass.csv.gz: the mbarrier loop).
template <int NC, bool SINGLE, bool IDENT, int MINB>
__global__ void __launch_bounds__(32, MINB > 0 ? MINB : 1) es_nuclear_stream_kernel(const __grid_constant__ NuclearParams P, const BatchPtrs B, const int list_len) {
    constexpr int TB = 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const RunConstants &C = P.C;
    const int S = IDENT ? NC + 2 : C.s, S3 = 3 * S;
    const unsigned out_bytes = (unsigned)(TB * S3 * sizeof(double));
    const unsigned in_bytes = (unsigned)(TB * S3 * sizeof(uint16_t)), in_stride = (in_bytes + 15u) & ~15u;
    double *s_post = reinterpret_cast<double *>(smem_raw); // [TB][S][3]
    double *s_single = s_post + (SINGLE ? TB * S3 : 0);
    unsigned char *s_in2 = reinterpret_cast<unsigned char *>(s_single + TB * S3); // [2][TB][S][3] uint16
    uint8_t *s_gt = s_in2 + 2 * in_stride;                                         // [TB][S]
    uint8_t *s_status = s_gt + ((TB * S + 15) & ~15);                              // [TB]
    uint8_t *s_flags2 = s_status + TB;                                             // [2][TB]: the flags travel with their tile
    __shared__ uint64_t bar;

    const int lane = threadIdx.x;
    const int64_t n_tiles = (B.V + TB - 1) / TB, n_full = B.V / TB;
    int64_t tile = (int64_t)blockIdx.x * list_len; // this block's tiles: list_len consecutive ones
    const int64_t list_end = min(n_tiles, tile + list_len);
    if (tile >= list_end) return;
    const unsigned tx_bytes = in_bytes + (B.flags ? (unsigned)TB : 0u);
    auto fetch = [&](int64_t t, unsigned buf) { // lane 0: tile t into buffer buf
        mbar_expect_tx(&bar, tx_bytes);
        bulk_load(s_in2 + buf * in_stride, B.pl + t * TB * S3, in_bytes, &bar);
        if (B.flags) bulk_load(s_flags2 + buf * TB, B.flags + t * TB, (unsigned)TB, &bar);
    };
    if (lane == 0) {
        mbar_init(&bar, 1);
        if (tile < n_full) fetch(tile, 0);
    }
    __syncwarp();
    unsigned phase = 0, it = 0;
    for (; tile < list_end; tile++, it ^= 1u) {
        const int64_t v0 = tile * TB, next = tile + 1;
        const int nv = (int)min((int64_t)TB, B.V - v0);
        const bool full = nv == TB;
        uint16_t *s_in = reinterpret_cast<uint16_t *>(s_in2 + it * in_stride);
        uint8_t *s_flags = s_flags2 + it * TB;
        if (full) {
            mbar_wait(&bar, phase); // issued a tile ago
            phase ^= 1u;
        } else {
            for (int k = lane; k < nv * S3; k += TB) s_in[k] = B.pl[v0 * S3 + k];
            if (B.flags && lane < nv) s_flags[lane] = B.flags[v0 + lane];
        }
        // Every lane has seen this tile's phase complete before the barrier is armed again: a lane still in front of the wait
        // when the NEXT phase completes would be waiting for the one after it (tests/test_nuclear_stream_cpu.py runs the
        // lanes as free-running threads and hangs without this).
        __syncwarp();
        // the next tile into the other buffer (its last readers finished a tile ago, and fenced); one copy in flight per barrier phase
        if (lane == 0 && next < list_end && next < n_full) fetch(next, it ^ 1u);
        if (lane == 0) bulk_wait_read(); // the previous tile's rows have left shared memory
        __syncwarp();
        // (a flag kept in a register across tiles gets spilled under the 72-register budget, and the spill waits for the load:
        // 17 % of the kernel, profiles/r2s_es_l3_sass.csv.gz -- so the flags ride on the tile's TMA transaction)
        const unsigned flag = (B.flags && lane < nv) ? s_flags[lane] : 0u;

        if (lane < nv)
            variant_thread<NC, true, SINGLE, IDENT>(P, flag, s_in + lane * S3, B.lut, s_post + lane * S3, s_single + lane * S3, s_gt + lane * S, s_status + lane);

        if (full) {
            fence_async_smem();
            __syncwarp();
            if (lane == 0) {
                bulk_store(B.post + v0 * S3, s_post, out_bytes);
                if (SINGLE) bulk_store(B.single + v0 * S3, s_single, out_bytes);
                bulk_store(B.gt + v0 * S, s_gt, (unsigned)(TB * S));
                bulk_store(B.status + v0, s_status, (unsigned)TB);
                bulk_commit();
            }
        } else {
            __syncwarp();
            for (int k = lane; k < nv * S3; k += TB) {
                B.post[v0 * S3 + k] = s_post[k];
                if (SINGLE) B.single[v0 * S3 + k] = s_single[k];
            }
            for (int k = lane; k < nv * S; k += TB) B.gt[v0 * S + k] = s_gt[k];
            if (lane < nv) B.status[v0 + lane] = s_status[lane];
        }
    }
    if (lane == 0) bulk_wait_read(); // shared memory must stay alive until the engine has read it
}

template <int NC, bool SINGLE, bool IDENT, int MINB>
cudaError_t launch_stream(const NuclearParams &P, const BatchPtrs &B, cudaStream_t stream) {
    constexpr int TB = 32;
    const size_t S = (size_t)P.C.s;
    const size_t in_bytes = (TB * S * 3 * sizeof(uint16_t) + 15) & ~(size_t)15;
    const size_t smem = (SINGLE ? 2 : 1) * TB * S * 3 * sizeof(double) + 2 * in_bytes + ((TB * S + 15) & ~(size_t)15) + 3 * TB;
    auto kernel = es_nuclear_stream_kernel<NC, SINGLE, IDENT, MINB>;
    cudaError_t rc = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc != cudaSuccess) return rc;
    int device = 0, n_sm = 0, per_sm = 0; // the grid: every block the device can hold at once
    if ((rc = cudaGetDevice(&device)) != cudaSuccess) return rc;
    if ((rc = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device)) != cudaSuccess) return rc;
    if ((rc = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, TB, smem)) != cudaSuccess) return rc;
    if (per_sm < 1) return cudaErrorLaunchOutOfResources;
    // A block takes a SHORT list of consecutive tiles, not its share of the whole batch.  Measured on 10 M trio variants
    // (profiles/r2u_stream.log, r2v_stream.log; fraction of the 167-byte roofline): 1 tile per block 0.805, 2 or 4 tiles 0.865,
    // 8 tiles 0.82, 16 tiles 0.79, one list per resident block 0.67 -- with equal shares the blocks of the slower SMs finish
    // last on their own (16 % of the warp slots empty over the run, profiles/r2s_r2s_es_l3.txt), so the balancing stays with the
    // block scheduler and the lists only have to be long enough to halve the block launches and keep a copy in flight.  Larger
    // sibships are less bandwidth-bound and like 8 (quads 0.72 -> 0.82, three children 0.67 -> 0.75).  Small batches get shorter
    // lists, down to the one-tile-per-block arrangement.
    const int64_t n_tiles = (B.V + TB - 1) / TB, resident = (int64_t)n_sm * per_sm;
    const int list_len = (int)std::max<int64_t>(1, std::min<int64_t>(P.stream_tiles > 0 ? P.stream_tiles : (NC == 1 ? 4 : 8), n_tiles / (2 * resident)));
    const unsigned grid = (unsigned)((n_tiles + list_len - 1) / list_len);
    kernel<<<grid, TB, smem, stream>>>(P, B, list_len);
    return cudaGetLastError();
}

template <int NC, int TB, bool PL, bool SINGLE, bool IDENT, int MINB>
cudaError_t launch_minb(const NuclearParams &P, const BatchPtrs &B, cudaStream_t stream) {
    const size_t S = (size_t)P.C.s;
    const size_t in_bytes = (TB * S * 3 * (PL ? sizeof(uint16_t) : sizeof(double)) + 15) & ~(size_t)15;
    const size_t smem = (SINGLE ? 2 : 1) * TB * S * 3 * sizeof(double) + in_bytes + ((TB * S + 15) & ~(size_t)15) + TB;
    cudaError_t rc = cudaFuncSetAttribute(es_nuclear_kernel<NC, TB, PL, SINGLE, IDENT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc != cudaSuccess) return rc;
    const unsigned grid = (unsigned)((B.V + TB - 1) / TB);
    es_nuclear_kernel<NC, TB, PL, SINGLE, IDENT, MINB><<<grid, TB, smem, stream>>>(P, B);
    return cudaGetLastError();
}

// Register budget per sibship size (one warp per block).  More resident warps beat more registers as long as nothing spills
// (profiles/r2n_nuclear.log, r2o_nuclear.log; fraction of the canonical HBM roofline): quads 0.60 -> 0.91 with 16 blocks per
// SM (128 registers) instead of the compiler's 138 registers, three children 0.69 -> 0.87 with 12 blocks (168 registers), four
// children 0.75 -> 0.80 with 12 blocks; five children keep the compiler's choice (248 registers, 0.78; 10 blocks spill: 0.56).
template <int NC, int TB, bool PL, bool SINGLE, bool IDENT> cudaError_t launch_ident(const NuclearParams &P, const BatchPtrs &B, cudaStream_t stream) {
    constexpr int kMinBlocks = NC == 1 ? 896 / TB : (NC == 2 ? 16 : (NC <= 4 ? 12 : 0));
    // (the flags ride on the tile's TMA transaction: 16-byte alignment, like every other array)
    if (PL && TB == 32 && P.stream_tiles >= 0 && (reinterpret_cast<uintptr_t>(B.flags) & 15u) == 0) return launch_stream<NC, SINGLE, IDENT, kMinBlocks>(P, B, stream);
    return launch_minb<NC, TB, PL, SINGLE, IDENT, kMinBlocks>(P, B, stream);
}

template <int NC, int TB, bool PL, bool SINGLE> cudaError_t launch_io(const NuclearParams &P, const BatchPtrs &B, cudaStream_t stream) {
    bool ident = P.allow_ident && P.C.s == NC + 2 && P.col_father == 0 && P.col_mother == 1;
    for (int c = 0; c < NC; c++) ident = ident && P.col_child[c] == 2 + c;
    // The specialisation for the identity column map (headline tile size only: compile time) saves ~120 of ~800 instructions per
    // trio variant, at the price of a few spilled registers under the 72-register cap.  Measured (profiles/r2j): compact input
    // 0.334 -> 0.317 ms (post + single), 0.282 -> 0.257 ms (post only) per 10 M trio variants; quads 0.53 -> 0.60, three-child
    // sibships 0.61 -> 0.69 of the HBM roofline; but the FP64-input trio kernel, which is HBM-bound, loses (0.345 -> 0.350 ms),
    // so that one keeps the general code.
    if (ident && TB == 32 && (PL || NC > 1)) return launch_ident<NC, 32, PL, SINGLE, true>(P, B, stream);
    return launch_ident<NC, TB, PL, SINGLE, false>(P, B, stream);
}

template <int NC, int TB> cudaError_t launch_nc(const NuclearParams &P, const BatchPtrs &B, cudaStream_t stream) {
    if (B.pl) return B.single ? launch_io<NC, TB, true, true>(P, B, stream) : launch_io<NC, TB, true, false>(P, B, stream);
    return B.single ? launch_io<NC, TB, false, true>(P, B, stream) : launch_io<NC, TB, false, false>(P, B, stream);
}

} // namespace

} // namespace famseq
