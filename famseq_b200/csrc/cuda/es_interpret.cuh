// es_interpret.cuh -- the Elston-Stewart message-program interpreter (host/es_program.hpp), one variant per thread in lock
// step, operands in a per-variant vector file in shared memory.  Shared by es_kernel.cu (one pedigree) and
// es_cohort_kernel.cu (one family program per block).  Compile with -fmad=false: every product is formed in the
// reference's association order, so the FP64 results are bit-identical to the reference CPU build.
#pragma once

#include "common.cuh"
#include "../host/es_program.hpp"

namespace famseq {

// Transmission table entry T[g][a][b] (child g | mother a, father b): table `sel` on chrX, the autosome table otherwise.
template <bool X> __device__ __forceinline__ double es_trans(const RunConstants &C, int sel, int g, int a, int b) {
    return X ? C.tab[sel][g * 9 + a * 3 + b] : C.tab[0][g * 9 + a * 3 + b];
}

// Per-variant vector file in shared memory (operand encoding of host/es_program.hpp): vector u, component g of this
// thread's variant is vec[(u * 3 + g) * (TB + 1)].  The odd row stride keeps both the transposing tile copy and the
// per-thread accesses free of bank conflicts.
template <int TB> struct EsThread {
    double *vec;
    VariantPriors pr;

    __device__ __forceinline__ void load(uint32_t u, double v[3]) const {
#pragma unroll
        for (int g = 0; g < 3; g++) v[g] = vec[(u * 3 + g) * (TB + 1)];
    }
    __device__ __forceinline__ void store(uint32_t u, const double v[3]) const {
#pragma unroll
        for (int g = 0; g < 3; g++) vec[(u * 3 + g) * (TB + 1)] = v[g];
    }
};

// Interprets the message program for one variant.  Returns true when a member's row sum was exactly
// zero (the reference returns false there, family.cpp:1305-1310).  `prog.word(pc)` is word pc of the program and
// `prog.col(c)` the output column of its input column c: the kernel parameters and the identity for es_kernel, a family's
// program and column map in global memory for the cohort kernel (es_cohort_kernel.cu).
// ACC: the conditioned program of bn_peel_kernel.cu, whose ES_OP_ACC stores (acc_first) or adds each member's
// unnormalised marginal into its accumulator; it exists only in that instantiation.
template <bool X, int TB, class Program, bool ACC = false>
__device__ bool es_interpret(const RunConstants &C, const Program &prog, const EsThread<TB> &t, double *post_row, uint8_t *gt_row,
                             bool acc_first = true) {
    bool failed = false;
    int pc = 0;
    for (;;) {
        const uint32_t w0 = prog.word(pc);
        const uint32_t op = w0 & 0xffu;
        if (op == ES_OP_END) break;
        if constexpr (ACC) {
            if (op == ES_OP_ACC) {
                const uint32_t w1 = prog.word(pc + 1), w2 = prog.word(pc + 2), acc = (w0 >> 8) & 0xffffu;
                double m[3], l[3], a[3];
                t.load(w1 & 0xffffu, m);
                t.load(w1 >> 16, l);
                t.load(w2 & 0xffffu, a);
#pragma unroll
                for (int g = 0; g < 3; g++) m[g] = (m[g] * l[g]) * a[g];
                if (!acc_first) { // never 0.0 + v on the first peel: it would turn a -0.0 into +0.0
                    double s[3];
                    t.load(acc, s);
#pragma unroll
                    for (int g = 0; g < 3; g++) m[g] = s[g] + m[g];
                }
                t.store(acc, m);
                pc += 3;
                continue;
            }
        }
        if (op == ES_OP_MUL) {
            const uint32_t w1 = prog.word(pc + 1);
            double a[3], b[3];
            t.load(w1 & 0xffffu, a);
            t.load(w1 >> 16, b);
#pragma unroll
            for (int g = 0; g < 3; g++) a[g] = a[g] * b[g];
            t.store((w0 >> 8) & 0xffffu, a);
            pc += 2;
        } else if (op == ES_OP_ANT) {
            const uint32_t w1 = prog.word(pc + 1);
            const int nsib = w0 >> 25;
            const int sel_c = ((w0 >> 24) & 1u) ? K_TAB_XM : K_TAB_XF;
            double wm[3], wf[3], sibs[3][3];
            t.load(w1 & 0xffffu, wm);
            t.load(w1 >> 16, wf);
            for (int k = 0; k < nsib; k++) {
                const uint32_t wk = prog.word(pc + 2 + k);
                const int sel_k = ((wk >> 16) & 1u) ? K_TAB_XM : K_TAB_XF;
                double d[3];
                t.load(wk & 0xffffu, d);
#pragma unroll
                for (int a = 0; a < 3; a++)
#pragma unroll
                    for (int b = 0; b < 3; b++) {
                        double sc = d[0] * es_trans<X>(C, sel_k, 0, a, b);
                        sc = sc + d[1] * es_trans<X>(C, sel_k, 1, a, b);
                        sc = sc + d[2] * es_trans<X>(C, sel_k, 2, a, b);
                        sibs[a][b] = (k == 0) ? sc : sibs[a][b] * sc;
                    }
            }
            double out[3];
#pragma unroll
            for (int g = 0; g < 3; g++) {
                double over_m = 0.0;
#pragma unroll
                for (int a = 0; a < 3; a++) {
                    double over_f = 0.0;
#pragma unroll
                    for (int b = 0; b < 3; b++) {
                        double term = wf[b] * es_trans<X>(C, sel_c, g, a, b);
                        if (nsib) term = term * sibs[a][b];
                        over_f = over_f + term;
                    }
                    over_m = over_m + wm[a] * over_f;
                }
                out[g] = over_m;
            }
            t.store((w0 >> 8) & 0xffffu, out);
            pc += 2 + nsib;
        } else if (op == ES_OP_POS) {
            const uint32_t w1 = prog.word(pc + 1);
            const int nkid = w0 >> 25;
            // autosome: table index is (g_i, g_j) whatever the sexes (family.cpp:1836);
            // chrX: (mother, father), so a male i goes second (family.cpp:1900-1921)
            const bool i_second = X && ((w0 >> 24) & 1u);
            double wj[3], kids[3][3];
            t.load(w1 & 0xffffu, wj);
            for (int k = 0; k < nkid; k++) {
                const uint32_t wk = prog.word(pc + 2 + 2 * k);
                const int sel_k = (prog.word(pc + 3 + 2 * k) & 1u) ? K_TAB_XM : K_TAB_XF;
                double lkc[3], mc[3];
                t.load(wk & 0xffffu, lkc);
                t.load(wk >> 16, mc);
#pragma unroll
                for (int g = 0; g < 3; g++)
#pragma unroll
                    for (int b = 0; b < 3; b++) {
                        double sc = 0.0;
#pragma unroll
                        for (int l = 0; l < 3; l++) {
                            const double tr = i_second ? es_trans<X>(C, sel_k, l, b, g) : es_trans<X>(C, sel_k, l, g, b);
                            const double term = (tr * lkc[l]) * mc[l];
                            sc = (l == 0) ? term : sc + term;
                        }
                        kids[g][b] = (k == 0) ? sc : kids[g][b] * sc;
                    }
            }
            double out[3];
#pragma unroll
            for (int g = 0; g < 3; g++) {
                double over_j = wj[0] * kids[g][0];
                over_j = over_j + wj[1] * kids[g][1];
                over_j = over_j + wj[2] * kids[g][2];
                out[g] = over_j;
            }
            t.store((w0 >> 8) & 0xffffu, out);
            pc += 2 + 2 * nkid;
        } else { // ES_OP_FIN
            const uint32_t w1 = prog.word(pc + 1), w2 = prog.word(pc + 2);
            double m[3], l[3], a[3];
            t.load(w1 & 0xffffu, m);
            t.load(w1 >> 16, l);
            t.load(w2 & 0xffffu, a);
#pragma unroll
            for (int g = 0; g < 3; g++) m[g] = (m[g] * l[g]) * a[g];
            const double sum = (m[0] + m[1]) + m[2];
            if (sum == 0.0) failed = true;
            if ((w0 >> 8) & 1u) {
                const int col = prog.col(w0 >> 9);
                double q0, q1, q2;
                div3(m[0], m[1], m[2], sum, q0, q1, q2);
                post_row[col * 3] = q0;
                post_row[col * 3 + 1] = q1;
                post_row[col * 3 + 2] = q2;
                gt_row[col] = call_genotype(q0, q1, q2); // get_postRlt (family.cpp:636-665), from registers
            }
            pc += 3;
        }
    }
    return failed;
}

} // namespace famseq
