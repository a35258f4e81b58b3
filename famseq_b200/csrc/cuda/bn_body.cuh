// bn_body.cuh -- the Bayesian-network kernel body, shared by bn_kernel (one pedigree, bn_kernel.cu) and bn_cohort_kernel
// (one family of a cohort ped file per block, bn_cohort_kernel.cu).
//
// bn_body<U, INDEP, FACTOR, COHORT> is bn_kernel's body.  Both kernels run its factor-table layout, enumeration, group
// reduction and normalisation, so a family enumerated by bn_cohort_kernel gets the bits fs_create BN gives that family
// alone.  COHORT switches, at compile time only, what differs:
//   * where the plan lives: the kernel parameter (BnParams), or the block's family's plan staged in shared memory;
//   * the head of each tile: bn_kernel's individual-only posteriors and LRC gate, or the status es_cohort_head_kernel
//     left (2: enumerate), and factor tables gathered through the family's column map (PL input decoded on the way);
//   * the end of each tile: bn_kernel's whole-row writes, or the family's members written at their global columns, a bin
//     sum <= 0 storing status 3.
// bn_kernel's instantiations (COHORT false) compile to the same SASS as the kernel written out in full did: the cohort
// code is discarded by `if constexpr`, and the body is the kernel's own text.  Both kernels compile it with the default
// -fmad=true.
#pragma once

#include "common.cuh"
#include "kernels.hpp"

namespace famseq {

namespace {

// bn_cohort_kernel's parameters: one launch class (kernels.hpp).  C.s is 0 (the body keeps no per-column state); s_row is
// the row's column count.
struct BnCohortLaunch {
    RunConstants C;
    const BnPlan *plans;
    const int32_t *fam_plan, *fam_col_off, *cols;
    int32_t begin, n_fam; // the class's families in device order
    int32_t s_row;
};

__device__ __forceinline__ int bn_row(uint64_t cfg, int sh_m, int sh_f) {
    return 3 * (int)((cfg >> sh_m) & 3u) + (int)((cfg >> sh_f) & 3u);
}

// Fully unrolled enumeration of the innermost U levels.  `off[x]` is the offset (in doubles) of the
// table row of unrolled level x given every digit chosen so far; returns the sum of the joints of the
// 3^(U-X) configurations below and adds them to the register bins acc[x][digit].
template <int X, int U> struct BnBlock {
    static __device__ __forceinline__ double run(const double *__restrict__ tab,
                                                 const int (&stride)[BN_MAX_UNROLL][BN_MAX_UNROLL],
                                                 const int (&off)[U], double prefix, double (&acc)[U][3]) {
        const double2 f01 = *reinterpret_cast<const double2 *>(tab + off[X]);
        if constexpr (X == U - 1) {
            // innermost level: each joint prefix*f[d] is formed inside the FMA that adds it to the member's bin; the
            // sum of the three joints is prefix * (f0+f1+f2), the row sum being tabulated next to the row
            const double2 f2s = *reinterpret_cast<const double2 *>(tab + off[X] + 2);
            acc[X][0] = fma(prefix, f01.x, acc[X][0]);
            acc[X][1] = fma(prefix, f01.y, acc[X][1]);
            acc[X][2] = fma(prefix, f2s.x, acc[X][2]);
            return prefix * f2s.y;
        }
        const double f2 = tab[off[X] + 2];
        double total = 0.0;
#pragma unroll
        for (int d = 0; d < 3; d++) {
            const double joint = prefix * (d == 0 ? f01.x : (d == 1 ? f01.y : f2));
            double below;
            if constexpr (X == U - 1) {
                below = joint;
            } else {
                int off2[U];
#pragma unroll
                for (int x = 0; x < U; x++) off2[x] = (x > X) ? off[x] + d * stride[x][X] : off[x];
                below = BnBlock<X + 1, U>::run(tab, stride, off2, joint, acc);
            }
            acc[X][d] += below;
            total = (d == 0) ? below : total + below;
        }
        return total;
    }
};

// The same enumeration when no unrolled level is the parent of another one (host/bn_plan.cpp puts childless
// members innermost, so this is the common case): the U factor vectors depend on outer digits only, are loaded
// once per block and the whole 3^U nest runs out of registers.
template <int X, int U> struct BnBlockRegs {
    // `inner` are the bins of the innermost level, one set per digit of the level above it: three times shorter
    // dependent FMA chains than a single set (they are summed once, after the enumeration)
    static __device__ __forceinline__ double run(const double (&f)[U][4], double prefix, double (&acc)[U][3],
                                                 double (&inner)[3][3], int above) {
        if constexpr (X == U - 1) { // see BnBlock: joints formed inside the FMAs, their sum is prefix * row sum
            inner[above][0] = fma(prefix, f[X][0], inner[above][0]);
            inner[above][1] = fma(prefix, f[X][1], inner[above][1]);
            inner[above][2] = fma(prefix, f[X][2], inner[above][2]);
            return prefix * f[X][3];
        } else {
            double total = 0.0;
#pragma unroll
            for (int d = 0; d < 3; d++) {
                const double joint = prefix * f[X][d];
                const double below = BnBlockRegs<X + 1, U>::run(f, joint, acc, inner, d);
                acc[X][d] += below;
                total = (d == 0) ? below : total + below;
            }
            return total;
        }
    }
};

// Opt-in (FAMSEQ_BN_FACTOR=1), INDEP only: the U innermost members are childless and their factor rows depend on outer
// digits only, so the sum over their 3^U configurations factorises:
//   bin[x][g] += prefix * f_x[g] * prod_{y != x} rowsum_y,      block total = prefix * prod_x rowsum_x
// -- 6U FP64 operations per block instead of ~2.5 * 3^U.  Same marginals up to summation order; the 3^U configurations
// of the block are then summed analytically instead of being visited, which is why it is not the default: the
// contract of this method (and its roofline accounting) is the exhaustive enumeration.
template <int U>
__device__ __forceinline__ double bn_block_factored(const double (&f)[U][4], double prefix, double (&acc)[U][3]) {
    double pre[U + 1];
    pre[0] = prefix;
#pragma unroll
    for (int x = 0; x < U; x++) pre[x + 1] = pre[x] * f[x][3];
    double suf = 1.0;
#pragma unroll
    for (int x = U - 1; x >= 0; x--) {
        const double w = pre[x] * suf; // prefix * row sums of every other unrolled member
        acc[x][0] = fma(w, f[x][0], acc[x][0]);
        acc[x][1] = fma(w, f[x][1], acc[x][1]);
        acc[x][2] = fma(w, f[x][2], acc[x][2]);
        suf *= f[x][3];
    }
    return pre[U];
}

__device__ __forceinline__ const BnPlan &bn_plan_of(const BnParams &P) { return P.plan; }

// The block's family: blockIdx.y + gridDim.y * blockIdx.z of the class.
__device__ __forceinline__ int bn_family(const BnCohortLaunch &) { return (int)(blockIdx.y + gridDim.y * blockIdx.z); }

// The block's family's plan, staged in shared memory (read once per block).
__device__ __forceinline__ const BnPlan &bn_plan_of(const BnCohortLaunch &P) {
    __shared__ int s_plan[sizeof(BnPlan) / sizeof(int)]; // raw words: BnPlan's member initialisers have no place in shared memory
    const int *src = reinterpret_cast<const int *>(P.plans + __ldg(P.fam_plan + P.begin + bn_family(P)));
    for (int k = threadIdx.x; k < (int)(sizeof(BnPlan) / sizeof(int)); k += blockDim.x) s_plan[k] = __ldg(src + k);
    __syncthreads();
    return *reinterpret_cast<const BnPlan *>(s_plan);
}

// bn_kernel's factor table of variant v, from the family's columns of the row (one table row per thread of the group).
__device__ __forceinline__ void bn_cohort_tables(const BnCohortLaunch &P, const BatchPtrs &B, const BnPlan &pl, double *tab,
                                                 bool active, int64_t v, bool chrx, const VariantPriors &pr, int code, int G) {
    if (!active) return;
    const RunConstants &C = P.C;
    const int32_t *cmap = P.cols + __ldg(P.fam_col_off + P.begin + bn_family(P)); // local -> global input column
    const int n_rows = pl.table_doubles >> 2;
    for (int q = code; q < n_rows; q += G) {
        const int L = pl.row_level[q], row = q - (pl.tab_off[L] >> 2);
        const bool founder = pl.founder[L] != 0, male = pl.male[L] != 0;
        const int col = pl.col[L];
        const int64_t at = v * 3 * (int64_t)P.s_row + (col >= 0 ? (int64_t)__ldg(cmap + col) * 3 : 0);
        const int kind = chrx ? (male ? K_TAB_XM : K_TAB_XF) : K_TAB_AUTO;
        double f[3];
#pragma unroll
        for (int g = 0; g < 3; g++) {
            const double lk = col < 0 ? 1.0 : (B.pl ? __ldg(B.lut + B.pl[at + g]) : __ldg(B.lk + at + g));
            const double base = founder ? (male ? pr.m[g] : pr.a[g]) : C.tab[kind][g * 9 + row];
            f[g] = __dmul_rn(base, lk); // the reference's indProb (family.cpp:899-909)
        }
        *reinterpret_cast<double2 *>(tab + 4 * q) = make_double2(f[0], f[1]);
        *reinterpret_cast<double2 *>(tab + 4 * q + 2) = make_double2(f[2], __dadd_rn(__dadd_rn(f[0], f[1]), f[2]));
    }
}

// The family's members of variant v normalised and called at their global columns, as bn_kernel writes them; a bin sum
// <= 0 fails the variant: status := 3, a plain store of a constant, so the blocks of the other families that share the
// variant cannot lose it (es_cohort_finish_kernel then writes the NA rows).
__device__ __forceinline__ void bn_cohort_write(const BnCohortLaunch &P, const BatchPtrs &B, const BnPlan &pl, const double *bins,
                                                bool active, int64_t v, int code, int G) {
    if (!active) return;
    const int32_t *cmap = P.cols + __ldg(P.fam_col_off + P.begin + bn_family(P));
    const int64_t S = P.s_row;
    for (int L = code; L < pl.n_levels; L += G) {
        const double b0 = bins[L * 3], b1 = bins[L * 3 + 1], b2 = bins[L * 3 + 2];
        const double sum = __dadd_rn(__dadd_rn(b0, b1), b2);
        if (sum <= 0.0) {
            B.status[v] = 3;
            continue;
        }
        const int c = pl.col[L];
        if (c < 0) continue;
        const int64_t gc = __ldg(cmap + c);
        const double p0 = b0 / sum, p1 = b1 / sum, p2 = b2 / sum;
        double *gp = B.post + (v * S + gc) * 3;
        gp[0] = p0;
        gp[1] = p1;
        gp[2] = p2;
        B.gt[v * S + gc] = call_genotype(p0, p1, p2);
    }
}

template <int U, bool INDEP, bool FACTOR, bool COHORT, class Params>
__device__ __forceinline__ void bn_body(const Params &P, const BatchPtrs &B, int n_tiles) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const RunConstants &C = P.C;
    if constexpr (COHORT)
        if (bn_family(P) >= P.n_fam) return;
    const BnPlan &pl = bn_plan_of(P);
    const int N = pl.n_levels, G = pl.group, VPB = pl.vpb, R = pl.r, H = pl.h, S = C.s;
    const int TD = pl.table_doubles;
    const int nthreads = blockDim.x;
    double *s_tab = reinterpret_cast<double *>(smem_raw);  // [VPB][TD] factor tables, rows of 4 doubles
    double *s_bins = s_tab + VPB * TD;                      // [VPB][N][3] marginal sums
    double *s_priv = s_bins + VPB * N * 3;                  // [R][5][nthreads]: prefix, 3 bins, pending mass of a rolled level
    double *s_red = s_priv + R * 5 * nthreads;              // [3U+1][nthreads]: unrolled bins, thread total
    double *s_single = s_red + (3 * U + 1) * nthreads;      // [VPB][S][3]
    int *s_state = reinterpret_cast<int *>(s_single + VPB * S * 3); // [VPB] bit 0: the pedigree is needed, bit 1: failed

    const int tid = threadIdx.x;
    const int slot = tid / G, code = tid - slot * G;
    const int first_unrolled = N - U;

    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t v = (int64_t)tile * VPB + slot;
        const bool live = slot < VPB && v < B.V;
        const unsigned flag = (live && B.flags) ? B.flags[v] : 0u;
        const bool chrx = (flag >> 1) & 1u;
        const VariantPriors pr = select_priors(C, flag);
        const double *lkv = B.lk + v * S * 3;

        if constexpr (COHORT) { // the head kernel did the column pass: enumerate the variants it left with status 2
            if (live && code == 0) s_state[slot] = B.status[v] == 2 ? 1 : 2;
            if (!__syncthreads_or(live && s_state[slot] == 1)) continue;
            bn_cohort_tables(P, B, pl, s_tab + slot * TD, live && s_state[slot] == 1, v, chrx, pr, code, G);
            __syncthreads();
        } else {
            // ---- individual-only posterior + LRC gate (family.cpp:1405-1499, :767-789) ------------------
            // one input column per thread of the variant's group; the verdicts meet in s_state (bit 0: some sample wants
            // the pedigree, bit 1: failed)
            if (live && code == 0) s_state[slot] = C.unseq_fail[flag & 3u] != 0 ? 2 : 0;
            __syncthreads();
            if (live) {
                int verdict = 0;
                for (int c = code; c < S; c += G) {
                    const double l0 = lkv[c * 3], l1 = lkv[c * 3 + 1], l2 = lkv[c * 3 + 2];
                    const bool male = C.col_male[c] != 0;
                    const double r0 = l0 * (male ? pr.m[0] : pr.a[0]);
                    const double r1 = l1 * (male ? pr.m[1] : pr.a[1]);
                    const double r2 = l2 * (male ? pr.m[2] : pr.a[2]);
                    const double rs = __dadd_rn(__dadd_rn(r0, r1), r2);
                    if (rs <= 0.0) verdict |= 2;
                    double *sg = s_single + (slot * S + c) * 3;
                    sg[0] = r0 / rs;
                    sg[1] = r1 / rs;
                    sg[2] = r2 / rs;
                    double big = 0.0;
                    if (big < l0) big = l0;
                    if (big < l1) big = l1;
                    if (big < l2) big = l2;
                    const double ls = __dadd_rn(__dadd_rn(l0, l1), l2);
                    if (big / ls < C.lrc) verdict |= 1;
                }
                if (verdict) atomicOr(&s_state[slot], verdict);
        }
        // ---- per-variant factor tables ---------------------------------------------------------------
        if (live) { // one table row (3 factors and their sum) per thread
            double *tab = s_tab + slot * TD;
            const int n_rows = TD >> 2;
            for (int q = code; q < n_rows; q += G) {
                const int L = pl.row_level[q], row = q - (pl.tab_off[L] >> 2);
                const bool founder = pl.founder[L] != 0, male = pl.male[L] != 0;
                const int col = pl.col[L];
                const int kind = chrx ? (male ? K_TAB_XM : K_TAB_XF) : K_TAB_AUTO;
                double f[3];
#pragma unroll
                for (int g = 0; g < 3; g++) {
                    const double lk = col >= 0 ? lkv[col * 3 + g] : 1.0;
                    const double base = founder ? (male ? pr.m[g] : pr.a[g]) : C.tab[kind][g * 9 + row];
                    f[g] = __dmul_rn(base, lk); // the reference's indProb (family.cpp:899-909)
                }
                *reinterpret_cast<double2 *>(tab + 4 * q) = make_double2(f[0], f[1]);
                *reinterpret_cast<double2 *>(tab + 4 * q + 2) = make_double2(f[2], __dadd_rn(__dadd_rn(f[0], f[1]), f[2]));
            }
        }
        __syncthreads();

        }
        // ---- enumeration -------------------------------------------------------------------------------
        double acc[U][3];
#pragma unroll
        for (int x = 0; x < U; x++) acc[x][0] = acc[x][1] = acc[x][2] = 0.0;
        double thread_total = 0.0;
        double inner[3][3]; // INDEP only: split bins of the innermost level
#pragma unroll
        for (int k = 0; k < 3; k++) inner[k][0] = inner[k][1] = inner[k][2] = 0.0;
        if (live && s_state[slot] == 1) { // pedigree needed and nothing failed
            const double *tab = s_tab + slot * TD;
            uint64_t cfg = 0;
            { // this thread's digits of the spread levels
                int c = code;
                for (int j = 0; j < H; j++) {
                    const int d = c % 3;
                    c /= 3;
                    cfg |= (uint64_t)d << (2 * j);
                }
            }
            double prefix = 10000000.0; // the reference's pre-scale, family.cpp:911
            for (int j = 0; j < H; j++)
                prefix *= tab[pl.tab_off[j] + 4 * bn_row(cfg, pl.sh_m[j], pl.sh_f[j]) + (int)((cfg >> (2 * j)) & 3u)];
            const double spread_prefix = prefix;
            // rolled levels start at digit 0; private state per rolled level: prefix, 3 bins, pending mass
            for (int q = 0; q < R; q++) {
                const int L = H + q;
                prefix *= tab[pl.tab_off[L] + 4 * bn_row(cfg, pl.sh_m[L], pl.sh_f[L])];
                double *pv = s_priv + (q * 5) * nthreads + tid;
                pv[0] = prefix;
                pv[nthreads] = pv[2 * nthreads] = pv[3 * nthreads] = pv[4 * nthreads] = 0.0;
            }
            int off[U];
            double f[INDEP ? U : 1][4];
            bool reload = true; // the unrolled levels' table rows depend on outer digits only
            for (;;) {
                if (reload) {
#pragma unroll
                    for (int x = 0; x < U; x++) {
                        const int L = first_unrolled + x;
                        off[x] = pl.tab_off[L] + 4 * bn_row(cfg, pl.sh_m[L], pl.sh_f[L]);
                    }
                    if constexpr (INDEP) {
#pragma unroll
                        for (int x = 0; x < U; x++) {
                            const double2 f01 = *reinterpret_cast<const double2 *>(tab + off[x]);
                            const double2 f2s = *reinterpret_cast<const double2 *>(tab + off[x] + 2);
                            f[x][0] = f01.x;
                            f[x][1] = f01.y;
                            f[x][2] = f2s.x;
                            f[x][3] = f2s.y;
                        }
                    }
                }
                double block_total;
                if constexpr (INDEP && FACTOR)
                    block_total = bn_block_factored<U>(f, prefix, acc);
                else if constexpr (INDEP)
                    block_total = BnBlockRegs<0, U>::run(f, prefix, acc, inner, 0);
                else
                    block_total = BnBlock<0, U>::run(tab, pl.ustride, off, prefix, acc);
                thread_total += block_total;
                if (R == 0) break;
                // Advance the odometer (innermost rolled level fastest) and book the block's mass into the bins of the
                // rolled levels hierarchically: a level's bin is touched only when its digit changes; what was
                // accumulated under an unchanged digit waits in the level's `pending` slot.
                double mass = block_total;
                int k = R - 1;
                bool finished = false;
                for (;;) {
                    const int L = H + k;
                    const int d = (int)((cfg >> (2 * L)) & 3u);
                    s_priv[(k * 5 + 1 + d) * nthreads + tid] += mass;
                    if (d < 2) {
                        cfg += 1ull << (2 * L);
                        if (k > 0) s_priv[((k - 1) * 5 + 4) * nthreads + tid] += mass;
                        break;
                    }
                    cfg &= ~(3ull << (2 * L));
                    if (k == 0) {
                        finished = true;
                        break;
                    }
                    k--;
                    mass += s_priv[(k * 5 + 4) * nthreads + tid];
                    s_priv[(k * 5 + 4) * nthreads + tid] = 0.0;
                }
                if (finished) break; // every rolled digit wrapped: done
                // levels k .. R-1 changed: rebuild their prefixes
                prefix = (k == 0) ? spread_prefix : s_priv[((k - 1) * 5) * nthreads + tid];
                for (int j = k; j < R; j++) {
                    const int L = H + j;
                    prefix *= tab[pl.tab_off[L] + 4 * bn_row(cfg, pl.sh_m[L], pl.sh_f[L]) + (int)((cfg >> (2 * L)) & 3u)];
                    s_priv[(j * 5) * nthreads + tid] = prefix;
                }
                reload = k <= pl.unrolled_dep;
            }
        } else {
                for (int q = 0; q < R; q++)
                    for (int k = 1; k < 4; k++) s_priv[(q * 5 + k) * nthreads + tid] = 0.0;
        }
        if constexpr (INDEP && !FACTOR) {
#pragma unroll
            for (int g = 0; g < 3; g++) acc[U - 1][g] = (inner[0][g] + inner[1][g]) + inner[2][g];
        }
#pragma unroll
        for (int x = 0; x < U; x++)
#pragma unroll
            for (int g = 0; g < 3; g++) s_red[(x * 3 + g) * nthreads + tid] = acc[x][g];
        s_red[(3 * U) * nthreads + tid] = thread_total;
        __syncthreads();

        // ---- sum the group's partial bins (fixed order) ------------------------------------------------
        {
            const int n_bins = VPB * N * 3;
            auto partial = [&](int bin, int c) -> double { // contribution of thread `c` of the group to `bin`
                const int sl = bin / (N * 3), rem = bin - sl * N * 3;
                const int L = rem / 3, g = rem - 3 * L;
                const int t = sl * G + c;
                if (L < H) {
                    int cc = c;
                    for (int j = 0; j < L; j++) cc /= 3;
                    return (cc % 3 == g) ? s_red[(3 * U) * nthreads + t] : 0.0;
                }
                if (L < H + R) return s_priv[((L - H) * 5 + 1 + g) * nthreads + t];
                return s_red[((L - first_unrolled) * 3 + g) * nthreads + t];
            };
            if (G >= 32) {
                const int lane = tid & 31, warp = tid >> 5, n_warps = nthreads >> 5;
                for (int bin = warp; bin < n_bins; bin += n_warps) {
                    double sum = 0.0;
                    for (int c = lane; c < G; c += 32) sum += partial(bin, c);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
                    if (lane == 0) s_bins[bin] = sum;
                }
            } else {
                for (int bin = tid; bin < n_bins; bin += nthreads) {
                    double sum = 0.0;
                    for (int c = 0; c < G; c++) sum += partial(bin, c);
                    s_bins[bin] = sum;
                }
            }
        }
        __syncthreads();

        if constexpr (COHORT) {
            bn_cohort_write(P, B, pl, s_bins + slot * N * 3, live && s_state[slot] == 1, v, code, G);
        } else {
            // ---- normalise, call, write (family.cpp:943-954, :576-665): one member / one column per thread -------------
            const bool enumerated = live && s_state[slot] == 1;
            if (enumerated) {
                const double *bins = s_bins + slot * N * 3;
                bool bad = false;
                for (int L = code; L < N; L += G)
                    if (__dadd_rn(__dadd_rn(bins[L * 3], bins[L * 3 + 1]), bins[L * 3 + 2]) <= 0.0) bad = true;
                if (bad) atomicOr(&s_state[slot], 2);
        }
        __syncthreads();
        if (live) {
            const int state = s_state[slot];
            const bool failed = (state & 2) != 0;
            double *gp = B.post + v * S * 3, *gs = B.single + v * S * 3;
            uint8_t *gg = B.gt + v * S;
            const double *sg = s_single + slot * S * 3;
            for (int c = code; c < S; c += G) { // GPP rows, and the FPP rows when the pedigree was not used
                const double q0 = failed ? 0.0 : sg[c * 3], q1 = failed ? 0.0 : sg[c * 3 + 1], q2 = failed ? 0.0 : sg[c * 3 + 2];
                gs[c * 3] = q0;
                gs[c * 3 + 1] = q1;
                gs[c * 3 + 2] = q2;
                if (failed || state == 0) {
                    gp[c * 3] = q0;
                    gp[c * 3 + 1] = q1;
                    gp[c * 3 + 2] = q2;
                    gg[c] = failed ? (uint8_t)255 : call_genotype(q0, q1, q2);
                }
            }
            if (!failed && state == 1) {
                const double *bins = s_bins + slot * N * 3;
                for (int L = code; L < N; L += G) {
                    const int c = pl.col[L];
                    if (c < 0) continue;
                    const double b0 = bins[L * 3], b1 = bins[L * 3 + 1], b2 = bins[L * 3 + 2];
                    const double sum = __dadd_rn(__dadd_rn(b0, b1), b2);
                    const double p0 = b0 / sum, p1 = b1 / sum, p2 = b2 / sum;
                    gp[c * 3] = p0;
                    gp[c * 3 + 1] = p1;
                    gp[c * 3 + 2] = p2;
                    gg[c] = call_genotype(p0, p1, p2);
                }
            }
            if (code == 0) B.status[v] = failed ? 1 : 0;
        }
        }
        __syncthreads();
    }
}


} // namespace

} // namespace famseq
