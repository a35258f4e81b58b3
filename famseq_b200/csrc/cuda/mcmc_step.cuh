// mcmc_step.cuh -- the single-site Gibbs step shared by the table-driven sampler of one pedigree (mcmc_kernel.cu) and the
// sampler of cohort ped files (mcmc_cohort_kernel.cu): the genotype vector, the Philox generator, the full conditional on
// the replicated transmission tables, the draw and the reciprocal of the Rao-Blackwell weights.  Both kernels run the same
// arithmetic in the same order, so a family's chain in the cohort kernel is bit for bit that family's part of the
// whole-file chain.
#pragma once

#include "common.cuh"

namespace famseq {

namespace {

constexpr int kCopies = 16;      // replicas of every table entry
constexpr int kEntries = 81 + 27; // 3 x 27 transmission entries followed by 27 ones
constexpr int kOnes = 81;

__device__ __forceinline__ double lds64(uint32_t shared_addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(shared_addr));
    return v;
}

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                              uint32_t &o0, uint32_t &o1, uint32_t &o2, uint32_t &o3) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0;
        c1 = lo1;
        c2 = n2;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    o0 = c0;
    o1 = c1;
    o2 = c2;
    o3 = c3;
}

// genotype vector, 2 bits per member in GW 64-bit words (GW = 1: up to 32 members, GW = 2: up to 64, GW = 4: up to 128);
// the member index is warp-uniform
template <int GW> struct Genotypes {
    uint64_t w[GW];
    __device__ __forceinline__ uint64_t word(int i) const {
        if (GW == 1) return w[0];
        if (GW == 2) return i < 32 ? w[0] : w[1];
        return i < 64 ? (i < 32 ? w[0] : w[1]) : (i < 96 ? w[2] : w[GW - 1]);
    }
    __device__ __forceinline__ int get(int i) const { return (int)((word(i) >> (2 * (i & 31))) & 3u); }
    __device__ __forceinline__ void set(int i, int g) {
        const uint64_t m = 3ull << (2 * (i & 31)), v = (uint64_t)g << (2 * (i & 31));
#pragma unroll
        for (int k = 0; k < GW; k++)
            if ((i >> 5) == k) w[k] = (w[k] & ~m) | v;
    }
};

// 1/s to ~1 ulp: hardware seed (MUFU.RCP64H) + two Newton steps; outside the safe range the IEEE divide.
__device__ __forceinline__ double fast_reciprocal(double s) {
    double x;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(s));
    double e = fma(-s, x, 1.0);
    x = fma(x, e, x);
    e = fma(-s, x, 1.0);
    x = fma(x, e, x);
    // rare: not a positive normal number with exponent in [-963, 963) (integer-pipe test on the high word)
    if (!(((unsigned)__double2hiint(s) - 0x03c00000u) < 0x78600000u)) x = 1.0 / s;
    return x;
}

// Own factor of member descriptor d (host/mcmc_plan.hpp) for genotype g: (1e6 * prior) * lk for founders, 1e6 * lk
// otherwise (family.cpp:2115-2126).
__device__ __forceinline__ double gibbs_own_factor(uint32_t d, const VariantPriors &pr, int g, double lk) {
    const bool founder = (d >> 14) & 1u, male = (d >> 15) & 1u;
    const double base = founder ? 1000000.0 * (male ? pick3(pr.m, g) : pick3(pr.a, g)) : 1000000.0;
    return base * lk;
}

// The full conditional of member descriptor d: w0..w2 hold its own factors and receive the weights; returns their sum.
// link[k] are the plan's link descriptors, tab_addr the shared-window address of this lane's copy of the tables.
// The step is written branch-light: founders and missing children multiply by a row of ones, the first two children are
// handled in line, shared memory is addressed with 32-bit shared-window addresses.
template <int GW, class Links>
__device__ __forceinline__ double gibbs_weights(uint32_t d, const Links &link, const Genotypes<GW> &cur, bool chrx, uint32_t tab_addr,
                                                double &w0, double &w1, double &w2) {
    const bool male = (d >> 15) & 1u, founder = (d >> 14) & 1u;
    const int xkind = male ? 2 * 27 : 27; // chrX table of this member / of a child, by sex
    {   // own factor: transmission from the parents' current genotypes (a row of ones for founders)
        const int row = cur.get(d & 127u) * 3 + cur.get((d >> 7) & 127u);
        const int e = founder ? kOnes : (chrx ? xkind : 0) + row;
        const uint32_t ta = tab_addr + (uint32_t)e * (kCopies * 8u);
        w0 *= lds64(ta);
        w1 *= lds64(ta + 9 * kCopies * 8);
        w2 *= lds64(ta + 18 * kCopies * 8);
    }
    const int lb = (d >> 16) & 0xffu;
    const int n_links = (!chrx || male) ? (int)(d >> 24) : 0; // chrX: only males get the children factor
    const uint32_t step = male ? kCopies * 8u : 3u * kCopies * 8u;     // this member sits in the father slot when male
    auto child_entry = [&](int k) -> int {
        const uint32_t l = link[k];
        const int kind = chrx ? (((l >> 14) & 1u) ? 2 * 27 : 27) : 0;
        const int other = cur.get((l >> 7) & 127u);
        return kind + cur.get(l & 127u) * 9 + (male ? other * 3 : other);
    };
    {   // first two children in line (a row of ones when there are fewer)
        const int e0 = n_links > 0 ? child_entry(lb) : kOnes;
        const int e1 = n_links > 1 ? child_entry(lb + 1) : kOnes;
        const uint32_t a0 = tab_addr + (uint32_t)e0 * (kCopies * 8u), a1 = tab_addr + (uint32_t)e1 * (kCopies * 8u);
        const double x0 = lds64(a0), x1 = lds64(a0 + step), x2 = lds64(a0 + 2 * step);
        const double y0 = lds64(a1), y1 = lds64(a1 + step), y2 = lds64(a1 + 2 * step);
        w0 = (w0 * x0) * y0;
        w1 = (w1 * x1) * y1;
        w2 = (w2 * x2) * y2;
    }
    for (int k = lb + 2; k < lb + n_links; k++) { // third and later children
        const uint32_t a0 = tab_addr + (uint32_t)child_entry(k) * (kCopies * 8u);
        w0 *= lds64(a0);
        w1 *= lds64(a0 + step);
        w2 *= lds64(a0 + 2 * step);
    }
    return __dadd_rn(__dadd_rn(w0, w1), w2); // not contracted into an FMA, whatever the calling kernel does with the weights
}

// The draw from random word u: rd = ((u >> 1) + 0.5) * 2^-31 (31 bits, like the reference's rand() / RAND_MAX);
// rd < w0/sum and rd > 1 - w2/sum decided without the division; a non-positive sum means all-zero weights in the
// reference, which then draws genotype 1 (family.cpp:2142-2173).
__device__ __forceinline__ int gibbs_draw(uint32_t u, double sum, double w0, double w2) {
    const double rd = ((double)(u >> 1) + 0.5) * (1.0 / 2147483648.0);
    const double thr = rd * sum;
    int g = (thr < w0) ? 0 : ((thr > sum - w2) ? 2 : 1);
    if (!(sum > 0.0)) g = 1;
    return g;
}

// 1/sum of the Rao-Blackwellised accumulation (family.cpp:2175-2178); all-zero weights add nothing.
__device__ __forceinline__ double gibbs_inv(double sum) { return sum > 0.0 ? fast_reciprocal(sum) : 0.0; }

} // namespace

} // namespace famseq
