// bn_plan.cpp -- see bn_plan.hpp.
#include <cstdlib>
#include <cstring>

#include "../../../include/famseq_b200.h"
#include "bn_plan.hpp"
#include "pedigree.hpp"

namespace famseq {

std::string bn_too_large_message(int n) {
    return "The Bayesian-network method enumerates 3^N genotype configurations; N = " + std::to_string(n) +
           " exceeds the kernel limit of " + std::to_string(BN_MAX_LEVELS) + " members.";
}

int build_bn_plan(const Pedigree &ped, BnPlan &out, std::string &err) {
    BnPlan p{};
    const int N = ped.n;
    if (N > BN_MAX_LEVELS) {
        err = bn_too_large_message(N);
        return FS_E_TOO_LARGE;
    }
    p.n_levels = N;

    // Enumeration order: parents before children; members who have children first (generation by
    // generation), childless members innermost.  Childless members' factors then depend only on
    // digits that are fixed outside the innermost loops.
    std::vector<int> order;
    std::vector<char> placed(N, 0);
    for (int pass = 0; pass < 2; pass++) {
        bool progress = true;
        while (progress) {
            progress = false;
            for (int i = 0; i < N; i++) {
                if (placed[i]) continue;
                const bool leaf = ped.children[i].empty();
                if ((pass == 0) == leaf) continue;
                if (!ped.founder(i) && (!placed[ped.mother[i]] || !placed[ped.father[i]])) continue;
                placed[i] = 1;
                order.push_back(i);
                progress = true;
            }
        }
    }
    if ((int)order.size() != N) { // cannot happen: a pedigree is a DAG
        err = "internal error: pedigree is not a DAG";
        return FS_E_ARG;
    }
    std::vector<int> level_of(N);
    for (int L = 0; L < N; L++) level_of[order[L]] = L;

    int n_leaves = 0;
    for (int i = 0; i < N; i++) n_leaves += ped.children[i].empty();
    // fully unrolled depth: 5 (243 configurations per block) only pays when the block can run out of registers,
    // i.e. when the five innermost members are all childless
    p.u = N < 3 ? N : (N >= 11 && n_leaves >= 5 ? 5 : (N >= 9 ? 4 : 3));
    if (const char *env = std::getenv("FAMSEQ_BN_UNROLL")) { // tuning knob: depth of the fully unrolled block
        const int u = std::atoi(env);
        if (u >= 1 && u <= BN_MAX_UNROLL && u <= N) p.u = u;
    }
    p.h = N - p.u < 5 ? N - p.u : 5;
    if (const char *env = std::getenv("FAMSEQ_BN_SPREAD")) { // tuning knob: levels spread over threads (3^h threads per variant)
        const int h = std::atoi(env);
        if (h >= 0 && h <= 5 && h <= N - p.u) p.h = h;
    }
    p.r = N - p.u - p.h;
    p.group = 1;
    for (int k = 0; k < p.h; k++) p.group *= 3;
    p.vpb = 256 / p.group;
    if (p.vpb < 1) p.vpb = 1;
    p.threads = ((p.vpb * p.group + 31) / 32) * 32;

    int off = 0;
    for (int L = 0; L < N; L++) {
        const int i = order[L];
        p.member[L] = (int16_t)i;
        p.col[L] = (int16_t)ped.col_of[i];
        p.male[L] = (uint8_t)ped.male[i];
        p.founder[L] = ped.founder(i);
        p.sh_m[L] = p.sh_f[L] = BN_ZERO_SHIFT;
        if (!ped.founder(i)) {
            p.sh_m[L] = (uint8_t)(2 * level_of[ped.mother[i]]);
            p.sh_f[L] = (uint8_t)(2 * level_of[ped.father[i]]);
        }
        p.tab_off[L] = off;
        for (int q = 0; q < (ped.founder(i) ? 1 : 9); q++) p.row_level[off / 4 + q] = (uint8_t)L;
        off += ped.founder(i) ? 4 : 36;
    }
    p.table_doubles = off;
    const int first_unrolled = N - p.u;
    for (int x = 0; x < p.u; x++) {
        const int i = order[first_unrolled + x];
        if (ped.founder(i)) continue;
        for (int y = 0; y < x; y++) {
            const int j = order[first_unrolled + y];
            if (ped.mother[i] == j) p.ustride[x][y] = 12; // row = 3*mother + father, 4 doubles per row
            if (ped.father[i] == j) p.ustride[x][y] = 4;
        }
    }
    p.unrolled_dep = -1;
    for (int x = 0; x < p.u; x++) {
        const int i = order[first_unrolled + x];
        if (ped.founder(i)) continue;
        for (int par : {ped.mother[i], ped.father[i]}) {
            const int q = level_of[par] - p.h; // rolled index of the parent, if it is a rolled level
            if (q >= 0 && q < p.r && q > p.unrolled_dep) p.unrolled_dep = q;
        }
    }
    p.independent = 1;
    for (int x = 0; x < p.u; x++)
        for (int y = 0; y < x; y++)
            if (p.ustride[x][y]) p.independent = 0;
    if (const char *env = std::getenv("FAMSEQ_BN_FACTOR")) p.factor_leaves = env[0] == '1';
    if (const char *env = std::getenv("FAMSEQ_BN_GENERIC")) // tuning / test knob: force the general unrolled block
        if (env[0] == '1') p.independent = 0;
    out = p;
    return FS_OK;
}

} // namespace famseq
