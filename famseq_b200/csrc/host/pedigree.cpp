// pedigree.cpp -- see pedigree.hpp.
#include "pedigree.hpp"

#include <cstring>
#include <numeric>
#include <unordered_map>

#include "../../../include/famseq_b200.h"

namespace famseq {

int Pedigree::n_founders() const {
    int k = 0;
    for (int i = 0; i < n; i++) k += founder(i);
    return k;
}

namespace {
struct UnionFind {
    std::vector<int> p;
    explicit UnionFind(int n) : p(n) { std::iota(p.begin(), p.end(), 0); }
    int find(int x) {
        while (p[x] != x) x = p[x] = p[p[x]];
        return x;
    }
    // returns false when x and y were already connected (the new edge closes a cycle)
    bool join(int x, int y) {
        x = find(x);
        y = find(y);
        if (x == y) return false;
        p[x] = y;
        return true;
    }
};
} // namespace

int build_pedigree(int n, const int32_t *id, const int32_t *mother_id, const int32_t *father_id,
                   const int32_t *gender, int s, const int32_t *cols, Pedigree &out, std::string &err) {
    if (n <= 0 || !id || !mother_id || !father_id || !gender || s < 0 || (s > 0 && !cols)) {
        err = "fs_pedigree: null array or non-positive size";
        return FS_E_ARG;
    }
    Pedigree p;
    p.n = n;
    p.mother.assign(n, -1);
    p.father.assign(n, -1);
    p.male.assign(n, 0);
    p.children.assign(n, {});
    p.spouses.assign(n, {});
    p.col_of.assign(n, -1);
    for (int i = 0; i < n; i++) p.male[i] = gender[i] == 1;

    // Parent lookup scans every row without stopping, so the LAST row carrying a matching id wins
    // (family.cpp:300-316).
    std::unordered_map<int32_t, int> row_of_id;
    row_of_id.reserve((size_t)n);
    for (int j = 0; j < n; j++) row_of_id[id[j]] = j;
    auto row_of = [&](int32_t x) {
        const auto it = row_of_id.find(x);
        return it == row_of_id.end() ? -1 : it->second;
    };
    for (int i = 0; i < n; i++) {
        const int m = row_of(mother_id[i]), f = row_of(father_id[i]);
        if ((m < 0) != (f < 0)) {
            err = "This is not a fulfill family. Please check the ped file."; // family.cpp:320
            return FS_E_HALF_PARENTS;
        }
        if (m < 0) continue;
        p.mother[i] = m;
        p.father[i] = f;
        p.children[m].push_back(i);
        p.children[f].push_back(i);
        bool known_couple = false;
        for (int sp : p.spouses[m]) known_couple |= (sp == f);
        if (!known_couple) {
            p.spouses[m].push_back(f);
            p.spouses[f].push_back(m);
        }
    }
    for (int i = 0; i < n; i++) { // family.cpp:204-219
        if (p.mother[i] < 0) continue;
        if (gender[p.mother[i]] != 2) {
            err = "Sample " + std::to_string(id[p.mother[i]]) + "'s a mother while she is not a female.";
            return FS_E_GENDER;
        }
        if (gender[p.father[i]] != 1) {
            err = "Sample " + std::to_string(id[p.mother[i]]) + "'s a father while she is not a male.";
            return FS_E_GENDER;
        }
    }
    for (int c = 0; c < s; c++) {
        if (cols[c] < 0 || cols[c] >= n) {
            err = "fs_pedigree.cols entry out of range";
            return FS_E_ARG;
        }
        if (p.col_of[cols[c]] >= 0) {
            // two input columns with the same sample name: the reference lets the later column overwrite the
            // earlier one's likelihoods; the command line resolves that before calling the engine
            err = "fs_pedigree.cols lists ped row " + std::to_string(cols[c]) + " twice";
            return FS_E_ARG;
        }
        p.cols.push_back(cols[c]);
        p.col_of[cols[c]] = c;
    }

    // Loop detection on the marriage-node graph: one node per member, one per couple; edges
    // spouse--couple and child--couple.  The pedigree is peelable iff this graph is a forest.
    {
        std::vector<std::pair<int, int>> couples;
        std::unordered_map<int64_t, int> couple_index;
        auto couple_id = [&](int m, int f) {
            const auto ins = couple_index.emplace((int64_t)m * n + f, (int)couples.size());
            if (ins.second) couples.emplace_back(m, f);
            return ins.first->second;
        };
        for (int i = 0; i < n; i++)
            if (p.mother[i] >= 0) couple_id(p.mother[i], p.father[i]);
        UnionFind uf(n + (int)couples.size());
        std::vector<char> linked(couples.size(), 0);
        for (int i = 0; i < n && !p.has_loop; i++) {
            if (p.mother[i] < 0) continue;
            int c = couple_id(p.mother[i], p.father[i]);
            if (!linked[c]) {
                linked[c] = 1;
                if (!uf.join(p.mother[i], n + c)) p.has_loop = true;
                if (!uf.join(p.father[i], n + c)) p.has_loop = true;
            }
            if (!uf.join(i, n + c)) p.has_loop = true;
        }
    }
    out = std::move(p);
    return FS_OK;
}

// ------------------------------------------------------------------------------------------------
// Transmission tables.
// ------------------------------------------------------------------------------------------------
namespace {
inline double &at(double *t, int g, int a, int b) { return t[g * 9 + a * 3 + b]; }

// Autosome.  A parent of genotype x carries alleles al[x][0], al[x][1]; one of the two haplotypes is
// picked (prob 1/2) and transmitted faithfully with prob 1-mu.  The reference sums the four
// (maternal pick, paternal pick) cases one after another (family.cpp:497-544): pass = 2*hm + hf, and
// inside a pass the child allele pair (k,l) runs (0,0),(0,1),(1,0),(1,1).  The accumulation order is
// kept because it decides the last bit of the heterozygote entries.
void autosome(double mu, double *t) {
    static const int al[3][2] = {{0, 0}, {0, 1}, {1, 1}};
    std::memset(t, 0, sizeof(double) * 27);
    for (int a = 0; a < 3; a++)
        for (int b = 0; b < 3; b++) {
            if (mu == 0) { // exact quarters, family.cpp:472-490
                for (int hm = 0; hm < 2; hm++)
                    for (int hf = 0; hf < 2; hf++) {
                        int g = al[a][hm] + al[b][hf];
                        at(t, g, a, b) = at(t, g, a, b) + 0.25;
                    }
                continue;
            }
            const double wrong = mu / (2 * (2 - 1)), right = (1 - mu) / 2;
            for (int pass = 0; pass < 4; pass++) {
                const int from_m = al[a][pass >> 1], from_f = al[b][pass & 1];
                for (int k = 0; k < 2; k++)
                    for (int l = 0; l < 2; l++) {
                        const double gm = (k == from_m) ? right : wrong;
                        const double gf = (l == from_f) ? right : wrong;
                        at(t, k + l, a, b) = at(t, k + l, a, b) + gm * gf;
                    }
            }
        }
}

// X chromosome, daughter (family.cpp:383-416): mother transmits one of her two X, father his only X
// (genotype 0 or 2; the het-father column is all zero).
void x_daughter(double mu, double *t) {
    const double q = 1.0 - mu;
    std::memset(t, 0, sizeof(double) * 27);
    const double hom_same[3] = {q * q, 2 * mu * q, mu * mu};     // mother RR x father R (and mirrored)
    const double hom_diff[3] = {q * mu, q * q + mu * mu, q * mu}; // mother RR x father A (and mirrored)
    const double het_lo = q * q / 2 + mu * q / 2;
    const double het_mid = mu * q + q * q / 2 + mu * mu / 2;
    const double het_hi = mu * mu / 2 + mu * q / 2;
    for (int g = 0; g < 3; g++) {
        at(t, g, 0, 0) = hom_same[g];
        at(t, g, 0, 2) = hom_diff[g];
        at(t, g, 2, 0) = hom_diff[g];
        at(t, g, 2, 2) = hom_same[2 - g];
    }
    at(t, 0, 1, 0) = het_lo;
    at(t, 1, 1, 0) = het_mid;
    at(t, 2, 1, 0) = het_hi;
    at(t, 0, 1, 2) = het_hi;
    at(t, 1, 1, 2) = het_mid;
    at(t, 2, 1, 2) = het_lo;
}

// X chromosome, son (family.cpp:418-445): only the mother matters, a het son is impossible.
void x_son(double mu, double *t) {
    std::memset(t, 0, sizeof(double) * 27);
    const double from_mother[3] = {mu, 0.5, 1 - mu}; // Pr(son carries A | mother genotype)
    for (int a = 0; a < 3; a++)
        for (int b = 0; b < 3; b += 2) {
            at(t, 2, a, b) = from_mother[a];
            at(t, 0, a, b) = (a == 1) ? 0.5 : from_mother[2 - a];
        }
}
} // namespace

void build_tables(double mu, double tab[3][27]) {
    autosome(mu, tab[TAB_AUTO]);
    x_daughter(mu, tab[TAB_XF]);
    x_son(mu, tab[TAB_XM]);
}

} // namespace famseq
