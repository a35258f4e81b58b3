// bn_peel.cpp -- see bn_peel.hpp.
#include "bn_peel.hpp"
#include "pedigree.hpp"

#include <map>
#include <numeric>

#include "../../../include/famseq_b200.h"

namespace famseq {
namespace {

// Cycle rank E - V + C of the member--marriage graph of the parent rows (a marriage is a parent pair with children; edges
// mother--marriage, father--marriage, child--marriage): the number of edges that close a cycle when added one by one.
int cycle_rank(const std::vector<int> &mother, const std::vector<int> &father) {
    const int n = (int)mother.size();
    std::map<std::pair<int, int>, int> couple;
    for (int i = 0; i < n; i++)
        if (mother[i] >= 0) couple.emplace(std::make_pair(mother[i], father[i]), (int)couple.size());
    std::vector<int> root(n + couple.size());
    std::iota(root.begin(), root.end(), 0);
    auto find = [&](int x) {
        while (root[x] != x) x = root[x] = root[root[x]];
        return x;
    };
    int closing = 0;
    auto join = [&](int x, int y) {
        x = find(x);
        y = find(y);
        if (x == y)
            closing++;
        else
            root[x] = y;
    };
    for (const auto &c : couple) {
        join(c.first.first, n + c.second);
        join(c.first.second, n + c.second);
    }
    for (int i = 0; i < n; i++)
        if (mother[i] >= 0) join(i, n + couple[std::make_pair(mother[i], father[i])]);
    return closing;
}

// The parent rows while marriages are being handed to copies; copies are appended founders.
struct Broken {
    std::vector<int> mother, father, male, copy_of; // copy_of[r]: the member row r copies, -1 for the pedigree's own rows
    int rank = 0;

    // b's marriages (mother, father), in the order of their first child
    std::vector<std::pair<int, int>> marriages(int b) const {
        std::vector<std::pair<int, int>> out;
        for (size_t i = 0; i < mother.size(); i++) {
            if (mother[i] != b && father[i] != b) continue;
            const auto m = std::make_pair(mother[i], father[i]);
            bool seen = false;
            for (const auto &o : out) seen |= o == m;
            if (!seen) out.push_back(m);
        }
        return out;
    }
    // Hands marriage m of b to a new copy of b when that marriage lies on a loop (the rank drops); otherwise changes nothing.
    bool move(int b, std::pair<int, int> m) {
        Broken t = *this;
        const int r = (int)t.mother.size();
        t.mother.push_back(-1);
        t.father.push_back(-1);
        t.male.push_back(male[b]);
        t.copy_of.push_back(b);
        for (int i = 0; i < r; i++)
            if (t.mother[i] == m.first && t.father[i] == m.second) (m.first == b ? t.mother[i] : t.father[i]) = r;
        t.rank = cycle_rank(t.mother, t.father);
        if (t.rank >= rank) return false;
        *this = std::move(t);
        return true;
    }
    // Every marriage of b on a loop, in order.  Returns how much the rank dropped.
    int condition(int b) {
        const int before = rank;
        for (const auto &m : marriages(b)) move(b, m);
        return before - rank;
    }
};

} // namespace

int bn_peel_cycle_rank(const Pedigree &ped) { return cycle_rank(ped.mother, ped.father); }

int build_bn_peel_program(const Pedigree &ped, BnPeelProgram &out, std::string &err) {
    out = BnPeelProgram();
    Broken cur;
    cur.mother = ped.mother;
    cur.father = ped.father;
    cur.male = ped.male;
    cur.copy_of.assign(ped.n, -1);
    cur.rank = cycle_rank(cur.mother, cur.father);

    // ---- the breakers: greedy on the rank drop, ties to the lowest ped row --------------------------------------------
    std::vector<int> breakers;
    std::vector<char> picked(ped.n, 0);
    while (cur.rank > 0) {
        if ((int)breakers.size() == BN_PEEL_MAX_BREAKERS) {
            err = "pedigree too large for conditioned peeling (-method 1 -peelLoops): more than " +
                  std::to_string(BN_PEEL_MAX_BREAKERS) + " loop breakers needed (" + std::to_string(breakers.size()) +
                  " picked, " + std::to_string(cur.rank) + " loops left)";
            return FS_E_TOO_LARGE;
        }
        int best = -1, best_gain = 0;
        Broken best_state;
        for (int b = 0; b < ped.n; b++) {
            if (picked[b]) continue;
            Broken t = cur;
            const int gain = t.condition(b);
            if (gain > best_gain) {
                best = b;
                best_gain = gain;
                best_state = std::move(t);
            }
        }
        if (best < 0) { // cannot happen: every loop runs through a marriage edge of one of its members
            err = "conditioned peeling: no loop breaker found";
            return FS_E_TOO_LARGE;
        }
        picked[best] = 1;
        breakers.push_back(best);
        cur = std::move(best_state);
    }

    // ---- the broken pedigree: build_pedigree's child and spouse order over the rewired parent rows ------------------
    const int n = (int)cur.mother.size(), K = (int)breakers.size(), S = ped.s();
    Pedigree q;
    q.n = n;
    q.mother = cur.mother;
    q.father = cur.father;
    q.male = cur.male;
    q.children.assign(n, {});
    q.spouses.assign(n, {});
    q.cols = ped.cols;
    q.col_of = ped.col_of;
    q.col_of.resize(n, -1);
    for (int i = 0; i < n; i++) {
        const int m = q.mother[i], f = q.father[i];
        if (m < 0) continue;
        q.children[m].push_back(i);
        q.children[f].push_back(i);
        bool known_couple = false;
        for (int sp : q.spouses[m]) known_couple |= (sp == f);
        if (!known_couple) {
            q.spouses[m].push_back(f);
            q.spouses[f].push_back(m);
        }
    }

    // ---- reserved vectors: clamped likelihoods, indicators, accumulators ----------------------------------------------
    EsConditioning cond;
    cond.n_real = ped.n;
    cond.lk_fixed.assign(n, -1);
    cond.ant_fixed.assign(n, -1);
    cond.acc_fixed.assign(ped.n, -1);
    for (int j = 0; j < K; j++) cond.lk_fixed[breakers[j]] = j;
    for (int r = ped.n; r < n; r++)
        for (int j = 0; j < K; j++)
            if (cur.copy_of[r] == breakers[j]) cond.ant_fixed[r] = K + j;
    for (int i = 0, u = 0; i < ped.n; i++) cond.acc_fixed[i] = 2 * K + (ped.col_of[i] >= 0 ? ped.col_of[i] : S + u++);
    cond.n_fixed = 2 * K + ped.n;

    const int rc = compile_es_program(q, out.prog, err, &cond);
    if (rc != FS_OK) {
        if (rc == FS_E_TOO_LARGE) err = "conditioned peeling (-method 1 -peelLoops): " + err;
        return FS_E_TOO_LARGE; // FS_E_LOOP cannot happen: the broken pedigree is a forest
    }
    out.n_breakers = K;
    for (int j = 0; j < K; j++) {
        out.breaker_row[j] = breakers[j];
        out.breaker_col[j] = ped.col_of[breakers[j]];
    }
    out.clamp_base = S + out.prog.n_slots + 3;
    out.acc_base = out.clamp_base + 2 * K;
    out.n_acc = ped.n;
    out.n_vectors = out.acc_base + ped.n;
    return FS_OK;
}

} // namespace famseq
