// families.cpp -- see families.hpp.
#include "families.hpp"

#include <numeric>

#include "../../../include/famseq_b200.h"
#include "pedigree.hpp"

namespace famseq {

int build_families(const Pedigree &p, const int32_t *id, FamilyTable &out, std::string &err) {
    const int n = p.n;
    // connected families: union-find over the parent links
    std::vector<int> up(n);
    std::iota(up.begin(), up.end(), 0);
    auto find = [&](int x) {
        while (up[x] != x) x = up[x] = up[up[x]];
        return x;
    };
    for (int i = 0; i < n; i++)
        if (!p.founder(i)) {
            up[find(i)] = find(p.mother[i]);
            up[find(i)] = find(p.father[i]);
        }
    FamilyTable t;
    t.family_of.assign(n, -1);
    std::vector<int> fam_of_root(n, -1), first_row;
    for (int i = 0; i < n; i++) {
        const int r = find(i);
        if (fam_of_root[r] < 0) {
            fam_of_root[r] = (int)first_row.size();
            first_row.push_back(i);
        }
        t.family_of[i] = fam_of_root[r];
    }
    const int F = (int)first_row.size();
    // members of each family in ped order (counting sort)
    std::vector<int> start(F + 1, 0), members(n);
    for (int i = 0; i < n; i++) start[t.family_of[i] + 1]++;
    for (int f = 0; f < F; f++) start[f + 1] += start[f];
    {
        std::vector<int> at(start.begin(), start.end() - 1);
        for (int i = 0; i < n; i++) members[at[t.family_of[i]]++] = i;
    }
    // classify: a lone individual, or two founders (a couple) with 1..5 childless children of both
    t.n_children.assign(F, 0);
    std::vector<int> father(F, -1), mother(F, -1);
    for (int f = 0; f < F; f++) {
        auto refuse = [&](const std::string &why) {
            err = "ped file family of " + std::to_string(id[first_row[f]]) + ": " + why +
                  "; fs_create_families takes lone individuals and nuclear families (two parents and 1.." +
                  std::to_string(FAMILY_MAX_CHILDREN) + " childless children of both)";
            return FS_E_TOO_LARGE;
        };
        const int size = start[f + 1] - start[f];
        if (size == 1) continue;
        int founders = 0, kids = 0;
        for (int k = start[f]; k < start[f + 1]; k++) {
            const int i = members[k];
            if (p.founder(i)) {
                founders++;
                continue;
            }
            if (!p.children[i].empty())
                return refuse("member " + std::to_string(id[i]) + " has both parents and children (more than two generations)");
            if (father[f] < 0) father[f] = p.father[i], mother[f] = p.mother[i];
            if (p.father[i] != father[f] || p.mother[i] != mother[f])
                return refuse("member " + std::to_string(id[i]) + " has other parents than a sibling (half-sibs or several spouses)");
            kids++;
        }
        if (founders != 2) return refuse(std::to_string(founders) + " founders (several spouses or half-sibs)");
        if (kids > FAMILY_MAX_CHILDREN) return refuse(std::to_string(kids) + " children");
        t.n_children[f] = kids;
    }
    // device order: by number of children, then by first row
    std::vector<int> order;
    order.reserve(F);
    for (int c = 0; c <= FAMILY_MAX_CHILDREN; c++) {
        for (int f = 0; f < F; f++)
            if (t.n_children[f] == c) order.push_back(f);
        t.class_end[c] = (int32_t)order.size();
        if (t.class_end[c] > (c ? t.class_end[c - 1] : 0)) t.nc_max = c;
    }
    t.col.assign((size_t)(2 + FAMILY_MAX_CHILDREN) * F, -1);
    t.male.assign(F, 0);
    for (int d = 0; d < F; d++) {
        const int f = order[d];
        auto put = [&](int role, int member) { t.col[(size_t)role * F + d] = p.col_of[member]; };
        if (t.n_children[f] == 0) {
            put(0, first_row[f]);
            t.male[d] = (uint8_t)p.male[first_row[f]];
            continue;
        }
        put(0, father[f]);
        put(1, mother[f]);
        int c = 0;
        for (int k = start[f]; k < start[f + 1]; k++) {
            const int i = members[k];
            if (p.founder(i)) continue;
            put(2 + c, i);
            t.male[d] |= (uint8_t)(p.male[i] << c);
            c++;
        }
    }
    out = std::move(t);
    return FS_OK;
}

} // namespace famseq
