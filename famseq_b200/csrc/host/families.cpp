// families.cpp -- see families.hpp.
#include "families.hpp"

#include <algorithm>
#include <cstring>
#include <map>
#include <memory>
#include <numeric>
#include <tuple>
#include <unordered_map>

#include "../../../include/famseq_b200.h"
#include "es_program.hpp"
#include "pedigree.hpp"

namespace famseq {

namespace {

constexpr int FAMILY_MAX_MEMBERS = 128; // fs_create's limit for one pedigree

// Family `members` (ped rows in file order) as a pedigree of its own: the same parents, children and spouses in the same
// order as in the whole file, so the message program recurses exactly as the reference does over the whole file.  Its
// columns are its sequenced members in increasing global input column; `global_cols` receives that map.
void sub_pedigree(const Pedigree &p, const int *members, int size, std::vector<int> &local, Pedigree &sub,
                  std::vector<int32_t> &global_cols) {
    for (int k = 0; k < size; k++) local[members[k]] = k;
    auto to_local = [&](const std::vector<int> &rows) {
        std::vector<int> v(rows.size());
        for (size_t j = 0; j < rows.size(); j++) v[j] = local[rows[j]];
        return v;
    };
    sub = Pedigree();
    sub.n = size;
    sub.mother.assign(size, -1);
    sub.father.assign(size, -1);
    sub.male.assign(size, 0);
    sub.children.resize(size);
    sub.spouses.resize(size);
    sub.col_of.assign(size, -1);
    std::vector<std::pair<int, int>> seq; // (global column, local row)
    for (int k = 0; k < size; k++) {
        const int i = members[k];
        if (!p.founder(i)) sub.mother[k] = local[p.mother[i]], sub.father[k] = local[p.father[i]];
        sub.male[k] = p.male[i];
        sub.children[k] = to_local(p.children[i]);
        sub.spouses[k] = to_local(p.spouses[i]);
        if (p.col_of[i] >= 0) seq.emplace_back(p.col_of[i], k);
    }
    std::sort(seq.begin(), seq.end());
    global_cols.clear();
    for (const auto &c : seq) {
        sub.col_of[c.second] = (int)sub.cols.size();
        sub.cols.push_back(c.second);
        global_cols.push_back(c.first);
    }
}

// FamilyMode::BN and MCMC: every family gets the plan `build(sub, size, plan, why)` makes for its own pedigree (the one
// fs_create builds for the family's rows alone), deduplicated by content; then the device order by launch class
// (`class_of(plan)`), plan and first row.
template <class Plan, class Build, class ClassOf>
int build_plan_families(const Pedigree &p, const int32_t *id, const std::vector<int> &start, const std::vector<int> &members,
                        const std::vector<int> &first_row, FamilyTable &t, std::vector<Plan> &plans, Build build, ClassOf class_of,
                        std::string &err) {
    const int F = (int)first_row.size();
    t.plan.assign(F, -1);
    t.col_off.assign(F, -1);
    std::unordered_map<std::string, int32_t> index;
    std::vector<int> local(p.n, -1);
    std::vector<int32_t> global_cols;
    Pedigree sub;
    Plan plan;
    for (int f = 0; f < F; f++) {
        const int size = start[f + 1] - start[f];
        t.n_children[f] = size - (int)std::count_if(members.begin() + start[f], members.begin() + start[f + 1],
                                                    [&](int i) { return p.founder(i); });
        std::string why;
        const int rc = build(&members[start[f]], size, local, sub, global_cols, plan, why);
        if (rc != FS_OK) {
            err = "ped file family of " + std::to_string(id[first_row[f]]) + ": " + why;
            return rc;
        }
        auto hit = index.emplace(std::string(reinterpret_cast<const char *>(&plan), sizeof plan), (int32_t)plans.size());
        if (hit.second) {
            plans.push_back(plan);
            t.plan_family.push_back(f);
        }
        t.plan[f] = hit.first->second;
        t.col_off[f] = (int32_t)t.cols.size();
        t.cols.insert(t.cols.end(), global_cols.begin(), global_cols.end());
    }
    // device order: by launch class, then by plan, then by first row (a stable sort of the families by (class, plan))
    std::vector<int32_t> by_plan(plans.size());
    std::iota(by_plan.begin(), by_plan.end(), 0);
    std::stable_sort(by_plan.begin(), by_plan.end(), [&](int a, int b) { return class_of(plans[a]) < class_of(plans[b]); });
    std::vector<int32_t> rank(plans.size());
    for (size_t k = 0; k < by_plan.size(); k++) rank[by_plan[k]] = (int32_t)k;
    std::vector<int32_t> at(plans.size() + 1, 0);
    for (int f = 0; f < F; f++) at[rank[t.plan[f]] + 1]++;
    for (size_t k = 0; k < plans.size(); k++) at[k + 1] += at[k];
    t.plan_order.assign(F, -1);
    for (int f = 0; f < F; f++) t.plan_order[at[rank[t.plan[f]]]++] = f;
    for (size_t k = 0; k < by_plan.size(); k++) // at[k] is now the end of the families of plan by_plan[k]
        if (k + 1 == by_plan.size() || class_of(plans[by_plan[k + 1]]) != class_of(plans[by_plan[k]]))
            t.plan_class_end.push_back(at[k]);
    return FS_OK;
}

} // namespace

int build_families(const Pedigree &p, const int32_t *id, FamilyTable &out, std::string &err, FamilyMode mode) {
    const bool any_shape = mode == FamilyMode::ANY_SHAPE;
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
    t.n_children.assign(F, 0);
    if (mode == FamilyMode::BN) {
        auto build = [&](const int *rows, int size, std::vector<int> &local, Pedigree &sub, std::vector<int32_t> &global_cols,
                         BnPlan &plan, std::string &why) {
            if (size > BN_MAX_LEVELS) { // no sub-pedigree for a family build_bn_plan refuses by its size
                why = bn_too_large_message(size);
                return (int)FS_E_TOO_LARGE;
            }
            sub_pedigree(p, rows, size, local, sub, global_cols);
            return build_bn_plan(sub, plan, why);
        };
        auto class_of = [](const BnPlan &b) { return std::make_tuple(b.u, b.independent, b.factor_leaves, b.group); };
        const int rc = build_plan_families(p, id, start, members, first_row, t, t.plans, build, class_of, err);
        if (rc == FS_OK) out = std::move(t);
        return rc;
    }
    if (mode == FamilyMode::MCMC) {
        auto build = [&](const int *rows, int size, std::vector<int> &local, Pedigree &sub, std::vector<int32_t> &global_cols,
                         McmcPlan &plan, std::string &why) {
            if (size > MCMC_MAX_MEMBERS) {
                why = std::to_string(size) + " members; the MCMC kernel supports families of up to " + std::to_string(MCMC_MAX_MEMBERS) +
                      " members";
                return (int)FS_E_TOO_LARGE;
            }
            sub_pedigree(p, rows, size, local, sub, global_cols);
            return build_mcmc_plan(sub, plan, why);
        };
        auto class_of = [](const McmcPlan &m) { return mcmc_cohort_width(m.n); };
        const int rc = build_plan_families(p, id, start, members, first_row, t, t.mcmc_plans, build, class_of, err);
        if (rc != FS_OK) return rc;
        t.rows.assign(members.begin(), members.end());
        t.row_off.assign(start.begin(), start.end());
        out = std::move(t);
        return FS_OK;
    }
    // classify: a lone individual, or two founders (a couple) with 1..5 childless children of both; any other family
    // is refused, or, with any_shape, peeled by a message program of its own
    std::vector<int> father(F, -1), mother(F, -1);
    std::vector<char> by_program(F, 0);
    for (int f = 0; f < F; f++) {
        std::string why;
        const int size = start[f + 1] - start[f];
        if (size == 1) continue;
        int founders = 0, kids = 0;
        for (int k = start[f]; k < start[f + 1] && why.empty(); k++) {
            const int i = members[k];
            if (p.founder(i)) {
                founders++;
                continue;
            }
            if (!p.children[i].empty()) {
                why = "member " + std::to_string(id[i]) + " has both parents and children (more than two generations)";
                break;
            }
            if (father[f] < 0) father[f] = p.father[i], mother[f] = p.mother[i];
            if (p.father[i] != father[f] || p.mother[i] != mother[f])
                why = "member " + std::to_string(id[i]) + " has other parents than a sibling (half-sibs or several spouses)";
            kids++;
        }
        if (why.empty() && founders != 2) why = std::to_string(founders) + " founders (several spouses or half-sibs)";
        if (why.empty() && kids > FAMILY_MAX_CHILDREN) why = std::to_string(kids) + " children";
        if (why.empty()) {
            t.n_children[f] = kids;
            continue;
        }
        if (!any_shape) {
            err = "ped file family of " + std::to_string(id[first_row[f]]) + ": " + why +
                  "; fs_create_families takes lone individuals and nuclear families (two parents and 1.." +
                  std::to_string(FAMILY_MAX_CHILDREN) + " childless children of both)";
            return FS_E_TOO_LARGE;
        }
        by_program[f] = 1;
        t.n_children[f] = size - (int)std::count_if(members.begin() + start[f], members.begin() + start[f + 1],
                                                    [&](int i) { return p.founder(i); });
    }
    // device order: by number of children, then by first row
    std::vector<int> order;
    order.reserve(F);
    for (int c = 0; c <= FAMILY_MAX_CHILDREN; c++) {
        for (int f = 0; f < F; f++)
            if (t.n_children[f] == c && !by_program[f]) order.push_back(f);
        t.class_end[c] = (int32_t)order.size();
        if (t.class_end[c] > (c ? t.class_end[c - 1] : 0)) t.nc_max = c;
    }
    const int D = t.n_peeled = (int)order.size();
    t.col.assign((size_t)(2 + FAMILY_MAX_CHILDREN) * D, -1);
    t.male.assign(D, 0);
    for (int d = 0; d < D; d++) {
        const int f = order[d];
        auto put = [&](int role, int member) { t.col[(size_t)role * D + d] = p.col_of[member]; };
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
    if (any_shape) {
        // one message program per family shape and sequencing pattern, compiled on the family's own pedigree
        t.program.assign(F, -1);
        t.col_off.assign(F, -1);
        std::map<std::pair<std::vector<uint32_t>, int32_t>, int32_t> index;
        std::vector<int> local(n, -1);
        std::vector<int32_t> global_cols;
        Pedigree sub;
        auto prog = std::make_unique<EsProgram>();
        for (int f = 0; f < F; f++) {
            if (!by_program[f]) continue;
            const int size = start[f + 1] - start[f];
            const std::string name = "ped file family of " + std::to_string(id[first_row[f]]) + ": ";
            if (size > FAMILY_MAX_MEMBERS) {
                err = name + std::to_string(size) + " members; a family of a cohort is one pedigree of at most " +
                      std::to_string(FAMILY_MAX_MEMBERS) + " members";
                return FS_E_TOO_LARGE;
            }
            sub_pedigree(p, &members[start[f]], size, local, sub, global_cols);
            std::string why;
            const int rc = compile_es_program(sub, *prog, why);
            if (rc != FS_OK) {
                err = name + why;
                return rc;
            }
            auto hit = index.emplace(std::make_pair(std::vector<uint32_t>(prog->words, prog->words + prog->n_words), prog->n_slots),
                                     t.n_programs());
            if (hit.second) {
                t.prog_off.push_back((int32_t)t.words.size());
                t.prog_slots.push_back(prog->n_slots);
                t.prog_cols.push_back(prog->n_cols);
                t.prog_family.push_back(f);
                t.words.insert(t.words.end(), prog->words, prog->words + prog->n_words);
                t.max_vectors = std::max(t.max_vectors, prog->n_cols + prog->n_slots);
            }
            t.program[f] = hit.first->second;
            t.col_off[f] = (int32_t)t.cols.size();
            t.cols.insert(t.cols.end(), global_cols.begin(), global_cols.end());
        }
        // device order: by program, then by first row (neighbouring blocks run the same program)
        std::vector<int32_t> at(t.n_programs() + 1, 0);
        for (int f = 0; f < F; f++)
            if (t.program[f] >= 0) at[t.program[f] + 1]++;
        for (int q = 0; q < t.n_programs(); q++) at[q + 1] += at[q];
        t.pf_order.assign(at.back(), -1);
        for (int f = 0; f < F; f++)
            if (t.program[f] >= 0) t.pf_order[at[t.program[f]]++] = f;
    }
    out = std::move(t);
    return FS_OK;
}

} // namespace famseq
