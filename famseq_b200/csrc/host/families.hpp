// families.hpp -- a ped file of many unrelated families (a cohort) split into its connected families for the
// cohort Elston-Stewart kernels.  Lone individuals and nuclear families (two founders and 1..5 childless children of both)
// are peeled by cuda/es_families_kernel.cu; with FamilyMode::ANY_SHAPE, every other loop-free family of at most 128 members
// gets an ES message program of its own (host/es_program.cpp), run by cuda/es_cohort_kernel.cu.  FamilyMode::BN gives every
// family, looped ones included, the Bayesian-network plan of its own pedigree (host/bn_plan.cpp), run by
// cuda/bn_cohort_kernel.cu; FamilyMode::MCMC gives every family the Gibbs sampler's plan of its own pedigree
// (host/mcmc_plan.cpp), run by cuda/mcmc_cohort_kernel.cu.
#pragma once

#include <cstdint>
#include <string>
#include <vector>

#include "bn_plan.hpp"
#include "mcmc_plan.hpp"

namespace famseq {

struct Pedigree; // host/pedigree.hpp

constexpr int FAMILY_MAX_CHILDREN = 5;

struct FamilyTable {
    std::vector<int32_t> family_of;  // [n] family of each ped row; families are numbered by their first row
    std::vector<int32_t> n_children; // [F] 0 for a lone individual; a program family: its non-founder members
    // Device order of the families the nuclear kernel peels: sorted by number of children (stable), structure-of-arrays.
    std::vector<int32_t> col;         // [2 + FAMILY_MAX_CHILDREN][n_peeled] input columns (-1 = unsequenced): father, mother,
                                      // children in ped order; a lone individual's column is in row 0
    std::vector<uint8_t> male;        // [n_peeled] bit c: child c is male; a lone individual: bit 0
    int32_t class_end[FAMILY_MAX_CHILDREN + 1] = {}; // device-order families [class_end[k-1], class_end[k]) have k children
    int32_t nc_max = 0;
    int32_t n_peeled = 0;             // families of the nuclear kernel (all of them without any_shape)

    // Program families (any_shape only).  Programs are deduplicated by (words, n_slots); their operands index the
    // family's own vector file: local columns (its sequenced members in increasing global input column), scratch, priors,
    // ones -- nothing depends on the cohort's column count.
    std::vector<int32_t> program;     // [F] program of each family, -1 for a family of the nuclear kernel
    std::vector<int32_t> col_off;     // [F] offset of the family's local -> global column map in `cols`, -1 likewise
    std::vector<int32_t> cols;        // concatenated column maps
    std::vector<uint32_t> words;      // concatenated programs
    std::vector<int32_t> prog_off, prog_slots, prog_cols; // [P] word offset, scratch vectors, local columns
    std::vector<int32_t> prog_family; // [P] first family that runs the program (names it in messages)
    std::vector<int32_t> pf_order;    // program families sorted by program, then family: the device order
    int32_t max_vectors = 0;          // largest local columns + scratch vectors of any program

    // FamilyMode::BN and MCMC: every family has a plan (nothing above is filled in but family_of, n_children, col_off and
    // cols).  Plans are deduplicated by content.  Device order: by launch class, then by plan, then by first row.  A BN
    // launch class is (u, independent, factor_leaves, group -- one kernel instantiation and block shape); an MCMC launch
    // class is the width of the genotype vector (mcmc_cohort_width).
    std::vector<BnPlan> plans;           // [P] BN
    std::vector<McmcPlan> mcmc_plans;    // [P] MCMC
    std::vector<int32_t> plan;           // [F] plan of each family
    std::vector<int32_t> plan_family;    // [P] first family that has the plan (names it in messages)
    std::vector<int32_t> plan_order;     // [F] the families in device order
    std::vector<int32_t> plan_class_end; // device-order families [plan_class_end[k-1], plan_class_end[k]) form launch class k
    // MCMC: the ped rows of family f, increasing, are rows[row_off[f] .. row_off[f + 1]); local member k of its plan is
    // ped row rows[row_off[f] + k] (the Philox counter of its random words)
    std::vector<int32_t> rows, row_off;

    int n_families() const { return (int)n_children.size(); }
    int n_programs() const { return (int)prog_off.size(); }
};

enum class FamilyMode {
    NUCLEAR,   // lone individuals and nuclear families only (fs_create_families)
    ANY_SHAPE, // and an ES message program for every other loop-free family (fs_create_cohort)
    BN,        // a Bayesian-network plan for every family, loops included (fs_create_cohort_bn)
    MCMC,      // a Gibbs sampler plan for every family, loops included (fs_create_cohort_mcmc)
};

// Launch class of an MCMC family of n members: the 64-bit words of its genotype vector (1: <= 32, 2: <= 64, 4: <= 128).
inline int mcmc_cohort_width(int n) { return n <= 32 ? 1 : n <= 64 ? 2 : 4; }

// FS_OK, or an error with a message naming the first ped id of the first family that is refused: FS_E_TOO_LARGE for a
// family of another shape (NUCLEAR), over a limit of the ES message program (ANY_SHAPE), over BN_MAX_LEVELS members (BN) or
// over MCMC_MAX_MEMBERS members (MCMC), FS_E_LOOP for a looped family (ANY_SHAPE).  Linear in the number of ped rows plus the compile time of the programs or
// plans.
int build_families(const Pedigree &p, const int32_t *id, FamilyTable &out, std::string &err, FamilyMode mode = FamilyMode::NUCLEAR);

} // namespace famseq
