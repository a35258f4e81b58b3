// families.hpp -- a ped file of many unrelated families (a cohort) split into its connected families for the
// cohort Elston-Stewart kernel (cuda/es_families_kernel.cu).  Each family must be a lone individual or a nuclear family:
// two founders and 1..5 childless children of both.
#pragma once

#include <cstdint>
#include <string>
#include <vector>

namespace famseq {

struct Pedigree; // host/pedigree.hpp

constexpr int FAMILY_MAX_CHILDREN = 5;

struct FamilyTable {
    std::vector<int32_t> family_of;  // [n] family of each ped row; families are numbered by their first row
    std::vector<int32_t> n_children; // [F] 0 for a lone individual
    // Device order: families sorted by number of children (stable), structure-of-arrays.
    std::vector<int32_t> col;         // [2 + FAMILY_MAX_CHILDREN][F] input columns (-1 = unsequenced): father, mother,
                                      // children in ped order; a lone individual's column is in row 0
    std::vector<uint8_t> male;        // [F] bit c: child c is male; a lone individual: bit 0
    int32_t class_end[FAMILY_MAX_CHILDREN + 1] = {}; // device-order families [class_end[k-1], class_end[k]) have k children
    int32_t nc_max = 0;
    int n_families() const { return (int)n_children.size(); }
};

// FS_OK, or FS_E_TOO_LARGE with a message naming the first ped id of the first family of another shape.  Linear in the
// number of ped rows.
int build_families(const Pedigree &p, const int32_t *id, FamilyTable &out, std::string &err);

} // namespace famseq
