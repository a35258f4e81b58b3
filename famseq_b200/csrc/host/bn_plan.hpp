// bn_plan.hpp -- enumeration plan for the Bayesian-network method: the order in which the members'
// genotypes are enumerated and how the 3^N joint configurations are split over threads.
//
// The reference (family.cpp:882-954) runs one odometer over all N digits and re-multiplies all N
// factors for every configuration.  The plan orders the members parents-before-children so that the
// joint probability can be carried as a prefix product down a loop nest:
//
//   levels 0 .. h-1          "spread" levels  : one thread per combination (3^h threads per variant)
//   levels h .. h+r-1        "rolled" levels  : an odometer inside every thread
//   levels h+r .. N-1        "unrolled" levels: a fully unrolled block of 3^u configurations
//
// Shared between host/bn_plan.cpp and cuda/bn_kernel.cu.
#pragma once

#include <cstdint>
#include <string>

namespace famseq {

struct Pedigree; // host/pedigree.hpp

constexpr int BN_MAX_LEVELS = 31; // 2 bits per level in a 64-bit word, field 31 stays zero
constexpr int BN_MAX_UNROLL = 5;
constexpr int BN_ZERO_SHIFT = 62; // bit position of the always-zero field (founders' "parents")

struct BnPlan {
    int32_t n_levels = 0; // = pedigree size N
    int32_t h = 0, r = 0, u = 0;
    int32_t group = 1;    // 3^h threads cooperate on one variant
    int32_t vpb = 1;      // variants per block
    int32_t threads = 32; // block size
    int32_t table_doubles = 0; // per-variant factor tables: 4 doubles per (level, parent-genotype row)
    // per level, outermost first
    int16_t member[32];  // ped row
    int16_t col[32];     // input column, -1 when unsequenced
    uint8_t male[32];
    uint8_t founder[32];
    uint8_t sh_m[32], sh_f[32]; // bit position in the packed configuration word of the mother's / father's digit
    int32_t tab_off[32];        // offset (doubles) of the level's table inside the variant's table block
    uint8_t row_level[288];     // level that owns table row q (row q starts at double 4q)
    // unrolled level x (0 = outermost unrolled): row stride (in doubles: 0, 4 or 12) contributed by the
    // digit of unrolled level y < x when y is its father / mother
    int32_t ustride[BN_MAX_UNROLL][BN_MAX_UNROLL];
    // 1 when no unrolled level is a parent of another unrolled level (all ustride are zero): the factor vectors of
    // the unrolled block then depend on outer digits only and are loaded once per block instead of once per use
    int32_t independent = 0;
    int32_t factor_leaves = 0; // FAMSEQ_BN_FACTOR=1: sum the unrolled (childless, independent) block analytically
    // largest rolled index (0 = outermost rolled level) that is a parent of an unrolled level, -1 if none: the
    // unrolled block's table rows must be re-read only when a rolled level <= this one changes
    int32_t unrolled_dep = -1;
};

// Host entry point (bn_plan.cpp): builds the enumeration plan.  Returns FS_OK or FS_E_TOO_LARGE.
int build_bn_plan(const Pedigree &ped, BnPlan &out, std::string &err);
// build_bn_plan's refusal of a pedigree of n > BN_MAX_LEVELS members.
std::string bn_too_large_message(int n);

} // namespace famseq
