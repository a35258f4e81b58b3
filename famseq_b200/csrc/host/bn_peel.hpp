// bn_peel.hpp -- exact BN posteriors of looped pedigrees by conditioned Elston-Stewart peeling (loop-cutset conditioning).
//
// A few loop-breaker members are picked; each of their marriages that lies on a loop is handed to a founder copy of the
// breaker's sex, which leaves a loop-free pedigree with the same connected families.  For every assignment of one
// genotype to each breaker (3^K "clamps"), the breaker's likelihood is multiplied by the indicator of its genotype and its
// copies take that indicator as their founder prior, so the broken pedigree's joint is the original joint restricted to
// the clamp.  Peeling it once per clamp and adding up every member's unnormalised marginal gives the exact marginal the
// Bayesian network enumerates; a loop-free pedigree has K = 0 and one peel, the ES program with FIN replaced by ACC.
#pragma once

#include <string>
#include <vector>

#include "es_program.hpp"

namespace famseq {

struct Pedigree; // host/pedigree.hpp

constexpr int BN_PEEL_MAX_BREAKERS = 8; // 3^8 = 6 561 peels per variant

// The conditioned program and what the kernel needs to drive it.  Vector file (es_program.hpp's, extended):
//   [0, S) likelihood rows, [S, S + n_slots) scratch, S + n_slots + 0/1/2 the special vectors, then
//   clamp_base + j        breaker j's clamped likelihood (lk (*) e_c, or e_c when it is unsequenced)
//   clamp_base + K + j    breaker j's indicator e_c (the founder prior of its copies)
//   acc_base + k          accumulator k: k < S the member behind input column k, then the unsequenced members in ped order
struct BnPeelProgram {
    EsProgram prog;
    int32_t n_breakers = 0;
    int32_t breaker_row[BN_PEEL_MAX_BREAKERS] = {}; // ped rows, in the order they were picked
    int32_t breaker_col[BN_PEEL_MAX_BREAKERS] = {}; // their input columns, -1 = unsequenced
    int32_t clamp_base = 0, acc_base = 0, n_acc = 0;
    int32_t n_vectors = 0; // the whole vector file
};

// Cycle rank E - V + C of the pedigree's member--marriage graph: the number of independent loops.
int bn_peel_cycle_rank(const Pedigree &ped);

// Picks the breakers, builds the broken pedigree and compiles its conditioned program.  Breakers are greedy: each round
// takes the member whose marriages, handed one by one to copies while they still lie on a loop, lower the cycle rank most
// (ties: lowest ped row), until the graph is a forest; so K <= the cycle rank.  A marriage that is not on a loop is never
// moved, which keeps every family connected.  FS_OK, or FS_E_TOO_LARGE with the reason in `err`: more than
// BN_PEEL_MAX_BREAKERS breakers, a program over ES_MAX_WORDS or a vector file over the 16-bit operand range.
int build_bn_peel_program(const Pedigree &ped, BnPeelProgram &out, std::string &err);

} // namespace famseq
