// kernels.hpp -- launch interface between the engine (engine.cu) and the three method kernels.
#pragma once

#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>
#include <vector>

#include "../host/bn_peel.hpp"
#include "../host/bn_plan.hpp"
#include "../host/es_program.hpp"
#include "../host/mcmc_plan.hpp"
#include "common.cuh"

struct fs_phred_fix; // include/famseq_b200.h

namespace famseq {

// ---- Elston-Stewart (es_kernel.cu) ----------------------------------------------------------------
struct EsParams {
    RunConstants C;
    EsProgram prog;
};
size_t es_smem_bytes(const EsParams &P, int tb);
int es_pick_block(const EsParams &P, size_t smem_limit);
cudaError_t launch_es(const EsParams &P, const BatchPtrs &B, int tb, cudaStream_t stream);

// ---- Bayesian network by conditioned peeling (bn_peel_kernel.cu) ---------------------------------------------
struct BnPeelParams {
    RunConstants C;
    BnPeelProgram peel;
};
// es_pick_block's rule for the conditioned program's vector file; 0 when not even 32 variants fit.
int bn_peel_pick_block(const BnPeelParams &P, size_t smem_limit);
cudaError_t launch_bn_peel(const BnPeelParams &P, const BatchPtrs &B, int tb, cudaStream_t stream);

// ---- Elston-Stewart, nuclear families (es_nuclear_kernel.cu) -------------------------------------------
constexpr int ES_NUCLEAR_MAX_CHILDREN = 5;
struct NuclearParams {
    RunConstants C;
    int32_t n_children;
    int32_t col_father, col_mother;               // input column or -1
    int32_t col_child[ES_NUCLEAR_MAX_CHILDREN];   // children in ped order
    int32_t male_child[ES_NUCLEAR_MAX_CHILDREN];
    int32_t allow_ident; // use the kernel specialised for the identity column map when it applies (FAMSEQ_ES_IDENT=0 turns it off)
    int32_t stream_tiles; // compact input: tiles per block, each prefetched under the one before (0: 4 for trios, 8 otherwise; -1: the one-tile kernel; FAMSEQ_ES_STREAM)
};
// Handles B.pl (compact input, decoded through B.lut) and B.single == nullptr itself.
cudaError_t launch_es_nuclear(const NuclearParams &P, const BatchPtrs &B, cudaStream_t stream);

// ---- Elston-Stewart, cohorts of nuclear families and lone individuals (es_families_kernel.cu) ----------------
// Families are ordered by class: [class_end[k-1], class_end[k]) have k children (k = 0: lone individuals).  The family table
// is structure-of-arrays in device memory, F entries per array.
constexpr int ES_FAMILIES_BLOCK = 128;
struct FamiliesParams {
    RunConstants C;           // C.s = S (may exceed FS_MAX_MEMBERS); C.col_male is unused, col_male below replaces it
    int32_t n_families;
    int32_t nc_max;           // largest sibship present (0..ES_NUCLEAR_MAX_CHILDREN)
    int32_t group;            // threads per variant: 4, 8, 16, 32, or ES_FAMILIES_BLOCK (the whole block)
    int32_t class_end[ES_NUCLEAR_MAX_CHILDREN + 1];
    const int32_t *fam_col;   // [2 + ES_NUCLEAR_MAX_CHILDREN][F] input columns (-1 = unsequenced): father, mother, children in ped
                              // order; a lone individual's column is in row 0
    const uint8_t *fam_male;  // [F] bit c: child c is male; a lone individual: bit 0
    const uint8_t *col_male;  // [S] gender == 1 of the member behind each input column
};
// Threads per variant for a row of S input columns.
int es_families_group(int S);
// Handles B.pl and B.single == nullptr itself, like the nuclear-family kernel.
cudaError_t launch_es_families(const FamiliesParams &P, const BatchPtrs &B, cudaStream_t stream);

// ---- Elston-Stewart, cohorts with families of any loop-free shape (es_cohort_kernel.cu) ------------------------
// The families es_families_kernel takes are peeled as there; every other family runs its deduplicated message program
// (host/families.hpp), one block per (variant tile, family).  The program arrays live in device memory.
struct CohortParams {
    FamiliesParams fam;         // the column pass, the nuclear families and lone individuals
    int32_t n_pf;               // families peeled by a program
    int32_t tb;                 // variants per block of the program kernel: 128, 64 or 32
    int32_t max_vectors;        // largest local columns + scratch vectors of any program: sizes the vector file
    const uint32_t *words;      // concatenated programs
    const int32_t *prog_off;    // [P] word offset of each program
    const int32_t *prog_slots;  // [P] scratch vectors
    const int32_t *prog_cols;   // [P] local columns
    const int32_t *pf_prog;     // [n_pf] program of each program family, sorted by program
    const int32_t *pf_col_off;  // [n_pf] offset of its local -> global column map in `cols`
    const int32_t *cols;        // concatenated column maps
};
// Shared memory of the program kernel's vector file at block size tb.
size_t es_cohort_smem_bytes(int max_vectors, int tb);
// Three launches whatever the number of families: the column pass and nuclear families, the programs, the failure rule.
// Handles B.pl and B.single == nullptr itself.
cudaError_t launch_es_cohort(const CohortParams &P, const BatchPtrs &B, cudaStream_t stream);
// Its first and last launch, for the cohort BN path too: es_cohort_head_kernel (individual-only posteriors, the whole-row
// gate and failure flag, the nuclear families of P; status := failed | needed << 1) and es_cohort_finish_kernel (NA rows of
// every failed variant, status := failed).
cudaError_t launch_es_cohort_head(const FamiliesParams &P, const BatchPtrs &B, cudaStream_t stream);
cudaError_t launch_es_cohort_finish(const BatchPtrs &B, int S, cudaStream_t stream);

// ---- Bayesian network (bn_kernel.cu) --------------------------------------------------------------
struct BnParams {
    RunConstants C;
    BnPlan plan;
};
size_t bn_smem_bytes(const BnParams &P);
cudaError_t launch_bn(const BnParams &P, const BatchPtrs &B, int sm_count, cudaStream_t stream);

// ---- Bayesian network, cohorts: every family enumerated on its own (bn_cohort_kernel.cu) --------------------------
// Families of one launch class share the instantiation bn_cohort_kernel<u, independent, factor_leaves> and the block shape
// (group threads per variant, 256 / group variants per block, 256 threads); they are [begin, end) of the device order.
struct BnCohortClass {
    int32_t u, independent, factor_leaves, group;
    int32_t begin, end;
    size_t smem; // the largest of bn_cohort_smem_bytes over the class's plans
};
struct BnCohortParams {
    FamiliesParams head;          // n_families = 0: es_cohort_head_kernel's column pass only
    const BnPlan *plans = nullptr;        // [P] deduplicated plans (device memory, like the arrays below)
    const int32_t *fam_plan = nullptr;    // [F] plan of each family, device order
    const int32_t *fam_col_off = nullptr; // [F] offset of its local -> global column map in `cols`
    const int32_t *cols = nullptr;        // concatenated column maps
    std::vector<BnCohortClass> classes;   // host side
};
// Dynamic shared memory of bn_cohort_kernel for a family of plan `pl`; the staged plan (sizeof(BnPlan)) is static.
size_t bn_cohort_smem_bytes(const BnPlan &pl);
// 2 + (launch classes) launches whatever the number of families: the head, one per class, the finish.  Handles B.pl and
// B.single == nullptr itself.
cudaError_t launch_bn_cohort(const BnCohortParams &P, const BatchPtrs &B, cudaStream_t stream);

// ---- Gibbs sampler (mcmc_kernel.cu) ---------------------------------------------------------------
struct McmcParams {
    RunConstants C;
    McmcPlan plan;
};
size_t mcmc_smem_bytes(const McmcParams &P, int tb);
int mcmc_pick_block(const McmcParams &P, size_t smem_limit, size_t smem_per_sm);
// Launch-time tuning, read from the environment once in fs_create (FAMSEQ_MCMC_BLOCKS, FAMSEQ_MCMC_WGLOBAL).
struct McmcTuning {
    int blocks_cap = 3; // resident blocks per SM when the own factors live in L2
    int wglobal = -1;   // own factors in L2 (1) / shared memory (0) / by pedigree size (-1)
};
// fixup: only variants whose status byte is 2 are processed (what the specialised kernel of gibbs_jit.cu left over);
// *fixup_count (device, may be null) is incremented once per such variant.
cudaError_t launch_mcmc(const McmcParams &P, const BatchPtrs &B, int tb, int burn, int rep, uint64_t seed,
                        int64_t v_offset, int sm_count, cudaStream_t stream, const McmcTuning &tune, bool fixup = false,
                        unsigned long long *fixup_count = nullptr);

// ---- Gibbs sampler, cohorts: every family's chain on its own (mcmc_cohort_kernel.cu) ----------------------------------
// Families of one launch class share the genotype-vector width gw (mcmc_cohort_width) and the block size tb; they are
// [begin, end) of the device order.  n_max, the class's largest family, sizes the shared memory.
struct McmcCohortClass {
    int32_t gw, tb, n_max;
    int32_t begin, end;
};
struct McmcCohortParams {
    FamiliesParams head;                  // n_families = 0: es_cohort_head_kernel's column pass only
    const McmcPlan *plans = nullptr;      // [P] deduplicated plans (device memory, like the arrays below)
    const int32_t *fam_plan = nullptr;    // [F] plan of each family, device order
    const int32_t *fam_col_off = nullptr; // [F] offset of its local -> global column map in `cols`
    const int32_t *fam_row_off = nullptr; // [F] offset of its local member -> global ped row map in `rows`
    const int32_t *cols = nullptr;        // concatenated column maps
    const int32_t *rows = nullptr;        // concatenated row maps
    std::vector<McmcCohortClass> classes; // host side
};
// Dynamic shared memory of mcmc_cohort_kernel for families of at most n members at block size tb (the staged plan and row /
// column maps, MCMC_COHORT_STATIC_SMEM bytes, are static).
size_t mcmc_cohort_smem_bytes(int n, int tb);
// mcmc_pick_block's rule for the cohort kernel: the block size that keeps the most chains resident per SM for families of
// at most n members; 0 when not even 32 chains fit.
int mcmc_cohort_pick_block(int n, size_t smem_limit, size_t smem_per_sm);
// 2 + (launch classes) launches whatever the number of families: the head, one per class, the finish.  Handles B.pl and
// B.single == nullptr itself.
cudaError_t launch_mcmc_cohort(const McmcCohortParams &P, const BatchPtrs &B, int burn, int rep, uint64_t seed, int64_t v_offset,
                               cudaStream_t stream);

// ---- compact input (engine.cu) ----------------------------------------------------------------------
// lk[k] = lut[pl[k]] for k < n: expands fs_run_pl input for the kernels that read FP64 likelihoods.
cudaError_t launch_pl_decode(const uint16_t *pl, const double *lut, double *lk, int64_t n, cudaStream_t stream);

// ---- Phred encoding of posteriors (phred_kernel.cu) --------------------------------------------------------
// out[k] = packed six-digit Phred code of p[k] (include/famseq_b200.h, FS_PHRED_*); values the device does not decide are
// appended to `fixes` (index0 + k, exact double), *n_fixes counts them even beyond `capacity`.
cudaError_t launch_phred_pack(const double *p, uint32_t *out, int64_t n, int64_t index0, struct ::fs_phred_fix *fixes, int64_t capacity,
                              unsigned long long *n_fixes, cudaStream_t stream);

} // namespace famseq
