// drivers.hpp -- the two record loops of the FamSeq command line, re-created around the batched engine:
// `FamSeq vcf` (reference: callGenoMVCF, src/file.cpp:108-1004) and `FamSeq LK` (callGenoLK, :1640-1886).
#pragma once

#include <string>
#include <vector>

#include "options.hpp"

namespace famseq_cli {

struct PedRows { // the five ped columns, file.cpp:24-62
    std::vector<int> id, mother_id, father_id, gender;
    std::vector<std::string> name;
};

bool read_ped(const std::string &path, PedRows &out);

// Checks the pedigree the way family::init does (half-specified parents, parent genders) before any output
// is written.  Prints the reference's messages; false = fatal.  family_bn (-familyBN -method 1): the ped file is checked
// as the cohort Bayesian-network engine takes it (every family on its own, loops allowed); mcmc (-method 3): a ped file past
// 128 members is checked as the cohort Gibbs sampler takes it (every family on its own, loops allowed).
// peel (-peelLoops -method 1): the pedigree must be one fs_create takes (at most 128 members, not with -familyBN) and its
// conditioned program must not be refused.
bool check_family(const PedRows &ped, bool family_bn, bool mcmc, bool peel);
// The engine method of the options: FS_METHOD_BN_PEEL for -method 1 -peelLoops, the -method value otherwise.
int engine_method(const CommonOptions &opt);

bool run_vcf(const VcfOptions &opt, const PedRows &ped);
bool run_lk(const LkOptions &opt, const PedRows &ped);

// Run statistics of the last driver call (written to stderr as one JSON line when FAMSEQ_STATS is set).
struct RunStats {
    long long records = 0, computed = 0, failed = 0, batches = 0;
    long long compact_batches = 0; // engine calls that shipped integer PL fields up and Phred codes down (fs_run_pl_phred)
    long long phred_fixes = 0;     // values of those the device left to the host formatter
    double parse_s = 0, engine_s = 0, kernel_ms = 0, write_s = 0, total_s = 0;
    double read_s = 0, start_wait_s = 0, drain_s = 0; // input file read, waiting for fs_create, waiting for the writer
    double alloc_s = 0, first_engine_s = 0;           // parts of engine_s: pinned buffers, the whole first block (first-use costs)
};
extern RunStats g_stats;

// True when the last run_* call failed inside the engine (CUDA error, pedigree refused by the chosen method):
// the command then exits 255.  File-open failures keep the reference's behaviour (message, exit status 0).
extern bool g_engine_failed;

} // namespace famseq_cli
