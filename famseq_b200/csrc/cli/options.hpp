// options.hpp -- the FamSeq command line (re-created from the behaviour of the reference's
// checkInputVCF / checkInputLK, src/checkInput.cpp:149-578 and :671-1067).
//
// Grammar: argv[1] is the mode (vcf | LK | -h); every later token that starts with '-' is an option, so
// negative numbers cannot be option values.  Unknown options and stray values only warn.  Return value of
// the parsers: 0 ok, 1 "some parameters were set to default" (warning), -1 fatal.
#pragma once

#include <string>
#include <vector>

namespace famseq_cli {

struct CommonOptions {
    std::string ped_file, output;
    int method = 1;                 // -method 1 BN | 2 ES | 3 MCMC (aliases BN/ES/MCMC accepted as an extension)
    double mrate = 1e-7;            // -mRate, [0, 0.5]
    std::vector<double> geno_prob_n, geno_prob_k, geno_prob_xn, geno_prob_xk; // empty = engine default
    int num_burn_in = 0, num_rep = 0;
    double lrc = 1.0;               // -LRC
    // extensions of this implementation (absent from the reference):
    int device = 0;                 // -device k | a,b,c | all   CUDA device(s); a batch is split between several
    std::vector<int> devices;       //   (filled from -device; empty = {device})
    unsigned long long seed = 1;    // -seed n     Philox key of the Gibbs sampler
    bool peel_loops = false;        // -peelLoops  with -method 1: exact BN posteriors by conditioned peeling (FS_METHOD_BN_PEEL)
    bool family_bn = false;         // -familyBN   with -method 1: each family of the ped file is its own Bayesian network
};

struct VcfOptions : CommonOptions {
    std::vector<std::string> vcf_files;
    std::string location_file;      // -l
    bool var_only = false;          // -v
    bool all_line = false;          // -a
    bool pos_order = false;         // -o (parsed, unused -- as in the reference)
    bool diff_only = false;         // -d
};

struct LkOptions : CommonOptions {
    std::string lk_file;
    int lk_type = 1;                // -lkType n(1) log10(2) ln(3) PS(4)
};

int parse_vcf_options(int argc, char **argv, VcfOptions &out);
int parse_lk_options(int argc, char **argv, LkOptions &out);

} // namespace famseq_cli
