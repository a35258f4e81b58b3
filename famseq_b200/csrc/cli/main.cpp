// main.cpp -- `FamSeq`: the reference's command line (src/FamSeq.cpp:28-156) in front of the B200 engine.
//
//   FamSeq vcf -vcfFile in.vcf -pedFile fam.ped -output out.vcf [-method 1|2|3] [-v|-a] [-mRate x] ...
//   FamSeq LK  -lkFile in.txt  -pedFile fam.ped -output out.txt [-lkType n|log10|ln|PS] ...
//   FamSeq -h
// Exit status: 255 (return -1) on fatal argument / file / pedigree errors, 0 otherwise, as the reference.
// Extensions: -method also accepts BN / ES / MCMC; -device k selects the GPU; -seed n keys the Gibbs sampler.
#include <cstdio>
#include <cstring>
#include <iostream>

#include <unistd.h>

#include "drivers.hpp"
#include "options.hpp"

using namespace famseq_cli;
using std::cout;
using std::endl;

static void usage_top() {
    cout << endl;
    cout << "Program: FamSeq (Sequence calling using pedigree information)" << endl;
    cout << "Version: 1.0.2 (B200-native engine)" << endl << endl;
    cout << "Usage:\tFamSeq <input type> [options]" << endl << endl;
    cout << "Input type: \tvcf\t\tinput vcf file" << endl;
    cout << "\t\tLK\t\tinput likelihood file" << endl;
    cout << endl;
    cout << "Type FamSeq -h for help." << endl;
    cout << endl;
}

static void usage_mode(const char *mode) {
    cout << endl;
    cout << "Usage:\tFamSeq " << mode << " [options]" << endl << endl;
    cout << "Call variants when the input data is in a vcf file." << endl;
    cout << endl;
    cout << "Type FamSeq -h for help." << endl;
}

static void help() {
    cout << "FamSeq: Version: 1.0.2 (B200-native engine)" << endl;
    cout << "Usage:\tFamSeq <input type> [options]" << endl << endl;
    cout << "FamSeq accepts two kinds of input files: vcf file and likelihood only format file. "
            "If the input is vcf file, type 'FamSeq vcf [options]' in the command line. "
            "Type 'FamSeq LK [options]' if the input is likelihood only format. The user can only use only of them."
         << endl << endl;
    cout << "Options:" << endl << endl;
    static const char *rows[][2] = {
        {"-vcfFile\t", "The name of input vcf file."},
        {"-lkFile\t\t", "The name of input likelihood only format file."},
        {"-lkType\t", "The likelihood type stored in the likelihood only format file. n:normal(default); log10: log10 scaled; ln: ln scaled; PS: phred scaled."},
        {"-pedFile\t", "The name of the file storing the pedigree information."},
        {"-output\t\t", "The name of output file"},
        {"-method\t\t", "Choose the method used in variant calling. 1(default): Bayesian network; 2: Elston-Stewart algorithm; 3: MCMC."},
        {"-mRate\t\t", "Mutation rate. The default value is 1e-7"},
        {"-v\t\t", "Only record the position at which the genotype is not RR in the output file. (R: reference allele, A: alternative allele)."},
        {"-a\t\t", "Record all the position in the output file."},
        {"-genoProbN\t", "Genotype probability of three kinds of genotype for autosome in population (Pr(G)) when the variant is not in dbSNP. The default value is:  0.9985, 0.001 and 0.0005. The dbSNP position should be provided in column ID in input vcf file. "},
        {"-genoProbK\t", "Genotype probability of three kinds of genotype for autosome in population (Pr(G)) when the variant is in dbSNP. The default value is: 0.45, 0.1 and 0.45."},
        {"-genoProbXN\t", "Genotype probability of two kinds of genotype for chromosome X for male in population (Pr(G)) when the variant is not in dbSNP. The default value is: 0.999 and 0.001."},
        {"-genoProbXK\t", "Genotype probability of two kinds of genotype for chromosome X for male in population (Pr(G)) when the variant is in dbSNP. The default value is: 0.5 and 0.5."},
        {"-numBurnIn\t", "Number of burn in when the user chooses the MCMC method. The default value is 1,000n, where n is the number of individuals in the pedigree. The default grows with the sample count: for a cohort ped file, give -numBurnIn and -numRep."},
        {"-numRep\t\t", "Number of iteration times when the user chooses MCMC method. The default value is 20,000n. With -method 3, a ped file of more than 128 individuals runs each family on its own chain, the whole file's chain restricted to that family (families of at most 128 members, loops allowed)."},
        {"-LRC\t\t", "Likelihood ratio criteria (default 1): the pedigree is ignored when every sample's largest normalised likelihood reaches it."},
        {"-l\t\t", "File of tab-separated 'chromosome position' lines; only these positions are processed (vcf mode)."},
        {"-device\t\t", "(this implementation) CUDA device to run on. The default is 0."},
        {"-seed\t\t", "(this implementation) Seed of the counter-based random number generator of the MCMC method. The default is 1."},
        {"-peelLoops\t", "(this implementation) With -method 1: compute the Bayesian network's exact posteriors by Elston-Stewart peeling with conditioned loop breakers instead of enumeration, so pedigrees with loops of more than 31 individuals (at most 128, at most 8 loop breakers) can be run. Posteriors equal those of -method 1 to 1e-9 relative; on a pedigree without loops the output is that of -method 2. Not with -familyBN."},
        {"-familyBN\t", "(this implementation) With -method 1: compute the Bayesian network of each family of the ped file on its own, for ped files of any size and families with loops (at most 31 members each). Members' posteriors equal those of the whole-file network except where its product of all members' probabilities leaves the double range."},
    };
    for (auto &r : rows) cout << r[0] << r[1] << endl << endl;
}

static int run(int argc, char *argv[]);

// Everything is written and closed when run() returns; leaving through _exit skips the CUDA runtime's tear-down of the
// context (0.3 - 1 s on a B200) and does not wait for a run-time compile that a short run no longer needs.
int main(int argc, char *argv[]) {
    const int rc = run(argc, argv);
    std::cout.flush();
    std::cerr.flush();
    std::fflush(nullptr);
    _exit(rc & 0xff);
}

static int run(int argc, char *argv[]) {
    if (argc == 1) {
        usage_top();
        return -1;
    }
    if (!std::strcmp(argv[1], "vcf")) {
        if (argc == 2) {
            usage_mode("vcf");
            return -1;
        }
        VcfOptions opt;
        const int rc = parse_vcf_options(argc, argv, opt);
        if (rc < 0) return -1;
        if (rc > 0) cout << "There are some improper parameters in the command line. Some parameters are set to default." << endl;
        PedRows ped;
        if (!read_ped(opt.ped_file, ped)) {
            cout << "Cannot read Ped file: " << opt.ped_file << "." << endl;
            cout << "Cannot set family." << endl;
            return -1;
        }
        if (!check_family(ped, opt.family_bn && opt.method == 1, opt.method == 3, opt.peel_loops && opt.method == 1)) {
            cout << "Cannot set family." << endl;
            return -1;
        }
        // like the reference, only the single-file case is implemented (FamSeq.cpp:78-86)
        if (opt.vcf_files.size() == 1 && !run_vcf(opt, ped) && g_engine_failed) return -1;
    } else if (!std::strcmp(argv[1], "LK")) {
        if (argc == 2) {
            usage_mode("LK");
            return -1;
        }
        LkOptions opt;
        const int rc = parse_lk_options(argc, argv, opt);
        if (rc < 0) return -1;
        if (rc > 0) cout << "There are some improper parameters in the command line. Some parameters are set to default." << endl;
        PedRows ped;
        if (!read_ped(opt.ped_file, ped)) {
            cout << "Cannot read Ped file: " << opt.ped_file << "." << endl;
            cout << "Cannot set Family." << endl;
            return -1;
        }
        if (!check_family(ped, opt.family_bn && opt.method == 1, opt.method == 3, opt.peel_loops && opt.method == 1)) {
            cout << "Cannot set Family." << endl;
            return -1;
        }
        if (!run_lk(opt, ped) && g_engine_failed) return -1;
    } else if (!std::strcmp(argv[1], "-h")) {
        help();
    } else {
        cout << "Cannot recognize the input type: \"" << argv[1] << "\"." << endl;
        cout << "The input type can only be vcf or LK" << endl;
        cout << endl;
        cout << "Type FamSeq -h for help." << endl;
        return -1;
    }
    return 0;
}
