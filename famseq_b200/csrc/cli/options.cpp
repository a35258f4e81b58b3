// options.cpp -- see options.hpp.  One table-driven scanner serves both modes; the user-visible
// messages are the reference's (checkInput.cpp), including its inherited wording quirks.
#include "options.hpp"

#include <string>

#include <cstdlib>
#include <cstring>
#include <iostream>

namespace famseq_cli {
namespace {

struct Scanner {
    int argc;
    char **argv;
    int i = 2;
    int warn = 0;

    bool more() const { return i < argc; }
    // true when the token after the current option is a value (exists and does not start with '-')
    bool value_follows() const { return i + 1 < argc && argv[i + 1][0] != '-'; }
    const char *take() { return argv[++i]; }
};

int method_from(const char *s) {
    if (!std::strcmp(s, "BN") || !std::strcmp(s, "bn")) return 1;
    if (!std::strcmp(s, "ES") || !std::strcmp(s, "es")) return 2;
    if (!std::strcmp(s, "MCMC") || !std::strcmp(s, "mcmc")) return 3;
    return std::atoi(s);
}

// -genoProbN / -genoProbK take three numbers, -genoProbXN / -genoProbXK two (stored as a,0,b).  If a value is
// missing the whole option is dropped with a warning and scanning resumes at the offending token.
void read_prior(Scanner &sc, int count, const char *missing_msg, std::vector<double> &dst) {
    std::vector<double> v(3, 0.0);
    for (int k = 0; k < count; k++) {
        if (!sc.value_follows()) {
            std::cout << missing_msg << std::endl;
            sc.warn = 1;
            return;
        }
        const double x = std::atof(sc.take());
        if (count == 3)
            v[k] = x;
        else
            v[k == 0 ? 0 : 2] = x;
    }
    dst = v;
}

// Options shared by both modes.  Returns 1 when `opt` was consumed, 0 when it is not a common option,
// -1 on a fatal error.
int common_option(Scanner &sc, const std::string &opt, CommonOptions &o) {
    auto fatal_path = [&](const char *msg, std::string &dst) {
        if (!sc.value_follows()) {
            std::cout << msg << std::endl;
            return -1;
        }
        dst = sc.take();
        return 1;
    };
    if (opt == "pedFile") return fatal_path("The ped file hasn't been set. Please check input.", o.ped_file);
    if (opt == "output") return fatal_path("The output file hasn't been set. Please check input.", o.output);
    if (opt == "method") {
        if (!sc.value_follows()) {
            std::cout << "Method hasn't been set. The default method (BN) will be used." << std::endl;
            sc.warn = 1;
        } else
            o.method = method_from(sc.take());
        return 1;
    }
    if (opt == "mRate") {
        if (!sc.value_follows()) {
            std::cout << "Mutation rate hasn't been set. The default (1e-7) will be used." << std::endl;
            sc.warn = 1;
        } else
            o.mrate = std::atof(sc.take());
        return 1;
    }
    if (opt == "genoProbN") {
        read_prior(sc, 3, "genoProbN hasn't been set. The default (0.9985,0.001,0.0005) will be used.", o.geno_prob_n);
        return 1;
    }
    if (opt == "genoProbK") {
        read_prior(sc, 3, "genoProbK hasn't been set. The default (0.45,0.1,0.45) will be used.", o.geno_prob_k);
        return 1;
    }
    if (opt == "genoProbXN") {
        read_prior(sc, 2, "genoProbN hasn't been set. The default (0.999,0.001) will be used.", o.geno_prob_xn);
        return 1;
    }
    if (opt == "genoProbXK") {
        read_prior(sc, 2, "genoProbN hasn't been set. The default (0.5,0.5) will be used.", o.geno_prob_xk);
        return 1;
    }
    if (opt == "numBurnIn") {
        if (!sc.value_follows()) {
            std::cout << "Number of burn in times hasn't been set. The default 1000 will be used." << std::endl;
            sc.warn = 1;
        } else
            o.num_burn_in = std::atoi(sc.take());
        return 1;
    }
    if (opt == "numRep") {
        if (!sc.value_follows()) {
            std::cout << "Number of MCMC repeat times hasn't been set. The default 100000 will be used." << std::endl;
            sc.warn = 1;
        } else
            o.num_rep = std::atoi(sc.take());
        return 1;
    }
    if (opt == "LRC") {
        if (!sc.value_follows()) {
            std::cerr << "Likelihood ratio criteria is not set. The default will be used." << std::endl;
            sc.warn = 1;
        } else
            o.lrc = std::atof(sc.take());
        return 1;
    }
    // extensions
    if (opt == "device" && sc.value_follows()) { // k, a comma-separated list, or "all" (resolved by the driver: -1)
        const std::string v = sc.take();
        o.devices.clear();
        if (v == "all") {
            o.devices.push_back(-1);
        } else {
            size_t pos = 0;
            while (pos <= v.size()) {
                const size_t comma = v.find(',', pos);
                const std::string item = v.substr(pos, comma == std::string::npos ? std::string::npos : comma - pos);
                if (!item.empty()) o.devices.push_back(std::atoi(item.c_str()));
                if (comma == std::string::npos) break;
                pos = comma + 1;
            }
        }
        o.device = (o.devices.empty() || o.devices[0] < 0) ? 0 : o.devices[0];
        return 1;
    }
    if (opt == "familyBN") {
        o.family_bn = true;
        return 1;
    }
    if (opt == "peelLoops") {
        o.peel_loops = true;
        return 1;
    }
    if (opt == "seed" && sc.value_follows()) {
        o.seed = std::strtoull(sc.take(), nullptr, 10);
        return 1;
    }
    return 0;
}

void unknown(Scanner &sc, const char *tok, bool is_option) {
    if (is_option)
        std::cout << "Cannot recognize option: \"" << (tok + 1) << "\" in the command." << std::endl;
    else
        std::cout << "Cannot recognize parameter: \"" << tok << "\" in the command." << std::endl;
    sc.warn = 1;
}

void check_common(Scanner &sc, CommonOptions &o) {
    if (o.method < 1 || o.method > 3) {
        std::cout << "Method could only be 1 or 3. The default method (BN) will be used." << std::endl;
        o.method = 1;
        sc.warn = 1;
    }
    if (o.mrate < 0 || o.mrate > 0.5) {
        std::cout << "Mutation rate is set out of range. The default (1e-7) will be used." << std::endl;
        o.mrate = 1e-7;
        sc.warn = 1;
    }
}

void check_lrc(Scanner &sc, CommonOptions &o) {
    if (o.lrc < 0) {
        std::cerr << "Likelihood ration criteria is not set correctly. The default will be used." << std::endl;
        o.lrc = 1;
        sc.warn = 1;
    }
}

} // namespace

int parse_vcf_options(int argc, char **argv, VcfOptions &o) {
    Scanner sc{argc, argv};
    o.num_burn_in = -999; // "not given": resolved to 1000 * S / 20000 * S by the driver (file.cpp:644-656)
    o.num_rep = -999;
    for (; sc.more(); sc.i++) {
        const char *tok = argv[sc.i];
        if (tok[0] != '-') {
            unknown(sc, tok, false);
            continue;
        }
        const std::string opt(tok + 1);
        if (opt == "vcfFile") {
            if (!sc.value_follows()) {
                std::cout << "The vcf file hasn't been set. Please check input." << std::endl;
                return -1;
            }
            while (sc.value_follows()) o.vcf_files.push_back(sc.take());
        } else if (opt == "l") {
            if (!sc.value_follows()) {
                std::cout << "The location file hasn't been set. Please check input." << std::endl;
                return -1;
            }
            o.location_file = sc.take();
        } else if (opt == "v") {
            o.var_only = true;
        } else if (opt == "o") {
            o.pos_order = true;
        } else if (opt == "a") {
            o.all_line = true;
        } else if (opt == "d") {
            o.diff_only = true;
        } else {
            const int rc = common_option(sc, opt, o);
            if (rc < 0) return -1;
            if (rc == 0) unknown(sc, tok, true);
        }
    }
    if (o.vcf_files.empty()) {
        std::cout << "The name of vcf file must be set. Please input the vcf file name." << std::endl;
        return -1;
    }
    if (o.ped_file.empty()) {
        std::cout << "The name of ped file must be set. Please input the ped file name." << std::endl;
        return -1;
    }
    if (o.output.empty()) {
        std::cout << "The name of output file must be set. Please input the output file name." << std::endl;
        return -1;
    }
    check_common(sc, o);
    if (o.var_only && o.all_line) {
        std::cout << "varOnly is setted, allLine is blocked." << std::endl;
        o.all_line = false;
        sc.warn = 1;
    }
    if (o.num_burn_in < 0) {
        if (o.num_burn_in != -999) {
            std::cout << "Number of burn in cannot be less than 0. The default 1000*n will be used." << std::endl;
            sc.warn = 1;
        }
        o.num_burn_in = -1;
    }
    if (o.num_rep <= 0) {
        if (o.num_rep != -999) {
            std::cout << "Number of MCMC repeat times cannot be less than 1. The default 20000*n will be used." << std::endl;
            sc.warn = 1;
        }
        o.num_rep = -1;
    }
    check_lrc(sc, o);
    return sc.warn;
}

int parse_lk_options(int argc, char **argv, LkOptions &o) {
    Scanner sc{argc, argv};
    o.num_burn_in = 1000; // checkInput.cpp:683-684
    o.num_rep = 100000;
    for (; sc.more(); sc.i++) {
        const char *tok = argv[sc.i];
        if (tok[0] != '-') {
            unknown(sc, tok, false);
            continue;
        }
        const std::string opt(tok + 1);
        if (opt == "lkFile") {
            if (!sc.value_follows()) {
                std::cout << "The likelihood file hasn't been set. Please check input." << std::endl;
                return -1;
            }
            o.lk_file = sc.take();
        } else if (opt == "lkType") {
            if (!sc.value_follows()) {
                std::cout << "Likelihood type hasn't been set. The default normal(n) will be used." << std::endl;
                sc.warn = 1;
                continue;
            }
            const std::string t = sc.take();
            if (t == "n")
                o.lk_type = 1;
            else if (t == "log10")
                o.lk_type = 2;
            else if (t == "ln")
                o.lk_type = 3;
            else if (t == "PS")
                o.lk_type = 4;
            else {
                std::cout << "Cannot recognize the likelihood type: " << t << ". The default normal (n) will be used." << std::endl;
                o.lk_type = 1;
                sc.warn = 1;
            }
        } else {
            const int rc = common_option(sc, opt, o);
            if (rc < 0) return -1;
            if (rc == 0) unknown(sc, tok, true);
        }
    }
    if (o.lk_file.empty()) {
        std::cout << "The name of likelihood file must be set. Please input the likelihood file name." << std::endl;
        return -1;
    }
    if (o.ped_file.empty()) {
        std::cout << "The name of ped file must be set. Please input the ped file name." << std::endl;
        return -1;
    }
    if (o.output.empty()) {
        std::cout << "The name of output file must be set. Please input the output file name." << std::endl;
        return -1;
    }
    check_common(sc, o);
    if (o.num_burn_in < 0) {
        std::cout << "Number of burn in cannot be less than 0. The default 1000 will be used." << std::endl;
        o.num_burn_in = 1000;
        sc.warn = 1;
    }
    if (o.num_rep <= 0) {
        std::cout << "Number of MCMC repeat times cannot be less than 1. The default 100000 will be used." << std::endl;
        o.num_rep = 100000;
        sc.warn = 1;
    }
    check_lrc(sc, o);
    return sc.warn;
}

} // namespace famseq_cli
