// engine.cu -- the C ABI of include/famseq_b200.h: engine life cycle, host-buffer pipeline and the
// dispatch to the three method kernels.  One engine drives one GPU; multi-GPU runs use one engine
// (one process, or one host thread) per device with the variants sharded between them.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <memory>
#include <cstdio>
#include <cstring>
#include <limits>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/famseq_b200.h"
#include "../host/families.hpp"
#include "../host/format_g.hpp"
#include "../host/pedigree.hpp"
#include "es_jit.hpp"
#include "gibbs_jit.hpp"
#include "kernels.hpp"

using namespace famseq;

static_assert((int)TAB_AUTO == (int)K_TAB_AUTO && (int)TAB_XF == (int)K_TAB_XF && (int)TAB_XM == (int)K_TAB_XM,
              "host and device table ids differ");

namespace {
thread_local std::string g_last_error;
int fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}
int cuda_fail(cudaError_t rc, const char *what) {
    return fail(FS_E_CUDA, std::string(what) + ": " + cudaGetErrorString(rc));
}
#define FS_CUDA(call)                                                                                        \
    do {                                                                                                     \
        cudaError_t rc__ = (call);                                                                           \
        if (rc__ != cudaSuccess) return cuda_fail(rc__, #call);                                              \
    } while (0)

constexpr int kPipelineDepth = 3;

struct DeviceChunk {
    cudaStream_t stream = nullptr;
    cudaEvent_t k0 = nullptr, k1 = nullptr;
    double *lk = nullptr, *post = nullptr, *single = nullptr; // lk / single are allocated when first needed
    uint16_t *pl = nullptr;
    uint32_t *post32 = nullptr, *single32 = nullptr; // Phred codes (fs_run_pl_phred), allocated when first needed
    uint8_t *flags = nullptr, *gt = nullptr, *status = nullptr;
    int64_t capacity = 0; // variants
    int64_t in_flight = 0;
};

// What one batch call reads and writes: FP64 likelihoods or compact PL input, `single` optional.
struct BatchIo {
    const double *lk = nullptr;
    const uint16_t *pl = nullptr;
    const uint8_t *flags = nullptr;
    double *post = nullptr, *single = nullptr;
    uint8_t *gt = nullptr, *status = nullptr;
    // compact output (fs_run_pl_phred): Phred codes instead of doubles, exceptions with their exact doubles
    uint32_t *post_phred = nullptr, *single_phred = nullptr;
    fs_phred_fix *fixes = nullptr;
    int64_t fix_capacity = 0;
    int64_t *n_fixes = nullptr;
    int64_t index_base = 0; // position of this batch's first value in the caller's arrays (multi-device slices)
    bool phred() const { return post_phred != nullptr; }
};

// Pedigree-specialised Gibbs kernel (gibbs_jit.cu).  FAMSEQ_MCMC_JIT: 0 = never, 1 = compile at the first MCMC batch and
// wait for it, unset = compile on a worker thread once a batch is large enough to be worth it and run the table-driven
// kernel until the cubin is ready (both kernels return the same bytes, so the switch is invisible).
// The compile job owns everything the worker touches, so an engine can be destroyed while the compiler is still
// running (the worker is detached and the job freed when it ends).
struct GibbsJitJob {
    enum { IDLE, COMPILING, COMPILED, FAILED, LOADED };
    McmcParams params;
    GibbsJitConfig cfg;
    std::string cubin, log, err;
    std::atomic<int> state{IDLE};
};
// The same for the generated Elston-Stewart kernel (es_jit.cu; pedigrees the nuclear-family kernel does not cover).
// FAMSEQ_ES_JIT: 0 = never, 1 = compile at the first ES batch, unset = on a worker thread after 2e10 variants (the
// interpreter does 1.5e9 variants/s, so only very long device-resident runs get there).
struct EsJitJob {
    enum { IDLE, COMPILING, COMPILED, FAILED, LOADED };
    EsParams params;
    std::string cubin, log, err;
    std::atomic<int> state{IDLE};
};
struct EsJitState {
    int mode = 2;
    double min_work = 2e10, work_seen = 0;
    std::shared_ptr<EsJitJob> job;
    std::thread worker;
    EsJitKernel *kernel = nullptr;
};
// Two generators (gibbs_jit.cu): [1] cached conditionals, fast where the chains sit still; [0] dense sweeps, whose speed does
// not depend on the data.  `pick` is the generator in use: it starts as the static choice of gibbs_jit_default_config and,
// unless FAMSEQ_JIT_CACHED fixes it, is settled by a pilot on the first large batch that is about to run the cached kernel:
// 256 sweeps over the first few thousand variants, counting how many groups the warps had to redo member by member.
struct GibbsJitState {
    int mode = 2;
    double min_work = 2e10; // Gibbs steps (variants x sweeps x members) seen by this engine before a compile is started
    double work_seen = 0;
    std::shared_ptr<GibbsJitJob> job[2];
    std::thread worker[2];
    GibbsJitKernel *kernel[2] = {nullptr, nullptr};
    int pick = -1;
    bool piloted = false;
    double pilot_serial_fraction = -1; // what the pilot measured (fs_get_info reports the generator)
    unsigned long long *d_vote_stats = nullptr;
};
// Uploads `v` to a new device array (nothing for an empty vector).
template <class T> cudaError_t upload(const std::vector<T> &v, const T **dst) {
    if (v.empty()) return cudaSuccess;
    T *d = nullptr;
    cudaError_t rc = cudaMalloc(&d, v.size() * sizeof(T));
    if (rc != cudaSuccess) return rc;
    *dst = d;
    return cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
}
} // namespace

struct fs_engine {
    Pedigree ped;
    fs_params params;
    RunConstants C;
    int device = -1;
    size_t smem_limit = 0;
    int sm_count = 0;

    EsParams es;
    int es_rc = FS_OK;
    std::string es_err;
    int es_tb = 0;
    NuclearParams nuclear;      // register-resident fast path for (father, mother, <= 5 childless children)
    bool is_nuclear = false;
    bool force_generic_es = false; // FAMSEQ_ES_GENERIC=1: run nuclear families through the message-program interpreter too

    BnParams bn;
    int bn_rc = FS_OK;
    std::string bn_err;

    BnPeelParams bn_peel; // FS_METHOD_BN_PEEL: the conditioned message program (host/bn_peel.hpp)
    int bn_peel_rc = FS_OK;
    std::string bn_peel_err;
    int bn_peel_tb = 0;

    McmcParams mcmc;
    int mcmc_rc = FS_OK;
    std::string mcmc_err;
    int mcmc_tb = 0;
    GibbsJitState jit;
    EsJitState es_jit;

    McmcTuning mcmc_tune;

    std::vector<double> pl_table;          // lut[pl] = pow(10, -pl/10), host libm (file.cpp:588-590)
    double *d_pl_table = nullptr;          // the same on the device, uploaded at the first fs_run_pl
    unsigned long long *d_fixups = nullptr; // chains redone by the table-driven kernel after the generated one
    fs_phred_fix *d_fixes = nullptr;        // Phred exceptions of the running call
    int64_t d_fix_capacity = 0;
    unsigned long long *d_n_fixes = nullptr;

    DeviceChunk chunk[kPipelineDepth];
    int64_t launches = 0, jit_launches = 0;
    int gibbs_generator = 0; // generated Gibbs kernel of the last MCMC launch: 0 none (table-driven), 1 dense sweeps, 2 cached conditionals
    double last_kernel_ms = 0;

    std::vector<fs_engine *> parts; // fs_create_multi: one single-device engine per GPU (this one then has device -1)

    // fs_create_families: a cohort of nuclear families and lone individuals, ES only (es_families_kernel.cu);
    // fs_create_cohort: families of any loop-free shape too, through per-family message programs (es_cohort_kernel.cu)
    bool families = false;
    FamilyTable fam_table;
    FamiliesParams fam; // its device arrays are owned by this engine
    CohortParams cohort; // fs_create_cohort with program families (cohort.n_pf > 0); its device arrays are owned too
    // fs_create_cohort_bn: every family enumerated on its own (bn_cohort_kernel.cu), BN only; its device arrays are owned too
    bool cohort_bn = false;
    BnCohortParams bn_cohort;
    // fs_create_cohort_mcmc: every family's Gibbs chain on its own (mcmc_cohort_kernel.cu), MCMC only; its device arrays are owned too
    bool cohort_mcmc = false;
    McmcCohortParams mcmc_cohort;
};

extern "C" {

void fs_default_params(fs_params *p) {
    if (!p) return;
    p->mrate = 1e-7;
    p->lrc = 1.0;
    const double n[3] = {0.9985, 0.001, 0.0005}, k[3] = {0.45, 0.1, 0.45};
    const double xn[3] = {0.999, 0, 0.001}, xk[3] = {0.5, 0, 0.5};
    std::memcpy(p->geno_prob_n, n, sizeof n);
    std::memcpy(p->geno_prob_k, k, sizeof k);
    std::memcpy(p->geno_prob_xn, xn, sizeof xn);
    std::memcpy(p->geno_prob_xk, xk, sizeof xk);
}

int fs_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

const char *fs_last_error(void) { return g_last_error.c_str(); }

int fs_warmup(int device) {
    FS_CUDA(cudaSetDevice(device));
    FS_CUDA(cudaFree(nullptr));
    return FS_OK;
}

static void release_chunks(fs_engine *e) {
    for (DeviceChunk &c : e->chunk) {
        cudaFree(c.lk);
        cudaFree(c.pl);
        cudaFree(c.post);
        cudaFree(c.single);
        cudaFree(c.post32);
        cudaFree(c.single32);
        cudaFree(c.flags);
        cudaFree(c.gt);
        cudaFree(c.status);
        if (c.k0) cudaEventDestroy(c.k0);
        if (c.k1) cudaEventDestroy(c.k1);
        if (c.stream) cudaStreamDestroy(c.stream);
        c = DeviceChunk();
    }
}

void fs_destroy(fs_engine *e) {
    if (!e) return;
    for (fs_engine *part : e->parts) fs_destroy(part);
    for (int g = 0; g < 2; g++)
        if (e->jit.worker[g].joinable()) { // do not wait for a compile nobody will use
            if (e->jit.job[g] && e->jit.job[g]->state.load(std::memory_order_acquire) == GibbsJitJob::COMPILING)
                e->jit.worker[g].detach();
            else
                e->jit.worker[g].join();
        }
    if (e->es_jit.worker.joinable()) {
        if (e->es_jit.job && e->es_jit.job->state.load(std::memory_order_acquire) == EsJitJob::COMPILING)
            e->es_jit.worker.detach();
        else
            e->es_jit.worker.join();
    }
    if (e->device >= 0) {
        cudaSetDevice(e->device);
        gibbs_jit_unload(e->jit.kernel[0]);
        gibbs_jit_unload(e->jit.kernel[1]);
        cudaFree(e->jit.d_vote_stats);
        es_jit_unload(e->es_jit.kernel);
        release_chunks(e);
        cudaFree(e->d_pl_table);
        cudaFree(e->d_fixups);
        cudaFree(e->d_fixes);
        cudaFree(e->d_n_fixes);
        cudaFree(const_cast<int32_t *>(e->fam.fam_col));
        cudaFree(const_cast<uint8_t *>(e->fam.fam_male));
        cudaFree(const_cast<uint8_t *>(e->fam.col_male));
        cudaFree(const_cast<uint32_t *>(e->cohort.words));
        for (const int32_t *a : {e->cohort.prog_off, e->cohort.prog_slots, e->cohort.prog_cols, e->cohort.pf_prog, e->cohort.pf_col_off, e->cohort.cols})
            cudaFree(const_cast<int32_t *>(a));
        cudaFree(const_cast<BnPlan *>(e->bn_cohort.plans));
        for (const int32_t *a : {e->bn_cohort.fam_plan, e->bn_cohort.fam_col_off, e->bn_cohort.cols}) cudaFree(const_cast<int32_t *>(a));
        cudaFree(const_cast<McmcPlan *>(e->mcmc_cohort.plans));
        for (const int32_t *a : {e->mcmc_cohort.fam_plan, e->mcmc_cohort.fam_col_off, e->mcmc_cohort.fam_row_off, e->mcmc_cohort.cols,
                                 e->mcmc_cohort.rows})
            cudaFree(const_cast<int32_t *>(a));
    }
    delete e;
}

static const char *creator(bool families, FamilyMode mode) {
    if (!families) return "fs_create";
    switch (mode) {
    case FamilyMode::BN: return "fs_create_cohort_bn";
    case FamilyMode::MCMC: return "fs_create_cohort_mcmc";
    case FamilyMode::ANY_SHAPE: return "fs_create_cohort";
    default: return "fs_create_families";
    }
}

// fs_create (families == false), and with families == true fs_create_families, fs_create_cohort, fs_create_cohort_bn or
// fs_create_cohort_mcmc by `mode`, on one device (-1: host side only).
static int create_engine(const fs_pedigree *ped, const fs_params *params, int device, bool families, FamilyMode mode, fs_engine **out) {
    const char *who = creator(families, mode);
    if (!ped || !out) return fail(FS_E_ARG, std::string(who) + ": null argument");
    *out = nullptr;
    fs_params prm;
    if (params)
        prm = *params;
    else
        fs_default_params(&prm);
    fs_engine *e = new (std::nothrow) fs_engine();
    if (!e) return fail(FS_E_NOMEM, "out of host memory");
    std::string err;
    int rc = build_pedigree(ped->n, ped->id, ped->mother_id, ped->father_id, ped->gender, ped->s, ped->cols,
                            e->ped, err);
    if (rc != FS_OK) {
        delete e;
        return fail(rc, err);
    }
    if (!families && e->ped.n > FS_MAX_MEMBERS) {
        delete e;
        return fail(FS_E_TOO_LARGE, "pedigree has more than " + std::to_string(FS_MAX_MEMBERS) + " members");
    }
    e->params = prm;
    e->device = device;

    // ---- per-run constants -----------------------------------------------------------------------
    RunConstants &C = e->C;
    std::memset(&C, 0, sizeof C);
    build_tables(prm.mrate, C.tab);
    std::memcpy(C.prior[0], prm.geno_prob_n, 24);
    std::memcpy(C.prior[1], prm.geno_prob_k, 24);
    std::memcpy(C.prior[2], prm.geno_prob_xn, 24);
    std::memcpy(C.prior[3], prm.geno_prob_xk, 24);
    C.lrc = prm.lrc;
    C.n = e->ped.n;
    C.s = e->ped.s();
    if (!families)
        for (int c = 0; c < C.s; c++) C.col_male[c] = (uint8_t)e->ped.male[e->ped.cols[c]];
    // calPostProbSingle fails the variant when ANY member's row sum is <= 0 (family.cpp:1433-1439);
    // for unsequenced members (lk = 1,1,1) that depends only on the prior vector in use.
    for (int f = 0; f < 4; f++) {
        const int known = f & 1, chrx = (f >> 1) & 1;
        bool bad = false;
        for (int i = 0; i < e->ped.n; i++) {
            if (e->ped.col_of[i] >= 0) continue;
            const double *pr = (chrx && e->ped.male[i]) ? C.prior[known ? 3 : 2] : C.prior[known ? 1 : 0];
            double r[3];
            for (int g = 0; g < 3; g++) r[g] = 1.0 * pr[g];
            double s = 0;
            for (int g = 0; g < 3; g++) s = s + r[g];
            if (s <= 0) bad = true;
        }
        C.unseq_fail[f] = bad;
    }

    // PL decode table: exactly the expression of the reference's VCF driver (file.cpp:588-590), evaluated by the host's libm
    e->pl_table.resize(FS_PL_TABLE_SIZE);
    for (int k = 0; k < FS_PL_TABLE_SIZE; k++) e->pl_table[k] = std::pow(10.0, -std::fabs((double)k) / 10.0);
    if (families) {
        rc = build_families(e->ped, ped->id, e->fam_table, err, mode);
        if (rc != FS_OK) {
            delete e;
            return fail(rc, err);
        }
        e->families = true;
        const FamilyTable &t = e->fam_table;
        e->fam.C = C;
        e->fam.n_families = t.n_peeled;
        e->fam.nc_max = t.nc_max;
        e->fam.group = es_families_group(C.s);
        std::memcpy(e->fam.class_end, t.class_end, sizeof t.class_end);
        e->bn_rc = e->mcmc_rc = FS_E_TOO_LARGE;
        e->bn_err = e->mcmc_err = "pedigree of " + std::to_string(e->ped.n) + " members in " + std::to_string(t.n_families()) +
                                  " families: only Elston-Stewart (-method 2) runs on ped files over " +
                                  std::to_string(FS_MAX_MEMBERS) + " members";
        e->mcmc_err += " (the Gibbs sampler on cohorts is fs_create_cohort_mcmc)";
        e->bn_peel_rc = FS_E_ARG;
        e->bn_peel_err = "conditioned peeling (method 4, -method 1 -peelLoops) runs on fs_create / fs_create_multi engines only, "
                         "not on " + std::string(who) + " engines";
        if (mode == FamilyMode::BN) {
            e->cohort_bn = true;
            e->bn_rc = FS_OK;
            e->es_rc = e->mcmc_rc = FS_E_ARG;
            e->es_err = e->mcmc_err = "pedigree of " + std::to_string(e->ped.n) + " members in " + std::to_string(t.n_families()) +
                                      " families: this engine runs the Bayesian network (-method 1) only; Elston-Stewart on "
                                      "cohorts is fs_create_cohort";
            // fs_get_info: the largest family's plan
            int big = 0;
            for (int q = 1; q < (int)t.plans.size(); q++)
                if (t.plans[q].n_levels > t.plans[big].n_levels) big = q;
            if (!t.plans.empty()) e->bn.plan = t.plans[big];
        }
        if (mode == FamilyMode::MCMC) {
            e->cohort_mcmc = true;
            e->mcmc_rc = FS_OK;
            e->es_rc = e->bn_rc = FS_E_ARG;
            e->es_err = e->bn_err = "pedigree of " + std::to_string(e->ped.n) + " members in " + std::to_string(t.n_families()) +
                                    " families: this engine runs the Gibbs sampler (-method 3) only; Elston-Stewart on cohorts is "
                                    "fs_create_cohort, the Bayesian network fs_create_cohort_bn";
            // fs_get_info: the largest family's plan
            int big = 0;
            for (int q = 1; q < (int)t.mcmc_plans.size(); q++)
                if (t.mcmc_plans[q].n > t.mcmc_plans[big].n) big = q;
            if (!t.mcmc_plans.empty()) e->mcmc.plan = t.mcmc_plans[big];
        }
    }

    // ---- pedigree compilers ----------------------------------------------------------------------
    if (!families) {
        e->es.C = C;
        e->es_rc = compile_es_program(e->ped, e->es.prog, e->es_err);
        { // nuclear family: exactly two founders who are the parents of every other member, nobody else has children
            const Pedigree &p = e->ped;
            int father = -1, mother = -1;
            bool ok = p.n >= 3 && p.n <= 2 + ES_NUCLEAR_MAX_CHILDREN && p.n_founders() == 2;
            for (int i = 0; ok && i < p.n; i++)
                if (!p.founder(i)) {
                    if (father < 0) {
                        father = p.father[i];
                        mother = p.mother[i];
                    }
                    ok = p.father[i] == father && p.mother[i] == mother && p.children[i].empty();
                }
            ok = ok && father >= 0 && p.founder(father) && p.founder(mother);
            if (ok) {
                NuclearParams &np = e->nuclear;
                std::memset(&np, 0, sizeof np);
                np.C = C;
                np.col_father = p.col_of[father];
                np.col_mother = p.col_of[mother];
                for (int i = 0; i < p.n; i++)
                    if (!p.founder(i)) {
                        np.col_child[np.n_children] = p.col_of[i];
                        np.male_child[np.n_children] = p.male[i];
                        np.n_children++;
                    }
                e->is_nuclear = true;
                np.allow_ident = 1;
                if (const char *env = std::getenv("FAMSEQ_ES_IDENT")) np.allow_ident = env[0] != '0';
                np.stream_tiles = 0;
                if (const char *env = std::getenv("FAMSEQ_ES_STREAM")) np.stream_tiles = std::max(-1, std::min(1 << 20, std::atoi(env)));
            }
            const char *env = std::getenv("FAMSEQ_ES_GENERIC");
            e->force_generic_es = env && env[0] == '1';
        }
        e->bn.C = C;
        e->bn_rc = build_bn_plan(e->ped, e->bn.plan, e->bn_err);
        e->bn_peel.C = C;
        e->bn_peel_rc = build_bn_peel_program(e->ped, e->bn_peel.peel, e->bn_peel_err);
        e->mcmc.C = C;
        e->mcmc_rc = build_mcmc_plan(e->ped, e->mcmc.plan, e->mcmc_err);
        if (const char *env = std::getenv("FAMSEQ_MCMC_JIT")) e->jit.mode = env[0] == '0' ? 0 : (env[0] == '1' ? 1 : 2);
        if (const char *env = std::getenv("FAMSEQ_JIT_MIN_WORK")) e->jit.min_work = std::atof(env);
        if (const char *env = std::getenv("FAMSEQ_ES_JIT")) e->es_jit.mode = env[0] == '0' ? 0 : (env[0] == '1' ? 1 : 2);
        if (const char *env = std::getenv("FAMSEQ_MCMC_BLOCKS")) e->mcmc_tune.blocks_cap = std::max(1, std::atoi(env));
        if (const char *env = std::getenv("FAMSEQ_MCMC_WGLOBAL")) e->mcmc_tune.wglobal = env[0] == '1';
    }

    if (device >= 0) {
        cudaError_t crc = cudaSetDevice(device);
        cudaDeviceProp prop;
        if (crc == cudaSuccess) crc = cudaGetDeviceProperties(&prop, device);
        if (crc != cudaSuccess) {
            delete e;
            return cuda_fail(crc, "fs_create: no usable CUDA device (there is no CPU fallback)");
        }
        if (prop.major < 10) {
            delete e;
            return fail(FS_E_CUDA, std::string("fs_create: device ") + prop.name + " is sm_" +
                                       std::to_string(prop.major * 10 + prop.minor) +
                                       "; this library carries sm_100a code only");
        }
        e->smem_limit = prop.sharedMemPerBlockOptin;
        e->sm_count = prop.multiProcessorCount;
        if (e->es_rc == FS_OK && !families) {
            e->es_tb = es_pick_block(e->es, e->smem_limit);
            if (e->es_tb == 0) {
                e->es_rc = FS_E_TOO_LARGE;
                e->es_err = "pedigree too large for the ES kernel: message scratch exceeds shared memory";
            }
        }
        if (e->bn_peel_rc == FS_OK && !families) {
            e->bn_peel_tb = bn_peel_pick_block(e->bn_peel, e->smem_limit);
            if (e->bn_peel_tb == 0) {
                e->bn_peel_rc = FS_E_TOO_LARGE;
                e->bn_peel_err = "pedigree too large for conditioned peeling (-method 1 -peelLoops): the vector file of " +
                                 std::to_string(e->bn_peel.peel.n_vectors) + " genotype vectors per variant exceeds shared memory";
            }
        }
        if (e->bn_rc == FS_OK && !families && bn_smem_bytes(e->bn) > e->smem_limit) {
            e->bn_rc = FS_E_TOO_LARGE;
            e->bn_err = "pedigree too large for the BN kernel: per-thread odometer state exceeds shared memory";
        }
        if (e->mcmc_rc == FS_OK && !families) {
            e->mcmc_tb = mcmc_pick_block(e->mcmc, e->smem_limit, prop.sharedMemPerMultiprocessor);
            if (e->mcmc_tb == 0) {
                e->mcmc_rc = FS_E_TOO_LARGE;
                e->mcmc_err = "pedigree too large for the MCMC kernel: chain state exceeds shared memory";
            }
        }
        if (families) { // the family table, structure-of-arrays
            const FamilyTable &t = e->fam_table;
            std::vector<uint8_t> col_male((size_t)C.s);
            for (int c = 0; c < C.s; c++) col_male[c] = (uint8_t)e->ped.male[e->ped.cols[c]];
            int32_t *d_col = nullptr;
            uint8_t *d_male = nullptr, *d_col_male = nullptr;
            crc = cudaMalloc(&d_col, std::max<size_t>(t.col.size(), 1) * sizeof(int32_t));
            if (crc == cudaSuccess) e->fam.fam_col = d_col, crc = cudaMalloc(&d_male, std::max<size_t>(t.male.size(), 1));
            if (crc == cudaSuccess) e->fam.fam_male = d_male, crc = cudaMalloc(&d_col_male, std::max<size_t>(col_male.size(), 1));
            if (crc == cudaSuccess) e->fam.col_male = d_col_male, crc = cudaMemcpy(d_col, t.col.data(), t.col.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
            if (crc == cudaSuccess) crc = cudaMemcpy(d_male, t.male.data(), t.male.size(), cudaMemcpyHostToDevice);
            if (crc == cudaSuccess) crc = cudaMemcpy(d_col_male, col_male.data(), col_male.size(), cudaMemcpyHostToDevice);
            if (crc == cudaSuccess && !t.pf_order.empty()) { // the program families
                CohortParams &P = e->cohort;
                P.fam = e->fam;
                P.n_pf = (int32_t)t.pf_order.size();
                P.max_vectors = t.max_vectors;
                // block size: es_pick_block's rule for the largest vector file of any program
                auto largest = std::make_unique<EsParams>();
                largest->C.s = t.max_vectors;
                P.tb = es_pick_block(*largest, e->smem_limit);
                if (P.tb == 0) {
                    int q = 0;
                    for (int k = 1; k < t.n_programs(); k++)
                        if (t.prog_cols[k] + t.prog_slots[k] > t.prog_cols[q] + t.prog_slots[q]) q = k;
                    const int32_t first_id = ped->id[std::find(t.family_of.begin(), t.family_of.end(), t.prog_family[q]) - t.family_of.begin()];
                    fs_destroy(e);
                    return fail(FS_E_TOO_LARGE, "ped file family of " + std::to_string(first_id) +
                                                    ": pedigree too large for the ES kernel: message scratch exceeds shared memory");
                }
                std::vector<int32_t> pf_prog, pf_col_off;
                for (int f : t.pf_order) {
                    pf_prog.push_back(t.program[f]);
                    pf_col_off.push_back(t.col_off[f]);
                }
                crc = upload(t.words, &P.words);
                if (crc == cudaSuccess) crc = upload(t.prog_off, &P.prog_off);
                if (crc == cudaSuccess) crc = upload(t.prog_slots, &P.prog_slots);
                if (crc == cudaSuccess) crc = upload(t.prog_cols, &P.prog_cols);
                if (crc == cudaSuccess) crc = upload(pf_prog, &P.pf_prog);
                if (crc == cudaSuccess) crc = upload(pf_col_off, &P.pf_col_off);
                if (crc == cudaSuccess) crc = upload(t.cols, &P.cols);
            }
            if (crc == cudaSuccess && e->cohort_bn) { // the plans, the column maps and the launch classes
                BnCohortParams &P = e->bn_cohort;
                P.head = e->fam;
                for (size_t q = 0; q < t.plans.size(); q++)
                    if (bn_cohort_smem_bytes(t.plans[q]) + sizeof(BnPlan) > e->smem_limit) {
                        const int32_t first_id = ped->id[std::find(t.family_of.begin(), t.family_of.end(), t.plan_family[q]) - t.family_of.begin()];
                        fs_destroy(e);
                        return fail(FS_E_TOO_LARGE, "ped file family of " + std::to_string(first_id) +
                                                        ": pedigree too large for the BN kernel: per-thread odometer state exceeds shared memory");
                    }
                std::vector<int32_t> fam_plan, fam_col_off;
                for (int f : t.plan_order) {
                    fam_plan.push_back(t.plan[f]);
                    fam_col_off.push_back(t.col_off[f]);
                }
                for (size_t k = 0, d = 0; k < t.plan_class_end.size(); k++) {
                    const BnPlan &first = t.plans[fam_plan[d]];
                    BnCohortClass c{first.u, first.independent, first.factor_leaves, first.group, (int32_t)d, t.plan_class_end[k], 0};
                    for (; (int32_t)d < c.end; d++) c.smem = std::max(c.smem, bn_cohort_smem_bytes(t.plans[fam_plan[d]]));
                    P.classes.push_back(c);
                }
                crc = upload(t.plans, &P.plans);
                if (crc == cudaSuccess) crc = upload(fam_plan, &P.fam_plan);
                if (crc == cudaSuccess) crc = upload(fam_col_off, &P.fam_col_off);
                if (crc == cudaSuccess) crc = upload(t.cols, &P.cols);
            }
            if (crc == cudaSuccess && e->cohort_mcmc) { // the plans, the column and row maps and the launch classes
                McmcCohortParams &P = e->mcmc_cohort;
                P.head = e->fam;
                std::vector<int32_t> fam_plan, fam_col_off, fam_row_off;
                for (int f : t.plan_order) {
                    fam_plan.push_back(t.plan[f]);
                    fam_col_off.push_back(t.col_off[f]);
                    fam_row_off.push_back(t.row_off[f]);
                }
                for (size_t k = 0, d = 0; k < t.plan_class_end.size(); k++) {
                    McmcCohortClass c{mcmc_cohort_width(t.mcmc_plans[fam_plan[d]].n), 0, 0, (int32_t)d, t.plan_class_end[k]};
                    int big = fam_plan[d];
                    for (; (int32_t)d < c.end; d++)
                        if (t.mcmc_plans[fam_plan[d]].n > c.n_max) c.n_max = t.mcmc_plans[big = fam_plan[d]].n;
                    c.tb = mcmc_cohort_pick_block(c.n_max, e->smem_limit, prop.sharedMemPerMultiprocessor);
                    if (c.tb == 0) {
                        const int32_t first_id = ped->id[std::find(t.family_of.begin(), t.family_of.end(), t.plan_family[big]) - t.family_of.begin()];
                        fs_destroy(e);
                        return fail(FS_E_TOO_LARGE, "ped file family of " + std::to_string(first_id) +
                                                        ": pedigree too large for the MCMC kernel: chain state exceeds shared memory");
                    }
                    P.classes.push_back(c);
                }
                crc = upload(t.mcmc_plans, &P.plans);
                if (crc == cudaSuccess) crc = upload(fam_plan, &P.fam_plan);
                if (crc == cudaSuccess) crc = upload(fam_col_off, &P.fam_col_off);
                if (crc == cudaSuccess) crc = upload(fam_row_off, &P.fam_row_off);
                if (crc == cudaSuccess) crc = upload(t.cols, &P.cols);
                if (crc == cudaSuccess) crc = upload(t.rows, &P.rows);
            }
            if (crc != cudaSuccess) {
                fs_destroy(e); // releases what was allocated
                return cuda_fail(crc, (std::string(who) + ": family table upload").c_str());
            }
        }
    }
    *out = e;
    return FS_OK;
}

int fs_create(const fs_pedigree *ped, const fs_params *params, int device, fs_engine **out) {
    return create_engine(ped, params, device, false, FamilyMode::NUCLEAR, out);
}

static int create_multi(const fs_pedigree *ped, const fs_params *params, const int *devices, int ndev, bool families, FamilyMode mode,
                        fs_engine **out) {
    const char *who = families ? creator(families, mode) : "fs_create_multi";
    if (!ped || !out || !devices || ndev < 1) return fail(FS_E_ARG, std::string(who) + ": null argument or no device");
    *out = nullptr;
    // a device may be listed more than once: every entry gets its own pipeline (streams, buffers) on that GPU
    for (int g = 0; g < ndev; g++)
        if (devices[g] < 0 && !(families && ndev == 1)) return fail(FS_E_ARG, std::string(who) + ": negative device");
    if (ndev == 1) return create_engine(ped, params, devices[0], families, mode, out);
    // the front engine holds the host side (pedigree, tables, info); the parts own the GPUs
    fs_engine *front = nullptr;
    int rc = create_engine(ped, params, -1, families, mode, &front);
    if (rc != FS_OK) return rc;
    for (int g = 0; g < ndev; g++) {
        fs_engine *part = nullptr;
        rc = create_engine(ped, params, devices[g], families, mode, &part);
        if (rc != FS_OK) {
            const std::string keep = g_last_error;
            fs_destroy(front);
            return fail(rc, keep);
        }
        front->parts.push_back(part);
    }
    *out = front;
    return FS_OK;
}

int fs_create_multi(const fs_pedigree *ped, const fs_params *params, const int *devices, int ndev, fs_engine **out) {
    return create_multi(ped, params, devices, ndev, false, FamilyMode::NUCLEAR, out);
}

int fs_create_families(const fs_pedigree *ped, const fs_params *params, const int *devices, int ndev, fs_engine **out) {
    return create_multi(ped, params, devices, ndev, true, FamilyMode::NUCLEAR, out);
}

int fs_create_cohort(const fs_pedigree *ped, const fs_params *params, const int *devices, int ndev, fs_engine **out) {
    return create_multi(ped, params, devices, ndev, true, FamilyMode::ANY_SHAPE, out);
}

int fs_create_cohort_bn(const fs_pedigree *ped, const fs_params *params, const int *devices, int ndev, fs_engine **out) {
    return create_multi(ped, params, devices, ndev, true, FamilyMode::BN, out);
}

int fs_create_cohort_mcmc(const fs_pedigree *ped, const fs_params *params, const int *devices, int ndev, fs_engine **out) {
    return create_multi(ped, params, devices, ndev, true, FamilyMode::MCMC, out);
}

int fs_get_families(const fs_engine *e, int32_t *family, int32_t *n_families, int32_t *n_children) {
    if (!e) return fail(FS_E_ARG, "fs_get_families: null engine");
    if (!e->families) return fail(FS_E_ARG, "fs_get_families: the engine was not made by fs_create_families or a cohort constructor");
    const FamilyTable &t = e->fam_table;
    if (family) std::memcpy(family, t.family_of.data(), t.family_of.size() * sizeof(int32_t));
    if (n_families) *n_families = t.n_families();
    if (n_children) std::memcpy(n_children, t.n_children.data(), t.n_children.size() * sizeof(int32_t));
    return FS_OK;
}

int fs_get_family_program(const fs_engine *e, int32_t f, uint32_t *words, int32_t capacity, int32_t *n_words, int32_t *n_slots,
                          int32_t *cols, int32_t *n_cols, int32_t *program) {
    if (!e) return fail(FS_E_ARG, "fs_get_family_program: null engine");
    if (!e->families) return fail(FS_E_ARG, "fs_get_family_program: the engine was not made by fs_create_families or fs_create_cohort");
    const FamilyTable &t = e->fam_table;
    if (f < 0 || f >= t.n_families()) return fail(FS_E_ARG, "fs_get_family_program: no family " + std::to_string(f));
    const int q = t.program.empty() ? -1 : t.program[f];
    const int nw = q < 0 ? 0 : (q + 1 < t.n_programs() ? t.prog_off[q + 1] : (int)t.words.size()) - t.prog_off[q];
    const int nc = q < 0 ? 0 : t.prog_cols[q];
    if (program) *program = q;
    if (n_words) *n_words = nw;
    if (n_slots) *n_slots = q < 0 ? 0 : t.prog_slots[q];
    if (n_cols) *n_cols = nc;
    if (words && nw) {
        if (capacity < nw) return fail(FS_E_ARG, "fs_get_family_program: buffer too small");
        std::memcpy(words, t.words.data() + t.prog_off[q], sizeof(uint32_t) * (size_t)nw);
    }
    if (cols && nc) std::memcpy(cols, t.cols.data() + t.col_off[f], sizeof(int32_t) * (size_t)nc);
    return FS_OK;
}

int fs_get_info(const fs_engine *e, fs_info *out) {
    if (!e || !out) return fail(FS_E_ARG, "fs_get_info: null argument");
    std::memset(out, 0, sizeof *out);
    out->n = e->ped.n;
    out->s = e->ped.s();
    out->n_founders = e->ped.n_founders();
    out->has_loop = e->ped.has_loop;
    out->es_ops = e->es_rc == FS_OK ? e->es.prog.n_ops : 0;
    out->es_slots = e->es_rc == FS_OK ? e->es.prog.n_slots : 0;
    out->bn_levels = e->bn_rc == FS_OK ? e->bn.plan.n_levels : 0;
    out->bn_group = e->bn_rc == FS_OK ? e->bn.plan.group : 0;
    out->mcmc_links = e->mcmc_rc == FS_OK ? e->mcmc.plan.n_links : 0;
    out->device = e->parts.empty() ? e->device : e->parts[0]->device;
    out->kernel_launches = e->launches;
    out->jit_launches = e->jit_launches;
    out->n_devices = e->parts.empty() ? (e->device >= 0 ? 1 : 0) : (int32_t)e->parts.size();
    out->gibbs_generator = e->parts.empty() ? e->gibbs_generator : e->parts[0]->gibbs_generator;
    for (const fs_engine *part : e->parts) {
        fs_info pi;
        const int rc = fs_get_info(part, &pi);
        if (rc != FS_OK) return rc;
        out->kernel_launches += pi.kernel_launches;
        out->jit_launches += pi.jit_launches;
        out->mcmc_fixups += pi.mcmc_fixups;
    }
    if (e->device >= 0 && e->d_fixups) {
        unsigned long long n = 0;
        FS_CUDA(cudaSetDevice(e->device));
        FS_CUDA(cudaMemcpy(&n, e->d_fixups, sizeof n, cudaMemcpyDeviceToHost));
        out->mcmc_fixups += (int64_t)n;
    }
    return FS_OK;
}

int fs_get_tables(const fs_engine *e, double *pcp2, double *pcp2_xf, double *pcp2_xm, int32_t *mother,
                  int32_t *father) {
    if (!e) return fail(FS_E_ARG, "fs_get_tables: null engine");
    if (pcp2) std::memcpy(pcp2, e->C.tab[TAB_AUTO], 27 * 8);
    if (pcp2_xf) std::memcpy(pcp2_xf, e->C.tab[TAB_XF], 27 * 8);
    if (pcp2_xm) std::memcpy(pcp2_xm, e->C.tab[TAB_XM], 27 * 8);
    for (int i = 0; i < e->ped.n; i++) {
        if (mother) mother[i] = e->ped.mother[i];
        if (father) father[i] = e->ped.father[i];
    }
    return FS_OK;
}

static int no_es_program(const fs_engine *e) {
    return fail(FS_E_TOO_LARGE, "pedigree of " + std::to_string(e->ped.n) + " members in " + std::to_string(e->fam_table.n_families()) +
                                    " families: peeled by the cohort kernel, which has no message program");
}

int fs_get_es_program(const fs_engine *e, uint32_t *words, int32_t capacity, int32_t *n_words, int32_t *n_slots) {
    if (!e) return fail(FS_E_ARG, "fs_get_es_program: null engine");
    if (e->families) return no_es_program(e);
    if (e->es_rc != FS_OK && e->es_rc != FS_E_TOO_LARGE) return fail(e->es_rc, e->es_err);
    const EsProgram &p = e->es.prog;
    if (n_words) *n_words = p.n_words;
    if (n_slots) *n_slots = p.n_slots;
    if (words) {
        if (capacity < p.n_words) return fail(FS_E_ARG, "fs_get_es_program: buffer too small");
        std::memcpy(words, p.words, sizeof(uint32_t) * (size_t)p.n_words);
    }
    return FS_OK;
}

int fs_get_bn_peel_program(const fs_engine *e, uint32_t *words, int32_t capacity, int32_t *n_words, int32_t *n_slots,
                           int32_t *breaker_rows, int32_t breaker_capacity, int32_t *n_breakers, int32_t *clamp_slots) {
    if (!e) return fail(FS_E_ARG, "fs_get_bn_peel_program: null engine");
    if (e->bn_peel_rc != FS_OK) return fail(e->bn_peel_rc, e->bn_peel_err);
    const BnPeelProgram &p = e->bn_peel.peel;
    if (n_words) *n_words = p.prog.n_words;
    if (n_slots) *n_slots = p.prog.n_slots;
    if (n_breakers) *n_breakers = p.n_breakers;
    if (words) {
        if (capacity < p.prog.n_words) return fail(FS_E_ARG, "fs_get_bn_peel_program: buffer too small");
        std::memcpy(words, p.prog.words, sizeof(uint32_t) * (size_t)p.prog.n_words);
    }
    if ((breaker_rows || clamp_slots) && breaker_capacity < p.n_breakers) return fail(FS_E_ARG, "fs_get_bn_peel_program: breaker buffer too small");
    for (int j = 0; j < p.n_breakers; j++) {
        if (breaker_rows) breaker_rows[j] = p.breaker_row[j];
        if (clamp_slots) {
            clamp_slots[2 * j] = p.clamp_base + j;
            clamp_slots[2 * j + 1] = p.clamp_base + p.n_breakers + j;
        }
    }
    return FS_OK;
}

int fs_get_gibbs_kernel(const fs_engine *e, int compile, char *text, size_t capacity, size_t *text_len, size_t *cubin_bytes) {
    if (!e) return fail(FS_E_ARG, "fs_get_gibbs_kernel: null engine");
    if (e->mcmc_rc != FS_OK) return fail(e->mcmc_rc, e->mcmc_err);
    const GibbsJitConfig cfg = gibbs_jit_default_config(e->mcmc);
    std::string out, cubin, err;
    if (compile) {
        const int rc = gibbs_jit_build(e->mcmc, cfg, cubin, out, err);
        if (rc != FS_OK) return fail(rc, err);
    } else {
        out = gibbs_jit_source(e->mcmc, cfg);
    }
    if (text_len) *text_len = out.size();
    if (cubin_bytes) *cubin_bytes = cubin.size();
    if (text && capacity) {
        const size_t n = std::min(capacity - 1, out.size());
        std::memcpy(text, out.data(), n);
        text[n] = 0;
    }
    return FS_OK;
}

int fs_get_es_kernel(const fs_engine *e, int compile, char *text, size_t capacity, size_t *text_len, size_t *cubin_bytes) {
    if (!e) return fail(FS_E_ARG, "fs_get_es_kernel: null engine");
    if (e->families) return no_es_program(e);
    if (e->es_rc != FS_OK) return fail(e->es_rc, e->es_err);
    if (!es_jit_fits(e->es, 227 * 1024))
        return fail(FS_E_TOO_LARGE, "pedigree too large for the generated ES kernel (the interpreter is used)");
    std::string out, cubin, err;
    if (compile) {
        const int rc = es_jit_build(e->es, cubin, out, err);
        if (rc != FS_OK) return fail(rc, err);
    } else {
        out = es_jit_source(e->es);
    }
    if (text_len) *text_len = out.size();
    if (cubin_bytes) *cubin_bytes = cubin.size();
    if (text && capacity) {
        const size_t n = std::min(capacity - 1, out.size());
        std::memcpy(text, out.data(), n);
        text[n] = 0;
    }
    return FS_OK;
}

int fs_get_pl_table(const fs_engine *e, double *out) {
    if (!e || !out) return fail(FS_E_ARG, "fs_get_pl_table: null argument");
    std::memcpy(out, e->pl_table.data(), sizeof(double) * FS_PL_TABLE_SIZE);
    return FS_OK;
}

void *fs_alloc_pinned(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void fs_free_pinned(void *p) {
    if (p) cudaFreeHost(p);
}

double fs_last_kernel_ms(const fs_engine *e) { return e ? e->last_kernel_ms : 0.0; }

// The Gibbs kernel of generator `which` if it is ready (loads it when the worker has finished, starts the worker when this
// batch is big enough); nullptr means: use the table-driven kernel for this batch.
static int gibbs_jit_poll(fs_engine *e, double work, int which, GibbsJitKernel **out) {
    GibbsJitState &J = e->jit;
    *out = nullptr;
    if (J.mode == 0) return FS_OK;
    J.work_seen += work;
    if (!J.job[which] && (J.mode == 1 || J.work_seen >= J.min_work)) {
        J.job[which] = std::make_shared<GibbsJitJob>();
        J.job[which]->params = e->mcmc;
        J.job[which]->cfg = gibbs_jit_config(e->mcmc, which);
        J.job[which]->state.store(GibbsJitJob::COMPILING, std::memory_order_release);
        std::shared_ptr<GibbsJitJob> job = J.job[which];
        auto build = [job]() {
            const int rc = gibbs_jit_build(job->params, job->cfg, job->cubin, job->log, job->err);
            job->state.store(rc == FS_OK ? GibbsJitJob::COMPILED : GibbsJitJob::FAILED, std::memory_order_release);
        };
        if (J.mode == 1)
            build();
        else
            J.worker[which] = std::thread(build);
    }
    if (!J.job[which]) return FS_OK;
    int st = J.job[which]->state.load(std::memory_order_acquire);
    if (st == GibbsJitJob::COMPILED) {
        if (J.worker[which].joinable()) J.worker[which].join();
        const int rc = gibbs_jit_load(e->mcmc, J.job[which]->cfg, J.job[which]->cubin, &J.kernel[which], J.job[which]->err);
        J.job[which]->cubin.clear();
        J.job[which]->cubin.shrink_to_fit();
        st = rc == FS_OK ? GibbsJitJob::LOADED : GibbsJitJob::FAILED;
        J.job[which]->state.store(st, std::memory_order_release);
    }
    if (st == GibbsJitJob::FAILED && J.mode == 1) return fail(FS_E_CUDA, "FAMSEQ_MCMC_JIT=1: " + J.job[which]->err);
    if (st == GibbsJitJob::LOADED) *out = J.kernel[which];
    return FS_OK;
}

// The pilot: the cached kernel on the head of the batch for 192 + 64 sweeps into throw-away outputs; *fraction receives the
// share of groups its warps redid member by member during the 64 sampling sweeps.  Synchronises the stream (once per engine).
static int gibbs_pilot(fs_engine *e, GibbsJitKernel *jk, const BatchPtrs &B, uint64_t seed, int64_t v_offset, cudaStream_t stream,
                       double *fraction) {
    GibbsJitState &J = e->jit;
    const int64_t n = std::min<int64_t>(B.V, 8192);
    const size_t S = (size_t)e->ped.s(), nd = std::max<size_t>((size_t)n * S * 3, 2) * sizeof(double);
    if (!J.d_vote_stats) FS_CUDA(cudaMalloc(&J.d_vote_stats, 2 * sizeof(unsigned long long)));
    double *post = nullptr, *single = nullptr;
    uint8_t *gt = nullptr, *status = nullptr;
    auto release = [&]() {
        cudaFree(post);
        cudaFree(single);
        cudaFree(gt);
        cudaFree(status);
    };
    cudaError_t rc = cudaMalloc(&post, nd);
    if (rc == cudaSuccess) rc = cudaMalloc(&single, nd);
    if (rc == cudaSuccess) rc = cudaMalloc(&gt, std::max<size_t>((size_t)n * S, 16));
    if (rc == cudaSuccess) rc = cudaMalloc(&status, (size_t)n);
    if (rc == cudaSuccess) rc = cudaMemsetAsync(J.d_vote_stats, 0, 2 * sizeof(unsigned long long), stream);
    BatchPtrs P{B.lk, B.flags, post, single, gt, status, n};
    if (rc == cudaSuccess) rc = gibbs_jit_launch(jk, P, 192, 64, seed, v_offset, e->sm_count, stream, J.d_vote_stats);
    unsigned long long stats[2] = {0, 0};
    if (rc == cudaSuccess) rc = cudaMemcpyAsync(stats, J.d_vote_stats, sizeof stats, cudaMemcpyDeviceToHost, stream);
    if (rc == cudaSuccess) rc = cudaStreamSynchronize(stream);
    release();
    if (rc != cudaSuccess) return cuda_fail(rc, "Gibbs pilot");
    e->launches++;
    *fraction = stats[1] ? (double)stats[0] / (double)stats[1] : 0.0;
    return FS_OK;
}

// The generated ES kernel if it is ready; nullptr means: use the interpreter for this batch.
static int es_jit_poll(fs_engine *e, double variants, EsJitKernel **out) {
    EsJitState &J = e->es_jit;
    *out = nullptr;
    if (J.mode == 0 || !es_jit_fits(e->es, e->smem_limit)) return FS_OK;
    J.work_seen += variants;
    if (!J.job && (J.mode == 1 || J.work_seen >= J.min_work)) {
        J.job = std::make_shared<EsJitJob>();
        J.job->params = e->es;
        J.job->state.store(EsJitJob::COMPILING, std::memory_order_release);
        std::shared_ptr<EsJitJob> job = J.job;
        auto build = [job]() {
            const int rc = es_jit_build(job->params, job->cubin, job->log, job->err);
            job->state.store(rc == FS_OK ? EsJitJob::COMPILED : EsJitJob::FAILED, std::memory_order_release);
        };
        if (J.mode == 1)
            build();
        else
            J.worker = std::thread(build);
    }
    if (!J.job) return FS_OK;
    int st = J.job->state.load(std::memory_order_acquire);
    if (st == EsJitJob::COMPILED) {
        if (J.worker.joinable()) J.worker.join();
        const int rc = es_jit_load(e->es, J.job->cubin, &J.kernel, J.job->err);
        J.job->cubin.clear();
        J.job->cubin.shrink_to_fit();
        st = rc == FS_OK ? EsJitJob::LOADED : EsJitJob::FAILED;
        J.job->state.store(st, std::memory_order_release);
    }
    if (st == EsJitJob::FAILED && J.mode == 1) return fail(FS_E_CUDA, "FAMSEQ_ES_JIT=1: " + J.job->err);
    if (st == EsJitJob::LOADED) *out = J.kernel;
    return FS_OK;
}

// The decode table on the device (uploaded once, at the first compact-input batch of this engine).
static int ensure_pl_table(fs_engine *e, cudaStream_t stream) {
    if (e->d_pl_table) return FS_OK;
    FS_CUDA(cudaMalloc(&e->d_pl_table, sizeof(double) * FS_PL_TABLE_SIZE));
    FS_CUDA(cudaMemcpyAsync(e->d_pl_table, e->pl_table.data(), sizeof(double) * FS_PL_TABLE_SIZE, cudaMemcpyHostToDevice, stream));
    FS_CUDA(cudaStreamSynchronize(stream)); // pl_table is pageable: do not leave a staged copy behind
    return FS_OK;
}

// Kernel launch(es) for `B.V` variants already on the device.  B.pl (compact input) and B.single == nullptr are
// handled by the nuclear-family kernel itself; every other kernel gets FP64 likelihoods (expanded into `lk_scratch`)
// and a place to put the individual-only posteriors (`single_scratch`); both scratch buffers are stream-ordered
// allocations when the caller (fs_run*_device) has none.
static int dispatch(fs_engine *e, int method, BatchPtrs B, int32_t burn, int32_t rep, uint64_t seed, int64_t v_offset,
                    cudaStream_t stream, double *lk_scratch = nullptr, double *single_scratch = nullptr) {
    if (B.V == 0) return FS_OK;
    if (method != FS_METHOD_ES && method != FS_METHOD_BN && method != FS_METHOD_MCMC && method != FS_METHOD_BN_PEEL)
        return fail(FS_E_ARG, "method must be 1 (BN), 2 (ES), 3 (MCMC) or 4 (BN by conditioned peeling)");
    if (method == FS_METHOD_ES && e->es_rc != FS_OK) return fail(e->es_rc, e->es_err);
    if (method == FS_METHOD_BN && e->bn_rc != FS_OK) return fail(e->bn_rc, e->bn_err);
    if (method == FS_METHOD_BN_PEEL && e->bn_peel_rc != FS_OK) return fail(e->bn_peel_rc, e->bn_peel_err);
    if (method == FS_METHOD_MCMC) {
        if (e->mcmc_rc != FS_OK) return fail(e->mcmc_rc, e->mcmc_err);
        if (burn < 0 || rep <= 0) return fail(FS_E_ARG, "MCMC needs burn >= 0 and rep >= 1");
    }
    if (B.pl) {
        const int rc = ensure_pl_table(e, stream);
        if (rc != FS_OK) return rc;
        B.lut = e->d_pl_table;
    }
    if (method == FS_METHOD_BN && e->cohort_bn) {
        FS_CUDA(launch_bn_cohort(e->bn_cohort, B, stream));
        e->launches += 2 + (int64_t)e->bn_cohort.classes.size();
        return FS_OK;
    }
    if (method == FS_METHOD_MCMC && e->cohort_mcmc) {
        FS_CUDA(launch_mcmc_cohort(e->mcmc_cohort, B, burn, rep, seed, v_offset, stream));
        e->launches += 2 + (int64_t)e->mcmc_cohort.classes.size();
        return FS_OK;
    }
    if (method == FS_METHOD_ES && e->families && e->cohort.n_pf > 0) {
        FS_CUDA(launch_es_cohort(e->cohort, B, stream));
        e->launches += 3;
        return FS_OK;
    }
    if (method == FS_METHOD_ES && e->families) {
        FS_CUDA(launch_es_families(e->fam, B, stream));
        e->launches++;
        return FS_OK;
    }
    const bool tma_ok = ((reinterpret_cast<uintptr_t>(B.gt) | reinterpret_cast<uintptr_t>(B.status) | reinterpret_cast<uintptr_t>(B.pl)) & 15u) == 0;
    if (method == FS_METHOD_ES && e->is_nuclear && tma_ok && !e->force_generic_es) {
        FS_CUDA(launch_es_nuclear(e->nuclear, B, stream));
        e->launches++;
        return FS_OK;
    }
    // ---- every other kernel: FP64 likelihoods in, individual-only posteriors out ------------------------------
    const size_t row_doubles = (size_t)B.V * (size_t)e->ped.s() * 3;
    double *owned_lk = nullptr, *owned_single = nullptr;
    auto release = [&]() {
        if (owned_lk) cudaFreeAsync(owned_lk, stream);
        if (owned_single) cudaFreeAsync(owned_single, stream);
    };
    if (B.pl) {
        if (!lk_scratch) {
            FS_CUDA(cudaMallocAsync(&owned_lk, std::max<size_t>(row_doubles, 2) * sizeof(double), stream));
            lk_scratch = owned_lk;
        }
        const cudaError_t rc = launch_pl_decode(B.pl, B.lut, lk_scratch, (int64_t)row_doubles, stream);
        if (rc != cudaSuccess) {
            release();
            return cuda_fail(rc, "launch_pl_decode");
        }
        e->launches++;
        B.lk = lk_scratch;
        B.pl = nullptr;
    }
    if (!B.single) {
        if (!single_scratch) {
            const cudaError_t rc = cudaMallocAsync(&owned_single, std::max<size_t>(row_doubles, 2) * sizeof(double), stream);
            if (rc != cudaSuccess) {
                release();
                return cuda_fail(rc, "cudaMallocAsync(single scratch)");
            }
            single_scratch = owned_single;
        }
        B.single = single_scratch;
    }
    cudaError_t krc = cudaSuccess;
    int frc = FS_OK;
    switch (method) {
    case FS_METHOD_ES: {
        EsJitKernel *jk = nullptr;
        if (tma_ok && !e->force_generic_es) frc = es_jit_poll(e, (double)B.V, &jk);
        if (frc != FS_OK) break;
        if (jk) {
            krc = es_jit_launch(jk, B, stream);
            e->jit_launches++;
        } else {
            krc = launch_es(e->es, B, e->es_tb, stream);
        }
        break;
    }
    case FS_METHOD_BN:
        krc = launch_bn(e->bn, B, e->sm_count, stream);
        break;
    case FS_METHOD_BN_PEEL:
        krc = launch_bn_peel(e->bn_peel, B, e->bn_peel_tb, stream);
        break;
    case FS_METHOD_MCMC: {
        GibbsJitState &J = e->jit;
        if (J.pick < 0) J.pick = gibbs_jit_default_config(e->mcmc).cached;
        GibbsJitKernel *jk = nullptr;
        const double work = (double)B.V * ((double)burn + rep) * e->ped.n;
        frc = gibbs_jit_poll(e, work, J.pick, &jk);
        if (frc != FS_OK) break;
        if (jk && J.pick == 1 && !J.piloted && !gibbs_jit_generator_forced() && B.V >= 2048 && (int64_t)burn + rep >= 1024) {
            // is this the data the cached kernel is made for?  (where the chains keep moving -- low coverage, Mendelian
            // inconsistencies -- its cache is always stale and the dense generator is ~8x faster)
            J.piloted = true;
            frc = gibbs_pilot(e, jk, B, seed, v_offset, stream, &J.pilot_serial_fraction);
            if (frc != FS_OK) break;
            if (J.pilot_serial_fraction > 0.4) {
                J.pick = 0;
                frc = gibbs_jit_poll(e, 0.0, 0, &jk);
                if (frc != FS_OK) break;
            }
        }
        if (jk) {
            // the specialised kernel covers chains whose weight sums stay positive normal numbers away from the exponent
            // limits; it marks the others with status 2 for a second pass of the table-driven kernel (counted in d_fixups)
            if (!e->d_fixups) {
                krc = cudaMalloc(&e->d_fixups, sizeof(unsigned long long));
                if (krc == cudaSuccess) krc = cudaMemset(e->d_fixups, 0, sizeof(unsigned long long));
                if (krc != cudaSuccess) break;
            }
            krc = gibbs_jit_launch(jk, B, burn, rep, seed, v_offset, e->sm_count, stream);
            if (krc == cudaSuccess)
                krc = launch_mcmc(e->mcmc, B, e->mcmc_tb, burn, rep, seed, v_offset, e->sm_count, stream, e->mcmc_tune, true, e->d_fixups);
            e->jit_launches++;
            e->launches++;
            e->gibbs_generator = 1 + J.pick;
        } else
            krc = launch_mcmc(e->mcmc, B, e->mcmc_tb, burn, rep, seed, v_offset, e->sm_count, stream, e->mcmc_tune);
        break;
    }
    }
    release();
    if (frc != FS_OK) return frc;
    if (krc != cudaSuccess) return cuda_fail(krc, "kernel launch");
    e->launches++;
    return FS_OK;
}

static int run_device(fs_engine *e, int method, int64_t V, const BatchIo &io, int32_t burn, int32_t rep, uint64_t seed,
                      int64_t v_offset, void *stream, const char *who) {
    if (!e) return fail(FS_E_ARG, std::string(who) + ": null engine");
    if (!e->parts.empty()) return fail(FS_E_ARG, std::string(who) + ": device buffers need a single-GPU engine (fs_create)");
    if (e->device < 0) return fail(FS_E_CUDA, "engine was created without a device (there is no CPU fallback)");
    if (V < 0 || (V > 0 && ((!io.lk && !io.pl) || !io.post || !io.gt || !io.status))) return fail(FS_E_ARG, std::string(who) + ": null buffer");
    if ((reinterpret_cast<uintptr_t>(io.lk) | reinterpret_cast<uintptr_t>(io.post) | reinterpret_cast<uintptr_t>(io.single)) & 15u)
        return fail(FS_E_ARG, std::string(who) + ": lk/post/single must be 16-byte aligned");
    FS_CUDA(cudaSetDevice(e->device));
    BatchPtrs B{io.lk, io.flags, io.post, io.single, io.gt, io.status, V};
    B.pl = io.pl;
    return dispatch(e, method, B, burn, rep, seed, v_offset, static_cast<cudaStream_t>(stream));
}

int fs_run_device(fs_engine *e, int method, int64_t V, const double *d_lk, const uint8_t *d_flags, int32_t burn,
                  int32_t rep, uint64_t seed, int64_t v_offset, double *d_post, double *d_single,
                  uint8_t *d_gt, uint8_t *d_status, void *stream) {
    BatchIo io;
    io.lk = d_lk, io.flags = d_flags, io.post = d_post, io.single = d_single, io.gt = d_gt, io.status = d_status;
    return run_device(e, method, V, io, burn, rep, seed, v_offset, stream, "fs_run_device");
}

int fs_run_pl_device(fs_engine *e, int method, int64_t V, const uint16_t *d_pl, const uint8_t *d_flags, int32_t burn,
                     int32_t rep, uint64_t seed, int64_t v_offset, double *d_post, double *d_single, uint8_t *d_gt,
                     uint8_t *d_status, void *stream) {
    BatchIo io;
    io.pl = d_pl, io.flags = d_flags, io.post = d_post, io.single = d_single, io.gt = d_gt, io.status = d_status;
    return run_device(e, method, V, io, burn, rep, seed, v_offset, stream, "fs_run_pl_device");
}

// Device buffers of the host pipeline: `cap` variants per slot; lk (FP64 input, or the expansion of compact input for the
// kernels that need it), pl and single only when this call uses them.
static int ensure_chunks(fs_engine *e, int64_t cap, bool need_lk, bool need_pl, bool need_single, bool need_post32 = false,
                         bool need_single32 = false) {
    const size_t S = (size_t)e->ped.s();
    for (DeviceChunk &c : e->chunk) {
        if (c.capacity < cap) {
            cudaStream_t st = c.stream;
            cudaEvent_t k0 = c.k0, k1 = c.k1;
            cudaFree(c.lk);
            cudaFree(c.pl);
            cudaFree(c.post);
            cudaFree(c.single);
            cudaFree(c.post32);
            cudaFree(c.single32);
            cudaFree(c.flags);
            cudaFree(c.gt);
            cudaFree(c.status);
            c = DeviceChunk();
            c.stream = st;
            c.k0 = k0;
            c.k1 = k1;
            if (!c.stream) FS_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
            if (!c.k0) FS_CUDA(cudaEventCreate(&c.k0));
            if (!c.k1) FS_CUDA(cudaEventCreate(&c.k1));
            const size_t nd = (size_t)cap * S * 3 * sizeof(double);
            FS_CUDA(cudaMalloc(&c.post, nd ? nd : 16));
            FS_CUDA(cudaMalloc(&c.flags, (size_t)cap));
            FS_CUDA(cudaMalloc(&c.gt, S ? (size_t)cap * S : 16));
            FS_CUDA(cudaMalloc(&c.status, (size_t)cap));
            c.capacity = cap;
        }
        const size_t nd = std::max<size_t>((size_t)c.capacity * S * 3 * sizeof(double), 16);
        if (need_lk && !c.lk) FS_CUDA(cudaMalloc(&c.lk, nd));
        if (need_single && !c.single) FS_CUDA(cudaMalloc(&c.single, nd));
        if (need_pl && !c.pl) FS_CUDA(cudaMalloc(&c.pl, std::max<size_t>((size_t)c.capacity * S * 3 * sizeof(uint16_t), 16)));
        if (need_post32 && !c.post32) FS_CUDA(cudaMalloc(&c.post32, nd / 2));
        if (need_single32 && !c.single32) FS_CUDA(cudaMalloc(&c.single32, nd / 2));
    }
    return FS_OK;
}

// The pipelined batch call of ONE GPU on host buffers.
static int run_host_one(fs_engine *e, int method, int64_t V, const BatchIo &io, int32_t burn, int32_t rep, uint64_t seed,
                        int64_t v_offset) {
    if (e->device < 0) return fail(FS_E_CUDA, "engine was created without a device (there is no CPU fallback)");
    if (V == 0) return FS_OK;
    FS_CUDA(cudaSetDevice(e->device));
    const size_t S = (size_t)e->ped.s();
    // Chunks of ~48 MB of FP64 likelihoods (a multiple of 1024 variants keeps every tile 16-byte aligned)
    // are cycled through kPipelineDepth streams so that the H2D copy of chunk k+1, the kernel of
    // chunk k and the D2H copy of chunk k-1 overlap.  The cohort kernel has no tiles: its chunks keep to ~48 MB
    // for rows of thousands of columns too (a multiple of 16 variants).
    const int64_t quantum = e->families ? 16 : 1024;
    int64_t cap = (int64_t)((48u << 20) / (S ? S * 24 : 24));
    cap = std::max<int64_t>(quantum, std::min<int64_t>(cap, 1 << 22)) & ~(quantum - 1);
    cap = std::min<int64_t>(cap, (V + quantum - 1) & ~(quantum - 1));
    // the kernel reads pl / skips single itself
    const bool fused = (method == FS_METHOD_ES && ((e->is_nuclear && !e->force_generic_es) || e->families)) ||
                       (method == FS_METHOD_BN && e->cohort_bn) || (method == FS_METHOD_MCMC && e->cohort_mcmc);
    const bool want_single = io.single != nullptr || io.single_phred != nullptr;
    int rc = ensure_chunks(e, cap, !io.pl || !fused, io.pl != nullptr, want_single || !fused, io.phred(), io.single_phred != nullptr);
    if (rc != FS_OK) return rc;
    if (io.phred()) { // exception list of this call
        const int64_t want = std::max<int64_t>(io.fix_capacity, 1);
        if (e->d_fix_capacity < want) {
            cudaFree(e->d_fixes);
            e->d_fixes = nullptr;
            e->d_fix_capacity = 0;
            FS_CUDA(cudaMalloc(&e->d_fixes, (size_t)want * sizeof(fs_phred_fix)));
            e->d_fix_capacity = want;
        }
        if (!e->d_n_fixes) FS_CUDA(cudaMalloc(&e->d_n_fixes, sizeof(unsigned long long)));
        FS_CUDA(cudaMemset(e->d_n_fixes, 0, sizeof(unsigned long long)));
    }

    e->last_kernel_ms = 0;
    auto drain = [&](DeviceChunk &c) -> int {
        if (!c.in_flight) return FS_OK;
        c.in_flight = 0;
        FS_CUDA(cudaStreamSynchronize(c.stream));
        float ms = 0;
        FS_CUDA(cudaEventElapsedTime(&ms, c.k0, c.k1));
        e->last_kernel_ms += ms;
        return FS_OK;
    };
    auto submit = [&](DeviceChunk &c, int64_t v0) -> int {
        const int64_t nv = std::min<int64_t>(cap, V - v0);
        const size_t nd = (size_t)nv * S * 3 * sizeof(double);
        c.in_flight = nv; // from here on the slot has work queued that touches the caller's buffers
        if (nd && io.pl)
            FS_CUDA(cudaMemcpyAsync(c.pl, io.pl + (size_t)v0 * S * 3, nd / 4, cudaMemcpyHostToDevice, c.stream));
        else if (nd)
            FS_CUDA(cudaMemcpyAsync(c.lk, io.lk + (size_t)v0 * S * 3, nd, cudaMemcpyHostToDevice, c.stream));
        if (io.flags) FS_CUDA(cudaMemcpyAsync(c.flags, io.flags + v0, (size_t)nv, cudaMemcpyHostToDevice, c.stream));
        BatchPtrs B{io.pl ? nullptr : c.lk, io.flags ? c.flags : nullptr, c.post, want_single ? c.single : nullptr, c.gt, c.status, nv};
        B.pl = io.pl ? c.pl : nullptr;
        FS_CUDA(cudaEventRecord(c.k0, c.stream));
        const int drc = dispatch(e, method, B, burn, rep, seed, v_offset + v0, c.stream, c.lk, c.single);
        if (drc != FS_OK) return drc;
        if (nd && io.phred()) { // Phred codes instead of doubles: 4 bytes per value cross PCIe
            const int64_t n3 = nv * (int64_t)S * 3, at = io.index_base + v0 * (int64_t)S * 3;
            FS_CUDA(launch_phred_pack(c.post, c.post32, n3, at, e->d_fixes, io.fix_capacity, e->d_n_fixes, c.stream));
            e->launches++;
            if (io.single_phred) {
                FS_CUDA(launch_phred_pack(c.single, c.single32, n3, at + FS_PHRED_FIX_SINGLE, e->d_fixes, io.fix_capacity, e->d_n_fixes, c.stream));
                e->launches++;
            }
        }
        FS_CUDA(cudaEventRecord(c.k1, c.stream));
        if (nd && io.phred()) {
            FS_CUDA(cudaMemcpyAsync(io.post_phred + (size_t)v0 * S * 3, c.post32, nd / 2, cudaMemcpyDeviceToHost, c.stream));
            if (io.single_phred)
                FS_CUDA(cudaMemcpyAsync(io.single_phred + (size_t)v0 * S * 3, c.single32, nd / 2, cudaMemcpyDeviceToHost, c.stream));
            FS_CUDA(cudaMemcpyAsync(io.gt + (size_t)v0 * S, c.gt, (size_t)nv * S, cudaMemcpyDeviceToHost, c.stream));
        } else if (nd) {
            FS_CUDA(cudaMemcpyAsync(io.post + (size_t)v0 * S * 3, c.post, nd, cudaMemcpyDeviceToHost, c.stream));
            if (io.single) FS_CUDA(cudaMemcpyAsync(io.single + (size_t)v0 * S * 3, c.single, nd, cudaMemcpyDeviceToHost, c.stream));
            FS_CUDA(cudaMemcpyAsync(io.gt + (size_t)v0 * S, c.gt, (size_t)nv * S, cudaMemcpyDeviceToHost, c.stream));
        }
        FS_CUDA(cudaMemcpyAsync(io.status + v0, c.status, (size_t)nv, cudaMemcpyDeviceToHost, c.stream));
        return FS_OK;
    };
    int slot = 0;
    for (int64_t v0 = 0; v0 < V && rc == FS_OK; v0 += cap, slot = (slot + 1) % kPipelineDepth) {
        DeviceChunk &c = e->chunk[slot];
        if ((rc = drain(c)) != FS_OK) break;
        rc = submit(c, v0);
    }
    if (rc != FS_OK) {
        // Something failed half way: copies into the caller's buffers may still be queued on the other slots.  Wait for
        // all of them (ignoring secondary errors) so that the caller may release its buffers, then report the first error.
        const std::string first = g_last_error;
        for (DeviceChunk &c : e->chunk)
            if (c.in_flight) {
                cudaStreamSynchronize(c.stream);
                c.in_flight = 0;
            }
        cudaGetLastError();
        return fail(rc, first);
    }
    for (DeviceChunk &c : e->chunk) {
        const int drc = drain(c);
        if (drc != FS_OK && rc == FS_OK) rc = drc; // keep draining the other slots
    }
    if (rc == FS_OK && io.phred()) { // the exceptions of the whole call
        unsigned long long n = 0;
        FS_CUDA(cudaMemcpy(&n, e->d_n_fixes, sizeof n, cudaMemcpyDeviceToHost));
        const int64_t have = std::min<int64_t>((int64_t)n, io.fix_capacity);
        if (have > 0) FS_CUDA(cudaMemcpy(io.fixes, e->d_fixes, (size_t)have * sizeof(fs_phred_fix), cudaMemcpyDeviceToHost));
        if (io.n_fixes) *io.n_fixes = (int64_t)n;
    }
    return rc;
}

// Host-buffer entry: argument checks, then one GPU, or (fs_create_multi) one contiguous slice per GPU on its own thread.
static int run_host(fs_engine *e, int method, int64_t V, const BatchIo &io, int32_t burn, int32_t rep, uint64_t seed,
                    int64_t v_offset, const char *who) {
    if (!e) return fail(FS_E_ARG, std::string(who) + ": null engine");
    if (V < 0 || (V > 0 && ((!io.lk && !io.pl) || (!io.post && !io.post_phred) || !io.gt || !io.status)))
        return fail(FS_E_ARG, std::string(who) + ": null buffer");
    if (io.phred() && (io.fix_capacity < 0 || (io.fix_capacity > 0 && !io.fixes))) return fail(FS_E_ARG, std::string(who) + ": bad exception buffer");
    if (io.n_fixes) *io.n_fixes = 0;
    if (e->parts.empty()) return run_host_one(e, method, V, io, burn, rep, seed, v_offset);
    const int G = (int)e->parts.size();
    const size_t S = (size_t)e->ped.s();
    std::vector<int> rcs(G, FS_OK);
    std::vector<std::string> errs(G);
    std::vector<std::vector<fs_phred_fix>> part_fixes(io.phred() ? G : 0);
    std::vector<int64_t> part_n(G, 0);
    auto work = [&](int g) {
        // slice boundaries on multiples of 1024 variants keep every GPU's tiles 16-byte aligned in the caller's buffers
        auto cut = [&](int k) { return k >= G ? V : std::min<int64_t>(V, (((V / G) * k) + 1023) & ~(int64_t)1023); };
        const int64_t a = cut(g), b = cut(g + 1);
        if (b <= a) return;
        BatchIo part = io;
        if (io.lk) part.lk = io.lk + (size_t)a * S * 3;
        if (io.pl) part.pl = io.pl + (size_t)a * S * 3;
        if (io.flags) part.flags = io.flags + a;
        if (io.post) part.post = io.post + (size_t)a * S * 3;
        if (io.single) part.single = io.single + (size_t)a * S * 3;
        if (io.phred()) {
            part.post_phred = io.post_phred + (size_t)a * S * 3;
            if (io.single_phred) part.single_phred = io.single_phred + (size_t)a * S * 3;
            part_fixes[g].resize((size_t)io.fix_capacity);
            part.fixes = part_fixes[g].data();
            part.n_fixes = &part_n[g];
            part.index_base = a * (int64_t)S * 3;
        }
        part.gt = io.gt + (size_t)a * S;
        part.status = io.status + a;
        rcs[g] = run_host_one(e->parts[g], method, b - a, part, burn, rep, seed, v_offset + a);
        if (rcs[g] != FS_OK) errs[g] = g_last_error; // thread-local: carry it to the caller's thread
    };
    std::vector<std::thread> threads;
    for (int g = 1; g < G; g++) threads.emplace_back(work, g);
    work(0);
    for (std::thread &t : threads) t.join();
    e->last_kernel_ms = 0;
    for (int g = 0; g < G; g++) e->last_kernel_ms = std::max(e->last_kernel_ms, e->parts[g]->last_kernel_ms);
    for (int g = 0; g < G; g++)
        if (rcs[g] != FS_OK) return fail(rcs[g], "device " + std::to_string(e->parts[g]->device) + ": " + errs[g]);
    if (io.phred()) { // the slices' exceptions, in slice order
        int64_t total = 0, stored = 0;
        for (int g = 0; g < G; g++) {
            const int64_t have = std::min<int64_t>(part_n[g], io.fix_capacity);
            for (int64_t k = 0; k < have && stored < io.fix_capacity; k++) io.fixes[stored++] = part_fixes[g][(size_t)k];
            total += part_n[g];
        }
        if (io.n_fixes) *io.n_fixes = total;
    }
    return FS_OK;
}

int fs_run(fs_engine *e, int method, int64_t V, const double *lk, const uint8_t *flags, int32_t burn, int32_t rep,
           uint64_t seed, int64_t v_offset, double *post, double *single, uint8_t *gt, uint8_t *status) {
    BatchIo io;
    io.lk = lk, io.flags = flags, io.post = post, io.single = single, io.gt = gt, io.status = status;
    return run_host(e, method, V, io, burn, rep, seed, v_offset, "fs_run");
}

int fs_run_pl(fs_engine *e, int method, int64_t V, const uint16_t *pl, const uint8_t *flags, int32_t burn, int32_t rep,
              uint64_t seed, int64_t v_offset, double *post, double *single, uint8_t *gt, uint8_t *status) {
    BatchIo io;
    io.pl = pl, io.flags = flags, io.post = post, io.single = single, io.gt = gt, io.status = status;
    return run_host(e, method, V, io, burn, rep, seed, v_offset, "fs_run_pl");
}

int fs_run_pl_phred(fs_engine *e, int method, int64_t V, const uint16_t *pl, const uint8_t *flags, int32_t burn, int32_t rep,
                    uint64_t seed, int64_t v_offset, uint32_t *post_phred, uint32_t *single_phred, uint8_t *gt, uint8_t *status,
                    fs_phred_fix *fixes, int64_t fix_capacity, int64_t *n_fixes) {
    BatchIo io;
    io.pl = pl, io.flags = flags, io.gt = gt, io.status = status;
    io.post_phred = post_phred, io.single_phred = single_phred, io.fixes = fixes, io.fix_capacity = fix_capacity, io.n_fixes = n_fixes;
    if (V > 0 && !post_phred) return fail(FS_E_ARG, "fs_run_pl_phred: null buffer");
    return run_host(e, method, V, io, burn, rep, seed, v_offset, "fs_run_pl_phred");
}

int fs_phred_encode(fs_engine *e, int64_t n, const double *p, uint32_t *out, fs_phred_fix *fixes, int64_t fix_capacity, int64_t *n_fixes) {
    if (!e) return fail(FS_E_ARG, "fs_phred_encode: null engine");
    if (!e->parts.empty()) e = e->parts[0];
    if (e->device < 0) return fail(FS_E_CUDA, "engine was created without a device (there is no CPU fallback)");
    if (n < 0 || (n > 0 && (!p || !out)) || fix_capacity < 0 || (fix_capacity > 0 && !fixes)) return fail(FS_E_ARG, "fs_phred_encode: bad argument");
    if (n_fixes) *n_fixes = 0;
    if (n == 0) return FS_OK;
    FS_CUDA(cudaSetDevice(e->device));
    double *d_p = nullptr;
    uint32_t *d_out = nullptr;
    fs_phred_fix *d_fix = nullptr;
    unsigned long long *d_n = nullptr, count = 0;
    auto release = [&]() {
        cudaFree(d_p);
        cudaFree(d_out);
        cudaFree(d_fix);
        cudaFree(d_n);
    };
    cudaError_t rc = cudaMalloc(&d_p, (size_t)n * sizeof(double));
    if (rc == cudaSuccess) rc = cudaMalloc(&d_out, (size_t)n * sizeof(uint32_t));
    if (rc == cudaSuccess) rc = cudaMalloc(&d_fix, (size_t)std::max<int64_t>(fix_capacity, 1) * sizeof(fs_phred_fix));
    if (rc == cudaSuccess) rc = cudaMalloc(&d_n, sizeof count);
    if (rc == cudaSuccess) rc = cudaMemset(d_n, 0, sizeof count);
    if (rc == cudaSuccess) rc = cudaMemcpy(d_p, p, (size_t)n * sizeof(double), cudaMemcpyHostToDevice);
    if (rc == cudaSuccess) rc = launch_phred_pack(d_p, d_out, n, 0, d_fix, fix_capacity, d_n, nullptr);
    if (rc == cudaSuccess) rc = cudaMemcpy(out, d_out, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    if (rc == cudaSuccess) rc = cudaMemcpy(&count, d_n, sizeof count, cudaMemcpyDeviceToHost);
    const int64_t have = std::min<int64_t>((int64_t)count, fix_capacity);
    if (rc == cudaSuccess && have > 0) rc = cudaMemcpy(fixes, d_fix, (size_t)have * sizeof(fs_phred_fix), cudaMemcpyDeviceToHost);
    release();
    if (rc != cudaSuccess) return cuda_fail(rc, "fs_phred_encode");
    e->launches++;
    if (n_fixes) *n_fixes = (int64_t)count;
    return FS_OK;
}

int fs_phred_text(uint32_t code, char *buf) {
    if (!buf) return -1;
    const uint32_t kind = code & (3u << 30);
    int n = 0;
    if (kind == FS_PHRED_FIX) {
        buf[0] = 0;
        return -1;
    }
    if (kind == FS_PHRED_ZERO) {
        buf[n++] = '0';
    } else if (kind == FS_PHRED_INF) {
        std::memcpy(buf, "99999", 5);
        n = 5;
    } else {
        n = famseq::emit_decimal6(buf, code & 0xfffffu, (int)((code >> 20) & 63u) - 32);
    }
    buf[n] = 0;
    return n;
}

int fs_phred_text_exact(double p, char *buf) { // file.cpp:702-749: -10*log10(p); +inf prints 99999, anything else its absolute value
    if (!buf) return -1;
    const double v = -10 * std::log10(p);
    std::string s;
    if (v == std::numeric_limits<double>::infinity())
        s = "99999";
    else
        famseq::append_g(s, std::fabs(v));
    std::memcpy(buf, s.c_str(), s.size() + 1);
    return (int)s.size();
}

} // extern "C"

// ---- compact input: lk[k] = lut[pl[k]] ----------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) pl_decode_kernel(const uint16_t *__restrict__ pl, const double *__restrict__ lut,
                                                        double *__restrict__ lk, int64_t n) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) lk[k] = __ldg(lut + pl[k]);
}
} // namespace

namespace famseq {
cudaError_t launch_pl_decode(const uint16_t *pl, const double *lut, double *lk, int64_t n, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const int grid = (int)std::min<int64_t>((n + 255) / 256, 148 * 16);
    pl_decode_kernel<<<grid, 256, 0, stream>>>(pl, lut, lk, n);
    return cudaGetLastError();
}
} // namespace famseq

// ---- FP64 roofline probe ----------------------------------------------------------------------------
// Register-resident DFMA chains (8 independent accumulators per thread): the measured FP64 peak that
// bench.py uses as the roofline denominator of the BN and MCMC kernels (MEASURED_PEAKS.json has none).
namespace {
__global__ void __launch_bounds__(256) fp64_probe_kernel(double *out, int iters, double a, double b) {
    double x0 = threadIdx.x * 1e-9, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    const double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 12345.678) out[0] = s; // never true; keeps the chains alive
}
} // namespace

extern "C" int fs_bench_fp64_tflops(int device, double *tflops) {
    if (!tflops) return fail(FS_E_ARG, "fs_bench_fp64_tflops: null argument");
    FS_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    FS_CUDA(cudaGetDeviceProperties(&prop, device));
    double *d = nullptr;
    FS_CUDA(cudaMalloc(&d, 8));
    cudaEvent_t e0, e1;
    FS_CUDA(cudaEventCreate(&e0));
    FS_CUDA(cudaEventCreate(&e1));
    const int iters = 4096, blocks = prop.multiProcessorCount * 8;
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        FS_CUDA(cudaEventRecord(e0));
        fp64_probe_kernel<<<blocks, 256>>>(d, iters, 1.0000001, 1e-9);
        FS_CUDA(cudaEventRecord(e1));
        FS_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        FS_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        const double flops = 2.0 * 64.0 * iters * 256.0 * blocks;
        if (rep > 0 && ms > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    *tflops = best;
    return FS_OK;
}
