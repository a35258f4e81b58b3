/* famseq_b200.h -- C ABI of the B200-native FamSeq posterior-genotype engine.
 *
 * This is the drop-in boundary for the reference's in-process seam `class family`
 * (/root/reference/src/family.h:62-390).  The reference is called once per variant from its
 * two record loops (src/file.cpp:595-682 / :833-920 for VCF, :1743-1806 for likelihood files);
 * this ABI is the batched equivalent: one call computes a whole block of variants on one GPU.
 *
 *   reference (per variant)                               this ABI (per batch)
 *   ----------------------------------------------------  -----------------------------------
 *   family(mem, mRate)            family.cpp:78-126       fs_create(ped, params, device, &eng)
 *   set_genoProb{N,K,XN,XK}       family.cpp:552-574        (fs_params.geno_prob_*)
 *   set_lc                        family.cpp:253-257        (fs_params.lrc)
 *   init / setRelation / checkPed family.cpp:221-238        (inside fs_create; same error rules)
 *   set_mapV2P / set_mapP2V       family.cpp:357-376        (fs_pedigree.cols)
 *   set_LK(N x 3)                 family.cpp:698-748      lk[V][S][3]   (sequenced columns only;
 *                                                           unsequenced members are (1,1,1))
 *   calPostProbBN(Known,chrType)  family.cpp:750-1124     fs_run(..., FS_METHOD_BN, ...)
 *   calPostProbPeeling(...)       family.cpp:1126-1403    fs_run(..., FS_METHOD_ES, ...)
 *   calPostProbMCMC(burn,rep,...) family.cpp:1932-2096    fs_run(..., FS_METHOD_MCMC, ...)
 *   bool return value             file.cpp:607-619        status[v] (1 = "hasn't been calculated")
 *   get_postProb(true)            family.cpp:576-604      post[V][S][3]
 *   get_postProbSingle(true)      family.cpp:606-634      single[V][S][3]
 *   get_postRlt()                 family.cpp:636-665      gt[V][S]  (0,1,2; 255 = the reference's -1)
 *   pow(10, -fabs(PL)/10)         file.cpp:588-590,       fs_run_pl(..., uint16 pl[V][S][3], ...): the caller ships
 *     (the VCF driver's decode)     :825-827                the integer PL fields, the device decodes them through
 *                                                           a table built on the host with the same libm call
 *
 * All entry points are plain C: pointers and sizes only.  Every function returns FS_OK (0) or a
 * negative FS_E_* code; fs_last_error() returns a thread-local message for the last failure.
 * There is no CPU fallback: without a usable sm_100 device fs_create fails with FS_E_CUDA.
 */
#ifndef FAMSEQ_B200_H_
#define FAMSEQ_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FS_ABI_VERSION 2

/* the CLI's -method 1|2|3; FS_METHOD_BN_PEEL is -method 1 -peelLoops.
 * FS_METHOD_BN_PEEL: the Bayesian network's answer -- each member's normalised exact marginal -- computed by Elston-Stewart
 * peeling with conditioned loop breakers (loop-cutset conditioning) instead of enumerating 3^n configurations, so it takes
 * looped pedigrees of any size fs_create takes (<= 128 members).  K breakers (K <= the pedigree's cycle rank, 0 for a
 * loop-free pedigree) each hand their marriages on loops to founder copies; the loop-free result is peeled once for each of
 * the 3^K genotype assignments of the breakers and the unnormalised marginals are added up.  Posteriors are those of
 * FS_METHOD_BN to 1e-9 relative; on a loop-free pedigree every output byte is that of FS_METHOD_ES.  Status 1 as BN: an
 * individual-only row sum <= 0, an unsequenced member's failing prior, or a member whose accumulated marginal sums to <= 0
 * (where the unscaled total likelihood underflows).  fs_create accepts the same pedigrees as without it; a run returns
 * FS_E_TOO_LARGE, with the reason, for a pedigree that needs more than 8 breakers, a program over ES_MAX_WORDS words or, on
 * a device, a vector file over shared memory.  Cohort engines refuse it with FS_E_ARG. */
enum fs_method { FS_METHOD_BN = 1, FS_METHOD_ES = 2, FS_METHOD_MCMC = 3, FS_METHOD_BN_PEEL = 4 };

enum fs_flag { FS_FLAG_KNOWN = 1, /* VCF ID != "."  (file.cpp:476-480) */
               FS_FLAG_CHRX = 2 /* CHROM in {X,chrX,CHRX} (file.cpp:482-486) */ };

enum fs_error {
    FS_OK = 0,
    FS_E_ARG = -1,          /* bad argument */
    FS_E_HALF_PARENTS = -2, /* exactly one parent known: "This is not a fulfill family" (family.cpp:318-322) */
    FS_E_GENDER = -3,       /* mother not female / father not male (family.cpp:204-219) */
    FS_E_LOOP = -4,         /* ES asked on a pedigree with a marriage/consanguinity loop (the reference crashes) */
    FS_E_TOO_LARGE = -5,    /* pedigree exceeds a kernel limit (message says which) */
    FS_E_CUDA = -6,         /* CUDA runtime failure or no sm_100 device */
    FS_E_NOMEM = -7
};

/* The ped rows (file.cpp:24-62) plus the input-column mapping built by the drivers
 * (file.cpp:204-223, :1673-1689). */
typedef struct fs_pedigree {
    int32_t n;                /* pedigree members (rows of the ped file)                              */
    const int32_t *id;        /* [n] individual id                                                    */
    const int32_t *mother_id; /* [n] mother's id, any id not present among `id` means "founder"       */
    const int32_t *father_id; /* [n]                                                                  */
    const int32_t *gender;    /* [n] 1 male, 2 female (anything else is treated as "not male")        */
    int32_t s;                /* sequenced input columns that matched a ped row                       */
    const int32_t *cols;      /* [s] ped row of each matched input column, in input-column order;
                               *     every ped row at most once                                        */
} fs_pedigree;

typedef struct fs_params {
    double mrate;           /* -mRate,     default 1e-7 (checkInput.cpp:157)           */
    double lrc;             /* -LRC,       default 1    (checkInput.cpp:167)           */
    double geno_prob_n[3];  /* -genoProbN, default 0.9985 0.001 0.0005 (family.cpp:97) */
    double geno_prob_k[3];  /* -genoProbK, default 0.45 0.1 0.45                       */
    double geno_prob_xn[3]; /* -genoProbXN a b -> (a,0,b), default 0.999 0 0.001       */
    double geno_prob_xk[3]; /* -genoProbXK a b -> (a,0,b), default 0.5 0 0.5           */
} fs_params;

typedef struct fs_engine fs_engine;

/* Fills *p with the reference defaults. */
void fs_default_params(fs_params *p);

/* Number of CUDA devices visible to the library (0 when there is none / no driver). */
int fs_device_count(void);

/* Builds the pedigree program (topology, transmission tables, ES message schedule, BN enumeration
 * plan, Gibbs neighbour lists) on the host and uploads it to `device`.  `device` < 0 builds the host
 * side only (no CUDA call is made; fs_run* then fail with FS_E_CUDA) -- used by CPU-only tests of the
 * pedigree compiler and by `FamSeq --check-ped`. */
int fs_create(const fs_pedigree *ped, const fs_params *params, int device, fs_engine **out);
void fs_destroy(fs_engine *e);

/* One engine that drives `ndev` GPUs (SURVEY section 8(b)/(e)): the pedigree program is replicated, every fs_run /
 * fs_run_pl call is cut into `ndev` contiguous slices of variants -- slice g = [g V/ndev, (g+1) V/ndev) on devices[g],
 * one host thread and one copy/compute pipeline per GPU -- and every GPU writes its slice of the caller's ordered
 * host buffers.  There is no inter-GPU collective; Gibbs streams are keyed by the global variant index, so the bytes
 * do not depend on ndev.  A device may be listed more than once (each entry is an independent pipeline on that GPU).
 * The *_device entry points need a single-GPU engine (FS_E_ARG otherwise). */
int fs_create_multi(const fs_pedigree *ped, const fs_params *params, const int *devices, int ndev, fs_engine **out);

/* A ped file of many unrelated families (a cohort), for Elston-Stewart.  The pedigree is split into its connected
 * families; each must be a lone individual or a nuclear family (two founders, 1..5 childless children of both, any
 * member unsequenced).  No limit on the total member count beyond memory.  Same validation and error codes as fs_create
 * for the ped rows themselves; a family of another shape is refused with FS_E_TOO_LARGE, the message naming its first ped
 * id.  Outputs are those of the reference peeling the whole file as one family: per-variant LRC gate and failure over all
 * samples.  ES only: BN / MCMC runs fail with FS_E_TOO_LARGE.  ndev == 1 gives a single-GPU engine (the *_device entry
 * points work, device -1 = host only); ndev > 1 slices batches like fs_create_multi. */
int fs_create_families(const fs_pedigree *ped, const fs_params *params, const int *devices, int ndev, fs_engine **out);
/* The same for cohorts whose families may have any shape: three generations, half-sibs, several spouses, sibships of six
 * or more.  Lone individuals and nuclear families (1..5 children) are peeled as by fs_create_families; every other family
 * is accepted when fs_create would run Elston-Stewart on it as a pedigree of its own (at most 128 members, no loop, a
 * message program within ES_MAX_WORDS and, on a device, a vector file that fits shared memory) and is peeled by its own
 * message program, compiled on its rows in file order with its sequenced members as columns in increasing input column.
 * Families of one shape and one sequencing pattern share one program.  Refusals name the family's first ped id
 * ("ped file family of <id>: ..."): FS_E_LOOP for a looped family, FS_E_TOO_LARGE for one over a limit.  Ped-row
 * validation, error codes, the whole-file LRC gate and failure rule, ES only and the device slicing are those of
 * fs_create_families.  A batch is three kernel launches (one without program families), whatever the number of families. */
int fs_create_cohort(const fs_pedigree *ped, const fs_params *params, const int *devices, int ndev, fs_engine **out);
/* The Bayesian network for cohort ped files: every family -- lone individuals, nuclear and extended families, looped
 * families too -- is enumerated on its own, with the plan fs_create builds for that family's rows alone (its rows in file
 * order, its sequenced members as columns in increasing input column); plans are shared by content.  The family split,
 * ped-row validation, error codes and device slicing are those of fs_create_cohort; no limit on the total member count.
 * Each member's FPP is its own family's normalised BN marginal: the reference's answer for the whole file, which
 * factorises by family, up to rounding -- it differs only where the whole-file product of every member's factor leaves
 * the double range and no single family's product does.  The whole-row rules are those of the cohort ES engines: the LRC
 * gate uses the pedigree for every sample once one sequenced sample asks for it, and a variant is NA for every sample
 * (status 1) when an individual-only row sum is <= 0, an unsequenced member's prior fails, or any member of any family
 * has a BN bin sum <= 0.  Refusals name the family ("ped file family of <first id>: ..."): FS_E_TOO_LARGE for a family
 * over BN_MAX_LEVELS (31) members or, on a device, one whose plan exceeds shared memory.  BN (-method 1) only: ES and
 * MCMC runs fail with FS_E_ARG (Elston-Stewart on cohorts is fs_create_cohort).  fs_get_info's bn_levels / bn_group
 * describe the largest family's plan.  A batch is 2 + (launch classes) kernel launches per chunk, whatever the number of
 * families: a launch class is the set of plans that share one kernel instantiation and block shape. */
int fs_create_cohort_bn(const fs_pedigree *ped, const fs_params *params, const int *devices, int ndev, fs_engine **out);
/* The Gibbs sampler (MCMC) for cohort ped files: every family -- lone individuals, nuclear and extended families, looped
 * families too -- runs its own chain, with the plan fs_create builds for that family's rows alone; plans are shared by
 * content.  The family split, ped-row validation, error codes and device slicing are those of fs_create_cohort_bn; no limit
 * on the total member count.  The chains are those of the whole file: fs_create's sampler visits the members in ped
 * order, a member's full conditional reads only its own family, and a member's random word depends only on (seed, global
 * site, sweep, global ped row).  So each family's chain, with its members swept in increasing ped row and its words drawn
 * with their global ped rows, is the whole-file chain restricted to that family, and the outputs are byte-identical to
 * fs_create's table-driven sampler (FAMSEQ_MCMC_JIT=0) on any file fs_create takes.  The whole-row rules are those of the
 * cohort ES engines: the LRC gate uses the pedigree for every sample once one sequenced sample asks for it, and a variant
 * is NA for every sample (status 1) when an individual-only row sum is <= 0, an unsequenced member's prior fails, or any
 * member of any family ends with a posterior row summing to <= 0.  Families with no sequenced member run their chains
 * too.  Refusals name the family ("ped file family of <first id>: ..."): FS_E_TOO_LARGE for a family over
 * MCMC_MAX_MEMBERS (128) members or, on a device, one whose chain state exceeds shared memory.  MCMC (-method 3) only:
 * ES and BN runs fail with FS_E_ARG (fs_create_cohort, fs_create_cohort_bn).  fs_get_info's mcmc_links describes the
 * largest family's plan, and gibbs_generator stays 0 (no generated kernel).  A batch is 2 + (launch classes) kernel
 * launches per chunk, whatever the number of families: a launch class is the set of families of one genotype-vector
 * width (at most 32, 64 or 128 members). */
int fs_create_cohort_mcmc(const fs_pedigree *ped, const fs_params *params, const int *devices, int ndev, fs_engine **out);
/* family[n]: family index of each ped row (families numbered by their first row); n_children[*n_families]: 0 for a lone
 * individual, the number of non-founder members for a family peeled by a program (fs_create_cohort) or enumerated by
 * fs_create_cohort_bn or run by fs_create_cohort_mcmc.  Either pointer may be NULL.  FS_E_ARG on an engine that fs_create
 * made. */
int fs_get_families(const fs_engine *e, int32_t *family, int32_t *n_families, int32_t *n_children);
/* Family f of an fs_create_cohort engine (numbered as in fs_get_families): the deduplicated message program it runs
 * (words: capacity in words; *n_words, *n_slots as fs_get_es_program), cols[*n_cols]: the global input column of each of
 * its local columns, *program: the program's index, or -1 for a family the nuclear kernel peels and for every family of an
 * fs_create_cohort_bn or fs_create_cohort_mcmc engine (then *n_words = 0 and *n_cols = 0).  Every pointer may be NULL.  Introspection: tests interpret the programs on the CPU. */
int fs_get_family_program(const fs_engine *e, int32_t f, uint32_t *words, int32_t capacity, int32_t *n_words, int32_t *n_slots,
                          int32_t *cols, int32_t *n_cols, int32_t *program);

/* Thread-local text of the last error raised on the calling thread. */
const char *fs_last_error(void);

/* Blocking batch call on HOST buffers (pinned memory recommended; see fs_alloc_pinned).
 *   lk      [V][S][3] FP64 raw likelihoods Pr(D|G), input-column order
 *   flags   [V]       FS_FLAG_* bits (NULL = all zero, as the LK driver does, file.cpp:1751)
 *   burn, rep         Gibbs burn-in / sampling sweeps (ignored for BN, ES)
 *   seed, v_offset    Philox key and global index of variant 0: variant v draws from the stream
 *                     keyed (seed, v_offset + v), so any sharding of the input gives identical bytes
 *   post, single [V][S][3], gt [V][S], status [V]   outputs (see the table above)
 *   single may be NULL: the individual-only posteriors are then neither stored nor copied back (a caller can
 *   recompute them from the likelihoods alone: single = lk * prior / sum, family.cpp:1405-1499)
 * The call is internally pipelined (H2D / kernel / D2H on separate streams).  On any error every copy already
 * queued into the caller's buffers has completed before the call returns. */
int fs_run(fs_engine *e, int method, int64_t V, const double *lk, const uint8_t *flags, int32_t burn,
           int32_t rep, uint64_t seed, int64_t v_offset, double *post, double *single, uint8_t *gt,
           uint8_t *status);

/* Same computation on DEVICE buffers, enqueued on `stream` (a cudaStream_t, NULL = default stream) and
 * not synchronised: this is the kernel-only path that bench.py times with CUDA events.  d_lk, d_post and d_single must be
 * 16-byte aligned (FS_E_ARG otherwise; cudaMalloc'ed arrays are); the byte arrays (flags, gt, status, and pl below) may
 * have any alignment -- 16-byte aligned ones take the kernels that move whole tiles with the copy engine. */
int fs_run_device(fs_engine *e, int method, int64_t V, const double *d_lk, const uint8_t *d_flags, int32_t burn,
                  int32_t rep, uint64_t seed, int64_t v_offset, double *d_post, double *d_single,
                  uint8_t *d_gt, uint8_t *d_status, void *stream);

/* Compact input (SURVEY section 8(f) rank 2, input half).  The reference's VCF driver turns every PL (or GL) field x
 * into the likelihood pow(10, -fabs(x)/10) (file.cpp:588-590, :825-827).  For the usual integer PL fields the caller
 * can ship the integers themselves: pl[V][S][3], uint16, 2 bytes per value instead of 8.  The engine decodes them on
 * the device through a 65 536-entry table that fs_create fills ON THE HOST with exactly that libm expression, so the
 * likelihoods -- and therefore every output byte -- are identical to fs_run on the decoded doubles.  Values above
 * 65 535 may be clamped to 65 535 by the caller (every PL >= 3240 decodes to exactly 0.0); missing samples are
 * (0, 0, 0) = likelihood (1, 1, 1) (file.cpp:802-811).  Non-integer or GL input takes fs_run.  `single` may be NULL. */
int fs_run_pl(fs_engine *e, int method, int64_t V, const uint16_t *pl, const uint8_t *flags, int32_t burn, int32_t rep,
              uint64_t seed, int64_t v_offset, double *post, double *single, uint8_t *gt, uint8_t *status);
int fs_run_pl_device(fs_engine *e, int method, int64_t V, const uint16_t *d_pl, const uint8_t *d_flags, int32_t burn,
                     int32_t rep, uint64_t seed, int64_t v_offset, double *d_post, double *d_single, uint8_t *d_gt,
                     uint8_t *d_status, void *stream);
/* Copies the decode table (65 536 doubles) the engine uses; works on host-only engines (tests compare it with libm). */
int fs_get_pl_table(const fs_engine *e, double *out);
#define FS_PL_TABLE_SIZE 65536

/* Compact output (SURVEY section 8(f) rank 2, output half).  The reference's drivers print a posterior p as
 * fabs(-10 * log10(p)) with ostream's default formatting ("%g", six significant digits), or 99999 when that is +inf
 * (file.cpp:702-761, :938-997, :1814-1873).  fs_run_pl_phred delivers exactly that, 4 bytes per value instead of 8: the
 * six decimal digits and the decimal exponent the text is made of, computed on the device.
 *   bits  0-19  m    six-digit integer 100000 .. 999999                         (kind FS_PHRED_NUMBER)
 *   bits 20-25  e+32 decimal exponent of the leading digit: value = m * 10^(e-5)
 *   bits 30-31  kind FS_PHRED_NUMBER 0 | FS_PHRED_ZERO (p = 1, prints "0") | FS_PHRED_INF (p = 0, prints "99999") |
 *                    FS_PHRED_FIX: the device did not decide this one (it sits within 3e-8 of a rounding boundary in the
 *                    sixth digit, where glibc's and CUDA's log10 could round differently, or p is not in [0, 1]); its index
 *                    and exact double come back in `fixes` and the host formats it the reference's way.  ~6 in 10^8.
 * fs_phred_text() turns a code into the text; tests compare it with the reference's formatting of the FP64 results. */
#define FS_PHRED_NUMBER 0u
#define FS_PHRED_ZERO (1u << 30)
#define FS_PHRED_INF (2u << 30)
#define FS_PHRED_FIX (3u << 30)
typedef struct fs_phred_fix {
    int64_t index; /* position in the [V][S][3] array; + FS_PHRED_FIX_SINGLE for an entry of `single_phred` */
    double p;      /* the exact probability */
} fs_phred_fix;
#define FS_PHRED_FIX_SINGLE ((int64_t)1 << 62)
/* Like fs_run_pl, with the posteriors Phred-encoded: post_phred, single_phred [V][S][3] uint32 (single_phred may be
 * NULL).  Up to `fix_capacity` exceptions are written to `fixes`; *n_fixes receives how many there were -- when it exceeds
 * the capacity the caller has to repeat the call with more room (or take fs_run_pl). */
int fs_run_pl_phred(fs_engine *e, int method, int64_t V, const uint16_t *pl, const uint8_t *flags, int32_t burn, int32_t rep,
                    uint64_t seed, int64_t v_offset, uint32_t *post_phred, uint32_t *single_phred, uint8_t *gt, uint8_t *status,
                    fs_phred_fix *fixes, int64_t fix_capacity, int64_t *n_fixes);
/* The encoder on its own: n probabilities on the HOST in, n codes out (device round trip inside). */
int fs_phred_encode(fs_engine *e, int64_t n, const double *p, uint32_t *out, fs_phred_fix *fixes, int64_t fix_capacity, int64_t *n_fixes);
/* Text of a code (at most 13 characters + NUL) into buf; returns its length, or -1 for FS_PHRED_FIX.  Host only. */
int fs_phred_text(uint32_t code, char *buf);
/* The reference's text of one probability (the formatting fs_phred_fix entries need): libm log10 + "%g".  Host only. */
int fs_phred_text_exact(double p, char *buf);

/* Introspection of the compiled pedigree program (all fields are counts). */
typedef struct fs_info {
    int32_t n, s;             /* members, sequenced columns                                          */
    int32_t n_founders;       /*                                                                      */
    int32_t has_loop;         /* 1 when the marriage graph has a cycle (ES unavailable)               */
    int32_t es_ops;           /* message-program length                                               */
    int32_t es_slots;         /* FP64 3-vectors of per-variant scratch the ES program needs           */
    int32_t bn_levels;        /* enumeration depth (= n)                                              */
    int32_t bn_group;         /* threads cooperating on one variant in the BN kernel                  */
    int32_t mcmc_links;       /* parent-child links visited per Gibbs sweep                           */
    int32_t device;           /* CUDA device or -1                                                    */
    int64_t kernel_launches;  /* kernels launched by this engine so far                               */
    int64_t jit_launches;     /* ... of which launches of the run-time compiled Gibbs / ES kernels    */
    int64_t mcmc_fixups;      /* chains the generated Gibbs kernel handed back (status 2) and the table-driven
                               * kernel redid; read from the device, so only exact once the work has completed */
    int32_t n_devices;        /* GPUs behind this engine (fs_create_multi), 1 for fs_create, 0 host-only        */
    int32_t gibbs_generator;  /* Gibbs kernel of the last MCMC launch: 0 table-driven, 1 generated dense sweeps,
                               * 2 generated cached conditionals (csrc/cuda/gibbs_jit.cu)                        */
} fs_info;
int fs_get_info(const fs_engine *e, fs_info *out);

/* Copies the 3 x 27 transmission tables [g][mother][father] (autosome, X daughter, X son) and the
 * parent rows (-1 = founder) the engine built; any pointer may be NULL. */
int fs_get_tables(const fs_engine *e, double *pcp2, double *pcp2_xf, double *pcp2_xm, int32_t *mother,
                  int32_t *father);

/* Copies the compiled Elston-Stewart message program (host/es_program.hpp describes the word format) into
 * `words` (capacity in words); *n_words / *n_slots receive its length and scratch size.  Introspection only:
 * tests interpret it on the CPU to check the pedigree compiler without a GPU.  FS_E_LOOP on looped pedigrees. */
int fs_get_es_program(const fs_engine *e, uint32_t *words, int32_t capacity, int32_t *n_words, int32_t *n_slots);

/* The conditioned program of FS_METHOD_BN_PEEL (host/bn_peel.hpp): its words (the format of fs_get_es_program plus
 * ES_OP_ACC), *n_words, *n_slots, the ped rows of its *n_breakers loop breakers in breaker_rows (breaker_capacity entries)
 * and, in clamp_slots[2 * breaker_capacity], the vector-file index of each breaker's clamped likelihood and of its
 * indicator.  The accumulators follow the indicators: input column c's member, then the unsequenced members in ped order.
 * Every pointer may be NULL.  Introspection: tests interpret the program on the CPU.  The run's error where the program is
 * refused. */
int fs_get_bn_peel_program(const fs_engine *e, uint32_t *words, int32_t capacity, int32_t *n_words, int32_t *n_slots,
                           int32_t *breaker_rows, int32_t breaker_capacity, int32_t *n_breakers, int32_t *clamp_slots);

/* The Gibbs sampler of large MCMC batches is a kernel the engine writes for this one pedigree and compiles for
 * sm_100a at run time (NVRTC; csrc/cuda/gibbs_jit.cu) -- it replaces the same reference functions as the table-driven
 * kernel, family::calPostProbMCMC / estGenoProb (src/family.cpp:1932-2299), and returns the same bytes.  Introspection:
 * compile == 0 copies the generated CUDA C++ into `text`; compile != 0 also compiles it (no device needed) and copies
 * the compiler log (ptxas -v: registers, spills) instead, with the cubin size in *cubin_bytes.  `text` is
 * NUL-terminated and truncated to `capacity`; *text_len receives the full length. */
int fs_get_gibbs_kernel(const fs_engine *e, int compile, char *text, size_t capacity, size_t *text_len, size_t *cubin_bytes);

/* The same for Elston-Stewart peeling of pedigrees that are not nuclear families: the message program as straight-line
 * code (csrc/cuda/es_jit.cu), replacing family::calPostProbPeeling + calAntProb[X] + calPosProb[X]
 * (src/family.cpp:1126-1403, :1501-1930) with the same doubles as the interpreter.  FAMSEQ_ES_JIT=1 uses it from the
 * first batch, unset: after 2e10 variants.  FS_E_LOOP on looped pedigrees. */
int fs_get_es_kernel(const fs_engine *e, int compile, char *text, size_t capacity, size_t *text_len, size_t *cubin_bytes);

/* Initialises the CUDA context of `device` and nothing else.  fs_create does it anyway; a caller that still has
 * input to read can run this on a helper thread first (the command line does) and hide the ~0.3 s it takes. */
int fs_warmup(int device);

/* Pinned host memory helpers for callers without their own CUDA runtime binding (portable: usable from every GPU of a
 * multi-device engine). */
void *fs_alloc_pinned(size_t bytes);
void fs_free_pinned(void *p);

/* Milliseconds the kernels of the last fs_run on this engine spent on the device (CUDA events). */
double fs_last_kernel_ms(const fs_engine *e);

/* Measures the device's plain (non-tensor) FP64 throughput with register-resident DFMA chains and writes
 * TFLOP/s to *tflops.  bench.py uses it as the roofline denominator of the BN and MCMC kernels. */
int fs_bench_fp64_tflops(int device, double *tflops);

#ifdef __cplusplus
}
#endif
#endif /* FAMSEQ_B200_H_ */
