// es_program.hpp -- the Elston-Stewart "message program": the reference's memoised mutual recursion
// (calAntProb / calPosProb, src/family.cpp:1501-1930) unrolled ONCE on the host into a flat,
// topologically ordered list of vector operations.  The schedule depends only on the pedigree, never
// on the variant, so one program drives every thread of the kernel (one variant per thread).
//
// Shared between the host compiler (es_program.cpp) and the interpreter kernel (cuda/es_kernel.cu).
#pragma once

#include <cstdint>
#include <string>
#include <vector>

#ifdef __CUDACC__
#define FS_HD __host__ __device__
#else
#define FS_HD
#endif

namespace famseq {

struct Pedigree; // host/pedigree.hpp

// Inside the compiler a "vector reference" names a genotype 3-vector by kind and index.  In the encoded program an
// operand is a 16-bit index into the per-variant VECTOR FILE the kernel keeps in shared memory:
//   [0, S)              likelihood rows of the input columns
//   [S, S + n_slots)    message scratch
//   S + n_slots + 0/1   founder prior of a non-male / male member (the latter is the chrX male prior on X)
//   S + n_slots + 2     the vector of ones (an unsequenced member's likelihood, an empty product)
// so the interpreter fetches any operand with three shared-memory loads and no case distinction.
enum EsRefKind : uint32_t {
    ES_REF_ONE = 0,   // (1,1,1): an unsequenced member's likelihood / an empty product. Never multiplied.
    ES_REF_SLOT = 1,  // per-thread scratch 3-vector `index`
    ES_REF_LK = 2,    // likelihood of input column `index`
    ES_REF_PRIOR = 3, // founder prior; index 1 = male (uses the chrX male prior on X), 0 = otherwise
    ES_REF_FIXED = 4, // conditioned program (host/bn_peel.hpp): reserved vector `index` behind the three special vectors
};
FS_HD constexpr uint32_t es_ref(EsRefKind k, uint32_t index) { return ((uint32_t)k << 13) | (index & 0x1fffu); }
FS_HD constexpr uint32_t es_ref_kind(uint32_t r) { return (r >> 13) & 7u; }
FS_HD constexpr uint32_t es_ref_index(uint32_t r) { return r & 0x1fffu; }

enum EsOpcode : uint32_t {
    // word0 = opcode | dst_slot<<8 ; word1 = a | b<<16                       dst = a (*) b element-wise
    ES_OP_MUL = 1,
    // anterior message of a non-founder (family.cpp:1609-1646 / :1714-1778):
    //   dst[g] = sum_a Wm[a] * ( sum_b ((Wf[b] * T_c[g][a][b]) * prod_k sum_l (D_k[l] * T_k[l][a][b])) )
    // word0 = opcode | dst<<8 | child_male<<24 | nsib<<25 ; word1 = Wm | Wf<<16 ;
    // then per full sib one word: D_k | sib_male<<16
    ES_OP_ANT = 2,
    // posterior message of i through the marriage with j (family.cpp:1817-1843 / :1881-1927):
    //   dst[g] = sum_b Wj[b] * prod_c sum_l ((T_c[l][g,b] * lk_c[l]) * M_c[l])
    // word0 = opcode | dst<<8 | i_male<<24 | nkid<<25 ; word1 = Wj ;
    // then per joint child two words: lk_c | M_c<<16 ; child_male
    ES_OP_POS = 3,
    // marginal of one member (family.cpp:1292-1314): v = (M (*) lk) (*) ant, row sum == 0 => variant fails,
    // otherwise, when the member is sequenced, post[col] = v / sum and gt[col] = arg max.
    // word0 = opcode | has_col<<8 | col<<9 ; word1 = M | lk<<16 ; word2 = ant
    ES_OP_FIN = 4,
    // conditioned peeling (host/bn_peel.hpp) in place of FIN: v = (M (*) lk) (*) ant is stored into (first peel) or added
    // to (later peels) the accumulator vector `acc`; no normalisation and no row-sum test.
    // word0 = opcode | acc<<8 ; word1 = M | lk<<16 ; word2 = ant
    ES_OP_ACC = 5,
    ES_OP_END = 0,
};

constexpr int ES_MAX_WORDS = 3072; // 12 KB of kernel-parameter space

struct EsProgram {
    int32_t n_words = 0;
    int32_t n_ops = 0;
    int32_t n_slots = 0; // scratch 3-vectors per variant after liveness-based reuse
    int32_t n_cols = 0;
    uint32_t words[ES_MAX_WORDS];
};

// Overrides of the conditioned program (host/bn_peel.cpp), in reserved vectors (ES_REF_FIXED, numbered from 0 right behind
// the three special vectors).  Members [0, n_real) are the pedigree's own; rows from n_real on are founder copies.
struct EsConditioning {
    int n_real = 0;
    std::vector<int> lk_fixed;  // [n] reserved vector replacing lk(i) (a breaker's clamped likelihood), or -1
    std::vector<int> ant_fixed; // [n] reserved vector replacing a founder copy's prior (the clamp indicator), or -1
    std::vector<int> acc_fixed; // [n_real] accumulator of member i: its FIN becomes ES_OP_ACC into this vector
    int n_fixed = 0;            // reserved vectors in all
};

// Host entry point of the pedigree compiler (es_program.cpp).  Returns FS_OK, FS_E_LOOP (pedigree is not
// peelable) or FS_E_TOO_LARGE; `err` receives the text.  With `cond`, the conditioned program of bn_peel.cpp.
int compile_es_program(const Pedigree &ped, EsProgram &out, std::string &err, const EsConditioning *cond = nullptr);

} // namespace famseq
