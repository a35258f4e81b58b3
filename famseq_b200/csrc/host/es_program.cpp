// es_program.cpp -- compiles a loop-free pedigree into the Elston-Stewart message program.
//
// The compiler walks the same mutual recursion as the reference (anterior message of a member needs
// the messages of both parents and of the full sibs; the posterior message of i through spouse j needs
// j's messages and the joint children's), but it runs once, symbolically, and records each message as
// one vector operation.  Products are emitted in exactly the reference's association order
// (family.cpp:1609-1646, :1817-1843, :1292-1303) so that the kernel, which is compiled without FMA
// contraction, reproduces the reference's doubles bit for bit.  Multiplications by an exact 1.0
// (unsequenced members, empty spouse products) are dropped -- they cannot change a double.
#include "es_program.hpp"
#include "pedigree.hpp"

#include <algorithm>
#include <map>

#include "../../../include/famseq_b200.h"

namespace famseq {
namespace {

struct Ref {
    EsRefKind kind = ES_REF_ONE;
    int index = 0;
    bool one() const { return kind == ES_REF_ONE; }
    bool operator<(const Ref &o) const { return kind != o.kind ? kind < o.kind : index < o.index; }
};

struct Item {
    Ref r0, r1;
    int male = 0;
};

struct Op {
    EsOpcode op = ES_OP_END;
    int dst = -1; // virtual slot
    Ref a, b, c;
    int male = 0;
    int col = -1;
    std::vector<Item> items;
};

class Compiler {
  public:
    Compiler(const Pedigree &p, const EsConditioning *c) : ped(p), cond(c), ant_slot(p.n, -1), ant_busy(p.n, 0) {}

    bool run(std::string &err) {
        const int n_fin = cond ? cond->n_real : ped.n; // founder copies have no marginal of their own
        for (int i = 0; i < n_fin && !loop; i++) {
            // family.cpp:1296-1301: postTmp = (prod_k pos(i,.,spouse k)) * lk(i,.) * ant(i,.)
            std::vector<Ref> below;
            for (int sp : ped.spouses[i]) below.push_back(pos(i, sp));
            Op f;
            f.op = ES_OP_FIN;
            f.a = product(below);
            f.b = lk(i);
            f.c = ant(i);
            f.col = ped.col_of[i];
            if (cond) {
                f.op = ES_OP_ACC;
                f.dst = cond->acc_fixed[i]; // a reserved vector, not a virtual slot
            }
            ops.push_back(f);
        }
        if (loop) {
            err = "The pedigree has a marriage or consanguinity loop: the Elston-Stewart method (-method 2) "
                  "needs a loop-free pedigree. Use -method 1 (BN) or -method 3 (MCMC).";
            return false;
        }
        return true;
    }

    std::vector<Op> ops;
    int n_virtual = 0;

  private:
    const Pedigree &ped;
    const EsConditioning *cond;
    std::vector<int> ant_slot;
    std::vector<char> ant_busy;
    std::map<std::pair<int, int>, int> pos_slot;
    std::map<std::pair<int, int>, char> pos_busy;
    std::map<std::vector<Ref>, Ref> chains;
    bool loop = false;

    Ref lk(int i) const {
        Ref r;
        if (cond && cond->lk_fixed[i] >= 0) {
            r.kind = ES_REF_FIXED;
            r.index = cond->lk_fixed[i];
        } else if (ped.col_of[i] >= 0) {
            r.kind = ES_REF_LK;
            r.index = ped.col_of[i];
        }
        return r;
    }
    Ref slot(int v) const {
        Ref r;
        r.kind = ES_REF_SLOT;
        r.index = v;
        return r;
    }

    // Left-to-right element-wise product of the non-unit entries (memoised by operand list).
    Ref product(std::vector<Ref> v) {
        v.erase(std::remove_if(v.begin(), v.end(), [](const Ref &r) { return r.one(); }), v.end());
        if (v.empty()) return Ref();
        if (v.size() == 1) return v[0];
        auto hit = chains.find(v);
        if (hit != chains.end()) return hit->second;
        Ref last = v.back();
        std::vector<Ref> head(v.begin(), v.end() - 1);
        Op m;
        m.op = ES_OP_MUL;
        m.a = product(head);
        m.b = last;
        m.dst = n_virtual++;
        ops.push_back(m);
        return chains[v] = slot(m.dst);
    }

    // ((ant(x) * lk(x)) * prod(pos(x, s) for the spouses s other than `except`))
    Ref weight(int x, int except) {
        Ref base = product({ant(x), lk(x)});
        std::vector<Ref> others;
        for (int sp : ped.spouses[x])
            if (sp != except) others.push_back(pos(x, sp));
        return product({base, product(others)});
    }

    Ref ant(int i) {
        if (ped.founder(i)) {
            Ref r;
            if (cond && cond->ant_fixed[i] >= 0) {
                r.kind = ES_REF_FIXED;
                r.index = cond->ant_fixed[i];
                return r;
            }
            r.kind = ES_REF_PRIOR;
            r.index = ped.male[i];
            return r;
        }
        if (ant_slot[i] >= 0) return slot(ant_slot[i]);
        if (loop) return Ref();
        if (ant_busy[i]) {
            loop = true;
            return Ref();
        }
        ant_busy[i] = 1;
        const int m = ped.mother[i], f = ped.father[i];
        Op a;
        a.op = ES_OP_ANT;
        a.male = ped.male[i];
        for (int c : ped.children[m]) { // full sibs, in the mother's child order (family.cpp:1576-1587)
            if (c == i || ped.father[c] != f) continue;
            std::vector<Ref> below;
            for (int sp : ped.spouses[c]) below.push_back(pos(c, sp));
            Item it;
            it.r0 = product({product(below), lk(c)}); // (mcs * lk), family.cpp:1627
            it.male = ped.male[c];
            a.items.push_back(it);
        }
        a.b = weight(f, m);
        a.a = weight(m, f);
        ant_busy[i] = 0;
        if (loop) return Ref();
        a.dst = n_virtual++;
        ant_slot[i] = a.dst;
        ops.push_back(a);
        return slot(a.dst);
    }

    Ref pos(int i, int j) {
        const auto key = std::make_pair(i, j);
        auto hit = pos_slot.find(key);
        if (hit != pos_slot.end()) return slot(hit->second);
        if (loop) return Ref();
        if (pos_busy[key]) {
            loop = true;
            return Ref();
        }
        pos_busy[key] = 1;
        Op p;
        p.op = ES_OP_POS;
        p.male = ped.male[i];
        p.a = weight(j, i);
        for (int c : ped.children[i]) { // joint children in i's child order (family.cpp:1806-1815)
            if (ped.mother[c] != j && ped.father[c] != j) continue;
            std::vector<Ref> below;
            for (int sp : ped.spouses[c]) below.push_back(pos(c, sp));
            Item it;
            it.r0 = lk(c);
            it.r1 = product(below);
            it.male = ped.male[c];
            p.items.push_back(it);
        }
        pos_busy[key] = 0;
        if (loop) return Ref();
        p.dst = n_virtual++;
        pos_slot[key] = p.dst;
        ops.push_back(p);
        return slot(p.dst);
    }
};

template <class F> void for_each_ref(Op &o, F f) {
    f(o.a);
    f(o.b);
    f(o.c);
    for (auto &it : o.items) {
        f(it.r0);
        f(it.r1);
    }
}


} // namespace

int compile_es_program(const Pedigree &ped, EsProgram &out, std::string &err, const EsConditioning *cond) {
    out = EsProgram();
    out.n_cols = ped.s();
    Compiler c(ped, cond);
    if (!c.run(err)) return FS_E_LOOP;

    // Liveness-based slot reuse: a virtual slot dies after its last reader; the destination of an
    // operation never aliases one of its own operands.
    const int nops = (int)c.ops.size();
    std::vector<int> last_use(c.n_virtual, -1);
    for (int k = 0; k < nops; k++)
        for_each_ref(c.ops[k], [&](Ref &r) {
            if (r.kind == ES_REF_SLOT) last_use[r.index] = k;
        });
    std::vector<int> phys(c.n_virtual, -1), free_list;
    std::vector<std::vector<int>> dying(nops);
    for (int v = 0; v < c.n_virtual; v++)
        if (last_use[v] >= 0) dying[last_use[v]].push_back(v);
    int n_phys = 0;
    for (int k = 0; k < nops; k++) {
        Op &o = c.ops[k];
        if (o.dst >= 0 && o.op != ES_OP_ACC) {
            if (free_list.empty()) {
                phys[o.dst] = n_phys++;
            } else {
                phys[o.dst] = free_list.back();
                free_list.pop_back();
            }
            if (last_use[o.dst] < 0) free_list.push_back(phys[o.dst]); // never read (cannot happen)
        }
        for (int v : dying[k]) free_list.push_back(phys[v]);
    }
    for (Op &o : c.ops) {
        for_each_ref(o, [&](Ref &r) {
            if (r.kind == ES_REF_SLOT) r.index = phys[r.index];
        });
        if (o.dst >= 0 && o.op != ES_OP_ACC) o.dst = phys[o.dst];
    }
    out.n_slots = n_phys;
    out.n_ops = nops;
    if (n_phys >= 0x1fff) {
        err = "pedigree too large for the ES message program (scratch slots)";
        return FS_E_TOO_LARGE;
    }

    // Operand encoding: index of a 3-vector in the per-variant vector file the kernel keeps in shared memory --
    // [0, S) likelihood rows of the input columns, [S, S + n_slots) message scratch, then the founder prior of a
    // non-male member, the founder prior of a male member, and the vector of ones; a conditioned program's reserved
    // vectors follow.
    const uint32_t S = (uint32_t)ped.s(), first_slot = S, special = S + (uint32_t)n_phys;
    const uint32_t n_fixed = cond ? (uint32_t)cond->n_fixed : 0u;
    auto enc = [&](const Ref &r) -> uint32_t {
        switch (r.kind) {
        case ES_REF_LK: return (uint32_t)r.index;
        case ES_REF_SLOT: return first_slot + (uint32_t)r.index;
        case ES_REF_PRIOR: return special + (r.index ? 1u : 0u);
        case ES_REF_FIXED: return special + 3u + (uint32_t)r.index;
        default: return special + 2u;
        }
    };
    if (special + 3u + n_fixed >= 0xffffu) {
        err = "pedigree too large for the ES message program (vector file)";
        return FS_E_TOO_LARGE;
    }
    std::vector<uint32_t> w;
    for (const Op &o : c.ops) {
        switch (o.op) {
        case ES_OP_MUL:
            w.push_back(ES_OP_MUL | (first_slot + (uint32_t)o.dst) << 8);
            w.push_back(enc(o.a) | enc(o.b) << 16);
            break;
        case ES_OP_ANT:
            w.push_back(ES_OP_ANT | (first_slot + (uint32_t)o.dst) << 8 | (uint32_t)o.male << 24 | (uint32_t)o.items.size() << 25);
            w.push_back(enc(o.a) | enc(o.b) << 16);
            for (const Item &it : o.items) w.push_back(enc(it.r0) | (uint32_t)it.male << 16);
            break;
        case ES_OP_POS:
            w.push_back(ES_OP_POS | (first_slot + (uint32_t)o.dst) << 8 | (uint32_t)o.male << 24 | (uint32_t)o.items.size() << 25);
            w.push_back(enc(o.a));
            for (const Item &it : o.items) {
                w.push_back(enc(it.r0) | enc(it.r1) << 16);
                w.push_back((uint32_t)it.male);
            }
            break;
        case ES_OP_FIN:
            w.push_back(ES_OP_FIN | (o.col >= 0 ? 1u << 8 : 0u) | (uint32_t)(o.col >= 0 ? o.col : 0) << 9);
            w.push_back(enc(o.a) | enc(o.b) << 16);
            w.push_back(enc(o.c));
            break;
        case ES_OP_ACC:
            w.push_back(ES_OP_ACC | (special + 3u + (uint32_t)o.dst) << 8);
            w.push_back(enc(o.a) | enc(o.b) << 16);
            w.push_back(enc(o.c));
            break;
        default:
            break;
        }
        if (o.items.size() > 127) {
            err = "pedigree too large for the ES message program (sibship of more than 127)";
            return FS_E_TOO_LARGE;
        }
    }
    w.push_back(ES_OP_END);
    if ((int)w.size() > ES_MAX_WORDS) {
        err = "pedigree too large for the ES message program (" + std::to_string(w.size()) + " words, limit " +
              std::to_string(ES_MAX_WORDS) + ")";
        return FS_E_TOO_LARGE;
    }
    out.n_words = (int)w.size();
    std::copy(w.begin(), w.end(), out.words);
    return FS_OK;
}

} // namespace famseq
