"""CPU-only checks of conditioned peeling (method 4, BN_PEEL; famseq_b200/csrc/host/bn_peel.cpp).

The conditioned program is fetched through the C ABI (fs_get_bn_peel_program, host-only engine) and interpreted here in
plain Python floats (IEEE doubles, no FMA) with the semantics of cuda/es_interpret.cuh and cuda/bn_peel_kernel.cu: one
peel per clamp of the loop breakers, ES_OP_ACC adding each member's unnormalised marginal.  The result is checked against
the C oracle's Bayesian network and, past its 31-member reach, against exact variable elimination written here in numpy.
This is test infrastructure: the product has no CPU compute path."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import famseq_b200 as fs
from famseq_b200 import synth
from oracle import oracle as O

from .test_es_program_cpu import interpret as es_interpret

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OP_END, OP_MUL, OP_ANT, OP_POS, OP_FIN, OP_ACC = 0, 1, 2, 3, 4, 5
TAB_AUTO, TAB_XF, TAB_XM = 0, 1, 2
MAX_BREAKERS = 8


def host_engine(ped, cols=None):
    return fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols() if cols is None else cols, device=-1)


def cycle_rank(ped):
    """E - V + C of the member--marriage graph."""
    par = ped.parents()
    couples = sorted({p for p in par if p[0] >= 0})
    root = list(range(ped.n + len(couples)))

    def find(x):
        while root[x] != x:
            root[x] = root[root[x]]
            x = root[x]
        return x

    closing = 0
    cidx = {c: ped.n + k for k, c in enumerate(couples)}
    edges = [(m, cidx[(m, f)]) for m, f in couples] + [(f, cidx[(m, f)]) for m, f in couples]
    edges += [(i, cidx[p]) for i, p in enumerate(par) if p[0] >= 0]
    for a, b in edges:
        a, b = find(a), find(b)
        if a == b:
            closing += 1
        else:
            root[a] = b
    return closing


def peel_interpret(words, n_slots, clamps, breaker_cols, n_members, tabs, priors, lk, flag):
    """One variant through the conditioned program.  Returns post [S][3], or None when a member's marginal sums to <= 0."""
    known, chrx = flag & 1, (flag >> 1) & 1
    pa = priors[1 if known else 0]
    pm = priors[(3 if known else 2)] if chrx else pa
    S, K = len(lk), len(breaker_cols)
    vec = [[float(x) for x in row] for row in lk] + [[0.0] * 3 for _ in range(n_slots)]
    vec += [[float(x) for x in pa], [float(x) for x in pm], [1.0, 1.0, 1.0]]
    vec += [[0.0] * 3 for _ in range(2 * K + n_members)]
    acc_base = S + n_slots + 3 + 2 * K

    def T(male, g, a, b):
        t = tabs[(TAB_XM if male else TAB_XF) if chrx else TAB_AUTO]
        return float(t[g * 9 + a * 3 + b])

    for c in range(3 ** K):
        rest = c
        for j in range(K):
            d = rest % 3
            rest //= 3
            e = [1.0 if g == d else 0.0 for g in range(3)]
            col = breaker_cols[j]
            vec[clamps[j][0]] = [vec[col][g] if g == d else 0.0 for g in range(3)] if col >= 0 else e
            vec[clamps[j][1]] = e
        pc = 0
        while True:
            w0 = int(words[pc]); op = w0 & 0xff
            if op == OP_END:
                break
            if op == OP_MUL:
                w1 = int(words[pc + 1]); a, b = vec[w1 & 0xffff], vec[w1 >> 16]
                vec[(w0 >> 8) & 0xffff] = [a[g] * b[g] for g in range(3)]
                pc += 2
            elif op == OP_ANT:
                w1 = int(words[pc + 1]); nsib = w0 >> 25; cmale = (w0 >> 24) & 1
                wm, wf = vec[w1 & 0xffff], vec[w1 >> 16]
                sibs = None
                for k in range(nsib):
                    wk = int(words[pc + 2 + k]); d = vec[wk & 0xffff]; smale = (wk >> 16) & 1
                    cur = [[(d[0] * T(smale, 0, a, b) + d[1] * T(smale, 1, a, b)) + d[2] * T(smale, 2, a, b) for b in range(3)] for a in range(3)]
                    sibs = cur if sibs is None else [[sibs[a][b] * cur[a][b] for b in range(3)] for a in range(3)]
                out = []
                for g in range(3):
                    over_m = 0.0
                    for a in range(3):
                        over_f = 0.0
                        for b in range(3):
                            term = wf[b] * T(cmale, g, a, b)
                            if nsib:
                                term = term * sibs[a][b]
                            over_f = over_f + term
                        over_m = over_m + wm[a] * over_f
                    out.append(over_m)
                vec[(w0 >> 8) & 0xffff] = out
                pc += 2 + nsib
            elif op == OP_POS:
                w1 = int(words[pc + 1]); nkid = w0 >> 25; i_second = bool(chrx and ((w0 >> 24) & 1))
                wj = vec[w1 & 0xffff]
                kids = None
                for k in range(nkid):
                    wk = int(words[pc + 2 + 2 * k]); kmale = int(words[pc + 3 + 2 * k]) & 1
                    lkc, mc = vec[wk & 0xffff], vec[wk >> 16]
                    cur = [[0.0] * 3 for _ in range(3)]
                    for g in range(3):
                        for b in range(3):
                            sc = None
                            for l in range(3):
                                tr = T(kmale, l, b, g) if i_second else T(kmale, l, g, b)
                                term = (tr * lkc[l]) * mc[l]
                                sc = term if sc is None else sc + term
                            cur[g][b] = sc
                    kids = cur if kids is None else [[kids[g][b] * cur[g][b] for b in range(3)] for g in range(3)]
                vec[(w0 >> 8) & 0xffff] = [(wj[0] * kids[g][0] + wj[1] * kids[g][1]) + wj[2] * kids[g][2] for g in range(3)]
                pc += 2 + 2 * nkid
            else:
                assert op == OP_ACC, op
                w1, w2 = int(words[pc + 1]), int(words[pc + 2])
                m, l, a = vec[w1 & 0xffff], vec[w1 >> 16], vec[w2 & 0xffff]
                v = [(m[g] * l[g]) * a[g] for g in range(3)]
                acc = (w0 >> 8) & 0xffff
                assert acc_base <= acc < acc_base + n_members
                vec[acc] = v if c == 0 else [vec[acc][g] + v[g] for g in range(3)]
                pc += 3
    post = [None] * S
    for k in range(n_members):
        a = vec[acc_base + k]
        s = (a[0] + a[1]) + a[2]
        if s <= 0.0:
            return None
        if k < S:
            post[k] = [a[g] / s for g in range(3)]
    return post


def run_program(e, ped, cols, lk, fl):
    words, n_slots, rows, clamps = e.bn_peel_program()
    a, xf, xm, _, _ = e.tables()
    col_of = {r: c for c, r in enumerate(cols)}
    bcols = [col_of.get(int(r), -1) for r in rows]
    return [peel_interpret(words, n_slots, clamps, bcols, ped.n, [a, xf, xm], e.params.priors(), lk[v], int(fl[v]))
            for v in range(len(lk))]


# ---- an exact oracle independent of the engine: variable elimination over the pedigree's factors ---------------------
def ve_marginals(ped, cols, tabs, priors, lk, flag):
    """Normalised exact marginal [n][3] of every member (None where the total is 0), by numpy variable elimination with a
    min-degree order."""
    known, chrx = flag & 1, (flag >> 1) & 1
    pa = priors[1 if known else 0]
    pm = priors[(3 if known else 2)] if chrx else pa
    par = ped.parents()
    male = [g == 1 for g in ped.genders]
    lk_of = {r: lk[c] for c, r in enumerate(cols)}
    base = []
    for i in range(ped.n):
        m, f = par[i]
        own = np.asarray(lk_of.get(i, np.ones(3)), np.float64)
        if m < 0:
            base.append(((i,), (pm if male[i] else pa) * own))
        else:
            t = tabs[(TAB_XM if male[i] else TAB_XF) if chrx else TAB_AUTO].reshape(3, 3, 3)  # [g][mother][father]
            base.append(((i, m, f), t * own[:, None, None]))
    out = []
    for q in range(ped.n):
        factors = list(base)
        left = set(range(ped.n)) - {q}
        while left:
            def degree(x):
                nb = set()
                for vs, _ in factors:
                    if x in vs:
                        nb |= set(vs)
                return len(nb)
            x = min(left, key=lambda y: (degree(y), y))
            left.discard(x)
            touch = [fc for fc in factors if x in fc[0]]
            factors = [fc for fc in factors if x not in fc[0]]
            vs = sorted(set(v for f_, _ in touch for v in f_))
            letters = {v: chr(97 + k) for k, v in enumerate(vs)}
            keep = [v for v in vs if v != x]
            spec = ",".join("".join(letters[v] for v in f_) for f_, _ in touch) + "->" + "".join(letters[v] for v in keep)
            factors.append((tuple(keep), np.einsum(spec, *[t for _, t in touch])))
        m = np.ones(3)
        for vs, t in factors:
            m = m * (t if vs else t * np.ones(3))
        s = m.sum()
        out.append(None if s <= 0 else m / s)
    return out


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    nz = b != 0
    assert np.array_equal(a == 0, b == 0) or np.max(np.abs(a - b)) < 1e-300
    return float(np.max(np.abs(a[nz] - b[nz]) / np.abs(b[nz]))) if nz.any() else 0.0


# ---- breakers ---------------------------------------------------------------------------------------------------
LOOPED = {"ped40": synth.ped40, "cousins_loop": synth.cousins_loop}
LOOP_FREE = ["trio", "ped14", "half_sibs", "three_wives", "ped100"]


@pytest.mark.parametrize("name", sorted(LOOPED) + LOOP_FREE)
def test_breakers_within_the_cycle_rank(name):
    ped = synth.PEDIGREES[name]()
    with host_engine(ped) as e:
        words, n_slots, rows, clamps = e.bn_peel_program()  # the broken pedigree compiled: no FS_E_LOOP
    K, rank = len(rows), cycle_rank(ped)
    assert K <= rank
    assert {"ped40": 3, "cousins_loop": 1}.get(name, 0) == rank
    if name == "cousins_loop":
        assert K == 1
    if name in LOOP_FREE:
        assert K == 0
    assert len(set(rows.tolist())) == K
    ops = [int(w) & 0xff for w in _op_words(words)]
    assert OP_FIN not in ops and ops.count(OP_ACC) == ped.n


def _op_words(words):
    """The first word of every operation of a program."""
    pc, out = 0, []
    while True:
        w0 = int(words[pc]); op = w0 & 0xff
        out.append(w0)
        if op == OP_END:
            return out
        pc += {OP_MUL: 2, OP_ANT: 2 + (w0 >> 25), OP_POS: 2 + 2 * (w0 >> 25)}.get(op, 3)


@pytest.mark.parametrize("seed", range(12))
def test_breakers_on_random_looped_pedigrees(seed):
    ped = synth.random_pedigree(seed, 40 + seed * 7, loops=True, shuffle=seed % 2 == 1)
    with host_engine(ped) as e:
        try:
            words, _, rows, _ = e.bn_peel_program()
        except fs.FamSeqError as err:  # past the breaker cap
            assert err.code == -5 and cycle_rank(ped) > MAX_BREAKERS
            return
    assert len(rows) <= cycle_rank(ped)
    with host_engine(ped) as e2:  # deterministic
        w2, _, r2, _ = e2.bn_peel_program()
    assert np.array_equal(words, w2) and np.array_equal(rows, r2)


@pytest.mark.parametrize("name", sorted(LOOPED))
def test_breakers_deterministic_on_shuffled_rows(name):
    ped = LOOPED[name]()
    rank = cycle_rank(ped)
    for seed in range(4):
        perm = np.random.default_rng(seed).permutation(ped.n)
        sp = synth.PedFile(*[[getattr(ped, k)[i] for i in perm] for k in ("ids", "mids", "fids", "genders", "names")])
        got = []
        for _ in range(2):
            with host_engine(sp) as e:
                words, _, rows, _ = e.bn_peel_program()
            got.append((words, rows))
        assert np.array_equal(got[0][0], got[1][0]) and np.array_equal(got[0][1], got[1][1])
        assert 1 <= len(got[0][1]) <= rank


def test_breaker_cap_refused_at_run_time():
    """Nine unrelated cousin marriages in one ped file: cycle rank 9 > 8.  fs_create accepts it, the program is refused."""
    ped, _ = synth.forest([synth.cousins_loop()] * 9)
    assert cycle_rank(ped) == 9
    with host_engine(ped) as e:  # fs_create succeeds
        with pytest.raises(fs.FamSeqError) as err:
            e.bn_peel_program()
    assert err.value.code == -5 and "loop breakers" in str(err.value) and "-peelLoops" in str(err.value)


# ---- K = 0: the ES program with FIN replaced by ACC ----------------------------------------------------------------
@pytest.mark.parametrize("name", LOOP_FREE + ["many_spouses", "three_generations", "random"])
def test_loop_free_program_is_the_es_program(name):
    if name == "many_spouses":
        ped = synth.many_spouses(5)
    elif name == "three_generations":
        ped = synth.three_generations()
    elif name == "random":
        ped = synth.random_pedigree(3, 30, shuffle=True, unsequenced=0.3)
    else:
        ped = synth.PEDIGREES[name]()
    cols = ped.sequenced_cols()
    with host_engine(ped) as e:
        es_words, es_slots = e.es_program()
        words, n_slots, rows, clamps = e.bn_peel_program()
    assert len(rows) == 0 and n_slots == es_slots and len(words) == len(es_words)
    S = len(cols)
    acc_base = S + n_slots + 3
    unseq = [i for i in range(ped.n) if i not in set(cols)]
    fin_rows = iter(range(ped.n))  # FIN / ACC come in ped-row order
    pc = 0
    while True:
        w0, a0 = int(es_words[pc]), int(words[pc])
        op = w0 & 0xff
        if op != OP_FIN:
            n = 1 if op == OP_END else {OP_MUL: 2, OP_ANT: 2 + (w0 >> 25), OP_POS: 2 + 2 * (w0 >> 25)}[op]
            assert np.array_equal(es_words[pc:pc + n], words[pc:pc + n]), f"{name}: word {pc}"
            if op == OP_END:
                break
            pc += n
            continue
        i = next(fin_rows)
        k = cols.index(i) if i in cols else S + unseq.index(i)
        assert a0 == OP_ACC | (acc_base + k) << 8
        assert es_words[pc + 1] == words[pc + 1] and es_words[pc + 2] == words[pc + 2]
        pc += 3


@pytest.mark.parametrize("name", ["ped14", "half_sibs", "three_wives"])
def test_loop_free_interpretation_bit_identical_to_es(name):
    ped = synth.PEDIGREES[name]()
    cols = ped.sequenced_cols()
    lk, fl = synth.synth_likelihoods(ped, 20, seed=5, x_fraction=0.4)
    with host_engine(ped) as e:
        got = run_program(e, ped, cols, lk, fl)
        words, n_slots = e.es_program()
        a, xf, xm, _, _ = e.tables()
        want = [es_interpret(words, n_slots, [a, xf, xm], e.params.priors(), lk[v], int(fl[v])) for v in range(20)]
    for g, w in zip(got, want):
        assert (g is None) == (w is None)
        if g is not None:
            assert np.array_equal(np.array(g), np.array(w))


# ---- looped pedigrees against the C oracle's BN ------------------------------------------------------------------
def looped_cases():
    yield "cousins_loop", synth.cousins_loop()
    found = 0
    for seed in range(200):
        ped = synth.random_pedigree(seed, 8 + seed % 5, loops=True, shuffle=True, unsequenced=0.25)
        if cycle_rank(ped) > 0:
            yield f"random{seed}", ped
            found += 1
            if found == 6:
                return


@pytest.mark.parametrize("name,ped", list(looped_cases()))
def test_matches_oracle_bn(name, ped):
    cols = ped.sequenced_cols()
    V = 24
    lk, fl = synth.synth_likelihoods(ped, V, seed=11, x_fraction=0.4)
    fl = fl | (np.arange(V) % 3 == 0).astype(np.uint8)  # Known rows too
    want = O.run(ped, cols, lk, fl, method=O.BN, lc=5.0)
    with host_engine(ped, cols) as e:
        assert len(e.bn_peel_program()[2]) >= 1
        got = run_program(e, ped, cols, lk, fl)
    checked = 0
    for v in range(V):
        if want["status"][v]:
            continue
        assert got[v] is not None, f"{name} variant {v}"
        assert rel(got[v], want["post"][v]) <= 1e-9, f"{name} variant {v}"
        checked += 1
    assert checked >= V // 2


# ---- past the oracle's reach: exact variable elimination ------------------------------------------------------------
def big_looped_cases():
    yield "ped40", synth.ped40()
    found = 0
    for seed in range(100):
        ped = synth.random_pedigree(1000 + seed, 40 + (seed * 7) % 21, loops=True, shuffle=True, unsequenced=0.2)
        if 1 <= cycle_rank(ped) <= 4:
            yield f"random{1000 + seed}", ped
            found += 1
            if found == 2:
                return


@pytest.mark.parametrize("name,ped", list(big_looped_cases()))
def test_matches_variable_elimination(name, ped):
    cols = ped.sequenced_cols()
    V = 3
    lk, fl = synth.synth_likelihoods(ped, V, seed=21, x_fraction=0.34)
    with host_engine(ped, cols) as e:
        got = run_program(e, ped, cols, lk, fl)
        a, xf, xm, _, _ = e.tables()
        priors = e.params.priors()
    for v in range(V):
        want = ve_marginals(ped, cols, [a, xf, xm], priors, lk[v], int(fl[v]))
        assert got[v] is not None
        for c, r in enumerate(cols):
            assert rel(got[v][c], want[r]) <= 1e-9, f"{name} variant {v} column {c}"


# ---- the Elston-Stewart kernels do not change: the ACC op exists only in bn_peel_kernel's instantiation -----------------
@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="needs nvcc")
def test_es_kernels_sass_unchanged_by_the_acc_op(tmp_path):
    """Cross-compiles es_kernel.cu and es_cohort_kernel.cu for sm_100a twice -- with cuda/es_interpret.cuh as it is, and with
    its `if constexpr (ACC)` block cut out -- and requires byte-identical SASS."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    csrc = os.path.join(ROOT, "famseq_b200", "csrc")
    src = open(os.path.join(csrc, "cuda", "es_interpret.cuh")).read()
    start = src.index("        if constexpr (ACC) {")
    end = src.index("        if (op == ES_OP_MUL) {")
    assert start < end
    stripped = tmp_path / "famseq_b200" / "csrc"
    shutil.copytree(csrc, stripped, ignore=shutil.ignore_patterns("build", "*.o"))
    (stripped / "cuda" / "es_interpret.cuh").write_text(src[:start] + src[end:])
    inc = tmp_path / "include"
    shutil.copytree(os.path.join(ROOT, "include"), inc)
    flags = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-fmad=false"]
    procs = []
    for tree in (csrc, str(stripped)):
        for name in ("es_kernel", "es_cohort_kernel"):
            out = tmp_path / f"{name}_{'new' if tree == csrc else 'stripped'}.o"
            procs.append((name, out, subprocess.Popen([nvcc, *flags, "-c", os.path.join(tree, "cuda", name + ".cu"), "-o", str(out)])))
    for _, _, p in procs:
        assert p.wait() == 0
    sass = {}
    for name, out, _ in procs:
        text = subprocess.run([cuobjdump, "-sass", str(out)], check=True, capture_output=True, text=True).stdout
        # the source path shows in the identifier line and, hashed, in the anonymous-namespace tag of mangled names
        text = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", re.sub(r"(?m)^identifier = .*$", "", text))
        sass.setdefault(name, []).append(text)
    for name, (a, b) in sass.items():
        assert len(a.splitlines()) > 1000 and a == b, f"{name}: SASS differs"
