"""Every kernel at the pedigree shapes where layouts change or limits sit, against the C oracle:

  * wide sibships (6..51 children): the nuclear fast path ends at 5 children, so the message-program interpreter runs long
    ANT / POS sibling products, whose order decides the bits; the generated ES kernel up to the largest sibship it takes;
    the ES program's word limit just below and above;
  * several families in one ped file (a forest), and each family's columns of it against the family run on its own;
  * 63 / 64 / 65 and 127 / 128 members: the Gibbs genotype vector goes from two to four 64-bit words, the generated
    Gibbs kernel moves draw thresholds from registers to shared memory, 128 members is the engine's limit;
  * the interpreter's block sizes 128 / 64 / 32 (es_pick_block);
  * one or two members without any parent-child link.

ES must return the oracle's doubles on every variant with status 0 and the same statuses; BN agrees to 1e-9; MCMC draws
from the oracle's Philox stream and agrees to 1e-9, and the generated Gibbs kernels run the same chains as the
table-driven one (assert_same_chains)."""
import numpy as np
import pytest

import famseq_b200 as fs
from famseq_b200 import synth
from oracle import oracle as O
from tests.util import REL_TOL, assert_parity, assert_same_chains, rel_err

pytestmark = pytest.mark.gpu

WIDE = [6, 7, 12, 16, 17, 22, 40, 51]
SEED, VOFF = 4242, 17  # MCMC stream


def engine(ped, cols, params=None, device=0):
    return fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=params, device=device)


def host_probe(ped, cols):
    """(ES program accepted, generated ES kernel accepted) by a host-only engine."""
    with engine(ped, cols, device=-1) as e:
        es_ok = e.info()["es_ops"] > 0
        try:
            e.es_kernel()
            jit_ok = True
        except fs.FamSeqError as x:
            assert x.code == -5
            jit_ok = False
    return es_ok, jit_ok


def wide_likelihoods(V, S, seed):
    """Random mantissas over a wide exponent range, with subnormal and zero entries and certain rows."""
    rng = np.random.default_rng(seed)
    lk = rng.random((V, S, 3)) * np.exp2(rng.integers(-1040, 1, (V, S, 3)).astype(np.float64))
    lk[rng.random((V, S, 3)) < 0.02] = 0.0
    lk[rng.random((V, S)) < 0.05] = 1.0
    return lk


def case_data(ped, cols, V, seed, n_wide=None):
    """Gene-dropped likelihoods of the sequenced members (chrX and Known flags mixed in), then rows with a wide exponent
    range, and a few rows made impossible; V is odd so that the last tile of every block size is ragged."""
    seq = synth._mk(list(zip(ped.ids, ped.mids, ped.fids, ped.genders)))
    lk, fl = synth.synth_likelihoods(seq, V, seed=seed, x_fraction=0.3)
    lk = lk[:, cols]
    n_wide = V // 4 if n_wide is None else n_wide
    lk[V - n_wide:] = wide_likelihoods(n_wide, len(cols), seed + 1)
    lk[3::101, len(cols) // 2] = 0.0  # an all-zero likelihood row: the variant fails
    return lk, fl


def assert_es_matches(got, want, what):
    assert np.array_equal(got.status, want["status"]), f"{what}: status differs"
    ok = want["status"] == 0
    assert np.array_equal(got.post[ok], want["post"][ok]), f"{what}: posteriors are not the oracle's doubles"
    assert np.array_equal(got.single[ok], want["single"][ok]), f"{what}: individual-only posteriors differ"
    assert np.array_equal(got.gt[ok], (want["gt"][ok] & 0xff).astype(np.uint8)), f"{what}: called genotypes differ"


def assert_not_vacuous(res, what, min_ok=0.5):
    ok = res.status == 0
    assert ok.mean() > min_ok, f"{what}: only {ok.mean():.2f} of the variants have status 0"
    assert (~ok).any(), f"{what}: no variant fails"
    assert (res.post[ok] != res.single[ok]).any(axis=(1, 2)).sum() > ok.sum() // 4, f"{what}: too few variants use the pedigree"


def run_es(ped, cols, lk, fl, monkeypatch, jit, params=None):
    """ES with FAMSEQ_ES_JIT=jit; returns (result, jit_launches, info)."""
    monkeypatch.setenv("FAMSEQ_ES_JIT", jit)
    with engine(ped, cols, params) as e:
        got = e.run(fs.ES, lk, fl)
        info = e.info()
    return got, info["jit_launches"], info


def check_es(ped, cols, lk, fl, monkeypatch, what, lc=1.0):
    """Interpreter against the oracle, then the generated kernel against the interpreter wherever the engine accepts it
    (and no generated kernel where it does not).  Returns the interpreter's result."""
    prm = fs.Params.default()
    prm.lrc = lc
    want = O.run(ped, cols, lk, fl, method=O.ES, lc=lc)
    interp, n_jit, info = run_es(ped, cols, lk, fl, monkeypatch, "0", prm)
    assert n_jit == 0
    assert_es_matches(interp, want, f"{what} interpreter")
    _, jit_ok = host_probe(ped, cols)
    got, n_jit, _ = run_es(ped, cols, lk, fl, monkeypatch, "1", prm)
    assert (n_jit >= 1) == jit_ok, f"{what}: generated ES kernel launches {n_jit}, accepted {jit_ok}"
    for k in ("status", "gt", "single", "post"):
        assert np.array_equal(getattr(got, k), getattr(interp, k)), f"{what}: generated ES kernel differs in {k}"
    return interp


def check_mcmc(ped, cols, lk, fl, monkeypatch, what, generators=(None,), burn=10, rep=60):
    """Table-driven Gibbs kernel against the oracle on the same Philox stream, then the generated kernel (each generator
    in `generators`: "0" dense, "1" cached, None the engine's pick) against the table-driven one.  Gene-dropped rows only:
    the kernels multiply by 1/sum where the oracle divides, which for subnormal results is not a 1e-9 agreement."""
    want = O.run(ped, cols, lk, fl, method=O.MCMC, burn=burn, rep=rep, rng=O.RNG_PHILOX, seed=SEED, v_offset=VOFF)
    monkeypatch.setenv("FAMSEQ_MCMC_JIT", "0")
    monkeypatch.delenv("FAMSEQ_JIT_CACHED", raising=False)
    with engine(ped, cols) as e:
        table = e.run(fs.MCMC, lk, fl, burn=burn, rep=rep, seed=SEED, v_offset=VOFF)
        assert e.info()["jit_launches"] == 0
    assert_parity(table, want, 1e-9, f"{what} table-driven MCMC")
    assert (table.status == 0).mean() > 0.5
    monkeypatch.setenv("FAMSEQ_MCMC_JIT", "1")
    for gen in generators:
        if gen is None:
            monkeypatch.delenv("FAMSEQ_JIT_CACHED", raising=False)
        else:
            monkeypatch.setenv("FAMSEQ_JIT_CACHED", gen)
        with engine(ped, cols) as e:
            got = e.run(fs.MCMC, lk, fl, burn=burn, rep=rep, seed=SEED, v_offset=VOFF)
            info = e.info()
        assert info["jit_launches"] >= 1, f"{what}: the generated Gibbs kernel did not run"
        if gen is not None:
            assert info["gibbs_generator"] == 1 + int(gen)
        assert_same_chains(got, table, f"{what} generated MCMC ({gen})")
    return table


def check_bn(ped, cols, lk, fl, what):
    want = O.run(ped, cols, lk, fl, method=O.BN)
    with engine(ped, cols) as e:
        got = e.run(fs.BN, lk, fl)
    assert_parity(got, want, REL_TOL, f"{what} BN")
    return got


def sibship_case(C):
    """C children, the father and the middle child unsequenced, input columns in a shuffled order."""
    ped = synth.sibship(C)
    ped.names[0] = ped.names[2 + C // 2] = "NA"
    cols = list(np.random.default_rng(C).permutation(ped.sequenced_cols()))
    return ped, cols


# ------------------------------------------------------------------------------------------------------
# wide sibships
# ------------------------------------------------------------------------------------------------------
def test_wide_sibships_straddle_the_limits():
    """The ES word limit and the generated ES kernel's limit, probed on host-only engines, fall between two sibship sizes of
    WIDE, so the parametrised tests run both sides of each."""
    def fits(C):
        ped = synth.sibship(C)
        return host_probe(ped, ped.sequenced_cols())
    es_max = next(C for C in range(6, 200) if not fits(C)[0]) - 1
    jit_max = next(C for C in range(6, 200) if not fits(C)[1]) - 1
    assert es_max in WIDE and jit_max in WIDE and jit_max + 1 in WIDE, (es_max, jit_max)
    for C in WIDE:
        es_ok, jit_ok = host_probe(*sibship_case(C))
        assert es_ok and jit_ok == (C <= jit_max), C


@pytest.mark.parametrize("C", WIDE)
def test_wide_sibship(C, monkeypatch):
    ped, cols = sibship_case(C)
    lk, fl = case_data(ped, cols, 2001, seed=900 + C)
    interp = check_es(ped, cols, lk, fl, monkeypatch, f"sibship C={C}")
    assert_not_vacuous(interp, f"sibship C={C}", min_ok=0.5)
    if C <= 15:
        check_bn(ped, cols, lk[:9], fl[:9], f"sibship C={C}")
    check_mcmc(ped, cols, lk[:120], fl[:120], monkeypatch, f"sibship C={C}", generators=("0", "1"))


def test_sibship_of_eight_in_three_generations(monkeypatch):
    """Long POS item lists (a father of 8) meet long ANT lists (each of 8 sibs lists 7) at every level."""
    ped = synth.three_generations(8)
    cols = ped.sequenced_cols()
    lk, fl = case_data(ped, cols, 1501, seed=31)
    assert_not_vacuous(check_es(ped, cols, lk, fl, monkeypatch, "three generations"), "three generations")
    check_mcmc(ped, cols, lk[:120], fl[:120], monkeypatch, "three generations")


def test_member_with_five_spouses(monkeypatch):
    ped = synth.many_spouses(5)
    cols = list(np.random.default_rng(5).permutation(ped.n))
    lk, fl = case_data(ped, cols, 1501, seed=32)
    assert_not_vacuous(check_es(ped, cols, lk, fl, monkeypatch, "five spouses"), "five spouses")
    check_mcmc(ped, cols, lk[:120], fl[:120], monkeypatch, "five spouses")


def test_sibships_past_the_es_limit(monkeypatch):
    """The first sibship the ES program refuses (probed) and 126 children (128 members): ES, and BN at 128 members, are
    refused with FS_E_TOO_LARGE; MCMC runs and matches the oracle."""
    C_refused = next(C for C in range(6, 200) if not host_probe(synth.sibship(C), list(range(C + 2)))[0])
    for C in (C_refused, 126):
        ped = synth.sibship(C)
        cols = ped.sequenced_cols()
        lk, fl = case_data(ped, cols, 61, seed=40 + C, n_wide=0)
        with engine(ped, cols) as e:
            with pytest.raises(fs.FamSeqError) as ei:
                e.run(fs.ES, lk, fl)
            assert ei.value.code == -5 and "words" in str(ei.value)
            if C == 126:
                with pytest.raises(fs.FamSeqError) as ei:
                    e.run(fs.BN, lk[:2], fl[:2])
                assert ei.value.code == -5
        check_mcmc(ped, cols, lk, fl, monkeypatch, f"sibship C={C}", burn=5, rep=40)


# ------------------------------------------------------------------------------------------------------
# several families in one ped file
# ------------------------------------------------------------------------------------------------------
def trios(t):
    return [synth.trio() for _ in range(t)]


def mix():
    return [synth.trio(), synth.ped14(), synth.half_sibs(), synth.sibship(5), synth._mk([(1, 0, 0, 2)])]


FORESTS = {"trios2": (trios(2), None), "trios21": (trios(21), None), "trios42": (trios(42), None), "mix": (mix(), None),
           "mix_shuffled": (mix(), 7)}


@pytest.mark.parametrize("name", list(FORESTS))
def test_forest_vs_oracle(name, monkeypatch):
    fams, shuffle = FORESTS[name]
    ped, _ = synth.forest(fams, shuffle)
    cols = ped.sequenced_cols()
    lk, fl = case_data(ped, cols, 1201, seed=60 + len(cols), n_wide=40)
    with engine(ped, cols, device=-1) as e:
        assert e.info()["n_founders"] > 2  # not the nuclear kernel
    assert_not_vacuous(check_es(ped, cols, lk, fl, monkeypatch, name), name)
    check_mcmc(ped, cols, lk[:100], fl[:100], monkeypatch, name, rep=40)


@pytest.mark.parametrize("name,bn", [("trios2", True), ("trios21", False), ("trios42", False), ("mix", False),
                                     ("mix_shuffled", False), ("trio_and_lone", True)])
def test_forest_equals_its_families(name, bn, monkeypatch):
    """-LRC 5: every variant takes the pedigree.  The columns of each family in the forest's run are the family's run on an
    engine of its own, bit for bit for ES (for a trio: the interpreter against the nuclear kernel), to 1e-9 for BN; the
    forest fails a variant exactly when one of its families does."""
    fams, shuffle = FORESTS[name] if name in FORESTS else ([synth.trio(), synth._mk([(1, 0, 0, 1)])], None)
    ped, rows = synth.forest(fams, shuffle)
    cols = ped.sequenced_cols()
    # BN sums over the whole forest, so the other families' factors underflow on wide-range rows: gene-dropped rows only
    lk, fl = case_data(ped, cols, 801 if not bn else 60, seed=70 + len(cols), n_wide=0 if bn else 20)
    prm = fs.Params.default()
    prm.lrc = 5.0
    monkeypatch.setenv("FAMSEQ_ES_JIT", "0")
    methods = (fs.ES, fs.BN) if bn else (fs.ES,)
    with engine(ped, cols, prm) as e:
        whole = {m: e.run(m, lk, fl) for m in methods}
    assert_not_vacuous(whole[fs.ES], name, min_ok=0.5)
    for m in methods:
        failed = np.zeros(len(lk), bool)
        ok = whole[m].status == 0
        for f, r in enumerate(rows):
            fam = synth._mk([(ped.ids[i], ped.mids[i], ped.fids[i], ped.genders[i]) for i in r])
            with engine(fam, list(range(fam.n)), prm) as e:
                part = e.run(m, lk[:, r], fl)
            failed |= part.status != 0
            got_post, got_single = whole[m].post[:, r][ok], whole[m].single[:, r][ok]
            if m == fs.ES:
                assert np.array_equal(got_post, part.post[ok]) and np.array_equal(got_single, part.single[ok]), f"{name} family {f}"
                assert np.array_equal(whole[m].gt[:, r][ok], part.gt[ok])
            else:
                assert rel_err(got_post, part.post[ok]) <= REL_TOL and rel_err(got_single, part.single[ok]) <= REL_TOL, f"{name} BN family {f}"
        assert np.array_equal(whole[m].status != 0, failed), f"{name}: the forest's status is not the OR of its families'"
    if bn:
        check_bn(ped, cols, lk[:30], fl[:30], name)


# ------------------------------------------------------------------------------------------------------
# member-count boundaries
# ------------------------------------------------------------------------------------------------------
SIZES = [(63, False), (64, False), (65, False), (127, False), (128, False), (65, True), (128, True)]


@pytest.mark.parametrize("n,loops", SIZES)
def test_member_count_boundaries(n, loops, monkeypatch):
    ped = synth.random_pedigree(0 if loops else n, n, loops=loops, shuffle=n % 2 == 1)
    cols = ped.sequenced_cols()
    with engine(ped, cols, device=-1) as e:
        assert e.info()["n"] == n and e.info()["has_loop"] == int(loops)
    lk, fl = case_data(ped, cols, 801, seed=80 + n, n_wide=30)
    if not loops:
        assert_not_vacuous(check_es(ped, cols, lk, fl, monkeypatch, f"random n={n}"), f"random n={n}")
    check_mcmc(ped, cols, lk[:100], fl[:100], monkeypatch, f"random n={n}", generators=("0", "1"), burn=5, rep=40)


def test_129_members_are_refused():
    ped = synth.random_pedigree(129, 129)
    with pytest.raises(fs.FamSeqError) as ei:
        engine(ped, ped.sequenced_cols())
    assert ei.value.code == -5


# ------------------------------------------------------------------------------------------------------
# interpreter block sizes
# ------------------------------------------------------------------------------------------------------
def pick_block(s, n_slots, smem_limit):
    """es_pick_block (es_kernel.cu): the block size that keeps the most variants resident, the larger one on a tie."""
    best, best_threads = 0, 0
    for tb in (128, 64, 32):
        smem = ((s + n_slots + 3) * 3 * (tb + 1) * 8 + 15) & ~15
        need = smem + 1024
        if need > smem_limit + 1024:
            continue
        threads = min(512, (smem_limit + 1024) // need * tb)
        if threads > best_threads:
            best, best_threads = tb, threads
    return best


def es_cases():
    """The loop-free pedigrees (and input columns) this file runs ES on."""
    out = {f"sibship C={C}": sibship_case(C) for C in WIDE}
    out["three generations"] = (synth.three_generations(8), None)
    out["five spouses"] = (synth.many_spouses(5), None)
    for name, (fams, shuffle) in FORESTS.items():
        out[name] = (synth.forest(fams, shuffle)[0], None)
    for n, loops in SIZES:
        if not loops:
            out[f"random n={n}"] = (synth.random_pedigree(n, n, shuffle=n % 2 == 1), None)
    return out


def test_es_cases_reach_every_interpreter_block_size():
    torch = pytest.importorskip("torch")
    smem = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    picks = {}
    for name, (ped, cols) in es_cases().items():
        cols = ped.sequenced_cols() if cols is None else cols
        with engine(ped, cols) as e:
            info = e.info()
        picks.setdefault(pick_block(info["s"], info["es_slots"], smem), []).append(name)
    assert {128, 64, 32} <= set(picks), {k: v[:3] for k, v in picks.items()}


# ------------------------------------------------------------------------------------------------------
# tiny pedigrees
# ------------------------------------------------------------------------------------------------------
TINY = {"lone": [(1, 0, 0, 2)], "two_founders": [(1, 0, 0, 1), (2, 0, 0, 2)],
        "lone_and_trio": [(1, 0, 0, 1), (2, 0, 0, 1), (3, 0, 0, 2), (4, 3, 2, 2)]}


@pytest.mark.parametrize("name", list(TINY))
def test_tiny_pedigrees(name, monkeypatch):
    ped = synth._mk(TINY[name])
    cols = ped.sequenced_cols()
    pl, fl = synth.synth_pl(ped, 3001, seed=11, x_fraction=0.3)
    pl[5::97, 0] = 65535  # decodes to 0: the variant fails
    lk = synth.pl_to_likelihood(pl)
    interp = check_es(ped, cols, lk, fl, monkeypatch, name)
    assert host_probe(ped, cols)[1], f"{name}: the generated ES kernel must take this pedigree"
    assert (interp.status == 0).mean() > 0.9 and (interp.status != 0).any()
    check_bn(ped, cols, lk[:200], fl[:200], name)
    check_mcmc(ped, cols, lk[:200], fl[:200], monkeypatch, name, generators=("0", "1"))
    # compact input: the same doubles as the decoded likelihoods, on every method and kernel
    for jit in ("0", "1"):
        monkeypatch.setenv("FAMSEQ_ES_JIT", jit)
        monkeypatch.setenv("FAMSEQ_MCMC_JIT", jit)
        with engine(ped, cols) as e:
            for m, V in ((fs.ES, 3001), (fs.BN, 200), (fs.MCMC, 200)):
                a = e.run_pl(m, pl[:V], fl[:V], burn=10, rep=60, seed=SEED, v_offset=VOFF)
                b = e.run(m, lk[:V], fl[:V], burn=10, rep=60, seed=SEED, v_offset=VOFF)
                for k in ("status", "gt", "single", "post"):
                    assert np.array_equal(getattr(a, k), getattr(b, k)), f"{name} run_pl method {m} jit={jit}: {k}"
            assert (e.info()["jit_launches"] >= 2) == (jit == "1")
