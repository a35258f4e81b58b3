"""Host-side limits of the pedigree compilers (host-only engines, no GPU) and the ES message programs of wide sibships and
of ped files with several families, interpreted in Python and compared with the oracle bit for bit.  The GPU side of the
same shapes is tests/test_pedigree_shapes_gpu.py."""
import numpy as np
import pytest

import famseq_b200 as fs
from famseq_b200 import synth
from oracle import oracle as O
from tests.test_es_program_cpu import interpret


def host(ped, cols=None):
    return fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols() if cols is None else cols, device=-1)


def test_129_members_are_refused():
    with host(synth.random_pedigree(128, 128)) as e:
        assert e.info()["n"] == 128
    with pytest.raises(fs.FamSeqError) as ei:
        host(synth.random_pedigree(129, 129))
    assert ei.value.code == -5 and "128" in str(ei.value)


def test_es_program_word_limit_sits_at_52_children():
    """Each child's ANT lists all its full sibs, so the program grows with the square of the sibship."""
    with host(synth.sibship(51)) as e:
        words, _ = e.es_program()
        assert e.info()["es_ops"] > 0 and len(words) <= 3072
    for C in (52, 126):
        with host(synth.sibship(C)) as e:
            assert e.info()["es_ops"] == 0
            with pytest.raises(fs.FamSeqError) as ei:
                e.es_kernel()
            assert ei.value.code == -5 and "words, limit 3072" in str(ei.value)


def test_generated_es_kernel_takes_up_to_16_children():
    with host(synth.sibship(16)) as e:
        assert len(e.es_program()[0]) <= 400
        text, _ = e.es_kernel()
        assert "famseq_es" in text
    with host(synth.sibship(17)) as e:
        assert len(e.es_program()[0]) > 400
        with pytest.raises(fs.FamSeqError) as ei:
            e.es_kernel()
        assert ei.value.code == -5


def test_bn_refused_past_31_members():
    for n, levels in ((31, 31), (32, 0)):
        with host(synth.sibship(n - 2)) as e:
            assert e.info()["bn_levels"] == levels, n


def test_mcmc_plan_of_a_father_of_126():
    with host(synth.sibship(126)) as e:
        assert e.info()["mcmc_links"] == 252
        assert "128 members" in e.gibbs_kernel()[0]


def run_program(ped, cols, V, seed, what):
    """The host compiler's ES program, interpreted in Python, against the oracle (-LRC 5: the pedigree is always used)."""
    seq = synth._mk(list(zip(ped.ids, ped.mids, ped.fids, ped.genders)))
    lk, fl = synth.synth_likelihoods(seq, V, seed=seed, x_fraction=0.4)
    lk = lk[:, cols]
    want = O.run(ped, cols, lk, fl, method=O.ES, lc=5.0)
    with host(ped, cols) as e:
        words, n_slots = e.es_program()
        a, xf, xm, _, _ = e.tables()
        priors = e.params.priors()
    assert (want["status"] == 0).mean() > 0.5
    for v in range(V):
        got = interpret(words, n_slots, [a, xf, xm], priors, lk[v], int(fl[v]))
        assert (got is None) == bool(want["status"][v]), f"{what} variant {v}"
        if got is not None:
            assert np.array_equal(np.array(got), want["post"][v]), f"{what} variant {v}"


@pytest.mark.parametrize("C", [6, 7, 12, 16, 17])
def test_wide_sibship_program(C):
    ped = synth.sibship(C)
    ped.names[0] = ped.names[2 + C // 2] = "NA"
    cols = list(np.random.default_rng(C).permutation(ped.sequenced_cols()))
    run_program(ped, cols, 12, 900 + C, f"sibship C={C}")


def test_three_generation_program():
    ped = synth.three_generations(8)
    run_program(ped, ped.sequenced_cols(), 8, 31, "three generations")


@pytest.mark.parametrize("families,shuffle", [("trios21", None), ("mix", None), ("mix", 7)])
def test_forest_program(families, shuffle):
    fams = [synth.trio() for _ in range(21)] if families == "trios21" else \
        [synth.trio(), synth.ped14(), synth.half_sibs(), synth.sibship(5), synth._mk([(1, 0, 0, 2)])]
    ped, rows = synth.forest(fams, shuffle)
    assert sorted(np.concatenate(rows).tolist()) == list(range(ped.n))
    run_program(ped, ped.sequenced_cols(), 8, 60, f"{families} shuffle={shuffle}")
