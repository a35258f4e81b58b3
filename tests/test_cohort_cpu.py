"""fs_create_cohort on host-only engines: which families of a cohort ped file get a message program of their own, how the
programs are shared, that each family's program returns the whole-file reference's doubles, what is refused, how fast a
large file builds, and the register budget of the cohort kernels."""
import os
import re
import subprocess
import time

import numpy as np
import pytest

import famseq_b200 as fs
from famseq_b200 import synth
from oracle import oracle as O
from tests.test_es_program_cpu import interpret

E_ARG, E_LOOP, E_TOO_LARGE = -1, -4, -5


def cohort_engine(ped, cols=None, params=None):
    cols = ped.sequenced_cols() if cols is None else cols
    return fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=params, device=-1, cohort=True)


def non_founders(p):
    return sum(1 for m in p.mids if m)


def test_which_families_get_programs():
    shapes = [synth.trio(), synth.three_generations(2), synth.sibship(6), synth.half_sibs(), synth.sibship(5),
              synth._mk([(1, 0, 0, 2)]), synth.many_spouses(3)]
    ped, rows = synth.forest(shapes, shuffle_seed=4)
    with cohort_engine(ped) as e:
        fam, kids = e.families()
        progs = [e.family_program(int(fam[r[0]])) for r in rows]
    by_program = [p[3] >= 0 for p in progs]
    assert by_program == [False, True, True, True, False, False, True]
    for shape, r, (words, n_slots, cols, prog) in zip(shapes, rows, progs):
        f = int(fam[r[0]])
        if prog < 0:
            assert len(words) == 0 and len(cols) == 0 and n_slots == 0
            assert kids[f] == non_founders(shape)  # what fs_create_families reports
        else:
            assert kids[f] == non_founders(shape) and len(cols) == shape.n and words[-1] == 0
            assert list(cols) == sorted(cols) and set(cols) == set(r.tolist())  # every row sequenced: column = row
    assert len({p[3] for p in progs if p[3] >= 0}) == 4


def test_identical_families_share_one_program():
    ped, rows = synth.forest([synth.three_generations(2)] * 50 + [synth.trio()] * 5)
    with cohort_engine(ped) as e:
        fam, _ = e.families()
        progs = {e.family_program(int(fam[r[0]]))[3] for r in rows[:50]}
        assert progs == {0} and e.family_program(int(fam[rows[50][0]]))[3] == -1
    ped.names[rows[17][3]] = "NA"  # one member of one family unsequenced: another program for that family
    with cohort_engine(ped) as e:
        fam, _ = e.families()
        progs = [e.family_program(int(fam[r[0]]))[3] for r in rows[:50]]
        words, _, cols, _ = e.family_program(int(fam[rows[17][0]]))
    assert sorted(set(progs)) == [0, 1] and progs.count(progs[17]) == 1
    assert len(cols) == len(rows[17]) - 1


SHAPES = {
    "three_generations": lambda: synth.three_generations(3),
    "half_sibs": synth.half_sibs,
    "three_wives": synth.three_wives,
    "many_spouses": lambda: synth.many_spouses(5),
    "sibship6": lambda: synth.sibship(6),
    "sibship16": lambda: synth.sibship(16),
    "sibship51": lambda: synth.sibship(51),
}


@pytest.mark.parametrize("name", list(SHAPES))
def test_family_programs_equal_the_whole_file_oracle(name):
    """Each program family's program, interpreted on its columns of the row, returns the oracle's doubles for the whole
    file (-LRC 5: the pedigree is always used).  Rows shuffled across families, input columns permuted, members of the
    extended family and of a trio unsequenced."""
    shapes = [synth.trio(), SHAPES[name](), synth.sibship(3), SHAPES[name](), synth._mk([(1, 0, 0, 1)])]
    ped, rows = synth.forest(shapes, shuffle_seed=len(name))
    ped.names[rows[1][1]] = ped.names[rows[1][-1]] = ped.names[rows[0][2]] = "NA"
    cols = ped.sequenced_cols()
    cols = [int(c) for c in np.random.default_rng(3).permutation(cols)]
    V = 6 if name == "sibship51" else 24
    lk, fl = synth.synth_likelihoods(synth._mk([(i + 1, 0, 0, 1) for i in range(len(cols))]), V, seed=5, x_fraction=0.4)
    want = O.run(ped, cols, lk, fl, method=O.ES, lc=5.0)
    assert (want["status"] == 0).any()
    with cohort_engine(ped, cols) as e:
        a, xf, xm, _, _ = e.tables()
        priors = e.params.priors()
        fam, _ = e.families()
        progs = [e.family_program(int(fam[rows[k][0]])) for k in (1, 3)]
    assert progs[0][3] >= 0 and progs[1][3] >= 0 and progs[0][3] != progs[1][3]  # the other one has all members sequenced
    for words, n_slots, fcols, _ in progs:
        assert len(fcols) and list(fcols) == sorted(fcols)
        for v in range(V):
            got = interpret(words, n_slots, [a, xf, xm], priors, lk[v][fcols], int(fl[v]))
            if want["status"][v]:
                continue
            assert got is not None, (name, v)
            assert np.array_equal(np.array(got), want["post"][v][fcols]), (name, v)


@pytest.mark.parametrize("shape, code, why", [(synth.cousins_loop, E_LOOP, "loop"), (lambda: synth.sibship(52), E_TOO_LARGE, "words"),
                                              (lambda: synth.sibship(127), E_TOO_LARGE, "129 members")])
def test_refusals_name_the_family(shape, code, why):
    ped, rows = synth.forest([synth.trio()] * 50 + [shape()] + [synth.three_generations(2)] * 3, shuffle_seed=9)
    first_id = ped.ids[min(rows[50])]
    with pytest.raises(fs.FamSeqError) as x:
        cohort_engine(ped)
    assert x.value.code == code
    msg = str(x.value)
    assert f"ped file family of {first_id}:" in msg and why in msg, msg


def test_ped_errors_are_those_of_fs_create():
    for rows in ([(1, 0, 0, 1), (2, 0, 0, 2), (3, 2, 9, 1)],  # a father id that is not in the file
                 [(1, 0, 0, 2), (2, 0, 0, 2), (3, 2, 1, 1)],  # a father who is not male
                 [(1, 0, 0, 1), (2, 0, 0, 2), (3, 2, 0, 1)]):  # one parent only
        ped = synth._mk(rows)
        codes, msgs = [], []
        for cohort in (False, True):
            with pytest.raises(fs.FamSeqError) as x:
                fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, [0, 1, 2], device=-1, cohort=cohort)
            codes.append(x.value.code)
            msgs.append(str(x.value))
        assert codes[0] == codes[1] < 0 and msgs[0] == msgs[1]


def test_nuclear_cohorts_match_fs_create_families_and_es_program_is_refused():
    ped, _ = synth.cohort(40, 5, 6, 4, seed=2, shuffle=True)
    args = (ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols())
    with fs.Engine(*args, device=-1, families=True) as a, fs.Engine(*args, device=-1, cohort=True) as b:
        for x, y in zip(a.families(), b.families()):
            assert np.array_equal(x, y)
        assert all(b.family_program(f)[3] == -1 for f in range(len(b.families()[1])))
        with pytest.raises(fs.FamSeqError) as x:
            b.es_program()
        assert x.value.code == E_TOO_LARGE
        with pytest.raises(fs.FamSeqError) as x:
            b.family_program(len(b.families()[1]))
        assert x.value.code == E_ARG


@pytest.mark.parametrize("shuffle", [False, True])
def test_a_large_cohort_with_extended_families_builds_quickly(shuffle):
    """10 000 families, 1 000 of them three-generation families, the rest trios.  In file order the 1 000 share one
    program; with the rows shuffled across families each has its own member order, so each compiles its own."""
    fams = [synth.trio()] * 9000 + [synth.three_generations(3)] * 1000
    ped, _ = synth.forest(fams, shuffle_seed=6 if shuffle else None)
    t0 = time.perf_counter()
    with cohort_engine(ped) as e:
        fam, kids = e.families()
        dt = time.perf_counter() - t0
        programs = {e.family_program(f)[3] for f in range(10000)}
    print(f"fs_create_cohort: {ped.n} members, 10 000 families, {len(programs) - 1} programs: {dt * 1e3:.1f} ms")
    assert dt < 1.0
    assert len(kids) == 10000 and (kids == 1).sum() == 9000 and (kids == non_founders(synth.three_generations(3))).sum() == 1000
    assert len(programs) == (1001 if shuffle else 2) and -1 in programs


def test_cohort_kernel_register_budget():
    """The sm_100a build of es_cohort_kernel.cu: the program kernel and the finish pass without local memory; the head
    kernel as es_families_kernel (tests/test_families_cpu.py): no local memory up to four children, and with five
    peel<5> alone takes nearly all 255 registers, so a few bytes spill (20 stores, 32 loads with nvcc 12.9)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = os.path.join(root, "famseq_b200", "csrc", "cuda", "es_cohort_kernel.cu")
    r = subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false", "-Xptxas", "-v",
                        "-c", src, "-o", os.devnull], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    pat = r"Compiling entry function '\w*?(es_cohort_kernel|es_cohort_finish_kernel|es_cohort_head_kernel)I(\w*?)E\w*' for 'sm_100a'\n.*?\n" \
          r"\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n.*?Used (\d+) registers"
    found = re.findall(pat, r.stderr)
    kinds = [k for k, *_ in found]
    assert kinds.count("es_cohort_kernel") == 6 and kinds.count("es_cohort_finish_kernel") == 2, r.stderr
    assert kinds.count("es_cohort_head_kernel") == 24, r.stderr
    for kind, targs, _, stores, loads, regs in found:
        if kind == "es_cohort_head_kernel" and targs.startswith("Li5"):
            assert int(stores) <= 24 and int(loads) <= 32, (kind, targs, stores, loads)
        else:
            assert stores == loads == "0", (kind, targs, stores, loads)
        if kind == "es_cohort_kernel":
            assert int(regs) <= 128, (targs, regs)  # 512 threads per SM, as es_pick_block assumes
