"""fs_create_families on host-only engines: how a cohort ped file is split into families, which family shapes it takes and
refuses, and how fast a large file builds."""
import time

import numpy as np
import pytest

import famseq_b200 as fs
from famseq_b200 import synth

E_TOO_LARGE, E_HALF_PARENTS, E_GENDER, E_ARG = -5, -2, -3, -1


def cohort_engine(ped, cols=None, device=-1):
    cols = ped.sequenced_cols() if cols is None else cols
    return fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, device=device, families=True)


def expected_families(ped):
    """(family[n], n_children[F]) from the ped rows, families numbered by their first row."""
    par = ped.parents()
    root = list(range(ped.n))

    def find(x):
        while root[x] != x:
            x = root[x]
        return x
    for i, (m, f) in enumerate(par):
        if m >= 0:
            root[find(i)] = find(m)
            root[find(i)] = find(f)
    index, fam = {}, []
    for i in range(ped.n):
        fam.append(index.setdefault(find(i), len(index)))
    kids = [0] * len(index)
    for i, (m, _) in enumerate(par):
        if m >= 0:
            kids[fam[i]] += 1
    return np.array(fam), np.array(kids)


@pytest.mark.parametrize("shuffle", [False, True])
def test_families_and_children_counts(shuffle):
    ped, rows = synth.cohort(7, 3, 6, 4, seed=2, shuffle=shuffle)
    with cohort_engine(ped) as e:
        fam, kids = e.families()
        info = e.info()
    want_fam, want_kids = expected_families(ped)
    assert np.array_equal(fam, want_fam) and np.array_equal(kids, want_kids)
    assert sorted(np.bincount(kids)[1:3].tolist()) == [3, 7] and (kids == 0).sum() == 4 and len(kids) == 20
    assert all(len(set(fam[r])) == 1 for r in rows)  # every family of the builder is one family of the engine
    assert fam[0] == 0 and np.all(np.diff(np.maximum.accumulate(fam)) <= 1)  # numbered by first row
    assert info["n"] == ped.n and info["s"] == ped.n and info["device"] == -1 and info["es_ops"] == 0


def test_sibships_of_one_to_five_with_unsequenced_members():
    ped, rows = synth.forest([synth.sibship(k) for k in (5, 1, 4, 2, 3)] + [synth._mk([(1, 0, 0, 2)])], shuffle_seed=3)
    ped.names[rows[0][0]] = "NA"  # a father
    ped.names[rows[2][-1]] = "NA"  # a child
    ped.names[rows[5][0]] = "NA"  # the lone individual
    with cohort_engine(ped) as e:
        fam, kids = e.families()
        assert e.info()["s"] == ped.n - 3
    want_fam, want_kids = expected_families(ped)
    assert np.array_equal(fam, want_fam) and sorted(kids.tolist()) == [0, 1, 2, 3, 4, 5]


def test_a_large_cohort_builds_quickly():
    ped, _ = synth.cohort(10000)
    t0 = time.perf_counter()
    with cohort_engine(ped) as e:
        fam, kids = e.families()
    assert time.perf_counter() - t0 < 0.5
    assert len(kids) == 10000 and (kids == 1).all() and fam[-1] == 9999


@pytest.mark.parametrize("shape, why", [(lambda: synth._mk([(1, 0, 0, 1), (2, 0, 0, 2), (3, 0, 0, 2), (4, 2, 1, 1), (5, 3, 1, 2)]), "half-sibs"), (lambda: synth.three_generations(2), "generations"),
                                        (lambda: synth.sibship(6), "6 children")])
def test_other_family_shapes_are_refused(shape, why):
    ped, rows = synth.forest([synth.trio()] * 50 + [shape()] + [synth.trio()] * 3, shuffle_seed=9)
    first_id = ped.ids[min(rows[50])]
    with pytest.raises(fs.FamSeqError) as x:
        cohort_engine(ped)
    assert x.value.code == E_TOO_LARGE
    msg = str(x.value)
    assert f"family of {first_id}:" in msg and why in msg, msg


def test_ped_errors_are_those_of_fs_create():
    for rows in ([(1, 0, 0, 1), (2, 0, 0, 2), (3, 2, 9, 1)],  # a father id that is not in the file
                 [(1, 0, 0, 2), (2, 0, 0, 2), (3, 2, 1, 1)]):  # a father who is not male
        ped = synth._mk(rows)
        codes, msgs = [], []
        for families in (False, True):
            with pytest.raises(fs.FamSeqError) as x:
                fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, [0, 1, 2], device=-1, families=families)
            codes.append(x.value.code)
            msgs.append(str(x.value))
        assert codes[0] == codes[1] in (E_HALF_PARENTS, E_GENDER) and msgs[0] == msgs[1]


def test_bn_and_mcmc_are_refused_and_fs_create_keeps_its_limit():
    ped, _ = synth.forest([synth.trio()] * 43)
    with pytest.raises(fs.FamSeqError) as x:
        fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols(), device=-1)
    assert x.value.code == E_TOO_LARGE
    with cohort_engine(ped) as e:  # (BN and MCMC runs are refused on the GPU: tests/test_families_gpu.py)
        with pytest.raises(fs.FamSeqError) as x:
            e.es_program()
        assert x.value.code == E_TOO_LARGE
    trio = synth.trio()
    with fs.Engine(trio.ids, trio.mids, trio.fids, trio.genders, [0, 1, 2], device=-1) as e:
        with pytest.raises(fs.FamSeqError) as x:
            e.families()
        assert x.value.code == E_ARG


def test_cohort_kernel_register_budget():
    """The sm_100a build of every es_families_kernel instantiation.  Cohorts whose largest sibship has at most four children
    run without local memory; with five, peel<5> alone takes nearly all 255 registers and 16 bytes spill."""
    import os
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = os.path.join(root, "famseq_b200", "csrc", "cuda", "es_families_kernel.cu")
    r = subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false", "-Xptxas", "-v",
                        "-c", src, "-o", os.devnull], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    found = re.findall(r"Compiling entry function '\w*es_families_kernelILi(\d)E\w*' for 'sm_100a'\n.*?\n\s*(\d+) bytes stack frame, "
                       r"(\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr)
    assert len(found) == 24, r.stderr
    for nc_max, _, stores, loads in found:
        if int(nc_max) < 5:
            assert stores == loads == "0", (nc_max, stores, loads)
        else:
            assert int(stores) <= 16 and int(loads) <= 32, (nc_max, stores, loads)
