"""fs_create_cohort_bn on host-only engines: the family split, looped families, refusals, build time, fs_get_info, and the
register budget of bn_cohort_kernel."""
import os
import re
import subprocess
import time

import numpy as np
import pytest

import famseq_b200 as fs
from famseq_b200 import synth

E_ARG, E_LOOP, E_TOO_LARGE = -1, -4, -5


def engine(ped, cols=None, **kw):
    cols = ped.sequenced_cols() if cols is None else cols
    return fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, device=-1, **kw)


def loop_free_forest():
    return [synth.trio(), synth.three_generations(2), synth.sibship(6), synth.half_sibs(), synth.sibship(5),
            synth._mk([(1, 0, 0, 2)]), synth.many_spouses(3), synth.ped14(), synth.three_wives(), synth._mk([(1, 0, 0, 1)])]


@pytest.mark.parametrize("shuffle", [None, 7])
def test_family_split_equals_fs_create_cohort(shuffle):
    ped, _ = synth.forest(loop_free_forest() * 3, shuffle_seed=shuffle)
    with engine(ped, cohort=True) as a, engine(ped, cohort_bn=True) as b:
        for x, y in zip(a.families(), b.families()):
            assert np.array_equal(x, y)
        assert all(b.family_program(f)[3] == -1 and len(b.family_program(f)[0]) == 0 for f in range(len(b.families()[1])))


def test_looped_families_build():
    ped, rows = synth.forest([synth.trio()] * 20 + [synth.cousins_loop()] * 2 + [synth.ped14()], shuffle_seed=3)
    with engine(ped, cohort_bn=True) as e:
        fam, kids = e.families()
        assert len(kids) == 23 and e.info()["has_loop"] == 1
        assert kids[fam[rows[20][0]]] == sum(1 for m in synth.cousins_loop().mids if m)
    with pytest.raises(fs.FamSeqError) as x:
        engine(ped, cohort=True)
    assert x.value.code == E_LOOP


def test_too_large_family_is_named():
    ped, rows = synth.forest([synth.trio()] * 50 + [synth.sibship(30)] + [synth.trio()] * 3, shuffle_seed=9)
    first_id = ped.ids[min(rows[50])]
    with pytest.raises(fs.FamSeqError) as x:
        engine(ped, cohort_bn=True)
    msg = str(x.value)
    assert x.value.code == E_TOO_LARGE and f"ped file family of {first_id}:" in msg and "31" in msg, msg


def test_ped_errors_are_those_of_fs_create():
    for rows in ([(1, 0, 0, 1), (2, 0, 0, 2), (3, 2, 9, 1)],  # a father id that is not in the file
                 [(1, 0, 0, 2), (2, 0, 0, 2), (3, 2, 1, 1)],  # a father who is not male
                 [(1, 0, 0, 1), (2, 0, 0, 2), (3, 2, 0, 1)]):  # one parent only
        ped = synth._mk(rows)
        got = []
        for kw in ({}, {"cohort_bn": True}):
            with pytest.raises(fs.FamSeqError) as x:
                fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, [0, 1, 2], device=-1, **kw)
            got.append((x.value.code, str(x.value)))
        assert got[0] == got[1] and got[0][0] < 0


@pytest.mark.parametrize("shuffle", [False, True])
def test_a_large_cohort_builds_quickly(shuffle):
    fams = [synth.trio()] * 9000 + [synth.three_generations(2)] * 1000
    ped, _ = synth.forest(fams, shuffle_seed=6 if shuffle else None)
    t0 = time.perf_counter()
    with engine(ped, cohort_bn=True) as e:
        dt = time.perf_counter() - t0
        _, kids = e.families()
    print(f"fs_create_cohort_bn: {ped.n} members, 10 000 families: {dt * 1e3:.1f} ms")
    assert dt < 1.0
    assert len(kids) == 10000 and (kids == 1).sum() == 9000


def test_info_describes_the_largest_family():
    big = synth.ped14()
    ped, _ = synth.forest([synth.trio(), big, synth.sibship(4), synth.cousins_loop()], shuffle_seed=2)
    with engine(big) as alone, engine(ped, cohort_bn=True) as e:
        want, got = alone.info(), e.info()
    assert (got["bn_levels"], got["bn_group"]) == (want["bn_levels"], want["bn_group"]) and got["bn_levels"] == big.n
    assert got["n"] == ped.n and got["es_ops"] == 0


def test_cohort_bn_kernel_register_budget():
    """The sm_100a build of bn_cohort_kernel.cu: within the 128 registers that two resident blocks of 256 threads allow
    (__launch_bounds__(256, 2), as bn_kernel), and without local memory except in the general four- and five-level
    unrolled blocks (U = 4, 5, not INDEP).  Those read the plan from shared memory where bn_kernel reads it from the
    parameter bank, and spill a few bytes (nvcc 12.9: 4 / 4 bytes of stores / loads at U = 4, 28 / 40 at U = 5, where
    bn_kernel's own U = 5 instantiation spills 24 / 36)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = os.path.join(root, "famseq_b200", "csrc", "cuda", "bn_cohort_kernel.cu")
    r = subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                        "-c", src, "-o", os.devnull], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    pat = r"Compiling entry function '\w*?bn_cohort_kernelI(Li\dELb\dELb\d)E\w*' for 'sm_100a'\n.*?\n" \
          r"\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n.*?Used (\d+) registers"
    found = re.findall(pat, r.stderr)
    assert len(found) == 13, r.stderr
    for targs, _, stores, loads, regs in found:
        if targs == "Li5ELb0ELb0":
            assert int(stores) <= 28 and int(loads) <= 40, (targs, stores, loads)
        elif targs == "Li4ELb0ELb0":
            assert int(stores) <= 4 and int(loads) <= 4, (targs, stores, loads)
        else:
            assert stores == loads == "0", (targs, stores, loads)
        assert int(regs) <= 128, (targs, regs)
