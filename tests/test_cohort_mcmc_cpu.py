"""fs_create_cohort_mcmc on host-only engines: the family split, looped families past the BN limit, refusals, build time,
fs_get_info, and the register budget of mcmc_cohort_kernel."""
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


def mixed_forest():
    return [synth.trio(), synth.three_generations(2), synth.sibship(6), synth.half_sibs(), synth.cousins_loop(), synth.sibship(5),
            synth._mk([(1, 0, 0, 2)]), synth.many_spouses(3), synth.ped14(), synth.three_wives(), synth._mk([(1, 0, 0, 1)])]


@pytest.mark.parametrize("shuffle", [None, 7])
def test_family_split_equals_fs_create_cohort_bn(shuffle):
    ped, _ = synth.forest(mixed_forest() * 3, shuffle_seed=shuffle)
    with engine(ped, cohort_bn=True) as a, engine(ped, cohort_mcmc=True) as b:
        for x, y in zip(a.families(), b.families()):
            assert np.array_equal(x, y)
        assert all(b.family_program(f)[3] == -1 for f in range(len(b.families()[1])))


@pytest.mark.parametrize("looped", ["ped40", "cousins_loop"])
def test_cohorts_the_other_constructors_refuse_build(looped):
    big = getattr(synth, looped)()
    ped, rows = synth.forest([synth.trio()] * 50 + [big] + [synth.sibship(3)] * 4, shuffle_seed=3)
    assert ped.n > 128
    with engine(ped, cohort_mcmc=True) as e:
        fam, kids = e.families()
        info = e.info()
    assert len(kids) == 55 and info["has_loop"] == 1 and info["gibbs_generator"] == 0
    assert kids[fam[rows[50][0]]] == sum(1 for m in big.mids if m)
    with engine(big) as alone:  # fs_get_info: the largest family's plan
        assert info["mcmc_links"] == alone.info()["mcmc_links"]
    with pytest.raises(fs.FamSeqError) as x:
        engine(ped, cohort=True)
    assert x.value.code == E_LOOP
    if looped == "ped40":
        with pytest.raises(fs.FamSeqError) as x:
            engine(ped, cohort_bn=True)
        assert x.value.code == E_TOO_LARGE


def test_too_large_family_is_named():
    ped, rows = synth.forest([synth.trio()] * 20 + [synth.sibship(127)] + [synth.trio()] * 3, shuffle_seed=9)
    assert len(rows[20]) == 129
    first_id = ped.ids[min(rows[20])]
    with pytest.raises(fs.FamSeqError) as x:
        engine(ped, cohort_mcmc=True)
    msg = str(x.value)
    assert x.value.code == E_TOO_LARGE and f"ped file family of {first_id}:" in msg and "128" in msg, msg
    ped, _ = synth.forest([synth.trio()] * 20 + [synth.sibship(126)], shuffle_seed=9)  # 128 members: taken
    with engine(ped, cohort_mcmc=True) as e:
        assert len(e.families()[1]) == 21


def test_ped_errors_are_those_of_fs_create():
    for rows in ([(1, 0, 0, 1), (2, 0, 0, 2), (3, 2, 9, 1)],  # a father id that is not in the file
                 [(1, 0, 0, 2), (2, 0, 0, 2), (3, 2, 1, 1)],  # a father who is not male
                 [(1, 0, 0, 1), (2, 0, 0, 2), (3, 2, 0, 1)]):  # one parent only
        ped = synth._mk(rows)
        got = []
        for kw in ({}, {"cohort_mcmc": True}):
            with pytest.raises(fs.FamSeqError) as x:
                fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, [0, 1, 2], device=-1, **kw)
            got.append((x.value.code, str(x.value)))
        assert got[0] == got[1] and got[0][0] < 0


@pytest.mark.parametrize("shuffle", [False, True])
def test_a_large_cohort_builds_quickly(shuffle):
    fams = [synth.trio()] * 9000 + [synth.three_generations(2)] * 990 + [synth.ped40()] * 10
    ped, _ = synth.forest(fams, shuffle_seed=6 if shuffle else None)
    t0 = time.perf_counter()
    with engine(ped, cohort_mcmc=True) as e:
        dt = time.perf_counter() - t0
        _, kids = e.families()
    print(f"fs_create_cohort_mcmc: {ped.n} members, 10 000 families: {dt * 1e3:.1f} ms")
    assert dt < 1.0
    assert len(kids) == 10000 and (kids == 1).sum() == 9000


def test_mcmc_cohort_kernel_register_budget():
    """The sm_100a build of mcmc_cohort_kernel.cu, compiled as the Makefile does: no spills, and few enough registers that
    a block of 256 chains (the largest block size the launcher picks) fits an SM's 64 K registers four times over.  The
    genotype vector of the 64- and 128-member classes sits in a 16- / 32-byte stack frame, as in mcmc_kernel (nvcc 12.9:
    48, 48 and 44 registers for GW = 1, 2, 4)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = os.path.join(root, "famseq_b200", "csrc", "cuda", "mcmc_cohort_kernel.cu")
    r = subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                        "-c", src, "-o", os.devnull], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    pat = r"Compiling entry function '\w*?mcmc_cohort_kernelILi(\d)E\w*' for 'sm_100a'\n.*?\n" \
          r"\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n.*?Used (\d+) registers"
    found = re.findall(pat, r.stderr)
    assert sorted(f[0] for f in found) == ["1", "2", "4"], r.stderr
    for gw, stack, stores, loads, regs in found:
        assert stores == loads == "0", (gw, stores, loads)
        assert int(stack) <= 8 * int(gw), (gw, stack)
        assert int(regs) * 256 * 4 <= 65536, (gw, regs)
