"""The cohort Elston-Stewart path with families of any loop-free shape (fs_create_cohort: es_cohort_head_kernel,
es_cohort_kernel, es_cohort_finish_kernel) on the GPU, bit for bit:

  * against fs_create (the interpreter peeling the whole file) on forests of at most 128 members that mix extended and
    nuclear families, with shuffled rows, permuted input columns and unsequenced members, at -LRC 1, 5 and 0.5, with
    chrX / Known, wide-exponent and failing rows, through every batch entry point, with and without single;
  * against fs_create_families on nuclear-only cohorts, with the same launch count;
  * past 128 members against the C oracle peeling the whole file;
  * the whole-row failure and gate rules across program families and nuclear families;
  * several pipelines on one GPU, the BN / MCMC refusal, and the command line on a VCF of about 200 samples."""
import os
import subprocess

import numpy as np
import pytest

import famseq_b200 as fs
from famseq_b200 import synth
from oracle import oracle as O
from tests.test_families_gpu import params, run_device, same
from tests.test_pedigree_shapes_gpu import case_data

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "famseq_b200", "bin", "FamSeq")


def forest(name):
    """Forests of at most 128 members: extended families next to nuclear families and lone individuals."""
    fams = [synth.ped14(), synth.trio(), synth.half_sibs(), synth.sibship(8), synth.three_wives(), synth.sibship(2),
            synth._mk([(1, 0, 0, 2)]), synth.three_generations(2), synth.sibship(5), synth.many_spouses(3)]
    ped, rows = synth.forest(fams, shuffle_seed=None if name == "mixed" else 12)
    if name == "mixed_unseq":  # a member of ped14, of the sibship of 8 and the trio's father
        ped.names[rows[0][4]] = ped.names[rows[3][-1]] = ped.names[rows[1][0]] = "NA"
    return ped, rows


def pl_rows(ped, cols, V, seed):
    pl, _ = synth.synth_pl(synth._mk(list(zip(ped.ids, ped.mids, ped.fids, ped.genders))), V, seed=seed, x_fraction=0.3)
    pl = pl[:, cols].astype(np.uint16)
    pl[5::97, 0] = 65535  # rows that decode to zeros: failing variants
    return pl


@pytest.mark.parametrize("lrc", [1.0, 5.0, 0.5])
@pytest.mark.parametrize("name", ["mixed", "mixed_shuffled", "mixed_unseq"])
def test_cohort_engine_matches_fs_create(name, lrc):
    ped, _ = forest(name)
    assert ped.n <= 128
    cols = ped.sequenced_cols()
    cols = list(np.random.default_rng(len(cols)).permutation(cols))
    lk, fl = case_data(ped, cols, 1201, seed=40 + len(cols), n_wide=200)
    pl = pl_rows(ped, cols, 1201, seed=41)
    prm = params(lrc)
    args = (ped.ids, ped.mids, ped.fids, ped.genders, cols)
    with fs.Engine(*args, params=prm, device=0) as ref, fs.Engine(*args, params=prm, device=0, cohort=True) as got:
        assert got.info()["kernel_launches"] == 0
        for want_single in (True, False):
            same(got.run(fs.ES, lk, fl, want_single=want_single), ref.run(fs.ES, lk, fl, want_single=want_single), f"{name} run")
            same(got.run_pl(fs.ES, pl, fl, want_single=want_single), ref.run_pl(fs.ES, pl, fl, want_single=want_single), f"{name} run_pl")
            for compact in (False, True):
                x = pl if compact else lk
                same(run_device(got, x, fl, compact, want_single), run_device(ref, x, fl, compact, want_single), f"{name} device {compact}")
        a, b = got.run_pl_phred(fs.ES, pl, fl), ref.run_pl_phred(fs.ES, pl, fl)
        for k in ("post", "single", "gt", "status"):
            assert np.array_equal(getattr(a, k), getattr(b, k)), f"{name} phred {k}"
        assert a.n_fixes == b.n_fixes and np.array_equal(a.fixes, b.fixes)
        n0 = got.info()["kernel_launches"]
        r = got.run(fs.ES, lk, fl)
        assert got.info()["kernel_launches"] - n0 == 3  # one chunk: three launches, whatever the number of families
        assert 0 < r.status.sum() < len(r.status)


def test_nuclear_only_cohorts_equal_fs_create_families():
    ped, _ = synth.cohort(300, 40, 30, 20, seed=5, shuffle=True)
    cols = ped.sequenced_cols()
    lk, fl = case_data(ped, cols, 300, seed=6, n_wide=40)
    pl = pl_rows(ped, cols, 300, seed=7)
    args = (ped.ids, ped.mids, ped.fids, ped.genders, cols)
    with fs.Engine(*args, device=0, families=True) as a, fs.Engine(*args, device=0, cohort=True) as b:
        for want_single in (True, False):
            same(b.run(fs.ES, lk, fl, want_single=want_single), a.run(fs.ES, lk, fl, want_single=want_single), "run")
            same(b.run_pl(fs.ES, pl, fl, want_single=want_single), a.run_pl(fs.ES, pl, fl, want_single=want_single), "run_pl")
        assert a.info()["kernel_launches"] == b.info()["kernel_launches"] == 4


def big_cohort(seed):
    rng = np.random.default_rng(seed)
    fams = [synth.trio()] * 150 + [synth._mk([(1, 0, 0, 1 + k % 2)]) for k in range(40)]
    fams += [synth.sibship(int(k)) for k in rng.integers(6, 13, 12)]
    fams += [synth.three_generations(2), synth.half_sibs(), synth.three_wives(), synth.many_spouses(4), synth.ped14()] * 4
    fams += [synth.sibship(int(k)) for k in rng.integers(1, 6, 60)]
    return synth.forest(fams, shuffle_seed=seed)


@pytest.mark.parametrize("lrc", [1.0, 5.0])
def test_past_128_members_matches_the_oracle(lrc):
    ped, rows = big_cohort(3)
    assert 1000 < ped.n <= 1500
    ped.names[rows[200][2]] = ped.names[rows[0][0]] = "NA"
    cols = ped.sequenced_cols()
    V = 120
    lk, fl = case_data(ped, cols, V, seed=8, n_wide=V // 6)
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=params(lrc), device=0, cohort=True) as e:
        got = e.run(fs.ES, lk, fl)
        assert e.info()["kernel_launches"] == 3
    want = O.run(ped, cols, lk, fl, method=O.ES, lc=lrc)
    assert np.array_equal(got.status, want["status"])
    assert 0 < (got.status == 0).sum() < V
    assert np.array_equal(got.post, want["post"]) and np.array_equal(got.single, want["single"])
    assert np.array_equal(got.gt, (want["gt"] & 0xff).astype(np.uint8))


def test_whole_row_failure_and_gate_across_families():
    """-LRC 0.5: rows of (0.6, 0.3, 0.1) keep the pedigree out, (0.3, 0.4, 0.3) asks for it."""
    ped, rows = synth.forest([synth.trio(), synth.three_generations(2), synth.sibship(3)], shuffle_seed=2)
    cols = ped.sequenced_cols()
    S, V = len(cols), 64
    ext = [cols.index(r) for r in rows[1]]
    nuc = [cols.index(r) for r in rows[0].tolist() + rows[2].tolist()]
    lk = np.zeros((V, S, 3))
    lk[...] = (0.6, 0.3, 0.1)
    lk[0::2][:, ext] = 1e-300  # the extended family asks for the pedigree, and its products underflow: FIN sums of zero
    lk[1::4][:, ext[3]] = (0.3, 0.4, 0.3)  # one sample of the extended family asks for the pedigree: every family is peeled
    fl = (np.arange(V) % 4).astype(np.uint8)
    args = (ped.ids, ped.mids, ped.fids, ped.genders, cols)
    with fs.Engine(*args, params=params(0.5), device=0) as ref, fs.Engine(*args, params=params(0.5), device=0, cohort=True) as got:
        for want_single in (False, True):
            a, b = got.run(fs.ES, lk, fl, want_single=want_single), ref.run(fs.ES, lk, fl, want_single=want_single)
            same(a, b, "cohort vs fs_create")
    assert (a.status[0::2] == 1).all() and (a.post[0::2] == 0).all() and (a.gt[0::2] == 255).all()
    assert (a.status[1::2] == 0).all()
    # the nuclear families were peeled where only the extended family asked for it, and not where nobody did
    assert (a.post[1::4][:, nuc] != b.single[1::4][:, nuc]).any(axis=(1, 2)).all()
    assert np.array_equal(a.post[3::4], b.single[3::4])


def test_repeated_device_gives_the_same_bytes_and_bn_is_refused():
    ped, _ = big_cohort(4)
    cols = ped.sequenced_cols()
    pl = pl_rows(ped, cols, 3000, seed=2)
    _, fl = synth.synth_pl(synth.trio(), 3000, seed=3, x_fraction=0.2)
    args = (ped.ids, ped.mids, ped.fids, ped.genders, cols)
    with fs.Engine(*args, device=[0], cohort=True) as a, fs.Engine(*args, device=[0, 0, 0], cohort=True) as b:
        assert b.info()["n_devices"] == 3
        same(a.run_pl(fs.ES, pl, fl), b.run_pl(fs.ES, pl, fl), "[0] vs [0, 0, 0]")
        for method in (fs.BN, fs.MCMC):
            with pytest.raises(fs.FamSeqError) as x:
                b.run(method, synth.pl_to_likelihood(pl[:4]), fl[:4], burn=10, rep=10)
            assert x.value.code == -5 and "only Elston-Stewart" in str(x.value)


def test_cli_on_a_cohort_vcf_with_extended_families(tmp_path):
    fams = [synth.trio()] * 30 + [synth.three_generations(2), synth.half_sibs(), synth.sibship(7), synth.ped14(), synth.three_wives()] * 2
    ped, _ = synth.forest(fams, shuffle_seed=3)
    assert 128 < ped.n <= 220
    cols = ped.sequenced_cols()
    pl, fl = synth.synth_pl(ped, 300, seed=8, x_fraction=0.2)
    ped.write(str(tmp_path / "cohort.ped"))
    synth.write_vcf(str(tmp_path / "cohort.vcf"), ped, pl, fl)
    argv = [BIN, "vcf", "-vcfFile", "cohort.vcf", "-pedFile", "cohort.ped", "-method", "2"]
    outs = []
    for dev in ("0", "0,0,0"):
        out = str(tmp_path / f"out_{dev}.vcf")
        r = subprocess.run(argv + ["-device", dev, "-output", out], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        outs.append(open(out, "rb").read())
    assert outs[0] == outs[1]
    want = O.run(ped, cols, synth.pl_to_likelihood(pl), fl, method=O.ES)
    body = [line.split("\t") for line in outs[0].decode().split("\n") if line and not line.startswith("#")]
    assert len(body) == len(pl) and (want["status"] == 0).mean() > 0.8
    for v in range(len(pl)):
        if want["status"][v]:
            continue
        for s in range(len(cols)):
            fields = body[v][9 + s].split(":")  # original field, GPP, FPP, FGT
            assert fields[-2].split(",") == [O.phred_text(p) for p in want["post"][v, s]], (v, s, body[v][9 + s])
            assert fields[-3].split(",") == [O.phred_text(p) for p in want["single"][v, s]], (v, s, body[v][9 + s])
