"""Conditioned peeling (method 4, BN_PEEL: bn_peel_kernel) on the GPU:

  * on loop-free pedigrees (no loop breaker, one peel) every output byte is Elston-Stewart's, through every entry point,
    with and without single, at -LRC 1, 5 and 0.5, with chrX / Known flags, failing and wide-exponent rows;
  * on looped pedigrees of at most 31 members it is the Bayesian network's answer (fs_run(BN)) to 1e-9 relative;
  * past 31 members (ped40, random looped pedigrees of 40-128 members) it is exact variable elimination's answer;
  * repeated devices, the cohort refusal, the breaker-cap refusal at run time, and the command line's -peelLoops."""
import json
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import famseq_b200 as fs
from famseq_b200 import synth
from tests.test_bn_peel_cpu import cycle_rank, ve_marginals
from tests.test_families_gpu import params, same
from tests.test_pedigree_shapes_gpu import case_data

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "famseq_b200", "bin", "FamSeq")
GOLDEN = os.path.join(ROOT, "tests", "golden", "cli")


def engine(ped, cols=None, lrc=1.0, device=0):
    return fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols() if cols is None else cols,
                     params=params(lrc), device=device)


def run_device(e, method, x, fl, compact, want_single):
    xd = torch.from_numpy(np.ascontiguousarray(x.astype(np.int16) if compact else x)).cuda()
    V, S = x.shape[:2]
    flags = torch.from_numpy(fl).cuda()
    post = torch.empty((V, S, 3), dtype=torch.float64, device="cuda")
    single = torch.empty_like(post) if want_single else None
    gt = torch.empty((V, S), dtype=torch.uint8, device="cuda")
    status = torch.empty(V, dtype=torch.uint8, device="cuda")
    f = e.run_pl_device if compact else e.run_device
    f(method, V, xd.data_ptr(), flags.data_ptr(), post.data_ptr(), single.data_ptr() if want_single else None, gt.data_ptr(),
      status.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return fs.Result(post.cpu().numpy(), single.cpu().numpy() if want_single else None, gt.cpu().numpy(), status.cpu().numpy())


def loop_free(name):
    if name == "many_spouses":
        return synth.many_spouses(5)
    if name == "three_generations":
        return synth.three_generations()
    if name.startswith("random"):
        return synth.random_pedigree(int(name[6:]), 20 + int(name[6:]) * 9, shuffle=True, unsequenced=0.25)
    return synth.PEDIGREES[name]()


LOOP_FREE = ["trio", "ped14", "half_sibs", "three_wives", "many_spouses", "three_generations", "ped100", "random1", "random5"]


@pytest.mark.parametrize("lrc", [1.0, 5.0, 0.5])
@pytest.mark.parametrize("name", LOOP_FREE)
def test_loop_free_bytes_are_es(name, lrc):
    ped = loop_free(name)
    cols = ped.sequenced_cols()
    lk, fl = case_data(ped, cols, 1037, seed=3)
    with engine(ped, cols, lrc) as e:
        want = e.run(fs.ES, lk, fl)
        same(e.run(fs.BN_PEEL, lk, fl), want, f"{name} fs_run")
        if lrc != 1.0:
            return
        nosingle = e.run(fs.BN_PEEL, lk, fl, want_single=False)
        assert np.array_equal(nosingle.post, want.post) and np.array_equal(nosingle.gt, want.gt)
        same(run_device(e, fs.BN_PEEL, lk, fl, False, True), want, f"{name} fs_run_device")
        dev = run_device(e, fs.BN_PEEL, lk, fl, False, False)
        assert np.array_equal(dev.post, want.post) and np.array_equal(dev.status, want.status)
        pl = np.clip(np.rint(-10 * np.log10(np.maximum(lk, 1e-300))), 0, 65535).astype(np.uint16)
        wpl = e.run_pl(fs.ES, pl, fl)
        same(e.run_pl(fs.BN_PEEL, pl, fl), wpl, f"{name} fs_run_pl")
        same(run_device(e, fs.BN_PEEL, pl, fl, True, True), wpl, f"{name} fs_run_pl_device")
        ph_want, ph_got = e.run_pl_phred(fs.ES, pl, fl), e.run_pl_phred(fs.BN_PEEL, pl, fl)
        assert np.array_equal(ph_got.post, ph_want.post) and np.array_equal(ph_got.single, ph_want.single)
        assert np.array_equal(ph_got.gt, ph_want.gt) and np.array_equal(ph_got.status, ph_want.status)
        assert np.array_equal(ph_got.fixes, ph_want.fixes)
    assert (want.status == 1).any() and (want.status == 0).mean() > 0.5


def assert_bn(got, want, what, tol=1e-9):
    assert np.array_equal(got.status, want.status), f"{what}: status"
    ok = want.status == 0
    for k in ("post", "single"):
        a, b = getattr(got, k)[ok], getattr(want, k)[ok]
        nz = b != 0
        assert np.array_equal(a == 0, b == 0) or np.abs(a - b).max() < 1e-300, f"{what}: {k} zeros"
        assert (np.abs(a[nz] - b[nz]) <= tol * np.abs(b[nz])).all(), f"{what}: {k} beyond {tol} relative"
    top = np.sort(want.post[ok], axis=-1)
    clear = (top[..., 2] - top[..., 1]) > 1e-9 * top[..., 2]
    assert np.array_equal(got.gt[ok][clear], want.gt[ok][clear]), f"{what}: gt"


def looped_small():
    yield "cousins_loop", synth.cousins_loop()
    found = 0
    for seed in range(300):
        ped = synth.random_pedigree(seed, 10 + seed % 16, loops=True, shuffle=seed % 2 == 0, unsequenced=0.2)
        if cycle_rank(ped) > 0:
            yield f"random{seed}_{ped.n}", ped
            found += 1
            if found == 6:
                return


@pytest.mark.parametrize("name,ped", list(looped_small()), ids=lambda x: x if isinstance(x, str) else "")
def test_looped_matches_bn_enumeration(name, ped):
    cols = ped.sequenced_cols()
    lk, fl = case_data(ped, cols, 777, seed=8, n_wide=0)
    for lrc in (1.0, 5.0):
        with engine(ped, cols, lrc) as e:
            want = e.run(fs.BN, lk, fl)
            got = e.run(fs.BN_PEEL, lk, fl)
            dev = run_device(e, fs.BN_PEEL, lk, fl, False, True)
        assert_bn(got, want, f"{name} lrc {lrc}")
        same(dev, got, f"{name} device")
        assert (want.status == 0).mean() > 0.5


def looped_big():
    yield "ped40", synth.ped40()
    found = 0
    for seed in range(300):
        ped = synth.random_pedigree(2000 + seed, 40 + (seed * 29) % 89, loops=True, shuffle=True, unsequenced=0.2)
        if 1 <= cycle_rank(ped) <= 4:
            yield f"random{2000 + seed}_{ped.n}", ped
            found += 1
            if found == 3:
                return


@pytest.mark.parametrize("name,ped", list(looped_big()), ids=lambda x: x if isinstance(x, str) else "")
def test_looped_past_31_matches_variable_elimination(name, ped):
    cols = ped.sequenced_cols()
    V = 24
    lk, fl = synth.synth_likelihoods(ped, V, seed=4, x_fraction=0.3)
    with engine(ped, cols, 5.0) as e:
        got = e.run(fs.BN_PEEL, lk, fl)
        with pytest.raises(fs.FamSeqError) as err:
            e.run(fs.BN, lk[:1], fl[:1])
        assert err.value.code == -5
        a, xf, xm, _, _ = e.tables()
        priors = e.params.priors()
    for v in range(V):
        want = ve_marginals(ped, cols, [a, xf, xm], priors, lk[v], int(fl[v]))
        assert got.status[v] == (any(w is None for w in want) or bool((got.single[v].sum(-1) <= 0).any()))
        if got.status[v]:
            continue
        for c, r in enumerate(cols):
            b = want[r]
            assert (np.abs(got.post[v, c] - b) <= 1e-9 * np.abs(b)).all(), f"{name} variant {v} column {c}"
    assert (got.status == 0).mean() > 0.5


def test_repeated_device_gives_the_bytes_of_one_gpu():
    ped = synth.ped40()
    lk, fl = case_data(ped, ped.sequenced_cols(), 3001, seed=12)
    with engine(ped) as e:
        want = e.run(fs.BN_PEEL, lk, fl)
    with engine(ped, device=[0, 0]) as e:
        same(e.run(fs.BN_PEEL, lk, fl), want, "devices [0, 0]")


def test_cohort_engines_refuse():
    ped, _ = synth.forest([synth.trio(), synth.cousins_loop()])
    lk, fl = synth.synth_likelihoods(ped, 4, seed=1)
    for kw in ({"cohort": True}, {"cohort_bn": True}, {"cohort_mcmc": True}, {"families": True}):
        if kw.get("families") or kw.get("cohort"):
            ped_k, _ = synth.forest([synth.trio(), synth.trio()])
            lk_k, _ = synth.synth_likelihoods(ped_k, 4, seed=1)
        else:
            ped_k, lk_k = ped, lk
        with fs.Engine(ped_k.ids, ped_k.mids, ped_k.fids, ped_k.genders, ped_k.sequenced_cols(), device=0, **kw) as e:
            with pytest.raises(fs.FamSeqError) as err:
                e.run(fs.BN_PEEL, lk_k, fl)
        assert err.value.code == -1 and "fs_create" in str(err.value), kw


def test_breaker_cap_refused_at_run_time():
    ped, _ = synth.forest([synth.cousins_loop()] * 9)
    lk, fl = synth.synth_likelihoods(ped, 8, seed=1)
    with engine(ped) as e:
        with pytest.raises(fs.FamSeqError) as err:
            e.run(fs.BN_PEEL, lk, fl)
        assert err.value.code == -5 and "loop breakers" in str(err.value)
        e.run(fs.MCMC, lk, fl, burn=10, rep=20)  # the engine itself is fine


# ---- command line -------------------------------------------------------------------------------------------------
MANIFEST = json.load(open(os.path.join(GOLDEN, "manifest.json")))


def run_cli(argv, out_path):
    return subprocess.run([BIN] + argv + ["-output", out_path], cwd=GOLDEN, capture_output=True, text=True)


@pytest.mark.parametrize("name", ["vcf_trio_es", "vcf_ped14_es", "vcf_fam01_es"])
def test_cli_loop_free_bytes_are_es(name, tmp_path):
    case = MANIFEST[name]
    argv = list(case["argv"])
    k = argv.index("-method")
    argv[k:k + 2] = ["-method", "1", "-peelLoops"]
    r = run_cli(argv, str(tmp_path / "out.vcf"))
    assert r.returncode == case["returncode"] and r.stdout == case["stdout"], r.stdout + r.stderr
    assert open(tmp_path / "out.vcf").read() == open(os.path.join(GOLDEN, name + ".expected")).read()


def test_cli_cousins_matches_reference_bn(tmp_path):
    case = MANIFEST["vcf_cousins_bn"]
    r = run_cli(case["argv"] + ["-peelLoops"], str(tmp_path / "out.vcf"))
    assert r.returncode == 0 and r.stdout == case["stdout"], r.stdout + r.stderr
    got = open(tmp_path / "out.vcf").read().split("\n")
    want = open(os.path.join(GOLDEN, "vcf_cousins_bn.expected")).read().split("\n")
    assert len(got) == len(want)
    differ = total = 0
    for g, w in zip(got, want):
        gt_, wt_ = re.split(r"([\t:,])", g), re.split(r"([\t:,])", w)
        assert len(gt_) == len(wt_), f"{g}\n{w}"
        for a, b in zip(gt_, wt_):
            total += 1
            if a == b:
                continue
            x, y = float(a), float(b)  # anything but a Phred number must be identical
            differ += 1
            # six significant digits of -10 log10(p): a 1e-9 relative change of p moves it by 4.4e-9 absolute
            assert abs(x - y) <= 0.5e-5 * max(abs(y), 1e-300) + 1e-8 or (abs(x) < 1e-8 and abs(y) < 1e-8), (a, b)
    assert differ < total // 20  # nearly every number is the golden text itself


def test_cli_runs_a_40_member_looped_ped(tmp_path):
    ped = synth.ped40()
    pl, fl = synth.synth_pl(ped, 50, seed=9)
    ped.write(str(tmp_path / "ped40.ped"))
    synth.write_vcf(str(tmp_path / "ped40.vcf"), ped, pl, fl)
    argv = ["vcf", "-vcfFile", str(tmp_path / "ped40.vcf"), "-pedFile", str(tmp_path / "ped40.ped"), "-method", "1"]
    r = subprocess.run([BIN] + argv + ["-output", str(tmp_path / "bn.vcf")], capture_output=True, text=True)
    assert r.returncode != 0  # the enumeration refuses 40 members
    r = subprocess.run([BIN] + argv + ["-peelLoops", "-output", str(tmp_path / "peel.vcf")], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    body = [ln for ln in open(tmp_path / "peel.vcf").read().split("\n") if ln and not ln.startswith("#")]
    assert len(body) == 50 and all(len(ln.rstrip("\t").split("\t")) == 9 + 40 for ln in body)


def test_cli_refusals(tmp_path):
    case = MANIFEST["vcf_cousins_bn"]
    r = run_cli(case["argv"] + ["-peelLoops", "-familyBN"], str(tmp_path / "o.vcf"))
    assert r.returncode == 255 and "-familyBN" in r.stdout
    big, _ = synth.forest([synth.trio()] * 43)
    big.write(str(tmp_path / "big.ped"))
    argv = ["vcf", "-vcfFile", "trio_syn.vcf", "-pedFile", str(tmp_path / "big.ped"), "-method", "1", "-peelLoops"]
    r = run_cli(argv, str(tmp_path / "o2.vcf"))
    assert r.returncode == 255 and "at most 128" in r.stdout
    many, _ = synth.forest([synth.cousins_loop()] * 9)
    many.write(str(tmp_path / "many.ped"))
    argv = ["vcf", "-vcfFile", "trio_syn.vcf", "-pedFile", str(tmp_path / "many.ped"), "-method", "1", "-peelLoops"]
    r = run_cli(argv, str(tmp_path / "o3.vcf"))
    assert r.returncode == 255 and "loop breakers" in r.stdout
