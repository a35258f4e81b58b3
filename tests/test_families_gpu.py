"""The cohort Elston-Stewart path (fs_create_families, es_families_kernel) on the GPU, bit for bit:

  * against fs_create on forests both constructors take (2, 21, 42 trios; sibships of 1..5 with lone individuals; shuffled
    rows, permuted input columns, an unsequenced father and child), at -LRC 1, 5 and 0.5 (the whole-file gate keeps the
    pedigree out of some rows), chrX and Known rows, wide-exponent rows and failing rows, through every batch entry point;
  * past 128 members against the C oracle peeling the whole file, and a 3 000-trio cohort against its families run one
    by one with the whole-file gate and failure rule applied in numpy;
  * several pipelines on one GPU, and the command line on a 180-sample VCF."""
import os
import subprocess

import numpy as np
import pytest
import torch

import famseq_b200 as fs
from famseq_b200 import synth
from oracle import oracle as O
from tests.test_pedigree_shapes_gpu import case_data

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "famseq_b200", "bin", "FamSeq")


def params(lrc):
    p = fs.Params.default()
    p.lrc = lrc
    return p


def unseq(ped, rows):
    """Marks the father of the first family and a child of the last one with children unsequenced."""
    first, last = rows[0], next(r for r in reversed(rows) if len(r) > 1)
    father = next(i for i in first if ped.mids[i] == 0 and ped.genders[i] == 1)
    child = next(i for i in last if ped.mids[i] != 0)
    ped.names[father] = ped.names[child] = "NA"
    return ped


def forest(name):
    if name.startswith("trios"):
        return synth.forest([synth.trio()] * int(name[5:]))
    fams = [synth.sibship(k) for k in (1, 2, 3, 4, 5, 2, 1)] + [synth._mk([(1, 0, 0, 1 + k % 2)]) for k in range(3)]
    return synth.forest(fams, shuffle_seed=5 if name == "mix_shuffled" else None)


FORESTS = ["trios2", "trios21", "trios42", "mix", "mix_shuffled", "mix_unseq"]


def same(a, b, what):
    assert np.array_equal(a.status, b.status), f"{what}: status"
    assert np.array_equal(a.post, b.post, equal_nan=True), f"{what}: post"
    assert np.array_equal(a.gt, b.gt), f"{what}: gt"
    if a.single is not None or b.single is not None:
        assert np.array_equal(a.single, b.single, equal_nan=True), f"{what}: single"


def run_device(e, pl_or_lk, fl, compact, want_single):
    """run_device / run_pl_device on torch buffers; returns a Result."""
    x = torch.from_numpy(np.ascontiguousarray(pl_or_lk.astype(np.int16) if compact else pl_or_lk)).cuda()
    V, S = pl_or_lk.shape[:2]
    flags = torch.from_numpy(fl).cuda()
    post = torch.empty((V, S, 3), dtype=torch.float64, device="cuda")
    single = torch.empty_like(post) if want_single else None
    gt = torch.empty((V, S), dtype=torch.uint8, device="cuda")
    status = torch.empty(V, dtype=torch.uint8, device="cuda")
    f = e.run_pl_device if compact else e.run_device
    f(fs.ES, V, x.data_ptr(), flags.data_ptr(), post.data_ptr(), single.data_ptr() if want_single else None, gt.data_ptr(),
      status.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return fs.Result(post.cpu().numpy(), single.cpu().numpy() if want_single else None, gt.cpu().numpy(), status.cpu().numpy())


@pytest.mark.parametrize("lrc", [1.0, 5.0, 0.5])
@pytest.mark.parametrize("name", FORESTS)
def test_cohort_engine_matches_fs_create(name, lrc):
    ped, rows = forest(name)
    if name == "mix_unseq":
        ped = unseq(ped, rows)
    cols = ped.sequenced_cols()
    cols = list(np.random.default_rng(len(cols)).permutation(cols))  # input columns in another order than the ped rows
    lk, fl = case_data(ped, cols, 1201, seed=90 + len(cols), n_wide=200)
    pl, _ = synth.synth_pl(synth._mk(list(zip(ped.ids, ped.mids, ped.fids, ped.genders))), 1201, seed=91, x_fraction=0.3)
    pl = pl[:, cols].astype(np.uint16)
    pl[5::97, 0] = 65535  # rows that decode to zeros: failing variants
    prm = params(lrc)
    args = (ped.ids, ped.mids, ped.fids, ped.genders, cols)
    with fs.Engine(*args, params=prm, device=0) as ref, fs.Engine(*args, params=prm, device=0, families=True) as got:
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
        info = got.info()
        assert info["es_ops"] == 0 and info["device"] == 0 and info["n"] == ped.n and info["s"] == len(cols)


@pytest.mark.parametrize("lrc", [1.0, 5.0])
@pytest.mark.parametrize("which", ["trios43", "cohort"])
def test_past_128_members_matches_the_oracle(which, lrc):
    ped, _ = synth.forest([synth.trio()] * 43) if which == "trios43" else synth.cohort(300, 50, 20, 20, seed=3, shuffle=True)
    cols = ped.sequenced_cols()
    V = 301 if which == "trios43" else 120
    lk, fl = case_data(ped, cols, V, seed=7, n_wide=V // 6)
    with pytest.raises(fs.FamSeqError):
        fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, device=-1)
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=params(lrc), device=0, families=True) as e:
        got = e.run(fs.ES, lk, fl)
    want = O.run(ped, cols, lk, fl, method=O.ES, lc=lrc)
    assert np.array_equal(got.status, want["status"])
    assert 0 < (got.status == 0).sum() < V
    assert np.array_equal(got.post, want["post"]) and np.array_equal(got.single, want["single"])
    assert np.array_equal(got.gt, (want["gt"] & 0xff).astype(np.uint8))


def test_3000_trios_equal_their_families_with_the_whole_file_rules():
    """-LRC 1 on the cohort = each trio at -LRC 5 on an fs_create engine, then the gate and failure of the whole row."""
    T, V, chunk = 3000, 10240, 1024
    ped, _ = synth.forest([synth.trio()] * T)
    cols = ped.sequenced_cols()
    S = len(cols)
    trio = synth.trio()
    male = np.array([ped.genders[c] == 1 for c in cols])
    pri = fs.Params.default().priors()
    rng = np.random.default_rng(11)
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, device=0, families=True) as e, \
            fs.Engine(trio.ids, trio.mids, trio.fids, trio.genders, [0, 1, 2], params=params(5.0), device=0) as t:
        for v0 in range(0, V, chunk):
            pl = rng.integers(0, 40, (chunk, S, 3)).astype(np.uint16)
            pl[np.arange(chunk)[:, None], np.arange(S)[None, :], rng.integers(0, 3, (chunk, S))] = 0
            pl[::7] = np.minimum(pl[::7], 2)  # nearly uninformative rows: most samples want the pedigree
            pl[1::9] = (0, 5000, 5000)  # certain samples only (every PL >= 3240 decodes to 0): the gate keeps the pedigree out
            pl[3::101, S // 2] = 65535  # an all-zero likelihood row: the variant fails
            fl = rng.integers(0, 4, chunk).astype(np.uint8)
            got = e.run_pl(fs.ES, pl, fl)
            fam = t.run_pl(fs.ES, pl.reshape(chunk * T, 3, 3), np.repeat(fl, T))
            post = fam.post.reshape(chunk, S, 3)
            single = fam.single.reshape(chunk, S, 3)
            gt = fam.gt.reshape(chunk, S)
            lk = synth.pl_table()[pl]
            big, ls = lk.max(-1), (lk[..., 0] + lk[..., 1]) + lk[..., 2]
            needed = (big < ls).any(1)
            chrx, known = (fl >> 1) & 1, fl & 1
            prior = np.where((chrx[:, None] == 1) & male[None, :], 2 + known[:, None], known[:, None])  # [V][S] prior row
            r = lk * pri[prior]
            ind_fail = (((r[..., 0] + r[..., 1]) + r[..., 2]) <= 0).any(1)
            failed = ind_fail | (needed & (fam.status.reshape(chunk, T) != 0).any(1))
            # FPP := GPP where no sample asks for the pedigree
            post = np.where(needed[:, None, None], post, single)
            single_gt = np.where(single.max(-1) > -1, single.argmax(-1), 255).astype(np.uint8)
            gt = np.where(needed[:, None], gt, single_gt)
            post[failed], single[failed], gt[failed] = 0.0, 0.0, 255
            assert needed.all() == False and needed.any(), "the gate must keep the pedigree out of some rows only"  # noqa: E712
            assert failed.any() and not failed.all()
            assert np.array_equal(got.status, failed.astype(np.uint8)), v0
            assert np.array_equal(got.post, post) and np.array_equal(got.single, single) and np.array_equal(got.gt, gt), v0


def test_repeated_device_gives_the_same_bytes():
    ped, _ = synth.cohort(200, 20, 10, 5, seed=4, shuffle=True)
    cols = ped.sequenced_cols()
    pl, fl = synth.synth_pl(synth._mk(list(zip(ped.ids, ped.mids, ped.fids, ped.genders))), 5000, seed=2, x_fraction=0.2)
    pl = pl[:, cols].astype(np.uint16)
    args = (ped.ids, ped.mids, ped.fids, ped.genders, cols)
    with fs.Engine(*args, device=[0], families=True) as a, fs.Engine(*args, device=[0, 0, 0], families=True) as b:
        assert b.info()["n_devices"] == 3
        same(a.run_pl(fs.ES, pl, fl), b.run_pl(fs.ES, pl, fl), "[0] vs [0, 0, 0]")
        with pytest.raises(fs.FamSeqError) as x:
            b.run(fs.BN, synth.pl_to_likelihood(pl[:4]), fl[:4])
        assert x.value.code == -5 and "only Elston-Stewart" in str(x.value)


def test_cli_on_a_cohort_vcf(tmp_path):
    ped, _ = synth.forest([synth.trio()] * 60)
    cols = ped.sequenced_cols()
    pl, fl = synth.synth_pl(ped, 400, seed=8, x_fraction=0.2)
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
    assert len(body) == len(pl) and (want["status"] == 0).mean() > 0.9
    for v in range(len(pl)):
        if want["status"][v]:
            continue
        for s in range(len(cols)):
            fields = body[v][9 + s].split(":")  # original field, GPP, FPP, FGT
            assert fields[-2].split(",") == [O.phred_text(p) for p in want["post"][v, s]], (v, s, body[v][9 + s])
            assert fields[-3].split(",") == [O.phred_text(p) for p in want["single"][v, s]], (v, s, body[v][9 + s])
    r = subprocess.run(argv[:-1] + ["1", "-output", str(tmp_path / "bn.vcf")], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode != 0 and "only Elston-Stewart" in r.stdout + r.stderr
