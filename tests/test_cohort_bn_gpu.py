"""The Bayesian network for cohort ped files (fs_create_cohort_bn: es_cohort_head_kernel, bn_cohort_kernel once per launch
class, es_cohort_finish_kernel) on the GPU:

  * each family's columns bit for bit as fs_create BN on that family alone, looped families included, with shuffled rows,
    permuted input columns and unsequenced members;
  * the whole-row gate and failure rules past 128 members, through every batch entry point, with and without single;
  * the C oracle's BN on each family, and fs_create BN on whole forests of at most 31 members;
  * the launch count, repeated devices, the ES / MCMC refusal, and the command line's -familyBN."""
import os
import subprocess

import numpy as np
import pytest
import torch

import famseq_b200 as fs
from famseq_b200 import synth
from famseq_b200.engine import PHRED_FIX_SINGLE, PHRED_KIND_FIX, phred_text, phred_text_exact
from oracle import oracle as O
from tests.test_families_gpu import params, same
from tests.test_pedigree_shapes_gpu import case_data

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "famseq_b200", "bin", "FamSeq")


def mixed(shuffle_seed=None):
    fams = [synth.trio(), synth._mk([(1, 0, 0, 1)]), synth.sibship(5), synth._mk([(1, 0, 0, 2)]), synth.sibship(8),
            synth.half_sibs(), synth.three_wives(), synth.three_generations(2), synth.many_spouses(3), synth.cousins_loop(),
            synth.ped14(), synth.trio()]
    return synth.forest(fams, shuffle_seed=shuffle_seed)


def family_engine(ped, rows, cols, prm):
    """fs_create on one family alone: its rows in file order, its sequenced members as columns in increasing global column.
    Returns (engine, global columns)."""
    rows = sorted(int(r) for r in rows)
    local = {r: k for k, r in enumerate(rows)}
    gcols = [c for c in range(len(cols)) if cols[c] in local]
    e = fs.Engine([ped.ids[r] for r in rows], [ped.mids[r] for r in rows], [ped.fids[r] for r in rows],
                  [ped.genders[r] for r in rows], [local[cols[c]] for c in gcols], params=prm, device=0)
    return e, gcols


def run_device(e, x, fl, compact, want_single):
    """run_device / run_pl_device (BN) on torch buffers; returns a Result."""
    xd = torch.from_numpy(np.ascontiguousarray(x.astype(np.int16) if compact else x)).cuda()
    V, S = x.shape[:2]
    flags = torch.from_numpy(fl).cuda()
    post = torch.empty((V, S, 3), dtype=torch.float64, device="cuda")
    single = torch.empty_like(post) if want_single else None
    gt = torch.empty((V, S), dtype=torch.uint8, device="cuda")
    status = torch.empty(V, dtype=torch.uint8, device="cuda")
    f = e.run_pl_device if compact else e.run_device
    f(fs.BN, V, xd.data_ptr(), flags.data_ptr(), post.data_ptr(), single.data_ptr() if want_single else None, gt.data_ptr(),
      status.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return fs.Result(post.cpu().numpy(), single.cpu().numpy() if want_single else None, gt.cpu().numpy(), status.cpu().numpy())


@pytest.mark.parametrize("name", ["file_order", "shuffled", "unsequenced"])
def test_each_family_equals_fs_create_on_that_family_alone(name):
    ped, rows = mixed(None if name == "file_order" else 17)
    if name == "unsequenced":  # a member of the looped family, of ped14 and the father of the first trio
        ped.names[rows[9][2]] = ped.names[rows[10][5]] = ped.names[rows[0][0]] = "NA"
    cols = [int(c) for c in np.random.default_rng(len(ped.sequenced_cols())).permutation(ped.sequenced_cols())]
    V = 301
    lk, fl = case_data(ped, cols, V, seed=60, n_wide=60)
    prm = params(5.0)
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=prm, device=0, cohort_bn=True) as e:
        got = e.run(fs.BN, lk, fl)
        assert e.info()["has_loop"] == 1
    status = np.zeros(V, np.uint8)
    for r in rows:
        fe, gcols = family_engine(ped, r, cols, prm)
        with fe:
            want = fe.run(fs.BN, lk[:, gcols], fl)
        status |= want.status
        ok = got.status == 0
        for k in ("post", "single", "gt"):
            assert np.array_equal(getattr(got, k)[ok][:, gcols], getattr(want, k)[ok]), (name, r[0], k)
    assert np.array_equal(got.status, status)
    assert 0 < got.status.sum() < V // 2


def reassemble(ped, rows, cols, lk, fl, prm):
    """The cohort's outputs from per-family runs, with the whole-row gate and failure rule applied in numpy.  -LRC 0 never
    uses the pedigree: its runs give the individual-only posteriors and the failures that do not depend on the pedigree;
    -LRC 5 always uses it: its runs give the BN posteriors and the BN failures."""
    V, S = lk.shape[:2]
    post, single, gt, single_gt = np.zeros((V, S, 3)), np.zeros((V, S, 3)), np.zeros((V, S), np.uint8), np.zeros((V, S), np.uint8)
    failed, bn_failed = np.zeros(V, bool), np.zeros(V, bool)
    for r in rows:
        for lrc in (0.0, 5.0):
            fe, gcols = family_engine(ped, r, cols, params(lrc))
            with fe:
                w = fe.run(fs.BN, lk[:, gcols], fl)
            if lrc == 0.0:
                single[:, gcols], single_gt[:, gcols] = w.single, w.gt
                failed |= w.status.astype(bool)
            else:
                post[:, gcols], gt[:, gcols] = w.post, w.gt
                bn_failed |= w.status.astype(bool)
    big, ls = lk.max(axis=2), (lk[..., 0] + lk[..., 1]) + lk[..., 2]
    needed = (big / ls < prm.lrc).any(axis=1)
    failed |= needed & bn_failed
    post = np.where(needed[:, None, None], post, single)
    gt = np.where(needed[:, None], gt, single_gt)
    post[failed], single[failed], gt[failed] = 0.0, 0.0, 255
    return fs.Result(post, single, gt, failed.astype(np.uint8))


@pytest.mark.parametrize("lrc", [1.0, 0.5])
def test_whole_row_rules_past_128_members_through_every_entry_point(lrc):
    fams = [synth.trio()] * 40 + [synth.cousins_loop(), synth.sibship(4), synth.half_sibs(), synth._mk([(1, 0, 0, 2)])]
    ped, rows = synth.forest(fams, shuffle_seed=4)
    assert ped.n > 128
    cols = ped.sequenced_cols()
    S, V = len(cols), 500
    pl, fl = synth.synth_pl(ped, V, seed=9, x_fraction=0.3)
    pl = pl.astype(np.uint16)
    pl[7::23, 5] = 65535  # rows that decode to zeros: failing variants
    pl[1::3] = np.where(pl[1::3] == 0, 0, 4000).astype(np.uint16)  # likelihoods (1, 0, 0): the gate keeps the pedigree out
    lk = synth.pl_to_likelihood(pl)
    prm = params(lrc)
    want = reassemble(ped, rows, cols, lk, fl, prm)
    assert 0 < want.status.sum() < V // 4
    args = (ped.ids, ped.mids, ped.fids, ped.genders, cols)
    with fs.Engine(*args, params=prm, device=0, cohort_bn=True) as e:
        for want_single in (True, False):
            w = want if want_single else fs.Result(want.post, None, want.gt, want.status)
            same(e.run(fs.BN, lk, fl, want_single=want_single), w, "run")
            same(e.run_pl(fs.BN, pl, fl, want_single=want_single), w, "run_pl")
            for compact in (False, True):
                same(run_device(e, pl if compact else lk, fl, compact, want_single), w, f"device {compact}")
        a, b = e.run_pl_phred(fs.BN, pl, fl), e.run_pl(fs.BN, pl, fl)
        codes, _, _ = e.phred_encode(b.post)
        assert np.array_equal(a.status, b.status) and np.array_equal(a.gt, b.gt)
        assert np.array_equal(a.post[a.post >> 30 != PHRED_KIND_FIX], codes[a.post >> 30 != PHRED_KIND_FIX])
    if lrc == 1.0:  # the gate both ways
        kept = (want.post == want.single).all(axis=(1, 2)) & (want.status == 0)
        assert 0 < kept.sum() < V


def test_against_the_oracle_and_fs_create_on_small_forests():
    fams = [synth.trio(), synth.sibship(2), synth._mk([(1, 0, 0, 1)]), synth.cousins_loop()]
    ped, rows = synth.forest(fams, shuffle_seed=5)
    assert ped.n <= 31
    cols = ped.sequenced_cols()
    V = 200
    lk, fl = synth.synth_likelihoods(ped, V, seed=11, x_fraction=0.3)
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, device=0, cohort_bn=True) as e, \
            fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, device=0) as whole:
        got, ref = e.run(fs.BN, lk, fl), whole.run(fs.BN, lk, fl)
    assert np.array_equal(got.status, ref.status) and np.array_equal(got.gt, ref.gt)
    # atol: where the whole-forest product of every member's factor leaves the double range, fs_create flushes a marginal to
    # zero (or a subnormal) that the family's own product keeps -- the one place the two may differ
    assert np.allclose(got.post, ref.post, rtol=1e-9, atol=1e-300) and np.array_equal(got.single, ref.single)
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=params(5.0), device=0, cohort_bn=True) as e:
        got = e.run(fs.BN, lk, fl)  # -LRC 5: the pedigree always used, so a family alone takes the cohort's gate
    for r in rows:  # the C oracle on each family, the looped one included
        sub = synth._mk([(ped.ids[i], ped.mids[i], ped.fids[i], ped.genders[i]) for i in r])
        gcols = [c for c in range(len(cols)) if cols[c] in set(r.tolist())]
        w = O.run(sub, [list(r).index(cols[c]) for c in gcols], lk[:, gcols], fl, method=O.BN, lc=5.0)
        assert (got.status[w["status"] != 0] == 1).all()
        ok = (w["status"] == 0) & (got.status == 0)
        assert np.allclose(got.post[ok][:, gcols], w["post"][ok], rtol=1e-9, atol=0)
        assert np.array_equal(got.gt[ok][:, gcols], (w["gt"][ok] & 0xff).astype(np.uint8))


def bn_class(p):
    """The launch class (u, independent, group) of the plan host/bn_plan.cpp builds for pedigree p (no tuning knobs set)."""
    n, par = p.n, p.parents()
    kids = [[] for _ in range(n)]
    for i, (m, f) in enumerate(par):
        if m >= 0:
            kids[m].append(i)
            kids[f].append(i)
    order, placed = [], [False] * n
    for leaves_pass in (False, True):  # parents before children; members with children first, childless innermost
        progress = True
        while progress:
            progress = False
            for i in range(n):
                m, f = par[i]
                if placed[i] or (not kids[i]) != leaves_pass or (m >= 0 and not (placed[m] and placed[f])):
                    continue
                placed[i] = progress = True
                order.append(i)
    leaves = sum(1 for k in kids if not k)
    u = n if n < 3 else (5 if n >= 11 and leaves >= 5 else (4 if n >= 9 else 3))
    unrolled = order[n - u:]
    independent = not any(par[i][0] in unrolled[:x] or par[i][1] in unrolled[:x] for x, i in enumerate(unrolled))
    return u, independent, 3 ** min(n - u, 5)


@pytest.mark.parametrize("shuffle", [None, 3])
def test_launch_count_does_not_depend_on_the_number_of_families(shuffle):
    counts = []
    for n in (10, 1000):
        ped, _ = synth.forest([synth.trio()] * n + [synth.cousins_loop(), synth.ped14()], shuffle_seed=shuffle)
        cols = ped.sequenced_cols()
        pl, fl = synth.synth_pl(ped, 64, seed=2, x_fraction=0.2)
        with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, device=0, cohort_bn=True) as e:
            e.run_pl(fs.BN, pl.astype(np.uint16), fl)
            counts.append(e.info()["kernel_launches"])
    # the head, one launch per class present, the finish
    classes = {bn_class(p) for p in (synth.trio(), synth.cousins_loop(), synth.ped14())}
    assert counts == [2 + len(classes)] * 2, (counts, classes)


def test_repeated_device_and_refusals():
    ped, _ = synth.forest([synth.trio()] * 100 + [synth.cousins_loop(), synth.sibship(3)] * 5, shuffle_seed=8)
    cols = ped.sequenced_cols()
    pl, fl = synth.synth_pl(ped, 3000, seed=2, x_fraction=0.2)
    pl = pl.astype(np.uint16)
    args = (ped.ids, ped.mids, ped.fids, ped.genders, cols)
    with fs.Engine(*args, device=[0], cohort_bn=True) as a, fs.Engine(*args, device=[0, 0, 0], cohort_bn=True) as b:
        assert b.info()["n_devices"] == 3
        same(a.run_pl(fs.BN, pl, fl), b.run_pl(fs.BN, pl, fl), "[0] vs [0, 0, 0]")
        for method in (fs.ES, fs.MCMC):
            with pytest.raises(fs.FamSeqError) as x:
                b.run(method, synth.pl_to_likelihood(pl[:4]), fl[:4], burn=10, rep=10)
            assert x.value.code == -1 and "-method 1" in str(x.value) and "fs_create_cohort" in str(x.value)


def cli(tmp_path, ped, pl, fl, extra, tag):
    ped.write(str(tmp_path / f"{tag}.ped"))
    synth.write_vcf(str(tmp_path / f"{tag}.vcf"), ped, pl, fl)
    out = str(tmp_path / f"{tag}_{'_'.join(extra).replace(',', '')}.vcf")
    r = subprocess.run([BIN, "vcf", "-vcfFile", f"{tag}.vcf", "-pedFile", f"{tag}.ped", "-method", "1", "-output", out] + extra,
                       cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return open(out, "rb").read()


def test_cli_family_bn(tmp_path):
    ped, _ = synth.forest([synth.trio()] * 60 + [synth.cousins_loop()], shuffle_seed=6)
    assert 180 < ped.n <= 220
    cols = ped.sequenced_cols()
    pl, fl = synth.synth_pl(ped, 300, seed=8, x_fraction=0.2)
    pl[5::37, 3] = 65535  # rows that decode to zeros: variants written as NA
    outs = [cli(tmp_path, ped, pl, fl, ["-familyBN", "-device", dev], "cohort") for dev in ("0", "0,0,0")]
    assert outs[0] == outs[1]
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, device=0, cohort_bn=True) as e:
        want = e.run_pl_phred(fs.BN, pl.astype(np.uint16), fl, fix_capacity=1 << 16)
    assert want.n_fixes <= 1 << 16
    fixes = {int(i): float(p) for i, p in want.fixes}

    def text(code, index):
        t = phred_text(int(code))
        return t if t is not None else phred_text_exact(fixes[index])
    body = [line.split("\t") for line in outs[0].decode().split("\n") if line and not line.startswith("#")]
    assert len(body) == len(pl) and 0.8 < (want.status == 0).mean() < 1
    S = len(cols)
    for v in range(len(pl)):  # GPP, FPP and FGT of every sample: the engine's codes as text, NA where the variant failed
        for s in range(S):
            at = (v * S + s) * 3
            if want.status[v]:
                calls = ["NA", "NA", "NA"]
            else:
                calls = [",".join(text(want.single[v, s, g], at + g + PHRED_FIX_SINGLE) for g in range(3)),
                         ",".join(text(want.post[v, s, g], at + g) for g in range(3)),
                         {0: "0/0", 1: "0/1"}.get(int(want.gt[v, s]), "1/1")]
            assert body[v][9 + s].split(":")[-3:] == calls, (v, s, body[v][9 + s])
    for shape in (synth.trio, synth.ped14):  # one family: the same bytes as fs_create BN
        p = shape()
        pl1, fl1 = synth.synth_pl(p, 400, seed=3, x_fraction=0.2)
        assert cli(tmp_path, p, pl1, fl1, ["-familyBN"], shape.__name__) == cli(tmp_path, p, pl1, fl1, [], shape.__name__)
