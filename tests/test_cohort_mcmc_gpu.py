"""The Gibbs sampler for cohort ped files (fs_create_cohort_mcmc: es_cohort_head_kernel, mcmc_cohort_kernel once per launch
class, es_cohort_finish_kernel) on the GPU:

  * bit for bit fs_create's table-driven sampler on forests of at most 128 members, looped families included, in file
    order and with shuffled rows, permuted columns, unsequenced members and a family with none sequenced, through every
    batch entry point, with and without single;
  * the C oracle's whole-file Philox chain past 128 members;
  * the whole-row rules, batch splits and repeated devices, the launch count, the ES / BN refusal, and the command line."""
import os
import subprocess

import numpy as np
import pytest
import torch

import famseq_b200 as fs
from famseq_b200 import synth
from oracle import oracle as O
from tests.test_families_gpu import params, same
from tests.test_pedigree_shapes_gpu import case_data
from tests.util import REL_TOL, assert_parity

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "famseq_b200", "bin", "FamSeq")
BURN, REP, SEED, V_OFFSET = 10, 60, 7, 1_000_003


def small_forest(shuffle_seed=None):
    """At most 128 members: every shape fs_create's sampler takes next to each other; family 9 has no sequenced member and
    a member of families 0, 6 and 7 is unsequenced."""
    fams = [synth.trio(), synth.sibship(5), synth.sibship(8), synth.half_sibs(), synth.three_wives(), synth.three_generations(2),
            synth.cousins_loop(), synth.ped14(), synth._mk([(1, 0, 0, 1)]), synth.trio(), synth._mk([(1, 0, 0, 2)]), synth.trio()]
    ped, rows = synth.forest(fams, shuffle_seed=shuffle_seed)
    assert ped.n <= 128
    for i in rows[9]:
        ped.names[i] = "NA"
    ped.names[rows[0][0]] = ped.names[rows[6][3]] = ped.names[rows[7][5]] = "NA"
    return ped, rows


def whole_engine(ped, cols, prm, monkeypatch):
    """fs_create on the whole file, with its table-driven sampler."""
    monkeypatch.setenv("FAMSEQ_MCMC_JIT", "0")
    e = fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=prm, device=0)
    monkeypatch.delenv("FAMSEQ_MCMC_JIT")
    return e


def run_device(e, x, fl, compact, want_single, v_offset=V_OFFSET):
    xd = torch.from_numpy(np.ascontiguousarray(x.astype(np.int16) if compact else x)).cuda()
    V, S = x.shape[:2]
    flags = torch.from_numpy(fl).cuda()
    post = torch.empty((V, S, 3), dtype=torch.float64, device="cuda")
    single = torch.empty_like(post) if want_single else None
    gt = torch.empty((V, S), dtype=torch.uint8, device="cuda")
    status = torch.empty(V, dtype=torch.uint8, device="cuda")
    f = e.run_pl_device if compact else e.run_device
    f(fs.MCMC, V, xd.data_ptr(), flags.data_ptr(), post.data_ptr(), single.data_ptr() if want_single else None, gt.data_ptr(),
      status.data_ptr(), burn=BURN, rep=REP, seed=SEED, v_offset=v_offset, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return fs.Result(post.cpu().numpy(), single.cpu().numpy() if want_single else None, gt.cpu().numpy(), status.cpu().numpy())


def inputs(ped, cols, V, seed):
    """FP64 rows from case_data (wide exponent range, all-zero rows, chrX and Known flags) and PL rows with a few that
    decode to zeros."""
    lk, fl = case_data(ped, cols, V, seed=seed, n_wide=V // 5)
    pl, _ = synth.synth_pl(synth._mk(list(zip(ped.ids, ped.mids, ped.fids, ped.genders))), V, seed=seed + 1, x_fraction=0.3)
    pl = pl[:, cols].astype(np.uint16)
    pl[5::37, len(cols) // 3] = 65535
    return lk, pl, fl


@pytest.mark.parametrize("lrc", [1.0, 5.0, 0.5])
@pytest.mark.parametrize("order", ["file", "shuffled"])
def test_bit_for_bit_fs_create_through_every_entry_point(order, lrc, monkeypatch):
    ped, _ = small_forest(None if order == "file" else 13)
    cols = [int(c) for c in np.random.default_rng(5).permutation(ped.sequenced_cols())]
    lk, pl, fl = inputs(ped, cols, 301, seed=40)
    prm = params(lrc)
    kw = dict(burn=BURN, rep=REP, seed=SEED, v_offset=V_OFFSET)
    with whole_engine(ped, cols, prm, monkeypatch) as w, \
            fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=prm, device=0, cohort_mcmc=True) as e:
        for want_single in (True, False):
            ref = w.run(fs.MCMC, lk, fl, want_single=want_single, **kw)
            same(e.run(fs.MCMC, lk, fl, want_single=want_single, **kw), ref, f"run {want_single}")
            same(run_device(e, lk, fl, False, want_single), ref, f"run_device {want_single}")
            ref = w.run_pl(fs.MCMC, pl, fl, want_single=want_single, **kw)
            same(e.run_pl(fs.MCMC, pl, fl, want_single=want_single, **kw), ref, f"run_pl {want_single}")
            same(run_device(e, pl, fl, True, want_single), ref, f"run_pl_device {want_single}")
        a, b = e.run_pl_phred(fs.MCMC, pl, fl, **kw), w.run_pl_phred(fs.MCMC, pl, fl, **kw)
        assert all(np.array_equal(getattr(a, k), getattr(b, k)) for k in ("post", "single", "gt", "status", "fixes"))
        assert e.info()["gibbs_generator"] == 0 and w.info()["gibbs_generator"] == 0
        res = e.run(fs.MCMC, lk, fl, **kw)
    ok = res.status == 0
    assert 0 < (~ok).sum() < len(ok) // 2
    chains = (res.post != res.single).any(axis=(1, 2)) & ok  # variants whose posteriors come from the chains
    assert lrc == 0.5 or chains.any()
    assert lrc != 5.0 or chains.sum() == ok.sum()


def test_unsequenced_prior_failure(monkeypatch):
    ped, _ = small_forest(3)
    cols = ped.sequenced_cols()
    lk, _, fl = inputs(ped, cols, 101, seed=8)
    fl[::2] |= 1  # Known
    prm = params(1.0)
    prm.geno_prob_k[0] = prm.geno_prob_k[1] = prm.geno_prob_k[2] = 0.0  # every Known variant fails on the unsequenced members
    kw = dict(burn=BURN, rep=REP, seed=SEED, v_offset=5)
    with whole_engine(ped, cols, prm, monkeypatch) as w, \
            fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=prm, device=0, cohort_mcmc=True) as e:
        got, ref = e.run(fs.MCMC, lk, fl, **kw), w.run(fs.MCMC, lk, fl, **kw)
    same(got, ref, "known prior")
    assert (got.status[(fl & 1) == 1] == 1).all() and (got.status[(fl & 1) == 0] == 0).any()


@pytest.mark.parametrize("size", ["300", "1000"])
def test_past_128_members_against_the_oracle(size):
    if size == "300":
        fams = [synth.trio()] * 70 + [synth.ped40(), synth.cousins_loop(), synth.sibship(5), synth._mk([(1, 0, 0, 2)])]
        V = 64
    else:
        fams = [synth.trio()] * 320 + [synth.ped40(), synth.sibship(8)] * 2
        V = 24
    ped, _ = synth.forest(fams, shuffle_seed=21)
    assert ped.n >= (250 if size == "300" else 1000)
    cols = ped.sequenced_cols()
    lk, fl = synth.synth_likelihoods(ped, V, seed=3, x_fraction=0.3)
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, device=0, cohort_mcmc=True) as e:
        got = e.run(fs.MCMC, lk, fl, burn=10, rep=80, seed=7, v_offset=11)
    want = O.run(ped, cols, lk, fl, method=O.MCMC, burn=10, rep=80, rng=O.RNG_PHILOX, seed=7, v_offset=11)
    assert_parity(got, want, REL_TOL, f"cohort of {ped.n}")
    assert (got.status == 0).sum() >= V // 4


def test_zero_row_in_one_family_fails_the_whole_variant():
    ped, rows = synth.forest([synth.trio()] * 50 + [synth.ped40()], shuffle_seed=2)
    cols = ped.sequenced_cols()
    lk, fl = synth.synth_likelihoods(ped, 40, seed=5, x_fraction=0.3)
    col40 = cols.index(int(rows[50][7]))
    lk[3, col40] = 0.0
    with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, device=0, cohort_mcmc=True) as e:
        got = e.run(fs.MCMC, lk, fl, burn=5, rep=20, seed=1)
    assert got.status[3] == 1 and (got.post[3] == 0).all() and (got.single[3] == 0).all() and (got.gt[3] == 255).all()


def test_split_batches_and_repeated_devices_give_the_same_bytes():
    ped, _ = synth.forest([synth.trio()] * 60 + [synth.ped40(), synth.cousins_loop()] * 2, shuffle_seed=8)
    cols = ped.sequenced_cols()
    pl, fl = synth.synth_pl(ped, 700, seed=2, x_fraction=0.2)
    pl = pl.astype(np.uint16)
    kw = dict(burn=8, rep=40, seed=3)
    args = (ped.ids, ped.mids, ped.fids, ped.genders, cols)
    with fs.Engine(*args, device=0, cohort_mcmc=True) as a, fs.Engine(*args, device=[0, 0, 0], cohort_mcmc=True) as b:
        one = a.run_pl(fs.MCMC, pl, fl, v_offset=100, **kw)
        h = 333
        x, y = a.run_pl(fs.MCMC, pl[:h], fl[:h], v_offset=100, **kw), a.run_pl(fs.MCMC, pl[h:], fl[h:], v_offset=100 + h, **kw)
        two = fs.Result(np.concatenate([x.post, y.post]), np.concatenate([x.single, y.single]), np.concatenate([x.gt, y.gt]),
                        np.concatenate([x.status, y.status]))
        same(two, one, "two halves")
        assert b.info()["n_devices"] == 3
        same(b.run_pl(fs.MCMC, pl, fl, v_offset=100, **kw), one, "[0] vs [0, 0, 0]")
        for method in (fs.ES, fs.BN):
            with pytest.raises(fs.FamSeqError) as err:
                b.run(method, synth.pl_to_likelihood(pl[:4]), fl[:4])
            msg = str(err.value)
            assert err.value.code == -1 and "-method 3" in msg and "fs_create_cohort" in msg and "fs_create_cohort_bn" in msg, msg


@pytest.mark.parametrize("shuffle", [None, 3])
def test_launch_count_does_not_depend_on_the_number_of_families(shuffle):
    counts = []
    for n in (10, 600):
        ped, _ = synth.forest([synth.trio()] * n + [synth.cousins_loop(), synth.ped40(), synth.ped100()], shuffle_seed=shuffle)
        pl, fl = synth.synth_pl(ped, 64, seed=2, x_fraction=0.2)
        with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, ped.sequenced_cols(), device=0, cohort_mcmc=True) as e:
            e.run_pl(fs.MCMC, pl.astype(np.uint16), fl, burn=2, rep=4)
            counts.append(e.info()["kernel_launches"])
    assert counts == [2 + 3] * 2, counts  # the head, the <= 32 / <= 64 / <= 128 member classes, the finish


def cli(tmp_path, ped, pl, fl, extra, tag):
    ped.write(str(tmp_path / f"{tag}.ped"))
    synth.write_vcf(str(tmp_path / f"{tag}.vcf"), ped, pl, fl)
    out = str(tmp_path / f"{tag}_{'_'.join(extra).replace(',', '')}.vcf")
    env = dict(os.environ, FAMSEQ_MCMC_JIT="0")
    r = subprocess.run([BIN, "vcf", "-vcfFile", f"{tag}.vcf", "-pedFile", f"{tag}.ped", "-method", "3", "-numBurnIn", "20",
                        "-numRep", "200", "-seed", "7", "-output", out] + extra, cwd=tmp_path, capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    return [line.split("\t") for line in open(out).read().split("\n") if line and not line.startswith("#")]


def test_cli_cohort_mcmc(tmp_path):
    fams = [synth.ped40()] + [synth.trio()] * 12 + [synth.cousins_loop()] + [synth.sibship(3)] * 2
    f_ped, _ = synth.forest(fams)
    assert f_ped.n <= 128 and f_ped.n + 60 > 128
    big, _ = synth.forest(fams + [synth._mk([(1, 0, 0, 1 + k % 2)]) for k in range(60)])  # 60 lone individuals appended
    assert list(big.ids[:f_ped.n]) == list(f_ped.ids) and big.n == f_ped.n + 60
    V = 120
    pl, fl = synth.synth_pl(big, V, seed=8, x_fraction=0.2)
    S = len(f_ped.sequenced_cols())
    alone = cli(tmp_path, f_ped, pl[:, :S], fl, [], "forest")
    outs = [cli(tmp_path, big, pl, fl, ["-device", dev], "cohort") for dev in ("0", "0,0,0")]
    assert outs[0] == outs[1]
    assert len(alone) == len(outs[0]) == V
    for a, b in zip(alone, outs[0]):  # the forest's columns: the same chains, so the same bytes
        assert a[:9 + S] == b[:9 + S]
    assert sum(1 for row in alone if not row[9].endswith(":NA")) > V // 2
