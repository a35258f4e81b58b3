"""Every Gibbs kernel with seeds and site counters past 32 bits.  Philox4x32-10 takes the 64-bit seed as its key (k0, k1)
and the global site as counter words (gv_lo, gv_hi); the command line reads -seed as a 64-bit integer, and a site counter
passes 2^32 in a long run.  Seeds 2^32 + 7 and 0x9E3779B97F4A7C15 (>= 2^63), batches at v_offset 2^32 - V / 2 (one
batch straddles 2^32) and 2^40 + 3:

  * the table-driven kernel against the C oracle's Philox chain, the generated kernels (dense and cached) against it with
    assert_same_chains, and the cohort kernel bit for bit as fs_create's table-driven one, on a trio, ped14 and a cohort
    forest of at most 128 members; the cohort kernel against the oracle on a cohort past 128 members;
  * the high words matter: changing only the seed's high word, or the site by 2^32, changes the chains; two devices
    give the bytes of one on the batch whose second slice starts at site 2^32."""
import numpy as np
import pytest

import famseq_b200 as fs
from famseq_b200 import synth
from oracle import oracle as O
from tests.test_families_gpu import same
from tests.util import REL_TOL, assert_parity, assert_same_chains

pytestmark = pytest.mark.gpu

V = 64
SEEDS = [2**32 + 7, 0x9E3779B97F4A7C15]
OFFSETS = [2**32 - V // 2, 2**40 + 3]
BURN, REP = 10, 60


def oracle_seed(seed):
    """The oracle's seed is an int64: the same 64 bits as two's complement."""
    return seed - 2**64 if seed >= 2**63 else seed


def pedigree(name):
    if name == "forest":  # GW 1 and GW 2 classes, shuffled rows, an unsequenced member
        ped, rows = synth.forest([synth.trio(), synth.ped14(), synth.sibship(5), synth.ped40(), synth.cousins_loop(),
                                  synth._mk([(1, 0, 0, 2)])], shuffle_seed=5)
        ped.names[rows[3][7]] = "NA"
        assert ped.n <= 128
        return ped
    return getattr(synth, name)()


def weak_likelihoods(ped, n, seed):
    """Gene-dropped PLs scaled down eightfold: uncertain genotypes, so the chains move between states and their
    posteriors depend on every random word."""
    pl, fl = synth.synth_pl(ped, n, seed=seed, x_fraction=0.3)
    return synth.pl_to_likelihood(pl // 8), fl


def engine(ped, cols, device=0, **kw):
    return fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, device=device, **kw)


def table_run(ped, cols, lk, fl, monkeypatch, seed, v_offset, device=0):
    monkeypatch.setenv("FAMSEQ_MCMC_JIT", "0")
    with engine(ped, cols, device) as e:
        res = e.run(fs.MCMC, lk, fl, burn=BURN, rep=REP, seed=seed, v_offset=v_offset)
        assert e.info()["jit_launches"] == 0
    monkeypatch.delenv("FAMSEQ_MCMC_JIT")
    return res


@pytest.mark.parametrize("v_offset", OFFSETS)
@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("name", ["trio", "ped14", "forest"])
def test_every_gibbs_kernel_with_64_bit_seed_and_site(name, seed, v_offset, monkeypatch):
    ped = pedigree(name)
    cols = ped.sequenced_cols()
    lk, fl = weak_likelihoods(ped, V, seed=len(cols))
    table = table_run(ped, cols, lk, fl, monkeypatch, seed, v_offset)
    want = O.run(ped, cols, lk, fl, method=O.MCMC, burn=BURN, rep=REP, rng=O.RNG_PHILOX, seed=oracle_seed(seed), v_offset=v_offset)
    assert_parity(table, want, REL_TOL, f"{name} table-driven")
    ok = table.status == 0
    assert ok.mean() > 0.25 and (table.post[ok] != table.single[ok]).any(axis=(1, 2)).mean() > 0.5
    monkeypatch.setenv("FAMSEQ_MCMC_JIT", "1")
    for cached in ("0", "1"):
        monkeypatch.setenv("FAMSEQ_JIT_CACHED", cached)
        with engine(ped, cols) as e:
            got = e.run(fs.MCMC, lk, fl, burn=BURN, rep=REP, seed=seed, v_offset=v_offset)
            info = e.info()
        assert info["jit_launches"] >= 1 and info["gibbs_generator"] == 1 + int(cached)
        assert_same_chains(got, table, f"{name} generated ({cached})")
    monkeypatch.delenv("FAMSEQ_MCMC_JIT")
    monkeypatch.delenv("FAMSEQ_JIT_CACHED")
    with engine(ped, cols, cohort_mcmc=True) as e:
        same(e.run(fs.MCMC, lk, fl, burn=BURN, rep=REP, seed=seed, v_offset=v_offset), table, f"{name} cohort")


@pytest.mark.parametrize("v_offset", OFFSETS)
@pytest.mark.parametrize("seed", SEEDS)
def test_cohort_past_128_members_against_the_oracle(seed, v_offset):
    ped, _ = synth.forest([synth.trio()] * 40 + [synth.ped40(), synth.sibship(5), synth._mk([(1, 0, 0, 1)])], shuffle_seed=3)
    assert ped.n > 128
    cols = ped.sequenced_cols()
    lk, fl = weak_likelihoods(ped, 24, seed=6)
    with engine(ped, cols, cohort_mcmc=True) as e:
        got = e.run(fs.MCMC, lk, fl, burn=BURN, rep=REP, seed=seed, v_offset=v_offset)
    want = O.run(ped, cols, lk, fl, method=O.MCMC, burn=BURN, rep=REP, rng=O.RNG_PHILOX, seed=oracle_seed(seed), v_offset=v_offset)
    assert_parity(got, want, REL_TOL, f"cohort of {ped.n}")
    assert (got.status == 0).mean() > 0.25


def changed(a, b):
    """Share of the variants both runs take whose posteriors differ."""
    ok = (a.status == 0) & (b.status == 0)
    assert ok.mean() > 0.25
    return (a.post[ok] != b.post[ok]).any(axis=(1, 2)).mean()


@pytest.mark.parametrize("cohort", [False, True])
def test_high_words_change_the_chains(cohort, monkeypatch):
    ped = pedigree("forest")
    cols = ped.sequenced_cols()
    lk, fl = weak_likelihoods(ped, V, seed=2)
    monkeypatch.setenv("FAMSEQ_MCMC_JIT", "0")
    with engine(ped, cols, cohort_mcmc=cohort) as e:
        def run(seed, v_offset):
            return e.run(fs.MCMC, lk, fl, burn=BURN, rep=REP, seed=seed, v_offset=v_offset)
        base = run(2**32 + 7, 2**40 + 3)
        assert changed(base, run(7, 2**40 + 3)) > 0.5  # seed's high word 1 -> 0
        assert changed(base, run(2**33 + 7, 2**40 + 3)) > 0.5  # 1 -> 2
        assert changed(base, run(2**32 + 7, 2**40 + 3 + 2**32)) > 0.5  # the site's high word
        assert changed(base, run(2**32 + 7, 2**40 + 3 - 2**32)) > 0.5


@pytest.mark.parametrize("cohort", [False, True])
def test_two_devices_split_at_site_2_32(cohort, monkeypatch):
    """fs_create_multi cuts at multiples of 1 024 variants: of 2 048, device 1 takes sites 2^32 .. 2^32 + 1 023."""
    ped = pedigree("forest")
    cols = ped.sequenced_cols()
    n = 2048
    lk, fl = weak_likelihoods(ped, n, seed=4)
    monkeypatch.setenv("FAMSEQ_MCMC_JIT", "0")
    kw = dict(burn=4, rep=20, seed=0x9E3779B97F4A7C15, v_offset=2**32 - n // 2)
    with engine(ped, cols, cohort_mcmc=cohort) as one, engine(ped, cols, device=[0, 0], cohort_mcmc=cohort) as two:
        assert two.info()["n_devices"] == 2
        a, b = one.run(fs.MCMC, lk, fl, **kw), two.run(fs.MCMC, lk, fl, **kw)
        same(b, a, "[0, 0] vs 0")
        low = one.run(fs.MCMC, lk[:n // 2], fl[:n // 2], **kw)
        high = one.run(fs.MCMC, lk[n // 2:], fl[n // 2:], **dict(kw, v_offset=2**32))
    same(fs.Result(np.concatenate([low.post, high.post]), np.concatenate([low.single, high.single]),
                   np.concatenate([low.gt, high.gt]), np.concatenate([low.status, high.status])), a, "halves")
    assert (a.status == 0).mean() > 0.25
