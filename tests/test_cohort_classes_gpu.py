"""The cohort kernels in every launch class their launchers can pick, with the launches read back from the profiler trace:

  A. mcmc_cohort_kernel<GW> at every (genotype-vector width, block size) pair mcmc_cohort_pick_block gives on this device,
     bit for bit as fs_create's table-driven sampler on the whole file;
  B. all 13 bn_cohort_kernel<U, INDEP, FACTOR> instantiations (FAMSEQ_BN_FACTOR / _GENERIC / _UNROLL), each family bit for
     bit as fs_create BN on that family alone under the same settings, and against the C oracle;
  C. more than 65 535 families in one class: the grid's z slices (BN, MCMC) and es_cohort_kernel's family loop, read
     through the device entry points into outputs pre-filled with NaN and 0xCD, so that a family no block wrote fails."""
import json
import os
import re

import numpy as np
import pytest
import torch

import famseq_b200 as fs
from famseq_b200 import synth
from oracle import oracle as O
from tests.test_cohort_bn_gpu import family_engine
from tests.test_cohort_classes_cpu import CLASS_SIZES, FIVE, FIVE_SEQUENCED, GRID_Y, LONE, regrouped, tiled, tiled_cols
from tests.test_cohort_mcmc_gpu import BURN, REP, SEED, V_OFFSET, inputs, whole_engine
from tests.test_families_gpu import params, same
from tests.test_pedigree_shapes_gpu import case_data
from tests.util import REL_TOL, rel_err

pytestmark = pytest.mark.gpu

KERNEL_NAME = re.compile(r"famseq::(?:\(anonymous namespace\)::)?(\w+_kernel(?:<[^>]*>)?)")


def famseq_launches(fn, tmp_path):
    """Runs fn() under torch.profiler (CUDA activity); returns (fn's result, [(kernel, grid, block)]) of the famseq kernels
    it launched, in launch order, the kernel as e.g. "bn_cohort_kernel<3, false, false>", grid and block as 3-tuples."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    path = str(tmp_path / "famseq_launches.json")
    prof.export_chrome_trace(path)
    with open(path) as fh:
        events = json.load(fh)["traceEvents"]
    os.remove(path)
    launches = []
    for ev in sorted((ev for ev in events if ev.get("cat") == "kernel"), key=lambda ev: float(ev["ts"])):
        m = KERNEL_NAME.search(ev["name"])
        if m:
            launches.append((m.group(1), tuple(ev["args"]["grid"]), tuple(ev["args"]["block"])))
    return out, launches


def device_props():
    p = torch.cuda.get_device_properties(0)
    return p.shared_memory_per_block_optin, p.shared_memory_per_multiprocessor


# ------------------------------------------------------------------------------------------------------
# A. mcmc_cohort_kernel: every (GW, TB) pair
# ------------------------------------------------------------------------------------------------------
MCMC_PLAN_BYTES = 1288  # sizeof(McmcPlan): n, n_links, member[128], link[256], col[128]


def mcmc_cohort_width(n):
    return 1 if n <= 32 else 2 if n <= 64 else 4


def mcmc_cohort_pick_block(n, smem_block, smem_sm):
    """mcmc_cohort_kernel.cu's pick: the block size (256 down to 32) that keeps the most chains resident on an SM, the
    larger one on a tie."""
    best, best_threads = 0, 0
    for tb in range(256, 31, -32):
        need = (108 * 16 + 2 * n * 3 * tb) * 8 + MCMC_PLAN_BYTES + 2 * 128 * 4 + 1024
        if need > smem_block + 1024:
            continue
        threads = min(2048, min(32, smem_sm // need) * tb)
        if threads > best_threads:
            best, best_threads = tb, threads
    return best


# (GW, TB) of a launch class by the member count of its largest family on a B200 (227 KB of shared memory per block,
# 228 KB per SM)
GIBBS_PAIRS = {(1, 256): [1, 3, 4, 7, 8, 14, 15, 16, 17], (1, 224): [2, 5, 9, 18, 19, 20], (1, 192): [6, 10, 21, 22, 23],
               (1, 160): [11, 12, 24, 25, 26, 27, 28], (1, 128): [29, 30, 31, 32], (1, 96): [13], (2, 128): [33, 34, 35],
               (2, 96): list(range(36, 47)), (2, 64): list(range(47, 65)), (4, 64): list(range(65, 71)),
               (4, 32): list(range(71, 129))}
GIBBS_PAIR = {n: pair for pair, ns in GIBBS_PAIRS.items() for n in ns}


def rp(seed, n):
    """A random pedigree of n members that is one family (seeds picked so), looped unless the seed gives a loop-free one."""
    p = synth.random_pedigree(seed, n, loops=True)
    assert p.n == n
    return p


def gibbs_forests():
    """Forests of at most 128 members whose launch classes' largest families reach all 11 pairs, the boundary sizes
    32 / 33, 64 / 65, 70 / 71 and 128 among them.  name: (families, shuffle seed)."""
    lone_m, lone_f = synth._mk([(1, 0, 0, 1)]), synth._mk([(1, 0, 0, 2)])
    return {"65_33_14": ([rp(5, 65), rp(4, 33), synth.ped14(), synth.trio(), lone_f], 11),
            "71_40_5": ([rp(10, 71), synth.ped40(), synth.sibship(3), synth.trio(), lone_m], None),
            "64_32": ([rp(5, 64), rp(4, 32), synth.trio(), synth.trio(), lone_m], 12),
            "70_13": ([rp(6, 70), synth.sibship(11), synth.sibship(8), synth.trio(), lone_f], None),
            "128": ([rp(10, 128)], 13),
            "50_12": ([rp(9, 50), synth.sibship(10), synth.three_generations(2), synth.half_sibs(), synth.trio(), lone_m], None),
            "40_22": ([synth.ped40(), rp(2, 22), synth.cousins_loop(), synth.sibship(2), lone_f], 14)}


def expected_gibbs_pairs(fams):
    largest = {}
    for p in fams:
        gw = mcmc_cohort_width(p.n)
        largest[gw] = max(largest.get(gw, 0), p.n)
    return {GIBBS_PAIR[n] for n in largest.values()}


def test_gibbs_block_table_is_the_devices():
    smem_block, smem_sm = device_props()
    got = {n: (mcmc_cohort_width(n), mcmc_cohort_pick_block(n, smem_block, smem_sm)) for n in range(1, 129)}
    assert got == GIBBS_PAIR, {n: (got[n], GIBBS_PAIR[n]) for n in got if got[n] != GIBBS_PAIR[n]}


def test_gibbs_forests_reach_every_pair():
    pairs = set()
    for fams, _ in gibbs_forests().values():
        assert sum(p.n for p in fams) <= 128
        pairs |= expected_gibbs_pairs(fams)
    assert pairs == set(GIBBS_PAIRS)
    assert {32, 33, 64, 65, 70, 71, 128} <= {p.n for fams, _ in gibbs_forests().values() for p in fams}


@pytest.mark.parametrize("lrc", [1.0, 5.0])
@pytest.mark.parametrize("name", list(gibbs_forests()))
def test_gibbs_class_bit_for_bit_fs_create(name, lrc, monkeypatch, tmp_path):
    fams, shuffle = gibbs_forests()[name]
    ped, rows = synth.forest(fams, shuffle_seed=shuffle)
    for i in range(2, ped.n, 9):  # unsequenced members
        ped.names[i] = "NA"
    cols = [int(c) for c in np.random.default_rng(ped.n).permutation(ped.sequenced_cols())]
    V = 301
    lk, pl, fl = inputs(ped, cols, V, seed=ped.n)
    prm = params(lrc)
    kw = dict(burn=BURN, rep=REP, seed=SEED, v_offset=V_OFFSET)
    cases = [(x, ws) for x in ("run", "run_pl") for ws in (True, False)]
    with whole_engine(ped, cols, prm, monkeypatch) as w, \
            fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=prm, device=0, cohort_mcmc=True) as e:
        fam, _ = e.families()
        sizes = np.bincount(fam)
        for r, p in zip(rows, fams):
            assert (fam[r] == fam[r[0]]).all() and sizes[fam[r[0]]] == p.n, (name, p.n)
        assert len(sizes) == len(fams)

        def cohort():
            return [getattr(e, x)(fs.MCMC, lk if x == "run" else pl, fl, want_single=ws, **kw) for x, ws in cases]
        got, launches = famseq_launches(cohort, tmp_path)
        want = [getattr(w, x)(fs.MCMC, lk if x == "run" else pl, fl, want_single=ws, **kw) for x, ws in cases]
    for g, r, (x, ws) in zip(got, want, cases):
        same(g, r, f"{name} {x} single={ws}")
    pairs = {(int(re.fullmatch(r"mcmc_cohort_kernel<(\d)>", k).group(1)), block[0]) for k, _, block in launches
             if k.startswith("mcmc_cohort_kernel")}
    assert pairs == expected_gibbs_pairs(fams), (name, pairs)
    assert sum(1 for k, _, _ in launches if k.startswith("mcmc_cohort_kernel")) == len(pairs) * len(cases)
    res = got[0]
    ok = res.status == 0
    chains = (res.post != res.single).any(axis=(1, 2)) & ok  # variants whose posteriors come from the chains
    assert 0 < (~ok).sum() and chains.sum() >= V // 4, (name, chains.sum())
    assert lrc != 5.0 or chains.sum() == ok.sum()


# ------------------------------------------------------------------------------------------------------
# B. bn_cohort_kernel: all 13 instantiations
# ------------------------------------------------------------------------------------------------------
BN_SETTINGS = {"default": {}, "factor": {"FAMSEQ_BN_FACTOR": "1"}, "generic": {"FAMSEQ_BN_GENERIC": "1"},
               "unroll2": {"FAMSEQ_BN_UNROLL": "2"}, "unroll2_factor": {"FAMSEQ_BN_UNROLL": "2", "FAMSEQ_BN_FACTOR": "1"}}
BN_INSTANTIATIONS = {"bn_cohort_kernel<1, false, false>"} | {
    f"bn_cohort_kernel<{u}, {indep}, {factor}>" for u in (2, 3, 4, 5)
    for indep, factor in (("false", "false"), ("true", "false"), ("true", "true"))}


def test_bn_cohort_every_instantiation(monkeypatch, tmp_path):
    # groups 1, 3, 9, 27, 81 and 243 (sibships of 2..5, ped14); U 1, 3, 4, 5 by default; U 2 under FAMSEQ_BN_UNROLL=2
    fams = [synth._mk([(1, 0, 0, 2)]), synth.trio(), synth.sibship(2), synth.sibship(3), synth.sibship(4), synth.sibship(5),
            synth.sibship(8), synth.three_generations(2), synth.cousins_loop(), synth.ped14()]
    ped, rows = synth.forest(fams, shuffle_seed=23)
    ped.names[rows[1][0]] = ped.names[rows[8][2]] = ped.names[rows[9][5]] = ped.names[rows[6][4]] = "NA"
    cols = [int(c) for c in np.random.default_rng(3).permutation(ped.sequenced_cols())]
    V, n_wide, n_oracle = 301, 60, 40
    lk, fl = case_data(ped, cols, V, seed=90, n_wide=n_wide)
    prm = params(5.0)
    oracle = {}
    for f, r in enumerate(rows):  # the C oracle's BN on each family, on gene-dropped rows
        sub = synth._mk([(ped.ids[i], ped.mids[i], ped.fids[i], ped.genders[i]) for i in r])
        gcols = [c for c in range(len(cols)) if cols[c] in set(r.tolist())]
        oracle[f] = O.run(sub, [list(r).index(cols[c]) for c in gcols], lk[:n_oracle, gcols], fl[:n_oracle], method=O.BN, lc=5.0)
    seen = set()
    for setting, env in BN_SETTINGS.items():
        for k in ("FAMSEQ_BN_FACTOR", "FAMSEQ_BN_GENERIC", "FAMSEQ_BN_UNROLL"):
            monkeypatch.delenv(k, raising=False)
        for k, x in env.items():
            monkeypatch.setenv(k, x)
        with fs.Engine(ped.ids, ped.mids, ped.fids, ped.genders, cols, params=prm, device=0, cohort_bn=True) as e:
            got, launches = famseq_launches(lambda: e.run(fs.BN, lk, fl), tmp_path)
        names = {k for k, _, _ in launches if k.startswith("bn_cohort_kernel")}
        seen |= names
        status = np.zeros(V, np.uint8)
        for f, r in enumerate(rows):
            fe, gcols = family_engine(ped, r, cols, prm)
            with fe:
                want = fe.run(fs.BN, lk[:, gcols], fl)
            status |= want.status
            ok = got.status == 0
            for k in ("post", "single", "gt"):
                assert np.array_equal(getattr(got, k)[ok][:, gcols], getattr(want, k)[ok]), (setting, f, k)
            w = oracle[f]
            assert (got.status[:n_oracle][w["status"] != 0] == 1).all(), (setting, f)
            ok = (w["status"] == 0) & (got.status[:n_oracle] == 0)
            assert rel_err(got.post[:n_oracle][ok][:, gcols], w["post"][ok]) <= REL_TOL, (setting, f)
            assert np.array_equal(got.gt[:n_oracle][ok][:, gcols], (w["gt"][ok] & 0xff).astype(np.uint8)), (setting, f)
        assert np.array_equal(got.status, status), setting
        assert 0 < got.status.sum() < V // 2 and (got.status[:n_oracle] == 0).sum() > n_oracle // 2, setting
    assert seen == BN_INSTANTIATIONS, sorted(BN_INSTANTIATIONS - seen)


# ------------------------------------------------------------------------------------------------------
# C. more than 65 535 families in one class
# ------------------------------------------------------------------------------------------------------
V_BIG = 8


def run_device_prefilled(e, method, lk, fl, **kw):
    """run_device into outputs pre-filled with NaN (post, single) and 0xCD (gt, status)."""
    V, S = lk.shape[:2]
    x, flags = torch.from_numpy(np.ascontiguousarray(lk)).cuda(), torch.from_numpy(fl).cuda()
    post = torch.full((V, S, 3), float("nan"), dtype=torch.float64, device="cuda")
    single = torch.full_like(post, float("nan"))
    gt = torch.full((V, S), 0xCD, dtype=torch.uint8, device="cuda")
    status = torch.full((V,), 0xCD, dtype=torch.uint8, device="cuda")
    e.run_device(method, V, x.data_ptr(), flags.data_ptr(), post.data_ptr(), single.data_ptr(), gt.data_ptr(), status.data_ptr(),
                 stream=torch.cuda.current_stream().cuda_stream, **kw)
    torch.cuda.synchronize()
    return fs.Result(post.cpu().numpy(), single.cpu().numpy(), gt.cpu().numpy(), status.cpu().numpy())


def stacked_data(fam, sequenced, F, seed):
    """Gene-dropped likelihoods of F copies of `fam` at V_BIG variants: row f * V_BIG + v of the stack is copy f at
    variant v.  Returns (stack [V_BIG F][k][3], cohort [V_BIG][F k][3], cohort flags [V_BIG]): chrX and Known mixed in."""
    p = synth._mk(list(zip(fam.ids, fam.mids, fam.fids, fam.genders)))
    p.names = ["NA" if i not in sequenced else f"s{i}" for i in range(p.n)]
    stack, _ = synth.synth_likelihoods(p, V_BIG * F, seed=seed)
    fl = (np.arange(V_BIG) % 4).astype(np.uint8)  # plain, Known, chrX, both
    return stack, fl


def to_cohort(stack, F):
    """[V_BIG F][k][...] stack rows -> [V_BIG][F k][...] cohort columns (copy f's members at columns f k .. f k + k - 1)."""
    k = stack.shape[1]
    return np.ascontiguousarray(stack.reshape((F, V_BIG, k) + stack.shape[2:]).swapaxes(0, 1).reshape((V_BIG, F * k) + stack.shape[2:]))


def expected_from_stack(ref, F):
    """The cohort's outputs from the stacked run: copy f's columns are its rows; a variant fails in every column when
    any copy fails it (the whole-row rule)."""
    failed = ref.status.reshape(F, V_BIG).any(axis=0)
    post, single, gt = to_cohort(ref.post, F), to_cohort(ref.single, F), to_cohort(ref.gt, F)
    post[failed], single[failed], gt[failed] = 0.0, 0.0, 255
    return fs.Result(post, single, gt, failed.astype(np.uint8))


def z_slices(F):
    return (F + GRID_Y - 1) // GRID_Y


@pytest.mark.parametrize("F", CLASS_SIZES)
@pytest.mark.parametrize("path", ["es", "bn_trio", "bn_lone"])
def test_past_65535_families_against_one_family_with_stacked_rows(path, F, tmp_path):
    fam, seq, kw, method = {"es": (FIVE, FIVE_SEQUENCED, dict(cohort=True), fs.ES),
                            "bn_trio": (synth.trio(), [0, 1, 2], dict(cohort_bn=True), fs.BN),
                            "bn_lone": (LONE, [0], dict(cohort_bn=True), fs.BN)}[path]
    stack, fl = stacked_data(fam, seq, F, seed=F % 1000)
    far = V_BIG // 2 + 1
    if path != "bn_lone":  # one variant fails only through the last family, in the far slice when F > 65 535
        stack[(F - 1) * V_BIG + far] = 1e-300
    lk = to_cohort(stack, F)
    prm = params(5.0)
    one = synth._mk(list(zip(fam.ids, fam.mids, fam.fids, fam.genders)))
    with fs.Engine(one.ids, one.mids, one.fids, one.genders, seq, params=prm, device=0) as w:
        ref = w.run(method, stack, np.tile(fl, F))
    want = expected_from_stack(ref, F)
    with fs.Engine(*tiled(fam, F), tiled_cols(fam.n, seq, F), params=prm, device=0, **kw) as e:
        got, launches = famseq_launches(lambda: run_device_prefilled(e, method, lk, fl), tmp_path)
    same(got, want, f"{path} F={F}")
    if path == "bn_lone":
        assert (got.status == 0).all()
    else:
        assert ref.status[(F - 1) * V_BIG + far] == 1 and ref.status.reshape(F, V_BIG)[:-1, far].sum() == 0
        assert got.status[far] == 1 and (got.post[far] == 0).all() and (got.single[far] == 0).all() and (got.gt[far] == 255).all()
        assert got.status.sum() == 1
    kernel = {"es": "es_cohort_kernel", "bn_trio": "bn_cohort_kernel<3, false, false>", "bn_lone": "bn_cohort_kernel<1, false, false>"}[path]
    mine = [(grid, block) for k, grid, block in launches if k == kernel or (path == "es" and k.startswith(kernel + "<"))]
    assert len(mine) == 1, launches
    grid = mine[0][0]
    assert grid[1] == GRID_Y and grid[2] == (1 if path == "es" else z_slices(F)), (path, F, grid)


@pytest.mark.parametrize("F", CLASS_SIZES)
def test_past_65535_families_gibbs_against_a_regrouped_file(F, tmp_path):
    """The trailing trios of a file of F trios (class GW 1; past device index 65 535 when F > 65 535) against the same
    trios in a file whose leading trios are regrouped into 45-member pedigrees (class GW 2), so that all the trailing ones
    sit in the first z slice: the same ped rows and columns, so the same chains and bytes."""
    trio = synth.trio()
    stack, fl = stacked_data(trio, [0, 1, 2], F, seed=7 + F % 1000)
    # autosomal sites only: the rows are gene-dropped as autosomes, and on chrX the sampler (as the C oracle) fails a
    # variant wherever a male's row calls a heterozygote -- about a third of the trios here, so every chrX variant
    fl &= 1
    lk = to_cohort(stack, F)
    prm = params(5.0)
    kw = dict(burn=4, rep=12, seed=SEED, v_offset=V_OFFSET)
    cols = np.arange(3 * F, dtype=np.int32)
    with fs.Engine(*tiled(trio, F), cols, params=prm, device=0, cohort_mcmc=True) as e:
        got, launches = famseq_launches(lambda: run_device_prefilled(e, fs.MCMC, lk, fl, **kw), tmp_path)
    ped2, R = regrouped(F)
    with fs.Engine(*ped2, cols, params=prm, device=0, cohort_mcmc=True) as e:
        ref, launches2 = famseq_launches(lambda: run_device_prefilled(e, fs.MCMC, lk, fl, **kw), tmp_path)
    assert (got.status == 0).all() and (ref.status == 0).all()
    assert not np.isnan(got.post).any() and not np.isnan(got.single).any() and not (got.gt == 0xCD).any()
    tail = slice(3 * R, 3 * F)
    same(fs.Result(got.post[:, tail], got.single[:, tail], got.gt[:, tail], got.status),
         fs.Result(ref.post[:, tail], ref.single[:, tail], ref.gt[:, tail], ref.status), f"trailing trios F={F}")
    chains = (got.post != got.single).any(axis=2)
    assert chains[:, tail].mean() > 0.5
    mine = [grid for k, grid, _ in launches if k.startswith("mcmc_cohort_kernel")]
    assert [k for k, _, _ in launches if k.startswith("mcmc_cohort_kernel")] == ["mcmc_cohort_kernel<1>"]
    assert mine[0][1] == GRID_Y and mine[0][2] == z_slices(F), (F, mine)
    classes = {k: grid for k, grid, _ in launches2 if k.startswith("mcmc_cohort_kernel")}
    assert set(classes) == {"mcmc_cohort_kernel<1>", "mcmc_cohort_kernel<2>"}
    assert classes["mcmc_cohort_kernel<1>"][1:] == (F - R, 1) and classes["mcmc_cohort_kernel<2>"][1:] == (R // 15, 1)
