"""Cohort ped files of more than 65 535 families in one launch class, built in linear time, on host-only engines: the family
split, each family's size and the build time.  tests/test_cohort_classes_gpu.py runs the same files on the GPU, where one
class spans one, two and three grid z slices (BN, MCMC) or passes of the program loop (ES)."""
import time

import numpy as np
import pytest

import famseq_b200 as fs
from famseq_b200 import synth

GRID_Y = 65535  # the launchers' cap on gridDim.y: families of one class past it go to blockIdx.z (or the next loop pass)
CLASS_SIZES = [GRID_Y, GRID_Y + 1, 2 * GRID_Y + 1]  # one, two and three slices

LONE = synth._mk([(1, 0, 0, 2)])
# three generations, five members: two founders, their son, his wife and a grandchild; the founder father and the
# grandchild are sequenced, so every copy runs as an ES program family
FIVE = synth._mk([(1, 0, 0, 1), (2, 0, 0, 2), (3, 2, 1, 1), (4, 0, 0, 2), (5, 4, 3, 2)])
FIVE_SEQUENCED = [0, 4]


# seeds for which synth.random_pedigree(seed, 45, loops=True) is one family (a member who marries a fresh founder and has
# no children with them leaves that founder on its own)
CONNECTED_45 = [2, 6, 12, 19, 20, 29, 30, 32]


def tiled(fam, F):
    """F copies of `fam` in one ped file, copy f on rows [f n, (f + 1) n) with its ids offset by f * max id, as int32
    arrays (ids, mother ids, father ids, genders).  Linear in the number of rows: synth.forest is quadratic in F."""
    off = (np.arange(F, dtype=np.int64) * max(fam.ids))[:, None]
    ids = np.asarray(fam.ids, np.int64)[None] + off
    par = [np.where(np.asarray(p)[None] == 0, 0, np.asarray(p, np.int64)[None] + off) for p in (fam.mids, fam.fids)]
    return tuple(a.ravel().astype(np.int32) for a in (ids, par[0], par[1])) + (np.tile(np.asarray(fam.genders, np.int32), F),)


def stacked(parts):
    """Several ped files one after the other, the ids of each offset past those of the ones before."""
    out, base = [[], [], [], []], 0
    for ids, mids, fids, genders in parts:
        out[0].append(ids + base)
        out[1].append(np.where(mids == 0, 0, mids + base))
        out[2].append(np.where(fids == 0, 0, fids + base))
        out[3].append(genders)
        base += int(ids.max())
    return tuple(np.concatenate(a).astype(np.int32) for a in out)


def tiled_cols(fam_n, sequenced, F):
    """The input columns of `tiled`: the sequenced members of each copy, copy by copy."""
    return (np.arange(F, dtype=np.int64)[:, None] * fam_n + np.asarray(sequenced)[None]).ravel().astype(np.int32)


def regrouped(F):
    """F trios in file order, except that the leading R trios are replaced by R / 15 random pedigrees of 45 members on the
    same rows and ids; the trailing F - R trios keep their rows, ids and columns.  R is the least multiple of 15 that
    leaves fewer than 65 536 trailing trios, so that they fit the first grid z slice.  Returns (ped arrays, R)."""
    R = 15 * max(1, -(-(F - GRID_Y) // 15))
    shapes = [synth.random_pedigree(s, 45, loops=True) for s in CONNECTED_45]
    assert all(p.n == 45 and p.ids == list(range(1, 46)) for p in shapes)
    lead = [tuple(np.asarray(getattr(shapes[k % len(shapes)], a), np.int32) for a in ("ids", "mids", "fids", "genders"))
            for k in range(R // 15)]
    return stacked(lead + [tiled(synth.trio(), F - R)]), R


def family_sizes(e):
    fam, kids = e.families()
    return np.bincount(fam, minlength=len(kids)), kids


@pytest.mark.parametrize("F", CLASS_SIZES)
def test_tiled_cohorts_split_into_their_copies(F):
    for fam, kw, seq in ((FIVE, dict(cohort=True), FIVE_SEQUENCED), (synth.trio(), dict(cohort_bn=True), [0, 1, 2]),
                         (LONE, dict(cohort_bn=True), [0]), (synth.trio(), dict(cohort_mcmc=True), [0, 1, 2])):
        ped = tiled(fam, F)
        cols = tiled_cols(fam.n, seq, F)
        t0 = time.perf_counter()
        with fs.Engine(*ped, cols, device=-1, **kw) as e:
            dt = time.perf_counter() - t0
            sizes, kids = family_sizes(e)
            fam_of = e.families()[0]
        print(f"{list(kw)[0]}: {F} families of {fam.n}: {dt * 1e3:.0f} ms")
        assert len(sizes) == F and (sizes == fam.n).all() and (kids == sum(1 for m in fam.mids if m)).all()
        assert np.array_equal(fam_of, np.repeat(np.arange(F), fam.n))  # families numbered by their first row: copy f is family f
        assert dt < 20.0


@pytest.mark.parametrize("F", CLASS_SIZES)
def test_regrouped_cohort_keeps_the_trailing_trios(F):
    (ids, mids, fids, genders), R = regrouped(F)
    assert len(ids) == 3 * F and R % 15 == 0 and 0 < F - R <= GRID_Y
    trios = tiled(synth.trio(), F)
    for a, b in zip((ids, mids, fids, genders), trios):
        assert np.array_equal(a[3 * R:], b[3 * R:])
    with fs.Engine(ids, mids, fids, genders, np.arange(3 * F, dtype=np.int32), device=-1, cohort_mcmc=True) as e:
        sizes, _ = family_sizes(e)
        fam_of = e.families()[0]
    assert len(sizes) == R // 15 + F - R
    assert (sizes[:R // 15] == 45).all() and (sizes[R // 15:] == 3).all()
    assert np.array_equal(fam_of[3 * R:], R // 15 + np.repeat(np.arange(F - R), 3))
