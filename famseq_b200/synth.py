"""Deterministic synthetic pedigrees and sequencing likelihoods (SURVEY.md section 8(d)).

Pedigrees: `trio`, `ped14` (3 generations, loop-free) and `ped40` (4 generations, 9 founders, marriage
and consanguinity loops).  Likelihoods: founder alleles ~ Bernoulli(AF), gene-dropped through the
pedigree without mutation, read depth ~ Poisson(30), alt reads ~ Binomial(depth, {0.01, 0.5, 0.99}[g]),
PL = round(-10 log10(L / Lmax)) clipped to [0, 2550], likelihood = 10^(-PL/10) exactly as the VCF
driver decodes it (file.cpp:588-590).  The stream is keyed by (seed, chunk of 65536 sites), so any slice
of a data set can be generated on its own (multi-GPU shards generate only their part).
"""
from __future__ import annotations

from dataclasses import dataclass, field

import math

import numpy as np

CHUNK = 65536
AFS = (0.01, 0.05, 0.2, 0.5)
ERR = np.array([0.01, 0.5, 0.99])


@dataclass
class PedFile:
    """Rows of a FamSeq ped file (file.cpp:24-62): id, mother id, father id, gender, sample name."""
    ids: list
    mids: list
    fids: list
    genders: list
    names: list = field(default_factory=list)

    @property
    def n(self) -> int:
        return len(self.ids)

    def sequenced_cols(self) -> list:
        return [i for i, nm in enumerate(self.names) if nm != "NA"]

    def write(self, path: str) -> None:
        with open(path, "w") as fh:
            fh.write("ID\tmID\tfID\tgender\tIndividualName\n")
            for r in zip(self.ids, self.mids, self.fids, self.genders, self.names):
                fh.write("\t".join(str(x) for x in r) + "\n")

    @staticmethod
    def read(path: str) -> "PedFile":
        ids, mids, fids, genders, names = [], [], [], [], []
        with open(path) as fh:
            fh.readline()
            for line in fh:
                line = line.rstrip("\n")
                if len(line) < 2:
                    break
                t = line.split()
                ids.append(int(t[0])); mids.append(int(t[1])); fids.append(int(t[2]))
                genders.append(int(t[3])); names.append(t[4] if len(t) > 4 else "")
        return PedFile(ids, mids, fids, genders, names)

    def parents(self):
        """(mother row, father row) per member, -1 for founders (last matching id wins, as the reference)."""
        row = {}
        for j, i in enumerate(self.ids):
            row[i] = j
        return [(row.get(m, -1), row.get(f, -1)) for m, f in zip(self.mids, self.fids)]


def _mk(rows, prefix="s") -> PedFile:
    ids, mids, fids, genders = (list(x) for x in zip(*rows))
    return PedFile(ids, mids, fids, genders, [f"{prefix}{i:02d}" for i in ids])


def trio() -> PedFile:
    return _mk([(1, 0, 0, 1), (2, 0, 0, 2), (3, 2, 1, 1)])


def ped14() -> PedFile:
    """Two founder couples -> 3 + 2 children; one inter-family couple and one couple with a married-in
    founder -> 2 + 2 grandchildren.  5 founders, loop-free."""
    return _mk([
        (1, 0, 0, 1), (2, 0, 0, 2), (3, 0, 0, 1), (4, 0, 0, 2),
        (5, 2, 1, 1), (6, 2, 1, 2), (7, 2, 1, 1), (8, 4, 3, 2), (9, 4, 3, 1),
        (10, 0, 0, 2),
        (11, 8, 5, 1), (12, 8, 5, 2), (13, 10, 9, 2), (14, 10, 9, 1),
    ])


def ped40() -> PedFile:
    """Four generations, 9 founders.  Loops: two brothers (5,6) marry two sisters (8,9); their children
    are double first cousins and 13 x 16 mate; 17 x 20 is a further first-cousin mating."""
    rows = [
        (1, 0, 0, 1), (2, 0, 0, 2), (3, 0, 0, 1), (4, 0, 0, 2),
        (5, 2, 1, 1), (6, 2, 1, 1), (7, 2, 1, 2), (8, 4, 3, 2), (9, 4, 3, 2), (10, 4, 3, 1),
        (11, 0, 0, 1), (12, 0, 0, 2),
        (13, 8, 5, 1), (14, 8, 5, 2), (15, 8, 5, 1), (16, 9, 6, 2), (17, 9, 6, 1), (18, 9, 6, 2),
        (19, 7, 11, 1), (20, 7, 11, 2), (21, 12, 10, 2), (22, 12, 10, 1),
        (23, 0, 0, 1), (24, 0, 0, 2), (25, 0, 0, 2),
        (26, 16, 13, 1), (27, 16, 13, 2), (28, 16, 13, 1),
        (29, 20, 17, 2), (30, 20, 17, 1), (31, 20, 17, 2),
        (32, 14, 23, 1), (33, 14, 23, 2), (34, 14, 23, 1),
        (35, 24, 15, 2), (36, 24, 15, 1), (37, 24, 15, 2),
        (38, 25, 22, 1), (39, 25, 22, 2), (40, 25, 22, 1),
    ]
    return _mk(rows)


def half_sibs() -> PedFile:
    """A man with two wives (half-sib families) and a grandchild: several spouses per member, loop-free."""
    return _mk([
        (1, 0, 0, 1), (2, 0, 0, 2), (3, 0, 0, 2),
        (4, 2, 1, 1), (5, 2, 1, 2), (6, 3, 1, 2), (7, 3, 1, 1),
        (8, 0, 0, 2), (9, 8, 4, 1), (10, 8, 4, 2),
    ])


def three_wives() -> PedFile:
    """A man with three wives: exercises the (ant*lk)*(pos*pos) association of the reference."""
    return _mk([
        (1, 0, 0, 1), (2, 0, 0, 2), (3, 0, 0, 2), (4, 0, 0, 2),
        (5, 2, 1, 1), (6, 3, 1, 2), (7, 4, 1, 1), (8, 4, 1, 2),
        (9, 0, 0, 1), (10, 6, 9, 2),
    ])


def cousins_loop() -> PedFile:
    """First-cousin marriage (9 members): the smallest consanguinity loop; ES must refuse it."""
    return _mk([
        (1, 0, 0, 1), (2, 0, 0, 2),
        (3, 2, 1, 1), (4, 2, 1, 2), (5, 0, 0, 2), (6, 0, 0, 1),
        (7, 5, 3, 1), (8, 4, 6, 2), (9, 8, 7, 1),
    ])


def ped100() -> PedFile:
    """100 members, loop-free: every child of a couple marries a founder and has three children of its own, breadth first
    (beyond the 64 members a two-register genotype vector holds; exercises the wide-vector Gibbs kernel)."""
    rows = [(1, 0, 0, 1), (2, 0, 0, 2)]
    couples = [(2, 1)]  # (mother id, father id)
    nxt = 3
    while len(rows) < 100:
        mother, father = couples.pop(0)
        for k in range(3):
            if len(rows) >= 100:
                break
            child, sex = nxt, 1 + (nxt + k) % 2
            rows.append((child, mother, father, sex))
            nxt += 1
            if len(rows) < 99:  # a founder spouse of the other sex; the pair queues up for children
                spouse = nxt
                rows.append((spouse, 0, 0, 3 - sex))
                nxt += 1
                couples.append((child, spouse) if sex == 2 else (spouse, child))
    return _mk(rows[:100])


def random_pedigree(seed: int, n_target: int, loops: bool = False, shuffle: bool = False, unsequenced: float = 0.0) -> PedFile:
    """A random pedigree for compiler tests: marriages with fresh founders (several spouses per member allowed), 1-3
    children per couple; with `loops`, marriages between existing members too (marriage / consanguinity loops).
    Without `loops` the marriage graph is a forest by construction, i.e. Elston-Stewart applies.  `shuffle` permutes
    the ped rows (children may precede their parents, as the reference allows), `unsequenced` is the fraction of
    members without a sample column."""
    rng = np.random.default_rng(seed)
    rows = [(1, 0, 0, 1), (2, 0, 0, 2)]  # id, mother, father, sex (1 male, 2 female)
    couples = [(2, 1)]
    sex = {1: 1, 2: 2}
    married = {(2, 1)}
    nxt = 3
    while len(rows) < n_target:
        act = rng.random()
        if act < 0.55 or not couples:  # children for a couple
            mother, father = couples[rng.integers(len(couples))]
            for _ in range(int(rng.integers(1, 4))):
                if len(rows) >= n_target:
                    break
                g = int(rng.integers(1, 3))
                rows.append((nxt, mother, father, g))
                sex[nxt] = g
                nxt += 1
        elif act < (0.7 if loops else 2.0):  # somebody marries a fresh founder
            p = int(rows[rng.integers(len(rows))][0])
            g = 3 - sex[p]
            rows.append((nxt, 0, 0, g))
            sex[nxt] = g
            pair = (p, nxt) if sex[p] == 2 else (nxt, p)
            couples.append(pair)
            married.add(pair)
            nxt += 1
        else:  # two existing members marry (may close a loop)
            a, b = (int(rows[i][0]) for i in rng.integers(len(rows), size=2))
            if sex[a] == sex[b]:
                continue
            pair = (a, b) if sex[a] == 2 else (b, a)
            if pair in married:
                continue
            parents = {r[0]: (r[1], r[2]) for r in rows}
            if pair[0] in parents[pair[1]] or pair[1] in parents[pair[0]]:
                continue  # no parent-child marriages
            couples.append(pair)
            married.add(pair)
            for _ in range(int(rng.integers(1, 3))):  # the marriage shows (and can close a loop) only through children
                if len(rows) >= n_target:
                    break
                g = int(rng.integers(1, 3))
                rows.append((nxt, pair[0], pair[1], g))
                sex[nxt] = g
                nxt += 1
    # couples without children are dropped by construction of the ped file (a marriage only shows through children)
    if shuffle:
        rows = [rows[i] for i in rng.permutation(len(rows))]
    ped = _mk(rows)
    if unsequenced > 0:
        for i in range(ped.n):
            if rng.random() < unsequenced:
                ped.names[i] = "NA"
        if not ped.sequenced_cols():
            ped.names[0] = "s00"
    return ped


def sibship(n_children: int) -> PedFile:
    """One couple (father 1, mother 2) and `n_children` full sibs of mixed sexes."""
    return _mk([(1, 0, 0, 1), (2, 0, 0, 2)] + [(3 + k, 2, 1, 1 + (k % 3 == 1)) for k in range(n_children)])


def many_spouses(n_spouses: int = 5) -> PedFile:
    """A man (1) with `n_spouses` wives, two or three children with each; one son has a family of his own."""
    rows = [(1, 0, 0, 1)]
    nxt = 2
    for w in range(n_spouses):
        wife = nxt
        rows.append((wife, 0, 0, 2))
        nxt += 1
        for k in range(2 + w % 2):
            rows.append((nxt, wife, 1, 1 + (nxt % 2)))
            nxt += 1
    son = next(r[0] for r in rows if r[2] == 1 and r[3] == 1)
    rows += [(nxt, 0, 0, 2), (nxt + 1, nxt, son, 1), (nxt + 2, nxt, son, 2)]
    return _mk(rows)


def three_generations(sibs: int = 8) -> PedFile:
    """A sibship of `sibs` in each of three generations: one son of each sibship marries a founder and has the next."""
    rows, father, mother, nxt = [(1, 0, 0, 1), (2, 0, 0, 2)], 1, 2, 3
    for gen in range(3):
        kids = [(nxt + k, mother, father, 1 + (k % 2 == 0)) for k in range(sibs)]
        rows += kids
        nxt += sibs
        if gen < 2:
            father = next(r[0] for r in kids if r[3] == 1)
            mother = nxt
            rows.append((mother, 0, 0, 2))
            nxt += 1
    return _mk(rows)


def forest(families, shuffle_seed=None):
    """Several unrelated families in one ped file: ids of family f are offset past those of the families before it.
    Returns (ped, rows): rows[f] are the ped rows of family f in the file's order (with `shuffle_seed`, the rows of all
    families are interleaved at random)."""
    out, fam, base = [], [], 0
    for f, p in enumerate(families):
        off = lambda i: i + base if i else 0
        out += [(off(i), off(m), off(fa), g) for i, m, fa, g in zip(p.ids, p.mids, p.fids, p.genders)]
        fam += [f] * p.n
        base += max(p.ids)
    order = np.arange(len(out)) if shuffle_seed is None else np.random.default_rng(shuffle_seed).permutation(len(out))
    ped = _mk([out[i] for i in order])
    fam = np.asarray(fam)[order]
    return ped, [np.nonzero(fam == f)[0] for f in range(len(families))]


PEDIGREES = {"trio": trio, "ped14": ped14, "ped40": ped40, "half_sibs": half_sibs, "three_wives": three_wives, "ped100": ped100,
             "cousins_loop": cousins_loop}


def _gene_drop(ped: PedFile, af: np.ndarray, chrx: np.ndarray, rng: np.random.Generator) -> np.ndarray:
    """Genotypes [V][N] (0,1,2) by dropping founder alleles through the pedigree, mutation-free."""
    V, N = af.shape[0], ped.n
    par = ped.parents()
    hap = np.zeros((V, N, 2), np.int8)  # [.,.,0] maternal allele, [.,.,1] paternal allele
    done = [False] * N
    pending = list(range(N))
    while pending:
        rest = []
        for i in pending:
            m, f = par[i]
            if m >= 0 and f >= 0 and not (done[m] and done[f]):
                rest.append(i)
                continue
            if m < 0 or f < 0:
                hap[:, i, 0] = rng.random(V) < af
                hap[:, i, 1] = rng.random(V) < af
            else:
                pick_m = rng.integers(0, 2, V)
                pick_f = rng.integers(0, 2, V)
                hap[:, i, 0] = np.take_along_axis(hap[:, m, :], pick_m[:, None], 1)[:, 0]
                hap[:, i, 1] = np.take_along_axis(hap[:, f, :], pick_f[:, None], 1)[:, 0]
            if ped.genders[i] == 1:  # males are hemizygous on X: both slots carry the maternal allele
                hap[:, i, 1] = np.where(chrx, hap[:, i, 0], hap[:, i, 1])
            done[i] = True
        pending = rest
    return (hap[:, :, 0] + hap[:, :, 1]).astype(np.int8)


def _chunk(ped: PedFile, seed: int, chunk: int, x_fraction: float):
    rng = np.random.Generator(np.random.Philox(key=[int(seed) & (2**64 - 1), int(chunk)]))
    site = np.arange(chunk * CHUNK, (chunk + 1) * CHUNK, dtype=np.int64)
    af = np.asarray(AFS)[site % 4]
    chrx = rng.random(CHUNK) < x_fraction if x_fraction > 0 else np.zeros(CHUNK, bool)
    geno = _gene_drop(ped, af, chrx, rng)
    cols = ped.sequenced_cols()
    g = geno[:, cols]
    depth = rng.poisson(30.0, g.shape)
    alt = rng.binomial(depth, ERR[g])
    ll = alt[..., None] * np.log10(ERR) + (depth - alt)[..., None] * np.log10(1.0 - ERR)
    pl = np.clip(np.rint(-10.0 * (ll - ll.max(-1, keepdims=True))), 0, 2550).astype(np.int32)
    flags = ((site % 3 == 0).astype(np.uint8)) | (chrx.astype(np.uint8) << 1)
    return pl, flags


def synth_pl(ped: PedFile, n_variants: int, seed: int, v0: int = 0, x_fraction: float = 0.0):
    """PL integers [V][S][3] and flags [V] (bit0 Known: every third site has an rs id; bit1 chrX)."""
    pls, fls = [], []
    first, last = v0 // CHUNK, (v0 + n_variants - 1) // CHUNK if n_variants > 0 else v0 // CHUNK - 1
    for c in range(first, last + 1):
        pl, fl = _chunk(ped, seed, c, x_fraction)
        lo = max(v0 - c * CHUNK, 0)
        hi = min(v0 + n_variants - c * CHUNK, CHUNK)
        pls.append(pl[lo:hi])
        fls.append(fl[lo:hi])
    S = len(ped.sequenced_cols())
    if not pls:
        return np.zeros((0, S, 3), np.int32), np.zeros(0, np.uint8)
    return np.concatenate(pls), np.concatenate(fls)


_PL_TABLE = None


def pl_table() -> np.ndarray:
    """pow(10, -pl/10) for pl = 0..65535 evaluated by libm (math.pow), like the reference's VCF driver and like the
    engine's fs_run_pl decode table; numpy's own power() differs from libm in the last bit for ~0.2 % of these."""
    global _PL_TABLE
    if _PL_TABLE is None:
        _PL_TABLE = np.array([math.pow(10.0, -abs(float(k)) / 10.0) for k in range(65536)], dtype=np.float64)
    return _PL_TABLE


def pl_to_likelihood(pl: np.ndarray) -> np.ndarray:
    """The VCF driver's decode: pow(10, -|PL|/10) (file.cpp:588-590); integer PLs beyond 65535 decode to 0 anyway."""
    return pl_table()[np.minimum(np.abs(pl.astype(np.int64)), 65535)]


def synth_likelihoods(ped: PedFile, n_variants: int, seed: int, v0: int = 0, x_fraction: float = 0.0):
    """Likelihoods [V][S][3] float64 and flags [V] uint8 for sites v0 .. v0+n_variants-1."""
    pl, flags = synth_pl(ped, n_variants, seed, v0, x_fraction)
    return pl_to_likelihood(pl), flags


def write_vcf(path: str, ped: PedFile, pl: np.ndarray, flags: np.ndarray, v0: int = 0) -> None:
    """A minimal multi-sample VCF carrying GT:DP:PL, in the shape the reference driver expects."""
    cols = ped.sequenced_cols()
    names = [ped.names[i] for i in cols]
    gt_txt = ("0/0", "0/1", "1/1")
    with open(path, "w") as fh:
        fh.write("##fileformat=VCFv4.1\n")
        fh.write('##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n')
        fh.write('##FORMAT=<ID=DP,Number=1,Type=Integer,Description="Depth">\n')
        fh.write('##FORMAT=<ID=PL,Number=G,Type=Integer,Description="Phred-scaled genotype likelihoods">\n')
        fh.write('##INFO=<ID=DP,Number=1,Type=Integer,Description="Total depth">\n')
        fh.write("##contig=<ID=1>\n")
        fh.write("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(names) + "\n")
        bases = "ACGT"
        for v in range(pl.shape[0]):
            site = v0 + v
            chrom = "X" if (flags[v] >> 1) & 1 else str(site % 22 + 1)
            rsid = f"rs{site}" if flags[v] & 1 else "."
            ref, alt = bases[site % 4], bases[(site + 1 + site // 4 % 3) % 4]
            fields = []
            for s in range(pl.shape[1]):
                p = pl[v, s]
                fields.append(f"{gt_txt[int(np.argmin(p))]}:30:{p[0]},{p[1]},{p[2]}")
            fh.write(f"{chrom}\t{1000 + site}\t{rsid}\t{ref}\t{alt}\t50\tPASS\tDP=90\tGT:DP:PL\t" + "\t".join(fields) + "\n")
