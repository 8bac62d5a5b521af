"""Gene assignments whose genes interleave in locus order, and checks of what the packers make of them.

Real group files list a gene's transcripts wherever the transcript list puts them, and transcripts missing from the file
become genes of their own with ids from len(groups) up (gbrs_b200.utils._gene_index).  So the genes of a class' loci,
read in locus order, can go A, B, A.  Both packers re-sort every class row by (gene, locus) and cut (class, gene) runs;
every gene-aware kernel relies on the pairs of one gene being adjacent in the row.  With contiguous genes (what
`synth.generate` and `tests/layouts.py` make) that order is locus order, and none of it is exercised.

`interleave(d, seed)` returns a copy of a `synth.SynthData` with a new gene assignment that has
  * for every class width K in 3..8, 9 and 40, a class with a gene split in locus order (A..B..A), and for K = 2 a class
    whose two loci are in descending gene order (so every fixed-width row pass and both row-pointer widths see a row the
    sort reorders);
  * genes spread over the whole locus range, one gene of at least MIN_BIG_GENE loci, single-locus genes;
  * about 10 % of the loci in no group, between grouped loci;
  * the layout's zero locus (if any) inside a multi-locus gene;
  * group lists in non-ascending locus order, genes listed in an order unrelated to their first locus, and one locus
    listed twice inside one group (harmless, as in the reference's group conversion matrix).
The copy is an `InterleavedSynth` whose `groups()` returns these lists, so `synth.to_apm`, `synth.write_group_file`,
`synth.genotype_mask` and `tests/boot_ref.compact_synth` follow it unchanged.  Its `gene_of` is the gene id of every locus
as the product computes it from the lists (ungrouped loci included).

`assert_genes_interleave(d, packed)` fails if a packed pattern does not contain those shapes; `assert_packed_structure`
checks the packed rows, runs and locus-major entries against the input, independently of either packer."""
from __future__ import annotations

import dataclasses

import numpy as np

from gbrs_b200 import synth
from gbrs_b200.utils import _gene_index
from tests.packed_emulation import unpack_entries

SPLIT_WIDTHS = (3, 4, 5, 6, 7, 8, 9, 40)  # widths that must hold a class with a gene split in locus order
REORDER_WIDTHS = (2,) + SPLIT_WIDTHS  # widths that must hold a class whose row the (gene, locus) sort reorders
MIN_BIG_GENE = 9  # more loci than a fixed-width row pass has pairs: the gene sums of k_gene_totals
UNGROUPED_FRAC = 0.1


@dataclasses.dataclass
class InterleavedSynth(synth.SynthData):
    group_lists: list = None  # gene -> locus ids, in the order of the group file

    def groups(self) -> list[list[int]]:
        return [list(g) for g in self.group_lists]


def gene_ids(d) -> np.ndarray:
    """int64 gene id per locus, as the product derives it from `d.groups()`"""
    return _gene_index(d.T, d.groups()).astype(np.int64)


def _class_loci(d):
    """sorted loci of every input class (classes without pairs: empty)"""
    pc, pl = np.asarray(d.pair_class), np.asarray(d.pair_locus)
    order = np.lexsort((pl, pc))
    bounds = np.searchsorted(pc[order], np.arange(d.N + 1))
    return np.split(pl[order], bounds[1:-1])


def interleave(d: synth.SynthData, seed: int = 0) -> InterleavedSynth:
    rng = np.random.default_rng(7919 + seed)
    T = d.T
    gene = np.full(T, -1, dtype=np.int64)  # provisional gene label per locus (-1: not yet placed)
    n_lab = 0
    loci_of = _class_loci(d)
    width = np.array([len(x) for x in loci_of])
    zero = getattr(d, "zero_locus", None)

    # 1. per width, a class with a split gene A..B..A: its first and last pair in gene A, a pair between in gene B
    for K in SPLIT_WIDTHS:
        done = not (width == K).any()  # (a width the input lacks: tests/layouts.py has them all)
        for n in rng.permutation(np.flatnonzero(width == K)):
            loci = loci_of[n]
            for i, k in [(0, K - 1)] + [(int(a), int(b)) for a, b in rng.integers(0, K, (4 * K, 2)) if b - a >= 2]:
                a = [int(gene[loci[i]]), int(gene[loci[k]])]
                labels = {x for x in a if x >= 0}
                if len(labels) > 1:
                    continue
                lab_a = labels.pop() if labels else None
                mids = [j for j in range(i + 1, k) if gene[loci[j]] < 0 or int(gene[loci[j]]) != lab_a]
                if not mids:
                    continue
                if lab_a is None:
                    lab_a, n_lab = n_lab, n_lab + 1
                gene[loci[i]] = gene[loci[k]] = lab_a
                j = mids[int(rng.integers(0, len(mids)))]
                if gene[loci[j]] < 0:
                    gene[loci[j]], n_lab = n_lab, n_lab + 1
                done = True
                break
            if done:
                break
        if not done:
            raise ValueError(f"no class of width {K} can hold a split gene")

    # 2. a width-2 class whose loci go to two different genes (listed so that the higher locus' gene comes first, below)
    descend = None
    for n in rng.permutation(np.flatnonzero(width == 2)):
        lo, hi = (int(x) for x in loci_of[n])
        if gene[lo] >= 0 and gene[hi] >= 0 and gene[lo] == gene[hi]:
            continue
        for t in (lo, hi):
            if gene[t] < 0:
                gene[t], n_lab = n_lab, n_lab + 1
        descend = (int(gene[lo]), int(gene[hi]))
        break
    if descend is None and (width == 2).any():
        raise ValueError("no class of width 2 can have two genes")

    # 3. about 10 % of the loci in no group, strictly between grouped loci; the zero locus stays grouped
    free = [t for t in range(1, T - 1) if gene[t] < 0 and t != zero]
    n_ungrouped = min(len(free), max(1, int(round(UNGROUPED_FRAC * T))))
    ungrouped = set(int(t) for t in rng.choice(free, n_ungrouped, replace=False)) if free else set()

    # 4. one big gene: the largest label so far grows to at least MIN_BIG_GENE loci, taken evenly over the locus range
    open_loci = [t for t in range(T) if gene[t] < 0 and t not in ungrouped]
    sizes = np.bincount(gene[gene >= 0], minlength=n_lab)
    big = int(np.argmax(sizes))
    need = max(0, MIN_BIG_GENE - int(sizes[big]))
    if need and open_loci:
        spread = {open_loci[i] for i in np.linspace(0, len(open_loci) - 1, need).round().astype(int)}
        for t in spread:
            gene[t] = big
        open_loci = [t for t in open_loci if t not in spread]
    rng.shuffle(open_loci)
    if zero is not None and gene[zero] < 0:
        gene[zero] = big
        open_loci = [t for t in open_loci if t != zero]

    # 5. everything else: single-locus genes and genes of 2-4 loci drawn from anywhere in the range
    while open_loci:
        t = open_loci.pop()
        r = rng.random()
        if r < 0.25:
            gene[t], n_lab = n_lab, n_lab + 1  # a single-locus gene
        elif r < 0.55:
            gene[t] = int(rng.integers(0, n_lab))  # joins an existing gene anywhere in the range
        else:
            k = min(int(rng.integers(1, 4)), len(open_loci))
            gene[t] = n_lab
            for _ in range(k):
                gene[open_loci.pop(int(rng.integers(0, len(open_loci))))] = n_lab
            n_lab += 1
    if zero is not None and np.count_nonzero(gene == gene[zero]) < 2:  # the zero locus joins a multi-locus gene
        gene[zero] = big

    # 6. group lists: loci shuffled (never ascending), genes in random order, one locus repeated inside one group
    labels = [lab for lab in range(n_lab) if (gene == lab).any()]
    order = [labels[i] for i in rng.permutation(len(labels))]
    if descend is not None:  # the width-2 class: the gene of its higher locus listed first
        a, b = order.index(descend[0]), order.index(descend[1])
        if a < b:
            order[a], order[b] = order[b], order[a]
    lists = []
    for lab in order:
        loci = [int(t) for t in rng.permutation(np.flatnonzero(gene == lab))]
        if len(loci) > 1 and loci == sorted(loci):
            loci.reverse()
        lists.append(loci)
    multi = [g for g, x in enumerate(lists) if len(x) > 1]
    dup = lists[multi[int(rng.integers(0, len(multi)))]]
    dup.insert(int(rng.integers(0, len(dup) + 1)), dup[int(rng.integers(0, len(dup)))])

    out = InterleavedSynth(**{f.name: getattr(d, f.name) for f in dataclasses.fields(synth.SynthData)},
                           group_lists=lists)
    out.lname = list(d.lname)
    out.gname = [f"IG{g:05d}" for g in range(len(lists))]
    out.gene_of = gene_ids(out)
    if zero is not None:
        out.zero_locus = zero
    if d.genotype is not None or d.H > 1:
        gi = np.sort(rng.integers(0, d.H, size=(len(lists), 2)), axis=1)
        out.genotype = [synth.HAPLOTYPES[a] + synth.HAPLOTYPES[b] for a, b in gi]
    else:
        out.genotype = ["AA"] * len(lists)
    _assert_assignment(out, zero)
    return out


def _assert_assignment(d, zero):
    """the properties the module docstring promises, on the group lists themselves"""
    lists = d.groups()
    gene = d.gene_of
    G = len(lists)
    listed = np.zeros(d.T, dtype=bool)
    for x in lists:
        listed[x] = True
    ungrouped = np.flatnonzero(~listed)
    assert ungrouped.size >= 1 and listed[0] and listed[-1], "ungrouped loci must sit between grouped ones"
    sizes = np.array([len(set(x)) for x in lists])
    assert sizes.max() >= MIN_BIG_GENE and (sizes == 1).any()
    big = lists[int(np.argmax(sizes))]
    assert max(big) - min(big) >= d.T // 2, "the big gene spans the locus range"
    assert any(len(x) > 1 and x != sorted(x) for x in lists)
    firsts = [min(x) for x in lists]
    assert firsts != sorted(firsts)
    assert any(len(x) != len(set(x)) for x in lists), "one locus listed twice inside a group"
    if zero is not None:
        assert gene[zero] < G and sizes[gene[zero]] > 1
    assert np.all(gene[ungrouped] >= G)


# ----------------------------------------------------------------------------------------------------------------------
# checks on packed patterns
# ----------------------------------------------------------------------------------------------------------------------
def _host_arrays(packed):
    return packed.arrays if getattr(packed, "arrays", None) else packed.to_host()


def _rows(arrays):
    rp = np.asarray(arrays["rowptr"], dtype=np.int64)
    pw = np.asarray(arrays["pairs"], dtype=np.int64)
    return rp, pw & 0xFFFFFF, pw >> 24


def interleave_summary(d, arrays) -> dict:
    """Per class width: how many packed classes the (gene, locus) sort reorders, and how many have a gene split in locus
    order (fewer genes than gene changes + 1).  Computed from the loci of each packed class and the genes of the input,
    not from the packer's row order."""
    gene = gene_ids(d)
    rp, loc, _ = _rows(arrays)
    reordered, split = {}, {}
    for n in range(rp.size - 1):
        loci = np.sort(loc[rp[n]:rp[n + 1]])
        K = int(loci.size)
        g = gene[loci]
        changes = int(np.count_nonzero(np.diff(g)))
        reordered[K] = reordered.get(K, 0) + int(bool((np.diff(g) < 0).any()))
        split[K] = split.get(K, 0) + int(np.unique(g).size < changes + 1)
    return dict(reordered=reordered, split=split)


def assert_genes_interleave(d, packed) -> dict:
    """For every width K in 2..8, 9 and 40 a class the sort reorders; for every K in 3..8, 9 and 40 a class with a gene
    split in locus order (A..B..A).  Genes enter neither the class order nor the item layout, so
    tests/layouts.assert_layout_covers still holds on the same pattern."""
    s = interleave_summary(d, _host_arrays(packed))
    missing = [K for K in REORDER_WIDTHS if not s["reordered"].get(K)]
    assert not missing, f"no class reordered by the (gene, locus) sort at widths {missing} ({s})"
    missing = [K for K in SPLIT_WIDTHS if not s["split"].get(K)]
    assert not missing, f"no class with a gene split in locus order at widths {missing} ({s})"
    return s


def input_rows(d, hapmask=None):
    """input class id -> sorted list of (locus, mask) (masks restricted by `hapmask`, empty pairs dropped)"""
    rows = {}
    for c, t, m in zip(np.asarray(d.pair_class), np.asarray(d.pair_locus), np.asarray(d.pair_mask)):
        m = int(m) & (int(hapmask[t]) if hapmask is not None else 0xFF)
        if m:
            rows.setdefault(int(c), []).append((int(t), m))
    return {c: sorted(v) for c, v in rows.items()}


def assert_packed_structure(d, info, arrays, hapmask=None) -> None:
    """The packed arrays against the input, for any packer:
      * row n holds exactly the (locus, mask) multiset of input class class_id[n], sorted by (gene, locus);
      * runptr[n + 1] - runptr[n] is the number of distinct genes of the class;
      * every real locus-major entry of locus t points (ent_pair) at a pair of locus t with the entry's mask inside the row
        of its class (ent_cls), and ent_run is runptr[class] plus that pair's run index;
      * gene_of is the product's gene index, gene_ptr / gene_loci its CSR (loci ascending per gene)."""
    gene = gene_ids(d)
    n_classes, n_pairs = int(info["n_classes"]), int(info["n_pairs"])
    rp, loc, msk = _rows(arrays)
    assert rp.size == n_classes + 1 and rp[-1] == n_pairs
    assert np.array_equal(np.asarray(arrays["gene_of"], dtype=np.int64), gene)
    G = int(gene.max()) + 1
    assert int(info["n_gene_ids"]) == G
    gp = np.asarray(arrays["gene_ptr"], dtype=np.int64)
    assert np.array_equal(gp, np.concatenate(([0], np.cumsum(np.bincount(gene, minlength=G)))))
    assert np.array_equal(np.asarray(arrays["gene_loci"], dtype=np.int64), np.argsort(gene, kind="stable"))
    want_rows = input_rows(d, hapmask)
    cid = np.asarray(arrays["class_id"], dtype=np.int64)
    assert cid.size == n_classes and np.unique(cid).size == n_classes and set(cid.tolist()) == set(want_rows)
    runptr = np.asarray(arrays["runptr"], dtype=np.int64)
    assert runptr.size == n_classes + 1 and runptr[0] == 0 and runptr[-1] == int(info["n_runs"])
    run_of_pair = np.zeros(n_pairs, dtype=np.int64)
    for n in range(n_classes):
        row = list(zip(loc[rp[n]:rp[n + 1]].tolist(), msk[rp[n]:rp[n + 1]].tolist()))
        want = sorted(want_rows[int(cid[n])], key=lambda p: (int(gene[p[0]]), p[0]))
        assert row == want, f"packed class {n} (input class {cid[n]}): row {row}, want (gene, locus) order {want}"
        g = gene[loc[rp[n]:rp[n + 1]]]
        assert runptr[n + 1] - runptr[n] == np.unique(g).size, f"packed class {n}: runs"
        run_of_pair[rp[n]:rp[n + 1]] = runptr[n] + np.concatenate(([0], np.cumsum(np.diff(g) != 0)))
    eb = int(info["entry_bytes"])
    idx_c, m_c = unpack_entries(np.asarray(arrays["ent_cls"]), eb)
    idx_p, m_p = unpack_entries(np.asarray(arrays["ent_pair"]), eb)
    idx_r, m_r = unpack_entries(np.asarray(arrays["ent_run"]), eb)
    assert np.array_equal(m_c, m_p) and np.array_equal(m_c, m_r)
    # the locus of an entry from the item layout (item_desc: entry range of each item; locus_desc: items of each locus)
    n_items = int(info["n_items"])
    desc = np.asarray(arrays["item_desc"], dtype=np.int64).reshape(-1, 4)[:n_items]
    begin, end = np.zeros(n_items, dtype=np.int64), np.zeros(n_items, dtype=np.int64)
    begin[desc[:, 2]], end[desc[:, 2]] = desc[:, 0], desc[:, 1]
    locus_of_entry = np.full(idx_c.size, -1, dtype=np.int64)
    for t, i0, i1, _ in np.asarray(arrays["locus_desc"], dtype=np.int64).reshape(-1, 4):
        for i in range(i0, i1):
            locus_of_entry[begin[i]:end[i]] = t
    real = m_c != 0
    assert np.count_nonzero(real) == n_pairs
    e_cls, e_pair, e_run, e_loc, e_msk = idx_c[real], idx_p[real], idx_r[real], locus_of_entry[real], m_c[real]
    assert np.all(e_pair < n_pairs) and np.all(e_cls < n_classes)
    assert np.all((rp[e_cls] <= e_pair) & (e_pair < rp[e_cls + 1])), "an entry's pair lies outside its class' row"
    assert np.array_equal(loc[e_pair], e_loc), "an entry's pair is not at the entry's locus"
    assert np.array_equal(msk[e_pair], e_msk)
    assert np.array_equal(run_of_pair[e_pair], e_run), "ent_run is not the run of the entry's pair"
    assert np.unique(e_pair).size == n_pairs  # every pair has exactly one entry
