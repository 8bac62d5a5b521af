"""Inputs whose packed layout is prescribed, and a check that the packer really produced it.

`make_layout(H, item_len)` builds a `synth.SynthData` in which every kind of work the EM kernels dispatch on occurs, each
at or one past the packer's thresholds (gbrs_b200/csrc/pack.cpp, step 6; L = item_len):
  * locus depths of exactly 8L (one mixed part: exactly 8 short items) and 8L+1 (split into a partial and a full part:
    9 items, a deep locus);
  * partial and full parts whose length mod L is in 1..4 and in 5..8, so that the last short item of the part has one
    quad or two quads of entry words; with L >= 16 the other short items have more than 8 words;
  * a partial and a full part of 32L+1 entries each (two long items each);
  * classes of every width 1..8 (the fixed-width row passes), 9 (the first row-pointer class) and 40;
  * classes with count 0, among them all classes of one locus (its theta' is exactly 0), and loci without entries;
  * full masks, the single highest haplotype 1 << (H-1) and, for H > 4, masks in the upper nibble only.
At item_len = 8 no short item can have more than 8 words (items of a part are item_len long, the part is padded to whole
quads), so the short-item classes "more than two quads" would be empty: 16 is the smallest item length that reaches all
seven column-pass segments.

`assert_layout_covers(packed)` reads the pack info, the width buckets and the item_desc trailer and fails if a kind of work
is missing.  Every test on a constructed layout calls it: if the packer or the constructor drifts, the test fails instead of
quietly covering less.

`make_empty_shards(kind, R)` builds inputs for which the class split of the packer leaves some of R row shards without a
class; `assert_empty_shards` checks that it did."""
from __future__ import annotations

import numpy as np

from gbrs_b200 import synth

KMAX = 8  # GBRS_KMAX: widths 1..8 take the fixed-width row passes, wider classes the row-pointer ones
DEEP_LOCUS_ITEMS = 8  # GBRS_DEEP_LOCUS_ITEMS
SEGMENTS = ("long", "short partial > 8 words", "short partial <= 8 words", "short partial <= 4 words",
            "short full > 8 words", "short full <= 8 words", "short full <= 4 words")
WIDTHS = tuple(range(1, KMAX + 2)) + (40,)


def _masks(rng, H, n, full_kind):
    """n pair masks: full ones for `full_kind`, otherwise never full -- a third the highest haplotype alone, a third (H > 4)
    in the upper nibble only, the rest anything else."""
    full = (1 << H) - 1
    if full_kind or H == 1:  # (with one haplotype every mask is full)
        return np.full(n, full, dtype=np.uint8)
    m = rng.integers(1, full, n)
    r = rng.random(n)
    m = np.where(r < 1 / 3, 1 << (H - 1), m)
    if H > 4:
        upper = rng.integers(1, 1 << (H - 4), n) << 4
        m = np.where((r >= 1 / 3) & (r < 2 / 3), upper, m)
    return m.astype(np.uint8)


def make_layout(H: int, item_len: int = 16, seed: int = 0) -> synth.SynthData:
    if not (1 <= H <= 8) or item_len % 8 or item_len < 16:
        raise ValueError("H in 1..8, item_len a multiple of 8 and at least 16")
    L = item_len
    rng = np.random.default_rng(1000 * H + L + seed)
    # (partial-mask entries, full-mask entries) per locus
    spec = [(4 * L, 4 * L),          # depth 8L: not split, 8 items
            (4 * L + 1, 4 * L),      # depth 8L+1: split; partial 4L+1 (4 items + one of one quad), full 4 items: 9 items
            (2 * L + 3, 7 * L + 6),  # partial tail of one quad, full tail of two quads
            (L + 6, 7 * L + 2),      # partial tail of two quads, full tail of one quad
            (32 * L + 1, 32 * L + 1)]  # two long partial items, two long full items
    if H == 1:  # no partial masks, so split loci are all full and never short: a locus of 9 long items is the deep one
        spec.append((0, 8 * 32 * L + 1))
    n_shallow, n_empty = 48, 3
    spec += [(int(a), int(b)) for a, b in rng.integers(0, L + 1, size=(n_shallow, 2))]
    spec = [(a, b) if a + b else (1, 0) for a, b in spec]
    z_slot = len(spec)  # the locus only count-0 classes reach
    spec += [(0, 0)] * (n_empty + 1)
    T = len(spec)
    where = rng.permutation(T)  # spec slot -> locus id
    rem = np.zeros((T, 2), dtype=np.int64)
    for s, (a, b) in enumerate(spec):
        rem[where[s]] = (a, b)
    z_locus = int(where[z_slot])
    shallow = where[len(spec) - n_shallow - n_empty - 1: len(spec) - n_empty - 1]

    classes = []  # (loci, kinds, count)

    def take(w):
        alive = np.flatnonzero(rem.sum(axis=1) > 0)
        w = min(w, alive.size)
        p = rem[alive].sum(axis=1).astype(np.float64)
        loci = rng.choice(alive, size=w, replace=False, p=p / p.sum())
        kinds = []
        for t in loci:
            a, b = rem[t]
            k = int(rng.random() >= a / (a + b))
            rem[t, k] -= 1
            kinds.append(k)
        return list(loci), kinds

    # three count-0 classes: the zero locus and a shallow locus each
    for i in range(3):
        t = int(shallow[i])  # (every shallow locus has at least one entry to give)
        k = 0 if rem[t, 0] else 1
        rem[t, k] -= 1
        classes.append(([z_locus, t], [0, k], 0.0))
    for w in WIDTHS:
        for _ in range(3 if w <= KMAX + 1 else 1):
            loci, kinds = take(w)
            assert len(loci) == w
            classes.append((loci, kinds, None))
    while rem.sum():
        loci, kinds = take(int(rng.choice([1, 1, 1, 2, 2, 3, 4, 5])))
        classes.append((loci, kinds, None))
    order = rng.permutation(len(classes))
    N = len(classes)
    pc, pl, pm, count = [], [], [], np.zeros(N)
    for new, old in enumerate(order):
        loci, kinds, c = classes[old]
        o = np.argsort(loci)
        pc += [new] * len(loci)
        pl += [int(loci[i]) for i in o]
        pm += [int(_masks(rng, H, 1, kinds[i])[0]) for i in o]
        count[new] = c if c is not None else (0.0 if rng.random() < 0.05 else float(rng.geometric(0.2)))
    pair_class, pair_locus, pair_mask = np.array(pc, np.int64), np.array(pl, np.int64), np.array(pm, np.uint8)
    # a count-0 class must still keep some (locus, haplotype) alive that a counted class reaches, or a later update would
    # leave it without any positive theta (0 / 0: the reference raises)
    bits = ((pair_mask[:, None] >> np.arange(H)) & 1).astype(bool)
    live = np.zeros((T, H), dtype=bool)
    live[pair_locus[:, None].repeat(H, 1)[bits & (count[pair_class] > 0)[:, None]],
         np.broadcast_to(np.arange(H), bits.shape)[bits & (count[pair_class] > 0)[:, None]]] = True
    reaches_live = np.zeros(N, dtype=bool)
    np.logical_or.at(reaches_live, pair_class, (bits & live[pair_locus]).any(axis=1))
    count[(count == 0) & ~reaches_live] = 1.0  # (count-0 classes at the zero locus reach their shallow locus)
    gsize = rng.integers(1, 5, T)
    gene_of = np.repeat(np.arange(T), gsize)[:T].astype(np.int64)
    lengths = rng.integers(300, 6000, size=(T, H)).astype(np.float64)
    d = synth.SynthData(T=T, H=H, N=N, pair_class=pair_class, pair_locus=pair_locus, pair_mask=pair_mask, count=count,
                        gene_of=gene_of, lengths=lengths, hname=synth.HAPLOTYPES[:H])
    d.lname = [f"T{t:05d}" for t in range(T)]
    d.gname = [f"G{g:05d}" for g in range(int(gene_of.max()) + 1)]
    d.zero_locus = z_locus
    widths = np.bincount(pair_class, minlength=N)
    assert set(WIDTHS) <= set(widths.tolist())
    assert np.all(count[np.unique(pair_class[pair_locus == z_locus])] == 0)
    return d


def make_heavy_first_class(T: int, seed: int = 0) -> synth.SynthData:
    """Class 0 hits every locus with a full mask of 8 haplotypes; the other T // 2 classes are single pairs of one
    haplotype.  Class 0 holds 16/17 of the nnz, more than (R - 1) / R for any R <= 8, so the packer's class split (class c
    to rank floor(cum_before(c) R / nnz)) sends class 0 to rank 0, everything else to rank R - 1 and nothing in between."""
    rng = np.random.default_rng(seed)
    n_small = T // 2
    pc = [0] * T + list(range(1, n_small + 1))
    pl = list(range(T)) + [int(t) for t in rng.integers(0, T, n_small)]
    pm = [0xFF] * T + [1 << int(h) for h in rng.integers(0, 8, n_small)]
    d = synth.SynthData(T=T, H=8, N=n_small + 1, pair_class=np.array(pc, np.int64), pair_locus=np.array(pl, np.int64),
                        pair_mask=np.array(pm, np.uint8), count=rng.integers(1, 20, n_small + 1).astype(np.float64),
                        gene_of=np.repeat(np.arange(T), 3)[:T].astype(np.int64),
                        lengths=rng.integers(300, 6000, size=(T, 8)).astype(np.float64), hname=synth.HAPLOTYPES[:8])
    d.lname = [f"T{t:04d}" for t in range(T)]
    d.gname = [f"G{g:04d}" for g in range(int(d.gene_of.max()) + 1)]
    return d


def make_empty_shards(kind: str, R: int) -> synth.SynthData:
    """An input that leaves some of R row shards without any class: "few classes" (fewer classes than ranks) or "heavy
    first class" (make_heavy_first_class)."""
    if kind == "few classes":
        return synth.generate(T=6, N=max(1, R - 3), H=8, sample_index=4)
    if kind == "heavy first class":
        return make_heavy_first_class(T=20, seed=R)
    raise ValueError(kind)


def assert_empty_shards(kind: str, d, classes, nnz) -> None:
    """`classes` / `nnz`: per shard, from the pack info.  The shards hold all of the nnz, and the ranks the input was built
    to leave empty really have no class."""
    R = len(classes)
    nnz = [int(n) for n in nnz]
    assert sum(nnz) == d.nnz, (nnz, d.nnz)
    empty = [r for r, c in enumerate(classes) if c == 0]
    assert all(nnz[r] == 0 for r in empty)
    if kind == "few classes":
        assert d.N < R and len(empty) >= R - d.N, classes
    else:
        assert empty == list(range(1, R - 1)) and classes[0] == 1, classes


def layout_summary(info, item_desc) -> dict:
    """Work items per column-pass segment (k_column_reduce's slot segments, in that order), long items per kind, classes
    per row-pass width bucket (1..8, then the row-pointer bucket), deep loci."""
    n, nl = int(info["n_items"]), int(info["n_long_items"])
    desc = np.asarray(item_desc).reshape(-1, 4).astype(np.int64)
    assert desc.shape[0] == n + 2
    p8, p4, f0, f8, f4 = (int(x) for x in desc[n:].ravel()[:5])
    assert nl <= p8 <= p4 <= f0 <= f8 <= f4 <= n
    long_full = int(desc[:nl, 3].sum())
    b = info["bucket_class0"]
    return dict(segments=[nl, p8 - nl, p4 - p8, f0 - p4, f8 - f0, f4 - f8, n - f4], long_partial=nl - long_full,
                long_full=long_full, widths=[int(b[k + 1] - b[k]) for k in range(KMAX + 1)],
                deep_loci=int(info["n_deep_loci"]), max_width=int(info["max_pairs_per_class"]))


def _host_arrays(packed):
    return packed.arrays if packed.arrays else packed.to_host()


def assert_layout_covers(packed) -> dict:
    """Every column-pass segment, every row-pass width bucket, deep loci and long items of both kinds are present.  With
    one haplotype every mask is full, so a split locus has no partial part: there the short full segments and the long
    partial items cannot exist and are required to be empty instead."""
    s = layout_summary(packed.info, _host_arrays(packed)["item_desc"])
    seg = s["segments"]
    missing = [SEGMENTS[k] for k in range(7 if packed.H > 1 else 4) if seg[k] == 0]
    assert not missing, f"column-pass segments without work: {missing} ({s})"
    if packed.H > 1:
        assert s["long_partial"] > 0 and s["long_full"] > 0, s
    else:
        assert seg[4:] == [0, 0, 0] and s["long_partial"] == 0 and s["long_full"] > 0, s
    assert all(w > 0 for w in s["widths"]), f"empty row-pass width bucket: {s['widths']}"
    assert s["deep_loci"] > 0 and s["max_width"] > 32, s
    return s


def locus_kinds(packed) -> list:
    """Per locus: its entry count and the column-pass segments of its items (failure reports)."""
    arrays = _host_arrays(packed)
    info = packed.info
    n = int(info["n_items"])
    desc = arrays["item_desc"].reshape(-1, 4).astype(np.int64)
    seg_start = [0, int(info["n_long_items"])] + [int(x) for x in desc[n:].ravel()[:5]]
    seg_of_pos = np.searchsorted(np.array(seg_start), np.arange(n), side="right") - 1
    seg_of_item = np.empty(n, dtype=np.int64)
    seg_of_item[desc[:n, 2]] = seg_of_pos
    words = np.zeros(n, dtype=np.int64)
    words[desc[:n, 2]] = desc[:n, 1] - desc[:n, 0]
    ld = arrays["locus_desc"].reshape(-1, 4).astype(np.int64)
    out = [""] * packed.T
    for t, i0, i1, _ in ld:
        kinds = sorted({SEGMENTS[k] for k in seg_of_item[i0:i1]})
        out[t] = f"{i1 - i0} items, {int(words[i0:i1].sum())} padded entry words, segments: {', '.join(kinds) or 'none'}"
    return out
