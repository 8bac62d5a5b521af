"""TEST INFRASTRUCTURE ONLY -- numpy reference of the bootstrap resampler (gbrs_boot_resample, include/gbrs_em.h):
Philox4x32-10 in uint64 arithmetic, the read index as the high half of a 128-bit product formed from 32-bit limbs, the
class by `np.searchsorted(P, k, side="right")` and the counts by `np.bincount`.  Also the matrix a replicate is the
ordinary EM of: the input with the resampled counts and the classes drawn 0 times removed."""
from __future__ import annotations

import numpy as np

MASK32 = np.uint64(0xFFFFFFFF)
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)

# Random123 known-answer vectors of philox4x32_10: (counter; key) -> output
KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


def philox4x32_10(ctr, key):
    """ctr: 4 arrays (or scalars) of 32-bit values, key: 2 values -> 4 uint64 arrays of 32-bit words."""
    c = [np.asarray(x, dtype=np.uint64) & MASK32 for x in ctr]
    k0, k1 = np.uint64(key[0]) & MASK32, np.uint64(key[1]) & MASK32
    with np.errstate(over="ignore"):
        for i in range(10):
            p0, p1 = _M0 * c[0], _M1 * c[2]  # 32 x 32 -> 64 bits: exact in uint64
            c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & MASK32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & MASK32]
            k0, k1 = (k0 + _W0) & MASK32, (k1 + _W1) & MASK32
    return c


def check_kat():
    for ctr, key, want in KAT:
        got = tuple(int(x) for x in philox4x32_10(ctr, key))
        assert got == want, ([hex(x) for x in got], [hex(x) for x in want])


check_kat()


def draws(M: int, seed: int, replicate: int) -> np.ndarray:
    """The M uint64 draws of replicate `replicate` of `seed`."""
    n_pairs = (M + 1) // 2
    j = np.arange(n_pairs, dtype=np.uint64)
    x = philox4x32_10((j & MASK32, j >> np.uint64(32), np.full(n_pairs, replicate, np.uint64), np.zeros(n_pairs, np.uint64)),
                      (seed & 0xFFFFFFFF, seed >> 32))
    u = np.empty(2 * n_pairs, dtype=np.uint64)
    u[0::2] = x[0] | (x[1] << np.uint64(32))
    u[1::2] = x[2] | (x[3] << np.uint64(32))
    return u[:M]


def mul64hi(u: np.ndarray, M: int) -> np.ndarray:
    """floor(u * M / 2^64) for uint64 u, from 32-bit limbs."""
    u = np.asarray(u, dtype=np.uint64)
    s32 = np.uint64(32)
    ul, uh = u & MASK32, u >> s32
    ml, mh = np.uint64(M & 0xFFFFFFFF), np.uint64(M >> 32)
    ll, lh, hl, hh = ul * ml, ul * mh, uh * ml, uh * mh
    mid = (ll >> s32) + (lh & MASK32) + (hl & MASK32)
    return hh + (lh >> s32) + (hl >> s32) + (mid >> s32)


def counts_of(count, N: int) -> np.ndarray:
    return np.ones(N, dtype=np.int64) if count is None else np.asarray(count, dtype=np.float64).astype(np.int64)


def resample(count, seed: int, replicate: int, N: int | None = None) -> np.ndarray:
    """Replicate counts (int64 [N], input class order); `count` None = all ones (then N is needed)."""
    c = counts_of(count, N if count is None else len(count))
    P = np.cumsum(c)
    M = int(P[-1])
    k = mul64hi(draws(M, seed, replicate), M).astype(np.int64)
    return np.bincount(np.searchsorted(P, k, side="right"), minlength=c.shape[0]).astype(np.int64)


def compact_synth(d, counts):
    """The SynthData a replicate is the ordinary EM of: the resampled counts, the classes drawn 0 times removed (the
    survivors keep their order), the same loci, lengths, genes and names."""
    import dataclasses

    counts = np.asarray(counts)
    keep = counts > 0
    new_id = np.cumsum(keep) - 1
    sel = keep[np.asarray(d.pair_class)]
    return dataclasses.replace(d, N=int(keep.sum()), pair_class=new_id[np.asarray(d.pair_class)[sel]].astype(np.int64),
                               pair_locus=np.asarray(d.pair_locus)[sel], pair_mask=np.asarray(d.pair_mask)[sel],
                               count=counts[keep].astype(np.float64))


def with_lonely_locus(d):
    """`d` plus one locus (its own gene) that a single new class of count 1 alone aligns to, on every haplotype."""
    import dataclasses

    T, N = d.T, d.N
    out = dataclasses.replace(
        d, T=T + 1, N=N + 1, pair_class=np.append(d.pair_class, N), pair_locus=np.append(d.pair_locus, T),
        pair_mask=np.append(d.pair_mask, np.uint8((1 << d.H) - 1)), count=np.append(d.count, 1.0),
        gene_of=np.append(d.gene_of, int(np.max(d.gene_of)) + 1), lengths=np.vstack([d.lengths, d.lengths[:1]]))
    out.lname = list(d.lname) + [f"lonely{T}"]
    out.gname = list(d.gname) + [f"lonelygene{T}"]
    return out


def seed_dropping(count, cls, replicate=0, start=0):
    """The first seed >= start whose replicate `replicate` draws class `cls` 0 times."""
    s = start
    while resample(count, s, replicate)[cls] != 0:
        s += 1
    return s
