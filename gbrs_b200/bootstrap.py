"""Bootstrap replicates of the allele-specific estimates (`EMfactory.bootstrap`, DESIGN.md section 7.2).

A replicate resamples the M reads of the input with replacement -- on the device, by a counter-based generator, so that
replicate r of seed s depends on (s, r, counts) alone -- and reruns prepare() + run() on the resampled class counts.
The spread of the replicates' estimates is the measure of how far the point estimate can be trusted.
"""
from __future__ import annotations

import numpy as np

GUIDE_BITS_MAX = 24  # kBootGuideBitsMax of the resampler (gbrs_b200/csrc/em_kernels.cu)


def replicate_indices(replicates) -> np.ndarray:
    """`replicates`: an int n (= range(n)) or a sequence of replicate indices -> int64 array; every index must fit uint32."""
    if isinstance(replicates, (int, np.integer)):
        if not 0 <= replicates <= 1 << 32:
            raise ValueError("the number of replicates must be in [0, 2^32] (replicate indices are uint32)")
        return np.arange(int(replicates), dtype=np.int64)
    idx = np.asarray(list(replicates))
    if idx.size and (idx.dtype.kind not in "iu" or idx.min() < 0 or idx.max() > 0xFFFFFFFF):
        raise ValueError("replicate indices must be integers in [0, 2^32)")
    return idx.astype(np.int64).reshape(-1)


def read_counts_of(count, n_classes: int) -> np.ndarray:
    """Input class counts (None = all ones) as int64, refused unless they are non-negative integers summing to at most
    2^53 (each replicate count is then exact in a double)."""
    if count is None:
        return np.ones(n_classes, dtype=np.int64)
    c = np.asarray(count, dtype=np.float64)
    if c.shape != (n_classes,):
        raise ValueError("count vector length does not match the number of classes")
    if not np.all(np.isfinite(c)) or np.any(c < 0) or np.any(c != np.floor(c)):
        raise ValueError("bootstrap needs non-negative integer class counts")
    # the int64 sum is exact unless the (rounded) double sum is already far past the limit
    if c.size and (float(np.sum(c)) > 2.0 ** 62 or int(c.astype(np.int64).sum()) > 2 ** 53):
        raise ValueError("bootstrap needs at most 2^53 reads in total")
    return c.astype(np.int64)


def resampler_bytes(N: int, M: int, n_classes: int) -> dict:
    """Bytes the resampler moves per replicate, from the shapes: the histogram is zeroed and written (one 8-byte atomic
    per draw), every draw reads two guide entries and the prefix entries of its search (about log2 of the guide spacing
    plus one, counted as 2), the scatter reads class_id and the histogram and writes one double per packed class.  The
    guide is built once per call: 4 (G + 1) bytes written, log2(N) prefix reads per entry."""
    bits = 0
    while bits < GUIDE_BITS_MAX and (1 << bits) < N:
        bits += 1
    G = 1 << bits
    per_replicate = 8 * N + M * (8 + 2 * 4 + 2 * 8) + n_classes * (4 + 8 + 8)
    guide = 4 * (G + 1) + 8 * G * max(bits, 1)
    return {"per_replicate": int(per_replicate), "guide_once": int(guide), "guide_entries": int(G + 1)}


class BootstrapResult:
    """Estimates of B bootstrap replicates (input locus / haplotype order).
      replicates            int64 [B]  the replicate indices
      seed, model           the generator seed and the EM model
      total_reads           M, the number of reads every replicate draws
      num_iters             int64 [B]  EM updates each replicate ran
      allelic_expression    float64 [B, H, T]  theta of each replicate (what `EMfactory.allelic_expression` holds)
      expected_read_counts  float64 [B, H, T]  (what `EMfactory.expected_read_counts()` returns)
    `tpm()` / `read_counts()` are the values the report tables hold (`report_depths` / `report_read_counts`)."""

    def __init__(self, replicates, seed, model, total_reads, num_iters, allelic_expression, expected_read_counts,
                 grp_conv_mat=None, lname=None, hname=None, gname=None):
        self.replicates = np.asarray(replicates, dtype=np.int64)
        self.seed, self.model, self.total_reads = int(seed), int(model), int(total_reads)
        self.num_iters = np.asarray(num_iters, dtype=np.int64)
        self.allelic_expression = allelic_expression
        self.expected_read_counts = expected_read_counts
        self.grp_conv_mat = grp_conv_mat
        self.lname, self.hname, self.gname = lname, hname, gname

    def __len__(self):
        return int(self.replicates.shape[0])

    def _group(self, x):
        if self.grp_conv_mat is None:
            raise RuntimeError("Group information matrix is missing.")
        return np.stack([np.asarray(x[b] * self.grp_conv_mat) for b in range(len(self))]) if len(self) else \
            np.zeros((0, x.shape[1], self.grp_conv_mat.shape[1]))

    def tpm(self, grp_wise: bool = False) -> np.ndarray:
        """[B, H, T] (or [B, H, G]) TPM per replicate, scaled as `report_depths(tpm=True)` scales."""
        depths = self._group(self.allelic_expression) if grp_wise else self.allelic_expression.copy()
        for b in range(len(self)):
            depths[b] *= 1000000.0 / depths[b].sum()
        return depths

    def read_counts(self, grp_wise: bool = False) -> np.ndarray:
        """[B, H, T] (or [B, H, G]) expected read counts per replicate, as `report_read_counts` reports them."""
        return self._group(self.expected_read_counts) if grp_wise else self.expected_read_counts.copy()

    def arrays(self) -> dict:
        out = {"replicate": self.replicates, "seed": np.uint64(self.seed), "model": np.int64(self.model),
               "total_reads": np.int64(self.total_reads), "num_iters": self.num_iters,
               "lname": np.asarray(self.lname, dtype=str), "hname": np.asarray(self.hname, dtype=str),
               "isoforms_tpm": self.tpm(), "isoforms_expected_read_counts": self.read_counts()}
        if self.grp_conv_mat is not None:
            out.update(gname=np.asarray(self.gname, dtype=str), genes_tpm=self.tpm(grp_wise=True),
                       genes_expected_read_counts=self.read_counts(grp_wise=True))
        return out

    def save(self, path) -> None:
        """Write the replicates as an npz: replicate, seed, model, total_reads, num_iters, lname, hname, isoforms_tpm,
        isoforms_expected_read_counts and, with groups, gname, genes_tpm, genes_expected_read_counts."""
        with open(path, "wb") as fh:  # np.savez would append ".npz" to a name without it
            np.savez(fh, **self.arrays())
