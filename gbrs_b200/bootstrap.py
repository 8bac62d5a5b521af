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


# ---------------------------------------------------------------------------------------------------------------------
# summaries (EMfactory.bootstrap_summary, DESIGN.md section 7.3)
# ---------------------------------------------------------------------------------------------------------------------
SUMMARY_MAX_REPLICATES = 16384  # GBRS_BOOT_SUMMARY_MAX_B of gbrs_boot_summarize: a column is sorted in shared memory
LEVELS = ("isoforms", "genes")
QUANTITIES = ("tpm", "expected_read_counts", "allelic_share")


def interval_quantiles(interval: float) -> np.ndarray:
    """The quantiles of a central interval: (1 - interval) / 2, 0.5, 1 - (1 - interval) / 2."""
    lo = (1.0 - float(interval)) / 2.0
    return np.array([lo, 0.5, 1.0 - lo])


def summarize_on_device(lib, stream, theta_all, acc_all, H: int, interval: float, genes=None) -> dict:
    """gbrs_boot_derive + gbrs_boot_summarize for every (level, quantity), one at a time through one [B][E] buffer.
    `theta_all` / `acc_all`: [B][T][8] device tensors; `genes`: (gene_ptr, gene_loci, number of real genes) or None;
    `stream`: a stream of the tensors' device, on which the kernels run (that device is made current for the calls).
    -> {(level, quantity): {"mean", "sd": [C, L], "q": [3, C, L], "n": int64 [L] (shares only)}} on the host, C = H + 1
    (the last row is the total column) or H for shares."""
    import ctypes as C

    import torch

    from . import _lib

    B, T = int(theta_all.shape[0]), int(theta_all.shape[1])
    q = interval_quantiles(interval)
    dev = theta_all.device
    # the launches go to the current device: make it the replicates' one (the factory's device need not be current)
    with torch.cuda.device(dev):
        values = torch.empty(B * T * (H + 1), dtype=torch.float64, device=dev)
        out = {}
        for level in LEVELS:
            if level == "genes" and genes is None:
                continue
            gp, gl, L = (None, None, T) if level == "isoforms" else (C.c_void_p(genes[0].data_ptr()),
                                                                    C.c_void_p(genes[1].data_ptr()), int(genes[2]))
            for quantity, code in zip(QUANTITIES, (_lib.BOOT_TPM, _lib.BOOT_COUNTS, _lib.BOOT_SHARE)):
                rows = H if code == _lib.BOOT_SHARE else H + 1
                E = rows * L
                src = acc_all if code == _lib.BOOT_COUNTS else theta_all
                mean = torch.empty(E, dtype=torch.float64, device=dev)
                sd = torch.empty(E, dtype=torch.float64, device=dev)
                qo = torch.empty((len(q), E), dtype=torch.float64, device=dev)
                n = torch.empty(E, dtype=torch.int32, device=dev)
                _lib.check(lib.gbrs_boot_derive(C.c_void_p(src.data_ptr()), B, T, H, code, gp, gl, L if gp else 0,
                                                C.c_void_p(values.data_ptr()), stream))
                _lib.check(lib.gbrs_boot_summarize(C.c_void_p(values.data_ptr()), B, E, q.ctypes.data, len(q),
                                                   C.c_void_p(mean.data_ptr()), C.c_void_p(sd.data_ptr()),
                                                   C.c_void_p(qo.data_ptr()), C.c_void_p(n.data_ptr()), stream))
                st = {"mean": mean.cpu().numpy().reshape(rows, L), "sd": sd.cpu().numpy().reshape(rows, L),
                      "q": qo.cpu().numpy().reshape(len(q), rows, L)}
                if code == _lib.BOOT_SHARE:  # whether a share is defined depends on the locus alone
                    st["n"] = n.cpu().numpy().reshape(rows, L)[0].astype(np.int64)
                out[(level, quantity)] = st
    return out


def _label(x: float) -> str:
    return f"{x:.6g}"


class BootstrapSummary:
    """Statistics of B bootstrap replicates per element, over the replicates in the order given.
      replicates, seed, model, total_reads, num_iters, interval, quantiles   as in BootstrapResult; quantiles =
                                                                          interval_quantiles(interval)
      stats[(level, quantity)]   level in LEVELS (genes only with groups), quantity in QUANTITIES:
          "mean", "sd"  float64 [C, L]; "q" float64 [3, C, L] (quantiles in order); "n" int64 [L] for allelic_share
          (replicates in which the locus' share is defined).  Rows: the haplotypes, then for tpm / expected_read_counts the
          total column.
      result   the BootstrapResult of the same replicates (keep_replicates=True), else None.
    `write(outbase)` writes one table per (level, quantity)."""

    def __init__(self, replicates, seed, model, total_reads, num_iters, interval, stats, lname=None, hname=None,
                 gname=None, result=None):
        self.replicates = np.asarray(replicates, dtype=np.int64)
        self.seed, self.model, self.total_reads = int(seed), int(model), int(total_reads)
        self.num_iters = np.asarray(num_iters, dtype=np.int64)
        self.interval = float(interval)
        self.quantiles = interval_quantiles(interval)
        self.stats = stats
        self.lname, self.hname, self.gname = lname, hname, gname
        self.result = result

    def __len__(self):
        return int(self.replicates.shape[0])

    def header(self, quantity: str, notes: bool = False) -> str:
        cols = list(self.hname) + ([] if quantity == "allelic_share" else ["total"])
        stats = ["mean", "sd"] + ["q" + _label(x) for x in self.quantiles]
        head = ["locus"] + [f"{c}.{s}" for c in cols for s in stats]
        if quantity == "allelic_share":
            head.append("n")
        if notes:
            head.append("notes")
        return "\t".join(head)

    def columns(self, level: str, quantity: str) -> np.ndarray:
        """[columns][loci] of the table: per haplotype (and total) mean, sd and the quantiles; n for shares."""
        st = self.stats[(level, quantity)]
        cols = []
        for c in range(st["mean"].shape[0]):
            cols += [st["mean"][c], st["sd"][c]] + [st["q"][j][c] for j in range(st["q"].shape[0])]
        if "n" in st:
            cols.append(st["n"].astype(np.float64))
        return np.vstack(cols)

    def write(self, outbase, notes_t=None, notes_g=None) -> list:
        """{outbase}.bootstrap.{isoforms,genes}.{tpm,expected_read_counts,allelic_share}.summary, one row per locus in
        input order, numbers formatted as the point reports format them.  Returns the paths written."""
        from . import utils

        paths = []
        for level, names, notes in (("isoforms", self.lname, notes_t), ("genes", self.gname, notes_g)):
            for quantity in QUANTITIES:
                if (level, quantity) not in self.stats:
                    continue
                path = f"{outbase}.bootstrap.{level}.{quantity}.summary"
                with open(path, "w") as fh:
                    fh.write(self.header(quantity, notes is not None) + "\n")
                    utils.write_table_rows(fh, names, self.columns(level, quantity), notes=notes)
                paths.append(path)
        return paths
