"""Time the bootstrap summaries (EMfactory.bootstrap_summary) at the benchmark shape.

    python tools/bench_bootstrap_summary.py [--replicates 100] [--out FILE]

Workload: C2 of bench.py (synth.generate(T=80000, N=5M, H=8), with its genes), model 4, tol 1e-4.
  * per (level, quantity): CUDA events around gbrs_boot_derive and gbrs_boot_summarize on the replicates of one
    bootstrap call (median of 5), bytes from the shapes (derive: its [B][T][8] reads, gene CSR, [B][E] write and, for
    TPM, two more passes over the row; summarize: one read of [B][E] and the outputs), and GB/s;
  * summary_s: wall time of bootstrap_summary(B) against host_s: bootstrap(B) followed by the same statistics in numpy
    on the host (tpm() / read_counts() / shares, mean, sd, nanquantile).
Prints one JSON document (also written to --out) with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.bench_posterior import card  # noqa: E402


def derive_bytes(B, T, H, L, quantity, nnz_genes=0):
    rows = H if quantity == "allelic_share" else H + 1
    read = B * (T if nnz_genes == 0 else nnz_genes) * 64 + (4 * (L + 1) + 4 * nnz_genes if nnz_genes else 0)
    write = B * rows * L * 8
    if quantity == "tpm":  # the row sum pass and the scaling pass
        read += B * H * L * 8 * 2
        write += B * rows * L * 8
    return read + write


def summarize_bytes(B, E, nq=3):
    return B * E * 8 + E * (8 * (2 + nq) + 4)


def host_summary(res, q):
    """what a user of bootstrap() had to do: the level values on the host, then the statistics in numpy"""
    out = {}
    for grp in (False, True):
        for name, x in (("tpm", res.tpm(grp)), ("expected_read_counts", res.read_counts(grp))):
            x = np.concatenate([x, x.sum(axis=1, keepdims=True)], axis=1)
            out[(grp, name)] = (x.mean(0), x.std(0, ddof=1), np.quantile(x, q, axis=0))
        th = res._group(res.allelic_expression) if grp else res.allelic_expression
        with np.errstate(all="ignore"):
            sh = th / th.sum(axis=1, keepdims=True)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            out[(grp, "allelic_share")] = (np.nanmean(sh, 0), np.nanstd(sh, 0, ddof=1), np.nanquantile(sh, q, axis=0),
                                           (~np.isnan(sh)).sum(0))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--replicates", type=int, default=100, help="B (1000 for the large case)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    from gbrs_b200 import _lib, synth
    from gbrs_b200.bootstrap import LEVELS, QUANTITIES, interval_quantiles
    from gbrs_b200.emfactory import EMfactory

    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    d = synth.generate(T=80_000, N=5_000_000, H=8)
    em = EMfactory(synth.to_apm(d))
    em.target_lengths = synth.effective_lengths(d)
    em.prepare()
    B, H, T = args.replicates, d.H, d.T
    q = interval_quantiles(0.95)
    em.bootstrap_summary([0, 1])  # warm-up: replicate state, graph capture, module load
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    summary = em.bootstrap_summary(B)
    torch.cuda.synchronize()
    summary_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    res = em.bootstrap(B)
    torch.cuda.synchronize()
    boot_s = time.perf_counter() - t0
    host_summary(res, q)
    host_s = time.perf_counter() - t0

    # the kernels, with events, on the replicates of one call
    pat = em._pattern
    p = em.probability
    reps, counts = em._check_bootstrap(B, 4, 0, 999)
    _, _, theta_all, acc_all = em._replicate_loop(reps, counts, 4, 0, 0.0, 1e-4, 999)
    lib, s = pat.lib, pat.stream()
    G = int(p.num_groups)
    nnz_genes = int(pat.dev["gene_ptr"][G].item())  # loci in real genes
    values = torch.empty(B * T * (H + 1), dtype=torch.float64, device="cuda")
    parts = []
    for level in LEVELS:
        gp, gl, L = (None, None, T) if level == "isoforms" else (pat.dev["gene_ptr"].data_ptr(),
                                                                pat.dev["gene_loci"].data_ptr(), G)
        for quantity, code in zip(QUANTITIES, (_lib.BOOT_TPM, _lib.BOOT_COUNTS, _lib.BOOT_SHARE)):
            rows = H if code == _lib.BOOT_SHARE else H + 1
            E = rows * L
            src = acc_all if code == _lib.BOOT_COUNTS else theta_all
            mean, sd = (torch.empty(E, dtype=torch.float64, device="cuda") for _ in range(2))
            qo, n = torch.empty((3, E), dtype=torch.float64, device="cuda"), torch.empty(E, dtype=torch.int32, device="cuda")
            der, summ = [], []
            for _ in range(6):
                e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                e[0].record()
                _lib.check(lib.gbrs_boot_derive(src.data_ptr(), B, T, H, code, gp, gl, L if gp else 0,
                                                values.data_ptr(), s))
                e[1].record()
                _lib.check(lib.gbrs_boot_summarize(values.data_ptr(), B, E, q.ctypes.data, 3, mean.data_ptr(),
                                                   sd.data_ptr(), qo.data_ptr(), n.data_ptr(), s))
                e[2].record()
                torch.cuda.synchronize()
                der.append(e[0].elapsed_time(e[1]))
                summ.append(e[1].elapsed_time(e[2]))
            der, summ = der[1:], summ[1:]  # the first pass warms the caches and the launch path
            db = derive_bytes(B, T, H, L, quantity, nnz_genes if level == "genes" else 0)
            sb = summarize_bytes(B, E)
            dm, sm = float(np.median(der)), float(np.median(summ))
            parts.append({"level": level, "quantity": quantity, "elements": E, "derive_ms": dm, "derive_bytes": db,
                          "derive_GBps": db / (dm * 1e-3) / 1e9, "summarize_ms": sm, "summarize_bytes": sb,
                          "summarize_GBps": sb / (sm * 1e-3) / 1e9})
    out = {
        "workload": "C2 (T=80000, N=5M, H=8, %d genes), model 4, tol 1e-4" % G, "replicates": B, "card": card(),
        "mean_iters": float(summary.num_iters.mean()),
        "parts": parts,
        "derive_plus_summarize_ms_total": sum(x["derive_ms"] + x["summarize_ms"] for x in parts),
        "bootstrap_summary_s": summary_s, "bootstrap_s": boot_s, "bootstrap_then_host_summary_s": host_s,
    }
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
