"""Time EMfactory.posterior_probability() and its device part (gbrs_em_posterior) at the benchmark shape.

    python tools/bench_posterior.py [--calls 20] [--warmup 3] [--e2e 3] [--out FILE]

Workload: C2 of bench.py (synth.generate(T=80000, N=5M, H=8), about 63 M stored entries).  Per model 4, 3, 2, 1, after
a few updates of that model:
  * device_ms: CUDA events around each gbrs_em_posterior call (the output pattern resident on the device), median over
    `--calls` calls after `--warmup`;
  * bytes: what the call moves, from the shapes (row pass: pair words, unit counts, weights out, subset tables; gather:
    per entry its class index, its class position, its weight and its value out, plus for models 1-3 the row pointers and
    the pair words a linear walk to the entry's pair reads, half a row on average); GB/s = bytes / device time;
  * e2e_s: wall time of posterior_probability() to a host AlignmentPropertyMatrix (output pattern up, values down, host
    CSC assembly), median of `--e2e` calls after one warm-up.
Prints one JSON document (also written to --out) with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = (x.strip() for x in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001 - report what is known
        import torch

        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def bytes_moved(info, T, nnz, index_bytes, model, classes_e, classes_k):
    """algorithmic bytes of one gbrs_em_posterior call"""
    Np, Pp, Rn = info["n_classes"], info["n_pairs"], info["n_runs"]
    widx = {4: Np, 3: Rn, 2: Pp, 1: 8 * Rn}[model]
    init = 4 * classes_e.size + 8 * Np + 4 * Np + 4 * Np  # class_pos fill, unit counts, class_id in, class_pos out
    tables = 64 * T + 256 * T + (0 if model == 4 else 64 * T + 64 * info["n_gene_ids"] + 8 * T)
    row = 4 * Pp + 8 * Np + 8 * widx + (0 if model == 4 else 8 * Np + 4 * Pp)
    gather = nnz * (index_bytes + 4 + 8 + 8) + 8 * 8 * (T + 1) + 64 * T
    if model != 4:  # row pointers + the pair words (and gene ids for models 1, 3) of a walk to the entry's pair
        per_word = 4 if model == 2 else 8
        gather += float(np.sum(classes_e * (8 + per_word * (classes_k + 1) / 2.0)))
    return {"init": int(init), "tables": int(tables), "row_pass": int(row), "gather": int(gather),
            "total": int(init + tables + row + gather)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--e2e", type=int, default=3)
    ap.add_argument("--updates", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    from gbrs_b200 import _lib, synth
    from gbrs_b200.emfactory import EMfactory, posterior_pattern

    if not torch.cuda.is_available():
        raise SystemExit("bench_posterior.py: no CUDA device")
    torch.cuda.set_device(0)
    t0 = time.perf_counter()
    d = synth.generate(T=80_000, N=5_000_000, H=8)
    apm = synth.to_apm(d)
    t_gen = time.perf_counter() - t0
    em = EMfactory(apm, device="cuda:0")
    em.target_lengths = synth.effective_lengths(d)
    em.prepare()
    pat = em._pattern
    info, T, H, N = pat.info, d.T, d.H, d.N
    pattern = posterior_pattern(apm)
    nnz = int(sum(a[1].size for a in pattern))
    index_bytes = pattern[0][1].dtype.itemsize
    classes_e = np.bincount(np.concatenate([a[1] for a in pattern]), minlength=N).astype(np.float64)
    classes_k = np.bincount(np.asarray(d.pair_class), minlength=N).astype(np.float64)
    keep = classes_e > 0
    classes_e, classes_k = classes_e[keep], classes_k[keep]
    d_ptr = [torch.from_numpy(np.ascontiguousarray(a[0], dtype=np.int64)).cuda() for a in pattern]
    d_idx = [torch.from_numpy(np.ascontiguousarray(a[1])).cuda() for a in pattern]
    vals = [torch.empty(max(a[1].size, 1), dtype=torch.float64, device="cuda:0") for a in pattern]
    P = C.c_void_p * H
    ptrs = (P(*[t.data_ptr() for t in d_ptr]), P(*[t.data_ptr() for t in d_idx]), P(*[t.data_ptr() for t in vals]))
    results = {}
    for model in (4, 3, 2, 1):
        if model != 4:
            pat.ensure_full(model)
        em.reset()
        em.run(model=model, tol=0.0, max_iters=args.updates, verbose=False)
        em.posterior_probability()  # uploads what the posterior reads (class_id, row pointers)
        nbytes = C.c_int64()
        _lib.check(pat.lib.gbrs_em_posterior_scratch_bytes(C.byref(pat.desc), model, N, C.byref(nbytes)))
        scratch = torch.empty(int(nbytes.value), dtype=torch.uint8, device="cuda:0")

        def call():
            _lib.check(pat.lib.gbrs_em_posterior(C.byref(pat.desc), model, C.c_void_p(pat.post_theta.data_ptr()),
                                                 C.c_void_p(pat.dev["class_id"].data_ptr()), N, ptrs[0], ptrs[1],
                                                 index_bytes, ptrs[2], C.c_void_p(scratch.data_ptr()), int(nbytes.value),
                                                 pat.stream()))

        for _ in range(args.warmup):
            call()
        ms = []
        for _ in range(args.calls):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            call()
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        em.posterior_probability()
        e2e = []
        for _ in range(args.e2e):
            t0 = time.perf_counter()
            post = em.posterior_probability()
            e2e.append(time.perf_counter() - t0)
        assert post.data[0].nnz == pattern[0][1].size
        b = bytes_moved(info, T, nnz, index_bytes, model, classes_e, classes_k)
        med = float(np.median(ms))
        results[str(model)] = {"device_ms_median": med, "device_ms_min": float(np.min(ms)), "device_ms_max": float(np.max(ms)),
                               "calls": args.calls, "bytes": b, "gb_per_s": b["total"] / (med * 1e-3) / 1e9,
                               "e2e_s_median": float(np.median(e2e)), "e2e_s_all": [round(x, 4) for x in e2e],
                               "values_d2h_bytes": 8 * nnz}
        print(f"model {model}: device {med:.3f} ms ({b['total'] / 1e9:.2f} GB, {results[str(model)]['gb_per_s']:.0f} GB/s), "
              f"end to end {np.median(e2e):.3f} s", file=sys.stderr, flush=True)
        del scratch
    out = {"tool": "tools/bench_posterior.py", "workload": "c2", "T": T, "H": H, "N": N, "nnz": nnz,
           "n_classes": info["n_classes"], "n_pairs": info["n_pairs"], "n_runs": info["n_runs"],
           "updates_before": args.updates, "generate_s": t_gen, "card": card(), "models": results}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
