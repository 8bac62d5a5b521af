"""Time EMfactory.bootstrap() and its parts at the benchmark shape.

    python tools/bench_bootstrap.py [--replicates 100] [--model 4] [--out FILE]

Workload: C2 of bench.py (synth.generate(T=80000, N=5M, H=8), M = 24,996,197 reads), model 4, tol 1e-4.
  * resample_ms: CUDA events around gbrs_boot_resample (zero the histogram, draw and count M reads, scatter into the
    packed counts), median over the replicates; bytes from the shapes (gbrs_b200.bootstrap.resampler_bytes);
  * em_ms / em_iters: CUDA events around prepare + run of each replicate on the replicate state, median, and the
    iteration counts;
  * bootstrap_s: wall time of one bootstrap(B) call (prefix upload, guide, B replicates, results to the host), against
    B times the wall time of one run() of the factory (run_s, median of 3).
Prints one JSON document (also written to --out) with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.bench_posterior import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--replicates", type=int, default=100)
    ap.add_argument("--model", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    from gbrs_b200 import _lib, synth
    from gbrs_b200.bootstrap import read_counts_of, resampler_bytes
    from gbrs_b200.emfactory import EMfactory

    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    d = synth.generate(T=80_000, N=5_000_000, H=8)
    em = EMfactory(synth.to_apm(d))
    em.target_lengths = synth.effective_lengths(d)
    em.prepare()
    B, model = args.replicates, args.model
    run_s = []
    for _ in range(3):
        em.prepare()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        em.run(model=model, tol=1e-4, verbose=False)
        torch.cuda.synchronize()
        run_s.append(time.perf_counter() - t0)
    point_iters = em.num_iters
    em.bootstrap([0], model=model)  # warm-up: replicate state, graph capture
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = em.bootstrap(B, model=model)
    torch.cuda.synchronize()
    boot_s = time.perf_counter() - t0

    # the parts, with events, on a replicate state of the same factory
    pat = em._pattern
    st = pat.replicate_state(model)
    lib = pat.lib
    counts = read_counts_of(d.count, d.N)
    M, N, n_cls = int(counts.sum()), d.N, int(pat.info["n_classes"])
    prefix = torch.from_numpy(np.cumsum(counts)).cuda()
    nbytes = C.c_int64()
    _lib.check(lib.gbrs_boot_scratch_bytes(N, C.byref(nbytes)))
    scratch = torch.empty(int(nbytes.value), dtype=torch.uint8, device="cuda")
    s = pat.stream()
    _lib.check(lib.gbrs_boot_guide(prefix.data_ptr(), N, M, scratch.data_ptr(), int(nbytes.value), s))
    res_ms, em_ms, iters = [], [], []
    errs = np.zeros(999)
    for r in range(min(B, 20)):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        _lib.check(lib.gbrs_boot_resample(prefix.data_ptr(), N, M, 0, r, pat.dev["class_id"].data_ptr(), n_cls,
                                          scratch.data_ptr(), int(nbytes.value), st.count.data_ptr(), s))
        e[1].record()
        _lib.check(lib.gbrs_em_prepare_local(C.byref(st.desc), s))
        _lib.check(lib.gbrs_em_prepare_finish(C.byref(st.desc), 0.0, s))
        n = C.c_int32(0)
        _lib.check(lib.gbrs_em_run_cb(C.byref(st.desc), model, 1e-4, 999, 4, s, C.byref(n), errs.ctypes.data, None, None))
        e[2].record()
        torch.cuda.synchronize()
        res_ms.append(e[0].elapsed_time(e[1]))
        em_ms.append(e[1].elapsed_time(e[2]))
        iters.append(int(n.value))
    nb = resampler_bytes(N, M, n_cls)
    out = {
        "workload": "C2 (T=80000, N=5M, H=8), model %d" % model, "total_reads": M, "classes": N, "packed_classes": n_cls,
        "replicates": B, "card": card(),
        "resample_ms_median": float(np.median(res_ms)), "resample_ms": res_ms,
        "resample_bytes_per_replicate": nb["per_replicate"], "guide_bytes_once": nb["guide_once"],
        "resample_GBps": nb["per_replicate"] / (np.median(res_ms) * 1e-3) / 1e9,
        "em_ms_median": float(np.median(em_ms)), "em_iters": iters, "em_ms": em_ms,
        "em_us_per_update": float(np.median(np.array(em_ms) / np.array(iters)) * 1e3),
        "bootstrap_s": boot_s, "bootstrap_iters_mean": float(res.num_iters.mean()),
        "run_s_median": float(np.median(run_s)), "run_iters": point_iters,
        "B_times_run_s": B * float(np.median(run_s)),
    }
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
