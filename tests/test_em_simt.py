"""The EM library itself -- kernels, launchers and C ABI of gbrs_b200/csrc/em_kernels.cu -- executed on the CPU through
the host SIMT shim (tests/simt_em.py: the source is rewritten mechanically, `<<<>>>` launches become thread-per-CUDA-thread
launches, the CUDA runtime is a stand-in) against the golden vectors of the reference: identical iteration counts,
theta / counts / error trajectory as on the GPU.  A check of the kernel CODE on machines without a GPU -- not a product
path: the package cannot load this library, and the product's entry points fail without a CUDA device.

By default a subset of the golden cases runs (one OS thread per CUDA thread is slow: 4-30 s per case); set
GBRS_SIMT_ALL=1 for all of them."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from gbrs_b200 import synth
from gbrs_b200.quantify import hapmask_bytes
from oracle import em_oracle as eo
from tests import helpers as hp
from tests import layouts, simt_em
from tests import xref as xr

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ is needed to build the SIMT emulation")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = [n for n in hp.golden_em_cases() if n.startswith("em_small")]
DEFAULT = ["em_small_m4", "em_small_m4_diploid", "em_small_m4_maxit5", "em_small_m4_pc", "em_small_m1_diploid",
           "em_small_m2_h3", "em_small_m3_h1"]
CASES = SMALL if os.environ.get("GBRS_SIMT_ALL") else DEFAULT


def pattern_for(g, d, **kw):
    hm = hapmask_bytes(g["gtmask"]) if g["masked"] else None
    return simt_em.HostPattern(synth.to_apm(d), gene_of=eo.gene_index(d.T, d.groups()), hapmask=hm, **kw)


@pytest.mark.parametrize("name", CASES)
def test_emulated_library_matches_reference_golden(name):
    g = hp.load_golden(name)
    d = hp.synth_from_golden(g)
    pat = pattern_for(g, d)
    theta0 = pat.prepare(eo.effective_length_table(d.lengths), g["pseudocount"])
    assert hp.relerr(theta0, g["theta0"]) < 1e-12
    out = pat.run(g["model"], g["tol"], g["max_iters"])
    assert out["iters"] == g["iters"]
    np.testing.assert_allclose(out["errs"], g["errs"], rtol=1e-7, atol=1e-7)
    assert hp.relerr(out["theta"], g["theta"]) < 1e-12 and hp.relerr(out["counts"], g["counts"]) < 1e-12
    assert abs(out["counts"].sum() - g["counts"].sum()) < 1e-9 * g["counts"].sum()


def test_emulated_wide_classes_short_items_and_alignment_counts():
    """Classes wider than GBRS_KMAX (row-pointer paths), 8-entry work items (many items per locus, long items), one
    update of every model against the oracle, and the alignment-count kernel (bit-exact) at locus and gene level."""
    d = synth.generate(T=120, N=1500, H=8, sample_index=9, wide_frac=0.08)
    gene_of = eo.gene_index(d.T, d.groups())
    pat = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of, item_len=8)
    assert pat.info["max_pairs_per_class"] > 8 and pat.info["n_long_items"] > 0
    eff = eo.effective_length_table(d.lengths)
    theta = pat.prepare(eff)
    oapm = eo.apm_from_pairs(d.T, d.H, d.N, d.pair_class, d.pair_locus, d.pair_mask, d.count)
    assert hp.relerr(theta, eo.prepare(oapm, eff, 0.0)) < 1e-12
    for model in (4, 3, 2, 1):
        want = eo.sum_read(oapm, eo.e_step(oapm, theta, model, gene_of))
        out = pat.run(model, tol=0.0, max_iters=1)
        assert out["iters"] == 1 and hp.relerr(out["counts"], want) < 1e-12
        theta = out["theta"]
        assert hp.relerr(theta, want / eff) < 1e-12
    aln, uniq, lu = pat.alignment_counts()
    want = eo.alignment_counts(oapm)
    assert np.array_equal(aln, want["aln"]) and np.array_equal(uniq, want["uniq"]) and np.array_equal(lu, want["locus_uniq"])
    groups = d.groups()
    aln, uniq, lu = pat.alignment_counts(gene_level=True, n_real_genes=len(groups))
    want = eo.alignment_counts(eo.bundle(oapm, groups))
    assert np.array_equal(aln, want["aln"]) and np.array_equal(uniq, want["uniq"]) and np.array_equal(lu, want["locus_uniq"])


def test_emulated_column_pass_size_classes():
    """Every kind of column-pass work in one problem -- long items (a whole warp), short items of more than two quads
    (eight lanes), of two quads (two lanes, sixteen per warp) and of one quad (one lane, thirty-two per warp), partial and
    full -- at the default item length, on a constructed layout (tests/layouts.py) so that all seven slot segments hold
    items; the trailer of item_desc agrees with the descriptors; updates of models 4 and 3 against the extended-precision
    reference, element-wise."""
    d = layouts.make_layout(8, 64)
    gene_of = eo.gene_index(d.T, d.groups())
    pat = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of)
    layouts.assert_layout_covers(pat.packed)
    n_items, nl = pat.info["n_items"], pat.info["n_long_items"]
    desc = pat.packed.arrays["item_desc"].reshape(-1, 4).astype(np.int64)
    assert desc.shape[0] == n_items + 2
    tr, desc = desc[n_items:].ravel(), desc[:n_items]
    lens = desc[:, 1] - desc[:, 0]
    p8, p4, f0, f8, f4 = (int(x) for x in tr[:5])
    assert 0 < nl < p8 < p4 < f0 < f8 < f4 < n_items  # every segment holds items
    assert np.all(lens[:nl] > 64) and np.all(lens[nl:p8] > 8) and np.all(lens[f0:f8] > 8)
    assert np.all((lens[p8:p4] > 4) & (lens[p8:p4] <= 8)) and np.all(lens[p4:f0] <= 4)
    assert np.all((lens[f8:f4] > 4) & (lens[f8:f4] <= 8)) and np.all(lens[f4:] <= 4)
    assert not desc[nl:f0, 3].any() and desc[f0:, 3].all()
    x = xr.XRef(d, gene_of)
    eff = eo.effective_length_table(d.lengths)
    theta = pat.prepare(eff)
    where = layouts.locus_kinds(pat.packed)
    xr.assert_elementwise(theta, x.prepare(eff), x.rtol_prepare(), "theta0", where)
    for model in (4, 3, 4):
        counts, _ = x.update(theta, model, eff)
        out = pat.run(model, tol=0.0, max_iters=1)
        assert out["iters"] == 1
        xr.assert_elementwise(out["counts"], counts, x.rtol_update(model), f"model {model} counts", where)
        theta = out["theta"]


@pytest.mark.parametrize("H", range(1, 9))
def test_emulated_elementwise_on_constructed_layouts(H):
    """One update of every model from a haplotype-asymmetric theta scattered over e^+-40 (some in-support slots exactly 0),
    on a layout that reaches every column-pass segment, row-pass width and lane mask of H haplotypes: expected counts and
    theta element by element against the extended-precision reference, within the error bound of tests/xref.py.  A theta'
    flushed to zero, a lost or doubled entry, a swapped haplotype: any of them fails here whatever its magnitude."""
    import ctypes as C

    xr.require_longdouble()
    d = layouts.make_layout(H)
    gene_of = eo.gene_index(d.T, d.groups())
    pat = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of, item_len=16)
    layouts.assert_layout_covers(pat.packed)
    where = layouts.locus_kinds(pat.packed)
    x = xr.XRef(d, gene_of)
    eff = eo.effective_length_table(d.lengths)
    xr.assert_elementwise(pat.prepare(eff), x.prepare(eff), x.rtol_prepare(), "theta0", where)
    theta = xr.random_theta(x, seed=H)
    tb = np.zeros((d.T, 8))  # referenced until the end: the library reads it through a raw pointer
    tb[:, :H] = theta.T
    for model in (4, 3, 2, 1):
        pat.check(pat.lib.gbrs_em_set_theta(C.byref(pat.desc), tb.ctypes.data, None))
        out = pat.run(model, tol=0.0, max_iters=1)
        counts, theta1 = x.update(theta, model, eff)
        rtol = x.rtol_update(model)
        xr.assert_elementwise(out["counts"], counts, rtol, f"H={H} model {model} counts", where)
        xr.assert_elementwise(out["theta"], theta1, rtol, f"H={H} model {model} theta", where)
        assert not out["counts"][:, d.zero_locus].any()


def test_emulated_standalone_estep_does_not_move_the_state():
    """update_probability_at_read_level semantics (EMfactory.py:146-212): the E-step alone leaves only the numerator
    behind.  Two stand-alone E-steps followed by a full update must give exactly what one update gives."""
    import ctypes as C

    d = synth.generate(T=60, N=600, H=8, sample_index=5)
    eff = eo.effective_length_table(d.lengths)
    oapm = eo.apm_from_pairs(d.T, d.H, d.N, d.pair_class, d.pair_locus, d.pair_mask, d.count)
    gene_of = eo.gene_index(d.T, d.groups())
    for model in (4, 2):
        pat = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of)
        theta = pat.prepare(eff)
        want_counts = eo.sum_read(oapm, eo.e_step(oapm, theta, model, gene_of))
        for _ in range(2):
            pat.check(pat.lib.gbrs_em_run_begin(C.byref(pat.desc), 0.0, 1, None))
            pat.check(pat.lib.gbrs_em_launch_estep(C.byref(pat.desc), model, None))
            assert hp.relerr(pat.acc[:, : pat.H].T, want_counts) < 1e-12
            assert np.array_equal(pat.current_theta(), theta)  # theta did not move
        out = pat.run(model, tol=0.0, max_iters=2)
        t1 = want_counts / eff
        t2 = eo.sum_read(oapm, eo.e_step(oapm, t1, model, gene_of)) / eff
        assert out["iters"] == 2 and hp.relerr(out["theta"], t2) < 1e-12


def test_emulated_zero_normaliser_is_reported():
    """theta = 0 on every alignment of a class -> 0/0 in the E-step: GBRS_E_NUMERIC (the reference raises
    FloatingPointError under np.seterr(all='raise'))."""
    d = synth.generate(T=40, N=300, H=4, sample_index=1)
    pat = simt_em.HostPattern(synth.to_apm(d))
    pat.prepare(None)
    zero = np.zeros((d.T, 8))
    pat.check(pat.lib.gbrs_em_set_theta(pat.desc, zero.ctypes.data, None))
    with pytest.raises(FloatingPointError):
        pat.run(4, tol=1e-4, max_iters=5)


def test_em_kernels_are_race_free_under_thread_sanitizer():
    """Five model-4 updates and one update of models 1-3 under ThreadSanitizer (intra-block ordering: blocks run one
    after the other in the emulation, so races between blocks are out of its reach)."""
    try:
        lib = simt_em.build(tsan=True)
    except RuntimeError as e:
        pytest.skip(f"ThreadSanitizer build unavailable: {e}")
    rt = subprocess.run(["g++", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(rt) or not os.path.exists(rt):
        pytest.skip("libtsan.so not found")
    code = f"""
import sys
sys.path.insert(0, {ROOT!r})
import numpy as np
from gbrs_b200 import synth
from oracle import em_oracle as eo
from tests import simt_em
simt_em._emul[False] = simt_em.load(tsan=True)
d = synth.generate(T=60, N=500, H=8, sample_index=3, wide_frac=0.05)
pat = simt_em.HostPattern(synth.to_apm(d), gene_of=eo.gene_index(d.T, d.groups()), item_len=8)
pat.prepare(eo.effective_length_table(d.lengths), 0.5)
out = pat.run(4, tol=0.0, max_iters=5)
for model in (3, 2, 1):
    out = pat.run(model, tol=0.0, max_iters=1)
assert np.isfinite(out["theta"]).all()
pat.alignment_counts()
print("TSAN-RUN-OK")
"""
    env = dict(os.environ, LD_PRELOAD=rt, TSAN_OPTIONS="halt_on_error=0 report_signal_unsafe=0 exitcode=0",
               OMP_NUM_THREADS="1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=1500)
    if "TSAN-RUN-OK" not in res.stdout:
        pytest.skip("the sanitizer run did not complete here: " + res.stderr[-400:])
    assert "ThreadSanitizer: data race" not in res.stderr, res.stderr[-4000:]


@pytest.mark.parametrize("model,R", [(4, 2), (2, 3)])
def test_emulated_row_shards_equal_the_unsharded_run(model, R):
    """The N > 1 compute path (gbrs_em_launch_local -> sum of the numerators over the shards -> gbrs_em_launch_update,
    every shard taking the same stop decision) on the emulated library: R shards, exchange by hand, against the
    single-shard run and the oracle.  Mirrors tests/test_sharded_gpu.py."""
    import ctypes as C

    from gbrs_b200 import _lib

    d = synth.generate(T=100, N=1200, H=8, sample_index=7)
    gene_of = eo.gene_index(d.T, d.groups())
    eff = eo.effective_length_table(d.lengths)
    apm = synth.to_apm(d)
    whole = simt_em.HostPattern(apm, gene_of=gene_of)
    whole.prepare(eff)
    ref = whole.run(model, tol=1e-3, max_iters=60)
    pats = [simt_em.HostPattern(apm, gene_of=gene_of, shard_rank=r, shard_count=R) for r in range(R)]
    assert sum(p.info["nnz"] for p in pats) == d.nnz
    lib = pats[0].lib

    def exchange():
        total = sum(p.acc for p in pats)
        for p in pats:
            p.acc[:] = total

    for p in pats:
        p.efflen[:, : d.H] = eff.T
        p.check(lib.gbrs_em_prepare_local(C.byref(p.desc), None))
    exchange()
    for p in pats:
        p.check(lib.gbrs_em_prepare_finish(C.byref(p.desc), 0.0, None))
        p.check(lib.gbrs_em_run_begin(C.byref(p.desc), 1e-3, 60, None))
    for it in range(1, 62):
        for p in pats:
            p.check(lib.gbrs_em_launch_local(C.byref(p.desc), model, None))
        exchange()
        for p in pats:
            p.check(lib.gbrs_em_launch_update(C.byref(p.desc), None))
        done = {int(p.ctrl[_lib.CTRL_DONE]) for p in pats}
        assert len(done) == 1  # every shard takes the same decision
        if done == {1}:
            break
    assert it == ref["iters"] == int(pats[0].ctrl[_lib.CTRL_ITERS])
    for p in pats:
        assert np.array_equal(p.current_theta(), pats[0].current_theta())
    assert hp.relerr(pats[0].current_theta(), ref["theta"]) < 1e-12
    assert hp.relerr(pats[0].acc[:, : d.H].T, ref["counts"]) < 1e-12
    o = hp.oracle_run(d, model, tol=1e-3, max_iters=60)
    assert o["iters"] == it and hp.relerr(ref["counts"], o["counts"]) < 1e-12


def _run_fused_ranks(d, model, R, tol, max_iters, tsan=False, poll=1, mode=2, timeout_ms=0, absent=()):
    """R ranks = R private instances of the emulated library running at the same time in R host threads, their
    symmetric exchange buffers in shared host memory: the fused NVLink exchange (k_locus_acc publishes and raises
    `ready`, the reduce step sums a slice with peer loads and raises `done`, the update waits for it) runs for real.
    One SM / one resident block per kernel ($GBRS_SIMT_SMS=1): the reduce + update launch needs all its blocks
    resident at once, and the emulation runs the blocks of a launch one after the other."""
    import ctypes as C
    import threading

    from gbrs_b200 import _lib

    os.environ["GBRS_SIMT_SMS"] = "1"
    try:
        gene_of = eo.gene_index(d.T, d.groups())
        eff = eo.effective_length_table(d.lengths)
        apm = synth.to_apm(d)
        pats = [simt_em.HostPattern(apm, gene_of=gene_of, shard_rank=r, shard_count=R,
                                    lib=simt_em.load_instance(f"rank{r}", tsan)) for r in range(R)]
        slice_len = ((8 * d.T + R - 1) // R + 1) & ~1
        n_doubles = R * slice_len + 8 * d.T + 16 if mode >= 2 else 2 * 8 * d.T + 16  # push, tag | pull layout
        bufs = [np.zeros(n_doubles) for _ in range(R)]
        for r, p in enumerate(pats):
            p.efflen[:, : d.H] = eff.T
            p.desc.xchg_enabled, p.desc.xchg_rank, p.desc.xchg_mc, p.desc.xchg_timeout_ms = mode, r, None, timeout_ms
            for q in range(R):
                p.desc.xchg_peer[q] = bufs[q].ctypes.data
        errors, iters = [], [0] * R

        def rank_main(r):
            p = pats[r]
            try:
                p.check(p.lib.gbrs_em_prepare_local(C.byref(p.desc), None))
                p.check(p.lib.gbrs_em_prepare_finish(C.byref(p.desc), 0.0, None))
                p.check(p.lib.gbrs_em_run_begin(C.byref(p.desc), tol, max_iters, None))
                while not p.ctrl[_lib.CTRL_DONE]:
                    for _ in range(poll):  # updates queued after the stop are no-ops, as in the product's graph replay
                        p.check(p.lib.gbrs_em_launch_local(C.byref(p.desc), model, None))
                        p.check(p.lib.gbrs_em_launch_update(C.byref(p.desc), None))
                    assert p.ctrl[_lib.CTRL_ERROR] == 0, int(p.ctrl[_lib.CTRL_ERROR])
                iters[r] = int(p.ctrl[_lib.CTRL_ITERS])
            except BaseException as e:  # noqa: BLE001 - reported by the main thread
                errors.append((r, repr(e)))

        threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(R) if r not in absent]
        for t in threads:
            t.start()
        for t in threads:
            t.join(timeout=900)
        assert not errors, errors
        assert not any(t.is_alive() for t in threads)
        return pats, iters
    finally:
        os.environ.pop("GBRS_SIMT_SMS", None)


@pytest.mark.parametrize("R,model,mode", [(2, 4, 2), (3, 2, 2), (3, 4, 1), (2, 4, 3), (3, 3, 3)])
def test_emulated_fused_exchange_between_concurrent_ranks(R, model, mode):
    """mode 2: the one-launch push form (k_locus_xchg); mode 1: the pull form; mode 3: the tag form (no flags: every
    double carries the parity of its exchange in its sign bit and is polled by the thread that needs it)."""
    d = synth.generate(T=70, N=900, H=8, sample_index=12)
    pats, iters = _run_fused_ranks(d, model, R, 1e-3, 60, poll=2, mode=mode)
    o = hp.oracle_run(d, model, tol=1e-3, max_iters=60)
    assert iters == [o["iters"]] * R
    for p in pats:  # bit-identical on every rank: each element of the numerator is summed by exactly one rank
        assert np.array_equal(p.current_theta(), pats[0].current_theta())
        assert np.array_equal(p.acc, pats[0].acc)
    assert hp.relerr(pats[0].current_theta(), o["theta"]) < 1e-12
    assert hp.relerr(pats[0].acc[:, : d.H].T, o["counts"]) < 1e-12


@pytest.mark.parametrize("mode", [2, 3])
def test_emulated_exchange_timeout_stops_every_block(mode):
    """A peer that never shows up: the wait is bounded by wall-clock time, the error flag (3) and the stop flag are
    raised and the kernel returns -- no block continues on partial sums, nothing hangs."""
    import ctypes as C
    import time

    from gbrs_b200 import _lib

    d = synth.generate(T=40, N=300, H=8, sample_index=3)
    os.environ["GBRS_SIMT_SMS"] = "1"
    try:
        R = 2
        p = simt_em.HostPattern(synth.to_apm(d), shard_rank=0, shard_count=R, lib=simt_em.load_instance("rank0"))
        slice_len = ((8 * d.T + R - 1) // R + 1) & ~1
        bufs = [np.zeros(R * slice_len + 8 * d.T + 16) for _ in range(R)]
        p.desc.xchg_enabled, p.desc.xchg_rank, p.desc.xchg_mc, p.desc.xchg_timeout_ms = mode, 0, None, 150
        for q in range(R):
            p.desc.xchg_peer[q] = bufs[q].ctypes.data
        t0 = time.time()
        p.check(p.lib.gbrs_em_prepare_local(C.byref(p.desc), None))  # rank 1 never raises its flag
        assert time.time() - t0 < 30
        assert int(p.ctrl[_lib.CTRL_ERROR]) == 3 and int(p.ctrl[_lib.CTRL_DONE]) == 1
        theta_before = p.theta.copy()
        p.check(p.lib.gbrs_em_launch_local(C.byref(p.desc), 4, None))  # stopped: queued work is a no-op
        assert np.array_equal(p.theta, theta_before)
    finally:
        os.environ.pop("GBRS_SIMT_SMS", None)


def test_emulated_tag_exchange_reports_a_negative_expression_value():
    """The tag form carries its "arrived" bit in the sign of every transported double, so a negative numerator cannot be
    transported: a theta with a negative value (not an expression estimate) raises the numeric error flag instead of being
    summed silently as its absolute value."""
    import ctypes as C
    import threading

    from gbrs_b200 import _lib

    d = synth.generate(T=30, N=300, H=8, sample_index=6)
    os.environ["GBRS_SIMT_SMS"] = "1"
    try:
        R = 2
        apm = synth.to_apm(d)
        pats = [simt_em.HostPattern(apm, shard_rank=r, shard_count=R, lib=simt_em.load_instance(f"rank{r}")) for r in range(R)]
        slice_len = ((8 * d.T + R - 1) // R + 1) & ~1
        bufs = [np.zeros(R * slice_len + 8 * d.T + 16) for _ in range(R)]
        for r, p in enumerate(pats):
            p.desc.xchg_enabled, p.desc.xchg_rank, p.desc.xchg_mc, p.desc.xchg_timeout_ms = 3, r, None, 0
            for q in range(R):
                p.desc.xchg_peer[q] = bufs[q].ctypes.data
        errors = []
        # a (locus, haplotype) slot none of whose classes has it as its only alignment: with a slightly negative theta there
        # every class normaliser stays positive, so the slot's numerator theta * sum(w) is negative
        nnz_of_class = np.bincount(d.pair_class, weights=synth._popcount8(d.pair_mask), minlength=d.N)
        t_neg = h_neg = None
        for t in np.argsort(-np.bincount(d.pair_locus, minlength=d.T)):
            sel = d.pair_locus == t
            for h in range(d.H):
                hit = sel & (((d.pair_mask >> h) & 1) == 1)
                if hit.any() and np.all(nnz_of_class[d.pair_class[hit]] >= 2):
                    t_neg, h_neg = int(t), h
                    break
            if t_neg is not None:
                break
        assert t_neg is not None

        def rank_main(r):
            p = pats[r]
            try:
                p.check(p.lib.gbrs_em_prepare_local(C.byref(p.desc), None))
                p.check(p.lib.gbrs_em_prepare_finish(C.byref(p.desc), 0.0, None))
                assert p.ctrl[_lib.CTRL_ERROR] == 0
                bad = np.zeros((d.T, 8))
                bad[:, : d.H] = p.current_theta().T
                bad[t_neg, h_neg] = -1e-9 * bad[:, : d.H].max()  # one slightly negative slot: its numerator is negative
                p.check(p.lib.gbrs_em_set_theta(C.byref(p.desc), bad.ctypes.data, None))
                p.check(p.lib.gbrs_em_run_begin(C.byref(p.desc), 0.0, 1, None))
                p.check(p.lib.gbrs_em_launch_local(C.byref(p.desc), 4, None))
            except BaseException as e:  # noqa: BLE001 - reported by the main thread
                errors.append((r, repr(e)))

        threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(R)]
        for t in threads:
            t.start()
        for t in threads:
            t.join(timeout=300)
        assert not errors, errors
        assert any(int(p.ctrl[_lib.CTRL_ERROR]) == 1 for p in pats)  # the rank(s) whose shard holds classes of that slot
    finally:
        os.environ.pop("GBRS_SIMT_SMS", None)


def test_fused_exchange_is_race_free_under_thread_sanitizer():
    """Two and three concurrent ranks under ThreadSanitizer: every access to a peer's numerator must be ordered by the
    ready / done flags (with the flag store weakened to a relaxed store the sanitizer reports the peer loads)."""
    try:
        simt_em.build(tsan=True)
    except RuntimeError as e:
        pytest.skip(f"ThreadSanitizer build unavailable: {e}")
    rt = subprocess.run(["g++", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(rt) or not os.path.exists(rt):
        pytest.skip("libtsan.so not found")
    code = f"""
import sys
sys.path.insert(0, {ROOT!r})
import numpy as np
from gbrs_b200 import synth
from tests.test_em_simt import _run_fused_ranks
d = synth.generate(T=40, N=400, H=8, sample_index=12)
pats, iters = _run_fused_ranks(d, 4, 2, 0.0, 4, tsan=True)
assert iters == [4, 4] and np.array_equal(pats[0].current_theta(), pats[1].current_theta())
pats, iters = _run_fused_ranks(d, 1, 3, 0.0, 2, tsan=True)
assert iters == [2, 2, 2]
pats, iters = _run_fused_ranks(d, 4, 3, 0.0, 3, tsan=True, mode=3)  # tag form: nothing but the 8-byte accesses themselves
assert iters == [3, 3, 3] and np.array_equal(pats[0].current_theta(), pats[2].current_theta())
print("TSAN-RUN-OK")
"""
    env = dict(os.environ, LD_PRELOAD=rt, TSAN_OPTIONS="halt_on_error=0 report_signal_unsafe=0 exitcode=0",
               OMP_NUM_THREADS="1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=1500)
    if "TSAN-RUN-OK" not in res.stdout:
        pytest.skip("the sanitizer run did not complete here: " + res.stderr[-400:])
    assert "ThreadSanitizer: data race" not in res.stderr, res.stderr[-4000:]


@pytest.mark.parametrize("knob", ["GBRS_FORCE_ENTRY64"])
def test_emulated_alternative_layouts(knob, monkeypatch):
    """64-bit locus-major entry words (what shards beyond 2^24 classes use): one update of every model on the forced
    layout against the oracle."""
    monkeypatch.setenv(knob, "1")
    d = synth.generate(T=90, N=1000, H=8, sample_index=13, wide_frac=0.04)
    gene_of = eo.gene_index(d.T, d.groups())
    pat = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of, item_len=8)
    assert pat.info["entry_bytes"] == 8
    eff = eo.effective_length_table(d.lengths)
    theta = pat.prepare(eff)
    oapm = eo.apm_from_pairs(d.T, d.H, d.N, d.pair_class, d.pair_locus, d.pair_mask, d.count)
    assert hp.relerr(theta, eo.prepare(oapm, eff, 0.0)) < 1e-12
    for model in (4, 3, 2, 1):
        want = eo.sum_read(oapm, eo.e_step(oapm, theta, model, gene_of))
        out = pat.run(model, tol=0.0, max_iters=1)
        assert hp.relerr(out["counts"], want) < 1e-12
        theta = out["theta"]


def _random_problem(rng):
    """A small problem of arbitrary shape: 1-44 loci, 1-8 haplotypes, 1-260 classes (some wide, some with count 0),
    random haplotype masks, random contiguous genes."""
    T, H, N = int(rng.integers(1, 45)), int(rng.integers(1, 9)), int(rng.integers(1, 260))
    kmax = int(rng.choice([1, 2, 4, 12, 30]))
    k = np.minimum(1 + rng.poisson(rng.uniform(0.2, 3.0), N), min(kmax, T)).astype(np.int64)
    cls = np.repeat(np.arange(N), k)
    key = np.unique(cls * T + rng.integers(0, T, cls.size))
    full = (1 << H) - 1
    mask = np.where(rng.random(key.size) < 0.4, full, rng.integers(1, full + 1, key.size)).astype(np.uint8)
    count = rng.integers(0 if rng.random() < 0.3 else 1, 9, N).astype(np.float64)
    _, gene_of = np.unique(np.sort(rng.integers(0, int(rng.integers(1, T + 1)), T)), return_inverse=True)
    d = synth.SynthData(T=T, H=H, N=N, pair_class=key // T, pair_locus=key % T, pair_mask=mask, count=count,
                        gene_of=gene_of.astype(np.int64), lengths=rng.integers(50, 4000, size=(T, H)).astype(np.float64),
                        hname=synth.HAPLOTYPES[:H])
    d.lname = [f"T{t:04d}" for t in range(T)]
    d.gname = [f"G{g:04d}" for g in range(int(gene_of.max()) + 1)]
    return d


@pytest.mark.parametrize("seed", range(100, 112))
def test_emulated_library_on_random_shapes(seed):
    """Seeded sample of the fuzz run that was done by hand over 440 problems (no failure): arbitrary small shapes, loci
    outside every gene, 1-3 row shards, 8-entry items, pseudocount, three models per problem, alignment counts."""
    import ctypes as C

    rng = np.random.default_rng(seed)
    d = _random_problem(rng)
    if d.count.sum() == 0:
        d.count[0] = 1.0
    groups = d.groups()
    if rng.random() < 0.3 and len(groups) > 1:  # a gene missing from the group file: its loci are on their own
        groups.pop(int(rng.integers(0, len(groups))))
    gene_of = eo.gene_index(d.T, groups)
    item_len, R = int(rng.choice([0, 8])), int(rng.choice([1, 1, 2, 3]))
    apm = synth.to_apm(d)
    eff = eo.effective_length_table(d.lengths)
    oapm = eo.apm_from_pairs(d.T, d.H, d.N, d.pair_class, d.pair_locus, d.pair_mask, d.count)
    pats = [simt_em.HostPattern(apm, gene_of=gene_of, item_len=item_len, shard_rank=r, shard_count=R) for r in range(R)]
    lib = pats[0].lib

    def exchange():
        total = sum(p.acc for p in pats)
        for p in pats:
            p.acc[:] = total

    for p in pats:
        p.efflen[:, : d.H] = eff.T
        p.check(lib.gbrs_em_prepare_local(C.byref(p.desc), None))
    exchange()
    pseudocount = float(rng.choice([0.0, 0.0, 0.7]))
    for p in pats:
        p.check(lib.gbrs_em_prepare_finish(C.byref(p.desc), pseudocount, None))
    theta = pats[0].current_theta()
    assert hp.relerr(theta, eo.prepare(oapm, eff, pseudocount)) < 1e-11
    for model in (int(m) for m in rng.permutation([1, 2, 3, 4])[:3]):
        with np.errstate(all="ignore"):
            want = eo.sum_read(oapm, eo.e_step(oapm, theta, model, gene_of))
        if not np.isfinite(want).all():
            break
        for p in pats:
            p.check(lib.gbrs_em_run_begin(C.byref(p.desc), 0.0, 1, None))
            p.check(lib.gbrs_em_launch_local(C.byref(p.desc), model, None))
        exchange()
        for p in pats:
            p.check(lib.gbrs_em_launch_update(C.byref(p.desc), None))
            assert int(p.ctrl[2]) == 0
        assert hp.relerr(pats[0].acc[:, : d.H].T, want) < 1e-11
        theta = pats[0].current_theta()
        assert hp.relerr(theta, want / eff) < 1e-11
    if R == 1:
        aln, uniq, lu = pats[0].alignment_counts()
        want = eo.alignment_counts(oapm)
        assert np.array_equal(aln, want["aln"]) and np.array_equal(uniq, want["uniq"]) and np.array_equal(lu, want["locus_uniq"])
