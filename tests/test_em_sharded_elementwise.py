"""Row-sharded EM updates with the cross-rank sum done inside the library's own kernels, element by element against the
extended-precision reference (tests/xref.py), at 2 to 8 ranks and through each exchange form:
  * push (xchg_enabled 2, the default between GPUs): k_locus_xchg<UNIT, false> -- every value is stored into its
    owner's slice, the owner sums its slice over the ranks and broadcasts the totals;
  * tag (3): k_locus_xchg<UNIT, true> -- the same slices, every double carrying its own "arrived" bit;
  * pull (1): k_locus_acc publishes the local numerator, the owner of each slice of 4T double2 pairs loads it from every
    peer (k_xchg_reduce in prepare(), k_locus_update<true, true> in an update).
R ranks are R private instances of the emulated library (tests/simt_em.py) running at the same time in R host threads,
their symmetric exchange buffers in shared host memory, as in tests/test_em_simt._run_fused_ranks.

The push and tag forms give each owner push_slice_len = (ceil(8T / R) + 1) & ~1 doubles, the pull form ceil(4T / R)
pairs: with few loci and many ranks the trailing owners get short or empty slices, and with few classes (or one class
holding most of the nnz) the class split of the packer leaves ranks without classes.  Each case states how many owners
are empty and how many ranks hold no class, so that a drift of the shapes fails instead of quietly covering less.

An element summed twice, dropped, taken from the wrong rank or left stale from the previous exchange fails here whatever
its magnitude: zeros must match exactly and every other element must lie within the error bound of its shape."""
import ctypes as C
import shutil
import threading

import numpy as np
import pytest

from gbrs_b200 import _lib, synth
from oracle import em_oracle as eo
from tests import layouts, simt_em
from tests import xref as xr

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ is needed to build the SIMT emulation")

FORMS = {"push": 2, "tag": 3, "pull": 1}
MODELS = (4, 3, 2, 1)


def push_slice_len(T, R):
    """doubles per owner in the push and tag forms (em_kernels.cu, push_slice_len)"""
    return ((8 * T + R - 1) // R + 1) & ~1


def empty_owners(T, R, form):
    """owners whose slice of the numerator is empty"""
    if form == "pull":
        n, per = 4 * T, (4 * T + R - 1) // R
    else:
        n, per = 8 * T, push_slice_len(T, R)
    return sum(1 for r in range(R) if per * r >= n)


class Ranks:
    """R emulated ranks of one problem, their fused exchange wired through host buffers."""

    def __init__(self, d, R, form, item_len=0, gene_of=None):
        self.d, self.R, self.form = d, R, form
        self.gene_of = eo.gene_index(d.T, d.groups()) if gene_of is None else gene_of
        self.eff = eo.effective_length_table(d.lengths)
        apm = synth.to_apm(d)
        self.pats = [simt_em.HostPattern(apm, gene_of=self.gene_of, item_len=item_len, shard_rank=r, shard_count=R,
                                         lib=simt_em.load_instance(f"rank{r}")) for r in range(R)]
        mode = FORMS[form]
        n = R * push_slice_len(d.T, R) + 8 * d.T + 16 if mode >= 2 else 2 * 8 * d.T + 16
        self.bufs = [np.zeros(n) for _ in range(R)]
        self.theta_in = np.zeros((d.T, 8))  # read by the library through a raw pointer: kept alive here
        for r, p in enumerate(self.pats):
            p.efflen[:, : d.H] = self.eff.T
            p.desc.xchg_enabled, p.desc.xchg_rank, p.desc.xchg_mc, p.desc.xchg_timeout_ms = mode, r, None, 0
            for q in range(R):
                p.desc.xchg_peer[q] = self.bufs[q].ctypes.data

    @property
    def classes(self):
        return [int(p.info["n_classes"]) for p in self.pats]

    def each(self, step):
        """step(p) on every rank at the same time (the exchange waits for all of them); returns the per-rank results"""
        out, errors = [None] * self.R, []

        def main(r):
            try:
                out[r] = step(self.pats[r])
            except BaseException as e:  # noqa: BLE001 - reported below
                errors.append((r, repr(e)))

        threads = [threading.Thread(target=main, args=(r,)) for r in range(self.R)]
        for t in threads:
            t.start()
        for t in threads:
            t.join(timeout=600)
        assert not any(t.is_alive() for t in threads), "a rank did not finish"
        assert not errors, errors
        return out

    def prepare(self, pseudocount):
        def step(p):
            p.check(p.lib.gbrs_em_prepare_local(C.byref(p.desc), None))
            p.check(p.lib.gbrs_em_prepare_finish(C.byref(p.desc), float(pseudocount), None))
            assert p.ctrl[_lib.CTRL_ERROR] == 0, int(p.ctrl[_lib.CTRL_ERROR])
            return p.current_theta()

        return self.each(step)

    def update(self, model, theta=None):
        """one update of `model` on every rank, from theta (H x T) if given, else from the current estimate: (summed
        numerator, theta') per rank"""
        if theta is not None:
            self.theta_in[:] = 0.0
            self.theta_in[:, : self.d.H] = theta.T

        def step(p):
            if theta is not None:
                p.check(p.lib.gbrs_em_set_theta(C.byref(p.desc), self.theta_in.ctypes.data, None))
            p.check(p.lib.gbrs_em_run_begin(C.byref(p.desc), 0.0, 1, None))
            p.check(p.lib.gbrs_em_launch_local(C.byref(p.desc), model, None))
            p.check(p.lib.gbrs_em_launch_update(C.byref(p.desc), None))
            assert p.ctrl[_lib.CTRL_ERROR] == 0, int(p.ctrl[_lib.CTRL_ERROR])
            assert int(p.ctrl[_lib.CTRL_ITERS]) == 1
            return p.acc.copy(), p.current_theta()

        return self.each(step)

    def run(self, model, pseudocount, tol, max_iters):
        def step(p):
            p.check(p.lib.gbrs_em_prepare_local(C.byref(p.desc), None))
            p.check(p.lib.gbrs_em_prepare_finish(C.byref(p.desc), float(pseudocount), None))
            p.check(p.lib.gbrs_em_run_begin(C.byref(p.desc), tol, max_iters, None))
            while not p.ctrl[_lib.CTRL_DONE]:
                p.check(p.lib.gbrs_em_launch_local(C.byref(p.desc), model, None))
                p.check(p.lib.gbrs_em_launch_update(C.byref(p.desc), None))
            assert p.ctrl[_lib.CTRL_ERROR] == 0, int(p.ctrl[_lib.CTRL_ERROR])
            n = int(p.ctrl[_lib.CTRL_ITERS])
            return n, p.err_log[:n].copy(), p.acc.copy(), p.current_theta()

        return self.each(step)


@pytest.fixture(autouse=True)
def one_resident_block(monkeypatch):
    """one SM, so one resident block per kernel: the exchange kernels need all their blocks resident at once, and the
    emulation runs the blocks of a launch one after the other"""
    xr.require_longdouble()
    monkeypatch.setenv("GBRS_SIMT_SMS", "1")


def check_one_update_each_model(rk, x, seed, where=None, pseudocounts=(0.0, 0.25)):
    """prepare() with each pseudocount, then one update of each model, the first from a random theta, each following one
    from the theta' the ranks computed before (the reference starts from the same float64 values): theta0, the summed
    numerator and theta' element-wise, bit-identical on every rank, the zero-count locus (if any) exactly 0."""
    d = rk.d
    for pc in pseudocounts:
        got = rk.prepare(pc)
        xr.assert_elementwise(got[0], x.prepare(rk.eff, pc), x.rtol_prepare(pc), f"R={rk.R} {rk.form} theta0 pc={pc}",
                              where)
        for g in got[1:]:
            assert np.array_equal(g, got[0])
    theta = xr.random_theta(x, seed=seed)
    for k, model in enumerate(MODELS):
        out = rk.update(model, theta if k == 0 else None)
        counts, theta1 = x.update(theta, model, rk.eff)
        rtol = x.rtol_update(model)
        what = f"R={rk.R} {rk.form} model {model}"
        acc0, th0 = out[0]
        xr.assert_elementwise(acc0[:, : d.H].T, counts, rtol, what + " counts", where)
        xr.assert_elementwise(th0, theta1, rtol, what + " theta", where)
        for acc, th in out[1:]:  # each element is summed by exactly one rank: the same bits everywhere
            assert np.array_equal(acc, acc0) and np.array_equal(th, th0), what
        if getattr(d, "zero_locus", None) is not None:
            assert not acc0[d.zero_locus].any()
        theta = th0


LAYOUT_CASES = [("push", R, 8) for R in range(2, 9)] + [("push", 5, 3)] + [
    (form, R, 8) for form in ("tag", "pull") for R in (2, 3, 5, 8)]


@pytest.mark.parametrize("form,R,H", LAYOUT_CASES)
def test_sharded_one_update_on_constructed_layout(form, R, H):
    """The constructed layouts of tests/layouts.py (every column-pass segment, row-pass width and lane mask), split over R
    ranks by the packer's class split."""
    d = layouts.make_layout(H)
    gene_of = eo.gene_index(d.T, d.groups())
    whole = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of, item_len=16)
    layouts.assert_layout_covers(whole.packed)
    rk = Ranks(d, R, form, item_len=16, gene_of=gene_of)
    assert sum(p.info["nnz"] for p in rk.pats) == d.nnz
    assert all(c > 0 for c in rk.classes)
    check_one_update_each_model(rk, xr.XRef(d, gene_of), seed=100 * R + H, where=layouts.locus_kinds(whole.packed))


# (form, R, T, owners with an empty slice).  T = 1 leaves the trailing owners without a slice; at R = 8 an odd T makes
# ceil(8T / R) odd (the rounding of push_slice_len) and 4T mod 8 != 0 (the last pull slice is short); at R = 5 and 7,
# 8T mod R != 0 and ceil(8T / R) is odd.  All three forms at R = 8; push and pull (the two slice arithmetics) at R = 5, 7.
EDGES = [(form, 8, T, e) for form in FORMS for T, e in ((1, 4), (3, 2), (5, 1))] + [
    ("push", 7, 1, 3), ("push", 7, 4, 1), ("pull", 7, 2, 3), ("pull", 7, 4, 1),
    ("push", 5, 1, 1), ("push", 5, 3, 1), ("pull", 5, 1, 1), ("pull", 5, 3, 1)]


def test_slice_edge_shapes_are_what_they_claim():
    ceil_odd = lambda R, T: (-(-8 * T // R)) % 2 == 1  # noqa: E731
    for form, R, T, e in EDGES:
        assert empty_owners(T, R, form) == e, (form, R, T)
        assert T == 1 or ceil_odd(R, T), (form, R, T)
        assert R == 8 or T == 1 or 8 * T % R != 0, (form, R, T)
    assert {R for _, R, _, _ in EDGES} == {5, 7, 8}
    assert all(4 * T % 8 for form, R, T, _ in EDGES if form == "pull" and R == 8)


@pytest.mark.parametrize("form,R,T,empty", EDGES)
def test_sharded_one_update_at_slice_edges(form, R, T, empty):
    """Few loci for many ranks: trailing owners with short or empty slices.  prepare() runs without a pseudocount only
    (the pseudocount is applied after the exchange, on every rank alike; the layout cases check it)."""
    d = synth.generate(T=T, N=12 * T + 8, H=8, sample_index=T + 3)
    rk = Ranks(d, R, form)
    assert empty_owners(T, R, form) == empty
    assert sum(p.info["nnz"] for p in rk.pats) == d.nnz
    check_one_update_each_model(rk, xr.XRef(d, rk.gene_of), seed=T, pseudocounts=(0.0,))


EMPTY_SHARDS = [("few classes", 8, "push"), ("few classes", 8, "tag"), ("few classes", 7, "pull"),
                ("heavy first class", 8, "push"), ("heavy first class", 5, "tag"), ("heavy first class", 6, "pull")]


@pytest.mark.parametrize("kind,R,form", EMPTY_SHARDS)
def test_sharded_one_update_with_empty_shards(kind, R, form):
    """Ranks that pack no class at all still take part in every exchange (they contribute zeros and own a slice)."""
    d = layouts.make_empty_shards(kind, R)
    rk = Ranks(d, R, form)
    layouts.assert_empty_shards(kind, d, rk.classes, [p.info["nnz"] for p in rk.pats])
    check_one_update_each_model(rk, xr.XRef(d, rk.gene_of), seed=R)


@pytest.mark.parametrize("model", [4, 2])
def test_sharded_run_to_convergence_eight_ranks(model):
    """run() at eight ranks, push form, after prepare() with a pseudocount: the reference's iteration count, its error
    trajectory to 1e-7, theta and the expected counts element-wise within the bound of that many updates."""
    d = synth.generate(T=70, N=900, H=8, sample_index=12)
    rk = Ranks(d, 8, "push")
    x = xr.XRef(d, rk.gene_of)
    want = x.run(x.prepare(rk.eff, 0.25), model, rk.eff, 1e-3, 60)
    assert want["iters"] < 60
    out = rk.run(model, 0.25, 1e-3, 60)
    n, errs, acc, theta = out[0]
    assert n == want["iters"]
    np.testing.assert_allclose(errs, want["errs"], rtol=1e-7, atol=1e-7)
    rtol = x.rtol_run(model, n, pseudocount=0.25)
    xr.assert_elementwise(theta, want["theta"], rtol, f"run model {model} theta")
    xr.assert_elementwise(acc[:, : d.H].T, want["counts"], rtol, f"run model {model} counts")
    for m, e, a, th in out[1:]:
        assert m == n and np.array_equal(e, errs) and np.array_equal(a, acc) and np.array_equal(th, theta)
