"""Posterior read-origin probabilities (gbrs_em_posterior, the kernels behind EMfactory.posterior_probability) executed on
the CPU through the host SIMT shim (tests/simt_em.py, tests/simt_posterior.py), element by element against the
extended-precision reference of tests/xref.py, on the constructed layouts of tests/layouts.py.  Also: the class permutation both packers emit, row
shards, the -G restriction, the error of a zero normaliser, and that the call leaves every buffer of the EM as it was."""
import ctypes as C
import shutil

import numpy as np
import pytest

from gbrs_b200 import synth
from gbrs_b200.emfactory import EMfactory, PackedPattern, posterior_pattern
from gbrs_b200.quantify import hapmask_bytes
from oracle import em_oracle as eo
from tests import layouts, simt_posterior
from tests import posterior_checks as pc
from tests import xref as xr

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ is needed to build the SIMT emulation")

MODELS = (4, 3, 2, 1)


def setup(H, item_len=16, **kw):
    xr.require_longdouble()
    d = layouts.make_layout(H, item_len)
    gene_of = eo.gene_index(d.T, d.groups())
    apm = synth.to_apm(d)
    pat = simt_posterior.PosteriorHostPattern(apm, gene_of=gene_of, item_len=item_len, **kw)
    return d, gene_of, apm, pat, xr.XRef(d, gene_of), eo.effective_length_table(d.lengths)


def T8(theta_HT, T):
    out = np.zeros((T, 8))
    out[:, : theta_HT.shape[0]] = theta_HT.T
    return out


def posterior(pat, apm, model, theta_T8, x, hapmask=None):
    ip, ix = pc.pattern_arrays(posterior_pattern(apm, hapmask))
    return pc.entry_values(pat.posterior(model, theta_T8, ip, ix), ip, ix, x)


def set_theta(pat, theta_T8):
    pat.check(pat.lib.gbrs_em_set_theta(C.byref(pat.desc), theta_T8.ctypes.data, None))


@pytest.mark.parametrize("H", range(1, 9))
def test_emulated_posterior_elementwise_on_constructed_layouts(H):
    """Every state of the reference's `probability`: after prepare() (theta = 1, model 4: 1 / entries of the class, with
    and without a pseudocount, which does not enter the posterior), after a stand-alone E-step from a random theta, after
    one update (the E-step of the theta that entered it) and after run() to convergence (the E-step of theta_{k-1}, the
    other half of the ping-pong)."""
    d, gene_of, apm, pat, x, eff = setup(H)
    layouts.assert_layout_covers(pat.packed)
    for pcount in (0.0, 0.25):
        pat.prepare(eff, pcount)
        got = posterior(pat, apm, 4, np.ones((d.T, 8)), x)
        pc.check(got, x.e_step(np.ones((H, d.T)), 4), pc.rtol_posterior(x, 4), f"H={H} prepare pc={pcount}")
    theta = xr.random_theta(x, seed=H)
    tb = T8(theta, d.T)
    for model in MODELS:
        rtol = pc.rtol_posterior(x, model)
        want = x.e_step(theta, model)
        pc.check(posterior(pat, apm, model, tb, x), want, rtol, f"H={H} model {model} E-step")
        set_theta(pat, tb)
        pat.run(model, tol=0.0, max_iters=1)
        prev = pat.copy_theta(previous=True)
        assert np.array_equal(prev, tb)  # the theta that entered the update, bit for bit
        pc.check(posterior(pat, apm, model, prev, x), want, rtol, f"H={H} model {model} after one update")
    model = MODELS[H % 4]
    pat.prepare(eff, 0.25)
    out = pat.run(model, tol=1e-5, max_iters=400)
    k = out["iters"]
    assert 1 < k < 400
    prev = pat.copy_theta(previous=True)
    want_prev = x.run(x.prepare(eff, 0.25), model, eff, 1e-5, k - 1)["theta"]
    xr.assert_elementwise(prev[:, :H].T, want_prev, x.rtol_run(model, k - 1, pseudocount=0.25), f"H={H} theta_(k-1)")
    assert np.array_equal(pat.copy_theta(previous=False)[:, :H].T, out["theta"])
    got = posterior(pat, apm, model, prev, x)
    pc.check(got, x.e_step(prev[:, :H].T, model), pc.rtol_posterior(x, model), f"H={H} model {model} after run ({k})")


@pytest.mark.parametrize("model", MODELS)
def test_emulated_posterior_invariants(model):
    """Per class the posterior sums to 1 within the bound; sum_n c_n P[n,t,h] of the returned values matches the expected
    read counts of the E-step from the same theta; zero-count classes get a posterior where theta > 0."""
    d, gene_of, apm, pat, x, eff = setup(5)
    pat.prepare(eff)
    theta = xr.random_theta(x, seed=7 + model)
    tb = T8(theta, d.T)
    got = posterior(pat, apm, model, tb, x)
    rtol = pc.rtol_posterior(x, model)
    sums = pc.class_sums(got, x)
    assert np.all(np.abs(sums - 1) <= 8 * x.k_max * rtol), float(np.abs(sums - 1).max())
    set_theta(pat, tb)
    pat.check(pat.lib.gbrs_em_run_begin(C.byref(pat.desc), 0.0, 1, None))
    pat.check(pat.lib.gbrs_em_launch_estep(C.byref(pat.desc), model, None))
    xr.assert_elementwise(pat.acc[:, : d.H].T, pc.counts_from(got, x), x.rtol_update(model), f"model {model} counts")
    zc = np.flatnonzero(np.asarray(d.count) == 0)
    assert zc.size > 0
    sel = np.isin(x.n, zc) & (theta[x.h, x.t] > 0)
    assert sel.any() and np.all(got[sel] > 0)


def test_emulated_posterior_leaves_the_em_untouched():
    """prepare, run(max_iters=3), posterior of every model, run to convergence: theta, counts, error log and iteration
    count bit-identical to the same sequence without the posterior calls; every EM buffer is unchanged by each call; two
    calls give identical bits."""
    d, gene_of, apm, _, x, eff = setup(8)
    results = []
    for with_posterior in (False, True):
        pat = simt_posterior.PosteriorHostPattern(apm, gene_of=gene_of, item_len=16)
        pat.prepare(eff)
        pat.run(2, tol=0.0, max_iters=3)
        if with_posterior:
            prev = pat.copy_theta(previous=True)
            bufs = ("theta", "efflen", "acc", "iso", "weights", "subsets", "wit", "part", "gene_hap", "gamma", "err_log",
                    "scal", "ctrl")
            for model in MODELS:
                before = {k: getattr(pat, k).copy() for k in bufs}
                a = posterior(pat, apm, model, prev, x)
                b = posterior(pat, apm, model, prev, x)
                assert np.array_equal(a.view(np.uint64), b.view(np.uint64))
                for k in bufs:
                    assert np.array_equal(getattr(pat, k).view(np.uint8), before[k].view(np.uint8)), k
        out = pat.run(2, tol=1e-6, max_iters=400)
        results.append(out)
    a, b = results
    assert a["iters"] == b["iters"]
    for k in ("theta", "counts", "errs"):
        assert np.array_equal(a[k].view(np.uint64), b[k].view(np.uint64)), k


def test_emulated_posterior_tile_layout():
    """A pattern that runs model 4 on the fused tile kernel: the posterior still takes the two-pass row pass."""
    d, gene_of, apm, pat, x, eff = setup(8, tiles=dict(max_loci=48, max_items=192))
    pat.prepare(eff)
    theta = xr.random_theta(x, seed=3)
    for model in (4, 1):
        got = posterior(pat, apm, model, T8(theta, d.T), x)
        pc.check(got, x.e_step(theta, model), pc.rtol_posterior(x, model), f"tiles model {model}")


def test_emulated_posterior_genotype_restriction():
    """-G: the masked (t, h) columns are empty in the output pattern, the rest matches XRef(gtmask=...)."""
    xr.require_longdouble()
    d = synth.generate(T=200, N=3000, H=8, sample_index=4, with_genotype=True)
    gene_of = eo.gene_index(d.T, d.groups())
    gtmask = synth.genotype_mask(d)
    hapmask = hapmask_bytes(gtmask)
    apm = synth.to_apm(d)
    pat = simt_posterior.PosteriorHostPattern(apm, gene_of=gene_of, hapmask=hapmask)
    x = xr.XRef(d, gene_of, gtmask=gtmask)
    pattern = posterior_pattern(apm, hapmask)
    for h, (ip, _, _) in enumerate(pattern):
        empty = ((hapmask >> h) & 1) == 0
        assert empty.any() and not np.diff(ip)[empty].any()
    theta = xr.random_theta(x, seed=11)
    for model in MODELS:
        got = posterior(pat, apm, model, T8(theta, d.T), x, hapmask=hapmask)
        pc.check(got, x.e_step(theta, model), pc.rtol_posterior(x, model), f"-G model {model}")


@pytest.mark.parametrize("model", MODELS)
def test_emulated_posterior_zero_normaliser_raises(model):
    """theta = 0 on every entry of a class: the reference divides 0 by 0 and raises FloatingPointError; so does the call."""
    d, gene_of, apm, pat, x, eff = setup(4)
    pat.prepare(eff)
    theta = xr.random_theta(x, seed=5)
    n0 = int(x.n[np.flatnonzero(np.bincount(x.n) > 1)[0] == x.n][0])
    theta[x.h[x.n == n0], x.t[x.n == n0]] = 0.0
    with pytest.raises(FloatingPointError):
        posterior(pat, apm, model, T8(theta, d.T), x)


@pytest.mark.parametrize("R", range(2, 9))
def test_emulated_posterior_row_shards_are_bit_identical(R):
    """Every shard fills its own classes and 0 elsewhere: the sum over R shards equals the unsharded posterior bit for bit,
    and class_id is a permutation of the shard's non-empty classes that matches its pairs."""
    d, gene_of, apm, whole, x, eff = setup(8)
    theta = T8(xr.random_theta(x, seed=R), d.T)
    ip, ix = pc.pattern_arrays(posterior_pattern(apm))
    pats = [simt_posterior.PosteriorHostPattern(apm, gene_of=gene_of, item_len=16, shard_rank=r, shard_count=R) for r in range(R)]
    seen = np.concatenate([p.packed.arrays["class_id"] for p in pats])
    assert np.array_equal(np.sort(seen), np.unique(x.n))
    for model in MODELS:
        want = whole.posterior(model, theta, ip, ix)
        parts = [p.posterior(model, theta, ip, ix) for p in pats]
        for h in range(d.H):
            got = np.zeros_like(want[h])
            for part in parts:
                assert not (np.asarray(part[h] != 0) & (got != 0)).any()  # disjoint supports
                got = got + part[h]
            assert np.array_equal(got.view(np.uint64), want[h].view(np.uint64)), (model, h)


def _assert_class_id(packed, apm):
    """class_id[p] is the input class whose (locus, mask) words the packed class p holds"""
    a = packed.arrays
    cid, rowptr, pairs = a["class_id"], a["rowptr"].astype(np.int64), a["pairs"]
    assert cid.size == packed.info["n_classes"] and np.unique(cid).size == cid.size
    T, H, N = apm.shape
    mask = np.zeros((N, T), dtype=np.int64)
    for h, m in enumerate(apm.data):
        coo = m.tocoo()
        mask[coo.row, coo.col] |= 1 << h
    for p in range(cid.size):
        w = pairs[rowptr[p]: rowptr[p + 1]].astype(np.int64)
        row = np.zeros(T, dtype=np.int64)
        row[w & 0xFFFFFF] = w >> 24
        assert np.array_equal(row, mask[cid[p]]), p


@pytest.mark.parametrize("R", [1, 3])
def test_packers_emit_the_class_permutation(R):
    """class_id of the host packer and of the device packer (through the emulation): the same array, a permutation of
    the shard's non-empty classes, matching the pairs."""
    d = synth.generate(T=150, N=2500, H=8, sample_index=5, wide_frac=0.05)
    gene_of = eo.gene_index(d.T, d.groups())
    apm = synth.to_apm(d)
    for r in range(R):
        host = PackedPattern(apm, gene_of=gene_of, shard_rank=r, shard_count=R)
        _assert_class_id(host, apm)
        class_id = simt_posterior.emulated_device_class_id(apm, gene_of=gene_of, shard_rank=r, shard_count=R)
        assert np.array_equal(class_id, host.arrays["class_id"])


def test_weighted_prepare_posterior_on_the_host():
    """prepare() of a matrix with stored values: normalize_reads(READ) of the values (explicit zeros stay in the pattern
    with the value 0); a class whose values sum to 0 raises FloatingPointError."""
    from scipy.sparse import csc_matrix

    from gbrs_b200 import AlignmentPropertyMatrix as APM

    rng = np.random.default_rng(3)
    T, H, N = 12, 3, 50
    dense = (rng.random((H, N, T)) < 0.2) * rng.integers(1, 4, (H, N, T)).astype(np.float64)
    mats = [csc_matrix(dense[h]) for h in range(H)]
    mats[0].data[::5] = 0.0  # explicit zeros
    apm = APM.from_csc(mats, [f"h{h}" for h in range(H)], [f"t{t}" for t in range(T)])
    pattern = posterior_pattern(apm)
    rows = sum(np.bincount(ix, weights=v, minlength=N) for _, ix, v in pattern)
    vals = EMfactory._weighted_posterior(pattern, N)
    for (ip, ix, v), got in zip(pattern, vals):
        np.testing.assert_array_equal(got, v / rows[ix])
        assert np.array_equal(got == 0, v == 0) and (got == 0).any() == (v == 0).any()
    n0 = int(mats[1].indices[0])
    for m in mats:
        m.data[m.indices == n0] = 0.0
    with pytest.raises(FloatingPointError):
        EMfactory._weighted_posterior(posterior_pattern(apm), N)
