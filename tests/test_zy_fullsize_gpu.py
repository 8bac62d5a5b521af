"""BASELINE.json's configurations at (or near) full size.

Oracle parity (the numpy restatement of the reference, oracle/em_oracle.py, on the host cores of the GPU box):
  * config 2 -- 80k transcripts x 8 haplotypes x 5M classes, model 4 -- at FULL size, a fixed number of updates:
    error trajectory to 1e-7 relative, theta / expected counts to 1e-9 (the north-star bar is 1e-6);
  * config 3 -- the same locus shape under models 1, 2 and 3 -- on a 1M-class slice;
  * config 4 -- diploid `-G` restriction -- on a 2M-class slice of the 20M-class shape.
Size-independent properties at the full single-GPU size of config 2:
  * every class' responsibilities sum to one  ->  expected counts add up to the class counts, in prepare() and after
    every update;
  * expected counts are finite, non-negative, and zero wherever a (locus, haplotype) has no alignment;
  * theta = counts / effective length (the M-step, EMfactory.py:228-232);
  * the result does not depend on the order of the alignment classes (a random relabelling of the 5M classes);
  * the result does not depend on row-sharding (two shards on one GPU, numerators summed by hand).
The run is cut at a fixed number of updates (tol = 0) so that both sides of a comparison do the same work.

Named to run after the parity tests of the EM (first executed on a device by the round-end driver)."""
import numpy as np
import pytest

from gbrs_b200 import synth
from tests import helpers as hp
from tests import xref as xr

UPDATES = 12


def relabel_classes(d, seed=5):
    """The same alignment classes under a random permutation of their ids."""
    perm = np.random.default_rng(seed).permutation(d.N)
    new_cls = perm[d.pair_class]
    order = np.argsort(new_cls, kind="stable")  # pairs stay locus-sorted inside a class
    count = np.empty_like(d.count)
    count[perm] = d.count
    d2 = synth.SynthData(T=d.T, H=d.H, N=d.N, pair_class=new_cls[order], pair_locus=d.pair_locus[order],
                         pair_mask=d.pair_mask[order], count=count, gene_of=d.gene_of, lengths=d.lengths, hname=d.hname)
    d2.lname, d2.gname = d.lname, d.gname
    return d2


def test_relabelling_keeps_the_problem():
    """CPU check of the helper: the oracle gives the same answer for the relabelled input."""
    d = synth.generate(T=60, N=900, H=8, sample_index=2)
    d2 = relabel_classes(d)
    assert not np.array_equal(d.count, d2.count) and d2.nnz == d.nnz and np.all(np.diff(d2.pair_class) >= 0)
    a, b = hp.oracle_run(d, 4), hp.oracle_run(d2, 4)
    assert a["iters"] == b["iters"] and hp.relerr(a["counts"], b["counts"]) < 1e-12


def run_fixed(d, eff):
    from gbrs_b200.emfactory import EMfactory

    em = EMfactory(synth.to_apm(d))
    em.target_lengths = eff
    em.prepare()
    theta0 = em.get_allelic_expression()
    em.run(model=4, tol=0.0, max_iters=UPDATES, verbose=False)
    assert em.num_iters == UPDATES
    return theta0, em.get_allelic_expression(), em.expected_read_counts().copy(), em.err_history.copy()


@pytest.mark.gpu
def test_full_size_properties_model4():
    from tests.test_sharded_gpu import run_sharded

    d = synth.generate(T=80_000, N=5_000_000, H=8)
    eff = synth.effective_lengths(d)
    total = d.count.sum()
    theta0, theta, counts, errs = run_fixed(d, eff)
    # conservation: prepare() distributes every class' count over its alignments, every E-step over its posterior
    assert abs((theta0 * eff).sum() - total) < 1e-9 * total
    assert abs(counts.sum() - total) < 1e-9 * total
    assert np.isfinite(counts).all() and counts.min() >= 0.0 and np.isfinite(errs).all() and errs.min() >= 0.0
    # support: no alignment, no expression
    support = np.zeros((d.H, d.T), dtype=bool)
    for h in range(d.H):
        support[h, d.pair_locus[((d.pair_mask >> h) & 1).astype(bool)]] = True
    assert not counts[~support].any() and not theta[~support].any()
    assert (counts[support] > 0).mean() > 0.99  # and (almost) every aligned slot keeps some
    # M-step: theta = counts / effective length
    assert hp.relerr(theta * eff, counts) < 1e-12
    # order of the classes is irrelevant
    _, theta_p, counts_p, errs_p = run_fixed(relabel_classes(d), eff)
    assert hp.relerr(counts_p, counts) < 1e-10 and hp.relerr(theta_p, theta) < 1e-10
    np.testing.assert_allclose(errs_p, errs, rtol=1e-8)
    # row-sharding is irrelevant
    s = run_sharded(d, 4, 2, tol=0.0, max_iters=UPDATES)
    assert s["iters"] == UPDATES
    assert hp.relerr(s["counts"], counts) < 1e-10 and hp.relerr(s["theta"], theta) < 1e-10


def gpu_fixed(d, model, updates, gtmask=None, **kw):
    from gbrs_b200.emfactory import EMfactory
    from gbrs_b200.quantify import hapmask_bytes

    em = EMfactory(synth.to_apm(d), locus_hapmask=None if gtmask is None else hapmask_bytes(gtmask), **kw)
    em.target_lengths = synth.effective_lengths(d)
    em.prepare()
    theta0 = em.get_allelic_expression()
    em.run(model=model, tol=0.0, max_iters=updates, verbose=False)
    return dict(theta0=theta0, theta=em.get_allelic_expression(), counts=em.expected_read_counts().copy(),
                errs=em.err_history.copy(), iters=em.num_iters)


def assert_parity(out, o, updates, d, model):
    assert out["iters"] == o["iters"] == updates
    assert hp.relerr(out["theta0"], o["theta0"]) < 1e-9
    np.testing.assert_allclose(out["errs"], o["errs"], rtol=1e-7)
    assert hp.relerr(out["theta"], o["theta"]) < 1e-9 and hp.relerr(out["counts"], o["counts"]) < 1e-9
    # element-wise against the float64 oracle: both sides are within the float64 error bound of tests/xref.py of the
    # exact result, so they are within twice that bound of each other (no absolute floor, zeros must match)
    rtol = 2 * xr.rtol_bound(*xr.shape_of(d), d.H, model, updates)
    xr.assert_elementwise(out["theta0"], o["theta0"], 2 * xr.rtol_bound(*xr.shape_of(d), d.H, model, 0), "theta0")
    xr.assert_elementwise(out["counts"], o["counts"], rtol, "counts")
    xr.assert_elementwise(out["theta"], o["theta"], rtol, "theta")


@pytest.mark.gpu
def test_config2_full_size_matches_oracle_model4():
    """BASELINE config 2 at its full 5M classes: 12 fixed updates of the GPU path against the oracle."""
    d = synth.generate(T=80_000, N=5_000_000, H=8)
    o = hp.oracle_run(d, 4, tol=0.0, max_iters=UPDATES)
    assert_parity(gpu_fixed(d, 4, UPDATES), o, UPDATES, d, 4)
    assert_parity(gpu_fixed(d, 4, UPDATES, tiles=True), o, UPDATES, d, 4)  # the opt-in single-pass tile kernel


@pytest.mark.gpu
@pytest.mark.parametrize("model", [1, 2, 3])
def test_config3_models_1_to_3_match_oracle_on_a_1m_class_slice(model):
    """BASELINE config 3 (the C2 locus shape under models 1-3) on a 1M-class slice, 6 fixed updates."""
    d = synth.generate(T=80_000, N=1_000_000, H=8)
    o = hp.oracle_run(d, model, tol=0.0, max_iters=6)
    assert_parity(gpu_fixed(d, model, 6), o, 6, d, model)


@pytest.mark.gpu
def test_config4_diploid_matches_oracle_on_a_2m_class_slice():
    """BASELINE config 4 (diploid -G restriction, 80k loci) on a 2M-class slice, 8 fixed updates."""
    d = synth.generate(T=80_000, N=2_000_000, H=8, with_genotype=True)
    gm = synth.genotype_mask(d)
    o = hp.oracle_run(d, 4, tol=0.0, max_iters=8, gtmask=gm)
    out = gpu_fixed(d, 4, 8, gtmask=gm)
    assert_parity(out, o, 8, d, 4)
    assert np.all(out["counts"][gm == 0] == 0.0)
