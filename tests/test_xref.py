"""The extended-precision reference (tests/xref.py) and the constructed layouts (tests/layouts.py) are themselves pinned: the
reference agrees element-wise with the float64 oracle and with every golden vector of the reference, the comparator sees
what a max-normalised check cannot, and every constructed layout reaches every kind of kernel work."""
import numpy as np
import pytest

from gbrs_b200 import synth
from gbrs_b200.emfactory import PackedPattern
from oracle import em_oracle as eo
from tests import helpers as hp
from tests import layouts
from tests import xref as xr


@pytest.mark.parametrize("name", hp.golden_em_cases())
def test_xref_matches_reference_golden_elementwise(name):
    xr.require_longdouble()
    g = hp.load_golden(name)
    d = hp.synth_from_golden(g)
    x = xr.XRef(d, eo.gene_index(d.T, d.groups()), g["gtmask"] if g["masked"] else None)
    eff = eo.effective_length_table(d.lengths)
    theta0 = x.prepare(eff, g["pseudocount"])
    xr.assert_elementwise(g["theta0"], theta0, 1e-13, f"{name} theta0")
    out = x.run(theta0, g["model"], eff, g["tol"], g["max_iters"])
    assert out["iters"] == g["iters"]
    np.testing.assert_allclose(out["errs"], g["errs"], rtol=1e-9, atol=1e-9)
    xr.assert_elementwise(g["theta"], out["theta"], 1e-13, f"{name} theta")
    xr.assert_elementwise(g["counts"], out["counts"], 1e-13, f"{name} counts")


@pytest.mark.parametrize("H", range(1, 9))
def test_xref_matches_oracle_on_constructed_layouts(H):
    """One update of every model from a theta scattered over e^+-40, and prepare() with a pseudocount."""
    xr.require_longdouble()
    d = layouts.make_layout(H)
    gene_of = eo.gene_index(d.T, d.groups())
    x = xr.XRef(d, gene_of)
    oapm = eo.apm_from_pairs(d.T, d.H, d.N, d.pair_class, d.pair_locus, d.pair_mask, d.count)
    eff = eo.effective_length_table(d.lengths)
    xr.assert_elementwise(eo.prepare(oapm, eff, 0.5), x.prepare(eff, 0.5), 1e-13, "theta0")
    theta = xr.random_theta(x, seed=H)
    for model in (4, 3, 2, 1):
        with np.errstate(all="raise", under="ignore"):
            want = eo.sum_read(oapm, eo.e_step(oapm, theta, model, gene_of))
        counts, theta1 = x.update(theta, model, eff)
        xr.assert_elementwise(want, counts, 1e-13, f"model {model} counts")
        xr.assert_elementwise(want / eff, theta1, 1e-13, f"model {model} theta")
        assert np.all(counts[:, d.zero_locus] == 0) and np.all(theta1[:, d.zero_locus] == 0)


def test_comparator_sees_what_max_normalisation_misses():
    want = np.array([[1.0, 1e-30, 0.0], [2.0, 3e-200, 5.0]])
    assert xr.assert_elementwise(want.copy(), want, 1e-15) == 0.0
    flushed = want.copy()
    flushed[0, 1] = 0.0
    assert hp.relerr(flushed, want) < 1e-29  # invisible to the max-normalised check
    with pytest.raises(AssertionError, match=r"zero pattern differs .*h=0, t=1"):
        xr.assert_elementwise(flushed, want, 1e-6)
    doubled = want.copy()
    doubled[1, 1] *= 2
    with pytest.raises(AssertionError, match=r"relative error 1\.000e\+00 over the bound .*h=1, t=1.*locus 1: depth 2"):
        xr.assert_elementwise(doubled, want, 1e-6, where=["", "depth 2", ""])
    with pytest.raises(AssertionError, match="non-finite"):
        xr.assert_elementwise(np.full_like(want, np.nan), want, 1e-6)


@pytest.mark.parametrize("item_len", [16, 64])
@pytest.mark.parametrize("H", range(1, 9))
def test_constructed_layout_covers_every_kernel_path(H, item_len):
    d = layouts.make_layout(H, item_len)
    gene_of = eo.gene_index(d.T, d.groups())
    packed = PackedPattern(synth.to_apm(d), gene_of=gene_of, item_len=item_len)
    s = layouts.assert_layout_covers(packed)
    depth = np.bincount(d.pair_locus, minlength=d.T)
    assert {8 * item_len, 8 * item_len + 1} <= set(depth.tolist())
    items = np.diff(packed.arrays["locus_item_ptr"].astype(np.int64))
    assert {8, 9} <= set(items.tolist()) or H == 1
    assert np.bincount(d.pair_class).max() > 32 and s["widths"][layouts.KMAX] > 0
    assert (depth == 0).sum() >= 3


def test_layout_check_fails_when_a_segment_is_missing():
    """Without the deep loci the constructor stops producing full items: the coverage check must say so."""
    d = layouts.make_layout(8)
    depth = np.bincount(d.pair_locus, minlength=d.T)
    drop = np.isin(d.pair_locus, np.flatnonzero(depth > 8 * 16))
    d.pair_class, d.pair_locus, d.pair_mask = d.pair_class[~drop], d.pair_locus[~drop], d.pair_mask[~drop]
    packed = PackedPattern(synth.to_apm(d), gene_of=eo.gene_index(d.T, d.groups()), item_len=16)
    with pytest.raises(AssertionError, match="short full"):
        layouts.assert_layout_covers(packed)
