"""Every output element of the device EM against the extended-precision reference (tests/xref.py), on layouts built to
reach every kernel path (tests/layouts.py): each haplotype count H = 1..8, models 1-4, each code path of the update
(two-pass kernels, 64-bit entry words, the fused tile kernel with wide and tiny tiles, row shards).  The tolerance of an element is the error bound of tests/xref.py computed from the shape; zeros must match
exactly.  Each check prints one ELEMENTWISE line (largest relative error, and the bound at that shape) under `pytest -s`."""
import ctypes as C

import numpy as np
import pytest

from gbrs_b200 import _lib, synth
from gbrs_b200.emfactory import DevicePattern, EMfactory, PackedPattern
from oracle import em_oracle as eo
from tests import layouts
from tests import xref as xr

pytestmark = pytest.mark.gpu

ITEM_LEN = 16
MODELS = (4, 3, 2, 1)
# the default tile caps hold classes of up to 16 loci; the constructed layouts have a class of 40
PATHS = {"two-pass": {}, "entry64": {}, "tiles": dict(tiles=True, tile_params=dict(max_loci=48, max_items=192)),
         "tiles-tiny": dict(tiles=True, tile_params=dict(max_classes=40, max_loci=48, max_items=96, item_len=4))}


def check(got, want, rtol, what, where=None):
    err = xr.assert_elementwise(got, want, rtol, what, where)
    print(f"ELEMENTWISE {what}: max rel err {err:.3e}, bound {float(np.min(rtol)):.3e}..{float(np.max(rtol)):.3e}")


def problem(H, item_len=ITEM_LEN):
    xr.require_longdouble()
    d = layouts.make_layout(H, item_len)
    gene_of = eo.gene_index(d.T, d.groups())
    return d, gene_of, xr.XRef(d, gene_of), eo.effective_length_table(d.lengths)


def factory(d, **kw):
    em = EMfactory(synth.to_apm(d), **kw)
    em.target_lengths = synth.effective_lengths(d)
    em.prepare()
    return em


def host_packed(d, gene_of, item_len=ITEM_LEN):
    return PackedPattern(synth.to_apm(d), gene_of=gene_of, item_len=item_len)


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("H", range(1, 9))
def test_gpu_one_update_elementwise(H, path, monkeypatch):
    """prepare(), then per model from one random theta: a stand-alone E-step and one update_allelic_expression."""
    if path == "entry64":
        monkeypatch.setenv("GBRS_FORCE_ENTRY64", "1")
    d, gene_of, x, eff = problem(H)
    em = factory(d, item_len=ITEM_LEN, **PATHS[path])
    pat = em._pattern
    layouts.assert_layout_covers(pat.packed)
    assert pat.info["entry_bytes"] == (8 if path == "entry64" else 4)
    assert (pat.tiled is not None) == path.startswith("tiles")
    where = layouts.locus_kinds(pat.packed)
    check(em.get_allelic_expression(), x.prepare(eff), x.rtol_prepare(), f"H={H} {path} theta0", where)
    theta = xr.random_theta(x, seed=H)
    for model in MODELS:
        counts, theta1 = x.update(theta, model, eff)
        rtol = x.rtol_update(model)
        em.allelic_expression = theta
        em.update_probability_at_read_level(model=model)
        check(em.expected_read_counts(), counts, rtol, f"H={H} {path} model {model} E-step counts", where)
        em.allelic_expression = theta
        em.update_allelic_expression(model=model)
        check(em.expected_read_counts(), counts, rtol, f"H={H} {path} model {model} counts", where)
        check(em.allelic_expression, theta1, rtol, f"H={H} {path} model {model} theta", where)
        assert not em.allelic_expression[:, d.zero_locus].any()


@pytest.mark.parametrize("R", [2, 3])
@pytest.mark.parametrize("H", range(1, 9))
def test_gpu_row_shards_one_update_elementwise(H, R):
    """R row shards on one GPU (the sequence of tests/test_sharded_gpu.run_sharded, numerators summed by hand): one update
    of every model from one random theta."""
    import torch

    d, gene_of, x, eff = problem(H)
    layouts.assert_layout_covers(host_packed(d, gene_of))
    apm = synth.to_apm(d)
    pats = [DevicePattern(apm, gene_of=gene_of, shard_rank=r, shard_count=R, item_len=ITEM_LEN) for r in range(R)]
    lib = pats[0].lib
    for p in pats:
        p.set_lengths(synth.effective_lengths(d))
        p.ensure_full(1)

    def exchange():
        total = torch.zeros_like(pats[0].acc)
        for p in pats:
            total += p.acc
        for p in pats:
            p.acc.copy_(total)

    for p in pats:
        _lib.check(lib.gbrs_em_prepare_local(C.byref(p.desc), p.stream()))
    exchange()
    for p in pats:
        _lib.check(lib.gbrs_em_prepare_finish(C.byref(p.desc), 0.0, p.stream()))
    theta = xr.random_theta(x, seed=10 + H)
    for model in MODELS:
        for p in pats:
            p.set_theta_HT(theta)
            _lib.check(lib.gbrs_em_run_begin(C.byref(p.desc), 0.0, 1, p.stream()))
            _lib.check(lib.gbrs_em_launch_local(C.byref(p.desc), model, p.stream()))
        exchange()
        for p in pats:
            _lib.check(lib.gbrs_em_launch_update(C.byref(p.desc), p.stream()))
            assert int(p.read_ctrl()[0][_lib.CTRL_ERROR]) == 0
        counts, theta1 = x.update(theta, model, eff)
        rtol = x.rtol_update(model)
        check(pats[0].acc_HT(), counts, rtol, f"H={H} R={R} model {model} counts")
        for p in pats:
            check(p.current_theta_HT(), theta1, rtol, f"H={H} R={R} model {model} theta")


@pytest.mark.parametrize("H", range(1, 9))
def test_gpu_run_to_convergence_elementwise(H):
    """run(): the same number of iterations as the reference, the error trajectory to 1e-7, theta and the expected counts
    element-wise within the bound of that many updates after prepare() with a pseudocount."""
    d, gene_of, x, eff = problem(H)
    model = MODELS[H % 4]
    em = EMfactory(synth.to_apm(d), item_len=ITEM_LEN)
    em.target_lengths = synth.effective_lengths(d)
    em.prepare(pseudocount=0.25)
    layouts.assert_layout_covers(em._pattern.packed)
    em.run(model=model, tol=1e-5, max_iters=400, verbose=False)
    want = x.run(x.prepare(eff, 0.25), model, eff, 1e-5, 400)
    assert em.num_iters == want["iters"] < 400
    np.testing.assert_allclose(em.err_history, want["errs"], rtol=1e-7, atol=1e-7)
    rtol = x.rtol_run(model, want["iters"], pseudocount=0.25)
    where = layouts.locus_kinds(em._pattern.packed)
    check(em.allelic_expression, want["theta"], rtol, f"H={H} run model {model} ({want['iters']} updates) theta", where)
    check(em.expected_read_counts(), want["counts"], rtol, f"H={H} run model {model} counts", where)
