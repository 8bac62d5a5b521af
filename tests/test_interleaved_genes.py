"""Genes whose loci interleave in locus order (tests/interleaved.py), on the CPU: the packed rows, runs and entries of the
host packer and of the device packer (run through the host SIMT shim) against the input, and the gene-aware kernels of
the EM library (tests/simt_em.py) element by element against the extended-precision reference of tests/xref.py: one
update and a stand-alone E-step of models 1-3 (model 4 as a control), row shards, run() to convergence, a relabelling of
the loci, the posterior, the gene-level alignment counts and a bootstrap replicate.

Every test calls tests/layouts.assert_layout_covers and tests/interleaved.assert_genes_interleave on the pattern it
runs, so the interleaving reaches every fixed-width row pass and both row-pointer widths."""
import ctypes as C
import dataclasses
import shutil

import numpy as np
import pytest

from gbrs_b200 import synth
from gbrs_b200.emfactory import PackedPattern, posterior_pattern
from oracle import em_oracle as eo
from tests import boot_ref as br
from tests import interleaved as il
from tests import layouts, simt_em, simt_posterior
from tests import posterior_checks as pc
from tests import xref as xr
from tests.test_bootstrap import emulated_replicate
from tests.test_pack import _assert_same_pack

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ is needed to build the SIMT emulation")

ITEM_LEN = 16
MODELS = (4, 3, 2, 1)


def problem(H, seed=0):
    xr.require_longdouble()
    d = il.interleave(layouts.make_layout(H, ITEM_LEN), seed=H + seed)
    gene_of = il.gene_ids(d)
    return d, gene_of, xr.XRef(d, gene_of), eo.effective_length_table(d.lengths)


def covers(d, packed):
    layouts.assert_layout_covers(packed)
    il.assert_genes_interleave(d, packed)


def shard_counts(x, theta, model, classes):
    """expected read counts of the input classes `classes` alone (one row shard's numerator before the exchange)"""
    keep = np.zeros(x.N, dtype=bool)
    keep[np.asarray(classes, dtype=np.int64)] = True
    val = x.e_step(theta, model) * np.where(keep[x.n], x.count[x.n], xr.LD(0))
    out = np.zeros(x.H * x.T, dtype=xr.LD)
    out[x.by_ht.keys] = x.by_ht.sums(val)
    return out.reshape(x.H, x.T)


def T8(theta_HT, T):
    out = np.zeros((T, 8))
    out[:, : theta_HT.shape[0]] = theta_HT.T
    return out


# ---- packed structure -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H", range(1, 9))
def test_host_packer_sorts_rows_by_gene_and_cuts_runs(H):
    d, gene_of, _, _ = problem(H)
    p = PackedPattern(synth.to_apm(d), gene_of=gene_of, item_len=ITEM_LEN)
    covers(d, p)
    il.assert_packed_structure(d, p.info, p.arrays)


@pytest.mark.parametrize("entry64", [False, True], ids=["entry32", "entry64"])
@pytest.mark.parametrize("H", [2, 8])
def test_emulated_device_packer_sorts_rows_by_gene_and_cuts_runs(H, entry64, monkeypatch):
    """gpu_pack.cu through the host shim: the structure against the input, and every array bit-identical to the host
    packer's, at 32- and 64-bit entry words."""
    if entry64:
        monkeypatch.setenv("GBRS_FORCE_ENTRY64", "1")
    d, gene_of, _, _ = problem(H)
    apm = synth.to_apm(d)
    info, arrays = simt_em.emulated_device_pack(apm, gene_of=gene_of, item_len=ITEM_LEN)
    arrays["class_id"] = simt_posterior.emulated_device_class_id(apm, gene_of=gene_of)
    assert info["entry_bytes"] == (8 if entry64 else 4)
    host = PackedPattern(apm, gene_of=gene_of, item_len=ITEM_LEN)
    covers(d, host)
    il.assert_packed_structure(d, info, arrays)
    _assert_same_pack(info, arrays, host)


def test_constructor_on_a_generated_problem():
    """interleave() also takes synth.generate's shapes (no zero locus, not every width): every split width the input has
    gets a split gene, and the packed structure holds with and without a -G restriction"""
    from gbrs_b200.quantify import hapmask_bytes

    d = il.interleave(synth.generate(T=300, N=4000, H=8, sample_index=3, wide_frac=0.02, wide_max=40), seed=1)
    gene_of = il.gene_ids(d)
    hm = hapmask_bytes(synth.genotype_mask(d))
    for hapmask in (None, hm):
        p = PackedPattern(synth.to_apm(d), gene_of=gene_of, hapmask=hapmask)
        il.assert_packed_structure(d, p.info, p.arrays, hapmask=hapmask)
    s = il.interleave_summary(d, PackedPattern(synth.to_apm(d), gene_of=gene_of).arrays)
    present = [K for K in il.SPLIT_WIDTHS if K in s["split"]]
    assert set(present) >= {3, 4, 5, 6, 9} and all(s["split"][K] for K in present), s


# ---- EM element-wise --------------------------------------------------------------------------------------------------
def one_update_each_model(pat, d, x, eff, theta, what, where, estep=True):
    """per model from `theta`: a stand-alone E-step (counts) and one update (counts and theta), element-wise"""
    tb = T8(theta, d.T)
    for model in MODELS:
        counts, theta1 = x.update(theta, model, eff)
        rtol = x.rtol_update(model)
        if estep:
            pat.check(pat.lib.gbrs_em_set_theta(C.byref(pat.desc), tb.ctypes.data, None))
            pat.check(pat.lib.gbrs_em_run_begin(C.byref(pat.desc), 0.0, 1, None))
            pat.check(pat.lib.gbrs_em_launch_estep(C.byref(pat.desc), model, None))
            xr.assert_elementwise(pat.acc[:, : d.H].T, counts, rtol, f"{what} model {model} E-step counts", where)
        pat.check(pat.lib.gbrs_em_set_theta(C.byref(pat.desc), tb.ctypes.data, None))
        out = pat.run(model, tol=0.0, max_iters=1)
        xr.assert_elementwise(out["counts"], counts, rtol, f"{what} model {model} counts", where)
        xr.assert_elementwise(out["theta"], theta1, rtol, f"{what} model {model} theta", where)
        assert not out["counts"][:, d.zero_locus].any()


@pytest.mark.parametrize("H", range(1, 9))
def test_emulated_one_update_elementwise(H):
    d, gene_of, x, eff = problem(H)
    pat = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of, item_len=ITEM_LEN)
    covers(d, pat.packed)
    where = layouts.locus_kinds(pat.packed)
    xr.assert_elementwise(pat.prepare(eff), x.prepare(eff), x.rtol_prepare(), f"H={H} theta0", where)
    one_update_each_model(pat, d, x, eff, xr.random_theta(x, seed=H), f"H={H}", where)


@pytest.mark.parametrize("H", [3, 8])
def test_emulated_one_update_elementwise_entry64(H, monkeypatch):
    monkeypatch.setenv("GBRS_FORCE_ENTRY64", "1")
    d, gene_of, x, eff = problem(H)
    pat = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of, item_len=ITEM_LEN)
    assert pat.info["entry_bytes"] == 8
    covers(d, pat.packed)
    pat.prepare(eff)
    one_update_each_model(pat, d, x, eff, xr.random_theta(x, seed=30 + H), f"H={H} entry64", None, estep=False)


@pytest.mark.parametrize("R", [2, 3])
def test_emulated_row_shards_one_update_elementwise(R):
    """R row shards, numerators summed by hand: one update of every model, every shard holding the same theta'"""
    H = 8 if R == 2 else 5
    d, gene_of, x, eff = problem(H)
    apm = synth.to_apm(d)
    covers(d, PackedPattern(apm, gene_of=gene_of, item_len=ITEM_LEN))
    pats = [simt_em.HostPattern(apm, gene_of=gene_of, item_len=ITEM_LEN, shard_rank=r, shard_count=R) for r in range(R)]
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
    theta = xr.random_theta(x, seed=10 + H)
    tb = T8(theta, d.T)
    for model in MODELS:
        for p in pats:
            p.check(lib.gbrs_em_set_theta(C.byref(p.desc), tb.ctypes.data, None))
            p.check(lib.gbrs_em_run_begin(C.byref(p.desc), 0.0, 1, None))
            p.check(lib.gbrs_em_launch_local(C.byref(p.desc), model, None))
        counts, theta1 = x.update(theta, model, eff)
        rtol = x.rtol_update(model)
        for r, p in enumerate(pats):  # each shard's own numerator, before the exchange sums them
            want = shard_counts(x, theta, model, p.packed.arrays["class_id"])
            xr.assert_elementwise(p.acc[:, : d.H].T, want, rtol, f"R={R} shard {r} model {model} local counts")
        exchange()
        for p in pats:
            p.check(lib.gbrs_em_launch_update(C.byref(p.desc), None))
        xr.assert_elementwise(pats[0].acc[:, : d.H].T, counts, rtol, f"R={R} model {model} counts")
        for p in pats:
            xr.assert_elementwise(p.current_theta(), theta1, rtol, f"R={R} model {model} theta")


@pytest.mark.parametrize("H", [2, 7])
def test_emulated_run_to_convergence_elementwise(H):
    """prepare() with a pseudocount, run(): the reference's iteration count, its error log to 1e-7, theta and counts
    within the bound of that many updates"""
    d, gene_of, x, eff = problem(H)
    model = (2, 3)[H % 2]
    pat = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of, item_len=ITEM_LEN)
    covers(d, pat.packed)
    pat.prepare(eff, 0.25)
    out = pat.run(model, tol=1e-5, max_iters=400)
    want = x.run(x.prepare(eff, 0.25), model, eff, 1e-5, 400)
    assert out["iters"] == want["iters"] < 400
    np.testing.assert_allclose(out["errs"], want["errs"], rtol=1e-7, atol=1e-7)
    rtol = x.rtol_run(model, want["iters"], pseudocount=0.25)
    xr.assert_elementwise(out["theta"], want["theta"], rtol, f"H={H} run model {model} theta")
    xr.assert_elementwise(out["counts"], want["counts"], rtol, f"H={H} run model {model} counts")


def relabel_loci(d, seed):
    """`d` with locus t renamed perm[t] (a random permutation): the same problem, with its genes interleaved.  Returns
    (relabelled data, perm)."""
    perm = np.random.default_rng(seed).permutation(d.T)
    inv = np.argsort(perm)
    out = il.InterleavedSynth(**{f.name: getattr(d, f.name) for f in dataclasses.fields(synth.SynthData)},
                              group_lists=[[int(perm[t]) for t in g] for g in d.groups()])
    out.pair_locus = perm[np.asarray(d.pair_locus)]
    out.lengths = np.asarray(d.lengths)[inv]
    out.lname = [d.lname[t] for t in inv]
    out.gname = list(d.gname)
    out.gene_of = il.gene_ids(out)
    return out, perm


RELABEL_H, RELABEL_SEED = 8, 3  # a permutation of the 8-haplotype layout that splits a gene at every width in SPLIT_WIDTHS


def relabelled_layout():
    """(contiguous-gene layout, its relabelled copy, perm); the copy reaches every kernel path and every width's sort"""
    d = layouts.make_layout(RELABEL_H, ITEM_LEN)
    e, perm = relabel_loci(d, RELABEL_SEED)
    covers(e, PackedPattern(synth.to_apm(e), gene_of=il.gene_ids(e), item_len=ITEM_LEN))
    return d, e, perm


def check_relabelled_run(run, d, e, perm, model):
    """run(d) and run(e), e = d with its loci relabelled by perm: the same iteration count, theta and counts the permuted
    ones.  No reference is involved: each run carries its own rounding error of at most the bound of that many updates
    (tests/xref.py) relative to the exact result, so the two differ by at most twice that bound."""
    a, b = run(d), run(e)
    assert a["iters"] == b["iters"]
    x = xr.XRef(d, il.gene_ids(d))
    rtol = 2 * x.rtol_run(model, a["iters"], pseudocount=0.5)
    xr.assert_elementwise(b["theta"][:, perm], a["theta"], rtol, f"model {model} relabelled theta")
    xr.assert_elementwise(b["counts"][:, perm], a["counts"], rtol, f"model {model} relabelled counts")
    return a["iters"]


@pytest.mark.parametrize("model", [3, 1])
def test_emulated_relabelled_loci_give_the_permuted_run(model):
    xr.require_longdouble()
    d, e, perm = relabelled_layout()

    def run(dd):
        pat = simt_em.HostPattern(synth.to_apm(dd), gene_of=il.gene_ids(dd), item_len=ITEM_LEN)
        pat.prepare(eo.effective_length_table(dd.lengths), 0.5)
        return pat.run(model, tol=1e-4, max_iters=400)

    assert check_relabelled_run(run, d, e, perm, model) < 400


# ---- the other gene-aware outputs -------------------------------------------------------------------------------------
@pytest.mark.parametrize("H", [2, 8])
def test_emulated_posterior_elementwise(H):
    """gbrs_em_posterior of models 1-3 (and 4) from a random theta, element-wise against the reference's E-step"""
    d, gene_of, x, eff = problem(H)
    apm = synth.to_apm(d)
    pat = simt_posterior.PosteriorHostPattern(apm, gene_of=gene_of, item_len=ITEM_LEN)
    covers(d, pat.packed)
    pat.prepare(eff)
    theta = xr.random_theta(x, seed=40 + H)
    ip, ix = pc.pattern_arrays(posterior_pattern(apm, None))
    for model in MODELS:
        got = pc.entry_values(pat.posterior(model, T8(theta, d.T), ip, ix), ip, ix, x)
        xr.assert_elementwise(np.asarray(got)[None, :], x.e_step(theta, model)[None, :], pc.rtol_posterior(x, model),
                              f"H={H} model {model} posterior")


@pytest.mark.parametrize("H", [1, 4, 8])
def test_emulated_gene_level_alignment_counts(H):
    """gbrs_em_alignment_counts at gene level, bit-exact against the reference's bundle-then-count: ungrouped loci
    scattered between grouped ones vanish, and n_real_genes is below the number of gene ids"""
    d, gene_of, _, _ = problem(H)
    groups = d.groups()
    assert int(gene_of.max()) + 1 > len(groups)
    pat = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of, item_len=ITEM_LEN)
    covers(d, pat.packed)
    oapm = eo.apm_from_pairs(d.T, d.H, d.N, d.pair_class, d.pair_locus, d.pair_mask, d.count)
    aln, uniq, lu = pat.alignment_counts(gene_level=True, n_real_genes=len(groups))
    want = eo.alignment_counts(eo.bundle(oapm, groups))
    assert np.array_equal(aln, want["aln"]) and np.array_equal(uniq, want["uniq"])
    assert np.array_equal(lu, want["locus_uniq"])


@pytest.mark.parametrize("model", [3, 2, 1])
def test_emulated_bootstrap_replicate_elementwise(model):
    """one replicate: the reference's run on the compacted matrix, same iteration count, every element within the bound"""
    d, gene_of, _, eff = problem(4)
    covers(d, PackedPattern(synth.to_apm(d), gene_of=gene_of, item_len=ITEM_LEN))
    seed = 5 + model
    out = emulated_replicate(d, gene_of, seed, 0, model)
    dc = br.compact_synth(d, br.resample(d.count, seed, 0))
    assert isinstance(dc, il.InterleavedSynth) and dc.groups() == d.groups()
    x = xr.XRef(dc, gene_of)
    o = x.run(x.prepare(eff), model, eff, 1e-3, 60)
    assert out["iters"] == o["iters"]
    rtol = x.rtol_run(model, o["iters"])
    xr.assert_elementwise(out["theta"], o["theta"], rtol, f"model {model} replicate theta")
    xr.assert_elementwise(out["counts"], o["counts"], rtol, f"model {model} replicate counts")
