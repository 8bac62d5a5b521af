"""Genes whose loci interleave in locus order (tests/interleaved.py) on the device: the device packer's rows, runs and
entries against the input and bit for bit against the host packer; every output element of the gene-aware EM paths
against the extended-precision reference of tests/xref.py (one update and a stand-alone E-step of models 1-3 with model 4
as a control, two-pass kernels and 64-bit entry words, row shards, run() to convergence,
a relabelling of the loci); the posterior, the gene-level alignment counts, bootstrap replicates, and `quantify` end to
end with the group file written out, with and without a genotype file.  Each check prints one ELEMENTWISE line under
`pytest -s`."""
import ctypes as C
import time

import numpy as np
import pytest

from gbrs_b200 import _lib, synth
from gbrs_b200.emfactory import DevicePacked, DevicePattern, EMfactory, PackedPattern
from gbrs_b200.quantify import hapmask_bytes, quantify
from oracle import em_oracle as eo
from tests import interleaved as il
from tests import layouts
from tests import posterior_checks as pc
from tests import xref as xr
from tests.test_bootstrap_gpu import check_replicates
from tests.test_interleaved_genes import check_relabelled_run, relabelled_layout, shard_counts
from tests.test_pack import _assert_same_pack
from tests.test_quantify_gpu import read_table

pytestmark = pytest.mark.gpu

ITEM_LEN = 16
MODELS = (4, 3, 2, 1)


def check(got, want, rtol, what):
    err = xr.assert_elementwise(got, want, rtol, what)
    print(f"ELEMENTWISE {what}: max rel err {err:.3e}, bound {float(np.min(rtol)):.3e}..{float(np.max(rtol)):.3e}")


def problem(H, seed=0):
    xr.require_longdouble()
    d = il.interleave(layouts.make_layout(H, ITEM_LEN), seed=H + seed)
    gene_of = il.gene_ids(d)
    return d, gene_of, xr.XRef(d, gene_of), eo.effective_length_table(d.lengths)


def factory(d, pseudocount=0.0, **kw):
    em = EMfactory(synth.to_apm(d), item_len=ITEM_LEN, **kw)
    em.target_lengths = synth.effective_lengths(d)
    em.prepare(pseudocount=pseudocount)
    return em


def covers(d, packed):
    layouts.assert_layout_covers(packed)
    il.assert_genes_interleave(d, packed)


# ---- the device packer ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H", range(1, 9))
def test_device_packer_sorts_rows_by_gene_and_cuts_runs(H, monkeypatch):
    d, gene_of, _, _ = problem(H)
    apm = synth.to_apm(d)
    for entry64 in (False, True):
        if entry64:
            monkeypatch.setenv("GBRS_FORCE_ENTRY64", "1")
        dp = DevicePacked(apm, "cuda:0", gene_of=gene_of, item_len=ITEM_LEN)
        assert dp.info["entry_bytes"] == (8 if entry64 else 4)
        covers(d, dp)
        arrays = dp.to_host()
        il.assert_packed_structure(d, dp.info, arrays)
        _assert_same_pack(dp.info, arrays, PackedPattern(apm, gene_of=gene_of, item_len=ITEM_LEN))


def test_device_packer_at_the_c2_locus_shape():
    """1M classes over 80k loci, genes interleaved: host == device bit for bit; the device packer's time next to the same
    input with contiguous genes (its per-class insertion sort is quadratic in the width when genes descend)"""
    import torch

    d0 = synth.generate(T=80_000, N=1_000_000, H=8)
    d = il.interleave(d0, seed=3)
    times = {}
    for what, dd in (("contiguous", d0), ("interleaved", d)):
        apm, gene_of = synth.to_apm(dd), il.gene_ids(dd)
        best = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dp = DevicePacked(apm, "cuda:0", gene_of=gene_of)
            torch.cuda.synchronize()
            best.append(time.perf_counter() - t0)
        times[what] = min(best)
        if what == "interleaved":
            _assert_same_pack(dp.info, dp.to_host(), PackedPattern(apm, gene_of=gene_of))
    print(f"PACKTIME device packer, {torch.cuda.get_device_name(0)}, 80k loci x 1M classes: "
          f"contiguous genes {times['contiguous'] * 1e3:.1f} ms, interleaved genes {times['interleaved'] * 1e3:.1f} ms")


# ---- EM element-wise --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["two-pass", "entry64"])
@pytest.mark.parametrize("H", range(1, 9))
def test_gpu_one_update_elementwise(H, path, monkeypatch):
    """prepare(), then per model from one random theta: a stand-alone E-step and one update_allelic_expression"""
    if path == "entry64":
        monkeypatch.setenv("GBRS_FORCE_ENTRY64", "1")
    d, gene_of, x, eff = problem(H)
    em = factory(d)
    covers(d, em._pattern.packed)
    assert em._pattern.info["entry_bytes"] == (8 if path == "entry64" else 4)
    check(em.get_allelic_expression(), x.prepare(eff), x.rtol_prepare(), f"interleaved H={H} {path} theta0")
    theta = xr.random_theta(x, seed=H)
    for model in MODELS:
        counts, theta1 = x.update(theta, model, eff)
        rtol = x.rtol_update(model)
        em.allelic_expression = theta
        em.update_probability_at_read_level(model=model)
        check(em.expected_read_counts(), counts, rtol, f"interleaved H={H} {path} model {model} E-step counts")
        em.allelic_expression = theta
        em.update_allelic_expression(model=model)
        check(em.expected_read_counts(), counts, rtol, f"interleaved H={H} {path} model {model} counts")
        check(em.allelic_expression, theta1, rtol, f"interleaved H={H} {path} model {model} theta")
        assert not em.allelic_expression[:, d.zero_locus].any()


@pytest.mark.parametrize("H", range(1, 9))
def test_gpu_run_to_convergence_elementwise(H):
    d, gene_of, x, eff = problem(H)
    model = (3, 2, 1)[H % 3]
    em = factory(d, pseudocount=0.25)
    covers(d, em._pattern.packed)
    em.run(model=model, tol=1e-5, max_iters=400, verbose=False)
    want = x.run(x.prepare(eff, 0.25), model, eff, 1e-5, 400)
    assert em.num_iters == want["iters"] < 400
    np.testing.assert_allclose(em.err_history, want["errs"], rtol=1e-7, atol=1e-7)
    rtol = x.rtol_run(model, want["iters"], pseudocount=0.25)
    check(em.allelic_expression, want["theta"], rtol, f"interleaved H={H} run model {model} ({want['iters']} updates) theta")
    check(em.expected_read_counts(), want["counts"], rtol, f"interleaved H={H} run model {model} counts")


@pytest.mark.parametrize("R", [2, 3])
@pytest.mark.parametrize("H", [2, 5, 8])
def test_gpu_row_shards_one_update_elementwise(H, R):
    import torch

    d, gene_of, x, eff = problem(H)
    apm = synth.to_apm(d)
    covers(d, PackedPattern(apm, gene_of=gene_of, item_len=ITEM_LEN))
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
        for r, p in enumerate(pats):  # each shard's own numerator, before the exchange sums them
            want = shard_counts(x, theta, model, il._host_arrays(p.packed)["class_id"])
            check(p.acc_HT(), want, x.rtol_update(model), f"interleaved H={H} R={R} shard {r} model {model} local counts")
        exchange()
        for p in pats:
            _lib.check(lib.gbrs_em_launch_update(C.byref(p.desc), p.stream()))
            assert int(p.read_ctrl()[0][_lib.CTRL_ERROR]) == 0
        counts, theta1 = x.update(theta, model, eff)
        rtol = x.rtol_update(model)
        check(pats[0].acc_HT(), counts, rtol, f"interleaved H={H} R={R} model {model} counts")
        for p in pats:
            check(p.current_theta_HT(), theta1, rtol, f"interleaved H={H} R={R} model {model} theta")


@pytest.mark.parametrize("model", [3, 2, 1])
def test_gpu_relabelled_loci_give_the_permuted_run(model):
    """a contiguous-gene problem and the same problem with its loci relabelled (its genes then interleave): the same
    iteration count, theta and counts the permuted ones within the bound"""
    xr.require_longdouble()
    d, e, perm = relabelled_layout()

    def run(dd):
        em = factory(dd, pseudocount=0.5)
        layouts.assert_layout_covers(em._pattern.packed)
        em.run(model=model, tol=1e-4, max_iters=400, verbose=False)
        return dict(iters=em.num_iters, theta=em.allelic_expression.copy(), counts=em.expected_read_counts().copy())

    iters = check_relabelled_run(run, d, e, perm, model)
    assert iters < 400
    print(f"ELEMENTWISE interleaved relabelled loci model {model} ({iters} updates): theta and counts within twice the bound")


# ---- the other gene-aware outputs -------------------------------------------------------------------------------------
@pytest.mark.parametrize("H", range(1, 9))
def test_gpu_posterior_elementwise(H):
    """posterior_probability() after a stand-alone E-step of every model from a random theta"""
    d, gene_of, x, eff = problem(H)
    em = factory(d)
    covers(d, em._pattern.packed)
    theta = xr.random_theta(x, seed=40 + H)
    for model in MODELS:
        em.allelic_expression = theta
        em.update_probability_at_read_level(model=model)
        got = pc.apm_entry_values(em.posterior_probability(), x)
        pc.check(got, x.e_step(theta, model), pc.rtol_posterior(x, model), f"interleaved H={H} model {model} posterior")


@pytest.mark.parametrize("H", [1, 2, 5, 8])
def test_gpu_gene_level_alignment_counts(H):
    """bit-exact against the reference's bundle-then-count; ungrouped loci between grouped ones vanish.  (The count
    pattern the product packs itself, from the group file, is checked by test_quantify_end_to_end.)"""
    d, gene_of, _, _ = problem(H)
    groups = d.groups()
    apm = synth.to_apm(d)
    pattern = DevicePattern(apm, gene_of=gene_of, item_len=ITEM_LEN)  # (the item length the layout is built for)
    covers(d, pattern.packed)
    aln, uniq, lu = apm._alignment_count_tables(gene_level=True, pattern=pattern)
    assert aln.shape == (d.H, len(groups)) and int(gene_of.max()) + 1 > len(groups)
    want = eo.alignment_counts(eo.bundle(eo.apm_from_pairs(d.T, d.H, d.N, d.pair_class, d.pair_locus, d.pair_mask,
                                                           d.count), groups))
    assert np.array_equal(aln, want["aln"]) and np.array_equal(uniq, want["uniq"])
    assert np.array_equal(lu, want["locus_uniq"])


@pytest.mark.parametrize("model", [3, 2, 1])
@pytest.mark.parametrize("H", [2, 8])
def test_gpu_bootstrap_replicate_elementwise(H, model):
    d, _, _, _ = problem(H)
    em = factory(d)
    covers(d, em._pattern.packed)
    check_replicates(d, em.bootstrap([1], model=model, seed=5, tol=1e-3, max_iters=60), model,
                     what=f"interleaved H={H} model {model}")


# ---- quantify end to end ----------------------------------------------------------------------------------------------
def reference_tables(d, model, gtmask):
    """the reference's quantify tables of `d` in long double (xref's run, grouping as the reference's grp_conv_mat: a
    locus listed twice in a group counts once) and the bound of one of their elements"""
    gene_of = il.gene_ids(d)
    groups = [sorted(set(g)) for g in d.groups()]
    x = xr.XRef(d, gene_of, gtmask)
    eff = eo.effective_length_table(d.lengths)
    o = x.run(x.prepare(eff), model, eff, 1e-4, 999)
    theta, counts = o["theta"], o["counts"]

    def gsum(m):
        return np.stack([m[:, g].sum(axis=1) for g in groups], axis=1)

    iso_tpm = theta * (xr.LD(1e6) / theta.sum())
    gene_tpm = gsum(iso_tpm)
    gene_tpm = gene_tpm * (xr.LD(1e6) / gene_tpm.sum())
    tables = {"isoforms.tpm": iso_tpm, "isoforms.expected_read_counts": counts, "genes.tpm": gene_tpm,
              "genes.expected_read_counts": gsum(counts)}
    rtol = float(np.max(x.rtol_run(model, o["iters"]))) + xr.SAFETY * (d.H * d.T + 2 * x.g_max + xr.C_OPS) * xr.U
    oapm = eo.apm_from_pairs(d.T, d.H, d.N, d.pair_class, d.pair_locus, d.pair_mask, d.count)
    exact = {"isoforms.alignment_counts": eo.alignment_counts(oapm),
             "genes.alignment_counts": eo.alignment_counts(eo.bundle(oapm, d.groups()))}
    return tables, exact, rtol, o["iters"]


@pytest.mark.parametrize("model,genotype", [(1, False), (2, False), (3, False), (3, True), (1, True)])
def test_quantify_end_to_end(model, genotype, tmp_path, capsys):
    d = il.interleave(synth.generate(T=300, N=4000, H=8, sample_index=6, wide_frac=0.03, wide_max=40), seed=model)
    p = PackedPattern(synth.to_apm(d), gene_of=il.gene_ids(d))
    assert all(il.interleave_summary(d, p.arrays)["split"].get(K) for K in (3, 4, 5))
    paths = {k: str(tmp_path / f"{k}.tsv") for k in ("grp", "len", "gt")}
    synth.write_group_file(d, paths["grp"])
    synth.write_length_file(d, paths["len"])
    synth.write_genotype_file(d, paths["gt"])
    aln = str(tmp_path / "aln.emase")
    synth.to_apm(d).save(aln)
    outbase = str(tmp_path / "out")
    capsys.readouterr()
    quantify(alignment_file=aln, group_file=paths["grp"], length_file=paths["len"],
             genotype_file=paths["gt"] if genotype else None, outbase=outbase, multiread_model=model,
             report_alignment_counts=True)
    iters = sum("/ 1000000" in line for line in capsys.readouterr().out.splitlines())
    gtmask = synth.genotype_mask(d) if genotype else None
    if genotype:  # what the EM ran on: a genotype restriction per listed gene, ungrouped loci removed entirely
        assert not gtmask[:, ~np.isin(np.arange(d.T), np.concatenate(d.groups()))].any()
    tables, exact, rtol, want_iters = reference_tables(d, model, gtmask)
    assert iters == want_iters
    kind = "diploid" if genotype else "multiway"
    for sfx, want in tables.items():
        header, names, got, _ = read_table(f"{outbase}.{kind}.{sfx}")
        assert header[1:1 + d.H] == list(d.hname) and header[1 + d.H] == "total"
        assert names == (list(d.gname) if sfx.startswith("genes") else list(d.lname)), sfx
        want_full = np.vstack([want, want.sum(axis=0, keepdims=True)])
        check(got.T, want_full, rtol, f"interleaved quantify model {model} {kind} {sfx}")
    for sfx, want in exact.items():
        _, names, got, _ = read_table(f"{outbase}.{kind}.{sfx}")
        assert names == (list(d.gname) if sfx.startswith("genes") else list(d.lname)), sfx
        assert np.array_equal(got, np.hstack([want["aln"].T, want["uniq"].T, want["locus_uniq"][:, None]])), sfx
