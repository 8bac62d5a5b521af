"""EMfactory.bootstrap on the device: resampled counts bit-identical to the numpy reference (tests/boot_ref.py), every
replicate element by element against the extended-precision reference (tests/xref.py) on the compacted matrix, replicate
independence across calls, packers and layouts, the zero-count row pass, state invariance of the factory, the refusals,
the CLI, and C2 at full size against the float64 oracle."""
import ctypes as C
import os

import numpy as np
import pytest

from gbrs_b200 import _lib, synth
from gbrs_b200.emfactory import EMfactory
from gbrs_b200.quantify import hapmask_bytes
from oracle import em_oracle as eo
from tests import boot_ref as br
from tests import helpers as hp
from tests import layouts
from tests import xref as xr

pytestmark = pytest.mark.gpu

TOL, MAXIT = 1e-3, 60


def device_resample(count, seed, replicates, N=None):
    """gbrs_boot_guide + gbrs_boot_resample with the identity class_id -> [B][N] histograms (float64)"""
    import torch

    lib = _lib.load()
    c = br.counts_of(count, N if count is None else len(count))
    N = c.shape[0]
    prefix = torch.from_numpy(np.cumsum(c)).cuda()
    M = int(c.sum())
    cid = torch.arange(N, dtype=torch.int32).cuda()
    nbytes = C.c_int64()
    _lib.check(lib.gbrs_boot_scratch_bytes(N, C.byref(nbytes)))
    scratch = torch.full((int(nbytes.value),), 0xAB, dtype=torch.uint8, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.gbrs_boot_guide(prefix.data_ptr(), N, M, scratch.data_ptr(), int(nbytes.value), stream))
    out = torch.empty((len(replicates), N), dtype=torch.float64, device="cuda")
    for b, r in enumerate(replicates):
        _lib.check(lib.gbrs_boot_resample(prefix.data_ptr(), N, M, seed, r, cid.data_ptr(), N, scratch.data_ptr(),
                                          int(nbytes.value), out[b].data_ptr(), stream))
    return out.cpu().numpy()


def factory(d, pseudocount=0.0, **kw):
    em = EMfactory(synth.to_apm(d), item_len=16, **kw)
    em.target_lengths = synth.effective_lengths(d)
    em.prepare(pseudocount=pseudocount)
    return em


def check_replicates(d, res, model, pseudocount=0.0, gtmask=None, what=""):
    """each replicate against xref's run on the compacted matrix: same iteration count, every element within the bound"""
    xr.require_longdouble()
    gene_of = eo.gene_index(d.T, d.groups())
    eff = eo.effective_length_table(d.lengths)
    worst = 0.0
    for b, r in enumerate(res.replicates.tolist()):
        dc = br.compact_synth(d, br.resample(d.count, res.seed, r))
        x = xr.XRef(dc, gene_of, gtmask)
        o = x.run(x.prepare(eff, pseudocount), model, eff, TOL, MAXIT)
        assert res.num_iters[b] == o["iters"], (what, r, res.num_iters[b], o["iters"])
        rtol = x.rtol_run(model, o["iters"], pseudocount)
        worst = max(worst, xr.assert_elementwise(res.allelic_expression[b], o["theta"], rtol, f"{what} r={r} theta"),
                    xr.assert_elementwise(res.expected_read_counts[b], o["counts"], rtol, f"{what} r={r} counts"))
    print(f"ELEMENTWISE bootstrap {what}: worst relative error {worst:.2e}")


@pytest.mark.parametrize("seed", [0, 77, 0xDEADBEEF12345678])
def test_device_counts_equal_numpy(seed):
    cases = [np.array([3, 0, 5, 1, 7, 2, 0, 5], float), np.array([37.0]), np.array([1, 0, 2000, 1, 1], float),
             np.random.default_rng(seed & 0xFFFF).integers(0, 9, 20000).astype(float)]
    for count in cases:
        got = device_resample(count, seed, (0, 1, 0xFFFFFFFF))
        for b, r in enumerate((0, 1, 0xFFFFFFFF)):
            assert np.array_equal(got[b], br.resample(count, seed, r).astype(np.float64))
    got = device_resample(None, seed, (3,), N=1000)
    assert np.array_equal(got[0], br.resample(None, seed, 3, N=1000).astype(np.float64))


@pytest.mark.parametrize("H", range(1, 9))
def test_model4_replicates_match_xref(H):
    d = layouts.make_layout(H, 16)
    em = factory(d)
    check_replicates(d, em.bootstrap([0, 3], model=4, seed=H, tol=TOL, max_iters=MAXIT), 4, what=f"H={H} model 4")


@pytest.mark.parametrize("H", [2, 8])
@pytest.mark.parametrize("model", [1, 2, 3])
def test_models_1_to_3_replicates_match_xref(H, model):
    d = layouts.make_layout(H, 16)
    em = factory(d)
    check_replicates(d, em.bootstrap([1], model=model, seed=5, tol=TOL, max_iters=MAXIT), model, what=f"H={H} model {model}")


def replicate_path(path):
    """one replicate of model 4 on the 8-haplotype layout through `path`"""
    d = layouts.make_layout(8, 16)
    kw, pc, gtmask = {}, 0.0, None
    if path == "pseudocount":
        pc = 0.5
    elif path == "genotype":
        rng = np.random.default_rng(4)
        gtmask = np.zeros((d.H, d.T))
        for t in range(d.T):
            gtmask[rng.choice(d.H, 2, replace=False), t] = 1.0
        kw = dict(locus_hapmask=hapmask_bytes(gtmask))
    elif path == "host-packer":
        kw = dict(pack="host")
    em = factory(d, pseudocount=pc, **kw)
    assert em._pattern.info["entry_bytes"] == (8 if path == "entry64" else 4)
    assert em._pattern.on_device == (path != "host-packer")
    res = em.bootstrap([2], model=4, seed=9, pseudocount=pc, tol=TOL, max_iters=MAXIT)
    check_replicates(d, res, 4, pseudocount=pc, gtmask=gtmask, what=path)


@pytest.mark.parametrize("path", ["pseudocount", "genotype", "host-packer", "entry64"])
def test_replicate_paths_match_xref(path, monkeypatch):
    if path == "entry64":
        monkeypatch.setenv("GBRS_FORCE_ENTRY64", "1")
    replicate_path(path)


def test_replicates_do_not_depend_on_the_call_packer_or_layout():
    d = layouts.make_layout(8, 16)
    full = factory(d).bootstrap(8, seed=3, tol=TOL, max_iters=MAXIT)
    for kw in ({}, dict(pack="host"), dict(tiles=True, tile_params=dict(max_loci=48, max_items=192)), dict(tiles=False)):
        part = factory(d, **kw).bootstrap([5, 2], seed=3, tol=TOL, max_iters=MAXIT)
        assert part.replicates.tolist() == [5, 2]
        for b, r in enumerate((5, 2)):
            assert np.array_equal(part.allelic_expression[b], full.allelic_expression[r]), kw
            assert np.array_equal(part.expected_read_counts[b], full.expected_read_counts[r]), kw
            assert part.num_iters[b] == full.num_iters[r]


def test_replicate_dropping_the_only_class_of_a_locus():
    d = br.with_lonely_locus(synth.generate(T=300, N=4000, H=4, sample_index=2))
    seed = br.seed_dropping(d.count, d.N - 1)
    em = factory(d)
    res = em.bootstrap([0], model=4, seed=seed, tol=TOL, max_iters=MAXIT)
    assert not res.allelic_expression[0][:, d.T - 1].any() and not res.expected_read_counts[0][:, d.T - 1].any()
    check_replicates(d, res, 4, what="lonely locus")
    # the same counts on an ordinary factory (count-0 class present): model 4 still raises, as before
    d0 = br.with_lonely_locus(synth.generate(T=300, N=4000, H=4, sample_index=2))
    d0.count = br.resample(d.count, seed, 0).astype(np.float64)
    em0 = factory(d0)
    with pytest.raises(FloatingPointError):
        em0.run(model=4, tol=TOL, max_iters=MAXIT, verbose=False)


def test_bootstrap_leaves_the_factory_state_alone():
    d = layouts.make_layout(4, 16)
    em = factory(d)
    em.run(model=4, tol=TOL, max_iters=MAXIT, verbose=False)
    before = (em.get_allelic_expression(), em.expected_read_counts().copy(), em.num_iters, em.err_history.copy(),
              [m.data.copy() for m in em.posterior_probability().data])
    em.bootstrap(3, model=4, seed=1, tol=TOL, max_iters=MAXIT)
    em.bootstrap([4], model=2, seed=1, tol=TOL, max_iters=MAXIT)
    after = (em.get_allelic_expression(), em.expected_read_counts().copy(), em.num_iters, em.err_history.copy(),
             [m.data.copy() for m in em.posterior_probability().data])
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
    assert before[2] == after[2] and np.array_equal(before[3], after[3])
    assert all(np.array_equal(a, b) for a, b in zip(before[4], after[4]))
    ref = factory(d)
    ref.run(model=4, tol=TOL, max_iters=MAXIT, verbose=False)
    em.prepare()
    em.run(model=4, tol=TOL, max_iters=MAXIT, verbose=False)
    assert np.array_equal(em.get_allelic_expression(), ref.get_allelic_expression())
    assert np.array_equal(em.expected_read_counts(), ref.expected_read_counts())


def test_refusals():
    d = synth.generate(T=50, N=600, H=4)
    em = EMfactory(synth.to_apm(d))
    with pytest.raises(RuntimeError):
        em.bootstrap(2)  # no prepare()
    em.prepare()
    with pytest.raises(ValueError):
        em.bootstrap([2 ** 32])
    with pytest.raises(ValueError):
        em.bootstrap([-1])
    for bad in (np.where(np.arange(d.N) == 3, -1.0, d.count), d.count + 0.5, np.zeros(d.N)):
        apm = synth.to_apm(d)
        apm.count = bad
        e = EMfactory(apm)
        if bad.min() >= 0 and bad.sum() > 0:
            e.prepare()
        else:
            e._pattern, e._post = object(), ("incidence",)  # the checks come before any device work
        with pytest.raises(ValueError):
            e.bootstrap(1)
    apm = synth.to_apm(d)
    apm.count = np.full(d.N, 2.0 ** 44)
    e = EMfactory(apm)
    e.prepare()
    with pytest.raises(ValueError):
        e.bootstrap(1)  # 600 * 2^44 reads > 2^53
    apm = synth.to_apm(d)
    apm.data[0].data[:] = 0.5  # a weighted file
    e = EMfactory(apm)
    e.prepare()
    with pytest.raises(NotImplementedError):
        e.bootstrap(1)
    e = EMfactory(synth.to_apm(d), shard="local")
    e.prepare()
    with pytest.raises(NotImplementedError):
        e.bootstrap(1)


def test_cli_quantify_bootstrap(tmp_path):
    from typer.testing import CliRunner

    from gbrs_b200 import commands

    gdir = os.path.join(hp.GOLDEN, "quantify_multiway")
    z = np.load(os.path.join(gdir, "input.npz"))
    d = synth.generate(T=int(z["T"]), N=int(z["N"]), H=int(z["H"]), with_genotype=True)
    aln = os.path.join(str(tmp_path), "aln.emase")
    from tests.test_pack import make_apm

    make_apm(d).save(aln)
    args = ["quantify", "-i", aln, "-g", os.path.join(gdir, "grp.tsv"), "-L", os.path.join(gdir, "len.tsv"), "-M", "4", "-a"]
    plain, boot = os.path.join(str(tmp_path), "plain"), os.path.join(str(tmp_path), "boot")
    for out, extra in ((plain, []), (boot, ["--bootstrap", "3", "--bootstrap-seed", "12"])):
        res = CliRunner().invoke(commands.app, args + ["-o", out] + extra)
        assert res.exit_code == 0, res.output
    for sfx in ["isoforms.tpm", "isoforms.expected_read_counts", "genes.tpm", "genes.expected_read_counts",
                "isoforms.alignment_counts", "genes.alignment_counts"]:
        with open(f"{plain}.multiway.{sfx}", "rb") as a, open(f"{boot}.multiway.{sfx}", "rb") as b:
            assert a.read() == b.read(), sfx
    assert not os.path.exists(f"{plain}.multiway.bootstrap.npz")
    z = np.load(f"{boot}.multiway.bootstrap.npz")
    from gbrs_b200.apm import AlignmentPropertyMatrix

    em = EMfactory(AlignmentPropertyMatrix(h5file=aln, grpfile=os.path.join(gdir, "grp.tsv")))
    em.prepare(lenfile=os.path.join(gdir, "len.tsv"))
    api = em.bootstrap(3, model=4, seed=12)
    want = api.arrays()
    assert sorted(z.files) == sorted(want)
    for k in want:
        assert np.array_equal(z[k], want[k]), k
    assert z["total_reads"] == int(d.count.sum()) and z["replicate"].tolist() == [0, 1, 2]


def test_c2_full_size():
    """C2 (80k x 8 x 5M classes): two replicates' counts bit-identical to numpy, one replicate against the float64 oracle
    on its compacted matrix for 12 fixed updates (the bound of the full-size parity test)."""
    updates = 12
    d = synth.generate(T=80_000, N=5_000_000, H=8)
    M = int(d.count.sum())
    got = device_resample(d.count, 0, (0, 1))
    for b in range(2):
        want = br.resample(d.count, 0, b)
        assert np.array_equal(got[b], want.astype(np.float64)) and int(got[b].sum()) == M
    em = EMfactory(synth.to_apm(d))
    em.target_lengths = synth.effective_lengths(d)
    em.prepare()
    res = em.bootstrap([1], model=4, seed=0, tol=0.0, max_iters=updates)
    assert res.total_reads == M and res.num_iters[0] == updates
    dc = br.compact_synth(d, br.resample(d.count, 0, 1))
    o = hp.oracle_run(dc, 4, tol=0.0, max_iters=updates)
    rtol = 2 * xr.rtol_bound(*xr.shape_of(dc), dc.H, 4, updates)
    worst = max(xr.assert_elementwise(res.expected_read_counts[0], o["counts"], rtol, "C2 replicate counts"),
                xr.assert_elementwise(res.allelic_expression[0], o["theta"], rtol, "C2 replicate theta"))
    print(f"ELEMENTWISE bootstrap C2 replicate: worst relative error {worst:.2e}")
