"""EMfactory.bootstrap_summary on the device: every statistic against the replicates of bootstrap() reduced in numpy
(tests/boot_summary_checks.py), `.result` bit-identical to bootstrap(), the factory's state untouched, identical bytes
from two calls, the refusals, and the CLI's summary tables."""
import os

import numpy as np
import pytest

from gbrs_b200 import synth
from gbrs_b200.bootstrap import SUMMARY_MAX_REPLICATES
from gbrs_b200.emfactory import EMfactory
from gbrs_b200.quantify import hapmask_bytes
from tests import boot_summary_checks as bs
from tests import helpers as hp
from tests import layouts

pytestmark = pytest.mark.gpu

TOL, MAXIT = 1e-3, 60


def factory(d, **kw):
    em = EMfactory(synth.to_apm(d), item_len=16, **kw)
    em.target_lengths = synth.effective_lengths(d)
    em.prepare()
    return em


def genotype_mask(d, seed=4):
    rng = np.random.default_rng(seed)
    gtmask = np.zeros((d.H, d.T))
    for t in range(d.T):
        gtmask[rng.choice(d.H, min(2, d.H), replace=False), t] = 1.0
    return hapmask_bytes(gtmask)


@pytest.mark.parametrize("H", [2, 8])
@pytest.mark.parametrize("model", [1, 2, 3, 4])
def test_summary_matches_the_replicates(model, H):
    d = layouts.make_layout(H, 16)
    em = factory(d, locus_hapmask=genotype_mask(d))
    kw = dict(model=model, seed=7, tol=TOL, max_iters=MAXIT)
    summary = em.bootstrap_summary(6, interval=0.9, keep_replicates=True, **kw)
    res = em.bootstrap(6, **kw)
    bs.assert_same_result(summary.result, res)
    assert np.array_equal(summary.num_iters, res.num_iters) and summary.total_reads == res.total_reads
    worst = bs.check_summary(em, summary, res)
    print(f"SUMMARY model {model} H={H}: derived values within {worst:.2e} of the host")


def test_summary_without_groups_leaves_the_gene_level_out():
    d = synth.generate(T=120, N=3000, H=4, sample_index=1)
    apm = synth.to_apm(d)
    apm.groups, apm.gname, apm.num_groups = None, None, 0
    em = EMfactory(apm)
    em.prepare()
    summary = em.bootstrap_summary([3, 1, 4], tol=TOL, max_iters=MAXIT, keep_replicates=True)
    assert {lv for lv, _ in summary.stats} == {"isoforms"}
    bs.check_summary(em, summary, summary.result)


def test_factory_state_and_repeatability():
    d = layouts.make_layout(4, 16)
    em = factory(d)
    em.run(model=4, tol=TOL, max_iters=MAXIT, verbose=False)
    before = (em.get_allelic_expression(), em.expected_read_counts().copy(), em.num_iters, em.err_history.copy(),
              [m.data.copy() for m in em.posterior_probability().data])
    a = em.bootstrap_summary(5, seed=2, tol=TOL, max_iters=MAXIT)
    b = em.bootstrap_summary(5, seed=2, tol=TOL, max_iters=MAXIT)
    assert a.result is None and b.result is None
    for key in a.stats:
        for stat in a.stats[key]:
            assert a.stats[key][stat].tobytes() == b.stats[key][stat].tobytes(), (key, stat)
    after = (em.get_allelic_expression(), em.expected_read_counts().copy(), em.num_iters, em.err_history.copy(),
             [m.data.copy() for m in em.posterior_probability().data])
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
    assert before[2] == after[2] and np.array_equal(before[3], after[3])
    assert all(np.array_equal(x, y) for x, y in zip(before[4], after[4]))
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
        em.bootstrap_summary(2)  # no prepare()
    em.prepare()
    for bad in (dict(replicates=1), dict(replicates=[7]), dict(replicates=SUMMARY_MAX_REPLICATES + 1),
                dict(replicates=3, interval=0.0), dict(replicates=3, interval=1.0), dict(replicates=3, interval=1.5),
                dict(replicates=[2 ** 32, 1])):
        with pytest.raises(ValueError):
            em.bootstrap_summary(**bad)
    apm = synth.to_apm(d)
    apm.data[0].data[:] = 0.5  # a weighted file
    e = EMfactory(apm)
    e.prepare()
    with pytest.raises(NotImplementedError):
        e.bootstrap_summary(3)


def write_inputs(tmp_path, case="quantify_multiway"):
    gdir = os.path.join(hp.GOLDEN, case)
    z = np.load(os.path.join(gdir, "input.npz"))
    d = synth.generate(T=int(z["T"]), N=int(z["N"]), H=int(z["H"]), with_genotype=True)
    aln = os.path.join(str(tmp_path), "aln.emase")
    from tests.test_pack import make_apm

    make_apm(d).save(aln)
    return d, aln, os.path.join(gdir, "grp.tsv"), os.path.join(gdir, "len.tsv")


def read_table(path):
    with open(path) as fh:
        lines = fh.read().splitlines()
    return lines[0].split("\t"), [line.split("\t") for line in lines[1:]]


def test_cli_summary_tables(tmp_path):
    from typer.testing import CliRunner

    from gbrs_b200 import commands
    from gbrs_b200.apm import AlignmentPropertyMatrix

    d, aln, grp, lenf = write_inputs(tmp_path)
    args = ["quantify", "-i", aln, "-g", grp, "-L", lenf, "-M", "4", "--bootstrap", "4", "--bootstrap-seed", "3"]
    outs = {}
    for mode in ("npz", "summary", "both"):
        outs[mode] = os.path.join(str(tmp_path), mode)
        res = CliRunner().invoke(commands.app, args + ["-o", outs[mode], "--bootstrap-output", mode,
                                                       "--bootstrap-interval", "0.8"])
        assert res.exit_code == 0, res.output
    em = EMfactory(AlignmentPropertyMatrix(h5file=aln, grpfile=grp))
    em.prepare(lenfile=lenf)
    want = em.bootstrap(4, model=4, seed=3).arrays()
    for mode in ("npz", "both"):
        z = np.load(f"{outs[mode]}.multiway.bootstrap.npz")
        assert sorted(z.files) == sorted(want)
        assert all(np.array_equal(z[k], want[k]) for k in want)
    assert not os.path.exists(f"{outs['summary']}.multiway.bootstrap.npz")
    assert not any(".summary" in f for f in os.listdir(str(tmp_path)) if f.startswith("npz."))
    summary = em.bootstrap_summary(4, model=4, seed=3, interval=0.8)
    H = d.H
    for mode in ("summary", "both"):
        for level, names in (("isoforms", em.probability.lname), ("genes", em.probability.gname)):
            for quantity in ("tpm", "expected_read_counts", "allelic_share"):
                path = f"{outs[mode]}.multiway.bootstrap.{level}.{quantity}.summary"
                head, rows = read_table(path)
                cols = H if quantity == "allelic_share" else H + 1
                assert head[0] == "locus" and len(head) == 1 + 5 * cols + (quantity == "allelic_share")
                assert head[1:6] == [f"{d.hname[0]}.mean", f"{d.hname[0]}.sd", f"{d.hname[0]}.q0.1",
                                     f"{d.hname[0]}.q0.5", f"{d.hname[0]}.q0.9"]
                if quantity != "allelic_share":
                    assert head[-5] == "total.mean"
                else:
                    assert head[-1] == "n"
                assert [r[0] for r in rows] == list(names) and all(len(r) == len(head) for r in rows)
                got = np.array([[float(x) for x in r[1:]] for r in rows]).T
                assert np.array_equal(got, summary.columns(level, quantity), equal_nan=True), path


def test_cli_summary_without_groups_and_with_notes(tmp_path):
    from typer.testing import CliRunner

    from gbrs_b200 import commands

    d, aln, grp, lenf = write_inputs(tmp_path)
    out = os.path.join(str(tmp_path), "run")
    res = CliRunner().invoke(commands.app, ["run", "-i", aln, "-L", lenf, "-o", out, "--bootstrap", "3",
                                            "--bootstrap-output", "summary"])
    assert res.exit_code == 0, res.output
    written = sorted(f for f in os.listdir(str(tmp_path)) if f.startswith("run.bootstrap."))
    assert written == sorted(f"run.bootstrap.isoforms.{q}.summary" for q in ("tpm", "expected_read_counts",
                                                                               "allelic_share"))
    head, rows = read_table(f"{out}.bootstrap.isoforms.tpm.summary")
    assert head[5] == f"{d.hname[0]}.q0.975" and len(rows) == d.T
    d, aln, grp, lenf = write_inputs(tmp_path, "quantify_diploid")
    geno = os.path.join(hp.GOLDEN, "quantify_diploid", "gt.tsv")
    out = os.path.join(str(tmp_path), "dip")
    res = CliRunner().invoke(commands.app, ["quantify", "-i", aln, "-g", grp, "-L", lenf, "-G", geno, "-o", out,
                                            "--bootstrap", "3", "--bootstrap-output", "summary"])
    assert res.exit_code == 0, res.output
    for level in ("isoforms", "genes"):
        for quantity in ("tpm", "expected_read_counts", "allelic_share"):
            head, rows = read_table(f"{out}.diploid.bootstrap.{level}.{quantity}.summary")
            with open(f"{out}.diploid.{level}.tpm") as fh:
                point_head = fh.readline().rstrip("\n").split("\t")
            assert point_head[-1] == "notes" and head[-1] == "notes"
            assert head[-2] == ("n" if quantity == "allelic_share" else f"total.q0.975")
            assert all(len(r) == len(head) for r in rows) and len(rows) > 0


def test_summary_of_a_factory_on_another_device():
    """A factory on the last device while device 0 is current: every launch goes to the factory's device, and the
    statistics are those of the same factory on device 0, bit for bit."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    d = layouts.make_layout(4, 16)
    last = torch.cuda.device_count() - 1
    torch.cuda.set_device(0)
    kw = dict(seed=5, tol=TOL, max_iters=MAXIT)
    want = factory(d, device="cuda:0").bootstrap_summary(4, **kw)
    got = factory(d, device=f"cuda:{last}").bootstrap_summary(4, keep_replicates=True, **kw)
    assert torch.cuda.current_device() == 0
    assert set(got.stats) == set(want.stats)
    for key in want.stats:
        for stat in want.stats[key]:
            assert got.stats[key][stat].tobytes() == want.stats[key][stat].tobytes(), (key, stat)
    bs.assert_same_result(got.result, factory(d, device="cuda:0").bootstrap(4, **kw))
