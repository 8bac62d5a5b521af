"""EMfactory.posterior_probability() on the device, element by element against the extended-precision reference
(tests/xref.py, bound of tests/posterior_checks.py) on the constructed layouts of tests/layouts.py: every state the
reference's `probability` can be in, on each code path of the update (two-pass kernels, 64-bit entry words, the tile
layout, the host packer), the -G restriction, weighted files, row shards on one GPU and
under torchrun, the export, and full-size problems against the float64 oracle.  Each check prints one ELEMENTWISE line
under `pytest -s`."""
import os
import signal
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from gbrs_b200 import synth
from gbrs_b200.emfactory import DevicePattern, EMfactory, posterior_pattern
from gbrs_b200.quantify import hapmask_bytes
from oracle import em_oracle as eo
from tests import layouts
from tests import posterior_checks as pc
from tests import xref as xr

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODELS = (4, 3, 2, 1)
PATHS = {"two-pass": {}, "entry64": {}, "host-packer": dict(pack="host"),
         "tiles": dict(tiles=True, tile_params=dict(max_loci=48, max_items=192))}


def problem(H):
    xr.require_longdouble()
    d = layouts.make_layout(H, 16)
    gene_of = eo.gene_index(d.T, d.groups())
    return d, gene_of, xr.XRef(d, gene_of), eo.effective_length_table(d.lengths)


def factory(d, pseudocount=0.0, **kw):
    em = EMfactory(synth.to_apm(d), item_len=16, **kw)
    em.target_lengths = synth.effective_lengths(d)
    em.prepare(pseudocount=pseudocount)
    return em


def states(H, path, em, d, x, eff):
    """prepare(), a stand-alone E-step and one update of every model from a random theta, run() to convergence"""
    tag = f"H={H} {path}"
    pc.check(pc.apm_entry_values(em.posterior_probability(), x), x.e_step(np.ones((H, d.T)), 4), pc.rtol_posterior(x, 4),
             f"{tag} prepare")
    theta = xr.random_theta(x, seed=H)
    for model in MODELS:
        want = x.e_step(theta, model)
        rtol = pc.rtol_posterior(x, model)
        em.allelic_expression = theta
        em.update_probability_at_read_level(model=model)
        got = pc.apm_entry_values(em.posterior_probability(), x)
        pc.check(got, want, rtol, f"{tag} model {model} E-step")
        xr.assert_elementwise(em.expected_read_counts(), pc.counts_from(got, x), x.rtol_update(model), f"{tag} counts")
        em.allelic_expression = theta
        em.update_allelic_expression(model=model)
        pc.check(pc.apm_entry_values(em.posterior_probability(), x), want, rtol, f"{tag} model {model} one update")
    model = MODELS[H % 4]
    em.reset(pseudocount=0.25)
    pc.check(pc.apm_entry_values(em.posterior_probability(), x), x.e_step(np.ones((H, d.T)), 4), pc.rtol_posterior(x, 4),
             f"{tag} reset pc=0.25")
    em.run(model=model, tol=1e-5, max_iters=400, verbose=False)
    k = em.num_iters
    prev = x.run(x.prepare(eff, 0.25), model, eff, 1e-5, k - 1)["theta"]
    # the E-step of theta_(k-1), whose own error is that of k - 1 updates: P moves by at most twice theta's relative error
    rtol = pc.rtol_posterior(x, model) + 2 * float(np.max(x.rtol_run(model, k - 1, pseudocount=0.25)))
    pc.check(pc.apm_entry_values(em.posterior_probability(), x), x.e_step(prev, model), rtol, f"{tag} run ({k} updates)")


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("H", range(1, 9))
def test_gpu_posterior_states_elementwise(H, path, monkeypatch):
    if path == "entry64":
        monkeypatch.setenv("GBRS_FORCE_ENTRY64", "1")
    d, gene_of, x, eff = problem(H)
    em = factory(d, **PATHS[path])
    pat = em._pattern
    assert pat.info["entry_bytes"] == (8 if path == "entry64" else 4)
    assert (pat.tiled is not None) == (path == "tiles") and pat.on_device == (path in ("two-pass", "entry64"))
    states(H, path, em, d, x, eff)


def test_gpu_posterior_model4_run_uploads_nothing_new():
    """A model-4 run on the host packer's pattern keeps class_id on the host; the first posterior call uploads it."""
    d, gene_of, x, eff = problem(8)
    em = factory(d, pack="host")
    em.run(model=4, tol=1e-5, max_iters=50, verbose=False)
    assert "class_id" not in em._pattern.dev
    em.posterior_probability()
    assert "class_id" in em._pattern.dev


def test_gpu_posterior_weighted_file_and_export(tmp_path):
    """A matrix with stored values: after prepare() the normalised values, after reset() the incidence posterior; the
    export with values round-trips through AlignmentPropertyMatrix(h5file=...); the default export writes exactly the
    arrays of `probability.save`."""
    from gbrs_b200 import AlignmentPropertyMatrix as APM

    d, gene_of, x, eff = problem(4)
    apm = synth.to_apm(d)
    rng = np.random.default_rng(1)
    for m in apm.data:
        m.data = rng.integers(1, 5, m.data.size).astype(np.float64)
    em = EMfactory(apm, item_len=16)
    em.target_lengths = synth.effective_lengths(d)
    em.prepare()
    pattern = posterior_pattern(apm)
    rows = sum(np.bincount(ix, weights=v, minlength=d.N) for _, ix, v in pattern)
    got = em.posterior_probability()
    for h, (ip, ix, v) in enumerate(pattern):
        np.testing.assert_array_equal(got.data[h].data, v / rows[ix])
    em.reset()
    pc.check(pc.apm_entry_values(em.posterior_probability(), x), x.e_step(np.ones((4, d.T)), 4), pc.rtol_posterior(x, 4),
             "weighted reset")
    em.run(model=3, tol=1e-5, max_iters=5, verbose=False)
    post = em.posterior_probability()
    f = tmp_path / "post.npz"
    em.export_posterior_probability(str(f), incidence_only=False)
    back = APM(h5file=str(f))
    assert back.shape == post.shape and list(back.hname) == list(post.hname)
    for a, b in zip(back.data, post.data):
        assert np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices)
        assert np.array_equal(a.data.view(np.uint64), b.data.view(np.uint64))
    f1, f2 = tmp_path / "default.npz", tmp_path / "save.npz"
    em.export_posterior_probability(str(f1))
    apm.save(h5file=str(f2), title="Posterior Probability")
    with np.load(f1) as z1, np.load(f2) as z2:  # (the zip members carry their write time: compare the arrays' bytes)
        assert sorted(z1.files) == sorted(z2.files) and "h0_data" not in z1.files
        for k in z1.files:
            assert z1[k].dtype == z2[k].dtype and z1[k].tobytes() == z2[k].tobytes(), k


def test_gpu_posterior_genotype_restriction_and_zero_class():
    """-G through locus_hapmask: masked columns empty, the rest as XRef(gtmask=...); a class whose entries all have
    theta 0 raises FloatingPointError."""
    xr.require_longdouble()
    d = synth.generate(T=200, N=3000, H=8, sample_index=4, with_genotype=True)
    gene_of = eo.gene_index(d.T, d.groups())
    gtmask = synth.genotype_mask(d)
    hapmask = hapmask_bytes(gtmask)
    x = xr.XRef(d, gene_of, gtmask=gtmask)
    em = EMfactory(synth.to_apm(d), locus_hapmask=hapmask)
    em.prepare()
    theta = xr.random_theta(x, seed=2)
    for model in MODELS:
        em.allelic_expression = theta
        em.update_probability_at_read_level(model=model)
        post = em.posterior_probability()
        for h, m in enumerate(post.data):
            assert not np.diff(m.indptr)[((hapmask >> h) & 1) == 0].any()
        pc.check(pc.apm_entry_values(post, x), x.e_step(theta, model), pc.rtol_posterior(x, model), f"-G model {model}")
    n0 = int(x.n[0])
    theta[x.h[x.n == n0], x.t[x.n == n0]] = 0.0
    for model in MODELS:
        em.allelic_expression = theta
        em.update_probability_at_read_level(model=model)
        with pytest.raises(FloatingPointError):
            em.posterior_probability()


def test_gpu_posterior_leaves_the_run_untouched():
    """prepare, run(max_iters=3), posterior, run to convergence: bit-identical to the same without the posterior."""
    d, gene_of, x, eff = problem(8)
    out = []
    for with_posterior in (False, True):
        em = factory(d)
        em.run(model=1, tol=0.0, max_iters=3, verbose=False)
        if with_posterior:
            a, b = em.posterior_probability(), em.posterior_probability()
            for m1, m2 in zip(a.data, b.data):
                assert np.array_equal(m1.data.view(np.uint64), m2.data.view(np.uint64))
        em.run(model=1, tol=1e-6, max_iters=400, verbose=False)
        out.append((em.allelic_expression.copy(), em.expected_read_counts().copy(), em.err_history.copy(), em.num_iters))
    (t1, c1, e1, n1), (t2, c2, e2, n2) = out
    assert n1 == n2 and np.array_equal(t1, t2) and np.array_equal(c1, c2) and np.array_equal(e1, e2)


@pytest.mark.parametrize("R", [2, 3])
def test_gpu_posterior_row_shards_on_one_gpu(R):
    """R shards of one GPU, one theta set by hand: the sum of the shards' posteriors equals the unsharded one bit for bit."""
    import torch

    d, gene_of, x, eff = problem(8)
    apm = synth.to_apm(d)
    theta = torch.zeros((d.T, 8), dtype=torch.float64)
    theta[:, : d.H] = torch.from_numpy(xr.random_theta(x, seed=R).T)
    theta = theta.cuda()
    ip, ix = pc.pattern_arrays(posterior_pattern(apm))
    whole = DevicePattern(apm, gene_of=gene_of, item_len=16)
    pats = [DevicePattern(apm, gene_of=gene_of, shard_rank=r, shard_count=R, item_len=16) for r in range(R)]
    for model in MODELS:
        want = whole.posterior(model, theta, ip, ix)
        parts = [p.posterior(model, theta, ip, ix) for p in pats]
        for h in range(d.H):
            got = sum(part[h] for part in parts)
            assert np.array_equal(got.view(np.uint64), want[h].view(np.uint64)), (model, h)
        pc.check(pc.entry_values(want, ip, ix, x), x.e_step(theta[:, : d.H].T.cpu().numpy(), model),
                 pc.rtol_posterior(x, model), f"R={R} model {model}")


def full_size_check(d, model, updates):
    """`updates` fixed updates, then the posterior against the float64 oracle's E-step of the theta that entered the last
    one, element-wise within twice the bound"""
    gene_of = eo.gene_index(d.T, d.groups())
    em = EMfactory(synth.to_apm(d))
    em.target_lengths = synth.effective_lengths(d)
    em.prepare()
    em.run(model=model, tol=0.0, max_iters=updates - 1, verbose=False)
    theta = em.get_allelic_expression()
    em.update_allelic_expression(model=model)
    post = em.posterior_probability()
    oapm = eo.apm_from_pairs(d.T, d.H, d.N, d.pair_class, d.pair_locus, d.pair_mask, d.count)
    want = eo.e_step(oapm, theta, model, gene_of)
    k_max = int(np.bincount(np.asarray(d.pair_class)).max())
    g_max = int(np.bincount(np.asarray(gene_of)).max())
    terms = 8 * k_max + xr.C_OPS + (0 if model == 4 else 3 * 8 * k_max + 2 * 8 * g_max)
    rtol = 2 * xr.SAFETY * terms * xr.U
    entries = SimpleNamespace(T=d.T, N=d.N, h=oapm.ent_h, n=oapm.ent_n, t=oapm.ent_t)
    got = pc.apm_entry_values(post, entries)
    pc.check(got, want, rtol, f"full size model {model} ({updates} updates, {got.size} entries)")


def test_gpu_posterior_full_size_model4():
    """C2 (80k loci x 8 haplotypes, 5M classes) after 12 updates of model 4."""
    full_size_check(synth.generate(T=80_000, N=5_000_000, H=8), 4, 12)


@pytest.mark.parametrize("model", [1, 2, 3])
def test_gpu_posterior_full_size_models_1_to_3(model):
    """The C2 locus shape under models 1-3 on a 1M-class slice, after 6 updates."""
    full_size_check(synth.generate(T=80_000, N=1_000_000, H=8), model, 6)


WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["GBRS_ROOT"])
import numpy as np
import torch
import torch.distributed as dist
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
from gbrs_b200 import synth
from gbrs_b200.emfactory import DevicePattern, EMfactory, posterior_pattern
from oracle import em_oracle as eo
from tests import layouts
from tests import posterior_checks as pc
from tests import xref as xr
d = layouts.make_layout(8)
gene_of = eo.gene_index(d.T, d.groups())
x = xr.XRef(d, gene_of)
apm = synth.to_apm(d)
em = EMfactory(apm, shard=True, item_len=16)
em.target_lengths = synth.effective_lengths(d)
em.prepare()
assert em.fused_exchange and em.exchange_mode == "push", (em.fused_exchange, em.exchange_mode)
theta = xr.random_theta(x, seed=3)
ip, ix = pc.pattern_arrays(posterior_pattern(apm))
single = DevicePattern(apm, gene_of=gene_of, item_len=16)  # the whole matrix on this GPU
t8 = torch.zeros((d.T, 8), dtype=torch.float64)
t8[:, : d.H] = torch.from_numpy(theta.T)
t8 = t8.cuda()
for model in (4, 3, 2, 1):
    em.allelic_expression = theta
    em.update_allelic_expression(model=model)
    post = em.posterior_probability()
    want = single.posterior(model, t8, ip, ix)
    for h in range(d.H):
        got = torch.from_numpy(post.data[h].data.view(np.int64)).cuda()
        lo, hi = got.clone(), got.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        assert torch.equal(lo, hi), "ranks differ"
        assert np.array_equal(post.data[h].data.view(np.uint64), want[h].view(np.uint64)), (model, h)
    if rank == 0:
        pc.check(pc.apm_entry_values(post, x), x.e_step(theta, model), pc.rtol_posterior(x, model), f"W={world} model {model}")
dist.destroy_process_group()
print("rank", rank, "ok", flush=True)
'''


def test_multi_gpu_posterior_push_form(tmp_path):
    """W = min(devices, 8) ranks under torchrun, push form: every rank returns the same bits, equal to a single-GPU
    computation from the same theta."""
    import torch

    xr.require_longdouble()
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"needs at least two GPUs (this box has {n})")
    world = min(n, 8)
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, GBRS_ROOT=ROOT, MASTER_ADDR="127.0.0.1", GBRS_XCHG="push")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", "29541", str(script)]
    # a session of its own: on a timeout the whole process group (torchrun and its workers) is killed
    proc = subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, start_new_session=True)
    try:
        out, err = proc.communicate(timeout=900)
    except subprocess.TimeoutExpired:
        os.killpg(proc.pid, signal.SIGKILL)
        out, err = proc.communicate()
        pytest.fail(f"W={world}: no result within 900 s\n" + out[-3000:] + err[-3000:])
    print("\n".join(line for line in out.splitlines() if line.startswith("ELEMENTWISE")))
    assert proc.returncode == 0, out[-3000:] + err[-3000:]
    assert out.count(" ok") == world, out[-3000:]
