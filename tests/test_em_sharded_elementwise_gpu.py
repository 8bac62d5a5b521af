"""Row-sharded EM on the device, every output element against the extended-precision reference (tests/xref.py), at 2 to
8 row shards.

* One GPU, R = 4..8 shards, the numerators summed by hand between the two halves of an update: the class split of the
  device packer and the local kernels on shards that are tiny or hold no class at all (constructed layouts, one locus,
  fewer classes than shards, one class holding nearly all of the nnz), on the two-pass kernels and on the tile kernel.
* Every GPU of the box (W = min(devices, 8), and W = 3 where there are more than three): `EMfactory(shard=True)` under
  torchrun through each exchange form (push, tag, pull, nvls, nccl): prepare(), one update of every model, run() to
  convergence, element-wise and bit-identical on every rank.

Each check prints one ELEMENTWISE line (largest relative error, and the bound at that shape) under `pytest -s`."""
import ctypes as C
import os
import signal
import subprocess
import sys

import numpy as np
import pytest

from gbrs_b200 import _lib, synth
from gbrs_b200.emfactory import DevicePattern
from oracle import em_oracle as eo
from tests import layouts
from tests import xref as xr
from tests.test_em_elementwise_gpu import check

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODELS = (4, 3, 2, 1)
KINDS = ("layout", "layout tiles", "one locus", "few classes", "heavy first class")
TILE_PARAMS = dict(max_loci=48, max_items=192)  # the default caps hold classes of up to 16 loci; the layouts have 40


def one_gpu_problem(kind, R):
    if kind.startswith("layout"):
        return layouts.make_layout(8), 16
    if kind == "one locus":  # 8T = 8 doubles over R owners: the trailing owners have an empty slice
        return synth.generate(T=1, N=20, H=8, sample_index=4), 0
    return layouts.make_empty_shards(kind, R), 0


@pytest.mark.parametrize("R", range(4, 9))
@pytest.mark.parametrize("kind", KINDS)
def test_gpu_row_shards_elementwise(kind, R):
    """R row shards on one GPU (numerators summed by hand): prepare() without and with a pseudocount, then one update of
    every model from one random theta, on every shard element-wise and bit-identical."""
    import torch

    xr.require_longdouble()
    d, item_len = one_gpu_problem(kind, R)
    gene_of = eo.gene_index(d.T, d.groups())
    x, eff = xr.XRef(d, gene_of), eo.effective_length_table(d.lengths)
    apm = synth.to_apm(d)
    tiles = dict(tiles=True, tile_params=TILE_PARAMS) if kind == "layout tiles" else {}
    pats = [DevicePattern(apm, gene_of=gene_of, shard_rank=r, shard_count=R, item_len=item_len, **tiles)
            for r in range(R)]
    classes, nnz = [int(p.info["n_classes"]) for p in pats], [int(p.info["nnz"]) for p in pats]
    if kind in ("few classes", "heavy first class"):
        layouts.assert_empty_shards(kind, d, classes, nnz)
    else:
        assert sum(nnz) == d.nnz and all(c > 0 for c in classes), classes
    if tiles:
        assert all(p.tiled is not None for p in pats)
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

    def same_on_every_shard(get, what):
        first = get(pats[0])
        for p in pats[1:]:
            assert np.array_equal(get(p), first), what

    tag = f"{kind} R={R}"
    for pc in (0.0, 0.25):
        for p in pats:
            _lib.check(lib.gbrs_em_prepare_local(C.byref(p.desc), p.stream()))
        exchange()
        for p in pats:
            _lib.check(lib.gbrs_em_prepare_finish(C.byref(p.desc), pc, p.stream()))
        check(pats[0].current_theta_HT(), x.prepare(eff, pc), x.rtol_prepare(pc), f"{tag} theta0 pc={pc}")
        same_on_every_shard(lambda p: p.current_theta_HT(), f"{tag} theta0 pc={pc}")
    theta = xr.random_theta(x, seed=30 + R)
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
        check(pats[0].acc_HT(), counts, rtol, f"{tag} model {model} counts")
        check(pats[0].current_theta_HT(), theta1, rtol, f"{tag} model {model} theta")
        same_on_every_shard(lambda p: p.current_theta_HT(), f"{tag} model {model} theta")
        if kind.startswith("layout"):
            assert not pats[0].acc_HT()[:, d.zero_locus].any()


WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["GBRS_ROOT"])
import numpy as np, torch, torch.distributed as dist
from gbrs_b200 import synth
from gbrs_b200.emfactory import EMfactory
from oracle import em_oracle as eo
from tests import layouts
from tests import xref as xr

local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
rank, world = dist.get_rank(), dist.get_world_size()
form = os.environ["GBRS_XCHG"]


def gather(v):
    t = torch.tensor([int(v)], dtype=torch.int64, device="cuda")
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [int(o.item()) for o in out]


def verify(got, want, rtol, what):
    err = xr.assert_elementwise(got, want, rtol, what)
    t = torch.from_numpy(np.ascontiguousarray(got, dtype=np.float64)).cuda()
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    assert torch.equal(lo, hi), what + ": ranks differ"
    if rank == 0:
        print(f"ELEMENTWISE W={world} {form} {what}: max rel err {err:.3e}, bound {float(np.min(rtol)):.3e}..{float(np.max(rtol)):.3e}",
              flush=True)


problems = [("layout", layouts.make_layout(8), 4), ("heavy first class", layouts.make_empty_shards("heavy first class", world), 2),
            ("one locus", synth.generate(T=1, N=20, H=8, sample_index=4), 3)]
for name, d, run_model in problems:
    gene_of = eo.gene_index(d.T, d.groups())
    x, eff = xr.XRef(d, gene_of), eo.effective_length_table(d.lengths)
    em = EMfactory(synth.to_apm(d), shard=True, item_len=16)
    em.target_lengths = synth.effective_lengths(d)
    em.prepare()
    assert em.world == world
    if form != "nccl":
        assert em.fused_exchange and em.exchange_mode == form, (em.fused_exchange, em.exchange_mode)
    else:
        assert not em.fused_exchange
    classes, nnz = gather(em._pattern.info["n_classes"]), gather(em._pattern.info["nnz"])
    if name == "heavy first class":
        layouts.assert_empty_shards(name, d, classes, nnz)
    else:
        assert sum(nnz) == d.nnz, (nnz, d.nnz)
    verify(em.get_allelic_expression(), x.prepare(eff), x.rtol_prepare(), f"{name} theta0")
    em.reset(pseudocount=0.25)
    verify(em.get_allelic_expression(), x.prepare(eff, 0.25), x.rtol_prepare(0.25), f"{name} theta0 pc=0.25")
    theta = xr.random_theta(x, seed=40 + world)
    for model in (4, 3, 2, 1):
        em.allelic_expression = theta
        em.update_allelic_expression(model=model)
        counts, theta1 = x.update(theta, model, eff)
        rtol = x.rtol_update(model)
        verify(em.expected_read_counts(), counts, rtol, f"{name} model {model} counts")
        verify(em.allelic_expression, theta1, rtol, f"{name} model {model} theta")
    em.reset(pseudocount=0.25)
    em.run(model=run_model, tol=1e-5, max_iters=400, verbose=False)
    want = x.run(x.prepare(eff, 0.25), run_model, eff, 1e-5, 400)
    assert em.num_iters == want["iters"] < 400, (name, em.num_iters, want["iters"])
    np.testing.assert_allclose(em.err_history, want["errs"], rtol=1e-7, atol=1e-7)
    rtol = x.rtol_run(run_model, want["iters"], pseudocount=0.25)
    verify(em.allelic_expression, want["theta"], rtol, f"{name} run model {run_model} ({want['iters']} updates) theta")
    verify(em.expected_read_counts(), want["counts"], rtol, f"{name} run model {run_model} counts")
dist.destroy_process_group()
print("rank", rank, "ok", flush=True)
'''


@pytest.mark.parametrize("xchg", ["push", "tag", "pull", "nvls", "nccl"])
@pytest.mark.parametrize("which", ["all", "three"])
def test_multi_gpu_sharded_elementwise(tmp_path, which, xchg):
    """W ranks under torchrun, one per GPU: W = min(devices, 8), and W = 3."""
    import torch

    xr.require_longdouble()
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"needs at least two GPUs (this box has {n})")
    if which == "three" and (n < 3 or min(n, 8) == 3):
        pytest.skip("W = 3 needs more than three GPUs to differ from W = min(devices, 8)")
    world = min(n, 8) if which == "all" else 3
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, GBRS_ROOT=ROOT, MASTER_ADDR="127.0.0.1", GBRS_XCHG=xchg)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", "29533", str(script)]
    # a session of its own: on a timeout the whole process group (torchrun and its workers) is killed
    proc = subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                            start_new_session=True)
    try:
        out, err = proc.communicate(timeout=900)
    except subprocess.TimeoutExpired:
        os.killpg(proc.pid, signal.SIGKILL)
        out, err = proc.communicate()
        pytest.fail(f"W={world} {xchg}: no result within 900 s\n" + out[-3000:] + err[-3000:])
    print("\n".join(line for line in out.splitlines() if line.startswith("ELEMENTWISE")))
    assert proc.returncode == 0, out[-3000:] + err[-3000:]
    assert out.count(" ok") == world, out[-3000:]
