"""Bootstrap summaries on the CPU: gbrs_boot_summarize and gbrs_boot_derive, compiled for the host SIMT shim
(tests/simt_em.py).  Quantiles and counts must equal numpy's nanquantile / the count bit for bit; mean and sd are held to
an extended-precision reference; derive to a long-double computation from the same [B][T][8] inputs."""
import os
import shutil
import subprocess
import sys
import warnings

import numpy as np
import pytest

from gbrs_b200 import _lib, utils
from gbrs_b200.bootstrap import SUMMARY_MAX_REPLICATES, interval_quantiles
from tests import simt_em
from tests import xref as xr

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ is needed to build the SIMT emulation")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUMMARY_SYMBOLS = ("gbrs_boot_derive", "gbrs_boot_summarize")


def emul_lib(tsan=False):
    lib = simt_em.load(tsan)
    for name in SUMMARY_SYMBOLS:
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = _lib.SYMBOLS[name]
    return lib


def emulated_summarize(values, q, lib=None):
    """[B][E] -> (mean [E], sd [E], quantiles [nq][E], n [E]) from the emulated gbrs_boot_summarize"""
    lib = lib or emul_lib()
    v = np.ascontiguousarray(values, dtype=np.float64)
    B, E = v.shape
    q = np.ascontiguousarray(q, dtype=np.float64)
    mean, sd = np.full(E, 7.0), np.full(E, 7.0)  # garbage: every element must be written
    qo, n = np.full((len(q), E), 7.0), np.full(E, -5, np.int32)
    rc = lib.gbrs_boot_summarize(v.ctypes.data, B, E, q.ctypes.data, len(q), mean.ctypes.data, sd.ctypes.data,
                                 qo.ctypes.data, n.ctypes.data, None)
    assert rc == 0, lib.gbrs_last_error()
    return mean, sd, qo, n


def check_summary(values, q):
    """quantiles and n exactly as numpy; mean within 1e-13 relative, sd within 1e-12 sd + 1e-13 mean of long double"""
    mean, sd, qo, n = emulated_summarize(values, q)
    defined = ~np.isnan(values)
    assert np.array_equal(n, defined.sum(axis=0))
    with warnings.catch_warnings():  # numpy warns about the all-NaN columns
        warnings.simplefilter("ignore", RuntimeWarning)
        want_q = np.nanquantile(values, q, axis=0, method="linear")
    assert np.array_equal(qo, want_q, equal_nan=True), np.argwhere(~((qo == want_q) | (np.isnan(qo) & np.isnan(want_q))))[:5]
    x = values.astype(np.longdouble)
    cnt = n.astype(np.longdouble)
    with np.errstate(all="ignore"):
        m = np.where(n > 0, np.where(defined, x, 0).sum(axis=0) / np.maximum(cnt, 1), np.nan)
        ss = np.where(defined, (x - m) ** 2, 0).sum(axis=0)
        s = np.where(n > 1, np.sqrt(ss / np.maximum(cnt - 1, 1)), np.nan)
    assert np.array_equal(np.isnan(mean), n == 0) and np.array_equal(np.isnan(sd), n < 2)
    ok = n > 0
    assert np.all(np.abs(mean[ok] - m[ok]) <= 1e-13 * np.abs(m[ok])), np.max(np.abs(mean[ok] - m[ok]))
    ok = n > 1
    assert np.all(np.abs(sd[ok] - s[ok]) <= 1e-12 * s[ok] + 1e-13 * np.abs(m[ok]))


def matrix(B, E, seed):
    """columns of several kinds: continuous, ties (small integers), all equal, zeros, NaN patterns that leave n = 0, 1,
    2 and about half defined"""
    rng = np.random.default_rng(seed)
    v = rng.gamma(2.0, 3.0, (B, E))
    kinds = np.arange(E) % 8
    v[:, kinds == 1] = rng.integers(0, 4, (B, int((kinds == 1).sum())))
    v[:, kinds == 2] = 0.37
    v[:, kinds == 3] = 0.0
    v[:, kinds == 4] = np.nan
    for kind, keep in ((5, 1), (6, 2)):
        for e in np.flatnonzero(kinds == kind):
            col = np.full(B, np.nan)
            idx = rng.choice(B, min(keep, B), replace=False)
            col[idx] = rng.random(len(idx))
            v[:, e] = col
    half = rng.random((B, E)) < 0.5
    v[:, kinds == 7] = np.where(half[:, kinds == 7], np.nan, v[:, kinds == 7])
    return v


@pytest.mark.parametrize("B", [2, 3, 31, 32, 33, 100])
@pytest.mark.parametrize("interval", [0.95, 0.5, 0.8, 0.999])
def test_emulated_summarize_equals_numpy(B, interval):
    E = 150 if B > 2 else 1100  # several tiles per block at B = 2 (grid-stride over tiles)
    check_summary(matrix(B, E, B * 1000 + int(interval * 1000)), interval_quantiles(interval))


def test_emulated_summarize_near_the_limit():
    B = SUMMARY_MAX_REPLICATES - 1  # a non-power of two: NaN padding fills the sort to 2^14
    assert B >= 4096
    check_summary(matrix(B, 9, 5), np.array([0.0, 0.025, 0.3, 0.5, 0.975, 1.0]))


def test_emulated_summarize_refusals():
    lib = emul_lib()
    v = np.zeros((SUMMARY_MAX_REPLICATES + 1, 1))
    out = np.zeros(4)
    n = np.zeros(1, np.int32)
    q = np.array([0.5])
    assert lib.gbrs_boot_summarize(v.ctypes.data, v.shape[0], 1, q.ctypes.data, 1, out.ctypes.data, out.ctypes.data,
                                   out.ctypes.data, n.ctypes.data, None) == _lib.GBRS_E_LIMIT
    for bad_q in (np.array([1.5]), np.array([np.nan])):
        assert lib.gbrs_boot_summarize(v.ctypes.data, 4, 1, bad_q.ctypes.data, 1, out.ctypes.data, out.ctypes.data,
                                       out.ctypes.data, n.ctypes.data, None) == _lib.GBRS_E_ARG
    assert lib.gbrs_boot_summarize(v.ctypes.data, 4, 1, q.ctypes.data, _lib.BOOT_MAX_QUANTILES + 1, out.ctypes.data,
                                   out.ctypes.data, out.ctypes.data, n.ctypes.data, None) == _lib.GBRS_E_ARG


# ---------------------------------------------------------------------------------------------------------------------
# derive
# ---------------------------------------------------------------------------------------------------------------------
def gene_csr(gene_of):
    """gene-major CSR over every gene id (ungrouped loci have ids >= n_genes), loci ascending"""
    order = np.argsort(gene_of, kind="stable")
    ptr = np.zeros(int(gene_of.max()) + 2, np.uint32)
    np.add.at(ptr, gene_of.astype(np.int64) + 1, 1)
    return np.cumsum(ptr).astype(np.uint32), order.astype(np.uint32)


def derive_inputs(B, T, H, seed):
    rng = np.random.default_rng(seed)
    src = np.zeros((B, T, 8))
    src[:, :, :H] = rng.gamma(0.7, 2.0, (B, T, H))
    src[:, :, :H][rng.random((B, T, H)) < 0.2] = 0.0
    src[:, 3, :H] = 0.0  # locus 3: theta 0 in every replicate (share undefined)
    src[::2, 5, :H] = 0.0  # locus 5: in every other replicate
    groups = [[0, 3], [1, 2, 4, 9], [5], [7, 8, 11]]  # loci 6, 10, 12.. belong to no gene
    return src, groups


def long_double_derive(src, H, quantity, groups):
    x = src[:, :, :H].astype(np.longdouble).transpose(0, 2, 1)  # [B, H, T]
    if groups is not None:
        x = np.stack([x[:, :, g].sum(axis=2) for g in groups], axis=2)
    tot = x.sum(axis=1, keepdims=True)
    if quantity == _lib.BOOT_SHARE:
        with np.errstate(all="ignore"):
            return np.where(tot != 0, x / tot, np.nan).reshape(x.shape[0], -1)
    if quantity == _lib.BOOT_TPM:
        x = x * (1e6 / x.sum(axis=(1, 2), keepdims=True))
    return np.concatenate([x, x.sum(axis=1, keepdims=True)], axis=1).reshape(x.shape[0], -1)


@pytest.mark.parametrize("H", [1, 2, 5, 8])
@pytest.mark.parametrize("level", ["isoforms", "genes"])
def test_emulated_derive_equals_long_double(H, level):
    xr.require_longdouble()
    B, T = 5, 13
    src, groups = derive_inputs(B, T, H, H)
    lib = emul_lib()
    if level == "genes":
        gene_of = utils.gene_index(T, groups)
        ptr, loci = gene_csr(gene_of)
        gp, gl, L = ptr.ctypes.data, loci.ctypes.data, len(groups)
    else:
        gp, gl, L, groups = None, None, T, None
    for quantity in (_lib.BOOT_TPM, _lib.BOOT_COUNTS, _lib.BOOT_SHARE):
        E = L * (H if quantity == _lib.BOOT_SHARE else H + 1)
        out = np.full((B, E), 7.0)
        assert lib.gbrs_boot_derive(src.ctypes.data, B, T, H, quantity, gp, gl, L if gp else 0, out.ctypes.data,
                                    None) == 0, lib.gbrs_last_error()
        want = long_double_derive(src, H, quantity, groups)
        assert np.array_equal(np.isnan(out), np.isnan(want)), quantity
        if quantity == _lib.BOOT_SHARE:
            assert np.isnan(out).any()  # the undefined shares are there
        ok = ~np.isnan(want)
        err = np.abs(out[ok] - want[ok].astype(np.float64))
        assert np.all(err <= 1e-13 * np.abs(want[ok]).astype(np.float64)), (quantity, err.max())


def test_emulated_derive_refusals():
    lib = emul_lib()
    src, out = np.zeros((1, 4, 8)), np.zeros(64)
    assert lib.gbrs_boot_derive(src.ctypes.data, 1, 4, 9, 0, None, None, 0, out.ctypes.data, None) == _lib.GBRS_E_ARG
    assert lib.gbrs_boot_derive(src.ctypes.data, 1, 4, 2, 3, None, None, 0, out.ctypes.data, None) == _lib.GBRS_E_ARG
    ptr = np.zeros(2, np.uint32)
    assert lib.gbrs_boot_derive(src.ctypes.data, 1, 4, 2, 0, ptr.ctypes.data, None, 1, out.ctypes.data, None) == _lib.GBRS_E_ARG


def test_summarize_kernel_is_race_free_under_thread_sanitizer():
    """One summarize call (two tiles, NaN columns) under ThreadSanitizer: the transpose, the per-column statistics, the
    bitonic stages and the quantile reads of one block must be ordered by its barriers."""
    try:
        simt_em.build(tsan=True)
    except RuntimeError as e:
        pytest.skip(f"ThreadSanitizer build unavailable: {e}")
    rt = subprocess.run(["g++", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(rt) or not os.path.exists(rt):
        pytest.skip("libtsan.so not found")
    code = f"""
import sys
sys.path.insert(0, {ROOT!r})
import numpy as np
from tests import test_bootstrap_summary as t
v = t.matrix(33, 70, 1)
mean, sd, qo, n = t.emulated_summarize(v, np.array([0.025, 0.5, 0.975]), lib=t.emul_lib(tsan=True))
assert np.array_equal(n, (~np.isnan(v)).sum(axis=0))
print("TSAN-RUN-OK")
"""
    env = dict(os.environ, LD_PRELOAD=rt, TSAN_OPTIONS="halt_on_error=0 report_signal_unsafe=0 exitcode=0",
               OMP_NUM_THREADS="1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=1500)
    if "TSAN-RUN-OK" not in res.stdout:
        pytest.skip("the sanitizer run did not complete here: " + res.stderr[-400:])
    assert "ThreadSanitizer: data race" not in res.stderr, res.stderr[-4000:]


@pytest.mark.parametrize("kw,match", [(dict(bootstrap=1, bootstrap_output="summary"), "2 to"),
                                      (dict(bootstrap=SUMMARY_MAX_REPLICATES + 1, bootstrap_output="both"), "2 to"),
                                      (dict(bootstrap=3, bootstrap_output="table"), "--bootstrap-output"),
                                      (dict(bootstrap=3, bootstrap_interval=1.0), "--bootstrap-interval")])
def test_bootstrap_flags_are_refused_before_the_input_is_read(kw, match, tmp_path):
    """quantify / run refuse bad bootstrap flags before they load anything (the alignment file does not exist)"""
    import importlib

    qm = importlib.import_module("gbrs_b200.quantify")  # the package re-exports the function of that name
    missing = str(tmp_path / "missing.h5")
    for fn in (qm.quantify, qm.run):
        with pytest.raises(ValueError, match=match):
            fn(alignment_file=missing, outbase=str(tmp_path / "out"), **kw)
