"""Checks shared by the device tests of the bootstrap summaries (tests/test_bootstrap_summary_gpu.py and the full-size
test): every statistic of a BootstrapSummary against the replicates of a BootstrapResult, reduced in numpy."""
import ctypes as C
import warnings

import numpy as np

from gbrs_b200 import _lib
from gbrs_b200.bootstrap import LEVELS, QUANTITIES


def host_values(res, level, quantity):
    """[B, C, L] from the BootstrapResult as the point reports compute them: tpm / read_counts with the total row, or
    the allelic shares (NaN where the locus' sum is 0)"""
    grp = level == "genes"
    if quantity == "allelic_share":
        x = res._group(res.allelic_expression) if grp else res.allelic_expression
        tot = x.sum(axis=1, keepdims=True)
        with np.errstate(all="ignore"):
            return np.where(tot != 0, x / tot, np.nan)
    x = res.tpm(grp) if quantity == "tpm" else res.read_counts(grp)
    return np.concatenate([x, x.sum(axis=1, keepdims=True)], axis=1)


def device_values(em, res, level, quantity):
    """gbrs_boot_derive on the replicates of `res` uploaded as [B][T][8] (bit for bit what bootstrap_summary derives
    from) -> [B, C, L]"""
    import torch

    B, H, T = res.allelic_expression.shape
    src = res.expected_read_counts if quantity == "expected_read_counts" else res.allelic_expression
    dev = torch.zeros((B, T, 8), dtype=torch.float64, device="cuda")
    dev[:, :, :H] = torch.from_numpy(np.ascontiguousarray(src.transpose(0, 2, 1))).cuda()
    code = {"tpm": _lib.BOOT_TPM, "expected_read_counts": _lib.BOOT_COUNTS, "allelic_share": _lib.BOOT_SHARE}[quantity]
    if level == "genes":
        pat = em._pattern
        gp, gl, L = pat.dev["gene_ptr"].data_ptr(), pat.dev["gene_loci"].data_ptr(), int(em.probability.num_groups)
    else:
        gp, gl, L = None, None, T
    rows = H if code == _lib.BOOT_SHARE else H + 1
    out = torch.empty((B, rows * L), dtype=torch.float64, device="cuda")
    _lib.check(_lib.load().gbrs_boot_derive(dev.data_ptr(), B, T, H, code, gp, gl, L if gp else 0, out.data_ptr(),
                                            C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out.cpu().numpy().reshape(B, rows, L)


def check_summary(em, summary, res, derive_rtol=1e-13):
    """derived values against the host computation within `derive_rtol`; quantiles bit for bit np.nanquantile of the
    device's derived values; n the count of defined values; mean within 1e-13 relative and sd within 1e-12 sd + 1e-13 mean
    of a long-double reduction.  Returns the worst relative deviation of the derived values."""
    worst = 0.0
    want_keys = {(lv, qn) for lv in LEVELS for qn in QUANTITIES if lv == "isoforms" or res.grp_conv_mat is not None}
    assert set(summary.stats) == want_keys
    for level, quantity in sorted(want_keys):
        st = summary.stats[(level, quantity)]
        dv = device_values(em, res, level, quantity)
        hv = host_values(res, level, quantity)
        what = f"{level}.{quantity}"
        assert np.array_equal(np.isnan(dv), np.isnan(hv)), what
        ok = ~np.isnan(hv)
        rel = np.abs(dv[ok] - hv[ok]) / np.maximum(np.abs(hv[ok]), 1e-300)
        rel[(dv[ok] == 0) & (hv[ok] == 0)] = 0.0
        worst = max(worst, float(rel.max(initial=0.0)))
        assert rel.max(initial=0.0) <= derive_rtol, (what, rel.max())
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            want_q = np.nanquantile(dv, summary.quantiles, axis=0, method="linear")
        assert np.array_equal(st["q"], want_q, equal_nan=True), what
        defined = ~np.isnan(dv)
        n = defined.sum(axis=0)
        if quantity == "allelic_share":
            assert np.array_equal(st["n"], n[0]), what
        x = np.where(defined, dv, 0).astype(np.longdouble)
        with np.errstate(all="ignore"):
            m = x.sum(axis=0) / n
            s = np.sqrt(np.where(defined, (dv.astype(np.longdouble) - m) ** 2, 0).sum(axis=0) / (n - 1))
        assert np.array_equal(np.isnan(st["mean"]), n == 0) and np.array_equal(np.isnan(st["sd"]), n < 2), what
        k = n > 0
        assert np.all(np.abs(st["mean"][k] - m[k]) <= 1e-13 * np.abs(m[k])), what
        k = n > 1
        assert np.all(np.abs(st["sd"][k] - s[k]) <= 1e-12 * s[k] + 1e-13 * np.abs(m[k])), what
    return worst


def assert_same_result(a, b):
    assert np.array_equal(a.replicates, b.replicates) and np.array_equal(a.num_iters, b.num_iters)
    assert a.seed == b.seed and a.model == b.model and a.total_reads == b.total_reads
    assert np.array_equal(a.allelic_expression, b.allelic_expression)
    assert np.array_equal(a.expected_read_counts, b.expected_read_counts)
