"""Shared by tests/test_posterior.py (CPU, SIMT emulation) and tests/test_posterior_gpu.py: the posterior read-origin
probabilities of a CSC pattern put in the entry order of tests/xref.XRef, and their error bound.

Bound of one posterior value (u = 2^-53, as in tests/xref.py, without a depth term: no sum over classes is involved).
Model 4: P = theta / s_n with s_n a sum of at most 8 k_max theta values, so |got - want| / want <= (8 k_max + c) u.
Models 1-3 add the three per-class normalisers (at most 8 k_max terms each) and the gene sums of theta (at most 8 g_max
terms, twice).  The bound is SAFETY times these counts times u, computed from the shape."""
from __future__ import annotations

import numpy as np

from tests import xref as xr


def rtol_posterior(x: xr.XRef, model: int) -> float:
    terms = 8 * x.k_max + xr.C_OPS + (0 if model == 4 else 3 * 8 * x.k_max + 2 * 8 * x.g_max)
    return xr.SAFETY * terms * xr.U


def pattern_arrays(pattern):
    """(indptr list, indices list) of gbrs_b200.emfactory.posterior_pattern()"""
    return [a[0] for a in pattern], [a[1] for a in pattern]


def entry_values(values, indptr, indices, x: xr.XRef) -> np.ndarray:
    """Values of the H CSC matrices (N x T, `indptr[h]` / `indices[h]` / `values[h]`) in the entry order of `x`.  The pattern
    must hold exactly the entries of `x`: nothing missing, nothing extra, no duplicate."""
    T, N = x.T, x.N
    keys, vals = [], []
    for h in range(len(indptr)):
        col = np.repeat(np.arange(T, dtype=np.int64), np.diff(np.asarray(indptr[h], dtype=np.int64)))
        keys.append((h * N + np.asarray(indices[h], dtype=np.int64)) * T + col)
        vals.append(np.asarray(values[h], dtype=np.float64))
    k, v = np.concatenate(keys), np.concatenate(vals)
    order = np.argsort(k, kind="stable")
    k, v = k[order], v[order]
    want = (x.h.astype(np.int64) * N + x.n) * T + x.t
    assert k.size == want.size and np.array_equal(np.unique(k), k), (k.size, want.size)
    pos = np.searchsorted(k, want)
    assert np.array_equal(k[np.minimum(pos, k.size - 1)], want), "the posterior pattern is not the EM's pattern"
    return v[pos]


def apm_entry_values(apm, x: xr.XRef) -> np.ndarray:
    """entry_values of an AlignmentPropertyMatrix (posterior_probability()); its matrices must be canonical CSC"""
    for m in apm.data:
        assert m.format == "csc" and m.has_sorted_indices and m.dtype == np.float64
    return entry_values([m.data for m in apm.data], [m.indptr for m in apm.data], [m.indices for m in apm.data], x)


def check(got, want, rtol, what):
    """element-wise (tests/xref.assert_elementwise: zeros exactly where the reference has zeros, no absolute floor)"""
    err = xr.assert_elementwise(np.asarray(got)[None, :], np.asarray(want)[None, :], rtol, what)
    print(f"ELEMENTWISE {what}: max rel err {err:.3e}, bound {float(rtol):.3e}")
    return err


def class_sums(vals, x: xr.XRef) -> np.ndarray:
    """sum of the posterior over every class that has entries, in long double"""
    s = np.zeros(x.N, dtype=xr.LD)
    np.add.at(s, x.n, np.asarray(vals).astype(xr.LD))
    return s[np.bincount(x.n, minlength=x.N) > 0]


def counts_from(vals, x: xr.XRef) -> np.ndarray:
    """sum_n c_n P[n,t,h] in long double (H x T), to compare with the expected read counts"""
    return x.sum_read(np.asarray(vals).astype(xr.LD))
