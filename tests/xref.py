"""Extended-precision reference of the EM update, an error bound for the float64 kernels, and an element-wise comparator.

The reference restates the reference's E-step / M-step (EMfactory.update_probability_at_read_level, models 1-4, and the
theta0 of prepare(), cf. oracle/em_oracle.py) in np.longdouble -- a 64-bit significand on x86, eps = 2^-63 -- with its own
segmented sums (a stable sort by segment key and np.add.reduceat), so that it shares no summation with the float64 oracle
and its own rounding (a few times 1e-19 relative) is negligible next to a float64 kernel's.

Error bound of the kernels (u = 2^-53, the unit round-off of float64).  Every quantity of an update is a sum, product or
quotient of non-negative numbers: a sum of m non-negative terms has a relative error of at most (m - 1) u whatever the
order, a product or quotient adds u (the device's reciprocal-Newton division a few u), and relative errors of the operands
add up.  One model-4 update of slot (h, t) is
    count_n / s_n summed over the depth_t classes n hitting (h, t), times theta(h, t),
with s_n a sum of at most 8 k_max theta values (k_max pairs of a class, 8 haplotypes), so
    |got - want| / want <= (depth_t + 8 k_max + c) u.
Models 1-3 add the per-class gene / haplotype normalisers (at most 8 k_max terms each, three of them) and the gene sums
of theta (at most 8 g_max terms, g_max loci per gene, twice).  prepare() sums depth_t terms and, with a pseudocount, the
whole of theta twice (H T terms).  To first order the errors of k updates add up: k times the bound of one.  The bound is
the sum of these counts times u times SAFETY, computed from the shape; it is not fitted to any output."""
from __future__ import annotations

import numpy as np
import pytest

U = 2.0 ** -53
SAFETY = 4.0
C_OPS = 64  # divisions, products and the final rounding, generously
LD = np.longdouble
HAVE_LONGDOUBLE = np.finfo(LD).eps <= 1.1e-19


def require_longdouble():
    if not HAVE_LONGDOUBLE:
        pytest.skip(f"np.longdouble has eps {np.finfo(LD).eps:.3g} here: no extended precision to compare against")


class _Seg:
    """Segments of equal integer key: sums in longdouble by sorted reduceat, broadcast back to the elements."""

    def __init__(self, key):
        key = np.asarray(key, dtype=np.int64)
        self.order = np.argsort(key, kind="stable")
        ks = key[self.order]
        first = np.ones(ks.size, dtype=bool)
        first[1:] = ks[1:] != ks[:-1]
        self.starts = np.flatnonzero(first)
        self.keys = ks[self.starts]
        self.inv = np.empty(key.size, dtype=np.int64)
        self.inv[self.order] = np.cumsum(first) - 1

    def sums(self, v):
        return np.add.reduceat(v[self.order], self.starts) if v.size else v[:0]

    def back(self, v):
        return self.sums(v)[self.inv]


def _div_on_pattern(val, den):
    """structural zeros stay 0 (the reference divides on the numerator's pattern after eliminate_zeros())"""
    out = np.zeros_like(val)
    nz = val != 0
    out[nz] = val[nz] / den[nz]
    return out


class XRef:
    """One problem in entry form: entry e = (class n, locus t, haplotype h) for every set bit of every pair mask (minus the
    (h, t) slots a genotype mask removes)."""

    def __init__(self, d, gene_of, gtmask=None):
        H, T = d.H, d.T
        bits = ((np.asarray(d.pair_mask)[:, None].astype(np.int64) >> np.arange(H)) & 1).astype(bool)
        p, h = np.nonzero(bits)
        n, t = np.asarray(d.pair_class)[p], np.asarray(d.pair_locus)[p]
        if gtmask is not None:
            keep = np.asarray(gtmask)[h, t] != 0
            n, t, h = n[keep], t[keep], h[keep]
        self.H, self.T, self.N = H, T, d.N
        self.n, self.t, self.h = n, t, h
        self.count = np.asarray(d.count, dtype=np.float64).astype(LD)
        self.gene_of = np.asarray(gene_of, dtype=np.int64)
        G = int(self.gene_of.max()) + 1
        g = self.gene_of[t]
        self.G = G
        self.by_n, self.by_nt = _Seg(n), _Seg(n * T + t)
        self.by_ng, self.by_ngh = _Seg(n * G + g), _Seg((n * G + g) * H + h)
        self.by_ht = _Seg(h * T + t)
        self.gene_seg = _Seg(self.gene_of)
        self.depth = np.bincount(np.asarray(d.pair_locus), minlength=T)  # classes hitting each locus
        self.k_max = int(np.bincount(np.asarray(d.pair_class), minlength=1).max()) if d.pairs else 0
        self.g_max = int(np.bincount(self.gene_of).max())

    def sum_read(self, val):
        out = np.zeros(self.H * self.T, dtype=LD)
        out[self.by_ht.keys] = self.by_ht.sums(val * self.count[self.n])
        return out.reshape(self.H, self.T)

    def _normalize_read(self, val):
        return val / self.by_n.back(val)

    def e_step(self, theta, model):
        """posterior of every entry (EMfactory.update_probability_at_read_level)"""
        theta = np.asarray(theta).astype(LD)
        n, t, h = self.n, self.t, self.h
        val = theta[h, t]
        with np.errstate(divide="raise", invalid="raise", over="raise"):
            if model == 4:
                return self._normalize_read(val)
            if model not in (1, 2, 3):
                raise RuntimeError("The read normalization model should be 1, 2, 3, or 4.")
            hg = np.zeros((self.H, self.G), dtype=LD)
            hg[:, self.gene_seg.keys] = np.add.reduceat(theta[:, self.gene_seg.order], self.gene_seg.starts, axis=1)
            hg = hg[:, self.gene_of]  # per haplotype: theta summed over the locus' gene
            gamma = hg.sum(axis=0)
            if model == 3:
                val = _div_on_pattern(val, self.by_ng.back(val)) * gamma[t]
            elif model == 2:
                val = _div_on_pattern(val, self.by_nt.back(val)) * theta.sum(axis=0)[t]
                val = _div_on_pattern(val, self.by_ng.back(val)) * gamma[t]
            else:
                val = _div_on_pattern(val, self.by_ngh.back(val)) * hg[h, t]
                val = _div_on_pattern(val, self.by_ng.back(val)) * gamma[t]
            return self._normalize_read(val)

    def update(self, theta, model, efflen):
        """(expected read counts, theta') of one update_allelic_expression"""
        counts = self.sum_read(self.e_step(theta, model))
        return counts, counts / np.asarray(efflen).astype(LD)

    def prepare(self, efflen, pseudocount=0.0):
        val = self._normalize_read(np.ones(self.n.size, dtype=LD))
        theta = self.sum_read(val) / np.asarray(efflen).astype(LD)
        if pseudocount > 0.0:
            s = theta.sum()
            nzloci = np.nonzero(theta)[1]
            theta[:, nzloci] += LD(pseudocount)
            theta *= s / theta.sum()
        return theta

    def run(self, theta0, model, efflen, tol, max_iters):
        """EMfactory.run: updates until the TPM change drops to 1e6 * tol"""
        theta, errs, counts = np.asarray(theta0).astype(LD), [], None
        err = LD(1e6)
        while err > LD(1e6) * LD(tol) and len(errs) < max_iters:
            prev = theta.sum(axis=0)
            prev *= LD(1e6) / prev.sum()
            counts, theta = self.update(theta, model, efflen)
            curr = theta.sum(axis=0)
            curr *= LD(1e6) / curr.sum()
            err = np.abs(curr - prev).sum()
            errs.append(err)
        return dict(theta=theta, counts=counts, iters=len(errs), errs=np.array(errs, dtype=np.float64))

    # -- error bound ------------------------------------------------------------------------------------------------
    def rtol_update(self, model):
        return rtol_bound(self.depth, self.k_max, self.g_max, self.H, model, updates=1, prepare=False)

    def rtol_prepare(self, pseudocount=0.0):
        return rtol_bound(self.depth, self.k_max, self.g_max, self.H, 4, updates=0, pseudocount=pseudocount)

    def rtol_run(self, model, k, pseudocount=0.0):
        return rtol_bound(self.depth, self.k_max, self.g_max, self.H, model, updates=k, pseudocount=pseudocount)


def rtol_bound(depth, k_max, g_max, H, model, updates, prepare=True, pseudocount=0.0):
    """H x T bound (module docstring) on the relative error of a float64 computation of `updates` updates of `model`,
    after prepare() if `prepare`: depth = classes hitting each locus, k_max = pairs of the widest class, g_max = loci of
    the largest gene."""
    depth = np.asarray(depth, dtype=np.float64)
    per_update = depth + 8 * k_max + C_OPS + (0 if model == 4 else 3 * 8 * k_max + 2 * 8 * g_max)
    terms = updates * per_update
    if prepare:
        terms = terms + depth + C_OPS + (2 * H * depth.size if pseudocount > 0.0 else 0)
    return np.broadcast_to(SAFETY * terms * U, (H, depth.size))


def shape_of(d):
    """(depth per locus, k_max, g_max) of a SynthData, for rtol_bound"""
    return (np.bincount(np.asarray(d.pair_locus), minlength=d.T), int(np.bincount(np.asarray(d.pair_class)).max()),
            int(np.bincount(np.asarray(d.gene_of)).max()))


def assert_elementwise(got, want, rtol, what="", where=None):
    """got (float64) against want (exact or longdouble), element by element: finite, zero exactly where want is zero,
    |got - want| <= rtol |want| everywhere else -- no normalisation by the largest value, no absolute floor.  `where[t]`
    describes locus t in a failure report.  Returns the largest relative error."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    rtol = np.broadcast_to(np.asarray(rtol, dtype=np.float64), want.shape)

    def report(idx, msg):
        h, t = (int(i) for i in idx)
        extra = f"; locus {t}: {where[t]}" if where is not None else ""
        return f"{what}: {msg} at (h={h}, t={t}): got {got[h, t]!r}, want {float(want[h, t])!r}{extra}"

    bad = ~np.isfinite(got)
    assert not bad.any(), report(np.argwhere(bad)[0], f"{int(bad.sum())} non-finite values")
    zg, zw = got == 0, want == 0
    bad = zg != zw
    assert not bad.any(), report(np.argwhere(bad)[0], f"zero pattern differs in {int(bad.sum())} elements")
    if not (~zw).any():
        return 0.0
    rel = np.zeros(want.shape, dtype=LD)
    nz = ~zw
    rel[nz] = np.abs(got[nz].astype(LD) - want[nz].astype(LD)) / np.abs(want[nz].astype(LD))
    ratio = np.where(nz, rel.astype(np.float64) / rtol, 0.0)
    worst = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    assert ratio[worst] <= 1.0, report(worst, f"relative error {float(rel[worst]):.3e} over the bound {rtol[worst]:.3e}")
    return float(rel.max())


def random_theta(x: XRef, seed, zero_frac=0.05):
    """log-uniform over e^-40 .. e^40 on every (h, t) slot with an entry (haplotype-asymmetric), some of them exactly 0; no
    class left with theta 0 on all its entries (its normaliser would be 0 / 0)."""
    rng = np.random.default_rng(seed)
    support = np.zeros((x.H, x.T), dtype=bool)
    support[x.h, x.t] = True
    theta = np.where(support, np.exp(rng.uniform(-40.0, 40.0, (x.H, x.T))), 0.0)
    theta[support & (rng.random((x.H, x.T)) < zero_frac)] = 0.0
    alive = np.zeros(x.N, dtype=bool)
    np.logical_or.at(alive, x.n, theta[x.h, x.t] > 0)
    for n in np.flatnonzero(~alive & (np.bincount(x.n, minlength=x.N) > 0)):
        e = int(np.flatnonzero(x.n == n)[0])
        theta[x.h[e], x.t[e]] = np.exp(rng.uniform(-40.0, 40.0))
    return theta
