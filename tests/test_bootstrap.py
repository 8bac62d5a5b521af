"""Bootstrap replicates on the CPU: the resampler kernels (gbrs_boot_guide / gbrs_boot_resample) and the zero-count row
pass of model 4, compiled for the host SIMT shim (tests/simt_em.py), against the numpy reference of tests/boot_ref.py;
one replicate end to end for models 1-4 against the extended-precision reference (tests/xref.py) on the compacted
matrix; and a statistical check of the numpy reference itself."""
import ctypes as C
import shutil

import numpy as np
import pytest

from gbrs_b200 import _lib, synth
from gbrs_b200.bootstrap import read_counts_of, replicate_indices
from oracle import em_oracle as eo
from tests import boot_ref as br
from tests import simt_em
from tests import simt_posterior as sp
from tests import xref as xr

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ is needed to build the SIMT emulation")

BOOT_SYMBOLS = ("gbrs_boot_scratch_bytes", "gbrs_boot_guide", "gbrs_boot_resample")


def emul_lib():
    lib = simt_em.load()
    for name in BOOT_SYMBOLS:
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = _lib.SYMBOLS[name]
    return lib


def emulated_resample(count, seed, replicates, class_id=None, N=None):
    """gbrs_boot_guide once, then gbrs_boot_resample per replicate on the emulated library -> [B][n_classes] doubles
    (`class_id` None: the identity, i.e. the whole histogram in input class order)."""
    lib = emul_lib()
    c = br.counts_of(count, N if count is None else len(count))
    N = c.shape[0]
    prefix = np.cumsum(c).astype(np.int64)
    M = int(prefix[-1])
    cid = np.arange(N, dtype=np.uint32) if class_id is None else np.ascontiguousarray(class_id, dtype=np.uint32)
    nbytes = C.c_int64()
    assert lib.gbrs_boot_scratch_bytes(N, C.byref(nbytes)) == 0
    raw = np.full(int(nbytes.value) + 256, 0xAB, np.uint8)  # garbage: the calls must not rely on a zeroed scratch
    scratch = raw.ctypes.data + (-raw.ctypes.data) % 256
    assert lib.gbrs_boot_guide(prefix.ctypes.data, N, M, scratch, int(nbytes.value), None) == 0, lib.gbrs_last_error()
    out = []
    for r in replicates:
        cnt = np.full(max(cid.shape[0], 1), np.nan)
        rc = lib.gbrs_boot_resample(prefix.ctypes.data, N, M, seed, r, cid.ctypes.data, cid.shape[0], scratch,
                                    int(nbytes.value), cnt.ctypes.data, None)
        assert rc == 0, lib.gbrs_last_error()
        out.append(cnt[: cid.shape[0]].copy())
    return np.array(out)


COUNT_CASES = {
    "M-even": np.array([3, 0, 5, 1, 7, 2, 0, 4], float),  # M = 22
    "M-odd": np.array([3, 0, 5, 1, 7, 2, 0, 5], float),  # M = 23
    "M=1": np.array([0, 0, 1, 0], float),
    "N=1": np.array([37], float),
    "zeros-at-ends": np.array([0, 0, 2, 9, 0, 1, 0, 0], float),
    "one-class-holds-almost-all": np.array([1, 0, 2000, 1, 1], float),
    "many-classes": np.random.default_rng(3).integers(0, 6, 700).astype(float),
}


def test_philox_known_answers():
    br.check_kat()


@pytest.mark.parametrize("case", sorted(COUNT_CASES))
def test_emulated_resampler_counts_equal_numpy(case):
    """Every replicate's histogram bit-identical to numpy; the counts sum to M exactly."""
    count = COUNT_CASES[case]
    M = int(count.sum())
    for seed in (0, 1, 0xDEADBEEF12345678):
        reps = (0, 1, 7, 0xFFFFFFFF)
        got = emulated_resample(count, seed, reps)
        for b, r in enumerate(reps):
            want = br.resample(count, seed, r)
            assert np.array_equal(got[b], want.astype(np.float64)), (case, seed, r, got[b], want)
            assert int(got[b].sum()) == M
            assert not np.any(got[b][count == 0])


def test_emulated_resampler_without_a_count_vector():
    got = emulated_resample(None, 5, (0, 3), N=50)
    for b, r in enumerate((0, 3)):
        assert np.array_equal(got[b], br.resample(None, 5, r, N=50).astype(np.float64))
        assert got[b].sum() == 50


@pytest.mark.parametrize("packer", ["host", "device"])
def test_emulated_resampler_scatters_through_class_id(packer):
    """count_out[p] = count of input class class_id[p], with the class order of either packer (-G restriction included,
    so that some input classes have no packed class)."""
    d = synth.generate(T=30, N=400, H=4, sample_index=1)
    apm = synth.to_apm(d)
    gene_of = eo.gene_index(d.T, d.groups())
    hapmask = np.random.default_rng(1).integers(1, 16, d.T).astype(np.uint8)
    if packer == "host":
        from gbrs_b200.emfactory import PackedPattern

        cid = PackedPattern(apm, gene_of=gene_of, hapmask=hapmask).arrays["class_id"].copy()
    else:
        cid = sp.emulated_device_class_id(apm, gene_of=gene_of, hapmask=hapmask)
    assert 0 < cid.shape[0] < d.N
    got = emulated_resample(d.count, 11, (0, 4), class_id=cid)
    for b, r in enumerate((0, 4)):
        assert np.array_equal(got[b], br.resample(d.count, 11, r)[cid].astype(np.float64))


def test_numpy_resampler_is_multinomial():
    """A guard on the reference itself: over B = 400 replicates the mean count of class n has variance
    c_n (1 - c_n / M) / B, so sum_n (mean - c)^2 / that variance is chi-square with N degrees of freedom."""
    count = np.random.default_rng(0).integers(1, 40, 60).astype(float)
    M, B = count.sum(), 400
    mean = np.mean([br.resample(count, 2024, r) for r in range(B)], axis=0)
    stat = float(np.sum((mean - count) ** 2 / (count * (1 - count / M) / B)))
    N = count.shape[0]
    assert abs(stat - N) <= 6 * np.sqrt(2 * N), stat


def test_refusals_of_the_host_checks():
    with pytest.raises(ValueError):
        replicate_indices([0, 2 ** 32])
    with pytest.raises(ValueError):
        replicate_indices([-1])
    with pytest.raises(ValueError):
        replicate_indices(2 ** 32 + 1)
    assert replicate_indices(3).tolist() == [0, 1, 2] and replicate_indices([5, 2]).tolist() == [5, 2]
    for bad in ([1.0, -1.0], [1.5, 2.0], [np.inf, 1.0], [2.0 ** 53, 1.0]):
        with pytest.raises(ValueError):
            read_counts_of(np.array(bad), 2)
    assert read_counts_of(None, 3).tolist() == [1, 1, 1]
    lib = emul_lib()
    nbytes = C.c_int64()
    assert lib.gbrs_boot_scratch_bytes(0, C.byref(nbytes)) == _lib.GBRS_E_ARG


# ---------------------------------------------------------------------------------------------------------------------
# one replicate end to end on the emulated library
# ---------------------------------------------------------------------------------------------------------------------
def emulated_replicate(d, gene_of, seed, r, model, tol=1e-3, max_iters=60, pseudocount=0.0):
    """What EMfactory.bootstrap does for one replicate, on the emulated library: resampled counts in packed order into the
    descriptor's count, the zero-count row pass, prepare + run."""
    pat = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of)
    cnt = emulated_resample(d.count, seed, (r,), class_id=pat.arr["class_id"])[0]
    pat.rep_count = np.ascontiguousarray(cnt)  # kept alive: the descriptor points at it
    pat.desc.count = pat.rep_count.ctypes.data
    pat.desc.zero_count_absent = 1
    pat.prepare(eo.effective_length_table(d.lengths), pseudocount)
    return pat.run(model, tol=tol, max_iters=max_iters)


@pytest.mark.parametrize("model", [4, 3, 2, 1])
def test_emulated_replicate_equals_the_em_of_the_compacted_matrix(model):
    """A replicate that drops the only class of a locus: that locus is exactly 0, every other element within the bound of
    the run, the same number of updates as the reference on the compacted matrix."""
    xr.require_longdouble()
    d = br.with_lonely_locus(synth.generate(T=24, N=160, H=4, sample_index=3))
    gene_of = eo.gene_index(d.T, d.groups())
    seed = br.seed_dropping(d.count, d.N - 1)
    counts = br.resample(d.count, seed, 0)
    assert counts[d.N - 1] == 0 and (counts == 0).sum() > 5
    out = emulated_replicate(d, gene_of, seed, 0, model)
    dc = br.compact_synth(d, counts)
    x = xr.XRef(dc, gene_of)
    eff = eo.effective_length_table(d.lengths)
    o = x.run(x.prepare(eff), model, eff, 1e-3, 60)
    assert out["iters"] == o["iters"], (out["iters"], o["iters"])
    rtol = x.rtol_run(model, o["iters"])
    xr.assert_elementwise(out["theta"], o["theta"], rtol, f"model {model} theta")
    xr.assert_elementwise(out["counts"], o["counts"], rtol, f"model {model} counts")
    assert not out["theta"][:, d.T - 1].any()


def test_emulated_zero_normaliser_of_a_present_class_still_raises():
    """Only a class of count 0 is absent: a class with a positive count whose entries all have theta 0 is 0 / 0."""
    d = br.with_lonely_locus(synth.generate(T=24, N=160, H=4, sample_index=3))
    gene_of = eo.gene_index(d.T, d.groups())
    pat = simt_em.HostPattern(synth.to_apm(d), gene_of=gene_of)
    pat.desc.zero_count_absent = 1
    pat.prepare()
    theta = pat.current_theta()
    theta[:, d.T - 1] = 0.0  # the lonely class (count 1) now has a zero normaliser
    staged = np.zeros((d.T, 8))
    staged[:, : d.H] = theta.T
    pat.check(pat.lib.gbrs_em_set_theta(C.byref(pat.desc), staged.ctypes.data, None))
    with pytest.raises(FloatingPointError):
        pat.run(4, tol=0.0, max_iters=1)
