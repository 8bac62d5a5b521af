"""Host packer (gbrs_pack_create) -- structure invariants, sharding, masking.  CPU only: no compute call."""
import numpy as np
import pytest

from gbrs_b200 import _lib, synth
from gbrs_b200.apm import AlignmentPropertyMatrix
from gbrs_b200.emfactory import PackedPattern
from gbrs_b200.utils import gene_index
from oracle import em_oracle as eo
from tests import helpers as hp
from tests.packed_emulation import deinterleave, em_update_model4, unpack_entries


def make_apm(d):
    return synth.to_apm(d)


def class_signatures(d, hapmask=None):
    """multiset of (count, ((locus, mask), ...)) over non-empty classes of the input."""
    sig = {}
    for c, t, m in zip(d.pair_class, d.pair_locus, d.pair_mask):
        m = int(m) & (int(hapmask[t]) if hapmask is not None else 0xFF)
        if m:
            sig.setdefault(int(c), []).append((int(t), m))
    out = sorted((float(d.count[c]), tuple(sorted(v))) for c, v in sig.items())
    return out


def packed_signatures(p):
    a = p.arrays
    rp = a["rowptr"].astype(np.int64)
    out = []
    for n in range(p.info["n_classes"]):
        w = a["pairs"][rp[n]:rp[n + 1]].astype(np.int64)
        out.append((float(a["count"][n]), tuple(sorted((int(x & 0xFFFFFF), int(x >> 24)) for x in w))))
    return sorted(out)


@pytest.fixture(scope="module")
def small():
    return synth.generate(T=120, N=1500, H=8, with_genotype=True)


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    import re, os
    hdr = open(os.path.join(os.path.dirname(_lib.HERE), "include", "gbrs_em.h")).read()
    declared = set(re.findall(r"\b(gbrs_[a-z_0-9]+)\s*\(", hdr))
    declared -= {"gbrs_pack", "gbrs_em", "gbrs_prof"}
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.gbrs_abi_version() == _lib.ABI_VERSION


def test_pack_preserves_pattern(small):
    d = small
    p = PackedPattern(make_apm(d), gene_of=gene_index(d.T, d.groups()))
    assert p.info["n_pairs"] == d.pairs and p.info["nnz"] == d.nnz == p.info["nnz_total"]
    assert packed_signatures(p) == class_signatures(d)
    a = p.arrays
    # classes ordered by (number of pairs capped at KMAX+1, smallest locus, second-smallest locus); bucket tables consistent
    # with rowptr
    rp = a["rowptr"].astype(np.int64)
    loci = [np.sort(a["pairs"][rp[n]:rp[n + 1]] & 0xFFFFFF) for n in range(p.info["n_classes"])]
    minloc = np.array([x[0] for x in loci], dtype=np.int64)
    secloc = np.array([x[1] if len(x) > 1 else 0 for x in loci], dtype=np.int64)
    width = np.minimum(np.diff(rp), _lib.GBRS_KMAX + 1)
    key = (width * (1 << 24) + minloc) * (1 << 24) + secloc
    assert np.all(np.diff(key) >= 0)
    bc, bp = p.info["bucket_class0"], p.info["bucket_pair0"]
    assert bc[0] == 0 and bc[-1] == p.info["n_classes"] and bp[-1] == p.info["n_pairs"]
    for k in range(1, _lib.GBRS_KMAX + 1):
        assert np.all(width[bc[k - 1]:bc[k]] == k)
        assert bp[k - 1] == rp[bc[k - 1]] and bp[k] - bp[k - 1] == k * (bc[k] - bc[k - 1])
    # locus-major entries mirror the class-major pairs
    idx_c, m_c = unpack_entries(a["ent_cls"], p.info["entry_bytes"])
    idx_p, m_p = unpack_entries(a["ent_pair"], p.info["entry_bytes"])
    idx_r, m_r = unpack_entries(a["ent_run"], p.info["entry_bytes"])
    assert np.array_equal(m_c, m_p) and np.array_equal(m_c, m_r)
    assert len(m_c) == p.info["n_entries"] and np.count_nonzero(m_c) == p.info["n_pairs"]
    real = m_c != 0  # padding words: empty mask, index one past the last real one
    assert np.all(idx_c[~real] == p.info["n_classes"]) and np.all(idx_p[~real] == p.info["n_pairs"])
    assert np.all(idx_r[~real] == p.info["n_runs"])
    pairs_ext = np.append(a["pairs"].astype(np.int64), 0)
    pw = pairs_ext[idx_p]
    assert np.array_equal(pw >> 24, m_p)
    cls_of_pair = np.append(np.repeat(np.arange(p.info["n_classes"]), np.diff(rp)), p.info["n_classes"])
    assert np.array_equal(cls_of_pair[idx_p], idx_c)
    # items tile the entries; every item belongs to one locus; entries of a locus are ascending in class id
    io, lip = a["item_off"].astype(np.int64), a["locus_item_ptr"].astype(np.int64)
    assert io[0] == 0 and io[-1] == p.info["n_entries"] and np.all(np.diff(io) > 0) and np.all(io % 4 == 0)
    lens = np.diff(io)
    assert p.info["n_long_items"] == np.count_nonzero(lens > 64) and lens.max() <= 32 * 64
    locus_of_entry = pw & 0xFFFFFF
    # inside an item the ascending sequence is dealt round-robin over the lanes; undo that before looking at the order
    real_stored = real
    idx_c, m_c, real = deinterleave(idx_c, io), deinterleave(m_c, io), deinterleave(real, io)
    locus_of_entry = deinterleave(locus_of_entry, io)
    for t in range(d.T):
        lo, hi = (io[lip[t]], io[lip[t + 1]]) if lip[t + 1] > lip[t] else (0, 0)
        rl = real[lo:hi]
        assert np.all(locus_of_entry[lo:hi][rl] == t)
        if np.count_nonzero(rl) > 8 * 64:  # deep locus: partial-mask entries first, then the full ones
            full = m_c[lo:hi][rl] == 0xFF
            assert np.all(np.diff(full.astype(int)) >= 0)
            assert np.all(np.diff(idx_c[lo:hi][rl][~full]) > 0) and np.all(np.diff(idx_c[lo:hi][rl][full]) > 0)
        else:
            assert np.all(np.diff(idx_c[lo:hi][rl]) > 0)
    assert lip[-1] == p.info["n_items"]
    order = a["item_order"].astype(np.int64) & 0x7FFFFFFF
    isfull = a["item_order"].astype(np.int64) >> 31
    assert sorted(order) == list(range(p.info["n_items"]))
    for i, f in zip(order, isfull):  # full items hold only full-mask entries
        assert not f or np.all(np.isin(m_c[io[i]:io[i + 1]], (0, 0xFF)))
    desc = a["item_desc"].astype(np.int64).reshape(-1, 4)
    # two-descriptor trailer: where the short items change kind / size class in the visiting order (k_column_reduce)
    assert desc.shape[0] == p.info["n_items"] + 2
    tr, desc = desc[p.info["n_items"]:].ravel(), desc[:p.info["n_items"]]
    lens_d, nl = desc[:, 1] - desc[:, 0], p.info["n_long_items"]
    short_p = (np.arange(len(desc)) >= nl) & (desc[:, 3] == 0)
    short_f = (np.arange(len(desc)) >= nl) & (desc[:, 3] == 1)
    f0 = nl + short_p.sum()
    assert list(tr[:5]) == [nl + (short_p & (lens_d > 8)).sum(), nl + (short_p & (lens_d > 4)).sum(), f0,
                            f0 + (short_f & (lens_d > 8)).sum(), f0 + (short_f & (lens_d > 4)).sum()] and not tr[5:].any()
    assert np.array_equal(desc[:, 2], order) and np.array_equal(desc[:, 3], isfull)
    assert np.array_equal(desc[:, 0], io[order]) and np.array_equal(desc[:, 1], io[order + 1])
    lo_ = a["locus_order"].astype(np.int64)
    assert sorted(lo_) == list(range(d.T)) and np.all(np.diff(np.diff(lip)[lo_]) <= 0)
    lens_o = np.diff(io)[order]
    key = np.where(lens_o > 64, 0, 2) + isfull
    assert np.all(np.diff(key) >= 0) and np.all(np.diff(lens_o)[np.diff(key) == 0] <= 0)
    # runs: consecutive pairs of one class in the same gene
    g = gene_index(d.T, d.groups())[pw_locus(a)]
    idx_p, idx_r = idx_p[real_stored], idx_r[real_stored]
    runptr = a["runptr"].astype(np.int64)
    run_of_pair = np.zeros(p.info["n_pairs"], dtype=np.int64)
    for n in range(p.info["n_classes"]):
        gg = g[rp[n]:rp[n + 1]]
        assert np.all(np.diff(gg) >= 0)
        run_of_pair[rp[n]:rp[n + 1]] = runptr[n] + np.concatenate(([0], np.cumsum(np.diff(gg) != 0)))
        assert runptr[n + 1] - runptr[n] == 1 + np.count_nonzero(np.diff(gg))
    assert np.array_equal(run_of_pair[idx_p], idx_r)


def pw_locus(a):
    return a["pairs"].astype(np.int64) & 0xFFFFFF


def test_pack_genotype_mask(small):
    d = small
    gm = synth.genotype_mask(d)
    hapmask = (gm.T.astype(np.uint8) << np.arange(8, dtype=np.uint8)[None, :]).sum(axis=1).astype(np.uint8)
    p = PackedPattern(make_apm(d), hapmask=hapmask)
    assert packed_signatures(p) == class_signatures(d, hapmask)
    # same thing through the host container path used by quantify -G
    apm = make_apm(d)
    apm.multiply(gm, axis=2)
    apm.eliminate_zeros()
    assert apm.is_pure_incidence()
    p2 = PackedPattern(apm)
    assert packed_signatures(p2) == packed_signatures(p)


@pytest.mark.parametrize("R", [2, 3, 8])
def test_pack_shards_partition_the_classes(small, R):
    d = small
    apm = make_apm(d)
    shards = [PackedPattern(apm, shard_rank=r, shard_count=R) for r in range(R)]
    allsig = sorted(s for p in shards for s in packed_signatures(p))
    assert allsig == class_signatures(d)
    nnz = [p.info["nnz"] for p in shards]
    assert sum(nnz) == d.nnz and all(p.info["nnz_total"] == d.nnz for p in shards)
    assert max(nnz) - min(nnz) <= 0.1 * d.nnz / R + 64  # balanced by nnz


def test_pack_handles_unsorted_indices_and_empty_classes():
    d = synth.generate(T=40, N=300, H=4)
    apm = make_apm(d)
    rng = np.random.default_rng(1)
    for m in apm.data:  # shuffle the entries inside every column
        for t in range(d.T):
            seg = m.indices[m.indptr[t]:m.indptr[t + 1]]
            rng.shuffle(seg)
        m.has_sorted_indices = False
    apm.shape = (d.T, d.H, d.N + 7)  # trailing classes without any alignment
    apm.num_reads = d.N + 7
    apm.data = [type(m)((m.data, m.indices, m.indptr), shape=(d.N + 7, d.T)) for m in apm.data]
    apm.count = np.concatenate([d.count, np.ones(7)])
    p = PackedPattern(apm)
    assert p.info["n_classes"] == len(class_signatures(d)) and packed_signatures(p) == class_signatures(d)


def test_pack_limits():
    d = synth.generate(T=10, N=20, H=2)
    apm = make_apm(d)
    apm.shape = (10, 9, 20)
    apm.data = apm.data + [apm.data[0]] * 7
    with pytest.raises(NotImplementedError):
        PackedPattern(apm)


@pytest.mark.parametrize("name", ["em_small_m4", "em_small_m4_diploid", "em_small_m4_h2"])
def test_packed_layout_reproduces_reference_model4(name):
    """One prepare + a few model-4 updates computed by walking the packed arrays equal the golden trajectory."""
    g = hp.load_golden(name)
    d = hp.synth_from_golden(g)
    hapmask = None
    if g["masked"]:
        hapmask = (g["gtmask"].T.astype(np.uint8) << np.arange(8, dtype=np.uint8)[None, :]).sum(axis=1).astype(np.uint8)
    p = PackedPattern(make_apm(d), hapmask=hapmask, item_len=16)
    eff = np.ones((d.T, 8))
    eff[:, :d.H] = eo.effective_length_table(d.lengths).T
    _, theta = em_update_model4(p.arrays, p.info, d.T, None, eff, unit=True)
    assert hp.relerr(theta[:, :d.H].T, g["theta0"]) < 1e-12
    acc = None
    for _ in range(g["iters"]):
        acc, theta = em_update_model4(p.arrays, p.info, d.T, theta, eff)
    assert hp.relerr(theta[:, :d.H].T, g["theta"]) < 1e-10
    assert hp.relerr(acc[:, :d.H].T, g["counts"]) < 1e-10


def test_pack_wide_classes_go_to_the_long_bucket():
    d = synth.generate(T=300, N=2000, H=8, sample_index=8, wide_frac=0.1)
    p = PackedPattern(make_apm(d), gene_of=gene_index(d.T, d.groups()))
    assert packed_signatures(p) == class_signatures(d)
    bc = p.info["bucket_class0"]
    rp = p.arrays["rowptr"].astype(np.int64)
    widths = np.diff(rp)
    assert bc[_lib.GBRS_KMAX] < p.info["n_classes"] and np.all(widths[bc[_lib.GBRS_KMAX]:] > _lib.GBRS_KMAX)
    assert np.all(widths[:bc[_lib.GBRS_KMAX]] <= _lib.GBRS_KMAX) and p.info["max_pairs_per_class"] == widths.max()


def test_pack_wide_entry_words(monkeypatch):
    monkeypatch.setenv("GBRS_FORCE_ENTRY64", "1")
    d = synth.generate(T=60, N=500, H=8)
    p = PackedPattern(make_apm(d))
    assert p.info["entry_bytes"] == 8 and p.arrays["ent_cls"].dtype == np.uint64
    idx, m = unpack_entries(p.arrays["ent_cls"], 8)
    assert np.count_nonzero(m) == d.pairs and idx.max() == p.info["n_classes"]
    assert packed_signatures(p) == class_signatures(d)


_DIGEST = r'''
import sys, hashlib, json, os
sys.path.insert(0, os.environ["GBRS_ROOT"])
import numpy as np
from gbrs_b200 import synth, utils
from gbrs_b200.compress import read_rows
from gbrs_b200.emfactory import PackedPattern
from gbrs_b200.quantify import hapmask_bytes
h = hashlib.sha256()
for kw, shard, item_len, mask in ((dict(T=900, N=60000, H=8), (0, 1), 0, False),
                                  (dict(T=400, N=30000, H=8, wide_frac=0.05), (1, 3), 8, False),
                                  (dict(T=700, N=40000, H=8, with_genotype=True), (0, 1), 0, True),
                                  (dict(T=300, N=20000, H=3, sample_index=2), (0, 2), 0, False)):
    d = synth.generate(**kw)
    hm = hapmask_bytes(synth.genotype_mask(d)) if mask else None
    p = PackedPattern(synth.to_apm(d), gene_of=utils.gene_index(d.T, d.groups()), hapmask=hm, shard_rank=shard[0],
                      shard_count=shard[1], item_len=item_len)
    for k in sorted(p.arrays):
        h.update(k.encode()); h.update(np.ascontiguousarray(p.arrays[k]).tobytes())
    h.update(json.dumps(p.info, sort_keys=True).encode())
    rowptr, words = read_rows(synth.to_csc_list(d), d.T, d.H)
    h.update(rowptr.tobytes()); h.update(words.tobytes())
print(h.hexdigest())
'''


def test_packer_and_row_builder_do_not_depend_on_the_thread_count(tmp_path):
    """The threaded host packer (gbrs_pack_create) and read-row builder (gbrs_rows_create) split their work by class /
    locus / read ranges: every array must come out bit-identical with 1, 3 and 13 OpenMP threads (13 oversubscribes
    the test machine, which is what shakes out ordering assumptions)."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "digest.py"
    script.write_text(_DIGEST)
    seen = set()
    for threads in ("1", "3", "13"):
        env = dict(os.environ, GBRS_ROOT=root, OMP_NUM_THREADS=threads)
        res = subprocess.run([sys.executable, str(script)], env=env, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        seen.add(res.stdout.strip())
    assert len(seen) == 1, seen


# ---- the device-side packer (gpu_pack.cu) against the host packer: every array, bit for bit ---------------------------------
def _device_pack_cases():
    from gbrs_b200.quantify import hapmask_bytes

    d = synth.generate(T=200, N=3000, H=8, sample_index=4, with_genotype=True)
    return [
        (synth.generate(T=60, N=900, H=8, sample_index=2), {}),
        (synth.generate(T=120, N=1500, H=8, sample_index=9, wide_frac=0.08), dict(item_len=8)),
        (synth.generate(T=40, N=300, H=3, sample_index=1), dict(no_genes=True)),
        (d, dict(hapmask=hapmask_bytes(synth.genotype_mask(d)))),
        (synth.generate(T=150, N=2500, H=8, sample_index=5), dict(shard_rank=1, shard_count=3, item_len=8)),
        (synth.generate(T=30, N=200, H=1, sample_index=1), {}),
    ]


def _assert_same_pack(info, arrays, host):
    bad = [k for k in info if info[k] != host.info[k]]
    assert not bad, [(k, info[k], host.info[k]) for k in bad]
    for k, a in arrays.items():
        h = host.arrays[k]
        assert a.shape == h.shape and np.array_equal(a, h), k


@pytest.mark.skipif(__import__("shutil").which("g++") is None, reason="g++ is needed to build the SIMT emulation")
@pytest.mark.parametrize("case", range(6))
def test_emulated_device_packer_equals_host_packer(case):
    """gpu_pack.cu executed on the CPU through the host SIMT shim (CUB served by a stable sort and a loop)."""
    from gbrs_b200.emfactory import PackedPattern
    from oracle import em_oracle as eo
    from tests import simt_em

    d, kw = _device_pack_cases()[case]
    kw = dict(kw)
    gene_of = None if kw.pop("no_genes", False) else eo.gene_index(d.T, d.groups())
    apm = synth.to_apm(d)
    info, arrays = simt_em.emulated_device_pack(apm, gene_of=gene_of, **kw)
    _assert_same_pack(info, arrays, PackedPattern(apm, gene_of=gene_of, **kw))


@pytest.mark.skipif(__import__("shutil").which("g++") is None, reason="g++ is needed to build the SIMT emulation")
def test_emulated_device_packer_empty_classes_and_masked_loci():
    """The device packer's transposition (stable sort of the locus-major entries) on the corner cases of the class
    boundaries: classes without any alignment at the start, in the middle and at the end of the id range, loci the
    genotype byte removes completely, and a matrix that is empty after masking."""
    from scipy.sparse import csc_matrix

    from gbrs_b200 import AlignmentPropertyMatrix as APM
    from gbrs_b200.emfactory import PackedPattern
    from tests import simt_em

    rng = np.random.default_rng(5)
    T, H, N = 23, 4, 400
    dense = (rng.random((H, N, T)) < 0.04).astype(np.float64)
    dense[:, :37, :] = 0       # no alignments for the first classes ...
    dense[:, 150:171, :] = 0   # ... for a block in the middle ...
    dense[:, N - 29:, :] = 0   # ... and for the last ones
    apm = APM(shape=(T, H, N))
    apm.data = [csc_matrix(dense[h]) for h in range(H)]
    apm.count = rng.integers(1, 9, N).astype(np.float64)
    apm.finalize()
    mask = rng.integers(0, 1 << H, T).astype(np.uint8)
    mask[[3, 11]] = 0  # loci dropped completely
    for hapmask in (None, mask):
        info, arrays = simt_em.emulated_device_pack(apm, hapmask=hapmask)
        _assert_same_pack(info, arrays, PackedPattern(apm, hapmask=hapmask))
        assert 0 < info["n_classes"] <= N - 37 - 21 - 29
    # nothing survives the mask: an empty problem, the same numbers from both packers (zero-length arrays are not compared:
    # the device packer never hands out a zero-byte allocation)
    info, _ = simt_em.emulated_device_pack(apm, hapmask=np.zeros(T, dtype=np.uint8))
    host = PackedPattern(apm, hapmask=np.zeros(T, dtype=np.uint8))
    assert info["n_classes"] == 0 and info["n_pairs"] == 0 and info["nnz"] == 0
    assert not [k for k in info if info[k] != host.info[k]]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(6))
def test_device_packer_equals_host_packer(case):
    from gbrs_b200.emfactory import DevicePacked, PackedPattern
    from oracle import em_oracle as eo

    d, kw = _device_pack_cases()[case]
    kw = dict(kw)
    gene_of = None if kw.pop("no_genes", False) else eo.gene_index(d.T, d.groups())
    apm = synth.to_apm(d)
    dp = DevicePacked(apm, "cuda:0", gene_of=gene_of, **kw)
    _assert_same_pack(dp.info, dp.to_host(), PackedPattern(apm, gene_of=gene_of, **kw))


@pytest.mark.gpu
def test_device_packer_equals_host_packer_at_size():
    """1M classes at the C2 locus shape, 64-bit class indices in the input."""
    from gbrs_b200.emfactory import DevicePacked, PackedPattern
    from oracle import em_oracle as eo

    d = synth.generate(T=80_000, N=1_000_000, H=8)
    apm = synth.to_apm(d)
    for m in apm.data:
        m.indices = m.indices.astype(np.int64)
    gene_of = eo.gene_index(d.T, d.groups())
    dp = DevicePacked(apm, "cuda:0", gene_of=gene_of)
    _assert_same_pack(dp.info, dp.to_host(), PackedPattern(apm, gene_of=gene_of))
