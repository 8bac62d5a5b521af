"""`EMfactory` -- the reference's EM coordinator interface, backed by the sm_100a kernels.

Same constructor / methods / attributes as /root/reference/src/gbrs/emase/EMfactory.py:15-392
(`prepare`, `reset`, `get_allelic_expression`, `update_probability_at_read_level`,
`update_allelic_expression`, `run`, `report_read_counts`, `report_depths`, `export_posterior_probability`;
attributes `probability`, `allelic_expression`, `grp_conv_mat`, `t2t_mat`, `target_lengths`).

Host code stays Python; all arithmetic of the loop runs in libgbrs_em.so through ctypes (gbrs_b200/_lib.py).
PyTorch tensors are used purely as device buffers (`tensor.data_ptr()`), and `torch.distributed` supplies the one
exchange step of a row-sharded run (sum of the T x H numerator).  There is no CPU fallback: without the built
library or without a CUDA device every compute call raises.

Differences from the reference that a caller can observe (DESIGN.md section 6):
  * the EM never materialises the posterior P[n,t,h]; after `run`, `self.probability` still holds the incidence pattern.
    Expected read counts come from the device-side numerator (identical to `probability.sum(READ)` of the last
    posterior).  `posterior_probability()` computes, on request, the matrix the reference's `probability` holds after
    the last call: a new `AlignmentPropertyMatrix` with P on the EM's pattern (DESIGN.md section 7.1).
  * classes are re-ordered internally; class-indexed results are returned in the input's class order.
"""
from __future__ import annotations

import copy
import ctypes as C
import os
import time

import numpy as np

from . import _lib, bootstrap as _boot, utils
from .apm import AlignmentPropertyMatrix as APM

logger = utils.get_logger("gbrs")

ERR_LOG_CAP = 1 << 16

_PACK_ARRAYS = {  # name -> numpy dtype (None = entry word, depends on entry_bytes)
    "rowptr": np.uint32, "pairs": np.uint32, "count": np.float64, "runptr": np.uint32, "class_id": np.uint32,
    "ent_cls": None, "ent_pair": None, "ent_run": None, "item_off": np.uint32, "item_order": np.uint32, "item_desc": np.uint32, "locus_order": np.uint32, "locus_desc": np.uint32,
    "locus_item_ptr": np.uint32,
    "gene_ptr": np.uint32, "gene_loci": np.uint32, "gene_of": np.int32,
}


# Packed arrays only the row / column passes of models 1-3, the wide-class row pass and the alignment counts read: made
# resident on first use (a model-4 run streams none of them).  The host-only ones describe the layout and are never
# read by a kernel.
_LAZY_ARRAYS = ("rowptr", "runptr", "ent_pair", "ent_run")
_HOST_ONLY_ARRAYS = ("item_off", "item_order", "locus_order", "locus_item_ptr")
# Read by the posterior only (gbrs_em_posterior): uploaded by its first call, never by an EM run.
_POSTERIOR_ARRAYS = ("class_id",)


_STAGING: dict = {}  # (device, T) -> pinned [T][8] staging buffer shared by the patterns of a process (used synchronously)
_TILE_ARRAYS = ("tile_blob", "tile_desc", "tile_locus_desc")
_GENE_ARRAYS = ("gene_ptr", "gene_loci", "gene_of")


def _tile_params_from_env():
    """GBRS_TILE_PARAMS="max_classes=1024,max_loci=64,..." (tuning / test knob); default: the builder's defaults."""
    out = {}
    for item in os.environ.get("GBRS_TILE_PARAMS", "").split(","):
        if "=" in item:
            k, v = item.split("=", 1)
            out[k.strip()] = int(v)
    return out


def _torch():
    import torch

    return torch


def _require_cuda(device=None):
    torch = _torch()
    if not torch.cuda.is_available():
        raise _lib.GbrsCudaError("no CUDA device is available; the gbrs_b200 EM has no CPU fallback")
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return torch.device(device)


def pack_input(apm: APM, gene_of=None, hapmask=None, shard_rank=0, shard_count=1, item_len=0):
    """The `gbrs_pack_input` record for an incidence matrix (host packer and device packer take the same one) and the
    list of arrays that must stay alive while it is in use."""
    T, H, N = apm.shape
    if not apm.finalized:
        raise RuntimeError("The original matrix must be finalized.")
    if H > _lib.GBRS_HPAD:
        raise NotImplementedError("more than 8 haplotypes is not supported by the packed mask layout")
    mats = [m if m.format == "csc" else m.tocsc() for m in apm.data]
    indptr = [np.ascontiguousarray(m.indptr, dtype=np.int64) for m in mats]
    wide = any(m.indices.dtype.itemsize == 8 for m in mats)
    idx_t = np.int64 if wide else np.int32
    indices = [np.ascontiguousarray(m.indices, dtype=idx_t) for m in mats]
    keep = [indptr, indices]
    inp = _lib.PackInput()
    inp.T, inp.H, inp.N = T, H, N
    inp.indptr = (C.c_void_p * H)(*[a.ctypes.data for a in indptr])
    inp.indices = (C.c_void_p * H)(*[a.ctypes.data for a in indices])
    inp.index_bytes = 8 if wide else 4
    inp.values = None
    count = None
    if apm.count is not None:
        count = np.ascontiguousarray(apm.count, dtype=np.float64)
        if count.shape[0] != N:
            raise RuntimeError("count vector length does not match the number of classes")
        inp.count = count.ctypes.data
    if hapmask is not None:
        hapmask = np.ascontiguousarray(hapmask, dtype=np.uint8)
        inp.locus_hapmask = hapmask.ctypes.data
    if gene_of is not None:
        gene_of = np.ascontiguousarray(gene_of, dtype=np.int32)
        inp.gene_of = gene_of.ctypes.data
    inp.shard_rank, inp.shard_count, inp.item_len = shard_rank, shard_count, item_len
    keep += [count, hapmask, gene_of]
    return inp, keep


def posterior_pattern(apm: APM, hapmask=None) -> list:
    """Per haplotype (indptr int64, indices, stored values) of the pattern the EM runs on: the input CSC in canonical form
    (sorted indices, duplicates summed), with the (t, h) columns a genotype restriction `hapmask` removes emptied."""
    out = []
    for h, m in enumerate(apm.data):
        m = m if m.format == "csc" else m.tocsc()
        if not m.has_canonical_format:
            m = m.copy()
            m.sum_duplicates()
        indptr, indices, data = np.asarray(m.indptr, dtype=np.int64), m.indices, m.data
        if hapmask is not None:
            keep = ((np.asarray(hapmask) >> h) & 1).astype(bool)
            lens = np.diff(indptr)
            sel = np.repeat(keep, lens)
            indices, data = indices[sel], data[sel]
            indptr = np.concatenate(([0], np.cumsum(np.where(keep, lens, 0)))).astype(np.int64)
        out.append((indptr, indices, data))
    return out


class _PackHandle:
    """Owns one gbrs_pack_t; the numpy views handed out by PackedPattern keep it alive through their ctypes buffers."""

    def __init__(self, lib, handle):
        self.lib, self.handle = lib, handle

    def __del__(self):
        if self.handle is not None and self.lib is not None:
            try:
                self.lib.gbrs_pack_free(self.handle)
            except Exception:  # noqa: BLE001 - interpreter shutdown
                pass
            self.handle = None


class PackedPattern:
    """Host result of gbrs_pack_create for one row shard.  The arrays are views into the packer's own memory (no copy
    of the few hundred megabytes); every view keeps the C object alive for as long as it is referenced."""

    def __init__(self, apm: APM, gene_of=None, hapmask=None, shard_rank=0, shard_count=1, item_len=0):
        lib = _lib.load()
        T, H, N = apm.shape
        inp, keep = pack_input(apm, gene_of=gene_of, hapmask=hapmask, shard_rank=shard_rank, shard_count=shard_count,
                               item_len=item_len)
        handle = C.c_void_p()
        t0 = time.perf_counter()
        _lib.check(lib.gbrs_pack_create(C.byref(inp), C.byref(handle)))
        owner = _PackHandle(lib, handle)  # frees the C object when the last view is gone (also if a call below fails)
        info = _lib.PackInfo()
        _lib.check(lib.gbrs_pack_get_info(handle, C.byref(info)))
        self.info = {f: getattr(info, f) for f, _ in _lib.PackInfo._fields_}
        self.info["bucket_class0"] = list(info.bucket_class0)
        self.info["bucket_pair0"] = list(info.bucket_pair0)
        self.arrays = {}
        entry_t = np.uint32 if info.entry_bytes == 4 else np.uint64
        for name, dt in _PACK_ARRAYS.items():
            ptr, nbytes = C.c_void_p(), C.c_int64()
            _lib.check(lib.gbrs_pack_get_array(handle, name.encode(), C.byref(ptr), C.byref(nbytes)))
            dt = entry_t if dt is None else dt
            if nbytes.value == 0:
                self.arrays[name] = np.zeros(0, dtype=dt)
            else:
                buf = (C.c_uint8 * nbytes.value).from_address(ptr.value)
                buf._gbrs_owner = owner  # the view's base: keeps the packer's memory alive
                self.arrays[name] = np.frombuffer(buf, dtype=dt)
        self._owner = owner
        self.pack_seconds = time.perf_counter() - t0
        self.T, self.H, self.N = T, H, N
        self.has_genes = gene_of is not None
        del keep

    def nbytes(self) -> int:
        return int(sum(a.nbytes for a in self.arrays.values()))


class DevicePacked:
    """Result of gbrs_pack_device: the packed arrays live in device memory only (`tensors`: name -> uint8 torch tensor);
    `info` / `T` / `H` / `has_genes` / `pack_seconds` as on PackedPattern.  There is no host copy (`arrays` is empty)."""

    def __init__(self, apm: APM, device, gene_of=None, hapmask=None, shard_rank=0, shard_count=1, item_len=0):
        torch = _torch()
        lib = _lib.load()
        T, H, N = apm.shape
        inp, keep = pack_input(apm, gene_of=gene_of, hapmask=hapmask, shard_rank=shard_rank, shard_count=shard_count,
                               item_len=item_len)
        kept, temps = {}, []

        def alloc(nbytes, tag, _user):
            try:
                t = torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)
            except Exception:  # noqa: BLE001 - out of device memory: the C side reports it
                return None
            tag = tag.decode()
            if tag.startswith("tmp:"):
                temps.append(t)
            else:
                kept[tag] = (t, int(nbytes))
            return t.data_ptr()

        cb = _lib.ALLOC_FN(alloc)
        info, out = _lib.PackInfo(), _lib.DevicePack()
        t0 = time.perf_counter()
        with torch.cuda.device(device):
            stream = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
            _lib.check(lib.gbrs_pack_device(C.byref(inp), cb, None, stream, C.byref(info), C.byref(out)))
        self.pack_seconds = time.perf_counter() - t0
        del temps, keep
        self.info = {f: getattr(info, f) for f, _ in _lib.PackInfo._fields_}
        self.info["bucket_class0"] = list(info.bucket_class0)
        self.info["bucket_pair0"] = list(info.bucket_pair0)
        self.tensors = {k: t[:max(n, 1)] for k, (t, n) in kept.items()}
        self.nbytes_exact = {k: n for k, (t, n) in kept.items()}
        self.arrays = {}
        self.T, self.H, self.N = T, H, N
        self.has_genes = gene_of is not None

    def nbytes(self) -> int:
        return int(sum(self.nbytes_exact.values()))

    def to_host(self) -> dict:
        """The packed arrays as numpy arrays (tests: comparison with the host packer)."""
        entry_t = np.uint32 if self.info["entry_bytes"] == 4 else np.uint64
        out = {}
        for k, t in self.tensors.items():
            dt = _PACK_ARRAYS.get(k, np.uint8)
            dt = entry_t if dt is None else dt
            out[k] = t[: self.nbytes_exact[k]].cpu().numpy().view(dt).copy()
        return out


class _TilesHandle:
    def __init__(self, lib, handle):
        self.lib, self.handle = lib, handle

    def __del__(self):
        if self.handle is not None and self.lib is not None:
            try:
                self.lib.gbrs_tiles_free(self.handle)
            except Exception:  # noqa: BLE001 - interpreter shutdown
                pass
            self.handle = None


class TiledPattern:
    """Host result of gbrs_tiles_create: the tile blobs of the fused model-4 update (include/gbrs_em.h).  Views into the
    builder's memory, like PackedPattern."""

    def __init__(self, packed: PackedPattern, **params):
        lib = _lib.load()
        prm = _lib.TilesParams()
        for k, v in params.items():
            setattr(prm, k, int(v))
        handle = C.c_void_p()
        t0 = time.perf_counter()
        _lib.check(lib.gbrs_tiles_create(packed._owner.handle, C.byref(prm), C.byref(handle)))
        owner = _TilesHandle(lib, handle)
        info = _lib.TilesInfo()
        _lib.check(lib.gbrs_tiles_get_info(handle, C.byref(info)))
        self.info = {f: getattr(info, f) for f, _ in _lib.TilesInfo._fields_}
        self.arrays = {}
        for name, dt in (("blob", np.uint8), ("tile_desc", np.uint32), ("locus_desc", np.uint32)):
            ptr, nbytes = C.c_void_p(), C.c_int64()
            _lib.check(lib.gbrs_tiles_get_array(handle, name.encode(), C.byref(ptr), C.byref(nbytes)))
            if nbytes.value == 0:
                self.arrays[name] = np.zeros(0, dtype=dt)
            else:
                buf = (C.c_uint8 * nbytes.value).from_address(ptr.value)
                buf._gbrs_owner = owner
                self.arrays[name] = np.frombuffer(buf, dtype=dt)
        self._owner = owner
        self.build_seconds = time.perf_counter() - t0

    def nbytes(self) -> int:
        return int(sum(a.nbytes for a in self.arrays.values()))


class DevicePattern:
    """Packed incidence + state vectors resident on one GPU, and the `gbrs_em_dev` descriptor pointing at them."""

    def __init__(self, apm: APM = None, gene_of=None, hapmask=None, device=None, shard_rank=0, shard_count=1,
                 item_len=0, packed: PackedPattern = None, pin=False, tiles=None, tile_params=None, pack=None):
        """`tiles`: also build the tile layout and run model 4 / prepare through the fused single-pass tile kernel
        (`k_tile_em`) instead of the two-pass kernels.  Opt-in (`tiles=True` or GBRS_TILES=1): parity-green and
        bit-reproducible, but on B200 it is the slower of the two formulations at the benchmark shape (DESIGN.md
        section 4: both are bound by instruction issue, and the tile kernel issues more).  A class touching more loci
        than a tile may hold keeps the pattern on the two-pass kernels."""
        torch = _torch()
        self.device = _require_cuda(device)
        self.lib = _lib.load()
        if tiles is None:
            tiles = os.environ.get("GBRS_TILES", "0") not in ("", "0")
        # `pack`: "gpu" (default) packs on the device (gbrs_pack_device: the CSC arrays go up as they are, the packed
        # arrays never exist on the host); "host" uses the OpenMP packer (gbrs_pack_create) and uploads -- also taken when
        # the device packer refuses the input or the tile layout (built from the host arrays) is wanted
        if pack is None:
            pack = os.environ.get("GBRS_PACK", "gpu")
        if packed is None and pack == "gpu" and not tiles:
            try:
                packed = DevicePacked(apm, self.device, gene_of=gene_of, hapmask=hapmask, shard_rank=shard_rank,
                                      shard_count=shard_count, item_len=item_len)
            except NotImplementedError as e:  # GBRS_E_LIMIT
                logger.info(f"device packer not used ({e}); packing on the host")
        if packed is None:
            packed = PackedPattern(apm, gene_of=gene_of, hapmask=hapmask, shard_rank=shard_rank,
                                   shard_count=shard_count, item_len=item_len)
        self.packed = packed
        self.on_device = isinstance(packed, DevicePacked)
        self.info = packed.info
        self.T, self.H = packed.T, packed.H
        self.n_ranks = shard_count
        self.tiled = None
        if tiles and not self.on_device:
            try:
                self.tiled = TiledPattern(packed, **(tile_params or _tile_params_from_env()))
            except NotImplementedError as e:  # GBRS_E_LIMIT: a class wider than a tile
                logger.info(f"tile layout not used ({e}); model 4 runs on the two-pass kernels")
        self.host = {}
        arrays = dict(packed.arrays)
        if self.tiled is not None:
            arrays.update(tile_blob=self.tiled.arrays["blob"], tile_desc=self.tiled.arrays["tile_desc"],
                          tile_locus_desc=self.tiled.arrays["locus_desc"])
        for k, a in arrays.items():
            # torch has no uint32/uint64 arithmetic needs here: ship raw bytes
            t = torch.from_numpy(a.view(np.uint8))
            self.host[k] = t.pin_memory() if pin else t
        self.dev = {}
        self.h2d_bytes = 0
        self.full = False
        i = self.info
        self._need_rowptr = i["bucket_class0"][_lib.GBRS_KMAX] < i["n_classes"]  # classes wider than GBRS_KMAX
        if self.on_device:  # everything is resident already (the CSC arrays went up instead of the packed ones)
            self.dev = dict(packed.tensors)
            self.full = True
            self.h2d_bytes = int(sum(m.indices.nbytes + m.indptr.nbytes for m in apm.data)) + (
                apm.count.nbytes if apm.count is not None else 0)
        self.upload()
        self._alloc_state()
        self._build_descriptor()

    # -- device residency -------------------------------------------------------------------------------------------
    def upload(self, lazy=False):
        """Host -> device copy of the packed arrays a model-4 run needs (`lazy=True`: of the remaining ones; once the
        pattern is `full`, a plain upload() refreshes everything)."""
        torch = _torch()
        with torch.cuda.device(self.device):
            for k, t in self.host.items():
                if k in _HOST_ONLY_ARRAYS or (k in _POSTERIOR_ARRAYS and k not in self.dev):
                    continue
                is_lazy = self._is_lazy(k)
                if is_lazy != lazy and not (self.full and not lazy):
                    continue
                if t.numel() == 0:  # keep a valid (non-null) pointer for empty shards
                    self.dev[k] = torch.zeros(16, dtype=torch.uint8, device=self.device)
                elif k in self.dev and self.dev[k].numel() == t.numel():
                    self.dev[k].copy_(t, non_blocking=True)
                else:
                    self.dev[k] = t.to(self.device, non_blocking=True)
                self.h2d_bytes += t.numel()

    def _is_lazy(self, k):
        """Arrays a model-4 run does not read stay on the host until a model-1-3 update or an alignment-count call asks
        for them.  With the tile layout that is every array of the two-pass kernels."""
        if k in _TILE_ARRAYS or k in _GENE_ARRAYS:
            return False
        if self.tiled is not None:
            return True
        return k in _LAZY_ARRAYS and not (k == "rowptr" and self._need_rowptr)

    def ensure_arrays(self, names):
        """Make the named packed arrays resident (each is uploaded once; the descriptor is rebuilt if any was missing)."""
        torch = _torch()
        missing = [k for k in names if k not in self.dev]
        if not missing:
            return
        with torch.cuda.device(self.device):
            for k in missing:
                t = self.host[k]
                self.dev[k] = torch.zeros(16, dtype=torch.uint8, device=self.device) if t.numel() == 0 else t.to(self.device)
                self.h2d_bytes += t.numel()
        self._build_descriptor()

    def _weights_len(self, model1: bool) -> int:
        """Slots of the E-step weight vector: one per class (model 4), pair (2) or (class, gene) run (3); model 1 keeps
        eight per run -- six times the others at the benchmark shape, so that size is only allocated when model 1 runs.
        + 8 trailing slots that stay zero (padding entries point there)."""
        i = self.info
        runs = i["n_runs"] if self.packed.has_genes else 0
        return max(i["n_classes"], i["n_pairs"], runs, 8 * runs if model1 else 0, 1) + 8

    def ensure_full(self, model=None):
        """Make the arrays of models 1-3 / the alignment counts resident too (no-op once done).  `model`: the model about to
        run (None: any) -- model 1 needs the large weight vector."""
        torch = _torch()
        rebuilt = False
        if not self.full:
            self.upload(lazy=True)
            self.full = True
            if self.tiled is not None:  # work arrays of the two-pass kernels were placeholders
                i = self.info
                self.weights = torch.zeros(self._weights_len(False), dtype=torch.float64, device=self.device)
                self.wit = torch.zeros((max(i["n_items"], 1), 8), dtype=torch.float64, device=self.device)
            rebuilt = True
        if model in (None, 1) and self.weights.numel() < self._weights_len(True):
            self.weights = torch.zeros(self._weights_len(True), dtype=torch.float64, device=self.device)
            rebuilt = True
        if rebuilt:
            self._build_descriptor()

    def _alloc_state(self):
        torch = _torch()
        T, dv, f64 = self.T, self.device, torch.float64
        i = self.info
        nw = self._weights_len(False)  # (model 1 grows it: ensure_full)
        n_wit = max(i["n_items"], 1)
        if self.tiled is not None:  # two-pass work arrays are allocated by ensure_full()
            nw, n_wit = 8, 1
            self.tile_partial = torch.zeros((max(self.tiled.info["n_slots"], 1), 8), dtype=f64, device=dv)
        self.theta = torch.zeros((2, T, 8), dtype=f64, device=dv)
        self.efflen = torch.ones((T, 8), dtype=f64, device=dv)
        self.acc = torch.zeros((T, 8), dtype=f64, device=dv)
        self.iso = torch.zeros((2, T), dtype=f64, device=dv)
        self.weights = torch.zeros(nw, dtype=f64, device=dv)  # trailing slots stay zero (read by padding entries)
        self.subsets = torch.zeros((T, 32), dtype=f64, device=dv)
        self.wit = torch.zeros((n_wit, 8), dtype=f64, device=dv)
        self.part = torch.zeros(_lib.GBRS_PART_SLOTS, dtype=f64, device=dv)
        self.gene_hap = torch.zeros((max(i["n_gene_ids"], 1), 8), dtype=f64, device=dv)
        self.gamma = torch.zeros(T, dtype=f64, device=dv)
        self.err_log = torch.zeros(ERR_LOG_CAP, dtype=f64, device=dv)
        self.scal = torch.zeros(8, dtype=f64, device=dv)
        self.ctrl = torch.zeros(16, dtype=torch.int32, device=dv)

    def _build_descriptor(self):
        d = getattr(self, "desc", None) or _lib.EmDev()  # updated in place: callers may hold a reference
        i = self.info
        d.T, d.H, d.n_gene_ids, d.entry_bytes = self.T, self.H, i["n_gene_ids"], i["entry_bytes"]
        d.n_classes, d.n_pairs, d.n_runs, d.n_items = i["n_classes"], i["n_pairs"], i["n_runs"], i["n_items"]
        d.n_long_items, d.n_entries = i["n_long_items"], i["n_entries"]
        d.n_ranks, d.max_iters_cap = self.n_ranks, ERR_LOG_CAP
        d.n_deep_loci = i["n_deep_loci"]
        for k in range(_lib.GBRS_KMAX + 2):
            d.bucket_class0[k] = i["bucket_class0"][k]
            d.bucket_pair0[k] = i["bucket_pair0"][k]
        for k in ("rowptr", "pairs", "count", "runptr", "ent_cls", "ent_pair", "ent_run", "item_off", "item_order",
                  "item_desc", "locus_order", "locus_desc", "locus_item_ptr"):
            setattr(d, k, self.dev[k].data_ptr() if k in self.dev else None)
        if self.packed.has_genes:
            for k in ("gene_of", "gene_ptr", "gene_loci"):
                setattr(d, k, self.dev[k].data_ptr())
            d.gene_hap, d.gamma = self.gene_hap.data_ptr(), self.gamma.data_ptr()
        else:
            d.gene_of = d.gene_ptr = d.gene_loci = d.gene_hap = d.gamma = None
        for k in ("theta", "efflen", "acc", "iso", "weights", "subsets", "wit", "part", "err_log", "scal", "ctrl"):
            setattr(d, k, getattr(self, k).data_ptr())
        if self.tiled is not None:
            ti = self.tiled.info
            for k in _TILE_ARRAYS:
                setattr(d, k, self.dev[k].data_ptr())
            d.tile_partial = self.tile_partial.data_ptr()
            d.n_tiles, d.n_tile_slots = ti["n_tiles"], ti["n_slots"]
            d.tile_max_classes, d.tile_max_loci, d.tile_max_items = ti["max_classes"], ti["max_loci"], ti["max_items"]
            d.tile_max_a_bytes, d.tile_max_b_bytes = ti["max_part_a_bytes"], ti["max_part_b_bytes"]
            d.tile_n_deep_loci = ti["n_deep_loci"]
        else:
            d.tile_blob = d.tile_desc = d.tile_locus_desc = d.tile_partial = None
            d.n_tiles = d.n_tile_slots = 0
        self.desc = d

    def stream(self):
        torch = _torch()
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # -- small conveniences -----------------------------------------------------------------------------------------
    def _staging(self):
        """One pinned [T][8] host buffer for the small state transfers (theta, lengths, numerator): pageable copies of
        these 5 MB tables cost more than ten EM updates each."""
        if getattr(self, "_stage", None) is None:
            key = (str(self.device), self.T)
            if key not in _STAGING:  # pinning 5 MB costs about a millisecond: one buffer per (device, T) and process
                if len(_STAGING) >= 4:
                    _STAGING.pop(next(iter(_STAGING)))
                _STAGING[key] = _torch().empty((self.T, 8), dtype=_torch().float64).pin_memory()
            self._stage = _STAGING[key]
        return self._stage

    def _fetch_T8(self, dev_tensor) -> np.ndarray:
        """device [T][8] -> host H x T (contiguous copy).  The transpose is done on the device (a strided numpy copy of
        these 640k doubles costs as much as ten EM updates), the transfer goes through the pinned staging buffer."""
        st = self._staging().view(-1)[: self.H * self.T].view(self.H, self.T)
        st.copy_(dev_tensor[:, : self.H].t(), non_blocking=True)
        _torch().cuda.current_stream(self.device).synchronize()
        return st.numpy().copy()

    def _sync(self):
        _torch().cuda.current_stream(self.device).synchronize()

    def set_lengths(self, target_lengths_HT):
        """H x T effective lengths -> device [T][8] (1.0 in unused slots).  The pinned staging buffer is always filled
        by ONE contiguous copy: `EMfactory._read_lengths` hands over the transpose of a [T][H] table (already the device
        layout); a C-contiguous H x T table goes up as it is and is transposed on the device (a strided host copy of
        these 640k doubles costs more than ten EM updates)."""
        torch = _torch()
        if target_lengths_HT is None:
            self.efflen.fill_(1.0)
            return
        st = self._staging()
        src = np.asarray(target_lengths_HT, dtype=np.float64)
        if src.shape != (self.H, self.T):
            raise ValueError(f"effective lengths must be {self.H} x {self.T}, got {src.shape}")
        if src.T.flags.c_contiguous:  # [T][H] in memory
            if self.H < 8:
                st[:, self.H:] = 1.0
            st[:, : self.H].copy_(torch.from_numpy(src.T))
            self.efflen.copy_(st, non_blocking=True)
        else:
            flat = st.view(-1)[: self.H * self.T].view(self.H, self.T)
            flat.copy_(torch.from_numpy(np.ascontiguousarray(src)))
            on_dev = flat.to(self.device, non_blocking=True)
            if self.H < 8:
                self.efflen[:, self.H:] = 1.0
            self.efflen[:, : self.H].copy_(on_dev.t())
        self._sync()  # the staging buffer is reused

    def read_ctrl(self):
        ctrl = np.zeros(16, dtype=np.int32)
        scal = np.zeros(8, dtype=np.float64)
        _lib.check(self.lib.gbrs_em_read_ctrl(C.byref(self.desc), self.stream(), ctrl.ctypes.data, scal.ctypes.data))
        return ctrl, scal

    def current_theta_HT(self) -> np.ndarray:
        ctrl, _ = self.read_ctrl()
        return self._fetch_T8(self.theta[int(ctrl[_lib.CTRL_PARITY])])

    def set_theta_HT(self, theta_HT):
        st = self._staging()
        t = st.numpy()
        t[:] = 0.0
        t[:, : self.H] = np.asarray(theta_HT, dtype=np.float64).T
        staged = st.to(self.device, non_blocking=True)
        _lib.check(self.lib.gbrs_em_set_theta(C.byref(self.desc), C.c_void_p(staged.data_ptr()), self.stream()))
        _torch().cuda.current_stream(self.device).synchronize()

    def acc_HT(self) -> np.ndarray:
        return self._fetch_T8(self.acc)

    def copy_theta(self, previous: bool):
        """Device copy of the current theta (or, `previous`, of the one that entered the last update) into `post_theta`,
        the source of the next posterior; queued on the stream, no synchronisation."""
        if getattr(self, "post_theta", None) is None:
            self.post_theta = _torch().empty((self.T, 8), dtype=_torch().float64, device=self.device)
        _lib.check(self.lib.gbrs_em_copy_theta(C.byref(self.desc), int(previous), self.post_theta.data_ptr(), self.stream()))

    def posterior(self, model: int, theta_src, indptr, indices, reduce=None):
        """gbrs_em_posterior: P = theta_src[t][h] * W[idx(n,t,h)] on the output pattern `indptr[h]` / `indices[h]` (host CSC
        arrays of N x T, one pair per haplotype) -> list of H host value arrays.  `theta_src`: device [T][8].  `reduce`:
        a callable summing a device tensor over the ranks of a row-sharded run (every rank fills its own classes only);
        it also receives the error flag, so that every rank raises together."""
        torch = _torch()
        i = self.info
        need = ["class_id", "pairs"]
        if model != 4 or self._need_rowptr:
            need.append("rowptr")
        if model != 4:
            if not self.packed.has_genes:
                raise _lib.GbrsError("Group information matrix is missing.")
            need.append("runptr")
        self.ensure_arrays(need)
        N = int(self.packed.N)
        H = self.H
        nbytes = C.c_int64()
        _lib.check(self.lib.gbrs_em_posterior_scratch_bytes(C.byref(self.desc), int(model), N, C.byref(nbytes)))
        wide = any(a.dtype.itemsize == 8 for a in indices)
        with torch.cuda.device(self.device):
            scratch = torch.empty(int(nbytes.value), dtype=torch.uint8, device=self.device)
            d_ptr = [torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(self.device) for a in indptr]
            d_idx = [torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64 if wide else np.int32)).to(self.device)
                     for a in indices]
            vals = [torch.empty(max(int(a.shape[0]), 1), dtype=torch.float64, device=self.device) for a in indices]
            P = C.c_void_p * H
            rc = self.lib.gbrs_em_posterior(
                C.byref(self.desc), int(model), C.c_void_p(theta_src.data_ptr()),
                C.c_void_p(self.dev["class_id"].data_ptr()) if i["n_classes"] > 0 else None, N,
                P(*[t.data_ptr() for t in d_ptr]), P(*[t.data_ptr() for t in d_idx]), 8 if wide else 4,
                P(*[t.data_ptr() for t in vals]), C.c_void_p(scratch.data_ptr()), int(nbytes.value), self.stream())
            if reduce is not None:  # every rank learns whether any rank failed before anyone raises
                flag = torch.tensor([-rc], dtype=torch.int32, device=self.device)
                reduce(flag, "max")
                worst = -int(flag.item())
                if worst != _lib.GBRS_OK and rc == _lib.GBRS_OK:
                    raise FloatingPointError("non-finite posterior probability on another rank") \
                        if worst == _lib.GBRS_E_NUMERIC else _lib.GbrsError("posterior failed on another rank")
            _lib.check(rc)
            if reduce is not None:
                for v in vals:
                    reduce(v, "sum")
            return [v[: a.shape[0]].cpu().numpy() for v, a in zip(vals, indices)]

    def replicate_state(self, model: int):
        """A second state set over the same packed arrays, for bootstrap replicates: its own theta ping-pong, numerator,
        isoform totals, subset / weight / partial-sum / gene tables, control block and error log, and a count buffer at
        a fixed address (the captured loop of gbrs_em_run_cb is keyed by the descriptor, so one graph serves every
        replicate).  Lengths are shared.  Always the two-pass kernels (the tile blob holds its own copy of the counts), and
        the model-4 row pass treats a class of count 0 as absent.  Nothing of this pattern's own state is touched."""
        torch = _torch()
        self.ensure_full(model=4)  # every array of the two-pass kernels resident (a tiled pattern has them lazy)
        st = copy.copy(self)
        st.tiled, st.desc, st._stage = None, None, None
        st.dev = dict(self.dev)
        st._alloc_state()
        st.efflen = self.efflen
        if model == 1:
            st.weights = torch.zeros(st._weights_len(True), dtype=torch.float64, device=self.device)
        st.count = torch.zeros(max(self.info["n_classes"], 1), dtype=torch.float64, device=self.device)
        st.dev["count"] = st.count
        st._build_descriptor()
        st.desc.n_ranks = 1
        st.desc.zero_count_absent = 1
        return st

    def alignment_counts(self, gene_level=False, n_real_genes=0):
        torch = _torch()
        self.ensure_full(model=4)  # the run tables, not model 1's weight vector
        rows = n_real_genes if gene_level else self.T
        alloc = max(self.info["n_gene_ids"], rows) if gene_level else self.T
        aln = torch.zeros((alloc, 8), dtype=torch.float64, device=self.device)
        uniq = torch.zeros((alloc, 8), dtype=torch.float64, device=self.device)
        lu = torch.zeros(alloc, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.gbrs_em_alignment_counts(C.byref(self.desc), int(gene_level), int(n_real_genes),
                                                     aln.data_ptr(), uniq.data_ptr(), lu.data_ptr(), self.stream()))
        H = self.H
        return (np.ascontiguousarray(aln.cpu().numpy()[:rows, :H].T), np.ascontiguousarray(uniq.cpu().numpy()[:rows, :H].T),
                lu.cpu().numpy()[:rows].copy())


class EMfactory:
    """A class that coordinates Expectation-Maximization (reference EMfactory.py:15-24)."""

    def __init__(self, alignments: APM, device=None, group=None, shard: bool | str | None = None, item_len: int = 0,
                 poll_every: int = 4, locus_hapmask=None, tiles: bool | None = None, tile_params: dict | None = None,
                 pack: str | None = None):
        """`alignments`: the incidence matrix.  Additions to the reference signature (all optional):
        `device` CUDA device; `group` a torch.distributed process group (or `shard=True` for the default group) over
        which the alignment classes are row-sharded -- every rank passes the same full matrix and packs only its own
        contiguous slice; `shard="local"` says the matrix passed in already is this rank's slice (each rank loaded
        different classes); `item_len` / `poll_every` are tuning knobs (column-pass work item size, iterations queued
        between reads of the device-side stop flag); `locus_hapmask` (uint8 [T], bit h = haplotype h of the locus is
        kept) applies the `-G` genotype restriction while packing, which is equivalent to -- and much cheaper than --
        `alignments.multiply(gtmask, axis=2)` followed by `eliminate_zeros()` on the host matrices; `tiles` /
        `tile_params` select the fused single-pass tile kernel for model 4, `pack` ("gpu" | "host") where the incidence is
        packed (see DevicePattern)."""
        self.probability = alignments
        self._theta_host = None   # host copy of theta; fetched from the device on first use after it went stale
        self._theta_stale = False  # the device holds a newer estimate than `_theta_host`
        self._theta_dirty = False  # the host copy was assigned by the caller and not yet sent to the device
        self.grp_conv_mat = None
        self._t2t_mat = None
        self.target_lengths = None
        self._device = device
        self._group = group
        self._item_len = item_len or int(os.environ.get("GBRS_ITEM_LEN", "0"))
        self._hapmask = None if locus_hapmask is None else np.ascontiguousarray(locus_hapmask, dtype=np.uint8)
        if self._hapmask is not None and self._hapmask.shape != (alignments.num_loci,):
            raise ValueError("locus_hapmask must hold one byte per locus")
        self._poll_every = poll_every
        self._tiles, self._tile_params, self._pack = tiles, tile_params, pack
        self._pattern: DevicePattern | None = None
        self._weighted = False
        self._gene_of = None
        self._counts_host = None
        # what the reference's `probability` would hold after the last call (posterior_probability()): None before
        # prepare(); ("incidence",) after reset(); ("weighted",) after prepare() of a matrix with stored values;
        # ("theta", model) after an E-step / update, the source theta being the pattern's `post_theta` snapshot
        self._post = None
        self.num_iters = 0
        self.err_history = np.zeros(0)
        self.rank, self.world = 0, 1
        self.fused_exchange = False
        self.nvls_exchange = False
        self.exchange_mode = "nccl"
        if shard is None:
            shard = group is not None
        self._presharded = shard == "local"
        if shard:
            import torch.distributed as dist

            if dist.is_available() and dist.is_initialized():
                self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)

    # ---------------------------------------------------------------------------------------------------------------
    # attributes mirrored from the reference
    # ---------------------------------------------------------------------------------------------------------------
    @property
    def allelic_expression(self):
        return self._theta()

    @allelic_expression.setter
    def allelic_expression(self, value):
        self._theta_host = None if value is None else np.array(value, dtype=np.float64, copy=True)
        self._theta_dirty = value is not None
        self._theta_stale = False

    def _theta(self):
        """The host copy of theta, fetched lazily: prepare() / run() / an update only mark it stale, so a caller that never
        looks (the cohort loop between prepare and run) pays no device-to-host copy."""
        if self._theta_stale and self._pattern is not None:
            self._theta_host = self._pattern.current_theta_HT()
            self._theta_stale = False
        return self._theta_host

    @property
    def t2t_mat(self):
        """T x T CSC: identity plus all same-gene pairs (EMfactory.py:48-59).  Built only on demand -- the kernels
        use the equivalent `gene_of` table."""
        if self._t2t_mat is None and self.grp_conv_mat is not None:
            from scipy.sparse import eye

            m = (self.grp_conv_mat @ self.grp_conv_mat.T + eye(self.probability.num_loci)).tocsc()
            m.data[:] = 1.0
            self._t2t_mat = m
        return self._t2t_mat

    # ---------------------------------------------------------------------------------------------------------------
    def _read_lengths(self, lenfile, read_length):
        """EMfactory.prepare length handling (EMfactory.py:60-94).  The reference walks the file line by line in
        Python (seconds at 640k lines); the table is parsed in bulk here and the line loop is kept as the fallback for
        anything unusual, so malformed files raise exactly what the reference raises."""
        p = self.probability
        tl = None
        if p.num_haplotypes > 0:
            try:
                tl = self._read_lengths_bulk(lenfile, read_length)
            except Exception:  # noqa: BLE001 - odd file: let the reference's loop decide what the error is
                tl = None
        if tl is None:
            tl = self._read_lengths_loop(lenfile, read_length)
        tl = tl.transpose()
        if not np.all(tl > 0.0):
            raise RuntimeError("There exist transcripts missing length information.")
        return tl

    def _read_lengths_bulk(self, lenfile, read_length):
        """Native parser (gbrs_parse_lengths); None if it met a line it does not take as well-formed."""
        p = self.probability
        lib = _lib.load()
        lnames = [str(x).encode() for x in p.lname]
        hnames = [str(x).encode() for x in p.hname]
        if len(set(lnames)) != len(lnames):
            return None
        c_l = (C.c_char_p * len(lnames))(*lnames)
        c_h = (C.c_char_p * len(hnames))(*hnames)
        tl = np.zeros((p.num_loci, p.num_haplotypes))
        bad = C.c_int64(0)
        _lib.check(lib.gbrs_parse_lengths(str(lenfile).encode(), c_l, p.num_loci, c_h, p.num_haplotypes,
                                          float(read_length), tl.ctypes.data, C.byref(bad)))
        return None if bad.value else tl

    def _read_lengths_loop(self, lenfile, read_length):
        p = self.probability
        hid = dict(zip(p.hname, np.arange(len(p.hname))))
        tl = np.zeros((p.num_loci, p.num_haplotypes))
        if p.num_haplotypes > 1:
            with open(lenfile) as fh:
                for curline in fh:
                    item = curline.rstrip().split("\t")
                    locus, hap = item[0].split("_")
                    tl[p.lid[locus], hid[hap]] = max(float(item[1]) - read_length + 1.0, 1.0)
        elif p.num_haplotypes > 0:
            with open(lenfile) as fh:
                for curline in fh:
                    item = curline.rstrip().split("\t")
                    tl[p.lid[item[0]], 0] = max(float(item[1]) - read_length + 1.0, 1.0)
        else:
            raise RuntimeError("There is something wrong with your emase-format alignment file.")
        return tl

    def _ensure_pattern(self):
        if self._pattern is None:
            p = self.probability
            # Stored values other than 1.0 (weighted or legacy files, explicit zeros): the reference's E-step starts with
            # probability.reset(), which sets EVERY stored entry to 1 (Sparse3DMatrix.py:220-228) -- so the EM runs on the
            # stored pattern, zeros included, and the values matter to prepare()'s initial normalisation only
            # (EMfactory.py:95-104).  The pattern is packed as it is; reset() takes theta0 from the values on the host.
            self._weighted = not p.is_pure_incidence(cache=True)
            if self._presharded:
                self._pattern = DevicePattern(p, gene_of=self._gene_of, hapmask=self._hapmask, device=self._device,
                                              item_len=self._item_len, tiles=self._tiles, tile_params=self._tile_params,
                                              pack=self._pack)
                self._pattern.n_ranks = self.world
                self._pattern._build_descriptor()
            else:
                self._pattern = DevicePattern(p, gene_of=self._gene_of, hapmask=self._hapmask, device=self._device,
                                              shard_rank=self.rank, shard_count=self.world, item_len=self._item_len,
                                              tiles=self._tiles, tile_params=self._tile_params, pack=self._pack)
            self._pattern.set_lengths(self.target_lengths)
            if self.world > 1:
                self.fused_exchange = self._setup_fused_exchange(self._pattern)
        return self._pattern

    def _exchange(self, pat):
        """The one exchange step of a row-sharded run: sum the T x H numerator over ranks (SURVEY.md 8e).  With the
        fused NVLink exchange enabled the kernels do it themselves (k_locus_acc -> k_xchg_reduce -> k_locus_update over
        peer memory) and this is a no-op; otherwise NCCL all-reduces `acc` in place."""
        if self.world > 1 and not pat.desc.xchg_enabled:
            import torch.distributed as dist

            dist.all_reduce(pat.acc, op=dist.ReduceOp.SUM, group=self._group)

    def _setup_fused_exchange(self, pat):
        """Give the kernels every rank's exchange buffer as peer memory (torch symmetric memory does the mapping:
        PyTorch as plumbing).  Falls back to the NCCL all-reduce if any rank cannot set it up."""
        torch = _torch()
        import torch.distributed as dist

        # GBRS_XCHG: push (default; also "fused") the one-launch push form | pull (also "p2p") the round-1 pull form: the
        # owner of a slice loads it from every peer | nvls: pull form with the in-switch reduction where the box has a
        # multicast mapping (a multimem f64 access moves 8 bytes per request: measured slower than peer loads on 2 and on
        # 8 ranks) | nccl: plain all-reduce between the two halves of an update.
        # tag: the push form without any flag -- every double carries its own "arrived" bit (the sign bit, free because the
        # numerator is non-negative) and is polled by the thread that needs it: no tickets, no fences, no handshakes.
        mode = os.environ.get("GBRS_XCHG", "push")
        mode = {"fused": "push", "p2p": "pull"}.get(mode, mode)
        if self.world < 2 or self.world > 8 or mode not in ("push", "tag", "pull", "nvls"):
            return False
        # the multicast mapping: the in-switch reduction of the nvls form; in the push form only the broadcast of the
        # slice totals goes through it (one 16-byte store replicated by the switch instead of one per peer)
        use_mc = mode == "nvls" or (mode in ("push", "tag") and os.environ.get("GBRS_XCHG_MC", "1") != "0")
        ok, buf, hdl, mc = 1, None, None, 0
        try:
            import torch.distributed._symmetric_memory as symm_mem

            if mode in ("push", "tag"):  # recv[R][slice] | total | flags (include/gbrs_em.h)
                slice_len = ((8 * pat.T + self.world - 1) // self.world + 1) & ~1
                n_doubles = self.world * slice_len + 8 * pat.T + 16
            else:  # acc_local | acc_total | flags
                n_doubles = 2 * 8 * pat.T + 16
            buf = symm_mem.empty(n_doubles, dtype=torch.float64, device=pat.device)
            buf.zero_()
            hdl = symm_mem.rendezvous(buf, group=self._group if self._group is not None else dist.group.WORLD)
            ptrs = list(hdl.buffer_ptrs)
            if len(ptrs) != self.world or any(int(p) == 0 for p in ptrs):
                ok = 0
            mc = int(getattr(hdl, "multicast_ptr", 0) or 0) if use_mc else 0
        except Exception as e:  # noqa: BLE001 - any failure means "use NCCL"
            logger.info(f"fused NVLink exchange unavailable ({e}); using the NCCL all-reduce")
            ok = 0
        # every rank must take the same path: fused only if all could map the buffers, NVLS only if all have the multicast
        flag = torch.tensor([ok, 1 if (ok and mc) else 0], dtype=torch.int32, device=pat.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self._group)  # also orders the zero-fill before first use
        torch.cuda.synchronize(pat.device)
        if int(flag[0].item()) != 1:
            return False
        self.nvls_exchange = bool(int(flag[1].item()))
        pat._xchg = (buf, hdl)
        pat.desc.xchg_enabled = {"push": 2, "tag": 3}.get(mode, 1)
        pat.desc.xchg_timeout_ms = int(os.environ.get("GBRS_XCHG_TIMEOUT_MS", "0"))
        self.exchange_mode = mode
        pat.desc.xchg_mc = mc if self.nvls_exchange else None
        pat.desc.xchg_rank = self.rank
        for r in range(self.world):
            pat.desc.xchg_peer[r] = int(ptrs[r])
        return True

    def _run_sharded(self, pat, model, tol, max_iters, on_poll=None):
        """Row-sharded loop: `poll_every` updates (local passes -> all-reduce of the numerator -> update + stop test)
        are captured once into a CUDA graph and replayed until the device-side stop flag is read back as set.  Every rank
        sees the same all-reduced numerator, hence the same error and the same decision, so no second collective is
        needed for the stop test."""
        torch = _torch()
        import torch.distributed as dist

        def body():
            for _ in range(self._poll_every):
                _lib.check(pat.lib.gbrs_em_launch_local(C.byref(pat.desc), model, pat.stream()))
                self._exchange(pat)
                _lib.check(pat.lib.gbrs_em_launch_update(C.byref(pat.desc), pat.stream()))

        use_graph = os.environ.get("GBRS_NO_GRAPH") is None and dist.get_backend(self._group) == "nccl"
        side = torch.cuda.Stream(device=pat.device)
        side.wait_stream(torch.cuda.current_stream(pat.device))
        with torch.cuda.stream(side):
            _lib.check(pat.lib.gbrs_em_run_begin(C.byref(pat.desc), tol, max_iters, pat.stream()))
            ctrl, _ = pat.read_ctrl()
            graph = None
            if use_graph and not ctrl[_lib.CTRL_DONE]:
                scratch = torch.zeros(8, dtype=torch.float64, device=pat.device)
                dist.all_reduce(scratch, group=self._group)  # communicator set-up must not happen during capture
                side.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side):
                    body()
            reported = 0
            while not ctrl[_lib.CTRL_DONE]:
                if graph is not None:
                    graph.replay()
                else:
                    body()
                ctrl, _ = pat.read_ctrl()
                if on_poll is not None and ctrl[_lib.CTRL_ITERS] > reported:
                    on_poll(reported, pat.err_log[reported:int(ctrl[_lib.CTRL_ITERS])].cpu().numpy())
                    reported = int(ctrl[_lib.CTRL_ITERS])
        torch.cuda.current_stream(pat.device).wait_stream(side)
        side.synchronize()
        return ctrl

    def _sync_theta_to_device(self):
        if self._theta_dirty:
            self._ensure_pattern().set_theta_HT(self._theta_host)
            self._theta_dirty = False

    def _fetch_theta(self):
        self._theta_stale = True
        self._theta_dirty = False

    # ---------------------------------------------------------------------------------------------------------------
    def prepare(self, pseudocount: float = 0.0, lenfile: str = None, read_length: int = 100) -> None:
        """Initializes the probability of read origin according to the alignment profile (EMfactory.py:27-111)."""
        p = self.probability
        if p.num_groups > 0:
            self.grp_conv_mat = utils.group_conversion_matrix(p.num_loci, p.groups)
            self._gene_of = utils.gene_index(p.num_loci, p.groups)
        if lenfile is not None:
            self.target_lengths = self._read_lengths(lenfile, read_length)
        self._pattern = None
        self.reset(pseudocount)
        if self._weighted:  # prepare() normalises the stored values; reset() replaces them by ones first
            self._post = ("weighted",)

    def reset(self, pseudocount: float = 0.0) -> None:
        """EMfactory.reset (EMfactory.py:113-138): theta0 from the incidence pattern."""
        fresh = self._pattern is None
        pat = self._ensure_pattern()
        if not fresh:  # a new pattern has just been given the lengths
            pat.set_lengths(self.target_lengths)
        if self._weighted:
            if self.world > 1:
                raise NotImplementedError("weighted alignment matrices are not supported in row-sharded runs")
            pat.set_theta_HT(self._weighted_theta0(float(pseudocount)))
        else:
            _lib.check(pat.lib.gbrs_em_prepare_local(C.byref(pat.desc), pat.stream()))
            self._exchange(pat)
            _lib.check(pat.lib.gbrs_em_prepare_finish(C.byref(pat.desc), float(pseudocount), pat.stream()))
        ctrl, _ = pat.read_ctrl()
        self._raise_on_ctrl_error(ctrl, "the initial expression estimate")
        self._fetch_theta()
        self._counts_host = None
        self._post = ("incidence",)
        self.num_iters = 0

    def _weighted_theta0(self, pseudocount: float) -> np.ndarray:
        """prepare()'s initial estimate for a matrix with stored values (EMfactory.py:95-111): normalize_reads(READ) on
        the values, count-weighted column sums, division by the effective lengths, pseudocount rule.  Host, one pass --
        initialisation only; the EM itself runs on the device on the stored pattern."""
        p = self.probability
        H, T = p.num_haplotypes, p.num_loci
        rows = np.zeros(p.shape[2])
        for m in p.data:
            rows += np.asarray(m.sum(axis=1)).ravel()
        cnt = np.ones(p.shape[2]) if p.count is None else np.asarray(p.count, dtype=np.float64)
        with np.errstate(divide="ignore", invalid="ignore"):
            scale = np.where(rows != 0.0, cnt / rows, 0.0)
        theta = np.vstack([np.asarray(m.T @ scale).ravel() for m in p.data])
        if self.target_lengths is not None:
            theta = theta / self.target_lengths
        if pseudocount > 0.0:
            total = theta.sum()
            nz = np.nonzero(theta)[1]
            theta[:, nz] += pseudocount
            theta *= total / theta.sum()
        assert theta.shape == (H, T)
        return theta

    def get_allelic_expression(self, at_group_level: bool = False):
        if at_group_level:
            return self._theta() * self.grp_conv_mat
        return self._theta().copy()

    def update_probability_at_read_level(self, model: int = 3) -> None:
        """E-step (EMfactory.py:146-212).  On the device the posterior is implicit: this queues the row pass and
        the column reduce for `model`, leaving the count-weighted numerator sum_n c[n] P[n,t,h] in `acc` -- and nothing
        else: like the reference's method it can be called repeatedly and does not move theta."""
        if model not in (1, 2, 3, 4):
            raise RuntimeError("The read normalization model should be 1, 2, 3, or 4.")
        pat = self._ensure_pattern()
        if model != 4:
            pat.ensure_full(model)
        self._sync_theta_to_device()
        _lib.check(pat.lib.gbrs_em_run_begin(C.byref(pat.desc), 0.0, 1, pat.stream()))
        _lib.check(pat.lib.gbrs_em_launch_estep(C.byref(pat.desc), int(model), pat.stream()))
        if self.world > 1:  # the stand-alone E-step never uses the fused exchange (it must not touch its flags)
            import torch.distributed as dist

            dist.all_reduce(pat.acc, op=dist.ReduceOp.SUM, group=self._group)
        self._counts_host = None
        pat.copy_theta(previous=False)  # theta does not move: the posterior is the E-step of the current one
        self._post = ("theta", int(model))

    def update_allelic_expression(self, model: int = 3) -> None:
        """A single EM step (EMfactory.py:214-232): E-step, then theta = numerator / effective length."""
        if model not in (1, 2, 3, 4):
            raise RuntimeError("The read normalization model should be 1, 2, 3, or 4.")
        pat = self._ensure_pattern()
        if model != 4:
            pat.ensure_full(model)
        self._sync_theta_to_device()
        _lib.check(pat.lib.gbrs_em_run_begin(C.byref(pat.desc), 0.0, 1, pat.stream()))
        _lib.check(pat.lib.gbrs_em_launch_local(C.byref(pat.desc), int(model), pat.stream()))
        self._exchange(pat)
        _lib.check(pat.lib.gbrs_em_launch_update(C.byref(pat.desc), pat.stream()))
        ctrl, _ = pat.read_ctrl()
        self._raise_on_ctrl_error(ctrl)
        self._fetch_theta()
        self._counts_host = None
        self._snapshot_posterior_source(pat, model, 1)

    def _snapshot_posterior_source(self, pat, model, n_updates):
        """After `n_updates` updates the posterior of the reference's `probability` is the E-step of the theta that
        entered the last one.  The loop has flipped the ping-pong after it (updates queued past the stop are no-ops), so
        that theta is the other half; it is copied before a later set_theta (e.g. after report_depths' in-place TPM
        scaling) can overwrite it.  No update: the previous posterior stays."""
        if n_updates > 0:
            pat.copy_theta(previous=True)
            self._post = ("theta", int(model))

    @staticmethod
    def _raise_on_ctrl_error(ctrl, what="the EM update"):
        """Device error flag -> the exception the reference (or the exchange) would raise."""
        err = int(ctrl[_lib.CTRL_ERROR])
        if err == 3:
            raise _lib.GbrsError("fused NVLink exchange timed out waiting for a peer rank")
        if err:
            raise FloatingPointError(f"non-finite value in {what} (zero normaliser or overflow)")

    def run(self, model: int, tol: float = 0.001, max_iters: int = 999, verbose: bool = True) -> None:
        """Runs EM iterations (EMfactory.py:234-287); the stop test runs on the device."""
        if model not in (1, 2, 3, 4):
            raise RuntimeError("The read normalization model should be 1, 2, 3, or 4.")
        if max_iters > ERR_LOG_CAP:
            raise ValueError(f"max_iters above {ERR_LOG_CAP} is not supported")
        pat = self._ensure_pattern()
        if model != 4:
            pat.ensure_full(model)
        self._sync_theta_to_device()
        show = verbose and self.rank == 0  # one table, from rank 0 (a sharded run would print it world times)
        if show:
            print("")
            print("Iter No  Time (hh:mm:ss)    Total change (TPM)  ")
            print("-------  ---------------  ----------------------")
        time0 = time.time()

        def print_rows(first, errs):
            # one row per iteration as the polls come back, stamped with the time of that poll (EMfactory.py:280-287)
            delmin, sec = divmod(int(time.time() - time0), 60)
            h, m = divmod(delmin, 60)
            for i, e in enumerate(errs):
                print(" %5d      %4d:%02d:%02d     %9.1f / 1000000" % (first + i + 1, h, m, sec, e), flush=True)

        if self.world == 1:
            iters = C.c_int32(0)
            errs = np.zeros(max(max_iters, 1), dtype=np.float64)
            cb = _lib.POLL_CB(lambda first, n, p, _u: print_rows(first, [p[i] for i in range(n)])) if show else None
            rc = pat.lib.gbrs_em_run_cb(C.byref(pat.desc), int(model), float(tol), int(max_iters), int(self._poll_every),
                                        pat.stream(), C.byref(iters), errs.ctypes.data,
                                        C.cast(cb, C.c_void_p) if cb is not None else None, None)
            _lib.check(rc)
            n = int(iters.value)
            self.err_history = errs[:n].copy()
        else:
            ctrl = self._run_sharded(pat, int(model), float(tol), int(max_iters), on_poll=print_rows if show else None)
            self._raise_on_ctrl_error(ctrl)
            n = int(ctrl[_lib.CTRL_ITERS])
            self.err_history = pat.err_log[:n].cpu().numpy()
        self.num_iters = n
        self._fetch_theta()
        self._counts_host = None
        self._snapshot_posterior_source(pat, model, n)

    # ---------------------------------------------------------------------------------------------------------------
    # bootstrap replicates
    # ---------------------------------------------------------------------------------------------------------------
    def bootstrap(self, replicates, model: int = 4, seed: int = 0, pseudocount: float = 0.0, tol: float = 0.0001,
                  max_iters: int = 999) -> _boot.BootstrapResult:
        """Bootstrap replicates of the estimates (DESIGN.md section 7.2).  `replicates`: an int n (= range(n)) or a
        sequence of replicate indices (uint32).  Replicate r of `seed` resamples the M = sum(count) reads of the input
        with replacement on the device (a pure function of seed, r and the counts: a subset of indices run alone gives
        the same bits as in a larger call, on any packer or layout) and is then prepare(pseudocount) + run(model, tol,
        max_iters) on the resampled counts, with the lengths, groups and -G restriction of this factory; classes drawn 0
        times are absent, exactly as if the resampled reads had been compressed again.  Needs prepare() first.  The
        replicates run on their own device state: everything this factory reports afterwards is bit-identical to before.
        Refused (before any device work): row-sharded factories, weighted files, counts that are not non-negative
        integers or sum to more than 2^53, M = 0."""
        reps, counts = self._check_bootstrap(replicates, model, seed, max_iters)
        M, iters, theta_all, acc_all = self._replicate_loop(reps, counts, model, seed, pseudocount, tol, max_iters)
        return self._host_result(reps, model, seed, M, iters, theta_all, acc_all)

    def bootstrap_summary(self, replicates, model: int = 4, seed: int = 0, pseudocount: float = 0.0, tol: float = 0.0001,
                          max_iters: int = 999, interval: float = 0.95,
                          keep_replicates: bool = False) -> _boot.BootstrapSummary:
        """Mean, standard deviation and percentile interval of the bootstrap replicates (DESIGN.md section 7.3), reduced on
        the device: TPM, expected read counts and allelic shares at isoform and (with groups) gene level.  The replicates
        are those of `bootstrap()` with the same arguments; `interval` in (0, 1) gives the quantiles (1 - interval) / 2,
        0.5 and 1 - (1 - interval) / 2.  Nothing [B, H, T]-sized comes to the host unless `keep_replicates`, which also
        returns `.result`, the BootstrapResult of `bootstrap()` bit for bit.  Refused as `bootstrap()` refuses, and for
        fewer than 2 or more than `bootstrap.SUMMARY_MAX_REPLICATES` replicates or `interval` outside (0, 1)."""
        reps, counts = self._check_bootstrap(replicates, model, seed, max_iters)
        if not 0.0 < float(interval) < 1.0:
            raise ValueError("the bootstrap interval must be in (0, 1)")
        if not 2 <= reps.shape[0] <= _boot.SUMMARY_MAX_REPLICATES:
            raise ValueError(f"bootstrap summaries need 2 to {_boot.SUMMARY_MAX_REPLICATES} replicates")
        pat = self._pattern
        p = self.probability
        M, iters, theta_all, acc_all = self._replicate_loop(reps, counts, model, seed, pseudocount, tol, max_iters)
        genes = None
        if p.num_groups > 0:
            genes = (pat.dev["gene_ptr"], pat.dev["gene_loci"], int(p.num_groups))
        stats = _boot.summarize_on_device(pat.lib, pat.stream(), theta_all, acc_all, p.num_haplotypes, interval, genes)
        result = None
        if keep_replicates:
            result = self._host_result(reps, model, seed, M, iters, theta_all, acc_all)
        return _boot.BootstrapSummary(reps, int(seed), model, M, iters, float(interval), stats, lname=p.lname,
                                      hname=p.hname, gname=p.gname if p.num_groups > 0 else None, result=result)

    def _check_bootstrap(self, replicates, model, seed, max_iters):
        """The refusals of bootstrap() (before any device work) -> (replicate indices, int64 input class counts)."""
        if model not in (1, 2, 3, 4):
            raise RuntimeError("The read normalization model should be 1, 2, 3, or 4.")
        if max_iters > ERR_LOG_CAP:
            raise ValueError(f"max_iters above {ERR_LOG_CAP} is not supported")
        if self.world > 1 or self._presharded:
            raise NotImplementedError("bootstrap replicates of a row-sharded factory are not supported")
        if self._pattern is None or self._post is None:
            raise RuntimeError("bootstrap needs prepare() first")
        if self._weighted:
            raise NotImplementedError("bootstrap replicates of a weighted alignment file (stored values other than 1) "
                                      "are not supported")
        p = self.probability
        if model != 4 and p.num_groups == 0:
            raise _lib.GbrsError("Group information matrix is missing.")
        reps = _boot.replicate_indices(replicates)
        counts = _boot.read_counts_of(p.count, p.shape[2])
        if int(counts.sum()) == 0:
            raise ValueError("bootstrap needs at least one read (the counts sum to 0)")
        if not 0 <= int(seed) < 2 ** 64:
            raise ValueError("the bootstrap seed must fit 64 bits")
        return reps, counts

    def _replicate_loop(self, reps, counts, model, seed, pseudocount, tol, max_iters):
        """The replicates of checked arguments on the replicate state -> (M, iteration counts, theta_all, acc_all), the
        last two [B][T][8] device tensors."""
        T, H, N = self.probability.shape
        M = int(counts.sum())
        torch = _torch()
        pat = self._pattern
        pat.ensure_arrays(["class_id"])
        st = pat.replicate_state(model)
        B, n_cls = int(reps.shape[0]), int(pat.info["n_classes"])
        lib = pat.lib
        with torch.cuda.device(pat.device):
            prefix = torch.from_numpy(np.cumsum(counts)).to(pat.device)
            nbytes = C.c_int64()
            _lib.check(lib.gbrs_boot_scratch_bytes(N, C.byref(nbytes)))
            scratch = torch.empty(int(nbytes.value), dtype=torch.uint8, device=pat.device)
            _lib.check(lib.gbrs_boot_guide(C.c_void_p(prefix.data_ptr()), N, M, C.c_void_p(scratch.data_ptr()),
                                           int(nbytes.value), pat.stream()))
            theta_all = torch.empty((B, T, 8), dtype=torch.float64, device=pat.device)
            acc_all = torch.empty((B, T, 8), dtype=torch.float64, device=pat.device)
            iters = np.zeros(B, dtype=np.int64)
            errs = np.zeros(max(max_iters, 1), dtype=np.float64)
            class_id = C.c_void_p(pat.dev["class_id"].data_ptr()) if n_cls > 0 else None
            for b, r in enumerate(reps.tolist()):
                _lib.check(lib.gbrs_boot_resample(C.c_void_p(prefix.data_ptr()), N, M, int(seed), int(r), class_id, n_cls,
                                                  C.c_void_p(scratch.data_ptr()), int(nbytes.value),
                                                  C.c_void_p(st.count.data_ptr()), pat.stream()))
                _lib.check(lib.gbrs_em_prepare_local(C.byref(st.desc), pat.stream()))
                _lib.check(lib.gbrs_em_prepare_finish(C.byref(st.desc), float(pseudocount), pat.stream()))
                n = C.c_int32(0)
                _lib.check(lib.gbrs_em_run_cb(C.byref(st.desc), int(model), float(tol), int(max_iters),
                                              int(self._poll_every), pat.stream(), C.byref(n), errs.ctypes.data, None, None))
                iters[b] = n.value
                _lib.check(lib.gbrs_em_copy_theta(C.byref(st.desc), 0, C.c_void_p(theta_all[b].data_ptr()), pat.stream()))
                acc_all[b].copy_(st.acc)
        return M, iters, theta_all, acc_all

    def _host_result(self, reps, model, seed, M, iters, theta_all, acc_all) -> _boot.BootstrapResult:
        p = self.probability
        H = p.num_haplotypes
        with _torch().cuda.device(self._pattern.device):
            theta = theta_all[:, :, :H].permute(0, 2, 1).contiguous().cpu().numpy()
            acc = acc_all[:, :, :H].permute(0, 2, 1).contiguous().cpu().numpy()
        return _boot.BootstrapResult(reps, int(seed), model, M, iters, theta, acc, grp_conv_mat=self.grp_conv_mat,
                                     lname=p.lname, hname=p.hname, gname=p.gname if p.num_groups > 0 else None)

    # ---------------------------------------------------------------------------------------------------------------
    # reports
    # ---------------------------------------------------------------------------------------------------------------
    def expected_read_counts(self) -> np.ndarray:
        """H x T count-weighted posterior sums of the last E-step (`probability.sum(axis=READ)`, EMfactory.py:302)."""
        if self._counts_host is None:
            self._counts_host = self._ensure_pattern().acc_HT()
        return self._counts_host

    @staticmethod
    def _order(total, reorder, n):
        if reorder == "decreasing":
            return np.argsort(total.flatten())[::-1]
        if reorder == "increasing":
            return np.argsort(total.flatten())
        return np.arange(n)

    def _write_report(self, filename, lname, data, reorder, notes):
        total = data.sum(axis=0)
        order = self._order(total, reorder, len(lname))
        cntdata = np.vstack((data, total))
        with open(filename, "w") as fh:
            fh.write("locus\t" + "\t".join(self.probability.hname) + "\ttotal")
            if notes is not None:
                fh.write("\tnotes")
            fh.write("\n")
            utils.write_table_rows(fh, lname, cntdata, notes=notes, order=order)

    def report_read_counts(self, filename, grp_wise=False, reorder="as-is", notes=None):
        """Export read counts (EMfactory.py:289-331)."""
        counts = self.expected_read_counts()
        if grp_wise:
            lname = self.probability.gname
            counts = counts * self.grp_conv_mat
        else:
            lname = self.probability.lname
        self._write_report(filename, lname, np.asarray(counts), reorder, notes)

    def report_depths(self, filename, tpm=True, grp_wise=False, reorder="as-is", notes=None) -> None:
        """Exports expected depths (EMfactory.py:333-380).  As in the reference, the isoform-level TPM report scales
        `allelic_expression` in place (:352-354)."""
        if grp_wise:
            lname = self.probability.gname
            depths = np.asarray(self._theta() * self.grp_conv_mat)
        else:
            lname = self.probability.lname
            depths = self._theta()
        if tpm:
            depths *= 1000000.0 / depths.sum()
            if not grp_wise:
                self._theta_dirty = True
        self._write_report(filename, lname, depths, reorder, notes)

    def export_posterior_probability(self, filename: str, title: str = "Posterior Probability",
                                     incidence_only: bool = True) -> None:
        """Writes the pattern + counts, exactly what the reference's default `incidence_only=True` save emits
        (EMfactory.py:382-392, AlignmentPropertyMatrix.py:484).  `incidence_only=False`: the values of
        `posterior_probability()` as well (the reference's `probability.save(..., incidence_only=False)`)."""
        if incidence_only:
            self.probability.save(h5file=filename, title=title)
        else:
            self.posterior_probability().save(h5file=filename, title=title, incidence_only=False)

    # ---------------------------------------------------------------------------------------------------------------
    # posterior read-origin probabilities
    # ---------------------------------------------------------------------------------------------------------------
    def posterior_probability(self) -> APM:
        """The posterior read-origin probabilities the reference's `probability` holds after the last call
        (EMfactory.update_probability_at_read_level, EMfactory.py:146-212): a new AlignmentPropertyMatrix with the shape,
        names, counts and groups of `probability` and, per haplotype, a float64 CSC in canonical form holding
        P[n,t,h] on the EM's pattern (stored entries, minus the columns of a `locus_hapmask` restriction).
          after prepare() / reset():            the stored values normalised per class (1 / entries of the class for
                                                a pure incidence matrix; reset() sets the values to 1 first)
          after update_probability_at_read_level(model):  the E-step of `model` from the current theta
          after update_allelic_expression(model) / run(model, ...): the E-step of the theta that entered the last update
        Row-sharded runs: every rank computes its own classes and the values are summed over the group, so every rank
        returns the whole matrix (`shard="local"`: the posterior of the matrix this rank was given).  A class whose
        normaliser is 0 raises FloatingPointError, as the reference does.  `probability` itself is not changed."""
        from scipy.sparse import csc_matrix

        if self._post is None:
            raise RuntimeError("no posterior yet: call prepare() first")
        p = self.probability
        T, H, N = p.shape
        pattern = posterior_pattern(p, self._hapmask)
        if self._post[0] == "weighted":
            values = self._weighted_posterior(pattern, N)
        else:
            torch = _torch()
            pat = self._ensure_pattern()
            if self._post[0] == "incidence":
                model, theta_src = 4, torch.ones((T, 8), dtype=torch.float64, device=pat.device)
            else:
                model, theta_src = self._post[1], pat.post_theta
            reduce = None
            if self.world > 1 and not self._presharded:
                import torch.distributed as dist

                def reduce(t, op):
                    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM, group=self._group)

            values = pat.posterior(model, theta_src, [a[0] for a in pattern], [a[1] for a in pattern], reduce=reduce)
        out = APM()
        out.shape = p.shape
        out.num_loci, out.num_haplotypes, out.num_reads = p.shape
        out.finalized = True
        out.count = None if p.count is None else np.array(p.count, copy=True)
        out._copy_names(p)
        out._copy_group_info(p)
        out.data = [csc_matrix((values[h], np.array(pattern[h][1], copy=True), pattern[h][0]), shape=(N, T))
                    for h in range(H)]
        return out

    @staticmethod
    def _weighted_posterior(pattern, N):
        """prepare()'s posterior of a matrix with stored values: normalize_reads(READ) of the values (host, like the
        initial estimate computed from them)."""
        rows = np.zeros(N)
        for _, indices, data in pattern:
            rows += np.bincount(indices, weights=data, minlength=N)
        out = []
        for _, indices, data in pattern:
            den = rows[indices]
            if np.any(den == 0.0):
                raise FloatingPointError("a class whose stored values sum to 0 has no posterior (0 / 0)")
            out.append(np.asarray(data, dtype=np.float64) / den)
        return out
