"""ctypes binding of libgbrs_em.so (the C ABI in include/gbrs_em.h).

There is deliberately no fallback: if the shared library has not been built (`python -m gbrs_b200.csrc.build` or
`__graft_entry__.build()`), loading raises; if no CUDA device is present, the compute entry points return
GBRS_E_CUDA and `check()` raises `GbrsCudaError`.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GBRS_LIB_PATH") or os.path.join(HERE, "_C", "libgbrs_em.so")  # override: tuning builds

GBRS_HPAD = 8
GBRS_KMAX = 8
GBRS_PART_SLOTS = 4096
ABI_VERSION = 8
CTRL_ITERS, CTRL_DONE, CTRL_ERROR, CTRL_PARITY, CTRL_MAX_ITERS, CTRL_PREPARED = range(6)
SCAL_ERR, SCAL_SUM_PREV, SCAL_TARGET, SCAL_SUM_CUR = range(4)

BOOT_TPM, BOOT_COUNTS, BOOT_SHARE = range(3)  # gbrs_boot_derive quantities
BOOT_MAX_QUANTILES, BOOT_SUMMARY_MAX_B = 16, 16384

GBRS_OK, GBRS_E_ARG, GBRS_E_LIMIT, GBRS_E_CUDA, GBRS_E_NUMERIC, GBRS_E_NOMEM, GBRS_E_STATE = 0, -1, -2, -3, -4, -5, -6


class GbrsError(RuntimeError):
    pass


class GbrsCudaError(GbrsError):
    pass


class PackInput(C.Structure):
    _fields_ = [("T", C.c_int32), ("H", C.c_int32), ("N", C.c_int64),
                ("indptr", C.POINTER(C.c_void_p)), ("indices", C.POINTER(C.c_void_p)), ("index_bytes", C.c_int32),
                ("values", C.POINTER(C.c_void_p)), ("count", C.c_void_p), ("locus_hapmask", C.c_void_p),
                ("gene_of", C.c_void_p), ("shard_rank", C.c_int32), ("shard_count", C.c_int32),
                ("item_len", C.c_int32)]


class PackInfo(C.Structure):
    _fields_ = [("n_classes", C.c_int64), ("n_pairs", C.c_int64), ("n_runs", C.c_int64), ("n_items", C.c_int64),
                ("n_entries", C.c_int64), ("n_long_items", C.c_int64), ("nnz", C.c_int64), ("nnz_total", C.c_int64), ("n_classes_total", C.c_int64),
                ("entry_bytes", C.c_int32), ("n_gene_ids", C.c_int32), ("max_pairs_per_class", C.c_int32),
                ("n_deep_loci", C.c_int32), ("bucket_class0", C.c_int64 * (GBRS_KMAX + 2)),
                ("bucket_pair0", C.c_int64 * (GBRS_KMAX + 2))]


class DevicePack(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("rowptr", "pairs", "count", "runptr", "class_id", "ent_cls", "ent_pair", "ent_run",
                                          "item_desc", "locus_desc", "gene_of", "gene_ptr", "gene_loci")]


ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_int64, C.c_char_p, C.c_void_p)


class TilesParams(C.Structure):
    _fields_ = [("max_classes", C.c_int32), ("max_loci", C.c_int32), ("max_pairs", C.c_int32),
                ("max_entries", C.c_int32), ("max_items", C.c_int32), ("item_len", C.c_int32)]


class TilesInfo(C.Structure):
    _fields_ = [("n_tiles", C.c_int64), ("n_slots", C.c_int64), ("blob_bytes", C.c_int64), ("n_entries", C.c_int64),
                ("n_items", C.c_int64), ("n_pairs", C.c_int64), ("n_classes", C.c_int64),
                ("max_classes", C.c_int32), ("max_loci", C.c_int32), ("max_items", C.c_int32),
                ("max_part_a_bytes", C.c_int32), ("max_part_b_bytes", C.c_int32), ("max_planes", C.c_int32),
                ("max_slots_per_locus", C.c_int32), ("item_len", C.c_int32), ("n_deep_loci", C.c_int32),
                ("reserved", C.c_int32)]


# blob header words / tile descriptor words (include/gbrs_em.h)
(TH_CLASSES, TH_LOCI, TH_PLANES, TH_RUNS, TH_ITEMS, TH_SLICES, TH_A_BYTES, TH_FULL, TH_PAIRS, TH_ENTRIES, TH_B_BYTES,
 TH_SELL_WORDS) = range(12)
TH_WORDS = 12
TD_WORDS = 16
CTRL_TILE_NEXT = 13


class EmDev(C.Structure):
    _fields_ = [("T", C.c_int32), ("H", C.c_int32), ("n_gene_ids", C.c_int32), ("entry_bytes", C.c_int32),
                ("n_classes", C.c_int64), ("n_pairs", C.c_int64), ("n_runs", C.c_int64), ("n_items", C.c_int64),
                ("n_entries", C.c_int64), ("n_long_items", C.c_int64), ("n_ranks", C.c_int32), ("max_iters_cap", C.c_int32),
                ("bucket_class0", C.c_int64 * (GBRS_KMAX + 2)), ("bucket_pair0", C.c_int64 * (GBRS_KMAX + 2)),
                ("xchg_enabled", C.c_int32), ("xchg_rank", C.c_int32), ("xchg_peer", C.c_void_p * 8), ("xchg_mc", C.c_void_p),
                ("rowptr", C.c_void_p), ("pairs", C.c_void_p), ("count", C.c_void_p), ("runptr", C.c_void_p),
                ("ent_cls", C.c_void_p), ("ent_pair", C.c_void_p), ("ent_run", C.c_void_p),
                ("item_off", C.c_void_p), ("item_order", C.c_void_p), ("item_desc", C.c_void_p),
                ("locus_order", C.c_void_p), ("locus_desc", C.c_void_p), ("locus_item_ptr", C.c_void_p),
                ("gene_of", C.c_void_p), ("gene_ptr", C.c_void_p), ("gene_loci", C.c_void_p),
                ("tile_blob", C.c_void_p), ("tile_desc", C.c_void_p), ("tile_locus_desc", C.c_void_p),
                ("tile_partial", C.c_void_p), ("n_tiles", C.c_int64), ("n_tile_slots", C.c_int64),
                ("n_deep_loci", C.c_int32), ("xchg_timeout_ms", C.c_int32),
                ("tile_max_classes", C.c_int32), ("tile_max_loci", C.c_int32), ("tile_max_items", C.c_int32),
                ("tile_max_a_bytes", C.c_int32), ("tile_max_b_bytes", C.c_int32), ("tile_n_deep_loci", C.c_int32),
                ("theta", C.c_void_p), ("efflen", C.c_void_p), ("acc", C.c_void_p), ("iso", C.c_void_p),
                ("weights", C.c_void_p), ("subsets", C.c_void_p), ("wit", C.c_void_p), ("part", C.c_void_p), ("gene_hap", C.c_void_p),
                ("gamma", C.c_void_p), ("err_log", C.c_void_p), ("scal", C.c_void_p), ("ctrl", C.c_void_p),
                ("zero_count_absent", C.c_int32), ("reserved", C.c_int32)]


POLL_CB = C.CFUNCTYPE(None, C.c_int32, C.c_int32, C.POINTER(C.c_double), C.c_void_p)


class HmmChain(C.Structure):
    _fields_ = [("gene0", C.c_int64), ("tprob0", C.c_int64), ("n_genes", C.c_int32), ("n_steps", C.c_int32),
                ("state0", C.c_int64)]


# every symbol include/gbrs_em.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "gbrs_last_error": (C.c_char_p, []),
    "gbrs_abi_version": (C.c_int, []),
    "gbrs_pack_create": (C.c_int, [C.POINTER(PackInput), C.POINTER(C.c_void_p)]),
    "gbrs_pack_get_info": (C.c_int, [C.c_void_p, C.POINTER(PackInfo)]),
    "gbrs_pack_get_array": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "gbrs_pack_free": (C.c_int, [C.c_void_p]),
    "gbrs_pack_device": (C.c_int, [C.POINTER(PackInput), ALLOC_FN, C.c_void_p, C.c_void_p, C.POINTER(PackInfo),
                                   C.POINTER(DevicePack)]),
    "gbrs_tiles_create": (C.c_int, [C.c_void_p, C.POINTER(TilesParams), C.POINTER(C.c_void_p)]),
    "gbrs_tiles_get_info": (C.c_int, [C.c_void_p, C.POINTER(TilesInfo)]),
    "gbrs_tiles_get_array": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "gbrs_tiles_free": (C.c_int, [C.c_void_p]),
    "gbrs_em_prepare_local": (C.c_int, [C.POINTER(EmDev), C.c_void_p]),
    "gbrs_em_prepare_finish": (C.c_int, [C.POINTER(EmDev), C.c_double, C.c_void_p]),
    "gbrs_em_set_theta": (C.c_int, [C.POINTER(EmDev), C.c_void_p, C.c_void_p]),
    "gbrs_em_current_theta": (C.c_int, [C.POINTER(EmDev), C.c_void_p, C.POINTER(C.c_void_p)]),
    "gbrs_em_run_begin": (C.c_int, [C.POINTER(EmDev), C.c_double, C.c_int, C.c_void_p]),
    "gbrs_em_launch_local": (C.c_int, [C.POINTER(EmDev), C.c_int, C.c_void_p]),
    "gbrs_em_launch_estep": (C.c_int, [C.POINTER(EmDev), C.c_int, C.c_void_p]),
    "gbrs_em_launch_update": (C.c_int, [C.POINTER(EmDev), C.c_void_p]),
    "gbrs_prof_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "gbrs_em_launch_local_profiled": (C.c_int, [C.POINTER(EmDev), C.c_int, C.c_void_p, C.c_void_p]),
    "gbrs_prof_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                 C.POINTER(C.c_int32)]),
    "gbrs_prof_free": (C.c_int, [C.c_void_p]),
    "gbrs_em_run": (C.c_int, [C.POINTER(EmDev), C.c_int, C.c_double, C.c_int, C.c_int, C.c_void_p,
                              C.POINTER(C.c_int32), C.c_void_p]),
    "gbrs_em_run_cb": (C.c_int, [C.POINTER(EmDev), C.c_int, C.c_double, C.c_int, C.c_int, C.c_void_p,
                                 C.POINTER(C.c_int32), C.c_void_p, C.c_void_p, C.c_void_p]),
    "gbrs_em_read_ctrl": (C.c_int, [C.POINTER(EmDev), C.c_void_p, C.c_void_p, C.c_void_p]),
    "gbrs_em_posterior_scratch_bytes": (C.c_int, [C.POINTER(EmDev), C.c_int, C.c_int64, C.POINTER(C.c_int64)]),
    "gbrs_em_posterior": (C.c_int, [C.POINTER(EmDev), C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p),
                                    C.POINTER(C.c_void_p), C.c_int32, C.POINTER(C.c_void_p), C.c_void_p, C.c_int64,
                                    C.c_void_p]),
    "gbrs_em_copy_theta": (C.c_int, [C.POINTER(EmDev), C.c_int, C.c_void_p, C.c_void_p]),
    "gbrs_boot_scratch_bytes": (C.c_int, [C.c_int64, C.POINTER(C.c_int64)]),
    "gbrs_boot_guide": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    "gbrs_boot_resample": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_int64,
                                     C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "gbrs_boot_derive": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_int32, C.c_void_p, C.c_void_p]),
    "gbrs_boot_summarize": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "gbrs_write_table": (C.c_int, [C.c_char_p, C.c_char_p, C.POINTER(C.c_char_p), C.c_int64, C.c_void_p, C.c_int32,
                                   C.POINTER(C.c_char_p), C.c_void_p, C.c_int32]),
    "gbrs_parse_lengths": (C.c_int, [C.c_char_p, C.POINTER(C.c_char_p), C.c_int64, C.POINTER(C.c_char_p), C.c_int32,
                                     C.c_double, C.c_void_p, C.POINTER(C.c_int64)]),
    "gbrs_format_double": (C.c_int, [C.c_double, C.c_char_p, C.c_int32]),
    "gbrs_rows_create": (C.c_int, [C.POINTER(PackInput), C.POINTER(C.c_void_p)]),
    "gbrs_rows_get": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "gbrs_rows_free": (C.c_int, [C.c_void_p]),
    "gbrs_ec_workspace_bytes": (C.c_int, [C.c_int64, C.POINTER(C.c_int64)]),
    "gbrs_ec_build": (C.c_int, [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(C.c_int64),
                                C.POINTER(C.c_int64)]),
    "gbrs_em_alignment_counts": (C.c_int, [C.POINTER(EmDev), C.c_int, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p]),
    "gbrs_hmm_emission": (C.c_int, [C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double,
                                    C.c_double, C.c_void_p, C.c_void_p]),
    "gbrs_hmm_run": (C.c_int, [C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built -- there is no CPU fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GbrsError(f"{LIB_PATH} is missing: build it with `python -m gbrs_b200.csrc.build` "
                            "(the multiway EM has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if lib.gbrs_abi_version() != ABI_VERSION:
            raise GbrsError("libgbrs_em.so ABI version mismatch; rebuild")
        _lib = lib
    return _lib


def last_error() -> str:
    return (load().gbrs_last_error() or b"").decode()


def check(rc: int) -> None:
    if rc == GBRS_OK:
        return
    msg = last_error()
    if rc == GBRS_E_CUDA:
        raise GbrsCudaError(msg)
    if rc == GBRS_E_NUMERIC:
        raise FloatingPointError(msg)  # reference: np.seterr(all='raise') in EMfactory.run
    if rc == GBRS_E_LIMIT:
        raise NotImplementedError(msg)
    if rc == GBRS_E_NOMEM:
        raise MemoryError(msg)
    raise GbrsError(msg)
