"""TEST INFRASTRUCTURE ONLY -- the posterior entry points of the EM library (gbrs_em_posterior, gbrs_em_copy_theta) on the
emulated library of tests/simt_em.py: `PosteriorHostPattern` is tests/simt_em.HostPattern with the calls of
gbrs_b200.emfactory.DevicePattern.copy_theta / .posterior, and `emulated_device_class_id` returns the `class_id` array of
the device packer run through the host shim."""
from __future__ import annotations

import ctypes as C

import numpy as np

from gbrs_b200 import _lib
from tests import simt_em

SYMBOLS = ("gbrs_em_posterior_scratch_bytes", "gbrs_em_posterior", "gbrs_em_copy_theta")


def bind(lib):
    """argument types of the posterior symbols on an emulated library (simt_em.load binds the EM update's only)"""
    for name in SYMBOLS:
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = _lib.SYMBOLS[name]
    return lib


class PosteriorHostPattern(simt_em.HostPattern):
    def __init__(self, apm, **kw):
        super().__init__(apm, **kw)
        bind(self.lib)

    def copy_theta(self, previous):
        """gbrs_em_copy_theta into a new [T][8] array: the current theta, or (`previous`) the other ping-pong half."""
        out = np.zeros((self.T, 8))
        self.check(self.lib.gbrs_em_copy_theta(C.byref(self.desc), int(previous), out.ctypes.data, None))
        return out

    def posterior(self, model, theta_src, indptr, indices):
        """DevicePattern.posterior: gbrs_em_posterior from `theta_src` ([T][8]) on the output pattern indptr[h] /
        indices[h] -> list of H value arrays.  The EM's own buffers are not touched."""
        N = int(self.packed.N)
        nbytes = C.c_int64()
        self.check(self.lib.gbrs_em_posterior_scratch_bytes(C.byref(self.desc), int(model), N, C.byref(nbytes)))
        scratch = np.zeros(int(nbytes.value) + 256, np.uint8)
        base = (-scratch.ctypes.data) % 256  # 256-byte aligned, as device allocations are
        wide = any(np.asarray(a).dtype.itemsize == 8 for a in indices)
        ip = [np.ascontiguousarray(a, dtype=np.int64) for a in indptr]
        ix = [np.ascontiguousarray(a, dtype=np.int64 if wide else np.int32) for a in indices]
        ix = [a if a.size else np.zeros(1, a.dtype) for a in ix]
        vals = [np.full(max(int(np.asarray(a).shape[0]), 1), np.nan) for a in indices]
        th = np.ascontiguousarray(theta_src, dtype=np.float64)
        P = C.c_void_p * self.H
        self.check(self.lib.gbrs_em_posterior(
            C.byref(self.desc), int(model), th.ctypes.data, self.arr["class_id"].ctypes.data, N,
            P(*[a.ctypes.data for a in ip]), P(*[a.ctypes.data for a in ix]), 8 if wide else 4,
            P(*[v.ctypes.data for v in vals]), scratch.ctypes.data + base, int(nbytes.value), None))
        return [v[: np.asarray(a).shape[0]].copy() for v, a in zip(vals, indices)]


def emulated_device_class_id(apm, gene_of=None, hapmask=None, shard_rank=0, shard_count=1):
    """`class_id` of gbrs_pack_device run through the host shim ("device" memory = host memory from a numpy allocator)"""
    from gbrs_b200.emfactory import pack_input

    lib = C.CDLL(simt_em.build_gpack())
    lib.gbrs_pack_device.restype, lib.gbrs_pack_device.argtypes = _lib.SYMBOLS["gbrs_pack_device"]
    lib.gbrs_last_error.restype = C.c_char_p
    inp, keep = pack_input(apm, gene_of=gene_of, hapmask=hapmask, shard_rank=shard_rank, shard_count=shard_count)
    bufs = {}

    def alloc(nbytes, tag, _user):
        a = np.zeros(max(int(nbytes), 1) + 64, dtype=np.uint8)
        bufs.setdefault(tag.decode(), []).append((a, int(nbytes)))
        return a.ctypes.data

    cb = _lib.ALLOC_FN(alloc)
    info, out = _lib.PackInfo(), _lib.DevicePack()
    rc = lib.gbrs_pack_device(C.byref(inp), cb, None, None, C.byref(info), C.byref(out))
    assert rc == 0, (rc, lib.gbrs_last_error())
    del keep
    a, nbytes = bufs["class_id"][-1]
    assert out.class_id == a.ctypes.data
    return a[:nbytes].view(np.uint32).copy()
