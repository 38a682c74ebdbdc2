"""TEST INFRASTRUCTURE ONLY: ctypes front end of tests/dc_pack_ref.c, the sequential statement of the packed item stream
(include/dark_bwt.h) the GPU's stream is compared with.  The C file is compiled on first use into the temporary
directory (the tree may be read-only), keyed by its contents."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "dc_pack_ref.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        so = os.path.join(tempfile.gettempdir(), "dc_pack_ref_%d_%s.so" % (os.getuid(), hashlib.sha1(src).hexdigest()[:16]))
        if not os.path.exists(so):
            tmp = "%s.%d" % (so, os.getpid())
            subprocess.check_call(["gcc", "-O2", "-std=gnu11", "-Wall", "-shared", "-fPIC", "-o", tmp, _SRC])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        vp, u64 = ctypes.c_void_p, ctypes.c_uint64
        L.dc_pack_ref.argtypes = [vp, vp, vp, vp, u64, vp]
        L.dc_pack_ref.restype = u64
        L.dc_unpack_ref.argtypes = [vp, u64, vp, vp, vp, vp, u64]
        L.dc_unpack_ref.restype = u64
        _lib = L
    return _lib


def pack(pos, dist, sym, rank):
    """The packed stream of the item arrays (np.uint8)."""
    pos, dist = np.ascontiguousarray(pos, np.uint32), np.ascontiguousarray(dist, np.uint32)
    sym, rank = np.ascontiguousarray(sym, np.uint8), np.ascontiguousarray(rank, np.uint8)
    m = pos.size
    assert dist.size == m and sym.size == m and rank.size == m
    out = np.empty(12 * m, np.uint8)
    k = lib().dc_pack_ref(pos.ctypes.data, dist.ctypes.data, sym.ctypes.data, rank.ctypes.data, m, out.ctypes.data)
    return out[:k]


def unpack(stream, max_items=None):
    """(pos, dist, sym, rank) arrays of a packed stream; ValueError for a malformed one.  Every item takes 4 bytes or more,
    so len(stream) // 4 items is the default room."""
    s = np.ascontiguousarray(stream, np.uint8)
    cap = s.size // 4 if max_items is None else int(max_items)
    pos, dist = np.empty(cap, np.uint32), np.empty(cap, np.uint32)
    sym, rank = np.empty(cap, np.uint8), np.empty(cap, np.uint8)
    k = lib().dc_unpack_ref(s.ctypes.data, s.size, pos.ctypes.data, dist.ctypes.data, sym.ctypes.data, rank.ctypes.data, cap)
    if k == 2 ** 64 - 1:
        raise ValueError("malformed packed item stream")
    return pos[:k], dist[:k], sym[:k], rank[:k]
