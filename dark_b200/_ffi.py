"""ctypes binding of include/dark_bwt.h (the same symbols a Rust -sys crate would bind)."""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.environ.get("DARK_BWT_LIB") or os.path.join(_HERE, "lib", "libdark_bwt.so")  # DARK_BWT_LIB: tuning builds (tools/)
_lib = None

MAX_ROUNDS = 40

OK, E_INVALID_N, E_INVALID_ARG, E_CUDA, E_NOMEM, E_INTERNAL = range(6)
F_DEFAULT, F_NO_ALPHABET_PACKING, F_DEVICE_ONLY = 0, 1, 2

# every symbol include/dark_bwt.h declares (tests/test_abi.py checks the .so exports all of them)
SYMBOLS = [
    "dark_bwt_abi_version", "dark_bwt_create", "dark_bwt_create_ex", "dark_bwt_capacity", "dark_bwt_forward",
    "dark_bwt_forward_batch", "dark_bwt_forward_many", "dark_bwt_forward_many_device", "dark_bwt_forward_device", "dark_bwt_inverse", "dark_bwt_inverse_device",
    "dark_bwt_inverse_batch", "dark_bwt_inverse_many", "dark_bwt_inverse_many_device", "dark_bwt_reuse", "dark_bwt_destroy", "dark_bwt_strerror", "dark_bwt_last_error",
    "dark_bwt_stream", "dark_bwt_sort_pairs_device", "dark_bwt_verify_sa_device", "dark_bwt_emit_device", "dark_bwt_lcp_profile_device",
    "dark_bwt_synth", "dark_bwt_dc_encode_device", "dark_bwt_dc_encode", "dark_bwt_forward_dc",
]


class Stats(ctypes.Structure):
    """dark_bwt_stats"""
    _fields_ = [
        ("n", ctypes.c_uint64), ("sigma", ctypes.c_uint32), ("bits_per_symbol", ctypes.c_uint32),
        ("symbols_per_key", ctypes.c_uint32), ("initial_symbols", ctypes.c_uint32), ("pair_rounds", ctypes.c_uint32),
        ("rounds", ctypes.c_uint32), ("sort_passes", ctypes.c_uint32),
        ("kernel_launches", ctypes.c_uint32), ("active", ctypes.c_uint64 * MAX_ROUNDS),
        ("passes", ctypes.c_uint32 * MAX_ROUNDS), ("sorted_elements", ctypes.c_uint64),
        ("device_ms", ctypes.c_float), ("init_ms", ctypes.c_float), ("sort_ms", ctypes.c_float), ("pass_ms", ctypes.c_float),
        ("keybuild_ms", ctypes.c_float), ("rerank_ms", ctypes.c_float), ("emit_ms", ctypes.c_float),
        ("h2d_ms", ctypes.c_float), ("d2h_ms", ctypes.c_float),
        ("gen_passes", ctypes.c_uint32), ("gen_pass_ms", ctypes.c_float), ("gen_elements", ctypes.c_uint64),
        ("host_syncs", ctypes.c_uint32), ("reserved_", ctypes.c_uint32),
    ]

    def as_dict(self):
        r = int(self.rounds)
        d = {k: getattr(self, k) for k, _ in self._fields_ if k not in ("active", "passes")}
        d["active"] = [int(self.active[i]) for i in range(r + 1)]
        d["passes"] = [int(self.passes[i]) for i in range(r + 1)]
        return d


class DcInfo(ctypes.Structure):
    """dark_bwt_dc_info"""
    _fields_ = [("init", ctypes.c_uint64 * 256), ("mtf_symbols", ctypes.c_uint8 * 256), ("num_unique", ctypes.c_uint32),
                ("reserved_", ctypes.c_uint32), ("num_items", ctypes.c_uint64), ("device_ms", ctypes.c_float),
                ("reserved2_", ctypes.c_uint32)]


class DarkBwtError(RuntimeError):
    """Raised where the Rust wrapper would panic! (the reference's assert!/unwrap convention)."""

    def __init__(self, code, message):
        super().__init__(message)
        self.code = code


def lib_path():
    return _LIB


def build_native(verbose=False):
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc")], stdout=out)
    return _LIB


def lib():
    """Load libdark_bwt.so.  Fails loudly if it has not been built — there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB):
        raise DarkBwtError(E_CUDA, f"{_LIB} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                   f"or `make -C dark_b200/csrc` (the forward BWT has no CPU fallback)")
    L = ctypes.CDLL(_LIB)
    vp, u64, u32, i32 = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int
    pp = ctypes.POINTER(vp)
    L.dark_bwt_abi_version.restype = i32
    L.dark_bwt_create.argtypes = [u64, i32, pp]
    L.dark_bwt_create_ex.argtypes = [u64, i32, u32, pp]
    L.dark_bwt_capacity.argtypes = [vp]
    L.dark_bwt_capacity.restype = u64
    L.dark_bwt_forward.argtypes = [vp, vp, u64, vp, ctypes.POINTER(u64), vp, ctypes.POINTER(Stats)]
    L.dark_bwt_forward_batch.argtypes = [vp, vp, vp, vp, vp, vp, u64, vp]
    L.dark_bwt_forward_device.argtypes = [vp, vp, u64, vp, ctypes.POINTER(u64), vp, ctypes.POINTER(Stats)]
    L.dark_bwt_forward_many.argtypes = [vp, vp, vp, vp, vp, u64, ctypes.POINTER(Stats)]
    L.dark_bwt_forward_many_device.argtypes = [vp, vp, vp, u64, vp, vp, vp, ctypes.POINTER(Stats)]
    L.dark_bwt_inverse.argtypes = [vp, vp, u64, u64, vp]
    L.dark_bwt_inverse_device.argtypes = [vp, vp, u64, u64, vp, ctypes.POINTER(ctypes.c_float)]
    L.dark_bwt_inverse_batch.argtypes = [vp, vp, vp, vp, vp, u64, vp]
    L.dark_bwt_inverse_many.argtypes = [vp, vp, vp, vp, vp, u64, vp]
    L.dark_bwt_inverse_many_device.argtypes = [vp, vp, vp, vp, u64, vp, vp]
    L.dark_bwt_reuse.argtypes = [vp, pp, ctypes.POINTER(u64)]
    L.dark_bwt_destroy.argtypes = [vp]
    L.dark_bwt_destroy.restype = None
    L.dark_bwt_strerror.argtypes = [i32]
    L.dark_bwt_strerror.restype = ctypes.c_char_p
    L.dark_bwt_last_error.argtypes = [vp]
    L.dark_bwt_last_error.restype = ctypes.c_char_p
    L.dark_bwt_stream.argtypes = [vp]
    L.dark_bwt_stream.restype = vp
    L.dark_bwt_sort_pairs_device.argtypes = [vp, vp, vp, vp, vp, u64, i32, i32, ctypes.POINTER(i32),
                                             ctypes.POINTER(ctypes.c_float)]
    L.dark_bwt_verify_sa_device.argtypes = [vp, vp, u64, vp, ctypes.POINTER(u64)]
    L.dark_bwt_emit_device.argtypes = [vp, vp, u64, vp, vp, ctypes.POINTER(u64)]
    L.dark_bwt_lcp_profile_device.argtypes = [vp, vp, u64, vp, ctypes.POINTER(u64), ctypes.POINTER(u32), ctypes.POINTER(u64)]
    L.dark_bwt_synth.argtypes = [ctypes.c_char_p, u64, vp, u64]
    L.dark_bwt_dc_encode_device.argtypes = [vp, vp, u64, vp, vp, vp, vp, vp, ctypes.POINTER(DcInfo)]
    L.dark_bwt_dc_encode.argtypes = [vp, vp, u64, vp, vp, vp, vp, vp, ctypes.POINTER(DcInfo)]
    L.dark_bwt_forward_dc.argtypes = [vp, vp, u64, vp, ctypes.POINTER(u64), vp, vp, vp, vp, vp, ctypes.POINTER(DcInfo), ctypes.POINTER(Stats)]
    _lib = L
    return L


def check(rc, ctx=None, what="dark_bwt"):
    if rc == OK:
        return
    L = lib()
    msg = L.dark_bwt_strerror(rc).decode()
    if ctx:
        detail = L.dark_bwt_last_error(ctx).decode()
        if detail:
            msg += f" [{detail}]"
    raise DarkBwtError(rc, f"{what}: {msg}")
