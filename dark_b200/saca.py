"""Host-side mirror of the reference's `saca` module (src/saca.rs) over the C ABI.

Same names, argument meaning and error behaviour as the Rust original so that the parity
tests read like the reference's own (`saca::test::some_detail`, src/saca.rs:393-407):

    Symbol = u8, Suffix = u32, SUF_INVALID = !0          src/saca.rs:18-22
    Constructor::new(max_n)                               src/saca.rs:351-360
    Constructor::capacity()                               src/saca.rs:363-365
    Constructor::compute(input) -> &[Suffix]              src/saca.rs:368-378   (asserts len == capacity)
    Constructor::reuse() -> &mut [Suffix]                 src/saca.rs:381-383
plus the fused entry the two call sites use instead of compute + TransformIterator
(src/block/dc.rs:45-50, src/block/raw.rs:39-44):
    Constructor::bwt(input) -> (Vec<u8>, usize)

Errors raise DarkBwtError where the Rust code panics (wrong length: saca.rs:369; n < 2:
saca.rs:69/300).
"""
import ctypes

import numpy as np

from . import _ffi

Symbol = np.uint8
Suffix = np.uint32
SUF_INVALID = 0xFFFFFFFF


def _as_u8(buf):
    if isinstance(buf, np.ndarray):
        return np.ascontiguousarray(buf, dtype=np.uint8)
    return np.frombuffer(bytes(buf) if not isinstance(buf, (bytes, bytearray, memoryview)) else buf, dtype=np.uint8)


class Constructor:
    """Suffix Array Constructor (GPU).  Not thread-safe, like `&mut self` in the reference."""

    def __init__(self, max_n, device=0, flags=_ffi.F_DEFAULT):
        self._L = _ffi.lib()
        self._ctx = ctypes.c_void_p()
        _ffi.check(self._L.dark_bwt_create_ex(int(max_n), int(device), int(flags), ctypes.byref(self._ctx)),
                   None, "Constructor::new")
        self.n = int(max_n)
        self.device = int(device)
        self.stats = _ffi.Stats()

    # -- reference API --------------------------------------------------------------------
    def capacity(self):
        return int(self._L.dark_bwt_capacity(self._ctx))

    def compute(self, input):
        """Suffix array of `input` (np.uint32[n]).  `len(input)` must equal capacity (saca.rs:369)."""
        t = _as_u8(input)
        if t.size != self.n:
            raise _ffi.DarkBwtError(_ffi.E_INVALID_N, f"assertion failed: input.len() == self.n ({t.size} != {self.n})")
        _, _, sa = self._forward(t, want_sa=True)
        return sa

    def reuse(self):
        """The context's host scratch as np.uint32 (>= capacity words; n + extra like saca.rs:353-357)."""
        p, cnt = ctypes.c_void_p(), ctypes.c_uint64()
        _ffi.check(self._L.dark_bwt_reuse(self._ctx, ctypes.byref(p), ctypes.byref(cnt)), self._ctx, "reuse")
        buf = (ctypes.c_uint32 * cnt.value).from_address(p.value)
        return np.frombuffer(buf, dtype=np.uint32)

    # -- the fused call-site entry -----------------------------------------------------------
    def bwt(self, input):
        """(BWT bytes np.uint8[n], origin) of a block of up to `capacity` bytes."""
        out, origin, _ = self._forward(_as_u8(input), want_sa=False)
        return out, origin

    def bwt_and_sa(self, input):
        return self._forward(_as_u8(input), want_sa=True)

    def _forward(self, t, want_sa):
        out = np.empty(t.size, dtype=np.uint8)
        sa = np.empty(t.size, dtype=np.uint32) if want_sa else None
        origin = ctypes.c_uint64(0)
        rc = self._L.dark_bwt_forward(self._ctx, t.ctypes.data if t.size else None, t.size, out.ctypes.data if t.size else None,
                                      ctypes.byref(origin), sa.ctypes.data if (want_sa and t.size) else None,
                                      ctypes.byref(self.stats))
        if rc == _ffi.E_INVALID_ARG and t.size == 0:
            rc = _ffi.E_INVALID_N
        _ffi.check(rc, self._ctx, "Constructor::bwt")
        return out, int(origin.value), sa

    def bwt_into(self, text_ptr, n, bwt_ptr, sa_ptr=None):
        """Host-buffer entry on raw addresses (e.g. pinned buffers): returns origin."""
        origin = ctypes.c_uint64(0)
        _ffi.check(self._L.dark_bwt_forward(self._ctx, text_ptr, int(n), bwt_ptr, ctypes.byref(origin), sa_ptr,
                                            ctypes.byref(self.stats)), self._ctx, "Constructor::bwt")
        return int(origin.value)

    def bwt_batch_into(self, text_ptrs, ns, bwt_ptrs, want_stats=False):
        """Pipelined host entry over several blocks (raw host addresses, ideally pinned):
        copy-in of block k+1 and copy-out of block k-1 overlap the transform of block k.
        Returns the list of origins (and the per-block stats if asked)."""
        cnt = len(ns)
        assert len(text_ptrs) == cnt and len(bwt_ptrs) == cnt
        T = (ctypes.c_void_p * cnt)(*text_ptrs)
        B = (ctypes.c_void_p * cnt)(*bwt_ptrs)
        N = (ctypes.c_uint64 * cnt)(*[int(x) for x in ns])
        O = (ctypes.c_uint64 * cnt)()
        S = (_ffi.Stats * cnt)() if want_stats else None
        _ffi.check(self._L.dark_bwt_forward_batch(self._ctx, T, N, B, O, None, cnt, S), self._ctx, "Constructor::bwt_batch")
        origins = [int(O[i]) for i in range(cnt)]
        return (origins, [S[i].as_dict() for i in range(cnt)]) if want_stats else origins

    def bwt_blocks(self, blocks):
        """[(bwt, origin), ...] for an iterable of host blocks, through the pipelined batch entry."""
        ts = [_as_u8(b) for b in blocks]
        outs = [np.empty(t.size, dtype=np.uint8) for t in ts]
        origins = self.bwt_batch_into([t.ctypes.data for t in ts], [t.size for t in ts], [o.ctypes.data for o in outs])
        return list(zip(outs, origins))

    def bwt_many_into(self, text_ptrs, ns, bwt_ptrs):
        """Many small host blocks in ONE device sort (dark_bwt_forward_many): raw host addresses; returns the origins.
        The blocks share the context's arena: sum(ns) <= capacity."""
        cnt = len(ns)
        assert len(text_ptrs) == cnt and len(bwt_ptrs) == cnt
        T = (ctypes.c_void_p * cnt)(*text_ptrs)
        B = (ctypes.c_void_p * cnt)(*bwt_ptrs)
        N = (ctypes.c_uint64 * cnt)(*[int(x) for x in ns])
        O = (ctypes.c_uint64 * cnt)()
        _ffi.check(self._L.dark_bwt_forward_many(self._ctx, T, N, B, O, cnt, ctypes.byref(self.stats)), self._ctx,
                   "Constructor::bwt_many")
        return [int(O[i]) for i in range(cnt)]

    def bwt_many(self, blocks):
        """[(bwt, origin), ...] for a list of small host blocks, sorted together in one pass over the GPU."""
        ts = [_as_u8(b) for b in blocks]
        outs = [np.empty(t.size, dtype=np.uint8) for t in ts]
        origins = self.bwt_many_into([t.ctypes.data for t in ts], [t.size for t in ts], [o.ctypes.data for o in outs])
        return list(zip(outs, origins))

    def bwt_many_device(self, d_text, d_starts, count, d_bwt, d_origins, d_sa=None):
        """Device-resident form: blocks back to back in d_text, offsets d_starts[0..count] (u32, on the device)."""
        _ffi.check(self._L.dark_bwt_forward_many_device(self._ctx, d_text, d_starts, int(count), d_bwt, d_origins, d_sa,
                                                        ctypes.byref(self.stats)), self._ctx, "Constructor::bwt_many_device")

    # -- the unpack side: compress::bwt::decode(&input, origin, &mut suffixes)  (block/dc.rs:154-156) ---------
    def inverse(self, bwt, origin):
        """Original block (np.uint8[n]) from its BWT bytes and origin index."""
        b = _as_u8(bwt)
        out = np.empty(b.size, dtype=np.uint8)
        _ffi.check(self._L.dark_bwt_inverse(self._ctx, b.ctypes.data if b.size else None, b.size, int(origin),
                                            out.ctypes.data if b.size else None), self._ctx, "bwt::decode")
        return out

    def inverse_device(self, d_bwt, n, origin, d_text):
        ms = ctypes.c_float(0)
        _ffi.check(self._L.dark_bwt_inverse_device(self._ctx, d_bwt, int(n), int(origin), d_text, ctypes.byref(ms)), self._ctx,
                   "bwt::decode")
        return float(ms.value)

    def inverse_many_into(self, bwt_ptrs, ns, origins, text_ptrs):
        """Many small host blocks inverted in ONE device pass (dark_bwt_inverse_many): raw host addresses; returns the
        device ms of the pass.  The blocks share the context's arena: sum(ns) + len(ns) <= capacity."""
        cnt = len(ns)
        assert len(bwt_ptrs) == cnt and len(origins) == cnt and len(text_ptrs) == cnt
        B = (ctypes.c_void_p * cnt)(*bwt_ptrs)
        T = (ctypes.c_void_p * cnt)(*text_ptrs)
        N = (ctypes.c_uint64 * cnt)(*[int(x) for x in ns])
        O = (ctypes.c_uint64 * cnt)(*[int(x) for x in origins])
        ms = ctypes.c_float(0)
        _ffi.check(self._L.dark_bwt_inverse_many(self._ctx, B, N, O, T, cnt, ctypes.byref(ms)), self._ctx, "bwt::decode (many)")
        return float(ms.value)

    def inverse_many(self, pairs):
        """[text, ...] for a list of (bwt, origin) pairs of small blocks, inverted together in one pass over the GPU."""
        bs = [_as_u8(b) for b, _ in pairs]
        outs = [np.empty(b.size, dtype=np.uint8) for b in bs]
        self.inverse_many_into([b.ctypes.data for b in bs], [b.size for b in bs], [int(o) for _, o in pairs],
                               [o.ctypes.data for o in outs])
        return outs

    def inverse_many_device(self, d_bwt, d_starts, d_origins, count, d_text):
        """Device-resident form, the layout bwt_many_device writes: blocks back to back in d_bwt, offsets d_starts[0..count]
        (u32) and origins d_origins[0..count) (u64), all on the device.  Returns the device ms of the pass."""
        ms = ctypes.c_float(0)
        _ffi.check(self._L.dark_bwt_inverse_many_device(self._ctx, d_bwt, d_starts, d_origins, int(count), d_text, ctypes.byref(ms)),
                   self._ctx, "bwt::decode (many)")
        return float(ms.value)

    def inverse_batch_into(self, bwt_ptrs, ns, origins, text_ptrs):
        """Pipelined host entry over several blocks (dark_bwt_inverse_batch; raw host addresses, ideally pinned): copy-in
        of block k+1 and copy-out of block k-1 overlap the inverse of block k.  Returns the per-block device ms."""
        cnt = len(ns)
        assert len(bwt_ptrs) == cnt and len(origins) == cnt and len(text_ptrs) == cnt
        B = (ctypes.c_void_p * cnt)(*bwt_ptrs)
        T = (ctypes.c_void_p * cnt)(*text_ptrs)
        N = (ctypes.c_uint64 * cnt)(*[int(x) for x in ns])
        O = (ctypes.c_uint64 * cnt)(*[int(x) for x in origins])
        ms = (ctypes.c_float * max(cnt, 1))()
        _ffi.check(self._L.dark_bwt_inverse_batch(self._ctx, B, N, O, T, cnt, ms), self._ctx, "bwt::decode (batch)")
        return [float(ms[i]) for i in range(cnt)]

    def inverse_blocks(self, pairs):
        """[text, ...] for an iterable of (bwt, origin) host blocks, through the pipelined batch entry."""
        pairs = list(pairs)
        bs = [_as_u8(b) for b, _ in pairs]
        outs = [np.empty(b.size, dtype=np.uint8) for b in bs]
        self.inverse_batch_into([b.ctypes.data for b in bs], [b.size for b in bs], [int(o) for _, o in pairs],
                                [o.ctypes.data for o in outs])
        return outs

    # -- distance coding + MTF: bwt::dc::encode(&output, suf, &mut mtf) and its item stream (block/dc.rs:52, 82-85) ---------
    def _dc_result(self, info, n, dist, pos, idist, sym, rank):
        k = int(info.num_items)
        return {"dist": dist, "init": np.array(list(info.init), dtype=np.uint64), "mtf_symbols": np.array(list(info.mtf_symbols), dtype=np.uint8),
                "num_unique": int(info.num_unique), "num_items": k, "item_pos": pos[:k], "item_dist": idist[:k], "item_sym": sym[:k],
                "item_rank": rank[:k], "device_ms": float(info.device_ms)}

    def dc_encode(self, bwt, want_dist=True):
        """Distance coding of a BWT block (host buffers): dict(dist u32[n] with filler n, init[256], mtf_symbols, num_unique,
        and the (distance, Context) items: item_pos/item_dist/item_sym/item_rank)."""
        b = _as_u8(bwt)
        n = b.size
        dist = np.empty(n, dtype=np.uint32) if want_dist else None
        pos, idist = np.empty(n, dtype=np.uint32), np.empty(n, dtype=np.uint32)
        sym, rank = np.empty(n, dtype=np.uint8), np.empty(n, dtype=np.uint8)
        info = _ffi.DcInfo()
        _ffi.check(self._L.dark_bwt_dc_encode(self._ctx, b.ctypes.data, n, dist.ctypes.data if want_dist else None, pos.ctypes.data,
                                              idist.ctypes.data, sym.ctypes.data, rank.ctypes.data, ctypes.byref(info)), self._ctx, "dc::encode")
        return self._dc_result(info, n, dist, pos, idist, sym, rank)

    def bwt_dc(self, input, want_dist=True):
        """block/dc.rs:45-52 in one call: (bwt, origin, dc dict) — the DC stage reads the BWT while it is still in HBM."""
        t = _as_u8(input)
        n = t.size
        out = np.empty(n, dtype=np.uint8)
        dist = np.empty(n, dtype=np.uint32) if want_dist else None
        pos, idist = np.empty(n, dtype=np.uint32), np.empty(n, dtype=np.uint32)
        sym, rank = np.empty(n, dtype=np.uint8), np.empty(n, dtype=np.uint8)
        info, origin = _ffi.DcInfo(), ctypes.c_uint64(0)
        _ffi.check(self._L.dark_bwt_forward_dc(self._ctx, t.ctypes.data, n, out.ctypes.data, ctypes.byref(origin),
                                               dist.ctypes.data if want_dist else None, pos.ctypes.data, idist.ctypes.data, sym.ctypes.data,
                                               rank.ctypes.data, ctypes.byref(info), ctypes.byref(self.stats)), self._ctx, "bwt + dc::encode")
        return out, int(origin.value), self._dc_result(info, n, dist, pos, idist, sym, rank)

    def dc_encode_device(self, d_bwt, n, d_dist=None, d_item_pos=None, d_item_dist=None, d_item_sym=None, d_item_rank=None):
        """Device pointers in, device pointers out (all outputs optional); returns the DcInfo header."""
        info = _ffi.DcInfo()
        _ffi.check(self._L.dark_bwt_dc_encode_device(self._ctx, d_bwt, int(n), d_dist, d_item_pos, d_item_dist, d_item_sym, d_item_rank,
                                                     ctypes.byref(info)), self._ctx, "dc::encode")
        return info

    # -- device-resident form (benches, pipelines that keep the block in HBM) ------------------
    def bwt_device(self, d_text, n, d_bwt, d_sa=None):
        """Raw device pointers (ints).  Returns origin; self.stats holds the device timings."""
        origin = ctypes.c_uint64(0)
        _ffi.check(self._L.dark_bwt_forward_device(self._ctx, d_text, int(n), d_bwt, ctypes.byref(origin), d_sa,
                                                   ctypes.byref(self.stats)), self._ctx, "Constructor::bwt_device")
        return int(origin.value)

    def verify_sa_device(self, d_text, n, d_sa):
        bad = ctypes.c_uint64(0)
        _ffi.check(self._L.dark_bwt_verify_sa_device(self._ctx, d_text, int(n), d_sa, ctypes.byref(bad)), self._ctx,
                   "verify_sa")
        return int(bad.value)

    def lcp_profile_device(self, d_text, n, d_sa):
        """SURVEY §8(d) profile on the GPU: dict(R, m[r], sum_m, max_lcp, b, P, b_alg)."""
        m = (ctypes.c_uint64 * 64)()
        rounds, mx = ctypes.c_uint32(0), ctypes.c_uint64(0)
        _ffi.check(self._L.dark_bwt_lcp_profile_device(self._ctx, d_text, int(n), d_sa, m, ctypes.byref(rounds), ctypes.byref(mx)),
                   self._ctx, "lcp_profile")
        R = int(rounds.value)
        ms = [int(m[i]) for i in range(R)]
        b = int(n).bit_length()                      # ceil(log2(n+1))
        P = (2 * b + 7) // 8
        return {"R": R, "m": ms, "sum_m": sum(ms), "max_lcp": int(mx.value), "b": b, "P": P,
                "b_alg": 243.0 * n + (48.0 + 24.0 * P) * sum(ms)}

    def emit_device(self, d_text, n, d_sa, d_bwt):
        origin = ctypes.c_uint64(0)
        _ffi.check(self._L.dark_bwt_emit_device(self._ctx, d_text, int(n), d_sa, d_bwt, ctypes.byref(origin)), self._ctx,
                   "emit")
        return int(origin.value)

    def sort_pairs_device(self, d_keys, d_vals, d_keys_alt, d_vals_alt, count, begin_bit=0, end_bit=64):
        in_alt, ms = ctypes.c_int(0), ctypes.c_float(0)
        _ffi.check(self._L.dark_bwt_sort_pairs_device(self._ctx, d_keys, d_vals, d_keys_alt, d_vals_alt, int(count),
                                                      begin_bit, end_bit, ctypes.byref(in_alt), ctypes.byref(ms)),
                   self._ctx, "sort_pairs")
        return bool(in_alt.value), float(ms.value)

    @property
    def stream(self):
        return self._L.dark_bwt_stream(self._ctx)

    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._L.dark_bwt_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def decode(bwt, origin, device=0):
    """`compress::bwt::decode(&input, origin, &mut suffixes)` collected: the original bytes."""
    b = _as_u8(bwt)
    with Constructor(max(b.size, 2), device=device) as con:
        return con.inverse(b, origin)


def transform(input, suf):
    """`compress::bwt::TransformIterator::new(input, suf)` collected: (bytes, origin).

    Host-side numpy statement of the emission rule, kept for callers that already hold a
    suffix array (the reference's tests do this, saca.rs:398-400).  The hot path uses
    Constructor.bwt, which never materialises the SA on the host."""
    t = _as_u8(input)
    s = np.asarray(suf, dtype=np.uint32)
    n = t.size
    idx = (s.astype(np.int64) + n - 1) % n
    origin = int(np.flatnonzero(s == 0)[0])
    return t[idx], origin
