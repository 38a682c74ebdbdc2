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

    def bwt_dc_batch_into(self, text_ptrs, ns, bwt_ptrs=None, dist_ptrs=None, pos_ptrs=None, idist_ptrs=None, sym_ptrs=None,
                          rank_ptrs=None, want_stats=False):
        """Pipelined block/dc.rs:45-52 over several blocks (dark_bwt_forward_dc_batch; raw host addresses, ideally pinned; needs
        a Constructor made with flags including _ffi.F_DC_BATCH): copy-in of block k+1 and copy-out of block k-1 overlap the
        forward + DC of block k.  Each output list is optional, and so is each entry (None).  The item arrays need room for n
        entries.  Returns (origins, DcInfo records) and the per-block stats if asked."""
        cnt = len(ns)
        assert len(text_ptrs) == cnt

        def arr(ptrs):
            if ptrs is None:
                return None
            assert len(ptrs) == cnt
            return (ctypes.c_void_p * max(cnt, 1))(*ptrs)
        O = (ctypes.c_uint64 * max(cnt, 1))()
        infos = (_ffi.DcInfo * max(cnt, 1))()
        S = (_ffi.Stats * max(cnt, 1))() if want_stats else None
        _ffi.check(self._L.dark_bwt_forward_dc_batch(self._ctx, arr(text_ptrs), (ctypes.c_uint64 * max(cnt, 1))(*[int(x) for x in ns]), cnt,
                                                     arr(bwt_ptrs), O, arr(dist_ptrs), arr(pos_ptrs), arr(idist_ptrs), arr(sym_ptrs),
                                                     arr(rank_ptrs), infos, S), self._ctx, "bwt + dc::encode (batch)")
        res = ([int(O[i]) for i in range(cnt)], [infos[i] for i in range(cnt)])
        return res + ([S[i].as_dict() for i in range(cnt)],) if want_stats else res

    def bwt_dc_blocks(self, texts, want_dist=True, want_bwt=True):
        """block/dc.rs:45-52 for a run of host blocks through the pipelined batch entry: [(bwt or None, origin, dc dict), ...],
        each what bwt_dc gives on that block alone."""
        ts = [_as_u8(t) for t in texts]
        ns = [t.size for t in ts]
        bwts = [np.empty(n, dtype=np.uint8) for n in ns] if want_bwt else None
        dists = [np.empty(n, dtype=np.uint32) for n in ns] if want_dist else None
        pos, idist = [np.empty(n, dtype=np.uint32) for n in ns], [np.empty(n, dtype=np.uint32) for n in ns]
        sym, rank = [np.empty(n, dtype=np.uint8) for n in ns], [np.empty(n, dtype=np.uint8) for n in ns]
        ptrs = lambda arrays: [a.ctypes.data for a in arrays] if arrays is not None else None  # noqa: E731
        origins, infos = self.bwt_dc_batch_into(ptrs(ts), ns, ptrs(bwts), ptrs(dists), ptrs(pos), ptrs(idist), ptrs(sym), ptrs(rank))
        return [(bwts[k] if want_bwt else None, origins[k],
                 self._dc_result(infos[k], ns[k], dists[k] if want_dist else None, pos[k], idist[k], sym[k], rank[k]))
                for k in range(len(ts))]

    def dc_encode_device(self, d_bwt, n, d_dist=None, d_item_pos=None, d_item_dist=None, d_item_sym=None, d_item_rank=None):
        """Device pointers in, device pointers out (all outputs optional); returns the DcInfo header."""
        info = _ffi.DcInfo()
        _ffi.check(self._L.dark_bwt_dc_encode_device(self._ctx, d_bwt, int(n), d_dist, d_item_pos, d_item_dist, d_item_sym, d_item_rank,
                                                     ctypes.byref(info)), self._ctx, "dc::encode")
        return info

    # -- the packed item stream (include/dark_bwt.h): sym, rank, varint(run length - 1), varint(dist) per item ----------
    def bwt_dc_packed(self, input, want_bwt=False):
        """block/dc.rs:45-52 with the items packed on the GPU (dark_bwt_forward_dc_packed): (bwt or None, origin,
        stream np.uint8 of its exact length, DcInfo)."""
        t = _as_u8(input)
        n = t.size
        out = np.empty(n, dtype=np.uint8) if want_bwt else None
        stream = np.empty(_ffi.dc_packed_max(n), dtype=np.uint8)
        info, origin, nbytes = _ffi.DcInfo(), ctypes.c_uint64(0), ctypes.c_uint64(0)
        _ffi.check(self._L.dark_bwt_forward_dc_packed(self._ctx, t.ctypes.data, n, out.ctypes.data if want_bwt else None,
                                                      ctypes.byref(origin), stream.ctypes.data, stream.size, ctypes.byref(nbytes),
                                                      ctypes.byref(info), ctypes.byref(self.stats)), self._ctx, "bwt + dc::encode (packed)")
        return out, int(origin.value), stream[:nbytes.value], info

    def bwt_dc_packed_batch_into(self, text_ptrs, ns, stream_ptrs, capacities, bwt_ptrs=None, want_stats=False):
        """Pipelined dark_bwt_forward_dc_packed over several blocks (dark_bwt_forward_dc_packed_batch; raw host addresses,
        ideally pinned; needs a Constructor made with flags including _ffi.F_DC_BATCH).  Returns (origins, stream sizes,
        DcInfo records) and the per-block stats if asked."""
        cnt = len(ns)
        assert len(text_ptrs) == cnt and len(stream_ptrs) == cnt and len(capacities) == cnt
        m = max(cnt, 1)
        arr = lambda ptrs: (ctypes.c_void_p * m)(*ptrs) if ptrs is not None else None  # noqa: E731
        O, B = (ctypes.c_uint64 * m)(), (ctypes.c_uint64 * m)()
        infos = (_ffi.DcInfo * m)()
        S = (_ffi.Stats * m)() if want_stats else None
        _ffi.check(self._L.dark_bwt_forward_dc_packed_batch(self._ctx, arr(text_ptrs), (ctypes.c_uint64 * m)(*[int(x) for x in ns]), cnt,
                                                            arr(bwt_ptrs), O, arr(stream_ptrs), (ctypes.c_uint64 * m)(*[int(c) for c in capacities]),
                                                            B, infos, S), self._ctx, "bwt + dc::encode (packed batch)")
        res = ([int(O[i]) for i in range(cnt)], [int(B[i]) for i in range(cnt)], [infos[i] for i in range(cnt)])
        return res + ([S[i].as_dict() for i in range(cnt)],) if want_stats else res

    def bwt_dc_packed_blocks(self, texts, want_bwt=False):
        """bwt_dc_packed for a run of host blocks through the pipelined batch entry: [(bwt or None, origin, stream, DcInfo), ...]."""
        ts = [_as_u8(t) for t in texts]
        ns = [t.size for t in ts]
        bwts = [np.empty(n, dtype=np.uint8) for n in ns] if want_bwt else None
        streams = [np.empty(_ffi.dc_packed_max(n), dtype=np.uint8) for n in ns]
        origins, sizes, infos = self.bwt_dc_packed_batch_into([t.ctypes.data for t in ts], ns, [s.ctypes.data for s in streams],
                                                              [s.size for s in streams], [b.ctypes.data for b in bwts] if want_bwt else None)
        return [(bwts[k] if want_bwt else None, origins[k], streams[k][:sizes[k]], infos[k]) for k in range(len(ts))]

    def dc_encode_packed_device(self, d_bwt, n, d_stream, capacity):
        """Device pointers: distance coding of d_bwt[0..n) with its items packed into d_stream (capacity bytes).  Returns
        (stream bytes, DcInfo)."""
        info, nbytes = _ffi.DcInfo(), ctypes.c_uint64(0)
        _ffi.check(self._L.dark_bwt_dc_encode_packed_device(self._ctx, d_bwt, int(n), d_stream, int(capacity), ctypes.byref(nbytes),
                                                            ctypes.byref(info)), self._ctx, "dc::encode (packed)")
        return int(nbytes.value), info

    # -- decoding the packed item stream: its block back, checked by re-encoding, then the text -------------------------------
    def inverse_dc_packed(self, stream, n, origin, want_bwt=False):
        """The unpack side of bwt_dc_packed (dark_bwt_inverse_dc_packed): (text np.uint8[n], bwt or None, DcInfo) from the
        packed item stream of the block's BWT and its origin.  A stream that is not exactly the packed stream of some block of
        n bytes raises DarkBwtError(E_INVALID_ARG)."""
        s = _as_u8(stream)
        n = int(n)
        text = np.empty(n, dtype=np.uint8)
        bwt = np.empty(n, dtype=np.uint8) if want_bwt else None
        info = _ffi.DcInfo()
        _ffi.check(self._L.dark_bwt_inverse_dc_packed(self._ctx, s.ctypes.data if s.size else None, s.size, n, int(origin),
                                                      text.ctypes.data if n else None, bwt.ctypes.data if want_bwt and n else None,
                                                      ctypes.byref(info)), self._ctx, "dc::decode (packed) + bwt::decode")
        return text, bwt, info

    def dc_decode_packed_device(self, d_stream, stream_bytes, n, d_bwt):
        """Device pointers: d_bwt[0..n) gets the block whose packed item stream is d_stream[0..stream_bytes)
        (dark_bwt_dc_decode_packed_device).  Returns the DcInfo the encoder gives for that block."""
        info = _ffi.DcInfo()
        _ffi.check(self._L.dark_bwt_dc_decode_packed_device(self._ctx, d_stream, int(stream_bytes), int(n), d_bwt, ctypes.byref(info)),
                   self._ctx, "dc::decode (packed)")
        return info

    # -- distance coding of many small blocks in one device pass -----------------------------------------------------
    def _dc_many_results(self, infos, ns, dist, item_starts, pos, idist, sym, rank):
        """Per-block dicts shaped like _dc_result, cut out of the concatenated outputs."""
        out, off = [], 0
        for k, n in enumerate(ns):
            a, e = int(item_starts[k]), int(item_starts[k + 1])
            d = dist[off:off + n] if dist is not None else None
            res = self._dc_result(infos[k], n, d, pos[a:e], idist[a:e], sym[a:e], rank[a:e])
            assert res["num_items"] == e - a
            out.append(res)
            off += n
        return out

    def _dc_many_outputs(self, total, count, want_dist):
        dist = np.empty(total, dtype=np.uint32) if want_dist else None
        starts = np.empty(count + 1, dtype=np.uint32)
        pos, idist = np.empty(total, dtype=np.uint32), np.empty(total, dtype=np.uint32)
        sym, rank = np.empty(total, dtype=np.uint8), np.empty(total, dtype=np.uint8)
        ptrs = [dist.ctypes.data if want_dist else None] + [a.ctypes.data for a in (starts, pos, idist, sym, rank)]
        return (dist, starts, pos, idist, sym, rank), ptrs

    def dc_encode_many(self, bwts, want_dist=True):
        """Distance coding of many small BWT blocks (host buffers) in ONE device pass (dark_bwt_dc_encode_many): a list of
        dicts shaped like dc_encode's, one per block, each what dc_encode gives on that block alone."""
        bs = [_as_u8(b) for b in bwts]
        cnt, ns = len(bs), [b.size for b in bs]
        arrays, ptrs = self._dc_many_outputs(sum(ns), cnt, want_dist)
        infos = (_ffi.DcInfo * max(cnt, 1))()
        ms = ctypes.c_float(0)
        _ffi.check(self._L.dark_bwt_dc_encode_many(self._ctx, (ctypes.c_void_p * max(cnt, 1))(*[b.ctypes.data for b in bs]),
                                                   (ctypes.c_uint64 * max(cnt, 1))(*ns), cnt, *ptrs, infos, ctypes.byref(ms)),
                   self._ctx, "dc::encode (many)")
        return self._dc_many_results(infos, ns, *arrays)

    def bwt_dc_many(self, texts, want_dist=True, want_bwt=True):
        """block/dc.rs:45-52 for many small blocks (dark_bwt_forward_dc_many): one sort of all blocks, then one DC pass over
        the BWTs while they are still in HBM.  [(bwt or None, origin, dc dict), ...]."""
        ts = [_as_u8(t) for t in texts]
        cnt, ns = len(ts), [t.size for t in ts]
        outs = [np.empty(n, dtype=np.uint8) for n in ns] if want_bwt else None
        arrays, ptrs = self._dc_many_outputs(sum(ns), cnt, want_dist)
        infos = (_ffi.DcInfo * max(cnt, 1))()
        origins = (ctypes.c_uint64 * max(cnt, 1))()
        bwt_ptrs = (ctypes.c_void_p * max(cnt, 1))(*[o.ctypes.data for o in outs]) if want_bwt else None
        _ffi.check(self._L.dark_bwt_forward_dc_many(self._ctx, (ctypes.c_void_p * max(cnt, 1))(*[t.ctypes.data for t in ts]),
                                                    (ctypes.c_uint64 * max(cnt, 1))(*ns), cnt, bwt_ptrs, origins, *ptrs, infos,
                                                    ctypes.byref(self.stats)), self._ctx, "bwt + dc::encode (many)")
        res = self._dc_many_results(infos, ns, *arrays)
        return [(outs[k] if want_bwt else None, int(origins[k]), res[k]) for k in range(cnt)]

    def dc_encode_many_device(self, d_bwt, d_starts, count, d_dist=None, d_item_starts=None, d_item_pos=None, d_item_dist=None,
                              d_item_sym=None, d_item_rank=None):
        """Device-resident form, the layout bwt_many_device writes: blocks back to back in d_bwt at the offsets d_starts[0..count]
        (u32, on the device); outputs are device pointers (all optional).  Returns (list of DcInfo headers, device ms)."""
        infos = (_ffi.DcInfo * max(int(count), 1))()
        ms = ctypes.c_float(0)
        _ffi.check(self._L.dark_bwt_dc_encode_many_device(self._ctx, d_bwt, d_starts, int(count), d_dist, d_item_starts, d_item_pos,
                                                          d_item_dist, d_item_sym, d_item_rank, infos, ctypes.byref(ms)),
                   self._ctx, "dc::encode (many)")
        return [infos[k] for k in range(int(count))], float(ms.value)

    # -- many small blocks with the packed item stream: the blocks' streams back to back, u64 offsets ------------------
    def bwt_dc_packed_many(self, texts, want_bwt=False):
        """bwt_dc_packed for many small blocks in one sort and one DC pass (dark_bwt_forward_dc_packed_many):
        [(bwt or None, origin, stream, DcInfo), ...] like bwt_dc_packed_blocks; the streams are slices of one buffer."""
        ts = [_as_u8(t) for t in texts]
        cnt, ns = len(ts), [t.size for t in ts]
        m = max(cnt, 1)
        outs = [np.empty(n, dtype=np.uint8) for n in ns] if want_bwt else None
        stream = np.empty(_ffi.dc_packed_max(sum(ns)), dtype=np.uint8)
        starts = np.empty(cnt + 1, dtype=np.uint64)
        infos, origins, nbytes = (_ffi.DcInfo * m)(), (ctypes.c_uint64 * m)(), ctypes.c_uint64(0)
        bwt_ptrs = (ctypes.c_void_p * m)(*[o.ctypes.data for o in outs]) if want_bwt else None
        _ffi.check(self._L.dark_bwt_forward_dc_packed_many(self._ctx, (ctypes.c_void_p * m)(*[t.ctypes.data for t in ts]),
                                                           (ctypes.c_uint64 * m)(*ns), cnt, bwt_ptrs, origins, stream.ctypes.data,
                                                           stream.size, starts.ctypes.data, ctypes.byref(nbytes), infos,
                                                           ctypes.byref(self.stats)), self._ctx, "bwt + dc::encode (packed many)")
        assert int(starts[cnt]) == nbytes.value
        return [(outs[k] if want_bwt else None, int(origins[k]), stream[int(starts[k]):int(starts[k + 1])], infos[k])
                for k in range(cnt)]

    def dc_encode_packed_many_device(self, d_bwt, d_starts, count, d_stream, capacity, d_stream_starts):
        """Device pointers, the layout dc_encode_many_device reads: the blocks' packed item streams back to back into d_stream
        (capacity bytes), their offsets into d_stream_starts (count + 1 u64).  Returns (total bytes, list of DcInfo, device ms)."""
        infos = (_ffi.DcInfo * max(int(count), 1))()
        nbytes, ms = ctypes.c_uint64(0), ctypes.c_float(0)
        _ffi.check(self._L.dark_bwt_dc_encode_packed_many_device(self._ctx, d_bwt, d_starts, int(count), d_stream, int(capacity),
                                                                 d_stream_starts, ctypes.byref(nbytes), infos, ctypes.byref(ms)),
                   self._ctx, "dc::encode (packed many)")
        return int(nbytes.value), [infos[k] for k in range(int(count))], float(ms.value)

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


def arena_bytes(max_n, flags=_ffi.F_DEFAULT):
    """Device bytes a Constructor(max_n, flags=flags) allocates, or 0 for a max_n or flags it rejects.  Touches no device:
    a caller can check that a block fits a card before creating the context."""
    return int(_ffi.lib().dark_bwt_arena_bytes(int(max_n), int(flags)))


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
