"""The packed item stream for many small blocks: dark_bwt_dc_encode_packed_many_device and dark_bwt_forward_dc_packed_many.
Block k's slice stream[stream_starts[k]:stream_starts[k+1]] must be what the single packed entries give for that block
alone, and what tests/dc_pack_ref.c packs block k's items of the unpacked many-block entries to."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import dc_pack_ref  # noqa: E402
from test_dc_many import MAX_MANY, RECORD, block_sets, fused_blocks, max_blocks  # noqa: E402

SYMBOLS = ["dark_bwt_dc_encode_packed_many_device", "dark_bwt_forward_dc_packed_many"]
SENTINEL = 0xA5
TILE = 2048  # items per tile of the pack kernels


# ---- CPU: exports and argument checks (no device work) ------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from dark_b200 import _ffi
    if not os.path.exists(_ffi.lib_path()):
        _ffi.build_native()
    return _ffi.lib()


def test_entries_are_declared_and_exported(lib):
    from dark_b200 import _ffi
    header = open(os.path.join(ROOT, "include", "dark_bwt.h")).read()
    for s in SYMBOLS:
        assert s in _ffi.SYMBOLS and hasattr(lib, s) and re.search(r"\b%s\s*\(" % s, header), s
    assert lib.dark_bwt_abi_version() == 2


def test_bad_arguments_are_rejected_before_any_device_work(lib):
    """A null context or required pointer is DARK_BWT_E_INVALID_ARG without touching CUDA, whatever the count."""
    from dark_b200 import _ffi
    p = (ctypes.c_void_p * 3)(1, 1, 1)
    ns = (ctypes.c_uint64 * 3)(10, 10, 10)
    u64s = (ctypes.c_uint64 * 4)()
    infos = (_ffi.DcInfo * 3)()
    one, ms = ctypes.c_uint64(), ctypes.c_float()
    D, H = lib.dark_bwt_dc_encode_packed_many_device, lib.dark_bwt_forward_dc_packed_many
    for count in (0, 1, 3):
        assert D(None, None, None, count, None, 0, None, None, None, None) == _ffi.E_INVALID_ARG
        assert D(None, 1, 1, count, 1, 80, 1, ctypes.byref(one), infos, ctypes.byref(ms)) == _ffi.E_INVALID_ARG
        assert H(None, None, None, count, None, None, None, 0, None, None, None, None) == _ffi.E_INVALID_ARG
        assert H(None, p, ns, count, None, u64s, 1, 240, u64s, ctypes.byref(one), infos, None) == _ffi.E_INVALID_ARG


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch as t
    if not t.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback)")
    return t


@pytest.fixture(scope="module")
def saca():
    from dark_b200 import saca as s
    return s


def as_u8(b):
    return b if isinstance(b, np.ndarray) else np.frombuffer(bytes(b), dtype=np.uint8)


def header_of(info):
    return ([int(x) for x in info.init], bytes(info.mtf_symbols), int(info.num_unique), int(info.num_items))


def header_of_dict(r):
    return ([int(x) for x in r["init"]], bytes(np.asarray(r["mtf_symbols"], np.uint8)), int(r["num_unique"]), int(r["num_items"]))


def items_of(r):
    return r["item_pos"], r["item_dist"], r["item_sym"], r["item_rank"]


def runs_block(nruns, seed, max_len=9, sigma=4, lo=97):
    """A block of exactly `nruns` runs (adjacent runs differ), run lengths 1..max_len."""
    r = np.random.default_rng(seed)
    syms = np.empty(nruns, np.int64)
    syms[0] = r.integers(0, sigma)
    steps = r.integers(1, sigma, nruns - 1)
    syms[1:] = (syms[0] + np.cumsum(steps)) % sigma
    return (np.repeat(syms, r.integers(1, max_len + 1, nruns)) + lo).astype(np.uint8)


def pack_sets():
    """Block lists aimed at the pack (each block's items are its runs)."""
    # first items of blocks at items 2047, 2048, 2049 (the last, first and second item of a tile) and around later tiles
    firsts = [0, 2047, 2048, 2049, 4095, 4096, 6143, 6144, 6151, 8192 + 7, 10_240]
    tile_edges = [runs_block(b - a, 300 + i, max_len=1 + (i % 3) * 150) for i, (a, b) in enumerate(zip(firsts, firsts[1:] + [12_000]))]
    # runs of >= 128 and >= 16,384 bytes at a block start (2 and 3 varint bytes), after blocks ending in the same byte
    rng = np.random.default_rng(7)
    long_runs = []
    for i, run in enumerate((127, 128, 129, 16_383, 16_384, 16_385, (1 << 21) + 1)):
        tail = rng.integers(98, 102, 500 + 37 * i).astype(np.uint8)
        long_runs += [np.concatenate([np.full(run, 97, np.uint8), tail, np.full(3, 97, np.uint8)])]
    # one run per byte: more than n / 2 runs, so there are more tiles of items than 4 KiB chunks of bytes
    alternating = [np.resize(np.array([65 + (k % 3), 66 + (k % 3)], np.uint8), 1500 + k) for k in range(200)]
    alternating += [np.resize(np.array([1, 2, 3], np.uint8), (1 << 20) + 5)]
    return {"tile_edges": tile_edges, "long_runs_at_block_starts": long_runs, "alternating_bytes": alternating}


def all_sets():
    s = block_sets()
    s.update(pack_sets())
    return s


def device_packed_many(con, torch, blocks, capacity=None):
    """dark_bwt_dc_encode_packed_many_device on the blocks back to back: (stream, offsets, infos, ms, total), read back
    from sentinel-filled buffers of `capacity` bytes (default DARK_BWT_DC_PACKED_MAX(total))."""
    starts = np.concatenate([[0], np.cumsum([b.size for b in blocks])]).astype(np.uint32)
    n, cnt = int(starts[-1]), len(blocks)
    cap = 8 * n if capacity is None else capacity
    d_bwt = torch.from_numpy(np.concatenate(blocks)).cuda()
    d_starts = torch.from_numpy(starts.view(np.int32)).cuda()
    d_stream = torch.full((max(cap, 1),), SENTINEL, dtype=torch.uint8, device="cuda")
    d_offs = torch.full((cnt + 1,), -1, dtype=torch.int64, device="cuda")
    total, infos, ms = con.dc_encode_packed_many_device(d_bwt.data_ptr(), d_starts.data_ptr(), cnt, d_stream.data_ptr(), cap,
                                                        d_offs.data_ptr())
    return d_stream.cpu().numpy(), d_offs.cpu().numpy().view(np.uint64), infos, ms, total, (d_bwt, d_starts, starts)


def check_device_form(saca, torch, blocks, single_every=1):
    """The device form against dc_encode_many_device's items through the reference pack (every block) and against
    dc_encode_packed_device on each single_every-th block alone (a fresh context)."""
    bs = [as_u8(b) for b in blocks]
    total = sum(b.size for b in bs)
    cap = max(total, (len(bs) * RECORD - 1024 + 7) // 8, 2)
    with saca.Constructor(cap) as con:
        stream, offs, infos, ms, nbytes, (d_bwt, d_starts, starts) = device_packed_many(con, torch, bs)
        assert int(offs[0]) == 0 and int(offs[-1]) == nbytes and np.all(np.diff(offs.astype(np.int64)) > 0)
        assert (stream[nbytes:] == SENTINEL).all()
        assert ms > 0 and all(i.device_ms == ms for i in infos)
        # the unpacked many-block entry on the same context, its items packed block by block by the reference
        n, cnt = total, len(bs)
        outs = [torch.zeros(n, dtype=torch.int32, device="cuda") for _ in range(2)] + [torch.zeros(n, dtype=torch.uint8, device="cuda")
                                                                                        for _ in range(2)]
        d_its = torch.zeros(cnt + 1, dtype=torch.int32, device="cuda")
        uinfos, _ = con.dc_encode_many_device(d_bwt.data_ptr(), d_starts.data_ptr(), cnt, None, d_its.data_ptr(),
                                              *[o.data_ptr() for o in outs])
        pos, idist, sym, rank = [o.cpu().numpy().view(dt) for o, dt in zip(outs, (np.uint32, np.uint32, np.uint8, np.uint8))]
        its = d_its.cpu().numpy().view(np.uint32)
        for k in range(cnt):
            a, e = int(its[k]), int(its[k + 1])
            want = dc_pack_ref.pack(pos[a:e], idist[a:e], sym[a:e], rank[a:e])
            got = stream[int(offs[k]):int(offs[k + 1])]
            assert np.array_equal(got, want), k
            assert header_of(infos[k]) == header_of(uinfos[k]), k
    with saca.Constructor(cap) as single:
        for k in range(0, cnt, single_every):
            nk = bs[k].size
            d_one = torch.full((8 * nk,), SENTINEL, dtype=torch.uint8, device="cuda")
            nb, info = single.dc_encode_packed_device(d_bwt.data_ptr() + int(starts[k]), nk, d_one.data_ptr(), 8 * nk)
            assert nb == int(offs[k + 1] - offs[k]), k
            assert np.array_equal(d_one.cpu().numpy()[:nb], stream[int(offs[k]):int(offs[k + 1])]), k
            assert header_of(info) == header_of(infos[k]), k
    return stream, offs, infos


def check_host_form(saca, texts, single_every=1, want_bwt=True):
    """The host form against dark_bwt_forward_dc_packed on each single_every-th block alone and, unpacked, against the
    items of dark_bwt_forward_dc_many (every block)."""
    ts = [as_u8(t) for t in texts]
    cap = max(sum(t.size for t in ts), (len(ts) * RECORD - 1024 + 7) // 8, 2)
    with saca.Constructor(cap) as con:
        res = con.bwt_dc_packed_many(ts, want_bwt=want_bwt)
        unpacked = con.bwt_dc_many(ts, want_dist=False, want_bwt=False)
    assert len(res) == len(ts)
    for k, ((b, o, s, info), (_, uo, r)) in enumerate(zip(res, unpacked)):
        assert o == uo and header_of(info) == header_of_dict(r), k
        assert (b is None) != want_bwt
        got = dc_pack_ref.unpack(s, int(info.num_items))
        assert got[0].size == int(info.num_items)
        for x, y in zip(got, items_of(r)):
            assert np.array_equal(x, y), k
        assert np.array_equal(dc_pack_ref.pack(*items_of(r)), s), k
    with saca.Constructor(cap) as single:
        for k in range(0, len(ts), single_every):
            b, o, s, info = res[k]
            rb, ro, rs, rinfo = single.bwt_dc_packed(ts[k], want_bwt=True)
            assert o == ro and np.array_equal(s, rs) and header_of(info) == header_of(rinfo), k
            if want_bwt:
                assert np.array_equal(b, rb), k
    return res


DEVICE_SETS = ["one_byte_blocks_256", "one_byte_blocks_small", "on_chunk_boundaries", "straddling_chunks", "many_in_one_chunk",
               "longer_than_a_scan_group", "equal_bytes_across_boundaries", "union_le_32_dna", "union_256", "text_slices",
               "tile_edges", "long_runs_at_block_starts", "alternating_bytes"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", DEVICE_SETS)
def test_device_form_block_sets(saca, torch, name):
    blocks = all_sets()[name]
    check_device_form(saca, torch, blocks, single_every=1 if len(blocks) <= 1000 else 37)


@pytest.mark.gpu
def test_tile_edges_land_where_planned(saca, torch):
    """The tile-edge blocks do open at items 2047, 2048, 2049, 4095 and 4096, and the alternating list has one run per
    byte (more tiles of 2,048 items than 4 KiB chunks of bytes)."""
    sets = pack_sets()
    _, _, infos = check_device_form(saca, torch, sets["tile_edges"][:6])
    firsts = np.concatenate([[0], np.cumsum([int(i.num_items) for i in infos])])
    assert {2047, 2048, 2049, 4095, 4096} <= set(firsts.tolist())
    alt = sets["alternating_bytes"]
    assert all(np.count_nonzero(np.diff(b)) == b.size - 1 for b in alt)


HOST_SETS = ["on_chunk_boundaries", "straddling_chunks", "union_le_32_dna", "text_slices", "tile_edges", "long_runs_at_block_starts",
             "alternating_bytes"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", HOST_SETS)
def test_host_form_block_sets(saca, torch, name):
    """Host form on the block sets, without their one-byte blocks (the sort needs two bytes)."""
    check_host_form(saca, [b for b in all_sets()[name] if len(b) >= 2])


@pytest.mark.gpu
def test_host_form_generators_with_and_without_bwt(saca, torch):
    """DNA, text, mixed and rep17 blocks of several sizes, with and without the BWTs."""
    texts = fused_blocks()
    check_host_form(saca, texts, want_bwt=True)
    check_host_form(saca, texts[:12], want_bwt=False)




def host_call(L, ctx, texts, stream_ptr, capacity, offs_ptr, bwt_ptrs=None):
    """dark_bwt_forward_dc_packed_many on raw host addresses: (rc, origins, total bytes, DcInfo array)."""
    from dark_b200 import _ffi
    cnt = len(texts)
    m = max(cnt, 1)
    O, nb, I = (ctypes.c_uint64 * m)(), ctypes.c_uint64(12345), (_ffi.DcInfo * m)()
    bp = (ctypes.c_void_p * m)(*bwt_ptrs) if bwt_ptrs is not None else None
    rc = L.dark_bwt_forward_dc_packed_many(ctx, (ctypes.c_void_p * m)(*[t.ctypes.data for t in texts]),
                                           (ctypes.c_uint64 * m)(*[t.size for t in texts]), cnt, bp, O, stream_ptr, capacity, offs_ptr,
                                           ctypes.byref(nb), I, None)
    return rc, [int(O[k]) for k in range(cnt)], int(nb.value), I


@pytest.mark.gpu
def test_capacity_rule(saca, torch):
    """total - 1 bytes: DARK_BWT_E_INVALID_ARG with the size needed, neither stream nor offsets written, the context usable;
    exactly total: OK.  Device form, and the host form on pageable and pinned buffers."""
    from dark_b200 import _ffi, synth
    texts = [synth.generate(("text", "dna", "mixed")[k % 3], 500 + k, 20_000 + 997 * k) for k in range(9)]
    texts += [synth.generate("mixed", 510, (1 << 20) + 3)]  # a stream above 1 MiB: the pageable copy takes the staging lanes
    cnt = len(texts)
    with saca.Constructor(sum(t.size for t in texts)) as ref:
        want = ref.bwt_dc_packed_many(texts, want_bwt=True)
    sizes = [s.size for _, _, s, _ in want]
    need = sum(sizes)
    assert need >= 1 << 20
    want_stream = np.concatenate([s for _, _, s, _ in want])
    want_offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    sentinel_u64 = np.uint64(0xA5A5A5A5A5A5A5A5)
    with saca.Constructor(sum(t.size for t in texts)) as con:
        L, ctx = con._L, con._ctx
        bwts = [b for b, _, _, _ in want]
        starts = np.concatenate([[0], np.cumsum([b.size for b in bwts])]).astype(np.uint32)
        d_bwt = torch.from_numpy(np.concatenate(bwts)).cuda()
        d_starts = torch.from_numpy(starts.view(np.int32)).cuda()
        for cap in (need - 1, need):
            d_stream = torch.full((need,), SENTINEL, dtype=torch.uint8, device="cuda")
            d_offs = torch.full((cnt + 1,), -1, dtype=torch.int64, device="cuda")
            nb, ms, infos = ctypes.c_uint64(0), ctypes.c_float(0), (_ffi.DcInfo * cnt)()
            rc = L.dark_bwt_dc_encode_packed_many_device(ctx, d_bwt.data_ptr(), d_starts.data_ptr(), cnt, d_stream.data_ptr(), cap,
                                                         d_offs.data_ptr(), ctypes.byref(nb), infos, ctypes.byref(ms))
            assert nb.value == need
            if cap < need:
                assert rc == _ffi.E_INVALID_ARG and str(need) in L.dark_bwt_last_error(ctx).decode()
                assert (d_stream.cpu().numpy() == SENTINEL).all() and (d_offs.cpu().numpy() == -1).all()
            else:
                assert rc == _ffi.OK
                assert np.array_equal(d_stream.cpu().numpy(), want_stream)
                assert np.array_equal(d_offs.cpu().numpy().view(np.uint64), want_offs)
                assert all(header_of(infos[k]) == header_of(want[k][3]) for k in range(cnt))
        for pinned in (False, True):
            for cap in (need - 1, need):
                if pinned:
                    keep = [torch.full((need,), SENTINEL, dtype=torch.uint8).pin_memory(),
                            torch.from_numpy(np.full(cnt + 1, sentinel_u64).view(np.int64)).pin_memory()]
                    keep += [torch.zeros(t.size, dtype=torch.uint8).pin_memory() for t in texts]
                    host = [keep[0].numpy(), keep[1].numpy().view(np.uint64)] + [b.numpy() for b in keep[2:]]
                    ptrs = [k.data_ptr() for k in keep]
                else:
                    host = [np.full(need, SENTINEL, np.uint8), np.full(cnt + 1, sentinel_u64, np.uint64)]
                    host += [np.zeros(t.size, np.uint8) for t in texts]
                    ptrs = [h.ctypes.data for h in host]
                rc, origins, nb, infos = host_call(L, ctx, texts, ptrs[0], cap, ptrs[1], ptrs[2:])
                assert nb == need, (pinned, cap)
                if cap < need:
                    assert rc == _ffi.E_INVALID_ARG and str(need) in L.dark_bwt_last_error(ctx).decode()
                    assert (host[0] == SENTINEL).all() and (host[1] == sentinel_u64).all(), pinned
                else:
                    assert rc == _ffi.OK, pinned
                    assert np.array_equal(host[0], want_stream) and np.array_equal(host[1], want_offs), pinned
                    for k in range(cnt):
                        assert origins[k] == want[k][1] and np.array_equal(host[2 + k], want[k][0]), (pinned, k)
                        assert header_of(infos[k]) == header_of(want[k][3]), (pinned, k)


@pytest.mark.gpu
def test_limits(saca, torch):
    """DARK_BWT_MAX_MANY_BLOCKS blocks are accepted; the record bound gives DARK_BWT_E_INVALID_N at the count
    dark_bwt_forward_dc_many refuses; the other refusals of the many-block entries."""
    from dark_b200 import _ffi

    def code(call):
        with pytest.raises(_ffi.DarkBwtError) as e:
            call()
        return e.value.code

    rng = np.random.default_rng(61)
    check_device_form(saca, torch, [rng.integers(0, 3, int(s)).astype(np.uint8) for s in rng.integers(1, 5, MAX_MANY)],
                      single_every=4099)
    check_host_form(saca, [rng.integers(0, 3, int(s)).astype(np.uint8) for s in rng.integers(2, 5, MAX_MANY)], single_every=4099,
                    want_bwt=False)
    cap = 15_972  # 8 * cap + 1024 = 100 records
    assert max_blocks(cap) == 100
    blocks = [rng.integers(0, 5, 150).astype(np.uint8) for _ in range(100)]
    with saca.Constructor(cap) as con:
        assert len(con.bwt_dc_packed_many(blocks)) == 100
        assert code(lambda: con.bwt_dc_many(blocks + [b"xy"])) == _ffi.E_INVALID_N
        assert code(lambda: con.bwt_dc_packed_many(blocks + [b"xy"])) == _ffi.E_INVALID_N
        assert code(lambda: device_packed_many(con, torch, blocks + [np.array([1], np.uint8)])) == _ffi.E_INVALID_N
        assert len(device_packed_many(con, torch, blocks)[2]) == 100
        assert code(lambda: device_packed_many(con, torch, [np.array([1, 2], np.uint8), np.zeros(0, np.uint8)])) == _ffi.E_INVALID_N
        assert code(lambda: con.bwt_dc_packed_many([b"abc", b"a"])) == _ffi.E_INVALID_N     # the sort needs 2 bytes
        assert code(lambda: con.bwt_dc_packed_many([b"a" * 10_000, b"b" * 6_000])) == _ffi.E_INVALID_N  # sum(ns) > capacity
        # count == 0: OK, total 0, stream_starts[0] = 0 (host form)
        L, ctx = con._L, con._ctx
        offs = np.full(1, 7, np.uint64)
        rc, _, nb, _ = host_call(L, ctx, [], np.zeros(8, np.uint8).ctypes.data, 8, offs.ctypes.data)
        assert rc == _ffi.OK and nb == 0 and int(offs[0]) == 0
        assert con.bwt_dc_packed_many([]) == []
        nbd, ms = ctypes.c_uint64(9), ctypes.c_float(0)
        d = torch.zeros(8, dtype=torch.uint8, device="cuda")
        assert L.dark_bwt_dc_encode_packed_many_device(ctx, d.data_ptr(), d.data_ptr(), 0, d.data_ptr(), 8, d.data_ptr(), ctypes.byref(nbd),
                                                       (_ffi.DcInfo * 1)(), ctypes.byref(ms)) == _ffi.OK and nbd.value == 0
    with saca.Constructor(MAX_MANY * 200) as con:                                            # count > DARK_BWT_MAX_MANY_BLOCKS
        assert code(lambda: con.bwt_dc_packed_many([b"ab"] * (MAX_MANY + 1))) == _ffi.E_INVALID_ARG
        assert code(lambda: device_packed_many(con, torch, [np.array([1, 2], np.uint8)] * (MAX_MANY + 1))) == _ffi.E_INVALID_ARG
    with saca.Constructor(1000, flags=_ffi.F_DEVICE_ONLY) as con:                            # the host form needs the staging buffers
        assert code(lambda: con.bwt_dc_packed_many([b"banana"])) == _ffi.E_INVALID_ARG
        assert len(device_packed_many(con, torch, [np.frombuffer(b"nnbaaa", np.uint8)])[2]) == 1


@pytest.mark.gpu
def test_interleaved_with_the_other_entries(saca, torch):
    """Both new entries, dark_bwt_forward_dc_packed, dark_bwt_forward_dc_many and dark_bwt_forward on one context keep
    giving what a fresh context gives (scratch left in keys[1], ranks or ranks_alt would show)."""
    from dark_b200 import synth
    big = synth.generate("mixed", 70, 1 << 20)
    small = [synth.generate("text", 71 + k, 2000 + 37 * k) for k in range(12)]
    alt = pack_sets()["alternating_bytes"][:40]
    texts = [synth.generate("dna", 90, 300_000), synth.generate("text", 91, 200_000)] + small[:4]
    cap = 1 << 21

    def fresh(f):
        with saca.Constructor(cap) as c:
            return f(c)
    f_pm = fresh(lambda c: c.bwt_dc_packed_many(texts, want_bwt=True))
    f_ps = fresh(lambda c: c.bwt_dc_packed_many(small))
    f_dev = fresh(lambda c: device_packed_many(c, torch, alt)[:3])
    f_p = fresh(lambda c: c.bwt_dc_packed(big, want_bwt=True))
    f_dm = fresh(lambda c: c.bwt_dc_many(texts))
    f_fwd = fresh(lambda c: c.bwt(big))

    def same_packed(got, ref):
        for (b, o, s, i), (rb, ro, rs, ri) in zip(got, ref):
            assert o == ro and np.array_equal(s, rs) and header_of(i) == header_of(ri)
            assert (b is None and rb is None) or np.array_equal(b, rb)
    with saca.Constructor(cap) as con:
        for _ in range(2):
            same_packed(con.bwt_dc_packed_many(texts, want_bwt=True), f_pm)
            same_packed([con.bwt_dc_packed(big, want_bwt=True)], [f_p])
            s, o, i = device_packed_many(con, torch, alt)[:3]
            assert np.array_equal(s, f_dev[0]) and np.array_equal(o, f_dev[1])
            assert [header_of(x) for x in i] == [header_of(x) for x in f_dev[2]]
            for (b, o, r), (fb, fo, fr) in zip(con.bwt_dc_many(texts), f_dm):
                assert o == fo and np.array_equal(b, fb) and header_of_dict(r) == header_of_dict(fr)
                assert all(np.array_equal(x, y) for x, y in zip(items_of(r), items_of(fr)))
            b, o = con.bwt(big)
            assert o == f_fwd[1] and np.array_equal(b, f_fwd[0])
            same_packed(con.bwt_dc_packed_many(small), f_ps)


@pytest.mark.gpu
@pytest.mark.parametrize("threads", ["0", "3"])
def test_pinned_and_pageable_buffers(threads):
    """A pageable stream of 1 MiB or more (through the staging lanes, or the driver's staging with 0 lanes) and pinned
    buffers give the same stream, offsets, BWTs and origins, equal to single packed calls."""
    code = (
        "import ctypes, numpy as np, torch, sys\n"
        "sys.path.insert(0, 'tests')\n"
        "from test_dc_packed_many import host_call, header_of\n"
        "from dark_b200 import saca, synth, _ffi\n"
        "blocks = [synth.generate('mixed', 31, 3 * (1 << 20) + 12345), synth.generate('dna', 32, 5000),\n"
        "          synth.generate('text', 33, (1 << 21) + 7), synth.generate('rep17', 34, 1 << 20), np.array([5, 5], np.uint8)]\n"
        "ns = [t.size for t in blocks]\n"
        "with saca.Constructor(max(ns)) as c:\n"
        "    ref = [c.bwt_dc_packed(t, want_bwt=True) for t in blocks]\n"
        "want = np.concatenate([s for _, _, s, _ in ref])\n"
        "offs = np.concatenate([[0], np.cumsum([s.size for _, _, s, _ in ref])]).astype(np.uint64)\n"
        "assert want.size >= 1 << 20\n"
        "with saca.Constructor(sum(ns)) as c:\n"
        "    for k, (b, o, s, i) in enumerate(c.bwt_dc_packed_many(blocks, want_bwt=True)):\n"
        "        assert o == ref[k][1] and np.array_equal(b, ref[k][0]) and np.array_equal(s, ref[k][2]), k\n"
        "        assert header_of(i) == header_of(ref[k][3]), k\n"
        "    cap = 8 * sum(ns)\n"
        "    for pinned_stream in (False, True):\n"
        "        st = torch.zeros(cap, dtype=torch.uint8).pin_memory() if pinned_stream else np.zeros(cap, np.uint8)\n"
        "        of = np.zeros(len(ns) + 1, np.uint64)\n"
        "        bw = [torch.zeros(n, dtype=torch.uint8).pin_memory() if pinned_stream else np.zeros(n, np.uint8) for n in ns]\n"
        "        ptr = lambda a: a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr()\n"
        "        h = lambda a: a if isinstance(a, np.ndarray) else a.numpy()\n"
        "        rc, origins, nb, infos = host_call(c._L, c._ctx, blocks, ptr(st), cap, of.ctypes.data, [ptr(b) for b in bw])\n"
        "        assert rc == 0 and nb == want.size and np.array_equal(h(st)[:nb], want) and np.array_equal(of, offs), pinned_stream\n"
        "        for k in range(len(blocks)):\n"
        "            assert origins[k] == ref[k][1] and np.array_equal(h(bw[k]), ref[k][0]), (pinned_stream, k)\n"
        "print('ok')\n")
    env = dict(os.environ, DARK_BWT_HOST_THREADS=threads)
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


@pytest.mark.gpu
def test_a_list_near_capacity(saca, torch):
    """256 mixed blocks of 1 MiB on a context of exactly their sum: every block unpacks to the items of
    dark_bwt_forward_dc_many, and every 17th equals dark_bwt_forward_dc_packed on it alone."""
    from dark_b200 import synth
    texts = [synth.generate("mixed", 1000 + k, 1 << 20) for k in range(256)]
    check_host_form(saca, texts, single_every=17, want_bwt=False)
