"""Forward + distance coding with the packed item stream (include/dark_bwt.h): dark_bwt_dc_encode_packed_device,
dark_bwt_forward_dc_packed and dark_bwt_forward_dc_packed_batch.  The stream must be byte-equal to the items of the
unpacked entries run through tests/dc_pack_ref.c, a sequential statement of the format, and the unpacked stream must give
those items back."""
import ctypes
import json
import os
import re
import subprocess
import sys
import zlib

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import dc_pack_ref  # noqa: E402
from test_alphabet_widths import DC_SIGMAS, alphabet, dc_runs  # noqa: E402

SYMBOLS = ["dark_bwt_dc_encode_packed_device", "dark_bwt_forward_dc_packed", "dark_bwt_forward_dc_packed_batch"]
KINDS = ("dna", "text", "mixed", "rep17")


def varint(v):
    out = []
    while v >= 0x80:
        out.append((v & 0x7F) | 0x80)
        v >>= 7
    return out + [v]


def pack_py(pos, dist, sym, rank):
    """The format as the header states it, item by item in Python: the check of the C statement."""
    out, prev = [], -1
    for p, d, s, r in zip(pos.tolist(), dist.tolist(), sym.tolist(), rank.tolist()):
        out += [s, r] + varint(p - prev - 1) + varint(d)
        prev = p
    return np.array(out, np.uint8)


def round_trip(pos, dist, sym, rank, n=None):
    stream = dc_pack_ref.pack(pos, dist, sym, rank)
    back = dc_pack_ref.unpack(stream)
    for a, b in zip(back, (pos, dist, sym, rank)):
        assert np.array_equal(a, np.asarray(b)), "unpack(pack(items)) differs"
    if n is not None:
        assert stream.size <= 8 * n
    return stream


# ---- CPU: exports, argument checks, the format ------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from dark_b200 import _ffi
    if not os.path.exists(_ffi.lib_path()):
        _ffi.build_native()
    return _ffi.lib()


def test_entries_and_bound_are_exported(lib):
    from dark_b200 import _ffi
    header = open(os.path.join(ROOT, "include", "dark_bwt.h")).read()
    for s in SYMBOLS:
        assert s in _ffi.SYMBOLS and hasattr(lib, s) and re.search(r"\b%s\s*\(" % s, header), s
    assert re.search(r"#define DARK_BWT_DC_PACKED_MAX\(n\) \(8ull \* \(uint64_t\)\(n\)\)", header)
    assert _ffi.dc_packed_max(5) == 40 and _ffi.dc_packed_max((1 << 32) - 2) == 8 * ((1 << 32) - 2)
    assert lib.dark_bwt_abi_version() == 2


def test_bad_arguments_are_rejected_before_any_device_work(lib):
    """A null context or required pointer is DARK_BWT_E_INVALID_ARG without touching CUDA, whatever the count."""
    from dark_b200 import _ffi
    p = (ctypes.c_void_p * 3)(1, 1, 1)
    ns = (ctypes.c_uint64 * 3)(10, 10, 10)
    caps = (ctypes.c_uint64 * 3)(80, 80, 80)
    u64s = (ctypes.c_uint64 * 3)()
    infos = (_ffi.DcInfo * 3)()
    one, info = ctypes.c_uint64(), _ffi.DcInfo()
    B = lib.dark_bwt_forward_dc_packed_batch
    for count in (0, 1, 3):
        assert B(None, None, None, count, None, None, None, None, None, None, None) == _ffi.E_INVALID_ARG
        assert B(None, p, ns, count, p, u64s, p, caps, u64s, infos, None) == _ffi.E_INVALID_ARG
        assert B(None, p, ns, count, None, u64s, None, caps, u64s, infos, None) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_dc_encode_packed_device(None, 1, 10, 1, 80, ctypes.byref(one), ctypes.byref(info)) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_dc_encode_packed_device(None, None, 10, None, 80, None, None) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_forward_dc_packed(None, 1, 10, None, ctypes.byref(one), 1, 80, ctypes.byref(one), ctypes.byref(info),
                                          None) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_forward_dc_packed(None, None, 10, None, None, None, 80, None, None, None) == _ffi.E_INVALID_ARG


def test_python_statement_matches_the_c_statement():
    rng = np.random.default_rng(3)
    m = 5000
    pos = np.cumsum(rng.integers(1, 300, m)).astype(np.uint32) - 1
    dist = (rng.integers(0, 1 << 32, m, dtype=np.uint64) >> rng.integers(0, 32, m).astype(np.uint64)).astype(np.uint32)
    sym, rank = rng.integers(0, 256, m).astype(np.uint8), rng.integers(0, 256, m).astype(np.uint8)
    assert np.array_equal(round_trip(pos, dist, sym, rank), pack_py(pos, dist, sym, rank))


@pytest.mark.parametrize("kind", KINDS)
def test_oracle_items_round_trip(oracle, kind):
    """The oracle's distance coding of every generator's BWT packs within 8 n bytes and unpacks to the same items."""
    t = oracle.gen(kind, 5, 300_007)
    bwt, _ = oracle.bwt_forward(t)
    dist, init, _, _ = oracle.dc_encode(bwt)
    items = oracle.dc_stream(bwt, dist, init)
    stream = round_trip(*items, n=t.size)
    assert stream.size >= 4 * items[0].size


@pytest.mark.parametrize("sigma", DC_SIGMAS)
def test_alphabet_width_items_round_trip(oracle, sigma):
    alpha = alphabet(sigma, sigma)
    for n in (4095, 4097, 70_001):
        b = dc_runs(alpha, n, n + sigma)
        dist, init, _, _ = oracle.dc_encode(b)
        round_trip(*oracle.dc_stream(b, dist, init), n=n)


def test_varint_boundaries_in_both_fields():
    """Run lengths - 1 and distances at every varint boundary, up to the largest run end and distance (2^32 - 2)."""
    edges = [0, 127, 128, (1 << 14) - 1, 1 << 14, (1 << 21) - 1, 1 << 21, (1 << 28) - 1, 1 << 28]
    lens1 = edges + [0] * 3
    pos = np.cumsum(np.array(lens1, np.uint64) + 1) - 1
    dist = np.array(edges[::-1] + [0, (1 << 32) - 2, (1 << 32) - 1], np.uint64)
    pos = np.append(pos, (1 << 32) - 2)                     # the last run ends at 2^32 - 2: its length - 1 is large too
    dist = np.append(dist, (1 << 32) - 2)
    m = pos.size
    sym, rank = np.arange(m, dtype=np.uint8), (255 - np.arange(m)).astype(np.uint8)
    pos, dist = pos.astype(np.uint32), dist.astype(np.uint32)
    stream = round_trip(pos, dist, sym, rank)
    assert np.array_equal(stream, pack_py(pos, dist, sym, rank))
    sizes = [2 + len(varint(int(a))) + len(varint(int(b))) for a, b in zip(np.diff(pos.astype(np.int64), prepend=-1) - 1, dist)]
    assert stream.size == sum(sizes)
    assert max(sizes) == 12 and min(sizes) == 4


def test_run_lengths_of_one_and_of_a_mebibyte():
    m = 1000
    for step in (1, 1 << 20):
        pos = (np.arange(m, dtype=np.uint64) * step + step - 1).astype(np.uint32)
        n = m * step
        dist = np.full(m, 5, np.uint32)
        stream = round_trip(pos, dist, np.zeros(m, np.uint8), np.ones(m, np.uint8), n=n)
        assert stream.size == m * (2 + len(varint(step - 1)) + 1)


def test_unpack_rejects_malformed_streams():
    good = dc_pack_ref.pack(np.array([3, 9], np.uint32), np.array([300, 2], np.uint32), np.zeros(2, np.uint8), np.zeros(2, np.uint8))
    for bad in (good[:-1], np.append(good, [1, 2, 0x80]), np.array([0, 0, 0x80, 0x80, 0x80, 0x80, 0x80, 0], np.uint8),
                np.array([0, 0, 0xFF, 0xFF, 0xFF, 0xFF, 0x1F, 0], np.uint8)):
        with pytest.raises(ValueError):
            dc_pack_ref.unpack(bad)


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


def header_of(info):
    return ([int(x) for x in info.init], bytes(info.mtf_symbols), int(info.num_unique), int(info.num_items))


def header_of_dict(r):
    return ([int(x) for x in r["init"]], bytes(np.asarray(r["mtf_symbols"], np.uint8)), int(r["num_unique"]), int(r["num_items"]))


def items_of(r):
    return r["item_pos"], r["item_dist"], r["item_sym"], r["item_rank"]


def device_blocks():
    """DC inputs: every generator, the alphabet-width blocks, n = 1 and 2, and 64 KiB +- 1 (DC of 64 KiB or less borrows
    the sort's status buffer)."""
    from dark_b200 import synth
    out = [(k, synth.generate(k, 21, n)) for k, n in zip(KINDS, (300_001, 1 << 20, 70_003, 2_000_000))]
    out += [("sigma%d" % s, dc_runs(alphabet(s, s), 100_003, s)) for s in DC_SIGMAS]
    out += [("n1", np.array([7], np.uint8)), ("n2", np.array([1, 2], np.uint8))]
    out += [("n%d" % n, synth.generate("mixed", n, n)) for n in (65_535, 65_536, 65_537)]
    return out


@pytest.mark.gpu
def test_device_form_equals_reference_pack_of_device_items(saca, torch):
    blocks = device_blocks()
    cap = max(t.size for _, t in blocks)
    with saca.Constructor(cap) as con:
        for name, t in blocks:
            n = t.size
            d_in = torch.from_numpy(t).cuda()
            d_items = [torch.zeros(n, dtype=dt, device="cuda") for dt in (torch.int32, torch.int32, torch.uint8, torch.uint8)]
            info = con.dc_encode_device(d_in.data_ptr(), n, None, *[a.data_ptr() for a in d_items])
            m = int(info.num_items)
            items = [a.cpu().numpy()[:m].view(dt) for a, dt in zip(d_items, (np.uint32, np.uint32, np.uint8, np.uint8))]
            want = dc_pack_ref.pack(*items)
            d_stream = torch.full((8 * n,), 0xA5, dtype=torch.uint8, device="cuda")
            nbytes, pinfo = con.dc_encode_packed_device(d_in.data_ptr(), n, d_stream.data_ptr(), 8 * n)
            got = d_stream.cpu().numpy()
            assert nbytes == want.size and np.array_equal(got[:nbytes], want), name
            assert (got[nbytes:] == 0xA5).all(), name
            assert header_of(pinfo) == header_of(info) and pinfo.device_ms > 0, name
            # an exact-size buffer at an odd address: the stores align to the buffer, not to its start
            d_odd = torch.full((nbytes + 17,), 0x5A, dtype=torch.uint8, device="cuda")
            assert con.dc_encode_packed_device(d_in.data_ptr(), n, d_odd.data_ptr() + 3, nbytes)[0] == nbytes
            odd = d_odd.cpu().numpy()
            assert np.array_equal(odd[3:3 + nbytes], want) and (odd[:3] == 0x5A).all() and (odd[3 + nbytes:] == 0x5A).all(), name


@pytest.mark.gpu
def test_capacity_is_checked_before_anything_is_written(saca, torch):
    from dark_b200 import _ffi, synth
    t = synth.generate("text", 3, 500_000)
    n = t.size
    with saca.Constructor(n, flags=_ffi.F_DC_BATCH) as con:
        L, ctx = con._L, con._ctx
        bwt, origin, want, info = con.bwt_dc_packed(t, want_bwt=True)
        need = want.size
        # device form, on the block's BWT
        d_in = torch.from_numpy(bwt).cuda()
        d_stream = torch.full((need,), 0xA5, dtype=torch.uint8, device="cuda")
        nb, dinfo = ctypes.c_uint64(0), _ffi.DcInfo()
        assert L.dark_bwt_dc_encode_packed_device(ctx, d_in.data_ptr(), n, d_stream.data_ptr(), need - 1, ctypes.byref(nb),
                                                  ctypes.byref(dinfo)) == _ffi.E_INVALID_ARG
        assert nb.value == need and str(need) in L.dark_bwt_last_error(ctx).decode()
        assert (d_stream.cpu().numpy() == 0xA5).all()
        assert con.dc_encode_packed_device(d_in.data_ptr(), n, d_stream.data_ptr(), need)[0] == need
        assert np.array_equal(d_stream.cpu().numpy(), want)
        # single host call: pageable and pinned sentinel buffers
        for pinned in (False, True):
            buf = torch.full((need - 1,), 0xA5, dtype=torch.uint8).pin_memory() if pinned else np.full(need - 1, 0xA5, np.uint8)
            ptr = buf.data_ptr() if pinned else buf.ctypes.data
            o, nb = ctypes.c_uint64(0), ctypes.c_uint64(0)
            assert L.dark_bwt_forward_dc_packed(ctx, t.ctypes.data, n, None, ctypes.byref(o), ptr, need - 1, ctypes.byref(nb),
                                                ctypes.byref(_ffi.DcInfo()), None) == _ffi.E_INVALID_ARG
            assert nb.value == need and str(need) in L.dark_bwt_last_error(ctx).decode()
            host = buf.numpy() if pinned else buf
            assert (host == 0xA5).all()
            b, o2, s, i = con.bwt_dc_packed(t, want_bwt=True)                     # usable after the refusal
            assert o2 == origin and np.array_equal(s, want) and header_of(i) == header_of(info)
        # exact size
        exact = np.empty(need, np.uint8)
        o, nb = ctypes.c_uint64(0), ctypes.c_uint64(0)
        _ffi.check(L.dark_bwt_forward_dc_packed(ctx, t.ctypes.data, n, None, ctypes.byref(o), exact.ctypes.data, need, ctypes.byref(nb),
                                                ctypes.byref(_ffi.DcInfo()), None), ctx, "exact")
        assert nb.value == need and np.array_equal(exact, want)


@pytest.mark.gpu
def test_single_call_equals_forward_dc_and_reference_pack(saca, oracle, torch):
    """dark_bwt_forward_dc_packed against dark_bwt_forward_dc + the reference pack: BWT, origin, stream, header; with and
    without bwt_out, pageable (staged for 1 MiB or more) and pinned buffers."""
    from dark_b200 import _ffi, synth
    blocks = [synth.generate("mixed", 41, 3 * (1 << 20) + 5), synth.generate("dna", 42, 5000), np.array([9, 9], np.uint8),
              synth.generate("rep17", 43, 65_536), synth.generate("text", 44, (1 << 21) + 1)]
    cap = max(t.size for t in blocks)
    with saca.Constructor(cap) as con:
        L, ctx = con._L, con._ctx
        for t in blocks:
            n = t.size
            rb, ro, rr = con.bwt_dc(t)
            want = dc_pack_ref.pack(*items_of(rr))
            assert want.size <= 8 * n
            for want_bwt in (False, True):
                b, o, s, info = con.bwt_dc_packed(t, want_bwt=want_bwt)
                assert o == ro and np.array_equal(s, want) and header_of(info) == header_of_dict(rr), (n, want_bwt)
                assert (b is None) != want_bwt and (b is None or np.array_equal(b, rb))
            pt = torch.from_numpy(t).pin_memory()
            ps = torch.zeros(8 * n, dtype=torch.uint8).pin_memory()
            pb = torch.zeros(n, dtype=torch.uint8).pin_memory()
            o, nb, info = ctypes.c_uint64(0), ctypes.c_uint64(0), _ffi.DcInfo()
            _ffi.check(L.dark_bwt_forward_dc_packed(ctx, pt.data_ptr(), n, pb.data_ptr(), ctypes.byref(o), ps.data_ptr(), 8 * n,
                                                    ctypes.byref(nb), ctypes.byref(info), ctypes.byref(con.stats)), ctx, "pinned")
            assert o.value == ro and nb.value == want.size and np.array_equal(ps.numpy()[:nb.value], want)
            assert np.array_equal(pb.numpy(), rb) and header_of(info) == header_of_dict(rr)
            bo, oo = oracle.bwt_forward(t)
            assert ro == oo and np.array_equal(rb, bo)


# ---- the pipelined batch ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ragged(saca, torch):
    """test_dc_batch's ragged blocks with each one's single dark_bwt_forward_dc_packed result (a context without the flag)."""
    from test_dc_batch import CAP, ragged_blocks
    blocks = ragged_blocks()
    with saca.Constructor(CAP) as con:
        ref = [con.bwt_dc_packed(t, want_bwt=True) for t in blocks]
    return CAP, blocks, ref


def same_packed(got, ref, k, want_bwt=True):
    b, o, s, info = got
    rb, ro, rs, rinfo = ref
    assert o == ro, k
    assert np.array_equal(s, rs), k
    assert header_of(info) == header_of(rinfo), k
    if want_bwt:
        assert np.array_equal(b, rb), k
    else:
        assert b is None


@pytest.mark.gpu
def test_ragged_batch_equals_single_calls(saca, torch, ragged):
    from dark_b200 import _ffi
    cap, blocks, ref = ragged
    with saca.Constructor(cap, flags=_ffi.F_DC_BATCH) as con:
        for want_bwt in (True, False):
            res = con.bwt_dc_packed_blocks(blocks, want_bwt=want_bwt)
            assert len(res) == len(blocks)
            for k, got in enumerate(res):
                same_packed(got, ref[k], k, want_bwt)
        with saca.Constructor(cap) as plain:                                        # against forward_dc + the reference pack
            for k, t in enumerate(blocks):
                rb, ro, rr = plain.bwt_dc(t)
                assert np.array_equal(ref[k][2], dc_pack_ref.pack(*items_of(rr))) and ref[k][1] == ro, k


@pytest.mark.gpu
@pytest.mark.parametrize("count", [1, 2, 3, 5])
def test_slot_alternation(saca, torch, ragged, count):
    from dark_b200 import _ffi
    cap, blocks, ref = ragged
    pick = [0, 1, 4, 6, 7][:count] if count == 5 else list(range(count))
    with saca.Constructor(cap, flags=_ffi.F_DC_BATCH) as con:
        for rep in range(2):
            for k, got in zip(pick, con.bwt_dc_packed_blocks([blocks[i] for i in pick], want_bwt=rep == 0)):
                same_packed(got, ref[k], k, rep == 0)


@pytest.mark.gpu
def test_too_small_capacity_at_block_two_of_five(saca, torch, ragged):
    """Blocks 0 and 1 are complete, the call reports block 2 and its size, block 3 on is not written, the context is usable."""
    from dark_b200 import _ffi
    cap, blocks, ref = ragged
    pick = [0, 2, 7, 1, 5]
    with saca.Constructor(cap, flags=_ffi.F_DC_BATCH) as con:
        L, ctx = con._L, con._ctx
        for pinned in (True, False):
            ts = [blocks[i] for i in pick]
            ns = [t.size for t in ts]
            sizes = [ref[i][2].size for i in pick]
            caps = [8 * n for n in ns]
            caps[2] = sizes[2] - 1
            if pinned:
                bufs = [torch.full((c,), 0xA5, dtype=torch.uint8).pin_memory() for c in caps]
                ptrs, host = [b.data_ptr() for b in bufs], [b.numpy() for b in bufs]
            else:
                host = [np.full(c, 0xA5, np.uint8) for c in caps]
                ptrs = [h.ctypes.data for h in host]
            m = len(ts)
            O, B, I = (ctypes.c_uint64 * m)(), (ctypes.c_uint64 * m)(), (_ffi.DcInfo * m)()
            rc = L.dark_bwt_forward_dc_packed_batch(ctx, (ctypes.c_void_p * m)(*[t.ctypes.data for t in ts]), (ctypes.c_uint64 * m)(*ns), m,
                                                    None, O, (ctypes.c_void_p * m)(*ptrs), (ctypes.c_uint64 * m)(*caps), B, I, None)
            assert rc == _ffi.E_INVALID_ARG
            err = L.dark_bwt_last_error(ctx).decode()
            assert "block 2" in err and str(sizes[2]) in err, err
            assert int(B[2]) == sizes[2]
            for j in (0, 1):
                assert int(B[j]) == sizes[j] and int(O[j]) == ref[pick[j]][1]
                assert np.array_equal(host[j][:sizes[j]], ref[pick[j]][2]) and (host[j][sizes[j]:] == 0xA5).all(), (pinned, j)
            for j in (2, 3, 4):
                assert (host[j] == 0xA5).all(), (pinned, j)
            for k, got in zip(pick, con.bwt_dc_packed_blocks(ts)):
                same_packed(got, ref[k], k, False)


@pytest.mark.gpu
def test_rejections_before_device_work(saca, torch, ragged):
    from dark_b200 import _ffi
    cap, blocks, ref = ragged
    small = [blocks[1], blocks[3]]

    def code(con, ts):
        with pytest.raises(_ffi.DarkBwtError) as e:
            con.bwt_dc_packed_blocks(ts)
        return e.value.code

    with saca.Constructor(cap) as con:                                            # no DC slots
        assert code(con, small) == _ffi.E_INVALID_ARG
        same_packed(con.bwt_dc_packed(blocks[1], want_bwt=True), ref[1], 1)
    with saca.Constructor(cap, flags=_ffi.F_DC_BATCH) as con:
        assert con.bwt_dc_packed_blocks([]) == []
        assert code(con, [small[0], np.zeros(1, np.uint8)]) == _ffi.E_INVALID_N
        assert code(con, [small[0], np.zeros(cap + 1, np.uint8)]) == _ffi.E_INVALID_N
        for k, got in zip((1, 3), con.bwt_dc_packed_blocks(small)):
            same_packed(got, ref[k], k, False)


@pytest.mark.gpu
def test_interleaved_with_the_other_entries(saca, torch, ragged):
    """packed batch, forward_dc_batch, forward, inverse and packed batch again on one context."""
    from dark_b200 import _ffi
    cap, blocks, ref = ragged
    idx = (0, 2, 1, 9)
    batch = [blocks[i] for i in idx]
    with saca.Constructor(cap, flags=_ffi.F_DC_BATCH) as con:
        for _ in range(2):
            for k, got in zip(idx, con.bwt_dc_packed_blocks(batch, want_bwt=True)):
                same_packed(got, ref[k], k)
            for k, (b, o, r) in zip(idx, con.bwt_dc_blocks(batch)):
                assert o == ref[k][1] and np.array_equal(b, ref[k][0]) and np.array_equal(dc_pack_ref.pack(*items_of(r)), ref[k][2]), k
            b, o = con.bwt(blocks[6])
            assert o == ref[6][1] and np.array_equal(b, ref[6][0])
            assert np.array_equal(con.inverse(ref[7][0], ref[7][1]), blocks[7])
            same_packed(con.bwt_dc_packed(blocks[5], want_bwt=True), ref[5], 5)


@pytest.mark.gpu
@pytest.mark.parametrize("threads", ["0", "3"])
def test_pinned_and_pageable_buffers(threads):
    """Pageable streams of 1 MiB or more (through the staging lanes, or the driver's staging with 0 lanes) and pinned ones
    give what single packed calls give."""
    code = (
        "import ctypes, numpy as np, torch\n"
        "from dark_b200 import saca, synth, _ffi\n"
        "blocks = [synth.generate('mixed', 31, 3 * (1 << 20) + 12345), synth.generate('dna', 32, 5000),\n"
        "          synth.generate('text', 33, (1 << 21) + 7), synth.generate('rep17', 34, 1 << 20)]\n"
        "ns = [t.size for t in blocks]\n"
        "with saca.Constructor(max(ns)) as c:\n"
        "    ref = [c.bwt_dc_packed(t, want_bwt=True) for t in blocks]\n"
        "with saca.Constructor(max(ns), flags=_ffi.F_DC_BATCH) as c:\n"
        "    for k, (b, o, s, i) in enumerate(c.bwt_dc_packed_blocks(blocks, want_bwt=True)):\n"
        "        assert o == ref[k][1] and np.array_equal(b, ref[k][0]) and np.array_equal(s, ref[k][2]), k\n"
        "    tx = [torch.from_numpy(t).pin_memory() for t in blocks]\n"
        "    for mixed in (False, True):\n"
        "        st = [np.zeros(8 * n, np.uint8) if mixed and k % 2 == 0 else torch.zeros(8 * n, dtype=torch.uint8).pin_memory() for k, n in enumerate(ns)]\n"
        "        bw = [np.zeros(n, np.uint8) if mixed else torch.zeros(n, dtype=torch.uint8).pin_memory() for n in ns]\n"
        "        ptr = lambda a: a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr()\n"
        "        h = lambda a: a if isinstance(a, np.ndarray) else a.numpy()\n"
        "        origins, sizes, infos = c.bwt_dc_packed_batch_into([t.data_ptr() for t in tx], ns, [ptr(a) for a in st], [8 * n for n in ns],\n"
        "                                                           [ptr(a) for a in bw])\n"
        "        for k in range(len(blocks)):\n"
        "            assert origins[k] == ref[k][1] and sizes[k] == ref[k][2].size, k\n"
        "            assert np.array_equal(h(st[k])[:sizes[k]], ref[k][2]) and np.array_equal(h(bw[k]), ref[k][0]), (mixed, k)\n"
        "print('ok')\n")
    env = dict(os.environ, DARK_BWT_HOST_THREADS=threads)
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


@pytest.mark.gpu
def test_full_size_blocks(saca, torch):
    """Two 256 MiB blocks of C2 and two of the first C5 block through one batch equal the single packed calls, and the
    streams unpack to the items dark_bwt_forward_dc gives."""
    from dark_b200 import _ffi, synth
    n = 1 << 28
    c2, c5 = synth.generate("dna", 1, n), synth.generate(*synth.c5_block(0))
    blocks = [c2, c5, c2, c5]
    with saca.Constructor(n, flags=_ffi.F_DC_BATCH) as con:
        res = con.bwt_dc_packed_blocks(blocks)
        for k, t in enumerate(blocks[:2]):
            single = con.bwt_dc_packed(t)
            same_packed(res[k], single, k, False)
            same_packed(res[k + 2], single, k + 2, False)
            _, _, r = con.bwt_dc(t, want_dist=False)
            got = dc_pack_ref.unpack(single[2], int(single[3].num_items))
            for a, b in zip(got, items_of(r)):
                assert np.array_equal(a, b), k
            del single, r, got


def crc(a):
    c = 0
    a = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    for i in range(0, a.size, 1 << 30):
        c = zlib.crc32(memoryview(a[i:i + (1 << 30)]), c)
    return "%08x" % c


@pytest.mark.gpu
def test_top_of_the_range(saca, torch):
    """The DNA block of 2^32 - 2 bytes through dark_bwt_forward_dc_packed on a default context: a stream of more than
    2^32 bytes (u64 tile offsets) that unpacks to the oracle's items of tests/golden/large_dc.json."""
    import gc
    from dark_b200 import synth
    top = (1 << 32) - 2
    with open(os.path.join(ROOT, "tests", "golden", "large_dc.json")) as f:
        g = json.load(f)
    assert g["block"] == "dna:1:%d" % top
    t = synth.generate("dna", 1, top)
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    con = saca.Constructor(top)
    try:
        _, origin, stream, info = con.bwt_dc_packed(t)
    finally:
        con.close()
    del t
    m = int(info.num_items)
    assert m == g["num_items"] and stream.size > 1 << 32 and stream.size <= 8 * top
    assert [int(x) for x in info.init] == g["init"] and int(info.num_unique) == g["num_unique"]
    items = dc_pack_ref.unpack(stream, m)
    del stream
    assert items[0].size == m
    got = {name + "_crc32": crc(a) for name, a in zip(("item_pos", "item_dist", "item_sym", "item_rank"), items)}
    print(got)
    assert got == {k: g[k] for k in got}
