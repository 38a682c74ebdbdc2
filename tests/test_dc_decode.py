"""Decoding the packed item stream (include/dark_bwt.h): dark_bwt_dc_decode_packed_device and dark_bwt_inverse_dc_packed.
A stream is accepted only if it is byte for byte the packed stream of the block it decodes to; the tests round-trip every
generator and shape through the encoder, and check that every kind of damaged stream is refused without touching the
caller's outputs, on a context that stays usable."""
import ctypes
import json
import os
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

SYMBOLS = ["dark_bwt_dc_decode_packed_device", "dark_bwt_inverse_dc_packed"]
KINDS = ("dna", "text", "mixed", "rep17")
CAP = (1 << 28) + 1          # room for one run whose length - 1 takes a 5-byte varint
TILE = 8192                  # kUnpackTile (dc_kernels.cuh): the parse's tile


def decode_py(stream, n):
    """The decode as a statement in Python: the items' run lengths and symbols expanded."""
    pos, _, sym, _ = dc_pack_ref.unpack(stream)
    runs = np.diff(pos.astype(np.int64), prepend=-1)
    assert runs.sum() == n
    return np.repeat(sym, runs)


def varint(v):
    out = []
    while v >= 0x80:
        out.append((v & 0x7F) | 0x80)
        v >>= 7
    return out + [v]


# ---- CPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from dark_b200 import _ffi
    if not os.path.exists(_ffi.lib_path()):
        _ffi.build_native()
    return _ffi.lib()


def test_entries_are_exported_and_declared(lib):
    import re
    from dark_b200 import _ffi
    header = open(os.path.join(ROOT, "include", "dark_bwt.h")).read()
    for s in SYMBOLS:
        assert s in _ffi.SYMBOLS and hasattr(lib, s) and re.search(r"\b%s\s*\(" % s, header), s


def test_null_arguments_are_refused_without_cuda(lib):
    from dark_b200 import _ffi
    info = _ffi.DcInfo()
    assert lib.dark_bwt_dc_decode_packed_device(None, 1, 10, 10, 1, ctypes.byref(info)) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_dc_decode_packed_device(None, None, 10, 10, None, None) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_inverse_dc_packed(None, 1, 10, 10, 0, 1, 1, ctypes.byref(info)) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_inverse_dc_packed(None, None, 10, 10, 0, None, None, None) == _ffi.E_INVALID_ARG


@pytest.mark.parametrize("kind", KINDS)
def test_python_statement_of_the_decode(oracle, kind):
    """unpack + np.repeat gives the oracle's BWT back from its packed items, for every generator."""
    t = oracle.gen(kind, 7, 100_003)
    bwt, _ = oracle.bwt_forward(t)
    dist, init, _, _ = oracle.dc_encode(bwt)
    stream = dc_pack_ref.pack(*oracle.dc_stream(bwt, dist, init))
    assert np.array_equal(decode_py(stream, t.size), bwt)


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch as t
    if not t.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback)")
    return t


@pytest.fixture
def con(torch):  # per test: test_top_of_the_range needs the card to itself
    from dark_b200 import saca
    c = saca.Constructor(CAP)
    yield c
    c.close()


def header_of(info):
    return ([int(x) for x in info.init], bytes(info.mtf_symbols), int(info.num_unique), int(info.num_items))


def encode_device(con, torch, block):
    """(stream, DcInfo) of a block through dark_bwt_dc_encode_packed_device."""
    n = block.size
    d_in = torch.from_numpy(block).cuda()
    d_stream = torch.empty(8 * n, dtype=torch.uint8, device="cuda")
    nb, info = con.dc_encode_packed_device(d_in.data_ptr(), n, d_stream.data_ptr(), 8 * n)
    return d_stream[:nb].cpu().numpy(), info


def decode_device(con, torch, stream, n, offset=0):
    """dark_bwt_dc_decode_packed_device of a host stream placed at `offset` bytes into an allocation, into an output at the
    same offset: (block, DcInfo)."""
    d_buf = torch.zeros(stream.size + 32, dtype=torch.uint8, device="cuda")
    d_buf[offset:offset + stream.size] = torch.from_numpy(stream).cuda()
    d_out = torch.full((n + 32,), 0xA5, dtype=torch.uint8, device="cuda")
    info = con.dc_decode_packed_device(d_buf.data_ptr() + offset, stream.size, n, d_out.data_ptr() + offset)
    out = d_out.cpu().numpy()
    assert (out[:offset] == 0xA5).all() and (out[offset + n:] == 0xA5).all(), "written outside [0, n)"
    return out[offset:offset + n], info


def device_round_trip(con, torch, block, offsets=(0,)):
    stream, info = encode_device(con, torch, block)
    for off in offsets:
        got, dinfo = decode_device(con, torch, stream, block.size, off)
        assert np.array_equal(got, block), off
        assert header_of(dinfo) == header_of(info) and dinfo.device_ms > 0, off
    return stream


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_round_trips(con, torch, kind):
    """forward_dc_packed -> inverse_dc_packed gives the text back; the BWT and the header are the encoder's; the device form
    decodes the same stream at byte offsets 0..15."""
    from dark_b200 import synth
    for n in (2, 3, 300_007, 768 * 1024, 16 << 20, 256 << 20):
        t = synth.generate(kind, 11, n)
        bwt, origin, stream, info = con.bwt_dc_packed(t, want_bwt=True)
        text, b, dinfo = con.inverse_dc_packed(stream, n, origin, want_bwt=True)
        assert np.array_equal(text, t) and np.array_equal(b, bwt), (kind, n)
        assert header_of(dinfo) == header_of(info) and dinfo.device_ms > 0, (kind, n)
        text2, none, _ = con.inverse_dc_packed(stream, n, origin)
        assert none is None and np.array_equal(text2, t), (kind, n)
        if n <= 300_007:
            for off in range(16):
                got, oinfo = decode_device(con, torch, stream, n, off)
                assert np.array_equal(got, bwt) and header_of(oinfo) == header_of(info), (kind, n, off)
        del t, bwt, stream, text, b, text2


@pytest.mark.gpu
def test_one_byte_block(con, torch):
    block = np.array([7], np.uint8)
    stream = device_round_trip(con, torch, block, offsets=range(16))
    text, b, _ = con.inverse_dc_packed(stream, 1, 0, want_bwt=True)
    assert text.tolist() == [7] and b.tolist() == [7]


@pytest.mark.gpu
def test_alphabet_widths(con, torch):
    for sigma in DC_SIGMAS:
        for n in (4095, 70_001):
            device_round_trip(con, torch, dc_runs(alphabet(sigma, sigma), n, n + sigma))


@pytest.mark.gpu
def test_one_run_at_every_varint_width(con, torch):
    """A block of one run: length - 1 takes 1, 2, 3, 4 and 5 bytes of varint."""
    for n in (1, 128, 129, (1 << 14) + 1, (1 << 21) + 1, (1 << 28) + 1):
        block = np.full(n, 0x3C, np.uint8)
        stream = device_round_trip(con, torch, block)
        assert stream.size == 2 + len(varint(n - 1)) + 1, n


@pytest.mark.gpu
def test_alternating_bytes(con, torch):
    block = np.tile(np.array([1, 2], np.uint8), 150_001)
    stream = device_round_trip(con, torch, block)
    assert dc_pack_ref.unpack(stream)[0].size == block.size


def random_runs(seed, n):
    """A block of n bytes in runs of 1..300 bytes (varints of 1 and 2 bytes), adjacent runs of different symbols."""
    rng = np.random.default_rng(seed)
    lens = np.minimum(rng.geometric(rng.choice([0.5, 0.05, 0.005]), n), 300)
    lens = lens[:np.searchsorted(np.cumsum(lens), n) + 1]
    lens[-1] -= lens.sum() - n
    syms = rng.integers(0, 255, lens.size)
    syms = np.cumsum(syms + 1) % 256  # consecutive symbols differ
    return np.repeat(syms.astype(np.uint8), lens)


def item_edges(stream):
    """Offsets of every item's first byte and every varint's last byte."""
    firsts, lasts, p = [], [], 0
    while p < stream.size:
        firsts.append(p)
        p += 2
        for _ in range(2):
            while stream[p] & 0x80:
                p += 1
            lasts.append(p)
            p += 1
    return np.array(firsts), np.array(lasts)


@pytest.mark.gpu
def test_items_and_varints_around_tile_edges(con, torch):
    """Blocks whose streams put an item's first byte, and a varint's last byte, at every offset within 12 bytes of the
    parse's first two tile edges."""
    want = set(range(TILE - 12, TILE + 12)) | set(range(2 * TILE - 12, 2 * TILE + 12))
    seen_first, seen_last = set(), set()
    for seed in range(400):
        block = random_runs(seed, 20_000 + seed)
        stream = device_round_trip(con, torch, block)
        f, last = item_edges(stream)
        seen_first |= want & set(f.tolist())
        seen_last |= want & set(last.tolist())
        if seen_first == want and seen_last == want:
            break
    assert seen_first == want and seen_last == want


@pytest.mark.gpu
def test_top_of_the_range():
    """The DNA block of 2^32 - 2 bytes: forward_dc_packed -> inverse_dc_packed on one context (a 12.9 GB stream), text and
    BWT CRCs of tests/golden/large_golden.json."""
    import gc
    import torch
    from dark_b200 import saca, synth
    top = (1 << 32) - 2
    with open(os.path.join(ROOT, "tests", "golden", "large_golden.json")) as f:
        g = json.load(f)["dna:1:%d" % top]
    t = synth.generate("dna", 1, top)
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    con = saca.Constructor(top)
    try:
        _, origin, stream, info = con.bwt_dc_packed(t)
        del t
        assert origin == g["origin"] and stream.size > 1 << 33
        text, bwt, dinfo = con.inverse_dc_packed(stream, top, origin, want_bwt=True)
    finally:
        con.close()
    del stream
    assert header_of(dinfo) == header_of(info)
    assert "%08x" % crc(text) == g["text_crc32"] and "%08x" % crc(bwt) == g["bwt_crc32"]


def crc(a):
    c = 0
    for i in range(0, a.size, 1 << 30):
        c = zlib.crc32(memoryview(a[i:i + (1 << 30)]), c)
    return c


# ---- rejections -----------------------------------------------------------------------------------------------------
def refused(con, stream, n, origin, nbytes=None):
    """dark_bwt_inverse_dc_packed on sentinel outputs: the code, and whether both outputs are untouched."""
    from dark_b200 import _ffi
    s = np.ascontiguousarray(stream, np.uint8)
    text, bwt = np.full(n, 0xA5, np.uint8), np.full(n, 0x5A, np.uint8)
    rc = con._L.dark_bwt_inverse_dc_packed(con._ctx, s.ctypes.data, s.size if nbytes is None else nbytes, n, origin,
                                           text.ctypes.data, bwt.ctypes.data, ctypes.byref(_ffi.DcInfo()))
    return rc, bool((text == 0xA5).all() and (bwt == 0x5A).all())


@pytest.fixture
def small(con):
    """A text block whose packed stream is about 1 KB, its BWT, origin and stream."""
    from dark_b200 import synth
    t = synth.generate("text", 5, 400)
    bwt, origin, stream, info = con.bwt_dc_packed(t, want_bwt=True)
    assert 600 < stream.size < 2000
    return t, bwt, origin, stream


def assert_refused(con, small, stream, origin=None, nbytes=None, n=None):
    from dark_b200 import _ffi
    t, bwt, o, good = small
    rc, clean = refused(con, stream, t.size if n is None else n, o if origin is None else origin, nbytes)
    assert rc == _ffi.E_INVALID_ARG and clean
    assert np.array_equal(con.inverse_dc_packed(good, t.size, o)[0], t)  # the context is usable


def repacked(stream, edit):
    pos, dist, sym, rank = [a.copy() for a in dc_pack_ref.unpack(stream)]
    edit(pos, dist, sym, rank)
    return dc_pack_ref.pack(pos, dist, sym, rank)


@pytest.mark.gpu
def test_every_truncation_and_a_trailing_byte(con, small):
    t, bwt, origin, stream = small
    for k in range(1, stream.size):
        assert_refused(con, small, stream[:k])
    assert_refused(con, small, np.append(stream, 0))


@pytest.mark.gpu
def test_run_lengths_off_by_one(con, small):
    t, bwt, origin, stream = small
    runs = np.diff(dc_pack_ref.unpack(stream)[0].astype(np.int64), prepend=-1)
    k = int(np.flatnonzero(runs >= 2)[0])

    def shorter(pos, dist, sym, rank):
        pos[k:] -= 1

    def longer(pos, dist, sym, rank):
        pos[k:] += 1
    assert_refused(con, small, repacked(stream, shorter))
    assert_refused(con, small, repacked(stream, longer))


@pytest.mark.gpu
def test_malformed_and_non_canonical_varints(con, small):
    t, bwt, origin, stream = small
    v = int(dc_pack_ref.unpack(stream)[0][0])  # the first run's length - 1
    first = varint(v)
    rest = stream[2 + len(first):]
    six = [(v & 0x7F) | 0x80, 0x80 | (v >> 7), 0x80, 0x80, 0x80, 0x00]
    assert_refused(con, small, np.concatenate([stream[:2], np.array(six, np.uint8), rest]))
    long_form = [b | 0x80 for b in first] + [0x00]
    assert_refused(con, small, np.concatenate([stream[:2], np.array(long_form, np.uint8), rest]))
    assert_refused(con, small, np.concatenate([stream[:2], np.array([0xFF] * 4 + [0x10], np.uint8), rest]))  # above 2^32 - 1


@pytest.mark.gpu
def test_equal_symbols_and_changed_distances_or_ranks(con, small):
    t, bwt, origin, stream = small

    def same_sym(pos, dist, sym, rank):
        sym[1] = sym[0]
    assert_refused(con, small, repacked(stream, same_sym))
    for k in (0, 7, 40):
        for d in (-1, 1):
            def dist_edit(pos, dist, sym, rank):
                dist[k] = int(dist[k]) + d if int(dist[k]) + d >= 0 else int(dist[k]) + 1

            def rank_edit(pos, dist, sym, rank):
                rank[k] = (int(rank[k]) + d) % 256
            assert_refused(con, small, repacked(stream, dist_edit))
            assert_refused(con, small, repacked(stream, rank_edit))


@pytest.mark.gpu
def test_bad_sizes_and_origin(con, small):
    from dark_b200 import _ffi
    t, bwt, origin, stream = small
    n = t.size
    big = np.concatenate([stream, np.zeros(8 * n, np.uint8)])
    assert refused(con, big, n, origin, nbytes=8 * n + 1) == (_ffi.E_INVALID_ARG, True)
    assert refused(con, stream, n, origin, nbytes=0) == (_ffi.E_INVALID_ARG, True)
    assert refused(con, stream, n, n) == (_ffi.E_INVALID_ARG, True)
    one = np.zeros(1, np.uint8)
    assert con._L.dark_bwt_inverse_dc_packed(con._ctx, stream.ctypes.data, stream.size, CAP + 1, 0, one.ctypes.data, None,
                                             None) == _ffi.E_INVALID_N
    assert np.array_equal(con.inverse_dc_packed(stream, n, origin)[0], t)


@pytest.mark.gpu
def test_valid_stream_of_a_block_that_is_not_a_bwt(con, small, torch):
    from dark_b200 import DarkBwtError
    rng = np.random.default_rng(9)
    for _ in range(100):
        block = rng.integers(0, 4, 1000).astype(np.uint8)
        try:
            con.inverse(block, 0)
        except DarkBwtError:
            break
    else:
        pytest.fail("no block the inverse refuses")
    stream, _ = encode_device(con, torch, block)
    assert_refused(con, small, stream, origin=0, n=block.size)


@pytest.mark.gpu
def test_random_byte_flips(con, small, torch):
    """A flipped byte is refused, or the stream decodes to a block whose own stream it is."""
    from dark_b200 import DarkBwtError, _ffi
    t, bwt, origin, stream = small
    rng = np.random.default_rng(17)
    accepted = 0
    for _ in range(2000):
        s = stream.copy()
        k = int(rng.integers(0, s.size))
        s[k] = (int(s[k]) + int(rng.integers(1, 256))) % 256
        try:
            got, _ = decode_device(con, torch, s, t.size)
        except DarkBwtError as e:
            assert e.code == _ffi.E_INVALID_ARG
            continue
        accepted += 1
        assert np.array_equal(encode_device(con, torch, got)[0], s)
    assert np.array_equal(con.inverse_dc_packed(stream, t.size, origin)[0], t)
    print("accepted flips:", accepted)


# ---- host buffers, context ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("threads", ["0", "3", None])
def test_pinned_and_pageable_buffers(threads):
    code = (
        "import ctypes, numpy as np, torch\n"
        "from dark_b200 import saca, synth, _ffi\n"
        "t = synth.generate('mixed', 31, 3 * (1 << 20) + 12345)\n"
        "n = t.size\n"
        "with saca.Constructor(n) as c:\n"
        "    bwt, origin, stream, info = c.bwt_dc_packed(t, want_bwt=True)\n"
        "    assert stream.size >= 1 << 20\n"
        "    text, b, _ = c.inverse_dc_packed(stream, n, origin, want_bwt=True)\n"
        "    assert np.array_equal(text, t) and np.array_equal(b, bwt)\n"
        "    ps = torch.from_numpy(stream).pin_memory()\n"
        "    pt, pb = torch.zeros(n, dtype=torch.uint8).pin_memory(), torch.zeros(n, dtype=torch.uint8).pin_memory()\n"
        "    _ffi.check(c._L.dark_bwt_inverse_dc_packed(c._ctx, ps.data_ptr(), stream.size, n, origin, pt.data_ptr(), pb.data_ptr(),\n"
        "                                              ctypes.byref(_ffi.DcInfo())), c._ctx, 'pinned')\n"
        "    assert np.array_equal(pt.numpy(), t) and np.array_equal(pb.numpy(), bwt)\n"
        "print('ok')\n")
    env = dict(os.environ)
    env.pop("DARK_BWT_HOST_THREADS", None)
    if threads is not None:
        env["DARK_BWT_HOST_THREADS"] = threads
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


@pytest.mark.gpu
def test_device_only_context(con, torch):
    from dark_b200 import _ffi, saca, synth
    t = synth.generate("dna", 3, 100_000)
    bwt, origin, stream, info = con.bwt_dc_packed(t, want_bwt=True)
    with saca.Constructor(t.size, flags=_ffi.F_DEVICE_ONLY) as dev:
        with pytest.raises(_ffi.DarkBwtError) as e:
            dev.inverse_dc_packed(stream, t.size, origin)
        assert e.value.code == _ffi.E_INVALID_ARG
        got, dinfo = decode_device(dev, torch, stream, t.size)
        assert np.array_equal(got, bwt) and header_of(dinfo) == header_of(info)


@pytest.mark.gpu
def test_decode_between_two_forward_calls(torch):
    """A decode on the context between two forward_dc_packed calls leaves their results unchanged (blocks of 64 KiB or
    less borrow the sort's status buffer for DC)."""
    from dark_b200 import saca, synth
    blocks = [synth.generate("text", 8, 50_000), synth.generate("mixed", 9, 65_536), synth.generate("dna", 10, 2_000_000)]
    with saca.Constructor(2_000_000) as ref:
        want = [ref.bwt_dc_packed(t, want_bwt=True) for t in blocks]
    with saca.Constructor(2_000_000) as c:
        for k, t in enumerate(blocks):
            other = blocks[(k + 1) % len(blocks)]
            o_bwt, o_origin, o_stream, _ = want[(k + 1) % len(blocks)]
            b, o, s, i = c.bwt_dc_packed(t, want_bwt=True)
            assert o == want[k][1] and np.array_equal(b, want[k][0]) and np.array_equal(s, want[k][2]), k
            text, _, _ = c.inverse_dc_packed(o_stream, other.size, o_origin)
            assert np.array_equal(text, other), k
            b, o, s, i = c.bwt_dc_packed(t, want_bwt=True)
            assert o == want[k][1] and np.array_equal(b, want[k][0]) and np.array_equal(s, want[k][2]), k
            assert header_of(i) == header_of(want[k][3]), k
