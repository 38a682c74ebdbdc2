"""Blocks above 2^31 bytes, up to the 2^32 - 2 the reference accepts (Suffix = u32), on one B200.

Above 2^31 the forward has no bit-31 tag in isa[] (every round builds its keys by gather), the radix passes use
64-bit tile status words, and a default-flag context keeps one host-entry staging pair (include/dark_bwt.h).  Each
large test closes its context and empties torch's cache first: the arenas nearly fill the card.  A create that
fails for lack of memory fails the test with the free and needed bytes."""
import json
import os
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOP = (1 << 32) - 2


def crc(a):
    c = 0
    a = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    for i in range(0, a.size, 1 << 30):
        c = zlib.crc32(memoryview(a[i:i + (1 << 30)]), c)
    return "%08x" % c


@pytest.fixture(scope="module")
def torch():
    import torch as t
    if not t.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU fallback for the forward BWT)")
    return t


@pytest.fixture(scope="module")
def saca():
    from dark_b200 import saca as s
    return s


def create(saca, torch, n, flags=0):
    """A context of capacity n on an otherwise empty card (as far as this process goes)."""
    import gc
    from dark_b200 import _ffi
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free, total = torch.cuda.mem_get_info()
    need = saca.arena_bytes(n, flags)
    try:
        return saca.Constructor(n, flags=flags)
    except _ffi.DarkBwtError as e:
        pytest.fail(f"create({n}, flags={flags}) needs {need} bytes, {free} of {total} free: {e}")


@pytest.fixture(scope="module")
def golden():
    """The oracle's records of the blocks above 2^31 (tests/golden/make_large_golden.py)."""
    with open(os.path.join(ROOT, "tests", "golden", "large_golden.json")) as f:
        return json.load(f)


def block(key):
    from dark_b200 import synth
    kind, seed, n = key.split(":")
    return synth.generate(kind, int(seed), int(n))


def test_device_resident_2_5_gib(saca, golden, torch):
    """mixed:4 of 2.5 GiB through dark_bwt_forward_device on a device-only context: the gather key build, 64-bit status
    words and the suffix array checked by the O(n) verifier and against the oracle."""
    from dark_b200 import _ffi
    key = "mixed:4:2684354560"
    t = block(key)
    n = t.size
    con = create(saca, torch, n, _ffi.F_DEVICE_ONLY)
    try:
        dt = torch.from_numpy(t).cuda()
        db = torch.empty(n, dtype=torch.uint8, device="cuda")
        ds = torch.empty(n, dtype=torch.int32, device="cuda")
        origin = con.bwt_device(dt.data_ptr(), n, db.data_ptr(), ds.data_ptr())
        bad = con.verify_sa_device(dt.data_ptr(), n, ds.data_ptr())
        got = {"text_crc32": crc(t), "origin": origin, "bwt_crc32": crc(db.cpu().numpy()), "sa_crc32": crc(ds.cpu().numpy())}
        del dt, db, ds
    finally:
        con.close()
    print(key, got)
    assert bad == 0
    g = golden[key]
    assert got == {k: g[k] for k in got}


@pytest.mark.parametrize("key", ["dna:1:%d" % TOP, "mixed:4:%d" % TOP])
def test_host_entry_at_the_top_of_the_range(saca, golden, torch, key):
    """2^32 - 2 bytes through the host entry on a default (one staging pair) context, then the inverse on the same
    context restores the text.  Row ids of the inverse reach 2^32 - 2, one below its nil sentinel."""
    t = block(key)
    con = create(saca, torch, TOP)
    try:
        bwt, origin = con.bwt(t)
        back = con.inverse(bwt, origin)
    finally:
        con.close()
    got = {"text_crc32": crc(t), "origin": origin, "bwt_crc32": crc(bwt)}
    print(key, got)
    assert np.array_equal(back, t)
    g = golden[key]
    assert got == {k: g[k] for k in got}


def test_distance_coding_at_the_top_of_the_range(saca, torch):
    """dark_bwt_forward_dc of the DNA block of 2^32 - 2 bytes: every output equals the oracle's distance coding of the
    oracle's BWT (tests/golden/large_dc.json), over 2^20-byte chunks whose tables and records are all in play."""
    t = block("dna:1:%d" % TOP)
    con = create(saca, torch, t.size)
    try:
        bwt, origin, dc = con.bwt_dc(t)
    finally:
        con.close()
    del t
    got = {"bwt_crc32": crc(bwt), "num_unique": dc["num_unique"], "num_items": dc["num_items"],
           **{name + "_crc32": crc(dc[name]) for name in ("dist", "item_pos", "item_dist", "item_sym", "item_rank")}}
    print(got)
    with open(os.path.join(ROOT, "tests", "golden", "large_dc.json")) as f:
        g = json.load(f)
    assert g["block"] == "dna:1:%d" % TOP
    assert got == {k: g[k] for k in got}
    assert dc["num_unique"] == g["num_unique"] and dc["num_items"] == g["num_items"]
    assert [int(x) for x in dc["init"]] == g["init"]
    nu = g["num_unique"]   # the MTF list is defined for the symbols that occur
    assert [int(x) for x in dc["mtf_symbols"][:nu]] == g["mtf_symbols"][:nu]


MANY = [("mixed", 31, 560000001), ("dna", 32, 536870912), ("rep17", 33, 500000000), ("text", 34, 530000017),
        ("mixed", 35, 511111111)]   # sum 2,637,981,141 > 2^31


def test_many_blocks_beyond_2_31(saca, torch):
    """forward_many, inverse_many and dc_encode_many with the blocks summing past 2^31 on a 2.5 GiB context: each block
    equals the single call on the same context."""
    from dark_b200 import synth
    blocks = [synth.generate(k, s, n) for k, s, n in MANY]
    assert sum(b.size for b in blocks) > 1 << 31
    con = create(saca, torch, 5 << 29)
    try:
        many = con.bwt_many(blocks)
        singles = [con.bwt(b) for b in blocks]
        for (bm, om), (bs, os_) in zip(many, singles):
            assert om == os_
            assert np.array_equal(bm, bs)
        texts = con.inverse_many([(b, o) for b, o in singles])
        for t, b in zip(texts, blocks):
            assert np.array_equal(t, b)
        dcs = con.dc_encode_many([b for b, _ in singles], want_dist=True)
        for d, (b, _) in zip(dcs, singles):
            s = con.dc_encode(b)
            assert d["num_items"] == s["num_items"] and d["num_unique"] == s["num_unique"]
            assert np.array_equal(d["init"], s["init"]) and np.array_equal(d["mtf_symbols"], s["mtf_symbols"])
            for name in ("dist", "item_pos", "item_dist", "item_sym", "item_rank"):
                assert np.array_equal(d[name], s[name]), name
    finally:
        con.close()


def test_batches_on_a_one_pair_context(saca, torch):
    """forward_batch and inverse_batch on a context above 2^31 (one staging pair: blocks run one after another) give
    what the single calls give, for pinned and pageable buffers."""
    from dark_b200 import synth
    blocks = [synth.generate(k, 40 + i, n) for i, (k, n) in
              enumerate([("mixed", 3 << 20), ("dna", 1 << 16), ("text", 5 << 20), ("rep17", 2 << 20), ("mixed", 77)])]
    pinned = [torch.from_numpy(b).pin_memory().numpy() for b in blocks]
    con = create(saca, torch, (1 << 31) + (1 << 20))
    try:
        singles = [con.bwt(b) for b in blocks]
        for src in (blocks, pinned):
            got = con.bwt_blocks(src)
            for (bb, ob), (bs, os_) in zip(got, singles):
                assert ob == os_ and np.array_equal(bb, bs)
        texts = con.inverse_blocks(singles)
        for t, b in zip(texts, blocks):
            assert np.array_equal(t, b)
        for t, (b, o) in zip(texts, singles):
            assert np.array_equal(con.inverse(b, o), t)
    finally:
        con.close()
