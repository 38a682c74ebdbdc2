"""Distance coding of many small blocks in one pass: dark_bwt_dc_encode_many / _many_device and the fused
dark_bwt_forward_dc_many.  Every block is compared with the CPU oracle's dc_encode / dc_stream (and decoded back), and
with a single dark_bwt_dc_encode call on that block alone."""
import ctypes
import os

import numpy as np
import pytest

NEW_SYMBOLS = ["dark_bwt_dc_encode_many", "dark_bwt_dc_encode_many_device", "dark_bwt_forward_dc_many"]
MAX_MANY = 65536  # DARK_BWT_MAX_MANY_BLOCKS
RECORD = 1288     # bytes per block staged on the device: count * RECORD <= 8 * capacity + 1024
FIELDS = ("dist", "init", "mtf_symbols", "num_unique", "num_items", "item_pos", "item_dist", "item_sym", "item_rank")


def max_blocks(capacity):
    return (8 * capacity + 1024) // RECORD


# ---- CPU: exports and argument checks (no device work) ---------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from dark_b200 import _ffi
    if not os.path.exists(_ffi.lib_path()):
        _ffi.build_native()
    return _ffi.lib()


def test_new_symbols_are_exported(lib):
    from dark_b200 import _ffi
    for name in NEW_SYMBOLS:
        assert name in _ffi.SYMBOLS
        assert hasattr(lib, name), name


def test_bad_arguments_are_rejected_before_any_device_work(lib):
    """Null context or required pointers give DARK_BWT_E_INVALID_ARG without touching CUDA, whatever the count."""
    from dark_b200 import _ffi
    p = (ctypes.c_void_p * 1)(1)
    ns = (ctypes.c_uint64 * 1)(10)
    info = (_ffi.DcInfo * 1)()
    for count in (0, 1, 3, MAX_MANY + 1):
        assert lib.dark_bwt_dc_encode_many(None, None, None, count, *([None] * 6), None, None) == _ffi.E_INVALID_ARG
        assert lib.dark_bwt_dc_encode_many(None, p, ns, count, *([None] * 6), info, None) == _ffi.E_INVALID_ARG
        assert lib.dark_bwt_dc_encode_many_device(None, None, None, count, *([None] * 6), None, None) == _ffi.E_INVALID_ARG
        assert lib.dark_bwt_dc_encode_many_device(None, 1, 1, count, *([None] * 6), info, None) == _ffi.E_INVALID_ARG
        assert lib.dark_bwt_forward_dc_many(None, None, None, count, None, None, *([None] * 6), None, None) == _ffi.E_INVALID_ARG
        origins = (ctypes.c_uint64 * 1)()
        assert lib.dark_bwt_forward_dc_many(None, p, ns, count, None, origins, *([None] * 6), info, None) == _ffi.E_INVALID_ARG


# ---- GPU ----------------------------------------------------------------------------------------------
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


def check_against_oracle(res, b, oracle):
    n = b.size
    dist, init, mtf, nu = oracle.dc_encode(b)
    pos, sd, sym, rk = oracle.dc_stream(b, dist, init)
    assert res["num_unique"] == nu and res["num_items"] == pos.size
    assert np.array_equal(res["init"], init)
    assert np.array_equal(res["mtf_symbols"][:nu], mtf[:nu])
    if res["dist"] is not None:
        assert np.array_equal(res["dist"], dist)
    assert np.array_equal(res["item_pos"], pos) and np.array_equal(res["item_dist"], sd)
    assert np.array_equal(res["item_sym"], sym) and np.array_equal(res["item_rank"], rk)
    assert np.array_equal(oracle.dc_decode(res["init"], res["item_dist"], n), b)


def same_result(a, b, fields=FIELDS):
    for f in fields:
        if a[f] is None or b[f] is None:
            continue
        assert np.array_equal(np.asarray(a[f]), np.asarray(b[f])), f


def check_many(saca, oracle, blocks, single_every=1):
    """dc_encode_many of `blocks` equals the oracle on every block and a single dc_encode call on every single_every-th."""
    bs = [as_u8(b) for b in blocks]
    total = sum(b.size for b in bs)
    cap = max(total, (len(bs) * RECORD - 1024 + 7) // 8, 2)
    with saca.Constructor(cap) as con:
        res = con.dc_encode_many(bs)
        assert len(res) == len(bs)
        for k, (b, r) in enumerate(zip(bs, res)):
            check_against_oracle(r, b, oracle)
            if k % single_every == 0:
                same_result(r, con.dc_encode(b))
            assert r["device_ms"] == res[0]["device_ms"] > 0
    return res


def block_sets():
    rng = np.random.default_rng(29)
    from dark_b200 import synth

    def runs(sigma, n, seed, lo=0):
        r = np.random.default_rng(seed)
        return (np.repeat(r.integers(0, sigma, n), r.integers(1, 9, n))[:n] + lo).astype(np.uint8)

    text = synth.generate("text", 3, 300_000)
    return {
        "one_byte_blocks_256": [bytes([int(c)]) for c in rng.integers(0, 256, 3000)],
        "one_byte_blocks_small": [bytes([int(c)]) for c in rng.integers(97, 100, 5000)],
        "on_chunk_boundaries": [runs(4, s, 10 + i) for i, s in enumerate((4096, 4096, 8192, 1, 4095, 1, 4096, 12288, 4097, 4095))],
        "straddling_chunks": [runs(26, s, 20 + i, 97) for i, s in enumerate((3000, 5000, 7001, 2, 9999, 4100, 123, 6000))],
        "many_in_one_chunk": [runs(3, int(s), 30 + i, 65) for i, s in enumerate(rng.integers(1, 17, 700))],
        "longer_than_a_scan_group": [runs(4, 100, 40), runs(4, (1 << 20) + 5000, 41, 65), runs(256, 3000, 42),
                                     runs(200, (1 << 21) + 17, 43)],
        "equal_bytes_across_boundaries": [b"aaaa", b"aaaa", b"a", b"ab", b"ba", b"aaaa", b"b", b"bbbb", b"\x00" * 5000, b"\x00" * 3],
        "identical_blocks": [text[:9973].tobytes()] * 9 + [b"rdarcaaaabb"] * 3,
        "union_le_32_dna": [runs(4, int(s), 50 + i, 65) for i, s in enumerate(rng.integers(1, 30_000, 40))],
        "union_256": [rng.integers(0, 256, int(s)).astype(np.uint8) for s in rng.integers(1, 20_000, 40)],
        "small_among_256": [rng.integers(0, 256, 5000).astype(np.uint8), runs(2, 4000, 60, 120), rng.integers(0, 256, 300).astype(np.uint8),
                            b"\x07" * 100, rng.integers(0, 256, 9000).astype(np.uint8), runs(3, 4096, 61, 1)],
        "text_slices": [text[i:i + 7919] for i in range(0, 290_000, 7919)],
    }


@pytest.mark.gpu
def test_dc_many_known_blocks(saca, oracle, torch):
    res = check_many(saca, oracle, [b"rdarcaaaabb", b"nnbaaa", b"z"])
    assert [r["num_items"] for r in res] == [7, 3, 1]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["one_byte_blocks_256", "one_byte_blocks_small", "on_chunk_boundaries", "straddling_chunks",
                                  "many_in_one_chunk", "longer_than_a_scan_group", "equal_bytes_across_boundaries",
                                  "identical_blocks", "union_le_32_dna", "union_256", "small_among_256", "text_slices"])
def test_dc_many_block_sets(saca, oracle, torch, name):
    check_many(saca, oracle, block_sets()[name])


@pytest.mark.gpu
def test_dc_many_max_blocks(saca, oracle, torch):
    """DARK_BWT_MAX_MANY_BLOCKS blocks of 1 to 4 bytes: the oracle on every block, a single call on every 251st."""
    rng = np.random.default_rng(31)
    blocks = [rng.integers(0, 3, int(s)).astype(np.uint8) for s in rng.integers(1, 5, MAX_MANY)]
    check_many(saca, oracle, blocks, single_every=251)


@pytest.mark.gpu
def test_dc_many_record_bound(saca, oracle, torch):
    """count * 1288 <= 8 * capacity + 1024: exactly at the bound passes, one block more is DARK_BWT_E_INVALID_N."""
    from dark_b200 import _ffi
    cap = 15_972  # 8 * cap + 1024 = 100 records
    assert max_blocks(cap) == 100 and max_blocks(cap - 1) == 99
    rng = np.random.default_rng(37)
    blocks = [rng.integers(0, 5, 150).astype(np.uint8) for _ in range(100)]
    with saca.Constructor(cap) as con:
        for b, r in zip(blocks, con.dc_encode_many(blocks)):
            check_against_oracle(r, b, oracle)
        for call in (lambda: con.dc_encode_many(blocks + [b"x"]), lambda: con.bwt_dc_many(blocks + [b"xy"])):
            with pytest.raises(_ffi.DarkBwtError) as e:
                call()
            assert e.value.code == _ffi.E_INVALID_N
        for t, (b, o, r) in zip(blocks, con.bwt_dc_many(blocks)):
            bwt_o, origin_o = oracle.bwt_forward(t)
            assert o == origin_o and np.array_equal(b, bwt_o)
            check_against_oracle(r, bwt_o, oracle)


def fused_blocks():
    from dark_b200 import synth
    rng = np.random.default_rng(41)
    blocks = [synth.generate("text", 3, 768_771), synth.generate("dna", 5, 300_007), synth.generate("mixed", 6, 200_003),
              synth.generate("rep17", 7, 100_001)]
    blocks += [synth.generate(("text", "dna", "mixed", "rep17")[k % 4], 100 + k, int(s)) for k, s in enumerate(rng.integers(2, 20_000, 28))]
    blocks += [np.array([9, 9], np.uint8), np.array([9, 9], np.uint8), np.array([1, 2], np.uint8)]
    return blocks


@pytest.mark.gpu
def test_forward_dc_many_equals_forward_dc(saca, oracle, torch):
    """BWT, origin and every DC output of each block equal a forward_dc call on that block, and the oracle."""
    texts = fused_blocks()
    with saca.Constructor(sum(t.size for t in texts)) as con:
        many = con.bwt_dc_many(texts)
        for k, (t, (bwt, origin, res)) in enumerate(zip(texts, many)):
            b1, o1, r1 = con.bwt_dc(t)
            assert origin == o1 and np.array_equal(bwt, b1), k
            same_result(res, r1)
            bwt_o, origin_o = oracle.bwt_forward(t)
            assert origin == origin_o and np.array_equal(bwt, bwt_o), k
            check_against_oracle(res, bwt_o, oracle)


@pytest.mark.gpu
def test_forward_dc_many_each_output_null(saca, oracle, torch):
    """Every nullable output left out in turn: the others are unchanged."""
    from dark_b200 import _ffi
    texts = fused_blocks()[4:]
    cnt, ns = len(texts), [t.size for t in texts]
    total = sum(ns)
    with saca.Constructor(total) as con:
        ref = con.bwt_dc_many(texts)
        L, ctx = con._L, con._ctx
        for skip in range(7):  # bwt_outs, dist, item_starts, item_pos, item_dist, item_sym, item_rank
            bwts = [np.zeros(n, np.uint8) for n in ns]
            arrays = [np.zeros(total, np.uint32), np.zeros(cnt + 1, np.uint32), np.zeros(total, np.uint32), np.zeros(total, np.uint32),
                      np.zeros(total, np.uint8), np.zeros(total, np.uint8)]
            ptrs = [a.ctypes.data for a in arrays]
            bp = (ctypes.c_void_p * cnt)(*[b.ctypes.data for b in bwts])
            if skip == 0:
                bp = None
            else:
                ptrs[skip - 1] = None
            infos = (_ffi.DcInfo * cnt)()
            origins = (ctypes.c_uint64 * cnt)()
            _ffi.check(L.dark_bwt_forward_dc_many(ctx, (ctypes.c_void_p * cnt)(*[t.ctypes.data for t in texts]), (ctypes.c_uint64 * cnt)(*ns),
                                                  cnt, bp, origins, *ptrs, infos, None), ctx, "forward_dc_many")
            dist, starts, pos, idist, sym, rank = arrays
            rs = np.concatenate([[0], np.cumsum([r["num_items"] for _, _, r in ref])])
            off = 0
            for k, (bwt, origin, r) in enumerate(ref):
                assert int(origins[k]) == origin and int(infos[k].num_items) == r["num_items"]
                assert np.array_equal(np.array(list(infos[k].init), np.uint64), r["init"])
                assert np.array_equal(np.array(list(infos[k].mtf_symbols), np.uint8), r["mtf_symbols"])
                if skip != 0:
                    assert np.array_equal(bwts[k], bwt)
                if skip != 1:
                    assert np.array_equal(dist[off:off + ns[k]], r["dist"])
                a, e = int(rs[k]), int(rs[k + 1])
                if skip != 2:
                    assert int(starts[k]) == a and int(starts[k + 1]) == e
                for j, (arr, f) in enumerate(((pos, "item_pos"), (idist, "item_dist"), (sym, "item_sym"), (rank, "item_rank"))):
                    if skip != 3 + j:
                        assert np.array_equal(arr[a:e], r[f]), (skip, f)
                off += ns[k]


@pytest.mark.gpu
def test_device_chain_forward_many_then_dc_many(saca, oracle, torch):
    """forward_many_device -> dc_encode_many_device on the same device buffers equals the host form on the BWTs."""
    from dark_b200 import _ffi, synth
    rng = np.random.default_rng(43)
    blocks = [synth.generate("text", 3 + 100 * k, int(s)) for k, s in enumerate(rng.integers(2, 40_000, 24))]
    blocks += [np.array([7, 7], np.uint8), synth.generate("dna", 9, 100_003), synth.generate("mixed", 10, 5000)]
    starts = np.concatenate([[0], np.cumsum([b.size for b in blocks])]).astype(np.uint32)
    n, cnt = int(starts[-1]), len(blocks)
    with saca.Constructor(n, flags=_ffi.F_DEVICE_ONLY) as con:
        dt = torch.from_numpy(np.concatenate(blocks)).cuda()
        ds = torch.from_numpy(starts.view(np.int32)).cuda()
        db = torch.empty(n, dtype=torch.uint8, device="cuda")
        do = torch.empty(cnt, dtype=torch.int64, device="cuda")
        con.bwt_many_device(dt.data_ptr(), ds.data_ptr(), cnt, db.data_ptr(), do.data_ptr())
        outs = [torch.full((n,), -1, dtype=torch.int32, device="cuda") for _ in range(2)] + \
            [torch.full((cnt + 1,), -1, dtype=torch.int32, device="cuda")] + [torch.zeros(n, dtype=torch.uint8, device="cuda") for _ in range(2)]
        dd, dsd, dst, dsym, drk = outs
        dpos = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        infos, ms = con.dc_encode_many_device(db.data_ptr(), ds.data_ptr(), cnt, dd.data_ptr(), dst.data_ptr(), dpos.data_ptr(),
                                              dsd.data_ptr(), dsym.data_ptr(), drk.data_ptr())
        assert ms > 0 and len(infos) == cnt
        hb = db.cpu().numpy()
        dist, its = dd.cpu().numpy().view(np.uint32), dst.cpu().numpy().view(np.uint32)
        pos, sd, sym, rk = dpos.cpu().numpy().view(np.uint32), dsd.cpu().numpy().view(np.uint32), dsym.cpu().numpy(), drk.cpu().numpy()
    bwts = [hb[int(starts[k]):int(starts[k + 1])] for k in range(cnt)]
    with saca.Constructor(n) as con:
        host = con.dc_encode_many(bwts)
    assert int(its[0]) == 0 and int(its[cnt]) == sum(r["num_items"] for r in host)
    for k in range(cnt):
        a, e = int(its[k]), int(its[k + 1])
        r = host[k]
        assert int(infos[k].num_items) == r["num_items"] == e - a
        assert np.array_equal(np.array(list(infos[k].init), np.uint64), r["init"])
        assert np.array_equal(dist[int(starts[k]):int(starts[k + 1])], r["dist"])
        for arr, f in ((pos, "item_pos"), (sd, "item_dist"), (sym, "item_sym"), (rk, "item_rank")):
            assert np.array_equal(arr[a:e], r[f]), (k, f)
        bwt_o, origin_o = oracle.bwt_forward(blocks[k])
        assert np.array_equal(bwts[k], bwt_o), k
        check_against_oracle(r, bwt_o, oracle)


@pytest.mark.gpu
def test_dc_many_rejects_bad_arguments(saca, oracle, torch):
    from dark_b200 import _ffi

    def code(call):
        with pytest.raises(_ffi.DarkBwtError) as e:
            call()
        return e.value.code

    with saca.Constructor(1000) as con:
        assert code(lambda: con.dc_encode_many([b"abc", b""])) == _ffi.E_INVALID_N            # an empty block
        assert code(lambda: con.bwt_dc_many([b"abc", b"a"])) == _ffi.E_INVALID_N              # the sort needs 2 bytes
        assert code(lambda: con.dc_encode_many([b"a" * 600, b"b" * 401])) == _ffi.E_INVALID_N  # sum(ns) > capacity
        assert code(lambda: con.bwt_dc_many([b"a" * 600, b"b" * 401])) == _ffi.E_INVALID_N
        assert con.dc_encode_many([]) == [] and con.bwt_dc_many([]) == []
        full = con.dc_encode_many([b"a" * 600, b"b" * 400])                                    # exactly full
        assert [r["num_items"] for r in full] == [1, 1]
        db = torch.frombuffer(bytearray(b"nnbaaaab"), dtype=torch.uint8).cuda()
        for starts, want in (([1, 8], _ffi.E_INVALID_ARG), ([0, 5, 3], _ffi.E_INVALID_N), ([0, 4, 4, 8], _ffi.E_INVALID_N),
                             ([0, 1001], _ffi.E_INVALID_N)):
            ds = torch.tensor(starts, dtype=torch.int32, device="cuda")
            assert code(lambda: con.dc_encode_many_device(db.data_ptr(), ds.data_ptr(), len(starts) - 1)) == want, starts
        ds = torch.tensor([0, 6, 8], dtype=torch.int32, device="cuda")
        infos, _ = con.dc_encode_many_device(db.data_ptr(), ds.data_ptr(), 2)
        assert [int(i.num_items) for i in infos] == [3, 2]
    with saca.Constructor(MAX_MANY * 200) as con:                                            # count > DARK_BWT_MAX_MANY_BLOCKS
        assert code(lambda: con.dc_encode_many([b"ab"] * (MAX_MANY + 1))) == _ffi.E_INVALID_ARG
        assert code(lambda: con.bwt_dc_many([b"ab"] * (MAX_MANY + 1))) == _ffi.E_INVALID_ARG
    with saca.Constructor(1000, flags=_ffi.F_DEVICE_ONLY) as con:                            # host forms need the staging buffers
        assert code(lambda: con.dc_encode_many([b"nnbaaa"])) == _ffi.E_INVALID_ARG
        assert code(lambda: con.bwt_dc_many([b"banana"])) == _ffi.E_INVALID_ARG


@pytest.mark.gpu
def test_dc_many_interleaved_on_one_context(saca, oracle, torch):
    """forward_dc, dc_encode_many (small total: borrows the sort's status buffer), forward, forward_dc_many and
    inverse_many on one context keep giving what a fresh context gives."""
    from dark_b200 import synth
    big = synth.generate("mixed", 70, 1 << 20)
    small = [synth.generate("text", 71 + k, 2000 + 37 * k) for k in range(12)]
    texts = [synth.generate("dna", 90, 300_000), synth.generate("text", 91, 200_000)] + small[:4]
    with saca.Constructor(1 << 21) as fresh:
        f_dc = fresh.bwt_dc(big)
    with saca.Constructor(1 << 21) as fresh:
        f_many = fresh.dc_encode_many(small)
    with saca.Constructor(1 << 21) as fresh:
        f_fwd = fresh.bwt(big)
    with saca.Constructor(1 << 21) as fresh:
        f_fdm = fresh.bwt_dc_many(texts)
    pairs = [(b, o) for b, o, _ in f_fdm]
    with saca.Constructor(1 << 21) as con:
        for _ in range(2):
            b, o, r = con.bwt_dc(big)
            assert o == f_dc[1] and np.array_equal(b, f_dc[0])
            same_result(r, f_dc[2])
            for r, f in zip(con.dc_encode_many(small), f_many):
                same_result(r, f)
            b, o = con.bwt(big)
            assert o == f_fwd[1] and np.array_equal(b, f_fwd[0])
            for (b, o, r), (fb, fo, fr) in zip(con.bwt_dc_many(texts), f_fdm):
                assert o == fo and np.array_equal(b, fb)
                same_result(r, fr)
            assert all(np.array_equal(x, t) for x, t in zip(con.inverse_many(pairs), texts))
    for t, (b, o, r) in zip(texts, f_fdm):
        bwt_o, origin_o = oracle.bwt_forward(t)
        assert o == origin_o and np.array_equal(b, bwt_o)
        check_against_oracle(r, bwt_o, oracle)
