"""The unpack side for many blocks: dark_bwt_inverse_many / _many_device (many small blocks in one device pass) and
dark_bwt_inverse_batch (host blocks pipelined like dark_bwt_forward_batch).  Every GPU result is compared bit-exactly
with the original text and with the CPU oracle's decode."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_SYMBOLS = ["dark_bwt_inverse_batch", "dark_bwt_inverse_many", "dark_bwt_inverse_many_device"]
MAX_MANY = 65536  # DARK_BWT_MAX_MANY_BLOCKS


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
    """Null pointers, and more than DARK_BWT_MAX_MANY_BLOCKS blocks, give DARK_BWT_E_INVALID_ARG without touching CUDA."""
    from dark_b200 import _ffi
    p = (ctypes.c_void_p * 1)(1)
    ns = (ctypes.c_uint64 * 1)(10)
    orgs = (ctypes.c_uint64 * 1)(0)
    for count in (1, 3, MAX_MANY + 1):
        assert lib.dark_bwt_inverse_many(None, None, None, None, None, count, None) == _ffi.E_INVALID_ARG
        assert lib.dark_bwt_inverse_many(None, p, ns, orgs, p, count, None) == _ffi.E_INVALID_ARG
        assert lib.dark_bwt_inverse_many_device(None, None, None, None, count, None, None) == _ffi.E_INVALID_ARG
        assert lib.dark_bwt_inverse_many_device(None, 1, 1, 1, count, 1, None) == _ffi.E_INVALID_ARG
        assert lib.dark_bwt_inverse_batch(None, None, None, None, None, count, None) == _ffi.E_INVALID_ARG
        assert lib.dark_bwt_inverse_batch(None, p, ns, orgs, p, count, None) == _ffi.E_INVALID_ARG


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


def fwd(oracle, blk):
    t = np.frombuffer(bytes(blk), dtype=np.uint8) if not isinstance(blk, np.ndarray) else blk
    if t.size < 2:
        return t.copy(), 0
    return oracle.bwt_forward(t)


def check_many(saca, oracle, blocks, capacity=None):
    """inverse_many of the oracle's forward transforms restores every block; equals the oracle's decode."""
    texts = [np.frombuffer(bytes(b), dtype=np.uint8) if not isinstance(b, np.ndarray) else b for b in blocks]
    pairs = [fwd(oracle, t) for t in texts]
    cap = capacity or max(sum(t.size for t in texts) + len(texts), 2)
    with saca.Constructor(cap) as con:
        outs = con.inverse_many(pairs)
        assert len(outs) == len(texts)
        for k, (t, (bwt, origin), out) in enumerate(zip(texts, pairs, outs)):
            assert np.array_equal(out, t), k
            assert np.array_equal(out, oracle.bwt_decode(bwt, origin)), k
    return pairs


def many_cases():
    rng = np.random.default_rng(17)
    from dark_b200 import synth
    text = synth.generate("text", 3, 200_000)
    return {
        "two_tiny": [b"abracadabra", b"banana"],
        "identical_blocks": [b"mississippi"] * 5 + [b"banana"] * 3,
        "prefix_blocks": [b"aaaa", b"aaaaaaaa", b"aa", b"aaab", b"baaa"],
        "minimal": [b"ab", b"ba", b"aa", b"\x00\x00", b"\xff\x00"],
        "binary_256": [rng.integers(0, 256, int(s)).astype(np.uint8).tobytes() for s in (300, 70_001, 2, 4096, 65_537)],
        "dna_ragged": [(rng.integers(0, 4, int(s)).astype(np.uint8) + 65).tobytes() for s in rng.integers(2, 50_000, 40)],
        "text_slices": [text[i:i + 9973].tobytes() for i in range(0, 190_000, 9973)],
        "periodic": [bytes(range(1, 18)) * 500, bytes(range(1, 18)) * 400 + b"x", b"\x07" * 30_000, b"\x07" * 29_999],
        "one_byte_blocks": [bytes([int(c)]) for c in rng.integers(0, 256, 300)] + [b"q"],
        "one_symbol_blocks": [b"z" * int(s) for s in rng.integers(1, 3000, 30)] + [b"\x00" * 5],
        "every_remainder": [rng.integers(0, 3, s).astype(np.uint8).tobytes() for s in range(1, 201)],
        "mixed_sizes": [b"x", b"xy"] + [rng.integers(0, 256, int(s)).astype(np.uint8).tobytes() for s in (1, 47, 48, 49, 95, 96, 97, 1)],
    }


@pytest.mark.gpu
def test_inverse_many_known_answers(saca, oracle, torch):
    # saca.rs:404-406 and 411-412: the KATs, decoded together
    with saca.Constructor(64) as con:
        outs = con.inverse_many([(b"rdarcaaaabb", 2), (b"nnbaaa", 3)])
    assert [o.tobytes() for o in outs] == [b"abracadabra", b"banana"]
    assert [oracle.bwt_decode(np.frombuffer(b, np.uint8), o).tobytes() for b, o in ((b"rdarcaaaabb", 2), (b"nnbaaa", 3))] == \
        [b"abracadabra", b"banana"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["two_tiny", "identical_blocks", "prefix_blocks", "minimal", "binary_256", "dna_ragged",
                                  "text_slices", "periodic", "one_byte_blocks", "one_symbol_blocks", "every_remainder",
                                  "mixed_sizes"])
def test_inverse_many_block_sets(saca, oracle, torch, name):
    check_many(saca, oracle, many_cases()[name])


@pytest.mark.gpu
def test_inverse_many_max_blocks_of_two_bytes(saca, oracle, torch):
    rng = np.random.default_rng(5)
    texts = [rng.integers(0, 4, 2).astype(np.uint8) for _ in range(MAX_MANY)]
    check_many(saca, oracle, texts)
    # one block too many is refused before any device work on the blocks
    from dark_b200 import _ffi
    with saca.Constructor(4 * (MAX_MANY + 1)) as con:
        with pytest.raises(_ffi.DarkBwtError) as e:
            con.inverse_many([(b"ab", 0)] * (MAX_MANY + 1))
        assert e.value.code == _ffi.E_INVALID_ARG


@pytest.mark.gpu
def test_inverse_many_single_block_equals_single_call(saca, oracle, torch):
    from dark_b200 import synth
    t = synth.generate("text", 3, 768771)
    bwt, origin = oracle.bwt_forward(t)
    with saca.Constructor(t.size + 1) as con:
        one = con.inverse(bwt, origin)
        (many,) = con.inverse_many([(bwt, origin)])
    assert np.array_equal(many, one) and np.array_equal(many, t)


@pytest.mark.gpu
def test_inverse_many_device_round_trip(saca, oracle, torch):
    """forward_many_device -> inverse_many_device on the same device buffers restores every block."""
    from dark_b200 import _ffi, synth
    rng = np.random.default_rng(23)
    blocks = [synth.generate("text", 3 + 100 * k, int(s)) for k, s in enumerate(rng.integers(2, 40_000, 24))]
    blocks += [np.array([7, 7], np.uint8), synth.generate("dna", 9, 100_003)]
    starts = np.concatenate([[0], np.cumsum([b.size for b in blocks])]).astype(np.uint32)
    n = int(starts[-1])
    with saca.Constructor(n + len(blocks), flags=_ffi.F_DEVICE_ONLY) as con:
        dt = torch.from_numpy(np.concatenate(blocks)).cuda()
        ds = torch.from_numpy(starts.view(np.int32)).cuda()
        db = torch.empty(n, dtype=torch.uint8, device="cuda")
        do = torch.empty(len(blocks), dtype=torch.int64, device="cuda")
        con.bwt_many_device(dt.data_ptr(), ds.data_ptr(), len(blocks), db.data_ptr(), do.data_ptr())
        dback = torch.zeros(n, dtype=torch.uint8, device="cuda")
        ms = con.inverse_many_device(db.data_ptr(), ds.data_ptr(), do.data_ptr(), len(blocks), dback.data_ptr())
        assert ms > 0
        assert torch.equal(dback, dt)
        hb, ho = db.cpu().numpy(), do.cpu().numpy()
    for k, blk in enumerate(blocks):
        a, e = int(starts[k]), int(starts[k + 1])
        assert np.array_equal(oracle.bwt_decode(hb[a:e], int(ho[k])), blk), k


@pytest.mark.gpu
def test_inverse_many_names_the_inconsistent_block(saca, oracle, torch):
    """A wrong origin inside a set: the call raises DarkBwtError naming that block, returns (no hang), and the context
    then inverts the corrected set."""
    from dark_b200 import DarkBwtError, synth
    texts = [synth.generate("text", 30 + k, 5000 + 777 * k) for k in range(8)]
    pairs = [oracle.bwt_forward(t) for t in texts]
    bad = 5
    with saca.Constructor(sum(t.size for t in texts) + len(texts)) as con:
        bwt, origin = pairs[bad]
        wrong = None
        for d in range(1, 200):  # an origin the single-block inverse rejects (some wrong origins decode to another text)
            cand = (origin + 97 * d) % bwt.size
            try:
                con.inverse(bwt, cand)
            except DarkBwtError:
                wrong = cand
                break
        assert wrong is not None
        broken = list(pairs)
        broken[bad] = (bwt, wrong)
        with pytest.raises(DarkBwtError, match=r"block %d\b" % bad):
            con.inverse_many(broken)
        outs = con.inverse_many(pairs)
        assert all(np.array_equal(o, t) for o, t in zip(outs, texts))


@pytest.mark.gpu
def test_inverse_many_rejects_bad_arguments(saca, oracle, torch):
    from dark_b200 import _ffi
    with saca.Constructor(100) as con:
        with pytest.raises(_ffi.DarkBwtError) as e:
            con.inverse_many([(b"nnbaaa", 3), (b"ab", 2)])          # origin >= n_b
        assert e.value.code == _ffi.E_INVALID_ARG
        with pytest.raises(_ffi.DarkBwtError) as e:
            con.inverse_many([(b"a" * 50, 0), (b"b" * 49, 0)])      # 99 bytes + 2 '$' rows > capacity
        assert e.value.code == _ffi.E_INVALID_N
        with pytest.raises(_ffi.DarkBwtError) as e:
            con.inverse_many([(b"", 0)])                            # an empty block
        assert e.value.code == _ffi.E_INVALID_N
        assert con.inverse_many([]) == []
        assert con.inverse_blocks([]) == []
        full = con.inverse_many([(b"a" * 49, 48), (b"b" * 49, 48)])  # 98 bytes + 2 rows: exactly full
        assert [o.tobytes() for o in full] == [b"a" * 49, b"b" * 49]
        # the device form checks offsets and origins it reads back from the device
        db = torch.frombuffer(bytearray(b"nnbaaa"), dtype=torch.uint8).cuda()
        out = torch.empty(6, dtype=torch.uint8, device="cuda")
        ds = torch.tensor([0, 6], dtype=torch.int32, device="cuda")
        for org, code in ((6, _ffi.E_INVALID_ARG), (1 << 40, _ffi.E_INVALID_ARG)):
            do = torch.tensor([org], dtype=torch.int64, device="cuda")
            with pytest.raises(_ffi.DarkBwtError) as e:
                con.inverse_many_device(db.data_ptr(), ds.data_ptr(), do.data_ptr(), 1, out.data_ptr())
            assert e.value.code == code
        do = torch.tensor([3], dtype=torch.int64, device="cuda")
        con.inverse_many_device(db.data_ptr(), ds.data_ptr(), do.data_ptr(), 1, out.data_ptr())
        assert bytes(out.cpu().numpy()) == b"banana"
    with saca.Constructor(100, flags=_ffi.F_DEVICE_ONLY) as con:         # host forms need the staging buffers
        for call in (lambda: con.inverse_many([(b"nnbaaa", 3)]), lambda: con.inverse_blocks([(b"nnbaaa", 3)])):
            with pytest.raises(_ffi.DarkBwtError) as e:
                call()
            assert e.value.code == _ffi.E_INVALID_ARG


@pytest.mark.gpu
@pytest.mark.parametrize("env_extra", [{"DARK_BWT_IBWT_TWO_WALKS": "1"}, {"DARK_BWT_IBWT_STRIDE": "1024"},
                                       {"DARK_BWT_IBWT_STRIDE": "400"}, {"DARK_BWT_IBWT_STRIDE": "2"}])
def test_inverse_many_forced_paths(env_extra):
    """The two-walk variant, long sublists written by the selective second walk, and the shortest stride."""
    code = (
        "import numpy as np, oracle\n"
        "from dark_b200 import saca, synth\n"
        "rng = np.random.default_rng(8)\n"
        "texts = [synth.generate('mixed', 4, 700001), synth.generate('dna', 2, 300007), synth.generate('rep17', 2, 200003),\n"
        "         synth.generate('text', 3, 5)] + [rng.integers(0, 3, s).astype(np.uint8) for s in range(1, 120)]\n"
        "pairs = [oracle.bwt_forward(t) if t.size > 1 else (t.copy(), 0) for t in texts]\n"
        "with saca.Constructor(sum(t.size + 1 for t in texts)) as c:\n"
        "    for o, t in zip(c.inverse_many(pairs), texts):\n"
        "        assert np.array_equal(o, t), t.size\n"
        "    for o, t in zip(c.inverse_blocks(pairs[:6]), texts[:6]):\n"
        "        assert np.array_equal(o, t), t.size\n"
        "print('ok')\n")
    env = dict(os.environ, **env_extra)
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


# ---- the pipelined batch entry --------------------------------------------------------------------------
@pytest.mark.gpu
def test_inverse_batch_ragged_pinned_and_pageable(saca, oracle, torch):
    """Sizes from 1 byte to several MiB; pageable numpy buffers (>= 1 MiB through the staging lanes) and pinned ones."""
    from dark_b200 import synth
    specs = [("text", 40, 1), ("mixed", 41, 3 * (1 << 20) + 17), ("dna", 42, 2), ("text", 43, 12345), ("rep17", 44, 1 << 20),
             ("mixed", 45, (1 << 22) - 3), ("dna", 46, 999_983), ("text", 47, 5 * (1 << 20) + 1)]
    texts = [synth.generate(k, s, n) for k, s, n in specs]
    pairs = [fwd(oracle, t) for t in texts]
    with saca.Constructor(max(t.size for t in texts)) as con:
        outs = con.inverse_blocks(pairs)                                   # pageable in and out
        for t, (b, o), out in zip(texts, pairs, outs):
            assert np.array_equal(out, t) and np.array_equal(out, oracle.bwt_decode(b, o))
        pin_in = [torch.from_numpy(b).pin_memory() for b, _ in pairs]
        pin_out = [torch.empty(t.size, dtype=torch.uint8).pin_memory() for t in texts]
        ms = con.inverse_batch_into([p.data_ptr() for p in pin_in], [t.size for t in texts], [o for _, o in pairs],
                                    [p.data_ptr() for p in pin_out])
        assert len(ms) == len(texts) and all(m > 0 for m in ms)
        for t, p in zip(texts, pin_out):
            assert np.array_equal(p.numpy(), t)
        # pinned in, pageable out, and the reverse
        pg = [np.empty(t.size, dtype=np.uint8) for t in texts]
        con.inverse_batch_into([p.data_ptr() for p in pin_in], [t.size for t in texts], [o for _, o in pairs], [p.ctypes.data for p in pg])
        assert all(np.array_equal(p, t) for p, t in zip(pg, texts))
        for p in pin_out:
            p.zero_()
        con.inverse_batch_into([b.ctypes.data for b, _ in pairs], [t.size for t in texts], [o for _, o in pairs],
                               [p.data_ptr() for p in pin_out])
        assert all(np.array_equal(p.numpy(), t) for p, t in zip(pin_out, texts))
        from dark_b200 import _ffi
        with pytest.raises(_ffi.DarkBwtError) as e:
            con.inverse_blocks([pairs[0], (pairs[3][0], 12345)])            # origin >= n
        assert e.value.code == _ffi.E_INVALID_ARG


@pytest.mark.gpu
def test_inverse_batch_large_blocks_round_trip(saca, golden, torch):
    """Three 256 MiB blocks (dna, mixed, rep17) through forward_batch -> inverse_batch, pinned buffers."""
    from dark_b200 import synth
    n = 1 << 28
    specs = [("dna", 1), ("mixed", 1000), ("rep17", 2)]
    texts = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in specs]
    for (kind, seed), t in zip(specs, texts):
        synth.generate(kind, seed, n, out=t.numpy())
    bwts = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in specs]
    backs = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in specs]
    with saca.Constructor(n) as con:
        origins = con.bwt_batch_into([t.data_ptr() for t in texts], [n] * 3, [b.data_ptr() for b in bwts])
        assert origins[0] == golden["dna:1:268435456"]["origin"]
        ms = con.inverse_batch_into([b.data_ptr() for b in bwts], [n] * 3, origins, [b.data_ptr() for b in backs])
    for (kind, _), t, b, m in zip(specs, texts, backs, ms):
        assert torch.equal(t, b), kind
        print("inverse_batch %s 256 MiB: %.2f ms device" % (kind, m))


@pytest.mark.gpu
def test_batch_entries_interleaved_on_one_context(saca, oracle, torch):
    """forward_batch, inverse_batch, inverse_many and forward on one context keep giving oracle results."""
    from dark_b200 import synth
    texts = [synth.generate("text", 50, 300_000), synth.generate("dna", 51, 1 << 20), synth.generate("mixed", 52, 77_777)]
    ref = [oracle.bwt_forward(t) for t in texts]
    with saca.Constructor(1 << 21) as con:
        for _ in range(2):
            fb = con.bwt_blocks(texts)
            for (b, o), (rb, ro) in zip(fb, ref):
                assert o == ro and np.array_equal(b, rb)
            back = con.inverse_blocks(fb)
            assert all(np.array_equal(x, t) for x, t in zip(back, texts))
            b1, o1 = con.bwt(texts[2])
            assert o1 == ref[2][1] and np.array_equal(b1, ref[2][0])
            many = con.inverse_many(ref)
            assert all(np.array_equal(x, t) for x, t in zip(many, texts))
            assert np.array_equal(con.inverse(*ref[1]), texts[1])
