"""GPU parity tests (run with `-m gpu` on a B200): the CUDA path, called through the C ABI
(dark_b200.saca.Constructor -> libdark_bwt.so), against the CPU oracle and the committed
golden fixtures.  Integer work: every comparison is bit-exact.

They mirror the reference's own tests: saca::test::detailed / roundtrips
(/root/reference/src/saca.rs:409-433) plus the differential and edge cases of SURVEY.md §4 (T1-T4).
"""
import ctypes
import os
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def crc(a):
    return "%08x" % (zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF)


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


@pytest.fixture(scope="module")
def con_small(saca, torch):
    c = saca.Constructor(1 << 16)
    yield c
    c.close()


def run_both_modes(saca, text):
    """(bwt, origin, sa) in default mode and in canonical (no alphabet packing) mode."""
    from dark_b200 import _ffi
    res = []
    for flags in (_ffi.F_DEFAULT, _ffi.F_NO_ALPHABET_PACKING):
        with saca.Constructor(len(text), flags=flags) as c:
            res.append(c.bwt_and_sa(text) + (c.stats.as_dict(),))
    return res


# ---- the reference's known answers: saca.rs:411-412 -------------------------------------------
KAT = [
    (b"abracadabra", [10, 7, 0, 3, 5, 8, 1, 4, 6, 9, 2], 2, b"rdarcaaaabb"),
    (b"banana", [5, 3, 1, 0, 4, 2], 3, b"nnbaaa"),
]


@pytest.mark.parametrize("text,sa_exp,origin_exp,bwt_exp", KAT)
def test_reference_known_answers(saca, oracle, torch, text, sa_exp, origin_exp, bwt_exp):
    # some_detail(): Constructor::new(len) -> compute -> TransformIterator -> decode (saca.rs:393-407)
    con = saca.Constructor(len(text))
    suf = con.compute(text)
    assert suf.tolist() == sa_exp
    out, origin = saca.transform(text, suf)
    assert origin == origin_exp and out.tobytes() == bwt_exp
    out2, origin2 = con.bwt(text)           # the fused call-site entry
    assert origin2 == origin_exp and out2.tobytes() == bwt_exp
    scratch = con.reuse()
    assert scratch.size >= len(text)
    assert oracle.bwt_decode(out2, origin2).tobytes() == text
    con.close()


def test_error_behaviour_matches_reference_panics(saca, torch):
    from dark_b200 import DarkBwtError
    con = saca.Constructor(16)
    assert con.capacity() == 16
    with pytest.raises(DarkBwtError):       # assert_eq!(input.len(), self.n)  saca.rs:369
        con.compute(b"too short")
    with pytest.raises(DarkBwtError):       # n == 1: assert at saca.rs:300
        con.bwt(b"x")
    with pytest.raises(DarkBwtError):       # n == 0: input[1..] panics, saca.rs:69
        con.bwt(b"")
    with pytest.raises(DarkBwtError):       # block larger than capacity: block/dc.rs:43
        con.bwt(b"y" * 17)
    out, origin = con.bwt(b"ba")            # smallest legal block, below capacity: SA = [1, 0]
    assert (out.tobytes(), origin) == (b"ba", 1)
    con.close()
    with pytest.raises(DarkBwtError):
        saca.Constructor(1)


# ---- differential against the oracle on small inputs ------------------------------------------
@pytest.mark.parametrize("sigma", [1, 2, 3, 4, 26, 256])
def test_small_random_differential(con_small, oracle, sigma):
    rng = np.random.default_rng(2000 + sigma)
    for it in range(60):
        n = int(rng.integers(2, 70)) if it < 40 else int(rng.integers(70, 9000))
        lo = int(rng.integers(0, 257 - sigma))
        t = (rng.integers(0, sigma, n) + lo).astype(np.uint8)
        bwt, origin, sa = con_small.bwt_and_sa(t)
        sa_o = oracle.saca(t)
        assert np.array_equal(sa, sa_o), (sigma, n, t[:80].tolist())
        bwt_o, origin_o = oracle.bwt_emit(t, sa_o)
        assert origin == origin_o and np.array_equal(bwt, bwt_o)


EDGE = [
    bytes([0, 0]), bytes([0, 1]), bytes([1, 0]), bytes([255, 255, 255]), bytes([0, 255, 0]),
    b"\x00" * 100, b"\xff" * 100, b"\x00" * 4097, b"ab" * 50, b"ab" * 50 + b"a", (b"abc" * 40)[:-1],
    b"a" * 63 + b"b", b"b" + b"a" * 63, bytes(range(256)), bytes(range(255, -1, -1)),
    b"\x00\x00\x00\x01\x00\x00\x00", b"aaaaaaaab" * 7 + b"aaaaaaaa", b"\x00" * 7 + b"\x01" + b"\x00" * 9,
    (b"oxvkjttpuoovephyk" * 300), (b"oxvkjttpuoovephyk" * 300)[:4099], b"ACGT" * 1025, b"A" * 5000 + b"C",
    bytes(range(256)) * 17,
]


@pytest.mark.parametrize("idx", range(len(EDGE)))
def test_edge_cases_both_modes(saca, oracle, torch, idx):
    # no in-band sentinel (0x00 and 0xFF are ordinary symbols), periodic tails, all-equal bytes,
    # n not a multiple of any tile (SURVEY §4 T4)
    t = EDGE[idx]
    sa_o = oracle.saca(t)
    bwt_o, origin_o = oracle.bwt_emit(t, sa_o)
    for bwt, origin, sa, _ in run_both_modes(saca, t):
        assert np.array_equal(sa, sa_o)
        assert origin == origin_o and np.array_equal(bwt, bwt_o)


# ---- medium: the App. D shapes, direct comparison + committed fixtures ------------------------
MEDIUM = ["text:3:768771", "dna:1:65536", "dna:1:1048576", "dna:7:1060921", "rep17:2:65536", "rep17:2:1048576",
          "rep17:2:4194304", "mixed:4:1048576", "mixed:1000:4194304", "text:5:100003"]


@pytest.mark.parametrize("key", MEDIUM)
def test_medium_shapes_vs_oracle_and_fixtures(saca, oracle, golden, torch, key):
    from dark_b200 import synth
    kind, seed, n = key.split(":")
    t = synth.generate(kind, int(seed), int(n))
    g = golden[key]
    assert crc(t) == g["text_crc32"]
    bwt_o, origin_o, sa_o = oracle.bwt_forward(t, want_sa=True)
    (bwt, origin, sa, st), (bwt2, origin2, sa2, st2) = run_both_modes(saca, t)
    assert np.array_equal(sa, sa_o) and np.array_equal(sa2, sa_o)
    assert origin == origin_o == origin2 == g["origin"]
    assert np.array_equal(bwt, bwt_o) and np.array_equal(bwt2, bwt_o)
    assert crc(bwt) == g["bwt_crc32"] and crc(sa) == g["sa_crc32"]
    # canonical mode (8 bytes per initial key): the per-round active counts are the profiler's m_r
    assert st2["symbols_per_key"] == 8
    assert st2["active"][1:] == g["profile"]["m"], (st2["active"], g["profile"]["m"])
    assert st2["rounds"] == g["profile"]["R"]
    # round trip like saca.rs:415-427
    assert np.array_equal(oracle.bwt_decode(bwt, origin), t)


FORCED_PATHS = [
    # (environment that forces a large-block code path on a small input, generator, seed, n)
    ({"DARK_BWT_FORCE_U64_STATUS": "1"}, "mixed", 4, 300001),       # 64-bit tile status (sorts of >= 2^30 pairs)
    ({"DARK_BWT_BUCKETED": "1"}, "mixed", 4, 3300001),               # bucketed rank scatter (isa[] larger than L2)
    ({"DARK_BWT_BUCKETED": "1"}, "rep17", 2, 1500007),
    ({"DARK_BWT_BUCKETED": "1"}, "dna", 5, 2000003),
    ({"DARK_BWT_EMIT_WINDOW_MB": "1"}, "mixed", 7, 5000011),         # windowed BWT emission (text larger than L2)
    ({"DARK_BWT_EMIT_WINDOW_MB": "1", "DARK_BWT_BUCKETED": "1"}, "text", 3, 2500000),
    ({"DARK_BWT_FUSE_ROUND0": "0", "DARK_BWT_BUCKETED": "1"}, "mixed", 4, 3300001),   # round 0 followed by separate partition passes
    ({"DARK_BWT_FUSE_ROUND0": "0", "DARK_BWT_BUCKETED": "1"}, "text", 3, 2500000),
    ({"DARK_BWT_PASS_IMPL": "0"}, "mixed", 9, 900001),               # the round-1 pass kernel (fallback of unaligned inputs / digits)
    ({"DARK_BWT_PASS_IMPL": "0"}, "dna", 7, 1000003),                # ... with its key-generating variant
    ({"DARK_BWT_PASS_IMPL": "0", "DARK_BWT_FORCE_U64_STATUS": "1"}, "rep17", 5, 600007),
    ({"DARK_BWT_RANK_SEARCH": "0"}, "dna", 6, 1500003),              # selective rank fill (bitmap + SA sweep) instead of the search
    ({"DARK_BWT_SPARSE_RERANK": "0"}, "dna", 9, 1400003),            # pruned round 0 re-ranked by the scan kernel instead of the sparse path
    ({"DARK_BWT_PAIRS": "0"}, "mixed", 4, 1300001),
    ({"DARK_BWT_TEXT_BUILD": "0"}, "mixed", 4, 1100001),             # rank gathers only, isa[] untagged
    ({"DARK_BWT_TEXT_BUILD": "0"}, "rep17", 2, 700001),
    ({"DARK_BWT_TEXT_BUILD": "1000000"}, "mixed", 5, 1200001),       # text-order key build in every round that may use it
    ({"DARK_BWT_TEXT_BUILD": "1000000"}, "rep17", 3, 900001),
    ({"DARK_BWT_TEXT_BUILD": "1000000"}, "text", 6, 800001),
    ({"DARK_BWT_TEXT_BUILD": "1000000", "DARK_BWT_BUCKETED": "1"}, "mixed", 6, 2100001),
    ({"DARK_BWT_TEXT_BUILD": "1000000", "DARK_BWT_BUCKETED": "1"}, "rep17", 4, 1000001),
    ({"DARK_BWT_TEXT_BUILD": "1000000", "DARK_BWT_RANK_SEARCH": "0"}, "dna", 6, 1500003),
    ({"DARK_BWT_CHECK_HIST": "1"}, "mixed", 4, 900001),              # q-gram histogram compared with the per-key count
    ({"DARK_BWT_CHECK_HIST": "1"}, "dna", 2, 1100003),
    ({"DARK_BWT_FORCE_U64_STATUS": "1"}, "dna", 8, 600011),          # key-generating pass with 64-bit tile status
    ({"DARK_BWT_INLINE_EMIT": "0"}, "dna", 3, 1200007),              # pruned initial sort WITHOUT inline emission
    ({"DARK_BWT_INLINE_EMIT": "0", "DARK_BWT_EMIT_WINDOW_MB": "1"}, "dna", 4, 3000001),        # ... emitted by the windowed gather
]


@pytest.mark.parametrize("idx", range(len(FORCED_PATHS)))
def test_large_block_code_paths_forced_on_small_inputs(oracle, idx):
    """Paths that only switch on for huge blocks (64-bit tile status, bucketed rank scatter, windowed
    emission) are forced through environment knobs in a fresh process and compared with the oracle."""
    import subprocess
    import sys
    env_extra, kind, seed, n = FORCED_PATHS[idx]
    code = (
        "import numpy as np, oracle\n"
        "from dark_b200 import saca, synth\n"
        f"t = synth.generate('{kind}', {seed}, {n})\n"
        "c = saca.Constructor(t.size)\n"
        "b, o, s = c.bwt_and_sa(t)\n"
        "bo, oo, so = oracle.bwt_forward(t, want_sa=True)\n"
        "assert o == oo and np.array_equal(b, bo) and np.array_equal(s, so)\n"
        "print('ok')\n")
    env = dict(os.environ, **env_extra)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=root, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


STAGING = [
    {},                                                                  # defaults: 12 lanes x 2 MiB
    {"DARK_BWT_HOST_THREADS": "1", "DARK_BWT_HOST_CHUNK_MB": "1"},       # one lane, many chunks
    {"DARK_BWT_HOST_THREADS": "16", "DARK_BWT_HOST_CHUNK_MB": "4"},      # more lanes than chunks
    {"DARK_BWT_HOST_THREADS": "0"},                                      # staging off: the driver's own bounce buffer
]


@pytest.mark.parametrize("idx", range(len(STAGING)))
def test_pageable_host_buffers_through_the_staging_lanes(oracle, idx):
    """The reference hands over a plain Vec<u8> and collects into a fresh one (src/main.rs:95, src/block/dc.rs:45-50):
    pageable buffers of 1 MiB or more go through the pinned staging lanes.  Ragged sizes (not a multiple of the lane
    chunk), the SA output (4n bytes through the same lanes), the batch entry, the inverse and the DC entry give what pinned
    buffers and the oracle give, for every lane setting."""
    import subprocess
    import sys
    code = (
        "import numpy as np, torch, oracle\n"
        "from dark_b200 import saca, synth\n"
        "n = 5 * (1 << 20) + 12345\n"
        "t = synth.generate('mixed', 21, n)\n"
        "c = saca.Constructor(n)\n"
        "b, o, s = c.bwt_and_sa(t)\n"                                   # pageable numpy buffers in and out
        "bo, oo, so = oracle.bwt_forward(t, want_sa=True)\n"
        "assert o == oo and np.array_equal(b, bo) and np.array_equal(s, so)\n"
        "pt = torch.from_numpy(t).pin_memory(); pb = torch.empty(n, dtype=torch.uint8).pin_memory()\n"
        "assert c.bwt_into(pt.data_ptr(), n, pb.data_ptr()) == oo and np.array_equal(pb.numpy(), bo)\n"   # pinned: straight DMA
        "blocks = [t, synth.generate('dna', 22, 3 * (1 << 20) + 7), synth.generate('text', 23, 4097), t[: 2 * (1 << 20)]]\n"
        "for blk, (bb, ob) in zip(blocks, c.bwt_blocks(blocks)):\n"      # pipelined batch entry, pageable in and out
        "    rb, ro = oracle.bwt_forward(blk)\n"
        "    assert ob == ro and np.array_equal(bb, rb)\n"
        "assert np.array_equal(c.inverse(bo, oo), t)\n"                  # unpack side, pageable
        "d = c.bwt_dc(t)\n"                                              # BWT + distance coding, 4n bytes of distances out
        "ref = oracle.dc_encode(bo)\n"
        "assert np.array_equal(d[0], bo) and d[1] == oo and np.array_equal(d[2]['dist'], ref[0]) and d[2]['num_unique'] == ref[3]\n"
        "print('ok')\n")
    env = dict(os.environ, **STAGING[idx])
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=root, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


# ---- building blocks (SURVEY §4 T1) -------------------------------------------------------------
@pytest.mark.parametrize("m,begin,end", [(1, 0, 64), (100, 0, 64), (4096, 0, 64), (4097, 0, 64), (1000003, 0, 64),
                                         (300000, 0, 40), (300000, 16, 48), (50000, 0, 8), (300000, 3, 40)])
def test_radix_sort_pairs_is_a_stable_sort(saca, oracle, torch, m, begin, end):
    from dark_b200 import synth
    rng = np.random.default_rng(m + begin)
    keys = rng.integers(0, 1 << 63, m, dtype=np.uint64) * 2 + rng.integers(0, 2, m, dtype=np.uint64)
    if m > 1000:
        keys[: m // 2] &= np.uint64(0x00FF00FF00FF00FF)      # skewed digits, many ties
    vals = np.arange(m, dtype=np.uint32)
    nbits = end - begin
    passes = (nbits + 7) // 8
    mask = np.uint64((1 << min(64 - begin, passes * 8)) - 1)
    sub = (keys >> np.uint64(begin)) & mask                   # whole 8-bit digits take part
    order = np.argsort(sub, kind="stable")
    con = saca.Constructor(max(m, 2))
    # off = 1: keys and values one element past 16-byte alignment, so the passes that read them take the round-1 kernel
    # (k_onesweep_pass) and those that read the aligned alt buffers take the TMA pass
    for off in (0, 1):
        dk = torch.empty(m + off, dtype=torch.int64, device="cuda")[off:]
        dv = torch.empty(m + off, dtype=torch.int32, device="cuda")[off:]
        dk.copy_(torch.from_numpy(keys.view(np.int64)))
        dv.copy_(torch.from_numpy(vals.view(np.int32)))
        dk2, dv2 = torch.empty_like(dk), torch.empty_like(dv)
        in_alt, _ = con.sort_pairs_device(dk.data_ptr(), dv.data_ptr(), dk2.data_ptr(), dv2.data_ptr(), m, begin, end)
        torch.cuda.synchronize()
        rk = (dk2 if in_alt else dk).cpu().numpy().view(np.uint64)
        rv = (dv2 if in_alt else dv).cpu().numpy().view(np.uint32)
        assert np.array_equal(rv, vals[order]), off
        assert np.array_equal(rk, keys[order]), off
    # a forward on the same context: its passes take over the sort status buffer from the sort's
    t = synth.generate("text", m, max(m, 2))
    b, o = con.bwt(t)
    rb, ro = oracle.bwt_forward(t)
    assert o == ro and np.array_equal(b, rb)
    con.close()


def test_emission_kernel_alone(saca, oracle, torch):
    from dark_b200 import synth
    for n in (2, 3, 5, 1023, 100003):
        t = synth.generate("text", 11, n)
        sa = oracle.saca(t)
        bwt_o, origin_o = oracle.bwt_emit(t, sa)
        con = saca.Constructor(n)
        dt = torch.from_numpy(t.copy()).cuda()
        ds = torch.from_numpy(sa.view(np.int32)).cuda()
        for off in (0, 1):                                    # aligned and unaligned output pointer
            db = torch.zeros(n + 8, dtype=torch.uint8, device="cuda")
            origin = con.emit_device(dt.data_ptr(), n, ds.data_ptr(), db.data_ptr() + off)
            assert origin == origin_o
            assert np.array_equal(db.cpu().numpy()[off:off + n], bwt_o)
        # a suffix array that is only 4-byte aligned (a slice of a larger buffer): no 128-bit SA loads
        ds_off = torch.zeros(n + 4, dtype=torch.int32, device="cuda")
        for shift in (1, 2, 3):
            ds_off[shift:shift + n] = ds
            db = torch.zeros(n + 8, dtype=torch.uint8, device="cuda")
            origin = con.emit_device(dt.data_ptr(), n, ds_off.data_ptr() + 4 * shift, db.data_ptr())
            assert origin == origin_o
            assert np.array_equal(db.cpu().numpy()[:n], bwt_o)
        con.close()


def test_gpu_verifier_accepts_and_rejects(saca, oracle, torch):
    from dark_b200 import synth
    t = synth.generate("mixed", 9, 200001)
    sa = oracle.saca(t)
    con = saca.Constructor(t.size)
    dt = torch.from_numpy(t.copy()).cuda()
    ds = torch.from_numpy(sa.view(np.int32)).cuda()
    assert con.verify_sa_device(dt.data_ptr(), t.size, ds.data_ptr()) == 0
    bad = sa.copy()
    bad[[1000, 1001]] = bad[[1001, 1000]]
    ds = torch.from_numpy(bad.view(np.int32)).cuda()
    assert con.verify_sa_device(dt.data_ptr(), t.size, ds.data_ptr()) > 0
    bad = sa.copy()
    bad[5] = bad[6]                                           # not a permutation
    ds = torch.from_numpy(bad.view(np.int32)).cuda()
    assert con.verify_sa_device(dt.data_ptr(), t.size, ds.data_ptr()) > 0
    con.close()


# ---- large: fixtures + the independent GPU verifier (SURVEY §4 T2/T3) ---------------------------
LARGE = ["dna:1:16777216", "mixed:4:16777216", "rep17:2:67108864", "dna:1:268435456", "mixed:1000:268435456",
         "mixed:4:2147483648"]   # the last one is C4: 2 GiB block, 64-bit offsets, 64-bit tile status


@pytest.mark.parametrize("key", LARGE)
def test_large_shapes_vs_fixtures_device_resident(saca, golden, torch, key):
    """C2 (256 MB DNA), C3 (64 MB period-17), a C5 block, device-resident through
    dark_bwt_forward_device; SA checked by the O(n) GPU verifier, BWT/SA/origin by CRC against
    the oracle's committed outputs."""
    from dark_b200 import synth, _ffi
    kind, seed, n = key.split(":")
    n = int(n)
    g = golden[key]
    t = synth.generate(kind, int(seed), n)
    assert crc(t) == g["text_crc32"]
    con = saca.Constructor(n, flags=_ffi.F_DEVICE_ONLY)
    dt = torch.from_numpy(t).cuda()
    db = torch.empty(n, dtype=torch.uint8, device="cuda")
    ds = torch.empty(n, dtype=torch.int32, device="cuda")
    origin = con.bwt_device(dt.data_ptr(), n, db.data_ptr(), ds.data_ptr())
    st = con.stats.as_dict()
    assert origin == g["origin"]
    assert con.verify_sa_device(dt.data_ptr(), n, ds.data_ptr()) == 0
    assert crc(db.cpu().numpy()) == g["bwt_crc32"]
    assert crc(ds.cpu().numpy()) == g["sa_crc32"]
    # without the SA output buffer the result is the same
    db2 = torch.empty(n, dtype=torch.uint8, device="cuda")
    assert con.bwt_device(dt.data_ptr(), n, db2.data_ptr(), None) == origin
    assert torch.equal(db, db2)
    print(key, {k: st[k] for k in ("sigma", "symbols_per_key", "rounds", "sort_passes", "device_ms")})
    con.close()


def test_pipelined_batch_entry_matches_single_calls(saca, oracle, torch):
    """dark_bwt_forward_batch: several blocks of different shapes and sizes through the double-buffered
    copy/compute pipeline give exactly what separate calls (and the oracle) give."""
    from dark_b200 import synth
    con = saca.Constructor(1 << 21)
    specs = [("mixed", 6, 1 << 21), ("dna", 3, 999983), ("text", 4, 12345), ("rep17", 5, 1 << 20), ("dna", 8, 2),
             ("mixed", 11, (1 << 21) - 1), ("text", 12, 300000)]
    blocks = [synth.generate(k, s, n) for k, s, n in specs]
    res = con.bwt_blocks(blocks)
    assert len(res) == len(blocks)
    for blk, (bwt, origin) in zip(blocks, res):
        bwt_o, origin_o = oracle.bwt_forward(blk)
        assert origin == origin_o and np.array_equal(bwt, bwt_o)
    # pinned buffers, repeated block, alternating outputs (what bench.py does)
    t = torch.from_numpy(blocks[0]).pin_memory()
    o1 = torch.empty(t.numel(), dtype=torch.uint8).pin_memory()
    o2 = torch.empty(t.numel(), dtype=torch.uint8).pin_memory()
    origins, stats = con.bwt_batch_into([t.data_ptr()] * 5, [t.numel()] * 5, [o1.data_ptr(), o2.data_ptr()] * 2 + [o1.data_ptr()],
                                        want_stats=True)
    assert origins == [res[0][1]] * 5 and len(stats) == 5
    assert np.array_equal(o1.numpy(), res[0][0]) and np.array_equal(o2.numpy(), res[0][0])
    con.close()


def test_idempotent_context_reuse(saca, oracle, torch):
    """One context, many blocks of different sizes (the Encoder keeps its Constructor)."""
    from dark_b200 import synth
    con = saca.Constructor(1 << 20)
    for kind, seed, n in (("dna", 3, 1 << 20), ("text", 4, 12345), ("rep17", 5, 999999), ("mixed", 6, 1 << 19),
                          ("dna", 3, 1 << 20)):
        t = synth.generate(kind, seed, n)
        bwt, origin = con.bwt(t)
        bwt_o, origin_o = oracle.bwt_forward(t)
        assert origin == origin_o and np.array_equal(bwt, bwt_o)
    con.close()


# ---- the unpack side: inverse BWT (SURVEY §8f) ---------------------------------------------------
@pytest.mark.parametrize("kind,seed,n", [("dna", 12, 500003), ("mixed", 13, 400001), ("text", 14, 300007), ("rep17", 15, 200003)])
def test_device_entry_with_unaligned_buffers(saca, oracle, torch, kind, seed, n):
    """d_text, d_bwt_out and d_sa_out may be arbitrary slices of larger device buffers: text and BWT at odd byte offsets,
    the suffix array only 4-byte aligned (no 128-bit accesses may be assumed on any of them)."""
    from dark_b200 import synth
    t = synth.generate(kind, seed, n)
    bwt_o, origin_o, sa_o = oracle.bwt_forward(t, want_sa=True)
    con = saca.Constructor(n)
    for toff, boff, soff in ((0, 0, 1), (1, 3, 3), (5, 2, 2)):
        dt = torch.zeros(n + 16, dtype=torch.uint8, device="cuda")
        dt[toff:toff + n] = torch.from_numpy(t).cuda()
        db = torch.zeros(n + 16, dtype=torch.uint8, device="cuda")
        ds = torch.zeros(n + 8, dtype=torch.int32, device="cuda")
        origin = con.bwt_device(dt.data_ptr() + toff, n, db.data_ptr() + boff, ds.data_ptr() + 4 * soff)
        assert origin == origin_o
        assert np.array_equal(db.cpu().numpy()[boff:boff + n], bwt_o)
        assert np.array_equal(ds.cpu().numpy()[soff:soff + n].view(np.uint32), sa_o)
    con.close()


def test_inverse_known_answers(saca, torch):
    # saca.rs:404-406: bwt::decode(&output, origin, suf) gives back the input of the KATs
    for text, _, origin, bwt in KAT:
        assert saca.decode(bwt, origin).tobytes() == text


@pytest.mark.parametrize("sigma", [1, 2, 4, 256])
def test_inverse_small_random_vs_oracle(con_small, oracle, sigma):
    rng = np.random.default_rng(3000 + sigma)
    for it in range(40):
        n = int(rng.integers(1, 70)) if it < 25 else int(rng.integers(70, 9000))
        t = rng.integers(0, sigma, n).astype(np.uint8)
        if n >= 2:
            bwt, origin = oracle.bwt_forward(t)
        else:
            bwt, origin = t.copy(), 0
        back = con_small.inverse(bwt, origin)
        assert np.array_equal(back, t), (sigma, n)
        assert np.array_equal(back, oracle.bwt_decode(bwt, origin))


@pytest.mark.parametrize("key", ["text:3:768771", "dna:1:1048576", "rep17:2:1048576", "mixed:4:1048576", "mixed:1000:4194304"])
def test_inverse_medium_shapes_roundtrip(saca, oracle, torch, key):
    from dark_b200 import synth
    kind, seed, n = key.split(":")
    t = synth.generate(kind, int(seed), int(n))
    with saca.Constructor(t.size) as con:
        bwt, origin = con.bwt(t)                     # forward on the GPU ...
        assert np.array_equal(con.inverse(bwt, origin), t)   # ... and back
        edge = EDGE[5]                                # all-equal bytes through the same context
        b2, o2 = oracle.bwt_forward(edge)
        assert con.inverse(b2, o2).tobytes() == edge


def test_inverse_rejects_inconsistent_input_without_hanging(saca, oracle, torch):
    from dark_b200 import DarkBwtError, synth
    t = synth.generate("text", 21, 50000)
    bwt, origin = oracle.bwt_forward(t)
    with saca.Constructor(t.size) as con:
        with pytest.raises(DarkBwtError):
            con.inverse(bwt, t.size)                  # origin out of range
        wrong = (origin + 12345) % t.size
        try:                                          # a wrong origin either fails loudly or decodes to another text,
            back = con.inverse(bwt, wrong)            # but never hangs and never returns the original
            assert not np.array_equal(back, t)
        except DarkBwtError:
            pass
        assert np.array_equal(con.inverse(bwt, origin), t)


def test_inverse_large_device_resident(saca, golden, torch):
    """C2 (256 MiB DNA): forward then inverse, both device-resident; the inverse restores the block."""
    from dark_b200 import synth, _ffi
    n = 1 << 28
    t = synth.generate("dna", 1, n)
    con = saca.Constructor(n, flags=_ffi.F_DEVICE_ONLY)
    dt = torch.from_numpy(t).cuda()
    db = torch.empty(n, dtype=torch.uint8, device="cuda")
    origin = con.bwt_device(dt.data_ptr(), n, db.data_ptr())
    assert origin == golden["dna:1:268435456"]["origin"]
    dback = torch.zeros(n, dtype=torch.uint8, device="cuda")
    ms = con.inverse_device(db.data_ptr(), n, origin, dback.data_ptr())
    assert torch.equal(dback, dt)
    print("inverse BWT 256 MiB: %.2f ms (%.1f GB/s)" % (ms, n / ms / 1e6))
    con.close()


def test_two_contexts_in_two_host_threads(saca, oracle, torch):
    """Distinct contexts are independent (INTEGRATION.md: one context per host thread): two threads drive
    two contexts on the same GPU at once (ctypes drops the GIL during the call)."""
    import threading
    from dark_b200 import synth
    blocks = [synth.generate("mixed", 31, 700001), synth.generate("dna", 32, 900001)]
    expect = [oracle.bwt_forward(b) for b in blocks]
    results = [None, None]

    def work(i):
        with saca.Constructor(blocks[i].size) as con:
            for _ in range(3):
                results[i] = con.bwt(blocks[i])

    threads = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for (bwt, origin), (bwt_o, origin_o) in zip(results, expect):
        assert origin == origin_o and np.array_equal(bwt, bwt_o)


def test_cpp_mirror_runs_the_reference_known_answers(torch, tmp_path):
    """examples/saca_cpp_demo.cpp: the C++ mirror of saca::Constructor on saca.rs:411-412, on the GPU."""
    import subprocess
    from dark_b200 import _ffi
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = tmp_path / "saca_cpp_demo"
    libdir = os.path.dirname(_ffi.lib_path())
    subprocess.check_call(["g++", "-std=c++17", "-I", root, os.path.join(root, "examples", "saca_cpp_demo.cpp"), "-L", libdir,
                           "-l:" + os.path.basename(_ffi.lib_path()), f"-Wl,-rpath,{libdir}", "-o", str(exe)])   # whichever build DARK_BWT_LIB names
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), (out.returncode, out.stdout, out.stderr)


@pytest.mark.parametrize("key", ["text:3:768771", "dna:1:1048576", "rep17:2:1048576", "mixed:4:1048576", "rep17:2:67108864",
                                 "dna:1:268435456"])
def test_gpu_lcp_profile_matches_the_oracle_profiler(saca, golden, torch, key):
    """dark_bwt_lcp_profile_device (SURVEY §8d/§8f): m_r, R, max LCP and B_alg from the GPU equal the oracle
    profiler's committed values, up to the full C2 and C3 blocks."""
    from dark_b200 import synth, _ffi
    kind, seed, n = key.split(":")
    n = int(n)
    g = golden[key]["profile"]
    t = synth.generate(kind, int(seed), n)
    con = saca.Constructor(n, flags=_ffi.F_DEVICE_ONLY)
    dt = torch.from_numpy(t).cuda()
    db = torch.empty(n, dtype=torch.uint8, device="cuda")
    ds = torch.empty(n, dtype=torch.int32, device="cuda")
    con.bwt_device(dt.data_ptr(), n, db.data_ptr(), ds.data_ptr())
    p = con.lcp_profile_device(dt.data_ptr(), n, ds.data_ptr())
    assert p["m"] == g["m"] and p["R"] == g["R"]
    assert p["max_lcp"] == g["max_lcp"]
    assert (p["b"], p["P"]) == (g["b"], g["P"])
    assert abs(p["b_alg"] - g["b_alg"]) <= 1.0
    con.close()


def _structured_inputs():
    fib = [b"a", b"ab"]
    while len(fib[-1]) < 300000:
        fib.append(fib[-1] + fib[-2])
    tm = bytearray(b"\x00")
    while len(tm) < 262144:
        tm += bytes(1 - x for x in tm)
    rng = np.random.default_rng(99)
    runs = np.repeat(rng.integers(0, 3, 4000).astype(np.uint8), rng.integers(1, 200, 4000))
    return {
        "fibonacci": fib[-1][:300007],
        "thue_morse": bytes(tm),
        "zeros_1M": bytes(1 << 20),
        "ff_then_00": b"\xff" * 70000 + b"\x00" * 70001,
        "long_runs": runs.tobytes(),
        "period_255": bytes(range(1, 256)) * 1200,
        "two_copies": (lambda x: x + x)(rng.integers(0, 256, 150000).astype(np.uint8).tobytes()),
    }


@pytest.mark.parametrize("name", ["fibonacci", "thue_morse", "zeros_1M", "ff_then_00", "long_runs", "period_255", "two_copies"])
def test_structured_worst_cases(saca, oracle, torch, name):
    """Highly repetitive inputs (long LCPs: many doubling rounds, giant groups, trivial digits everywhere)."""
    t = _structured_inputs()[name]
    bwt_o, origin_o, sa_o = oracle.bwt_forward(t, want_sa=True)
    with saca.Constructor(len(t)) as con:
        bwt, origin, sa = con.bwt_and_sa(t)
        assert origin == origin_o and np.array_equal(sa, sa_o) and np.array_equal(bwt, bwt_o)
        assert con.inverse(bwt, origin).tobytes() == t


# ---- pairs mode (late rounds in which every group is a pair) -----------------------------------
def _pairs_inputs():
    rng = np.random.default_rng(7)
    dna = rng.integers(0, 4, 2_000_003).astype(np.uint8) + 65
    planted = dna.copy()
    planted[1_200_000:1_200_000 + 5000] = planted[100_000:100_000 + 5000]      # one long repeat in random DNA
    nested = rng.integers(0, 256, 600_000).astype(np.uint8)
    nested[400_000:400_000 + 70_000] = nested[10_000:10_000 + 70_000]            # a pair of long copies ...
    nested[500_000:500_000 + 300] = nested[20_000:20_000 + 300]                  # ... and a triple inside it
    two = rng.integers(0, 256, 150_001).astype(np.uint8)
    return {"planted_dna": planted, "nested_repeats": nested, "two_copies_odd": np.concatenate([two, two]),
            "tail_repeat": np.concatenate([rng.integers(0, 256, 300_000).astype(np.uint8)] * 1 + [np.arange(40_000, dtype=np.uint8)])}


@pytest.mark.parametrize("name", ["planted_dna", "nested_repeats", "two_copies_odd", "tail_repeat"])
def test_pairs_mode_rounds(saca, oracle, torch, name):
    """Inputs whose late rounds hold nothing but pairs: the pairs kernel must take over (stats.pair_rounds > 0),
    leave the per-round active counts canonical and produce the oracle's bytes; both alphabet modes."""
    t = _pairs_inputs()[name]
    bwt_o, origin_o, sa_o = oracle.bwt_forward(t, want_sa=True)
    (bwt, origin, sa, st), (bwt2, origin2, sa2, st2) = run_both_modes(saca, t)
    assert origin == origin_o == origin2
    assert np.array_equal(sa, sa_o) and np.array_equal(sa2, sa_o)
    assert np.array_equal(bwt, bwt_o) and np.array_equal(bwt2, bwt_o)
    if name != "tail_repeat":
        assert st["pair_rounds"] > 0 and st2["pair_rounds"] > 0, (st["pair_rounds"], st2["pair_rounds"])
    prof = oracle.profile(t, sa_o)
    assert st2["active"][1:1 + len(prof["m"])] == prof["m"], (st2["active"], prof["m"])


def test_qgram_histogram_equals_per_key_histogram(oracle):
    """DARK_BWT_CHECK_HIST=1 makes the library count the round-0 digit histograms both ways (one q-gram
    histogram of the text vs eight digits per key) and fail on any difference; alphabets of 2, 4, 16 and 256
    symbols, sizes around the 56-position boundary correction, an unaligned device pointer."""
    import subprocess
    import sys
    code = (
        "import numpy as np, torch, oracle\n"
        "from dark_b200 import saca, _ffi\n"
        "rng = np.random.default_rng(5)\n"
        "for sigma in (2, 3, 4, 11, 16, 200, 256):\n"
        "    for n in (2, 3, 5, 8, 17, 55, 56, 57, 63, 64, 65, 100, 4097, 300007):\n"
        "        t = rng.integers(0, sigma, n).astype(np.uint8)\n"
        "        if sigma < 200: t = t * 7 + 3\n"
        "        with saca.Constructor(n) as c:\n"
        "            b, o, s = c.bwt_and_sa(t)\n"
        "        bo, oo, so = oracle.bwt_forward(t, want_sa=True)\n"
        "        assert o == oo and np.array_equal(b, bo) and np.array_equal(s, so), (sigma, n)\n"
        "n = 100003\n"
        "t = rng.integers(0, 4, n + 1).astype(np.uint8)\n"
        "d = torch.from_numpy(t).cuda()\n"
        "db = torch.empty(n, dtype=torch.uint8, device='cuda')\n"
        "with saca.Constructor(n, flags=_ffi.F_DEVICE_ONLY) as c:\n"
        "    o = c.bwt_device(d.data_ptr() + 1, n, db.data_ptr(), None)\n"
        "bo, oo = oracle.bwt_forward(np.ascontiguousarray(t[1:]))\n"
        "assert o == oo and np.array_equal(db.cpu().numpy(), bo)\n"
        "print('ok')\n")
    env = dict(os.environ, DARK_BWT_CHECK_HIST="1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=root, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


# ---- many small blocks in one sort (dark_bwt_forward_many) ---------------------------------------
def _many_cases():
    rng = np.random.default_rng(11)
    from dark_b200 import synth
    text = synth.generate("text", 3, 200_000)
    cases = {
        "two_tiny": [b"abracadabra", b"banana"],
        "identical_blocks": [b"mississippi"] * 5 + [b"banana"] * 3,      # equal suffixes in different blocks: ordered by block
        "prefix_blocks": [b"aaaa", b"aaaaaaaa", b"aa", b"aaab", b"baaa"],
        "minimal": [b"ab", b"ba", b"aa", b"\x00\x00", b"\xff\x00"],
        "binary_256": [rng.integers(0, 256, int(s)).astype(np.uint8).tobytes() for s in (300, 70_001, 2, 4096, 65_537)],
        "dna_ragged": [(rng.integers(0, 4, int(s)).astype(np.uint8) + 65).tobytes() for s in rng.integers(2, 50_000, 40)],
        "text_slices": [text[i:i + 9973].tobytes() for i in range(0, 190_000, 9973)],
        "periodic": [bytes(range(1, 18)) * 500, bytes(range(1, 18)) * 400 + b"x", b"\x07" * 30_000, b"\x07" * 29_999],
        "one_block": [text[:50_001].tobytes()],
    }
    return cases


@pytest.mark.parametrize("name", ["two_tiny", "identical_blocks", "prefix_blocks", "minimal", "binary_256", "dna_ragged",
                                  "text_slices", "periodic", "one_block"])
def test_many_small_blocks_in_one_sort(saca, oracle, torch, name):
    """dark_bwt_forward_many must give, block by block, exactly what the oracle gives for the block alone."""
    blocks = _many_cases()[name]
    total = sum(len(b) for b in blocks)
    with saca.Constructor(max(total, 2)) as con:
        res = con.bwt_many(blocks)
        assert len(res) == len(blocks)
        for k, (blk, (bwt, origin)) in enumerate(zip(blocks, res)):
            bwt_o, origin_o = oracle.bwt_forward(blk)
            assert origin == origin_o, (name, k, origin, origin_o)
            assert np.array_equal(bwt, bwt_o), (name, k)
        # the same context still does single blocks afterwards
        b1, o1 = con.bwt(blocks[0])
        bo, oo = oracle.bwt_forward(blocks[0])
        assert o1 == oo and np.array_equal(b1, bo)


def test_many_blocks_device_form_with_suffix_arrays(saca, oracle, torch):
    rng = np.random.default_rng(12)
    blocks = [rng.integers(0, 3, int(s)).astype(np.uint8) for s in (1000, 2, 33_333, 7, 12_345)]
    starts = np.concatenate([[0], np.cumsum([b.size for b in blocks])]).astype(np.uint32)
    n = int(starts[-1])
    from dark_b200 import _ffi
    with saca.Constructor(n, flags=_ffi.F_DEVICE_ONLY) as con:
        dt = torch.from_numpy(np.concatenate(blocks)).cuda()
        ds = torch.from_numpy(starts.view(np.int32)).cuda()
        db = torch.empty(n, dtype=torch.uint8, device="cuda")
        do = torch.empty(len(blocks), dtype=torch.int64, device="cuda")
        dsa = torch.empty(n, dtype=torch.int32, device="cuda")
        con.bwt_many_device(dt.data_ptr(), ds.data_ptr(), len(blocks), db.data_ptr(), do.data_ptr(), dsa.data_ptr())
        hb, ho, hs = db.cpu().numpy(), do.cpu().numpy(), dsa.cpu().numpy().view(np.uint32)
    for k, blk in enumerate(blocks):
        bwt_o, origin_o, sa_o = oracle.bwt_forward(blk, want_sa=True)
        a, e = int(starts[k]), int(starts[k + 1])
        assert int(ho[k]) == origin_o and np.array_equal(hb[a:e], bwt_o) and np.array_equal(hs[a:e], sa_o)


def test_many_blocks_rejects_bad_arguments(saca, torch):
    from dark_b200 import _ffi
    with saca.Constructor(1000) as con:
        with pytest.raises(_ffi.DarkBwtError):
            con.bwt_many([b"ab", b"x"])            # a block of one byte (the reference panics for n = 1, saca.rs:69)
        with pytest.raises(_ffi.DarkBwtError):
            con.bwt_many([b"a" * 600, b"b" * 600])  # the blocks share one arena: 1200 > capacity
        assert con.bwt_many([]) == []


@pytest.mark.parametrize("env_extra", [{"DARK_BWT_IBWT_TWO_WALKS": "1"}, {"DARK_BWT_IBWT_STRIDE": "1024"},
                                       {"DARK_BWT_IBWT_STRIDE": "400"}, {"DARK_BWT_IBWT_STRIDE": "2"}])
def test_inverse_forced_paths(env_extra):
    """The two-walk variant, and splitter strides that make most sublists longer than the stash chunk (they are then
    written by the second, selective walk) or as short as possible."""
    import subprocess
    import sys
    code = (
        "import numpy as np, oracle\n"
        "from dark_b200 import saca, synth\n"
        "for kind, seed, n in (('mixed', 4, 700001), ('dna', 2, 300007), ('rep17', 2, 200003), ('text', 3, 5)):\n"
        "    t = synth.generate(kind, seed, n)\n"
        "    b, o = oracle.bwt_forward(t)\n"
        "    with saca.Constructor(n) as c:\n"
        "        assert np.array_equal(c.inverse(b, o), t), (kind, n)\n"
        "print('ok')\n")
    env = dict(os.environ, **env_extra)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=root, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


def _sparse_fallback_inputs():
    rng = np.random.default_rng(21)
    a = (rng.integers(0, 4, 1_500_000).astype(np.uint8) + 65)
    motif = (rng.integers(0, 4, 300).astype(np.uint8) + 65)
    for k in range(150):
        a[5000 + 9000 * k: 5000 + 9000 * k + 300] = motif
    half = (rng.integers(0, 4, 600_000).astype(np.uint8) + 65)
    return {"planted_motif": a, "repeated_half": np.concatenate([half, half])}


def test_sparse_rerank_fallbacks(saca, oracle, torch):
    """Pruned round 0 (uniform DNA digits) whose survivors defeat the sparse re-rank: a motif planted 150 times (groups
    longer than the walk limit -> scan kernel), and a block whose second half repeats the first (more than n/16
    survivors -> scan kernel).  Both must still give the oracle's bytes."""
    for t in _sparse_fallback_inputs().values():
        bwt_o, origin_o, sa_o = oracle.bwt_forward(t, want_sa=True)
        with saca.Constructor(t.size) as con:
            bwt, origin, sa = con.bwt_and_sa(t)
            assert con.stats.initial_symbols < con.stats.symbols_per_key  # the initial sort was pruned
        assert origin == origin_o and np.array_equal(sa, sa_o) and np.array_equal(bwt, bwt_o)


# ---- distance coding + MTF on the GPU (SURVEY §8f rank 3; parity UNPINNED: checked against the restated oracle) ---------
def _check_dc(res, b, oracle):
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
    assert np.array_equal(oracle.dc_decode(res["init"], res["item_dist"], n), b)      # and back


@pytest.mark.gpu
def test_dc_small_random_and_structured(saca, oracle, torch):
    rng = np.random.default_rng(11)
    con = saca.Constructor(1 << 16)
    cases = [np.zeros(1, np.uint8), np.zeros(5000, np.uint8), np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8)[::-1].copy(),
             np.tile(np.arange(256, dtype=np.uint8), 40), np.repeat(np.arange(7, dtype=np.uint8), 4099)[:20000],
             np.frombuffer(b"rdarcaaaabb", dtype=np.uint8).copy(), np.frombuffer(b"nnbaaa", dtype=np.uint8).copy()]
    for trial in range(120):
        n = int(rng.integers(1, 9000))
        sigma = int(rng.choice([1, 2, 4, 26, 256]))
        b = rng.integers(0, sigma, n).astype(np.uint8)
        if trial % 2:
            b = np.repeat(b, rng.integers(1, 40, n))[: int(rng.integers(1, 60000))]
        cases.append(b)
    for b in cases:
        _check_dc(con.dc_encode(b), b, oracle)
    con.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,seed,n", [("text", 3, 768771), ("dna", 1, 1 << 20), ("mixed", 4, 1 << 22), ("rep17", 2, 1 << 20)])
def test_forward_dc_fused_entry(saca, oracle, torch, kind, seed, n):
    """block/dc.rs:45-52 in one call: forward BWT, then DC of the BWT while it is still in HBM; host buffers out."""
    from dark_b200 import synth
    t = synth.generate(kind, seed, n)
    con = saca.Constructor(n)
    bwt, origin, res = con.bwt_dc(t)
    bwt_o, origin_o = oracle.bwt_forward(t)
    assert origin == origin_o and np.array_equal(bwt, bwt_o)
    _check_dc(res, bwt_o, oracle)
    # device entry with caller-owned outputs
    db = torch.from_numpy(bwt_o).cuda()
    dd = torch.empty(n, dtype=torch.int32, device="cuda")
    dpos, ddist = torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.int32, device="cuda")
    dsym, drk = torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")
    info = con.dc_encode_device(db.data_ptr(), n, dd.data_ptr(), dpos.data_ptr(), ddist.data_ptr(), dsym.data_ptr(), drk.data_ptr())
    k = int(info.num_items)
    assert k == res["num_items"]
    assert np.array_equal(dd.cpu().numpy().view(np.uint32), res["dist"])
    assert np.array_equal(dpos.cpu().numpy().view(np.uint32)[:k], res["item_pos"])
    assert np.array_equal(drk.cpu().numpy()[:k], res["item_rank"])
    con.close()
