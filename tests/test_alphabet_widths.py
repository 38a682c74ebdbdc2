"""Every symbol width, on both sides of each packing boundary.

The number of distinct bytes in a block (sigma) decides which kernels run:
- single block (forward_device): s = max(1, bit_length(sigma - 1)) bits per symbol, K = 64 // s symbols per initial key.
  s in {1, 2, 4, 8} takes the packed key builder, the q-gram histograms and the key-generating pass, and only these widths
  can prune the initial sort.  s in {3, 5, 6, 7} takes the generic builder, whose keys leave 1 (s = 3, 7) or 4 (s = 5, 6)
  bits unused at the bottom, and is never pruned;
- many blocks (forward_many_device): s = bit_length(sigma) over the union alphabet (code 0 is "past the block's end");
- distance coding (k_dc_ranks): up to 32 symbols the last-occurrence table lives in registers, above 32 in shared memory;
  the many-block pass decides by the union alphabet.

Each generator is checked on the CPU to give exactly the sigma it is named for, and the oracle is cross-checked against the
reference's brute-force specification at every width.  Every GPU result is compared bit for bit with the CPU oracle, and
every GPU case also asserts through Constructor.stats that it took the path it is named for.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

PACKED = (1, 2, 4, 8)
COLLIDE_LIMIT = 1.5 / 256          # run_sort prunes only when every digit's collision rate is at most this
SIGMAS = [2, 3, 4, 5, 8, 9, 16, 17, 32, 33, 64, 65, 128, 129, 255, 256]
MANY_SIGMAS = [1, 3, 4, 7, 8, 15, 16, 31, 32, 63, 64, 127, 128, 255, 256]
DC_SIGMAS = [31, 32, 33, 34, 64, 128, 255]
N_SMALL = 5000
N_LARGE = (1 << 20) + 4099
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def single_width(sigma):
    return max(1, (sigma - 1).bit_length())


def many_width(sigma):
    return sigma.bit_length()


def uniform_prunes(sigma):
    """Whether sigma equiprobable symbols pass the pruning test: a digit holds 8 / s symbols, so two keys share it with
    probability sigma^(-8/s).  True for sigma = 2, 4, 16, 255, 256; false for 3, 9, 17, 129 and every generic width."""
    s = single_width(sigma)
    return s in PACKED and sigma ** (-8.0 / s) <= COLLIDE_LIMIT


# ---- generators -------------------------------------------------------------------------------------------------
def alphabet(sigma, seed):
    """`sigma` distinct bytes in ascending order, scattered over 0..255.  Even seeds include 0x00 and 0xFF; odd seeds take
    both sides of the 32-byte boundaries of k_build_lut's warp scan (31/32, 95/96, 159/160, 223/224) and, while sigma
    leaves room, neither 0x00 nor 0xFF."""
    if sigma == 256:
        return np.arange(256, dtype=np.uint8)
    rng = np.random.default_rng(1000 + seed)
    must = [0, 255] if seed % 2 == 0 else [31, 32, 95, 96, 159, 160, 223, 224]
    must = must[:sigma]
    banned = set(must) | ({0, 255} if seed % 2 and sigma <= 200 else set())
    rest = np.array([b for b in range(256) if b not in banned])
    pick = rng.choice(rest, sigma - len(must), replace=False)
    return np.sort(np.concatenate([must, pick])).astype(np.uint8)


def cover(t, alpha, rng):
    """Overwrite a few random positions with a permutation of the alphabet, so every symbol occurs."""
    pos = rng.choice(t.size, alpha.size, replace=False)
    t[pos] = rng.permutation(alpha)
    return t


def uniform(alpha, n, seed, planted=0):
    """Equiprobable symbols.  `planted` copies of one 400-byte segment leave a few hundred suffixes tied after round 0 (at
    most n/16), so round 1 reads its ranks off the sorted round-0 keys (k_build_keys_search) at every width."""
    rng = np.random.default_rng(seed)
    t = cover(alpha[rng.integers(0, alpha.size, n)], alpha, rng)
    for k in range(planted):
        at = int(rng.integers(2000, n - 400))
        t[at:at + 400] = t[1000:1400]
    return t


def skewed(alpha, n, seed):
    """Text-like: words of Zipf-distributed symbols from a 400-word vocabulary, words chosen with Zipf weights, separated
    by the most frequent symbol.  Every digit of the initial key collides far more often than 1.5/256."""
    rng = np.random.default_rng(seed)
    sigma = alpha.size
    by_rank = rng.permutation(alpha)                       # which byte is the most frequent is not tied to byte order
    p = 1.0 / np.arange(1, sigma + 1) ** 1.1
    p /= p.sum()
    vocab = [np.append(by_rank[rng.choice(sigma, int(rng.integers(2, 9)), p=p)], by_rank[0]) for _ in range(400)]
    q = 1.0 / np.arange(1, 401)
    q /= q.sum()
    words = rng.choice(400, n // 3 + 16, p=q)
    t = np.concatenate([vocab[w] for w in words])[:n].astype(np.uint8)
    assert t.size == n
    return cover(t, alpha, rng)


def end_edge(alpha, r, seed):
    """A random body, then r copies of the smallest byte: the last suffixes are runs of the smallest code, each a prefix
    of the next, around the length K of one initial key."""
    rng = np.random.default_rng(seed)
    body = cover(alpha[rng.integers(0, alpha.size, 1500 + alpha.size)], alpha, rng)
    return np.concatenate([body, np.full(r, alpha[0], np.uint8)])


def periodic(alpha, period, seed):
    """Every symbol once, then a body of period `period` (ending in a partial period): keys equal across shifts."""
    rng = np.random.default_rng(seed)
    unit = alpha[rng.integers(0, alpha.size, period)]
    reps = 4000 // period + 1
    return np.concatenate([rng.permutation(alpha), np.tile(unit, reps), unit[: period // 2 + 1]]).astype(np.uint8)


def eot_lengths(sigma):
    K = 64 // single_width(sigma)
    return [K - 2, K - 1, K, K + 1, 2 * K + 1]


def periods(sigma):
    K = 64 // single_width(sigma)
    return [K - 1, K, K + 1]


SHAPES = ["uniform_small", "uniform_large", "skewed", "end_of_text", "periodic"]


def shape_inputs(sigma, shape):
    """[(text, expect_pruned)] of one shape; expect_pruned None where the test does not predict it."""
    alpha = alphabet(sigma, sigma)
    s = single_width(sigma)
    if shape == "uniform_small":
        return [(uniform(alpha, N_SMALL, sigma), uniform_prunes(sigma))]
    if shape == "uniform_large":
        return [(uniform(alpha, N_LARGE + 2 * sigma, sigma + 1, planted=4), uniform_prunes(sigma))]
    if shape == "skewed":
        return [(skewed(alpha, N_LARGE + sigma, sigma + 2), False)]
    generic = None if s in PACKED else False
    if shape == "end_of_text":
        return [(end_edge(alpha, r, sigma + 3 + r), generic) for r in eot_lengths(sigma)]
    return [(periodic(alpha, p, sigma + 4 + p), generic) for p in periods(sigma)]


def digit_collisions(t, alpha):
    """The host's view of the initial sort (radix_sort.cuh k_scan_hist): per 8-bit digit of the MSB-aligned key of K dense
    codes, the probability that two keys share it."""
    s = single_width(alpha.size)
    K = 64 // s
    codes = np.searchsorted(alpha, t).astype(np.uint64)
    padded = np.concatenate([codes, np.zeros(K, np.uint64)])
    key = np.zeros(t.size, np.uint64)
    for c in range(K):
        key |= padded[c:c + t.size] << np.uint64(64 - s * (c + 1))
    out = []
    for p in range(8):
        cnt = np.bincount(((key >> np.uint64(8 * p)) & np.uint64(255)).astype(np.int64), minlength=256).astype(np.float64)
        out.append(float(((cnt / t.size) ** 2).sum()))
    return out


def prose(n, seed):
    """ASCII-like prose: a 30,000-word vocabulary (lower case, capitalised, numbers), words chosen with Zipf weights and
    joined by spaces and punctuation.  Built in 8 MiB pieces with one vocabulary, so the block repeats like text does."""
    rng = np.random.default_rng(seed)
    letters = np.frombuffer(b"etaoinshrdlcumwfgypbvkjxqz", np.uint8)
    lp = 1.0 / np.arange(1, 27) ** 0.9
    lp /= lp.sum()
    seps = [b" "] * 30 + [b", ", b". ", b"; ", b": ", b"!\n", b"?\n", b".\n\n", b" - ", b" (", b") ", b"\" ", b" '", b"' ",
                          b"/", b"[", b"] ", b"*", b"&", b"#", b"%", b"+", b"=", b"@", b"_", b"\t"]
    vocab = []
    for i in range(30000):
        r = rng.random()
        if r < 0.04:
            w = str(int(rng.integers(0, 100000))).encode()
        else:
            w = letters[rng.choice(26, int(rng.integers(1, 12)), p=lp)].tobytes()
            if r < 0.16:
                w = w.capitalize()
            elif r < 0.17:
                w = w.upper()
        vocab.append(w + seps[int(rng.integers(0, len(seps)))])
    flat = np.frombuffer(b"".join(vocab), np.uint8)
    lens = np.array([len(v) for v in vocab], np.int64)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]])
    q = 1.0 / np.arange(1, 30001) ** 1.05
    q /= q.sum()
    out = np.empty(n, np.uint8)
    filled = 0
    while filled < n:
        piece = min(8 << 20, n - filled)
        words = rng.choice(30000, piece // 2 + 64, p=q)
        wl = lens[words]
        ends = np.cumsum(wl)
        assert ends[-1] >= piece
        cut = int(np.searchsorted(ends, piece)) + 1
        words, wl, ends = words[:cut], wl[:cut], ends[:cut]
        idx = np.repeat(offs[words] - (ends - wl), wl) + np.arange(int(ends[-1]))
        out[filled:filled + piece] = flat[idx[:piece]]
        filled += piece
    return out


def large_width_inputs():
    """4-16 MiB blocks of other widths: (name, text, sigma, expect_pruned)."""
    rng = np.random.default_rng(77)
    b64 = np.frombuffer(b"ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/", np.uint8)
    base64 = b64[rng.integers(0, 64, 8 << 20)]
    lines = np.insert(base64, np.arange(76, base64.size, 76), 10)[: (8 << 20) + 33]     # 76-column lines: '\n' is a 65th symbol
    hexa = np.frombuffer(b"0123456789abcdef", np.uint8)[rng.integers(0, 16, (6 << 20) + 5)]
    eight = np.frombuffer(b"ACGTNRYK", np.uint8)[rng.integers(0, 8, (4 << 20) + 7)]
    binary = np.array([0, 255], np.uint8)[rng.integers(0, 2, (4 << 20) + 3)]
    return [("base64", base64, 64, False), ("base64_lines", lines, 65, False), ("hex", hexa, 16, True),
            ("eight_symbols", eight, 8, False), ("binary", binary, 2, True)]


def many_block_sets(sigma):
    """Block lists whose union alphabet has exactly `sigma` symbols."""
    alpha = alphabet(sigma, sigma + 5)
    rng = np.random.default_rng(500 + sigma)
    parts = np.array_split(rng.permutation(alpha), min(sigma, 6))
    disjoint = []
    for k, part in enumerate(parts):
        part = np.sort(part)
        n = int(rng.integers(max(2, part.size), 20000))
        disjoint.append(skewed(part, n, 600 + k) if part.size > 1 else np.full(n, part[0], np.uint8))
    one_symbol = [np.full(int(rng.integers(2, 300)), c, np.uint8) for c in rng.permutation(alpha)]
    block = uniform(alpha, max(2, sigma) + 2000, 700 + sigma)
    return {"disjoint": disjoint, "one_symbol": one_symbol, "identical": [block] * 5}


def dc_runs(alpha, n, seed):
    """BWT-like bytes over `alpha` (at least 3 symbols, n >= sigma + 3): Zipf symbols in runs of 1..8, every symbol once
    at the start.  The last symbol occurs only there, inside the first 4 KiB chunk, so every later chunk and scan group
    must carry its last occurrence; the second-to-last occurs once more, near the end."""
    rng = np.random.default_rng(seed)
    common, rare = alpha[:-1], alpha[-2]
    p = 1.0 / np.arange(1, common.size)
    p /= p.sum()
    t = np.repeat(common[rng.choice(common.size - 1, n, p=p)], rng.integers(1, 9, n))[:n].copy()   # never `rare`
    t[: alpha.size] = rng.permutation(alpha)
    t[n - 3] = rare
    return t


# ---- CPU: generators, width formulas and the oracle at every width --------------------------------------------------
def test_width_formulas():
    for sigma in range(1, 257):
        s = single_width(sigma)
        assert (1 << s) >= sigma and (s == 1 or (1 << (s - 1)) < sigma)
        assert (1 << many_width(sigma)) > sigma >= (1 << (many_width(sigma) - 1))
    assert [single_width(x) for x in SIGMAS] == [1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 8]
    assert [64 // single_width(x) for x in (5, 33, 65)] == [21, 10, 9]
    assert sorted({single_width(x) for x in SIGMAS}) == list(range(1, 9))
    assert sorted({many_width(x) for x in MANY_SIGMAS}) == list(range(1, 10))
    assert [x for x in SIGMAS if uniform_prunes(x)] == [2, 4, 16, 255, 256]
    for s in PACKED:   # uniform cases fall on both sides of the pruning threshold at every packed width but s = 1 (skewed covers it)
        side = {uniform_prunes(x) for x in SIGMAS if single_width(x) == s}
        assert side == ({True} if s == 1 else {True, False}), s


@pytest.mark.parametrize("sigma", SIGMAS)
def test_alphabets_and_shapes_have_their_sigma(sigma):
    alpha = alphabet(sigma, sigma)
    assert alpha.size == sigma and np.all(np.diff(alpha.astype(int)) > 0)
    if sigma % 2 == 0:
        assert alpha[0] == 0 and alpha[-1] == 255
    else:
        assert {31, 32} <= set(alpha.tolist()) or sigma < 2
        assert sigma > 200 or not ({0, 255} & set(alpha.tolist()))
    for shape in SHAPES:
        for t, _ in shape_inputs(sigma, shape):
            assert t.dtype == np.uint8
            assert np.array_equal(np.unique(t), alpha), (shape, sigma)


@pytest.mark.parametrize("sigma", SIGMAS)
def test_uniform_and_skewed_fall_on_their_side_of_the_pruning_threshold(sigma):
    """The collision rates the GPU's pruning decision reads, modelled on the host: the uniform bodies of packed widths are
    below 1.5/256 exactly when uniform_prunes() says so, the skewed ones clearly above (and generic widths never prune)."""
    alpha = alphabet(sigma, sigma)
    for shape in ("uniform_small", "skewed"):
        (t, expect), = shape_inputs(sigma, shape)
        worst = max(digit_collisions(t, alpha))
        if expect:
            assert worst < COLLIDE_LIMIT * 0.8, (shape, worst)
        else:
            assert worst > COLLIDE_LIMIT * 1.2, (shape, worst)


@pytest.mark.parametrize("sigma", MANY_SIGMAS)
def test_many_block_sets_have_their_union_sigma(sigma):
    for name, blocks in many_block_sets(sigma).items():
        assert all(b.size >= 2 and b.dtype == np.uint8 for b in blocks), name
        assert np.unique(np.concatenate(blocks)).size == sigma, name
        if name == "disjoint":
            sets = [set(np.unique(b).tolist()) for b in blocks]
            assert sum(len(x) for x in sets) == sigma
        if name == "one_symbol":
            assert all(np.unique(b).size == 1 for b in blocks)


@pytest.mark.parametrize("sigma", DC_SIGMAS)
def test_dc_inputs_have_their_sigma(sigma):
    alpha = alphabet(sigma, sigma)
    for n in (4095, 4096, 4097, 8193, (3 << 20) + 4097):
        t = dc_runs(alpha, n, n + sigma)
        assert t.size == n and np.unique(t).size == sigma, n
        last = np.flatnonzero(t == alpha[-1])
        assert last.size == 1 and last[0] < 4096
        assert np.count_nonzero(t == alpha[-2]) == 2 and t[n - 3] == alpha[-2]


def test_dc_many_sets_have_their_alphabets():
    sets = dc_many_alphabet_sets()
    for name, blocks in sets.items():
        union = np.unique(np.concatenate(blocks)).size
        per_block = max(np.unique(b).size for b in blocks)
        want = {"blocks_le_32_union_32": (32, 32), "blocks_le_32_union_33": (33, 32), "blocks_le_32_union_64_over_3_mib": (64, 32),
                "large_block_alphabets": (256, 256)}[name]
        assert union == want[0] and per_block <= want[1], (name, union, per_block)
    assert sum(b.size for b in sets["blocks_le_32_union_64_over_3_mib"]) > 3 << 20
    assert min(np.unique(b).size for b in sets["large_block_alphabets"][:12]) > 32


def test_large_inputs_have_their_sigma():
    for name, t, sigma, _ in large_width_inputs():
        assert np.unique(t).size == sigma, name
    t = prose(3 << 20, 5)
    sigma = np.unique(t).size
    assert 65 <= sigma <= 128 and single_width(sigma) == 7, sigma


@pytest.mark.parametrize("s", range(1, 9))
def test_oracle_matches_the_brute_force_specification_at_every_width(oracle, s):
    """oracle.saca against sort_direct (the reference's specification, saca.rs:25-35) at both ends of width s."""
    lo, hi = (1 << (s - 1)) + 1 if s > 1 else 1, 1 << s
    for sigma in sorted({lo, hi}):
        alpha = alphabet(sigma, sigma)
        texts = [uniform(alpha, 1900, sigma) if sigma > 1 else np.full(1900, 7, np.uint8), skewed(alpha, 2000, sigma) if sigma > 1
                 else np.full(7, 0, np.uint8)]
        if sigma > 1:
            texts += [end_edge(alpha, r, r)[-600:] for r in eot_lengths(sigma)]
            texts += [periodic(alpha, p, p) for p in periods(sigma)]
        for t in texts:
            t = np.ascontiguousarray(t)
            sa = oracle.saca(t)
            assert np.array_equal(sa, oracle.sort_direct(t)), (sigma, t.size)
            bwt, origin = oracle.bwt_emit(t, sa)
            assert np.array_equal(oracle.bwt_decode(bwt, origin), t)


# ---- GPU ------------------------------------------------------------------------------------------------------------
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


def _contexts(saca, cap):
    from dark_b200 import _ffi
    return saca.Constructor(cap), saca.Constructor(cap, flags=_ffi.F_NO_ALPHABET_PACKING)


@pytest.fixture(scope="module")
def cons_small(saca, torch):
    cs = _contexts(saca, 1 << 14)
    yield cs
    for c in cs:
        c.close()


@pytest.fixture(scope="module")
def cons_large(saca, torch):
    cs = _contexts(saca, N_LARGE + 1024)
    yield cs
    for c in cs:
        c.close()


def check_dc(res, b, oracle):
    dist, init, mtf, nu = oracle.dc_encode(b)
    pos, sd, sym, rk = oracle.dc_stream(b, dist, init)
    assert res["num_unique"] == nu and res["num_items"] == pos.size
    assert np.array_equal(res["init"], init)
    assert np.array_equal(res["mtf_symbols"][:nu], mtf[:nu])
    if res["dist"] is not None:
        assert np.array_equal(res["dist"], dist)
    assert np.array_equal(res["item_pos"], pos) and np.array_equal(res["item_dist"], sd)
    assert np.array_equal(res["item_sym"], sym) and np.array_equal(res["item_rank"], rk)
    assert np.array_equal(oracle.dc_decode(res["init"], res["item_dist"], b.size), b)


def check_single(cons, oracle, t, sigma, expect_pruned):
    """SA, BWT and origin equal the oracle with and without alphabet packing, on the path the case is named for; the
    inverse restores the text and distance coding of the BWT equals the oracle's."""
    con, canon = cons
    s = single_width(sigma)
    bwt_o, origin_o, sa_o = oracle.bwt_forward(t, want_sa=True)
    bwt, origin, sa = con.bwt_and_sa(t)
    st = con.stats
    assert (st.sigma, st.bits_per_symbol, st.symbols_per_key) == (sigma, s, 64 // s)
    pruned = st.initial_symbols < st.symbols_per_key
    if expect_pruned is not None:
        assert pruned == expect_pruned, (sigma, st.initial_symbols, st.symbols_per_key)
    assert origin == origin_o and np.array_equal(sa, sa_o) and np.array_equal(bwt, bwt_o)
    bwt2, origin2, sa2 = canon.bwt_and_sa(t)
    st = canon.stats
    assert (st.sigma, st.bits_per_symbol, st.symbols_per_key, st.initial_symbols) == (sigma, 8, 8, 8)
    assert origin2 == origin_o and np.array_equal(sa2, sa_o) and np.array_equal(bwt2, bwt_o)
    assert np.array_equal(con.inverse(bwt, origin), t)
    check_dc(con.dc_encode(bwt), bwt_o, oracle)
    return pruned


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("sigma", SIGMAS)
def test_single_block_every_width(oracle, cons_small, cons_large, sigma, shape):
    cons = cons_large if shape in ("uniform_large", "skewed") else cons_small
    for t, expect in shape_inputs(sigma, shape):
        check_single(cons, oracle, t, sigma, expect)


@pytest.mark.gpu
def test_realistic_prose_block_takes_the_large_block_paths(saca, oracle, torch):
    """ASCII-like prose, 100 MiB + 12,345 bytes, width 7 (sigma 65-128), device-resident with an SA output.  At this size
    every large-block path switches on by itself: the bucketed rank scatter (4n > 96 MiB), the fused round-0 sink
    (bucketed and an unpruned initial sort), windowed emission (n > 96 MiB, no inline emission without pruning) and the
    text-order key build in round 1 (it needs more than n/8 suffixes to survive round 0; on a B200 80 % of them did, with
    sigma = 87 and three doubling rounds)."""
    from dark_b200 import _ffi
    n = (100 << 20) + 12345
    t = prose(n, 2024)
    sigma = int(np.unique(t).size)
    assert 65 <= sigma <= 128
    con = saca.Constructor(n, flags=_ffi.F_DEVICE_ONLY)
    try:
        dt = torch.from_numpy(t).cuda()
        db = torch.empty(n, dtype=torch.uint8, device="cuda")
        ds = torch.empty(n, dtype=torch.int32, device="cuda")
        origin = con.bwt_device(dt.data_ptr(), n, db.data_ptr(), ds.data_ptr())
        st = con.stats.as_dict()
        assert (st["sigma"], st["bits_per_symbol"], st["symbols_per_key"], st["initial_symbols"]) == (sigma, 7, 9, 9)
        # the stats cannot show the bucketed scatter, the fused round-0 sink or windowed emission: they follow from n and
        # from the unpruned initial sort asserted above.  The text-order build also needs the survivors of round 0:
        assert st["rounds"] >= 1 and st["active"][1] * 8 > n
        print("prose: sigma %d, round-0 survivors %.1f %%, rounds %d" % (sigma, 100.0 * st["active"][1] / n, st["rounds"]))
        assert con.verify_sa_device(dt.data_ptr(), n, ds.data_ptr()) == 0
        bwt_o, origin_o, sa_o = oracle.bwt_forward(t, want_sa=True)
        assert origin == origin_o
        assert np.array_equal(db.cpu().numpy(), bwt_o)
        assert np.array_equal(ds.cpu().numpy().view(np.uint32), sa_o)
        del sa_o
        back = torch.zeros(n, dtype=torch.uint8, device="cuda")
        con.inverse_device(db.data_ptr(), n, origin, back.data_ptr())
        assert torch.equal(back, dt)
    finally:
        con.close()


@pytest.mark.gpu
def test_large_blocks_of_other_widths(saca, oracle, torch):
    """base64 (sigma 64, width 6) and base64 in 76-column lines (sigma 65, width 7), hex (pruned width 4), 8 symbols
    (width 3) and binary (pruned width 1), 4-8 MiB each."""
    inputs = large_width_inputs()
    with saca.Constructor(max(t.size for _, t, _, _ in inputs)) as con:
        for name, t, sigma, expect_pruned in inputs:
            s = single_width(sigma)
            bwt, origin, sa = con.bwt_and_sa(t)
            st = con.stats
            assert (st.sigma, st.bits_per_symbol, st.symbols_per_key) == (sigma, s, 64 // s), name
            assert (st.initial_symbols < st.symbols_per_key) == expect_pruned, name
            bwt_o, origin_o, sa_o = oracle.bwt_forward(t, want_sa=True)
            assert origin == origin_o and np.array_equal(sa, sa_o) and np.array_equal(bwt, bwt_o), name
            assert np.array_equal(con.inverse(bwt, origin), t), name


FORCED_KNOBS = [
    # each knob only changes what runs when the block reaches its path: the bucketed scatter, the fused round-0 sink and
    # the text-order key build need many suffixes to survive round 0 (the subprocess asserts more than n/8), and windowed
    # emission needs n > 1.5 x the window (emit() in dark_bwt.cu), so the blocks are N_FORCED > 1.5 MiB for a 1 MiB window
    {"DARK_BWT_BUCKETED": "1"},                                  # bucketed rank scatter
    {"DARK_BWT_EMIT_WINDOW_MB": "1"},                            # windowed emission: n > 1.5 MiB
    {"DARK_BWT_FORCE_U64_STATUS": "1"},                          # 64-bit tile status
    {"DARK_BWT_PASS_IMPL": "0"},                                 # the round-1 pass kernel
    {"DARK_BWT_PAIRS": "0"},                                     # no pairs mode
    {"DARK_BWT_TEXT_BUILD": "0"},                                # rank gathers only, isa[] untagged
    {"DARK_BWT_TEXT_BUILD": "1000000"},                          # text-order key build in every round
    {"DARK_BWT_FUSE_ROUND0": "0", "DARK_BWT_BUCKETED": "1"},     # round 0 followed by separate partition passes
]
GENERIC_SIGMAS = [8, 64, 128]   # widths 3, 6, 7
N_FORCED = (2 << 20) + 4099
EMIT_WINDOW = 1 << 20           # DARK_BWT_EMIT_WINDOW_MB=1


@pytest.fixture(scope="module")
def generic_cases(oracle, tmp_path_factory):
    """Skewed (text-like) bodies of widths 3, 6 and 7, about 2 MiB each, and their oracle results, saved for the knob
    subprocesses."""
    d = tmp_path_factory.mktemp("generic_widths")
    for sigma in GENERIC_SIGMAS:
        t = skewed(alphabet(sigma, sigma), N_FORCED + sigma, sigma + 9)
        assert t.size > EMIT_WINDOW + EMIT_WINDOW // 2
        bwt, origin, sa = oracle.bwt_forward(t, want_sa=True)
        np.savez(d / f"w{sigma}.npz", text=t, bwt=bwt, sa=sa, origin=np.uint64(origin))
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(len(FORCED_KNOBS)))
def test_forced_large_block_paths_at_generic_widths(generic_cases, idx):
    """The large-block paths, forced on ~2 MiB blocks by the same knobs as test_gpu_parity's FORCED_PATHS, at widths 3, 6
    and 7: one fresh process per knob set, running all three widths."""
    code = (
        "import sys, numpy as np\n"
        "from dark_b200 import saca\n"
        "for sigma in (%s):\n"
        "    z = np.load(sys.argv[1] + '/w%%d.npz' %% sigma)\n"
        "    t = z['text']\n"
        "    with saca.Constructor(t.size) as c:\n"
        "        b, o, s = c.bwt_and_sa(t)\n"
        "        st = c.stats\n"
        "    width = max(1, (sigma - 1).bit_length())\n"
        "    assert (st.sigma, st.bits_per_symbol, st.initial_symbols) == (sigma, width, 64 // width), sigma\n"
        "    assert st.rounds >= 1 and st.active[1] * 8 > t.size, (sigma, st.active[1])\n"
        "    assert o == int(z['origin']) and np.array_equal(b, z['bwt']) and np.array_equal(s, z['sa']), sigma\n"
        "print('ok')\n") % ", ".join(str(x) for x in GENERIC_SIGMAS)
    env = dict(os.environ, **FORCED_KNOBS[idx])
    out = subprocess.run([sys.executable, "-c", code, str(generic_cases)], env=env, cwd=REPO, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


@pytest.fixture(scope="module")
def con_many(saca, torch):
    c = saca.Constructor(1 << 20)
    yield c
    c.close()


def check_many(con, oracle, blocks, sigma):
    """forward_many, inverse_many, dc_encode_many and forward_dc_many of `blocks`, every block against the oracle."""
    s = many_width(sigma)
    res = con.bwt_many(blocks)
    st = con.stats
    assert (st.sigma, st.bits_per_symbol, st.symbols_per_key) == (sigma, s, 64 // s)
    expect = [oracle.bwt_forward(b) for b in blocks]
    for k, ((bwt, origin), (bwt_o, origin_o)) in enumerate(zip(res, expect)):
        assert origin == origin_o and np.array_equal(bwt, bwt_o), k
    back = con.inverse_many([(b, o) for b, o in expect])
    assert all(np.array_equal(x, t) for x, t in zip(back, blocks))
    for (bwt_o, _), r in zip(expect, con.dc_encode_many([b for b, _ in expect])):
        check_dc(r, bwt_o, oracle)
    fused = con.bwt_dc_many(blocks)
    assert con.stats.bits_per_symbol == s
    for k, ((bwt, origin, r), (bwt_o, origin_o)) in enumerate(zip(fused, expect)):
        assert origin == origin_o and np.array_equal(bwt, bwt_o), k
        check_dc(r, bwt_o, oracle)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["disjoint", "one_symbol", "identical"])
@pytest.mark.parametrize("sigma", MANY_SIGMAS)
def test_many_blocks_every_width(oracle, con_many, sigma, name):
    check_many(con_many, oracle, many_block_sets(sigma)[name], sigma)


@pytest.mark.gpu
@pytest.mark.parametrize("sigma", [64, 128])
def test_many_blocks_large_set(saca, oracle, torch, sigma):
    """64 blocks of 64 KiB over one alphabet: sigma 128 fills all 64 key bits with eight 8-bit codes; sigma 64 is width 7."""
    alpha = alphabet(sigma, sigma + 7)
    blocks = [skewed(alpha, 1 << 16, 800 + k) if k % 2 else uniform(alpha, 1 << 16, 800 + k) for k in range(64)]
    with saca.Constructor((64 << 16) + 64) as con:
        check_many(con, oracle, blocks, sigma)


@pytest.fixture(scope="module")
def con_dc(saca, torch):
    c = saca.Constructor(6 << 20)
    yield c
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("sigma", DC_SIGMAS)
def test_dc_register_and_shared_tables(oracle, torch, con_dc, sigma):
    """Alphabets around the 32-symbol switch of k_dc_ranks, over several 256-chunk scan groups and around one 4 KiB chunk,
    through dc_encode, dc_encode_device and dc_encode_many (each block also against a single call)."""
    alpha = alphabet(sigma, sigma)
    blocks = [dc_runs(alpha, n, n + sigma) for n in (4095, 4096, 4097, 8193, (3 << 20) + 4097)]
    singles = []
    for b in blocks:
        r = con_dc.dc_encode(b)
        assert r["num_unique"] == sigma
        check_dc(r, b, oracle)
        singles.append(r)
    b = blocks[-1]
    n = b.size
    dist, init, _, _ = oracle.dc_encode(b)
    pos, sd, sym, rk = oracle.dc_stream(b, dist, init)
    db = torch.from_numpy(b).cuda()
    dd = torch.empty(n, dtype=torch.int32, device="cuda")
    dpos, ddist = torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.int32, device="cuda")
    dsym, drk = torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")
    info = con_dc.dc_encode_device(db.data_ptr(), n, dd.data_ptr(), dpos.data_ptr(), ddist.data_ptr(), dsym.data_ptr(), drk.data_ptr())
    k = int(info.num_items)
    assert k == pos.size and int(info.num_unique) == sigma
    assert np.array_equal(np.array(list(info.init), np.uint64), init)
    assert np.array_equal(dd.cpu().numpy().view(np.uint32), dist)
    assert np.array_equal(dpos.cpu().numpy().view(np.uint32)[:k], pos) and np.array_equal(ddist.cpu().numpy().view(np.uint32)[:k], sd)
    assert np.array_equal(dsym.cpu().numpy()[:k], sym) and np.array_equal(drk.cpu().numpy()[:k], rk)
    for r, single, blk in zip(con_dc.dc_encode_many(blocks), singles, blocks):
        check_dc(r, blk, oracle)
        for f in ("dist", "init", "num_items", "item_pos", "item_dist", "item_sym", "item_rank"):
            assert np.array_equal(np.asarray(r[f]), np.asarray(single[f])), f


def dc_many_alphabet_sets():
    """Per-block alphabets against the union alphabet, which decides the table of the many-block pass."""
    rng = np.random.default_rng(91)
    a32, a33, a64, a256 = alphabet(32, 32), alphabet(33, 33), alphabet(64, 64), alphabet(256, 256)

    def blocks_over(union, per_block, sizes, seed):
        out = []
        for k, n in enumerate(sizes):
            sub = np.sort(np.random.default_rng(seed + k).choice(union, per_block, replace=False))
            out.append(dc_runs(sub, max(int(n), per_block + 3), seed + k))
        covered = np.unique(np.concatenate(out))
        missing = np.setdiff1d(union, covered)
        if missing.size:
            out.append(np.repeat(missing, 3))
        return out

    sizes = rng.integers(1, 70_000, 30)
    return {
        "blocks_le_32_union_32": blocks_over(a32, 12, sizes, 100),
        "blocks_le_32_union_33": blocks_over(a33, 32, sizes, 200),
        "blocks_le_32_union_64_over_3_mib": blocks_over(a64, 20, list(sizes) + [(3 << 20) + 11], 300),
        "large_block_alphabets": blocks_over(a256, 200, sizes[:12], 400) + blocks_over(a64, 40, sizes[:6], 500)
        + [dc_runs(a33, 5000, 600), dc_runs(a32, 4097, 601)],
    }


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["blocks_le_32_union_32", "blocks_le_32_union_33", "blocks_le_32_union_64_over_3_mib",
                                  "large_block_alphabets"])
def test_dc_many_union_alphabet(oracle, con_dc, name):
    blocks = dc_many_alphabet_sets()[name]
    union = np.unique(np.concatenate(blocks)).size
    assert union == {"blocks_le_32_union_32": 32, "blocks_le_32_union_33": 33}.get(name, union)
    if name.startswith("blocks_le_32"):
        assert max(np.unique(b).size for b in blocks) <= 32
    res = con_dc.dc_encode_many(blocks)
    for k, (b, r) in enumerate(zip(blocks, res)):
        check_dc(r, b, oracle)
        single = con_dc.dc_encode(b)
        for f in ("dist", "init", "num_items", "item_pos", "item_dist", "item_sym", "item_rank"):
            assert np.array_equal(np.asarray(r[f]), np.asarray(single[f])), (k, f)
