"""Inverse BWT layouts that the one-block and many-block forms share: head rows that fall on a splitter row, texts written to
unaligned device addresses with guard bytes around them, and the single-block consistency message.  Every entry
(inverse, inverse_device, inverse_many, inverse_many_device) is checked against the original text."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
STRIDE = 48  # the default splitter stride (DARK_BWT_IBWT_STRIDE): rows 0, 48, 96, ... start a walk
SENTINEL = 0xA5


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


def heads_on_splitters_single(oracle):
    """One-block (text, bwt, origin) whose head row origin + 1 is a splitter row, plus origin == 0 and origin == n - 1."""
    rng = np.random.default_rng(4801)
    found = []
    while len(found) < 4:  # about one text in 48 qualifies
        n = int(rng.integers(STRIDE, 6000))
        t = rng.integers(0, int(rng.choice([2, 4, 26, 256])), n).astype(np.uint8)
        b, o = oracle.bwt_forward(t)
        if (o + 1) % STRIDE == 0:
            found.append((t, b, o))
    low = rng.integers(1, 256, 1000).astype(np.uint8)
    low[0] = 0                                  # suffix 0 is the smallest: origin 0
    high = rng.integers(0, 255, 2 * STRIDE).astype(np.uint8)
    high[0] = 255                               # suffix 0 is the largest: origin n - 1, head row n on splitter 2
    for t, want in ((low, 0), (high, high.size - 1)):
        b, o = oracle.bwt_forward(t)
        assert o == want
        found.append((t, b, o))
    return found


def heads_on_splitters_many(oracle):
    """A block set in which every other block's head row starts[b] + b + origin_b + 1 is a multiple of the stride, among
    them an origin-0 block and an origin-(n_b - 1) block."""
    rng = np.random.default_rng(4802)
    blocks, first_row = [], 0  # first_row = starts[b] + b, the block's '$' row

    def add(t):
        nonlocal first_row
        b, o = oracle.bwt_forward(t) if t.size > 1 else (t.copy(), 0)
        blocks.append((t, b, o, (first_row + o + 1) % STRIDE == 0))
        first_row += t.size + 1

    for k in range(12):
        while True:
            t = rng.integers(0, int(rng.choice([2, 4, 256])), int(rng.integers(2, 3000))).astype(np.uint8)
            b, o = oracle.bwt_forward(t)
            if k % 2 or (first_row + o + 1) % STRIDE == 0:
                break
        add(t)
    n_fill = (STRIDE - 1 - first_row) % STRIDE + STRIDE - 1  # a filler that puts the next '$' row at 47 mod 48
    add(rng.integers(0, 4, n_fill).astype(np.uint8))
    low = rng.integers(1, 256, 700).astype(np.uint8)
    low[0] = 0                                  # origin 0: head row first_row + 1
    add(low)
    n_high = (-first_row) % STRIDE + STRIDE     # origin n - 1: head row first_row + n
    high = rng.integers(0, 255, n_high).astype(np.uint8)
    high[0] = 255
    add(high)
    assert blocks[-2][2] == 0 and blocks[-1][2] == n_high - 1
    assert sum(on for *_, on in blocks) >= 8
    return [(t, b, o) for t, b, o, _ in blocks]


def inverse_device(torch, con, bwt, origin):
    db = torch.from_numpy(bwt).cuda()
    dt = torch.empty(bwt.size, dtype=torch.uint8, device="cuda")
    con.inverse_device(db.data_ptr(), bwt.size, origin, dt.data_ptr())
    return dt.cpu().numpy()


def inverse_many_device(torch, con, pairs, d_text_ptr=None):
    starts = np.concatenate([[0], np.cumsum([b.size for b, _ in pairs])]).astype(np.uint32)
    db = torch.from_numpy(np.concatenate([b for b, _ in pairs])).cuda()
    ds = torch.from_numpy(starts.view(np.int32)).cuda()
    do = torch.tensor([o for _, o in pairs], dtype=torch.int64, device="cuda")
    dt = None
    if d_text_ptr is None:
        dt = torch.empty(int(starts[-1]), dtype=torch.uint8, device="cuda")
        d_text_ptr = dt.data_ptr()
    con.inverse_many_device(db.data_ptr(), ds.data_ptr(), do.data_ptr(), len(pairs), d_text_ptr)
    if dt is None:
        return None
    out = dt.cpu().numpy()
    return [out[starts[k]:starts[k + 1]] for k in range(len(pairs))]


def test_single_block_head_on_splitter(saca, oracle, torch):
    for t, b, o in heads_on_splitters_single(oracle):
        with saca.Constructor(t.size + 1) as con:
            assert np.array_equal(con.inverse(b, o), t), (t.size, o)
            assert np.array_equal(inverse_device(torch, con, b, o), t), (t.size, o)
            (many,) = con.inverse_many([(b, o)])
            assert np.array_equal(many, t), (t.size, o)
            (many,) = inverse_many_device(torch, con, [(b, o)])
            assert np.array_equal(many, t), (t.size, o)


def test_many_blocks_heads_on_splitters(saca, oracle, torch):
    blocks = heads_on_splitters_many(oracle)
    pairs = [(b, o) for _, b, o in blocks]
    with saca.Constructor(sum(t.size + 1 for t, _, _ in blocks)) as con:
        for k, (out, (t, _, _)) in enumerate(zip(con.inverse_many(pairs), blocks)):
            assert np.array_equal(out, t), k
        for k, (out, (t, _, _)) in enumerate(zip(inverse_many_device(torch, con, pairs), blocks)):
            assert np.array_equal(out, t), k
        for k, (t, b, o) in enumerate(blocks):
            assert np.array_equal(con.inverse(b, o), t), k
            assert np.array_equal(inverse_device(torch, con, b, o), t), k


def check_unaligned_outputs():
    """inverse_device and inverse_many_device into d_text + 1, + 2 and + 3 of a buffer filled with a sentinel: the text lands
    in [off, off + n) and no byte outside it changes.  Run in a fresh process so that the environment picks the walk."""
    import oracle
    import torch
    from dark_b200 import saca, synth
    singles = [synth.generate("mixed", 4, 300007), synth.generate("text", 3, 4099), np.array([7, 1, 7], np.uint8)]
    rng = np.random.default_rng(4803)
    many = [rng.integers(0, 256, s).astype(np.uint8) for s in (1, 2, 3, 5, 47, 48, 49, 1000, 4099)]
    many.append(synth.generate("dna", 2, 70001))
    many_pairs = [oracle.bwt_forward(t) if t.size > 1 else (t.copy(), 0) for t in many]
    many_text = np.concatenate(many)
    with saca.Constructor(max(300007, sum(t.size + 1 for t in many))) as con:
        for off in (1, 2, 3):
            for t in singles:
                b, o = oracle.bwt_forward(t)
                db = torch.from_numpy(b).cuda()
                buf = torch.full((t.size + 8,), SENTINEL, dtype=torch.uint8, device="cuda")
                con.inverse_device(db.data_ptr(), t.size, o, buf.data_ptr() + off)
                h = buf.cpu().numpy()
                assert np.array_equal(h[off:off + t.size], t), (off, t.size)
                assert (h[:off] == SENTINEL).all() and (h[off + t.size:] == SENTINEL).all(), (off, t.size)
            buf = torch.full((many_text.size + 8,), SENTINEL, dtype=torch.uint8, device="cuda")
            inverse_many_device(torch, con, many_pairs, buf.data_ptr() + off)
            h = buf.cpu().numpy()
            assert np.array_equal(h[off:off + many_text.size], many_text), off
            assert (h[:off] == SENTINEL).all() and (h[off + many_text.size:] == SENTINEL).all(), off


@pytest.mark.parametrize("env_extra", [{}, {"DARK_BWT_IBWT_TWO_WALKS": "1"}], ids=["stash", "two_walks"])
def test_unaligned_outputs_keep_guard_bytes(env_extra):
    code = "import sys; sys.path.insert(0, %r); import test_inverse_layouts as m; m.check_unaligned_outputs(); print('ok')" % HERE
    env = dict(os.environ, **env_extra)
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


def test_inconsistent_single_block_message(saca, oracle, torch):
    from dark_b200 import DarkBwtError, _ffi, synth
    t = synth.generate("text", 35, 9001)
    bwt, origin = oracle.bwt_forward(t)
    n = t.size
    with saca.Constructor(n + 1) as con:
        err = None
        for d in range(1, 200):  # an origin the inverse rejects (some wrong origins decode to another text)
            try:
                con.inverse(bwt, (origin + 97 * d) % n)
            except DarkBwtError as e:
                err = e
                break
        assert err is not None
        assert err.code == _ffi.E_INVALID_ARG
        m = re.search(r"is not a forward transform \(list covers (\d+) of (\d+) rows\)", str(err))
        assert m, str(err)
        assert int(m.group(2)) == n + 1 and 1 <= int(m.group(1)) <= n
        assert np.array_equal(con.inverse(bwt, origin), t)
