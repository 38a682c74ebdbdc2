"""Pipelined forward BWT + distance coding over a run of host blocks: dark_bwt_forward_dc_batch.  Every block must give
exactly what a dark_bwt_forward_dc call on it alone gives (and what the CPU oracle gives), whatever the mix of block
sizes, which outputs are asked for and where the host buffers live."""
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
from test_dc_many import FIELDS, check_against_oracle, same_result  # noqa: E402

OUTPUTS = ("bwt", "dist", "item_pos", "item_dist", "item_sym", "item_rank")  # the argument order of the entry


# ---- CPU: export, flag and argument checks (no device work) ------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from dark_b200 import _ffi
    if not os.path.exists(_ffi.lib_path()):
        _ffi.build_native()
    return _ffi.lib()


def test_entry_and_flag_are_exported(lib):
    from dark_b200 import _ffi
    assert "dark_bwt_forward_dc_batch" in _ffi.SYMBOLS and hasattr(lib, "dark_bwt_forward_dc_batch")
    header = open(os.path.join(ROOT, "include", "dark_bwt.h")).read()
    assert re.search(r"#define DARK_BWT_F_DC_BATCH 4u\b", header) and _ffi.F_DC_BATCH == 4


def test_bad_arguments_are_rejected_before_any_device_work(lib):
    """A null context or required pointer is DARK_BWT_E_INVALID_ARG without touching CUDA, whatever the count."""
    from dark_b200 import _ffi
    p = (ctypes.c_void_p * 1)(1)
    ns = (ctypes.c_uint64 * 1)(10)
    origins = (ctypes.c_uint64 * 1)()
    info = (_ffi.DcInfo * 1)()
    for count in (0, 1, 3):
        assert lib.dark_bwt_forward_dc_batch(None, None, None, count, *([None] * 8), None) == _ffi.E_INVALID_ARG
        assert lib.dark_bwt_forward_dc_batch(None, p, ns, count, None, origins, *([None] * 5), info, None) == _ffi.E_INVALID_ARG
        assert lib.dark_bwt_forward_dc_batch(None, p, ns, count, *([p] * 1), origins, *([p] * 5), info, None) == _ffi.E_INVALID_ARG


def test_create_rejects_dc_batch_with_device_only(lib):
    """DARK_BWT_F_DC_BATCH | DARK_BWT_F_DEVICE_ONLY is refused by the flag check, before any CUDA call."""
    from dark_b200 import _ffi
    out = ctypes.c_void_p(1)
    assert lib.dark_bwt_create_ex(1 << 20, 0, _ffi.F_DC_BATCH | _ffi.F_DEVICE_ONLY, ctypes.byref(out)) == _ffi.E_INVALID_ARG
    assert not out.value
    out = ctypes.c_void_p(1)
    flags = _ffi.F_DC_BATCH | _ffi.F_DEVICE_ONLY | _ffi.F_NO_ALPHABET_PACKING
    assert lib.dark_bwt_create_ex(1 << 20, 0, flags, ctypes.byref(out)) == _ffi.E_INVALID_ARG
    assert lib.dark_bwt_create_ex(1 << 20, 0, 8, ctypes.byref(out)) == _ffi.E_INVALID_ARG  # still no unknown flag


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


def ragged_blocks():
    """Twelve blocks: every generator, n = 2, one symbol, all 256 symbols, and blocks of 64 KiB or less (their DC borrows
    the sort's status buffer, which the next block's forward must clear) next to blocks of more than 1 MiB."""
    from dark_b200 import synth
    rng = np.random.default_rng(53)
    return [synth.generate("dna", 5, (1 << 21) + 3), synth.generate("text", 6, 40_000), synth.generate("mixed", 7, (1 << 20) + 11),
            np.array([3, 1], np.uint8), np.full(100_000, 65, np.uint8), rng.integers(0, 256, 300_000).astype(np.uint8),
            synth.generate("rep17", 8, 65_536), synth.generate("text", 10, 1 << 21), synth.generate("dna", 9, 5000),
            synth.generate("mixed", 11, 65_537), synth.generate("rep17", 12, 1_500_000), synth.generate("text", 13, 2)]


CAP = (1 << 21) + 3


@pytest.fixture(scope="module")
def reference(saca, torch):
    """Per-block bwt_dc on a context without the flag, with each block's stats."""
    blocks = ragged_blocks()
    out = []
    with saca.Constructor(CAP) as con:
        for t in blocks:
            b, o, r = con.bwt_dc(t)
            out.append((b, o, r, con.stats.as_dict()))
    return blocks, out


def same_block(got, ref, k):
    b, o, r = got
    rb, ro, rr = ref[:3]
    assert o == ro, k
    if b is not None:
        assert np.array_equal(b, rb), k
    same_result(r, rr)
    assert r["device_ms"] > 0


def untimed(st):
    return {k: v for k, v in st.items() if not k.endswith("_ms")}


@pytest.mark.gpu
def test_ragged_batch_equals_single_calls_and_oracle(saca, oracle, torch, reference):
    from dark_b200 import _ffi
    blocks, ref = reference
    with saca.Constructor(CAP, flags=_ffi.F_DC_BATCH) as con:
        res = con.bwt_dc_blocks(blocks)
        assert len(res) == len(blocks)
        for k, (t, got) in enumerate(zip(blocks, res)):
            same_block(got, ref[k], k)
            bwt_o, origin_o = oracle.bwt_forward(t)
            assert got[1] == origin_o and np.array_equal(got[0], bwt_o), k
            check_against_oracle(got[2], bwt_o, oracle)
        # the reference's path: items only, no BWT and no distances cross PCIe; stats as forward_dc reports them
        ns = [t.size for t in blocks]
        items = [[np.zeros(n, dt) for n in ns] for dt in (np.uint32, np.uint32, np.uint8, np.uint8)]
        origins, infos, stats = con.bwt_dc_batch_into([t.ctypes.data for t in blocks], ns, None, None,
                                                      *[[a.ctypes.data for a in arrs] for arrs in items], want_stats=True)
        for k in range(len(blocks)):
            m = ref[k][2]["num_items"]
            assert origins[k] == ref[k][1] and int(infos[k].num_items) == m, k
            for arrs, f in zip(items, FIELDS[5:]):
                assert np.array_equal(arrs[k][:m], ref[k][2][f]), (k, f)
            assert untimed(stats[k]) == untimed(ref[k][3]), k


@pytest.mark.gpu
@pytest.mark.parametrize("count", [1, 2, 3, 5])
def test_slot_alternation(saca, torch, reference, count):
    """Batches of 1, 2, 3 and 5 blocks: the last block lands in either slot, a slot is reused one or two times."""
    from dark_b200 import _ffi
    blocks, ref = reference
    pick = [0, 1, 4, 6, 7][:count] if count == 5 else list(range(count))
    with saca.Constructor(CAP, flags=_ffi.F_DC_BATCH) as con:
        for rep in range(2):
            for k, got in zip(pick, con.bwt_dc_blocks([blocks[i] for i in pick], want_dist=rep == 0)):
                same_block(got, ref[k], k)


@pytest.mark.gpu
def test_each_output_null(saca, torch, reference):
    """Each output array left null in turn, then a single entry of it: the other outputs are unchanged, the buffer of the
    null entry is not written."""
    from dark_b200 import _ffi
    blocks, ref = reference
    pick = [1, 0, 3, 2, 6]
    ts = [blocks[i] for i in pick]
    ns = [t.size for t in ts]
    dtypes = (np.uint8, np.uint32, np.uint32, np.uint32, np.uint8, np.uint8)
    with saca.Constructor(CAP, flags=_ffi.F_DC_BATCH) as con:
        for which in range(len(OUTPUTS)):
            for single in (False, True):
                arrays = [[np.zeros(n, dt) for n in ns] for dt in dtypes]
                ptrs = [[a.ctypes.data for a in arrs] for arrs in arrays]
                if single:
                    ptrs[which][1] = None
                else:
                    ptrs[which] = None
                origins, infos = con.bwt_dc_batch_into([t.ctypes.data for t in ts], ns, *ptrs)
                for j, k in enumerate(pick):
                    rb, ro, rr = ref[k][:3]
                    m = rr["num_items"]
                    assert origins[j] == ro and int(infos[j].num_items) == m
                    assert np.array_equal(np.array(list(infos[j].init), np.uint64), rr["init"])
                    want = [rb, rr["dist"], rr["item_pos"], rr["item_dist"], rr["item_sym"], rr["item_rank"]]
                    for o in range(len(OUTPUTS)):
                        got = arrays[o][j] if o < 2 else arrays[o][j][:m]
                        if o == which and (not single or j == 1):
                            assert not arrays[o][j].any(), (OUTPUTS[o], single, j)
                        else:
                            assert np.array_equal(got, want[o]), (OUTPUTS[which], single, OUTPUTS[o], j)


@pytest.mark.gpu
@pytest.mark.parametrize("threads", ["0", "3"])
def test_pinned_and_pageable_buffers(threads):
    """Pageable buffers of 1 MiB or more (through the staging lanes, or the driver's own staging with 0 lanes), pinned
    buffers, and a mix of both in one block's outputs give what single forward_dc calls give."""
    code = (
        "import numpy as np, torch\n"
        "from dark_b200 import saca, synth, _ffi\n"
        "blocks = [synth.generate('mixed', 31, 3 * (1 << 20) + 12345), synth.generate('dna', 32, 5000),\n"
        "          synth.generate('text', 33, (1 << 21) + 7), synth.generate('rep17', 34, 1 << 20)]\n"
        "ns = [t.size for t in blocks]\n"
        "cap = max(ns)\n"
        "with saca.Constructor(cap) as c:\n"
        "    ref = [c.bwt_dc(t) for t in blocks]\n"
        "def same(got, k):\n"
        "    b, o, r = got\n"
        "    rb, ro, rr = ref[k]\n"
        "    assert o == ro and np.array_equal(b, rb), k\n"
        "    for f in ('dist', 'num_items', 'item_pos', 'item_dist', 'item_sym', 'item_rank', 'init', 'num_unique'):\n"
        "        assert np.array_equal(np.asarray(r[f]), np.asarray(rr[f])), (k, f)\n"
        "with saca.Constructor(cap, flags=_ffi.F_DC_BATCH) as c:\n"
        "    for k, got in enumerate(c.bwt_dc_blocks(blocks)):\n"                       # pageable in and out
        "        same(got, k)\n"
        "    pin = lambda n, dt: torch.empty(n, dtype=dt).pin_memory()\n"
        "    tx = [torch.from_numpy(t).pin_memory() for t in blocks]\n"
        "    for mixed in (False, True):\n"                                            # pinned; then pageable BWT + distances
        "        bw = [np.empty(n, np.uint8) if mixed else pin(n, torch.uint8) for n in ns]\n"
        "        di = [np.empty(n, np.uint32) if mixed else pin(n, torch.int32) for n in ns]\n"
        "        it = [[pin(n, dt) for n in ns] for dt in (torch.int32, torch.int32, torch.uint8, torch.uint8)]\n"
        "        ptr = lambda a: a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr()\n"
        "        origins, infos = c.bwt_dc_batch_into([t.data_ptr() for t in tx], ns, [ptr(a) for a in bw], [ptr(a) for a in di],\n"
        "                                             *[[ptr(a) for a in arrs] for arrs in it])\n"
        "        for k in range(len(blocks)):\n"
        "            m = int(infos[k].num_items)\n"
        "            h = lambda a, dt: a if isinstance(a, np.ndarray) else a.numpy().view(dt)\n"
        "            r = {'dist': h(di[k], np.uint32), 'num_items': m, 'item_pos': h(it[0][k], np.uint32)[:m],\n"
        "                 'item_dist': h(it[1][k], np.uint32)[:m], 'item_sym': h(it[2][k], np.uint8)[:m], 'item_rank': h(it[3][k], np.uint8)[:m],\n"
        "                 'init': np.array(list(infos[k].init), np.uint64), 'num_unique': int(infos[k].num_unique)}\n"
        "            same((h(bw[k], np.uint8), origins[k], r), k)\n"
        "print('ok')\n")
    env = dict(os.environ, DARK_BWT_HOST_THREADS=threads)
    out = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


@pytest.mark.gpu
def test_forward_batch_suffix_arrays_through_the_copy_list(saca, oracle, torch):
    """dark_bwt_forward_batch with SA outputs (a copy that must finish before the next block reuses the SA buffer), pinned
    and pageable, with some SA entries left null."""
    from dark_b200 import _ffi, synth
    blocks = [synth.generate("mixed", 61, (1 << 21) - 5), synth.generate("dna", 62, 3000), synth.generate("text", 63, 1 << 20)]
    ns = [t.size for t in blocks]
    ref = [oracle.bwt_forward(t, want_sa=True) for t in blocks]
    with saca.Constructor(max(ns)) as con:
        L, ctx = con._L, con._ctx
        for pinned in (False, True):
            alloc = (lambda n, dt: torch.zeros(n, dtype=dt).pin_memory()) if pinned else (lambda n, dt: np.zeros(n, {torch.uint8: np.uint8, torch.int32: np.uint32}[dt]))
            ptr = (lambda a: a.data_ptr()) if pinned else (lambda a: a.ctypes.data)
            host = (lambda a, dt: a.numpy().view(dt)) if pinned else (lambda a, dt: a)
            bw = [alloc(n, torch.uint8) for n in ns]
            sa = [alloc(n, torch.int32) for n in ns]
            sp = [ptr(a) for a in sa]
            sp[1] = None
            cnt = len(blocks)
            O = (ctypes.c_uint64 * cnt)()
            _ffi.check(L.dark_bwt_forward_batch(ctx, (ctypes.c_void_p * cnt)(*[t.ctypes.data for t in blocks]), (ctypes.c_uint64 * cnt)(*ns),
                                                (ctypes.c_void_p * cnt)(*[ptr(a) for a in bw]), O, (ctypes.c_void_p * cnt)(*sp), cnt, None),
                       ctx, "forward_batch")
            for k, (rb, ro, rs) in enumerate(ref):
                assert int(O[k]) == ro and np.array_equal(host(bw[k], np.uint8), rb), (pinned, k)
                if k == 1:
                    assert not host(sa[k], np.uint32).any()
                else:
                    assert np.array_equal(host(sa[k], np.uint32), rs), (pinned, k)


@pytest.mark.gpu
def test_rejections_leave_the_context_usable(saca, torch, reference):
    from dark_b200 import _ffi
    blocks, ref = reference
    small = [blocks[1], blocks[3], blocks[8]]

    def code(call):
        with pytest.raises(_ffi.DarkBwtError) as e:
            call()
        return e.value.code

    with saca.Constructor(CAP) as con:                                           # no DC slots
        assert code(lambda: con.bwt_dc_blocks(small)) == _ffi.E_INVALID_ARG
        same_block(con.bwt_dc(blocks[1]), ref[1], 1)
    with saca.Constructor(CAP, flags=_ffi.F_DEVICE_ONLY) as con:                  # no staging either
        assert code(lambda: con.bwt_dc_blocks(small)) == _ffi.E_INVALID_ARG
    with pytest.raises(_ffi.DarkBwtError) as e:
        saca.Constructor(CAP, flags=_ffi.F_DC_BATCH | _ffi.F_DEVICE_ONLY)
    assert e.value.code == _ffi.E_INVALID_ARG
    with saca.Constructor(CAP, flags=_ffi.F_DC_BATCH) as con:
        assert con.bwt_dc_blocks([]) == []
        for bad, want in (([small[0], b"x", small[2]], _ffi.E_INVALID_N), ([small[0], np.zeros(CAP + 1, np.uint8), small[2]], _ffi.E_INVALID_N)):
            ts = [np.frombuffer(bytes(t), np.uint8) if isinstance(t, bytes) else t for t in bad]
            outs = [np.zeros(max(t.size, 1), np.uint8) for t in ts]
            with pytest.raises(_ffi.DarkBwtError) as e:
                con.bwt_dc_batch_into([t.ctypes.data for t in ts], [t.size for t in ts], [o.ctypes.data for o in outs])
            assert e.value.code == want
            assert not any(o.any() for o in outs)                              # nothing ran, not even block 0
        L, ctx = con._L, con._ctx
        cnt = len(small)
        T = (ctypes.c_void_p * cnt)(*[t.ctypes.data for t in small])
        T_null = (ctypes.c_void_p * cnt)(small[0].ctypes.data, None, small[2].ctypes.data)
        N = (ctypes.c_uint64 * cnt)(*[t.size for t in small])
        O = (ctypes.c_uint64 * cnt)()
        I = (_ffi.DcInfo * cnt)()
        nulls = [None] * 6
        assert L.dark_bwt_forward_dc_batch(ctx, T_null, N, cnt, *nulls[:1], O, *nulls[1:], I, None) == _ffi.E_INVALID_ARG
        assert L.dark_bwt_forward_dc_batch(ctx, T, N, cnt, *nulls[:1], None, *nulls[1:], I, None) == _ffi.E_INVALID_ARG
        assert L.dark_bwt_forward_dc_batch(ctx, T, N, cnt, *nulls[:1], O, *nulls[1:], None, None) == _ffi.E_INVALID_ARG
        assert L.dark_bwt_forward_dc_batch(ctx, T, None, cnt, *nulls[:1], O, *nulls[1:], I, None) == _ffi.E_INVALID_ARG
        for k, got in zip((1, 3, 8), con.bwt_dc_blocks(small)):
            same_block(got, ref[k], k)


@pytest.mark.gpu
def test_interleaved_with_the_other_entries(saca, torch, reference):
    """forward_dc_batch, forward_batch, forward_dc, forward_dc_many and forward_dc_batch again on one context."""
    from dark_b200 import _ffi
    blocks, ref = reference
    batch = [blocks[i] for i in (0, 2, 1, 9)]                                   # ends on a small block: the status buffer is dirty
    many = [blocks[i] for i in (1, 3, 8, 11)]
    with saca.Constructor(CAP, flags=_ffi.F_DC_BATCH) as con:
        for _ in range(2):
            for k, got in zip((0, 2, 1, 9), con.bwt_dc_blocks(batch)):
                same_block(got, ref[k], k)
            for k, (b, o) in zip((0, 2, 1, 9), con.bwt_blocks(batch)):
                assert o == ref[k][1] and np.array_equal(b, ref[k][0]), k
            same_block(con.bwt_dc(blocks[6]), ref[6], 6)
            for k, got in zip((1, 3, 8, 11), con.bwt_dc_many(many)):
                same_block(got, ref[k], k)


@pytest.mark.gpu
def test_full_size_blocks(saca, torch):
    """Three 256 MiB blocks (C2, a C5 block, C2 again) through one batch equal three bwt_dc calls."""
    from dark_b200 import _ffi, synth
    n = 1 << 28
    c2 = synth.generate("dna", 1, n)
    blocks = [c2, synth.generate(*synth.c5_block(0)), c2]
    with saca.Constructor(n, flags=_ffi.F_DC_BATCH) as con:
        res = con.bwt_dc_blocks(blocks)
        for k, t in enumerate(blocks):
            b, o, r = con.bwt_dc(t)
            same_block(res[k], (b, o, r), k)
            del b, r
