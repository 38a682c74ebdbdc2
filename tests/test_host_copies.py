"""Host-buffer copies of the single-call and many-block entries with pageable buffers of 1 MiB or more: dark_bwt_dc_encode,
dark_bwt_dc_encode_many, dark_bwt_forward_dc_many, dark_bwt_forward_dc with each output left null in turn,
dark_bwt_forward_dc_packed and dark_bwt_forward_dc_packed_many, and dark_bwt_forward_many and dark_bwt_inverse_many on blocks
on both sides of the 1 MiB staging threshold.  Every call gives what the CPU oracle gives, and the calls that run twice give
it on pageable and on pinned buffers, for each setting of the staging lanes.  Every blocking host entry that takes stats
times its copies (h2d_ms, d2h_ms > 0); the pipelined batch entries report 0 for both."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
MiB = 1 << 20

SETTINGS = [
    {},                                                                  # defaults: 12 lanes x 2 MiB
    {"DARK_BWT_HOST_THREADS": "0"},                                      # staging off: the driver's own bounce buffer
    {"DARK_BWT_HOST_THREADS": "1", "DARK_BWT_HOST_CHUNK_MB": "1"},       # one lane, many chunks
]
OUTPUTS = ("bwt", "dist", "item_pos", "item_dist", "item_sym", "item_rank")  # forward_dc's nullable outputs, in argument order


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(len(SETTINGS)))
def test_host_copies_pageable_and_pinned(idx):
    """The staging lanes are set up at create from the environment: one process per setting."""
    env = dict(os.environ, **SETTINGS[idx])
    out = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, cwd=ROOT, capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-3000:]


# ---- the subprocess --------------------------------------------------------------------------------------------
def host(n, dtype, pinned):
    """A zeroed host array: pageable numpy memory, or a numpy view of pinned memory."""
    if not pinned:
        return np.zeros(n, dtype)
    import torch
    return torch.zeros(n * np.dtype(dtype).itemsize, dtype=torch.uint8).pin_memory().numpy().view(dtype)


def placed(a, pinned):
    b = host(a.size, a.dtype, pinned)
    b[:] = a
    return b


def ptrs(arrays):
    return [a.ctypes.data if a is not None else None for a in arrays]


def dc_arrays(n, pinned):
    """dist, item_pos, item_dist, item_sym, item_rank with room for n entries each."""
    return [host(n, dt, pinned) for dt in (np.uint32, np.uint32, np.uint32, np.uint8, np.uint8)]


def dc_encode(con, bwt, pinned):
    from dark_b200 import _ffi
    b = placed(bwt, pinned)
    outs = dc_arrays(b.size, pinned)
    info = _ffi.DcInfo()
    _ffi.check(con._L.dark_bwt_dc_encode(con._ctx, b.ctypes.data, b.size, *ptrs(outs), ctypes.byref(info)), con._ctx, "dc_encode")
    return con._dc_result(info, b.size, *outs)


def dc_encode_many(con, bwts, pinned):
    from dark_b200 import _ffi
    bs = [placed(b, pinned) for b in bwts]
    cnt, ns = len(bs), [b.size for b in bs]
    dist, pos, idist, sym, rank = dc_arrays(sum(ns), pinned)
    starts = host(cnt + 1, np.uint32, pinned)
    infos = (_ffi.DcInfo * cnt)()
    _ffi.check(con._L.dark_bwt_dc_encode_many(con._ctx, (ctypes.c_void_p * cnt)(*ptrs(bs)), (ctypes.c_uint64 * cnt)(*ns), cnt,
                                              *ptrs([dist, starts, pos, idist, sym, rank]), infos, None), con._ctx, "dc_encode_many")
    return con._dc_many_results(infos, ns, dist, starts, pos, idist, sym, rank)


def forward_dc_many(con, texts, pinned):
    from dark_b200 import _ffi
    ts = [placed(t, pinned) for t in texts]
    cnt, ns = len(ts), [t.size for t in ts]
    bwts = [host(n, np.uint8, pinned) for n in ns]
    dist, pos, idist, sym, rank = dc_arrays(sum(ns), pinned)
    starts = host(cnt + 1, np.uint32, pinned)
    infos, origins, stats = (_ffi.DcInfo * cnt)(), (ctypes.c_uint64 * cnt)(), _ffi.Stats()
    _ffi.check(con._L.dark_bwt_forward_dc_many(con._ctx, (ctypes.c_void_p * cnt)(*ptrs(ts)), (ctypes.c_uint64 * cnt)(*ns), cnt,
                                               (ctypes.c_void_p * cnt)(*ptrs(bwts)), origins,
                                               *ptrs([dist, starts, pos, idist, sym, rank]), infos, ctypes.byref(stats)),
               con._ctx, "forward_dc_many")
    res = con._dc_many_results(infos, ns, dist, starts, pos, idist, sym, rank)
    return [(bwts[k], int(origins[k]), res[k]) for k in range(cnt)], stats.as_dict()


def forward_many(con, texts, pinned):
    """(BWTs, origins, stats) of one dark_bwt_forward_many call."""
    ts = [placed(t, pinned) for t in texts]
    bwts = [host(t.size, np.uint8, pinned) for t in ts]
    origins = con.bwt_many_into(ptrs(ts), [t.size for t in ts], ptrs(bwts))
    return bwts, origins, con.stats.as_dict()


def inverse_many(con, bwts, origins, pinned):
    """The texts of one dark_bwt_inverse_many call."""
    bs = [placed(b, pinned) for b in bwts]
    outs = [host(b.size, np.uint8, pinned) for b in bs]
    con.inverse_many_into(ptrs(bs), [b.size for b in bs], origins, ptrs(outs))
    return outs


def forward_dc(con, text, pinned, skip=None):
    """(origin, {output: array or None}, info, stats) of one dark_bwt_forward_dc call, OUTPUTS[skip] left null."""
    from dark_b200 import _ffi
    t = placed(text, pinned)
    n = t.size
    outs = [host(n, np.uint8, pinned)] + dc_arrays(n, pinned)
    if skip is not None:
        outs[skip] = None
    p = ptrs(outs)
    info, origin, stats = _ffi.DcInfo(), ctypes.c_uint64(0), _ffi.Stats()
    _ffi.check(con._L.dark_bwt_forward_dc(con._ctx, t.ctypes.data, n, p[0], ctypes.byref(origin), *p[1:], ctypes.byref(info),
                                          ctypes.byref(stats)), con._ctx, "forward_dc")
    m = int(info.num_items)
    got = {f: a if a is None or f in ("bwt", "dist") else a[:m] for f, a in zip(OUTPUTS, outs)}
    return int(origin.value), got, info, stats.as_dict()


def same_dc(a, b, what):
    for f in ("dist", "init", "mtf_symbols", "num_unique", "num_items", "item_pos", "item_dist", "item_sym", "item_rank"):
        assert np.array_equal(np.asarray(a[f]), np.asarray(b[f])), (what, f)


def run():
    import oracle
    from dark_b200 import _ffi, saca, synth
    from dc_pack_ref import pack
    from test_dc_many import check_against_oracle
    rng = np.random.default_rng(71)
    n = 3 * MiB + 12345
    text = rng.integers(0, 200, n).astype(np.uint8)     # short runs: more than 1 MiB of items
    bwt_o, origin_o = oracle.bwt_forward(text)
    dist_o, init_o, _, _ = oracle.dc_encode(bwt_o)
    want = dict(zip(OUTPUTS, (bwt_o,) + (dist_o,) + oracle.dc_stream(bwt_o, dist_o, init_o)))
    assert want["item_sym"].size >= MiB
    blocks = [rng.integers(0, 256, 700_000).astype(np.uint8), rng.integers(0, 200, 500_001).astype(np.uint8),
              synth.generate("dna", 72, 100_003), synth.generate("text", 73, 40_000), np.array([3, 1], np.uint8)]
    with saca.Constructor(n) as con:
        # distance coding of one pageable BWT: 12 MiB of distances, more than 1 MiB in each item array
        single = [dc_encode(con, bwt_o, pinned) for pinned in (False, True)]
        check_against_oracle(single[0], bwt_o, oracle)
        same_dc(single[0], single[1], "dc_encode")

        # many blocks: concatenated outputs of more than 1 MiB
        many = [dc_encode_many(con, blocks, pinned) for pinned in (False, True)]
        assert sum(r["num_items"] for r in many[0]) >= MiB
        for k, b in enumerate(blocks):
            check_against_oracle(many[0][k], b, oracle)
            same_dc(many[0][k], many[1][k], ("dc_encode_many", k))
        fused = [forward_dc_many(con, blocks, pinned) for pinned in (False, True)]
        host_stats = [("forward_dc_many", st) for _, st in fused]
        packed = con.bwt_dc_packed_many(blocks, want_bwt=True)
        host_stats.append(("forward_dc_packed_many", con.stats.as_dict()))
        for k, t in enumerate(blocks):
            bo, oo = oracle.bwt_forward(t)
            for bwt, origin, res in (fused[0][0][k], fused[1][0][k]):
                assert origin == oo and np.array_equal(bwt, bo), ("forward_dc_many", k)
            check_against_oracle(fused[0][0][k][2], bo, oracle)
            same_dc(fused[0][0][k][2], fused[1][0][k][2], ("forward_dc_many", k))
            res = fused[0][0][k][2]
            bwt, origin, stream, _ = packed[k]
            assert origin == oo and np.array_equal(bwt, bo), ("forward_dc_packed_many", k)
            assert np.array_equal(stream, pack(res["item_pos"], res["item_dist"], res["item_sym"], res["item_rank"])), k

        # one forward + DC call, every output given, then each left null in turn
        for pinned in (False, True):
            origin, got, info, st = forward_dc(con, text, pinned)
            assert origin == origin_o and int(info.num_items) == want["item_pos"].size
            for f in OUTPUTS:
                assert np.array_equal(got[f], want[f]), ("forward_dc", pinned, f)
            host_stats.append(("forward_dc", st))
        for skip in range(len(OUTPUTS)):
            origin, got, _, _ = forward_dc(con, text, False, skip)
            assert origin == origin_o
            for f in OUTPUTS:
                assert (got[f] is None) == (f == OUTPUTS[skip]), (skip, f)
                if got[f] is not None:
                    assert np.array_equal(got[f], want[f]), ("forward_dc", OUTPUTS[skip], f)

        # the BWT and the packed stream of one block leave in one copy-out
        bwt, origin, stream, _ = con.bwt_dc_packed(text, want_bwt=True)
        assert origin == origin_o and np.array_equal(bwt, bwt_o)
        assert stream.size >= MiB and np.array_equal(stream, pack(*(want[f] for f in OUTPUTS[2:])))
        host_stats.append(("forward_dc_packed", con.stats.as_dict()))
        bwt, origin = con.bwt(text)
        assert origin == origin_o and np.array_equal(bwt, bwt_o)
        host_stats.append(("forward", con.stats.as_dict()))

    # many blocks on both sides of the staging threshold: 3 MiB + 12,345 bytes, exactly 1 MiB, 1 MiB - 1 and a few KiB
    sized = [text, rng.integers(0, 256, MiB).astype(np.uint8), rng.integers(0, 4, MiB - 1).astype(np.uint8),
             synth.generate("text", 74, 5_000)]
    want_sized = [(bwt_o, origin_o)] + [oracle.bwt_forward(t) for t in sized[1:]]
    with saca.Constructor(sum(t.size + 1 for t in sized)) as con:  # the inverse's rows: one '$' per block
        for pinned in (False, True):
            bwts, origins, st = forward_many(con, sized, pinned)
            host_stats.append(("forward_many", st))
            texts = inverse_many(con, [b for b, _ in want_sized], [o for _, o in want_sized], pinned)
            for k, (t, (bo, oo)) in enumerate(zip(sized, want_sized)):
                assert origins[k] == oo and np.array_equal(bwts[k], bo), ("forward_many", pinned, k)
                assert np.array_equal(texts[k], t), ("inverse_many", pinned, k)

    # every blocking host entry that takes stats times the copies of the caller's buffers in each direction
    assert sorted({e for e, _ in host_stats}) == sorted(["forward", "forward_dc", "forward_dc_packed", "forward_many",
                                                         "forward_dc_many", "forward_dc_packed_many"])
    for entry, st in host_stats:
        assert st["h2d_ms"] > 0 and st["d2h_ms"] > 0, (entry, st)

    # the pipelined batch entries time no copies of their own
    with saca.Constructor(n, flags=_ffi.F_DC_BATCH) as con:
        ts = [text, blocks[0]]
        outs = [np.zeros(t.size, np.uint8) for t in ts]
        origins, stats = con.bwt_batch_into(ptrs(ts), [t.size for t in ts], ptrs(outs), want_stats=True)
        assert origins[0] == origin_o and np.array_equal(outs[0], bwt_o)
        origins, _, dc_stats = con.bwt_dc_batch_into(ptrs(ts), [t.size for t in ts], ptrs(outs), want_stats=True)
        assert origins[0] == origin_o and np.array_equal(outs[0], bwt_o)
        for st in stats + dc_stats:
            assert st["h2d_ms"] == 0 and st["d2h_ms"] == 0, st
    print("ok")


if __name__ == "__main__":
    sys.path[:0] = [ROOT, HERE]
    run()
