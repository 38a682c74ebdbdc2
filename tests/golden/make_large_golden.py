#!/usr/bin/env python3
"""Generate the fixtures of the blocks above 2^31 bytes with the CPU oracle (oracle/oracle_cli).

    python tests/golden/make_large_golden.py

writes tests/golden/large_golden.json: one record per block, shaped like those of oracle_golden.json
(make_golden.py).  The blocks run one after another, ~30 GB of RAM each; the two of 2^32 - 2 bytes run without
the LCP profile, which would need ~50 GB more.  Scaling the C4 run (15 min at 2 GiB), about 20, 20 and 35
minutes of one core.

It also writes tests/golden/large_dc.json: the CRC-32s of the oracle's distance coding (oracle_dc_encode,
oracle_dc_stream) of the DNA block's BWT, so that the GPU test need not hold the oracle's arrays.  Those arrays
(~40 GB at 2^32 - 2) go through memory-mapped files under $TMPDIR.
"""
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_golden import CLI, ROOT, key  # noqa: E402

OUT = os.path.join(HERE, "large_golden.json")
DC_OUT = os.path.join(HERE, "large_dc.json")
BLOCKS = [("mixed", 4, 5 << 29), ("dna", 1, (1 << 32) - 2), ("mixed", 4, (1 << 32) - 2)]
PROFILE = {("mixed", 4, 5 << 29)}
DC_BLOCK = ("dna", 1, (1 << 32) - 2)


def crc32_file(a, chunk=1 << 28):
    c = 0
    for i in range(0, a.size, chunk):
        c = zlib.crc32(memoryview(a[i:i + chunk]).cast("B"), c)
    return f"{c:08x}"


def dc_record(bwt_path, n):
    """CRC-32s of oracle_dc_encode / oracle_dc_stream on the BWT in bwt_path, arrays memory-mapped beside it."""
    sys.path.insert(0, ROOT)
    from oracle import lib
    L = lib()
    d = os.path.dirname(bwt_path)
    mm = lambda name, dt: np.memmap(os.path.join(d, name), dtype=dt, mode="w+", shape=(n,))  # noqa: E731
    bwt = np.memmap(bwt_path, dtype=np.uint8, mode="r", shape=(n,))
    dist = mm("dist", np.uint32)
    init = (ctypes.c_uint64 * 256)()
    mtf = (ctypes.c_uint8 * 256)()
    nu = ctypes.c_uint32(0)
    L.oracle_dc_encode.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                   ctypes.POINTER(ctypes.c_uint32)]
    assert L.oracle_dc_encode(bwt.ctypes.data, n, dist.ctypes.data, init, mtf, ctypes.byref(nu)) == 0
    pos, idist, sym, rk = mm("pos", np.uint32), mm("idist", np.uint32), mm("sym", np.uint8), mm("rank", np.uint8)
    L.oracle_dc_stream.restype = ctypes.c_uint64
    L.oracle_dc_stream.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p] + [ctypes.c_void_p] * 4
    k = int(L.oracle_dc_stream(bwt.ctypes.data, dist.ctypes.data, n, init, pos.ctypes.data, idist.ctypes.data,
                               sym.ctypes.data, rk.ctypes.data))
    return {"n": n, "bwt_crc32": crc32_file(bwt), "init": [int(x) for x in init], "mtf_symbols": [int(x) for x in mtf],
            "num_unique": int(nu.value), "num_items": k, "dist_crc32": crc32_file(dist),
            "item_pos_crc32": crc32_file(pos[:k]), "item_dist_crc32": crc32_file(idist[:k]),
            "item_sym_crc32": crc32_file(sym[:k]), "item_rank_crc32": crc32_file(rk[:k])}


def write(path, obj):
    with open(path, "w") as f:
        json.dump(obj, f, indent=1, sort_keys=True)
        f.write("\n")


def main():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
    gold = {}
    if os.path.exists(OUT):
        with open(OUT) as f:
            gold = json.load(f)
    for kind, seed, n in BLOCKS:
        with tempfile.TemporaryDirectory() as tmp:
            dump = ["--dump-bwt", os.path.join(tmp, "bwt")] if (kind, seed, n) == DC_BLOCK else []
            prof = ["--profile"] if (kind, seed, n) in PROFILE else []
            out = subprocess.check_output([CLI, kind, str(seed), str(n)] + prof + dump, text=True)
            if dump:
                rec = {"block": key(kind, seed, n), **dc_record(dump[1], n)}
                write(DC_OUT, rec)
                print(key(kind, seed, n), "dc items", rec["num_items"], flush=True)
        rec = json.loads(out)
        for k in ("saca_s", "emit_s", "mb_per_s"):   # timings are not golden
            rec.pop(k, None)
        gold[key(kind, seed, n)] = rec
        print(key(kind, seed, n), "origin", rec["origin"], "bwt", rec["bwt_crc32"], flush=True)
        write(OUT, gold)


if __name__ == "__main__":
    main()
