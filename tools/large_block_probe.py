#!/usr/bin/env python3
"""Blocks above 2^31 on one card: C4 (2^31) beside 3 GiB and 2^32 - 2, mixed and DNA, through the host entry on a
default-flag context (one staging pair above 2^31).  One JSON line per block after a card line (name, power limit,
free memory, the arena of every context made):
forward device ms and phase split, host-entry wall time, inverse and distance-coding device ms, CRC-32s.

    python tools/large_block_probe.py [out.jsonl]"""
import json
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from dark_b200 import saca, synth, _ffi  # noqa: E402

SIZES = [1 << 31, 3 << 30, (1 << 32) - 2]
KINDS = [("mixed", 4), ("dna", 1)]
PHASES = ("device_ms", "init_ms", "sort_ms", "keybuild_ms", "rerank_ms", "emit_ms", "rounds", "sort_passes")


def crc(a):
    c = 0
    for i in range(0, a.size, 1 << 30):
        c = zlib.crc32(memoryview(a[i:i + (1 << 30)]), c)
    return "%08x" % c


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    free, total = torch.cuda.mem_get_info()
    return {"card": q, "free_bytes": free, "total_bytes": total,
            "arena_bytes": {f"{n}:{f}": saca.arena_bytes(n, f) for n in SIZES for f in (_ffi.F_DEFAULT, _ffi.F_DEVICE_ONLY)}}


def main():
    out = open(sys.argv[1], "w") if len(sys.argv) > 1 else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()
    torch.cuda.init()
    emit(card())
    for n in SIZES:
        torch.cuda.empty_cache()
        free = torch.cuda.mem_get_info()[0]
        t0 = time.perf_counter()
        con = saca.Constructor(n)
        create_s = time.perf_counter() - t0
        for kind, seed in KINDS:
            t = synth.generate(kind, seed, n)
            bwt = np.empty(n, dtype=np.uint8)
            origin = con.bwt_batch_into([t.ctypes.data], [n], [bwt.ctypes.data])[0]   # warm: module load, staging lanes
            t0 = time.perf_counter()
            bwt, origin = con.bwt(t)
            wall_ms = (time.perf_counter() - t0) * 1e3
            st = con.stats.as_dict()
            back = np.empty(n, dtype=np.uint8)
            inv_ms = con.inverse_batch_into([bwt.ctypes.data], [n], [origin], [back.ctypes.data])[0]
            dc = con.dc_encode(bwt, want_dist=False)
            emit({"kind": kind, "seed": seed, "n": n, "arena_bytes": saca.arena_bytes(n), "free_before_create": free,
                  "create_s": round(create_s, 3), "origin": origin, "text_crc32": crc(t), "bwt_crc32": crc(bwt),
                  "round_trip": bool(np.array_equal(back, t)), "host_wall_ms": round(wall_ms, 2),
                  "h2d_ms": st["h2d_ms"], "d2h_ms": st["d2h_ms"], **{k: st[k] for k in PHASES},
                  "inverse_device_ms": inv_ms, "dc_device_ms": dc["device_ms"], "dc_items": dc["num_items"]})
            del t, bwt, back, dc
        con.close()


if __name__ == "__main__":
    main()
