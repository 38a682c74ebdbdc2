#!/usr/bin/env python3
"""Decoding the packed item stream on the GPU against the CPU path it replaces.  One JSON line per row, printed and written
to profiles/r4_dc_decode_probe.jsonl (--out to change); the first line names the card and its power limit, read in the
same run.

For each block (C2 = dna seed 1, 256 MiB; the first C5 block, mixed seed 1000, 256 MiB; C3 = rep17 seed 2, 64 MiB;
C1 = text seed 3, 768,771 bytes) the stream and origin come from dark_bwt_forward_dc_packed, and four arms are alternated
REPS times on one context, host clock around each call:
  gpu_pinned    dark_bwt_inverse_dc_packed, stream and text in pinned host memory
  gpu_pageable  the same with numpy (pageable) buffers
  cpu_unpack    the tests' reference unpack (tests/dc_pack_ref.c) + np.repeat to the BWT, then dark_bwt_inverse (pageable)
  bwt_only      dark_bwt_inverse of the BWT alone (pageable), the reference point
Every row checks the CRC-32 of each arm's text against the block's.  Device ms (CUDA events, device-resident buffers):
decode = dark_bwt_dc_decode_packed_device (parse, expand, check, compare), check = dark_bwt_dc_encode_packed_device of
the BWT (the DC + pack the check runs), parse_expand_compare = decode - check, inverse = dark_bwt_inverse_device.

    python tools/dc_decode_probe.py [--out PATH] [--reps R]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402
import dc_pack_ref  # noqa: E402
from dark_b200 import _ffi, saca, synth  # noqa: E402

BLOCKS = [("C2", "dna", 1, 1 << 28), ("C5 block 0", "mixed", 1000, 1 << 28), ("C3", "rep17", 2, 1 << 26), ("C1", "text", 3, 768_771)]
OUT = None


def emit(d):
    line = json.dumps(d)
    print(line, flush=True)
    OUT.write(line + "\n")
    OUT.flush()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    emit({"card": q[0] if q else torch.cuda.get_device_name(0), "torch_device": torch.cuda.get_device_name(0)})


def crc(a):
    return "%08x" % (zlib.crc32(memoryview(np.ascontiguousarray(a)).cast("B")) & 0xFFFFFFFF)


def med(xs):
    return round(float(np.median(xs)), 3)


def probe(con, name, kind, seed, n, reps):
    text = synth.generate(kind, seed, n)
    want = crc(text)
    bwt, origin, stream, info = con.bwt_dc_packed(text, want_bwt=True)
    S = stream.size
    L, ctx = con._L, con._ctx
    p_stream = torch.from_numpy(stream.copy()).pin_memory()
    p_text = torch.empty(n, dtype=torch.uint8).pin_memory()
    g_text = np.empty(n, np.uint8)

    def gpu_pinned():
        _ffi.check(L.dark_bwt_inverse_dc_packed(ctx, p_stream.data_ptr(), S, n, origin, p_text.data_ptr(), None, None), ctx, "pinned")
        return p_text.numpy()

    def gpu_pageable():
        _ffi.check(L.dark_bwt_inverse_dc_packed(ctx, stream.ctypes.data, S, n, origin, g_text.ctypes.data, None, None), ctx, "pageable")
        return g_text

    def cpu_unpack():
        pos, _, sym, _ = dc_pack_ref.unpack(stream, int(info.num_items))
        b = np.repeat(sym, np.diff(pos.astype(np.int64), prepend=-1))
        return con.inverse(b, origin)

    def bwt_only():
        return con.inverse(bwt, origin)

    arms = {"gpu_pinned": gpu_pinned, "gpu_pageable": gpu_pageable, "cpu_unpack": cpu_unpack, "bwt_only": bwt_only}
    for f in arms.values():  # warm-up: staging lanes, pages touched
        f()
    ms = {a: [] for a in arms}
    ok = True
    for _ in range(reps):
        for a, f in arms.items():
            t0 = time.perf_counter()
            out = f()
            ms[a].append((time.perf_counter() - t0) * 1e3)
            ok &= crc(out) == want
    # device split on device-resident buffers
    d_stream = torch.from_numpy(stream).cuda()
    d_bwt = torch.from_numpy(bwt).cuda()
    d_out = torch.empty(n, dtype=torch.uint8, device="cuda")
    d_enc = torch.empty(8 * n, dtype=torch.uint8, device="cuda")
    dec, chk, inv = [], [], []
    for _ in range(reps):
        dec.append(con.dc_decode_packed_device(d_stream.data_ptr(), S, n, d_out.data_ptr()).device_ms)
        chk.append(con.dc_encode_packed_device(d_bwt.data_ptr(), n, d_enc.data_ptr(), 8 * n)[1].device_ms)
        inv.append(con.inverse_device(d_bwt.data_ptr(), n, origin, d_out.data_ptr()))
    ok &= bool(torch.equal(d_out.cpu(), torch.from_numpy(text)))
    emit({"block": name, "kind": kind, "seed": seed, "n": n, "num_items": int(info.num_items), "stream_bytes": S, "reps": reps,
          "wall_ms": {a: med(v) for a, v in ms.items()}, "wall_ms_all": {a: [round(x, 3) for x in v] for a, v in ms.items()},
          "bytes_in": {"gpu_pinned": S, "gpu_pageable": S, "cpu_unpack": n, "bwt_only": n}, "bytes_out": n,
          "device_ms": {"decode": med(dec), "check": med(chk), "parse_expand_compare": round(med(dec) - med(chk), 3), "inverse": med(inv)},
          "text_crc32": want, "crc_ok": ok})
    del d_stream, d_bwt, d_out, d_enc
    torch.cuda.empty_cache()


def main():
    global OUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_dc_decode_probe.jsonl"))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    OUT = open(a.out, "w")
    card()
    with saca.Constructor(1 << 28) as con:
        for name, kind, seed, n in BLOCKS:
            probe(con, name, kind, seed, n, a.reps)


if __name__ == "__main__":
    main()
