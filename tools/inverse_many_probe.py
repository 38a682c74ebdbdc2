#!/usr/bin/env python3
"""The unpack side for many blocks, against the single-block calls it replaces.  One JSON line per measurement; the first
line names the card and its power limit, read in the same run.

  many   1, 4, 16, 64, 256 DISTINCT C1-sized text blocks (768,771 bytes, seeds 3 + 100 k as in small_blocks_probe.py)
         through dark_bwt_inverse_many (pinned host buffers): device ms and wall ms per call, against the same blocks
         through single dark_bwt_inverse_device calls (summed device ms) and single dark_bwt_inverse calls (summed wall
         ms), with per-block parity (original text, and many == single).
  batch  20 x 256 MiB pinned blocks (C2 dna and C5 mixed; one block repeated, outputs alternating between two buffers as
         bench.py does) through dark_bwt_inverse_batch, against 20 sequential dark_bwt_inverse calls, wall clock end to
         end; then one batch run on pageable numpy buffers.

    python tools/inverse_many_probe.py [many|batch|all]
"""
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from dark_b200 import _ffi, saca, synth  # noqa: E402

what = sys.argv[1] if len(sys.argv) > 1 else "all"


def emit(d):
    print(json.dumps(d), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    emit({"card": q[0] if q else torch.cuda.get_device_name(0), "torch_device": torch.cuda.get_device_name(0)})


def probe_many():
    kind, seed, n = synth.CONFIGS["c1"]
    for cnt in (1, 4, 16, 64, 256):
        texts = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(cnt)]
        for k in range(cnt):
            synth.generate(kind, seed + 100 * k, n, out=texts[k].numpy())
        bwts = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(cnt)]
        outs = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(cnt)]
        con = saca.Constructor(cnt * (n + 1))
        origins = con.bwt_many_into([t.data_ptr() for t in texts], [n] * cnt, [b.data_ptr() for b in bwts])
        bp, op = [b.data_ptr() for b in bwts], [o.data_ptr() for o in outs]
        con.inverse_many_into(bp, [n] * cnt, origins, op)  # warm-up
        reps = max(3, 256 // cnt)
        dev = 0.0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            dev += con.inverse_many_into(bp, [n] * cnt, origins, op)
        wall = (time.perf_counter() - t0) / reps
        dev /= reps
        many_ok = all(torch.equal(o, t) for o, t in zip(outs, texts))
        # the same blocks one call each: device-resident (device ms) and host (wall ms)
        d_bwt = torch.empty(n, dtype=torch.uint8, device="cuda")
        d_out = torch.empty(n, dtype=torch.uint8, device="cuda")
        single_out = torch.empty(n, dtype=torch.uint8).pin_memory()
        L, ctx = con._L, con._ctx
        L.dark_bwt_inverse(ctx, bp[0], n, origins[0], single_out.data_ptr())  # warm-up
        d_bwt.copy_(bwts[0])
        con.inverse_device(d_bwt.data_ptr(), n, origins[0], d_out.data_ptr())
        single_dev, single_wall, parity = 0.0, 0.0, True
        for k in range(cnt):
            d_bwt.copy_(bwts[k])
            torch.cuda.synchronize()
            single_dev += con.inverse_device(d_bwt.data_ptr(), n, origins[k], d_out.data_ptr())
            parity &= torch.equal(d_out.cpu(), outs[k])
            t0 = time.perf_counter()
            _ffi.check(L.dark_bwt_inverse(ctx, bp[k], n, origins[k], single_out.data_ptr()), ctx, "inverse")
            single_wall += time.perf_counter() - t0
            parity &= torch.equal(single_out, outs[k])
        emit({"many": cnt, "block_bytes": n, "calls": reps, "device_ms_per_call": dev, "wall_ms_per_call": wall * 1e3,
              "single_device_ms_sum": single_dev, "single_wall_ms_sum": single_wall * 1e3,
              "device_ratio_many_over_single": dev / single_dev, "wall_ratio_many_over_single": wall * 1e3 / (single_wall * 1e3),
              "many_device_MBps": cnt * n / 1e3 / dev, "many_wall_MBps": cnt * n / 1e6 / wall,
              "parity_text": "ok" if many_ok else "MISMATCH", "parity_many_vs_single": "ok" if parity else "MISMATCH"})
        con.close()
        del texts, bwts, outs


def probe_batch():
    n, cnt = 1 << 28, 20
    for name, (kind, seed) in (("c2", ("dna", 1)), ("c5", ("mixed", 1000))):
        text = torch.empty(n, dtype=torch.uint8).pin_memory()
        synth.generate(kind, seed, n, out=text.numpy())
        bwt = torch.empty(n, dtype=torch.uint8).pin_memory()
        o1 = torch.empty(n, dtype=torch.uint8).pin_memory()
        o2 = torch.empty(n, dtype=torch.uint8).pin_memory()
        con = saca.Constructor(n)
        origin = con.bwt_into(text.data_ptr(), n, bwt.data_ptr())
        L, ctx = con._L, con._ctx
        outs = [o1.data_ptr(), o2.data_ptr()] * (cnt // 2)
        con.inverse_batch_into([bwt.data_ptr()] * 2, [n] * 2, [origin] * 2, outs[:2])  # warm-up (both buffers)
        _ffi.check(L.dark_bwt_inverse(ctx, bwt.data_ptr(), n, origin, o1.data_ptr()), ctx, "inverse")
        res = {}
        for rep in range(2):  # alternate the two forms twice: the spread shows in the two figures of each
            o1.zero_(), o2.zero_()
            t0 = time.perf_counter()
            ms = con.inverse_batch_into([bwt.data_ptr()] * cnt, [n] * cnt, [origin] * cnt, outs)
            wall_b = time.perf_counter() - t0
            ok_b = torch.equal(o1, text) and torch.equal(o2, text)
            o1.zero_()
            t0 = time.perf_counter()
            for k in range(cnt):
                _ffi.check(L.dark_bwt_inverse(ctx, bwt.data_ptr(), n, origin, outs[k]), ctx, "inverse")
            wall_s = time.perf_counter() - t0
            ok_s = torch.equal(o1, text)
            res.setdefault("batch_e2e_GBps", []).append(cnt * n / wall_b / 1e9)
            res.setdefault("sequential_e2e_GBps", []).append(cnt * n / wall_s / 1e9)
            res.setdefault("batch_device_ms_mean", []).append(sum(ms) / cnt)
            res.setdefault("parity", []).append("ok" if ok_b and ok_s else "MISMATCH")
        emit(dict({"batch": name, "blocks": cnt, "block_bytes": n, "buffers": "pinned"}, **res))
        # pageable numpy buffers: the staging lanes in both directions
        pb = bwt.numpy().copy()
        p1, p2 = np.empty(n, dtype=np.uint8), np.empty(n, dtype=np.uint8)
        pouts = [p1.ctypes.data, p2.ctypes.data] * (cnt // 2)
        con.inverse_batch_into([pb.ctypes.data] * 2, [n] * 2, [origin] * 2, pouts[:2])  # warm-up (allocates the lanes)
        t0 = time.perf_counter()
        con.inverse_batch_into([pb.ctypes.data] * cnt, [n] * cnt, [origin] * cnt, pouts)
        wall_p = time.perf_counter() - t0
        tn = text.numpy()
        emit({"batch": name, "blocks": cnt, "block_bytes": n, "buffers": "pageable", "batch_e2e_GBps": cnt * n / wall_p / 1e9,
              "parity": "ok" if np.array_equal(p1, tn) and np.array_equal(p2, tn) else "MISMATCH"})
        con.close()
        del text, bwt, o1, o2, pb, p1, p2


if not torch.cuda.is_available():
    sys.exit("inverse_many_probe.py measures on the GPU: no CUDA device here")
card()
if what in ("many", "all"):
    probe_many()
if what in ("batch", "all"):
    probe_batch()
