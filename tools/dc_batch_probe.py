#!/usr/bin/env python3
"""The pipelined forward BWT + distance coding batch against the sequential calls it replaces.  One JSON line per row;
the first line names the card and its power limit, read in the same run.

For each workload (20 x 256 MiB blocks of C2 = dna seed 1, and of the first C5 block = mixed seed 1000), each host buffer
kind (pinned, then pageable numpy) and each output set (`items`: the four item arrays only, the reference's path; `all`:
BWT, distances and items), two arms are alternated twice on one context:
  batch       one dark_bwt_forward_dc_batch call over the 20 blocks;
  sequential  20 dark_bwt_forward_dc calls.
Block k writes into output set k & 1 (two sets, as bench.py alternates two BWT buffers).  A row reports wall ms per block,
input GB/s end to end, the bytes copied out per block, the D2H-only time of those same bytes (the same arrays copied from
device memory into pinned host buffers by cudaMemcpyAsync, 20 times, nothing else running: the copy bound, which a
pageable destination cannot beat either), and the CRC-32 of every output of both sets after each arm, which must agree.

    python tools/dc_batch_probe.py
"""
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
import torch  # noqa: E402
from dark_b200 import _ffi, saca, synth  # noqa: E402

N, COUNT, REPS = 1 << 28, 20, 2
ARRAYS = ("bwt", "dist", "item_pos", "item_dist", "item_sym", "item_rank")
WIDTH = {"bwt": 1, "dist": 4, "item_pos": 4, "item_dist": 4, "item_sym": 1, "item_rank": 1}
SETS = {"items": ARRAYS[2:], "all": ARRAYS}


def emit(d):
    print(json.dumps(d), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    emit({"card": q[0] if q else torch.cuda.get_device_name(0), "torch_device": torch.cuda.get_device_name(0)})


def host_set(pinned):
    """One output set: numpy views of host buffers (pinned tensors or plain numpy) for all six arrays."""
    out = {}
    for a in ARRAYS:
        dt = np.uint8 if WIDTH[a] == 1 else np.uint32
        if pinned:
            t = torch.empty(N * WIDTH[a], dtype=torch.uint8).pin_memory()
            out[a] = (t, t.numpy().view(dt))
        else:
            arr = np.empty(N, dt)
            out[a] = (None, arr)
    return out


def crcs(sets, which, items):
    r = {}
    for s, hs in enumerate(sets):
        for a in which:
            v = hs[a][1]
            v = v[:items] if a.startswith("item_") else v
            r[f"{a}[{s}]"] = "%08x" % (zlib.crc32(memoryview(np.ascontiguousarray(v)).cast("B")) & 0xFFFFFFFF)
    return r


def d2h_only_ms(sizes):
    """COUNT rounds of the same per-array D2H copies, device -> pinned host, on one stream, host clock to a synchronise."""
    dev = [torch.empty(b, dtype=torch.uint8, device="cuda") for b in sizes]
    host = [torch.empty(b, dtype=torch.uint8).pin_memory() for b in sizes]
    for h, d in zip(host, dev):  # warm-up
        h.copy_(d, non_blocking=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(COUNT):
        for h, d in zip(host, dev):
            h.copy_(d, non_blocking=True)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / COUNT
    del dev, host
    return ms


def probe(name, kind, seed):
    con = saca.Constructor(N, flags=_ffi.F_DC_BATCH)
    L, ctx = con._L, con._ctx
    pinned_text = torch.empty(N, dtype=torch.uint8).pin_memory()
    synth.generate(kind, seed, N, out=pinned_text.numpy())
    for buffers in ("pinned", "pageable"):
        pinned = buffers == "pinned"
        page_text = None if pinned else pinned_text.numpy().copy()
        text_ptr = pinned_text.data_ptr() if pinned else page_text.ctypes.data
        sets = [host_set(pinned), host_set(pinned)]
        info, origin = _ffi.DcInfo(), ctypes.c_uint64(0)
        for outputs, which in SETS.items():
            ptr = {a: ([sets[k & 1][a][1].ctypes.data for k in range(COUNT)] if a in which else None) for a in ARRAYS}

            def batch():
                return con.bwt_dc_batch_into([text_ptr] * COUNT, [N] * COUNT, *[ptr[a] for a in ARRAYS], want_stats=True)

            def sequential():
                for k in range(COUNT):
                    out = [ptr[a][k] if ptr[a] else None for a in ARRAYS]
                    _ffi.check(L.dark_bwt_forward_dc(ctx, text_ptr, N, out[0], ctypes.byref(origin), *out[1:], ctypes.byref(info), None),
                               ctx, "forward_dc")
            origins, infos, stats = batch()  # warm-up: both slots, the staging lanes, every host page touched
            sequential()
            items = int(infos[0].num_items)
            bytes_out = sum((items if a.startswith("item_") else N) * WIDTH[a] for a in which)
            row = {"workload": name, "buffers": buffers, "outputs": outputs, "blocks": COUNT, "block_bytes": N, "num_items": items,
                   "bytes_out_per_block": bytes_out, "origin": origins[0]}
            crc_arm = {}
            for rep in range(REPS):
                for arm in ("batch", "sequential"):
                    for s in sets:
                        for a in which:
                            s[a][1].fill(0)
                    t0 = time.perf_counter()
                    if arm == "batch":
                        origins, infos, stats = batch()
                    else:
                        sequential()
                    wall = (time.perf_counter() - t0) * 1e3
                    row.setdefault(f"{arm}_ms_per_block", []).append(wall / COUNT)
                    row.setdefault(f"{arm}_e2e_GBps", []).append(COUNT * N / (wall / 1e3) / 1e9)
                    if arm == "batch":
                        row.setdefault("batch_device_ms_per_block", []).append(
                            sum(s["device_ms"] + i.device_ms for s, i in zip(stats, infos)) / COUNT)
                        assert all(int(i.num_items) == items for i in infos) and all(o == row["origin"] for o in origins)
                    else:
                        assert int(info.num_items) == items and int(origin.value) == row["origin"]
                    crc_arm.setdefault(arm, []).append(crcs(sets, which, items))
            row["crc"] = crc_arm["batch"][0]
            same = all(c == row["crc"] for arm in crc_arm.values() for c in arm)
            row["parity_batch_vs_sequential"] = "ok" if same else "MISMATCH"
            row["d2h_only_pinned_ms_per_block"] = d2h_only_ms([(items if a.startswith("item_") else N) * WIDTH[a] for a in which])
            row["batch_over_d2h_only"] = float(np.median(row["batch_ms_per_block"])) / row["d2h_only_pinned_ms_per_block"]
            row["batch_speedup_over_sequential"] = float(np.median(row["sequential_ms_per_block"])) / float(np.median(row["batch_ms_per_block"]))
            emit(row)
        del sets, page_text
    con.close()


if not torch.cuda.is_available():
    sys.exit("dc_batch_probe.py measures on the GPU: no CUDA device here")
card()
probe("c2", "dna", 1)
probe("c5", *synth.c5_block(0)[:2])
