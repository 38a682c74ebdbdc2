#!/usr/bin/env python3
"""The packed item stream against the four item arrays, through the pipelined forward + DC batch.  One JSON line per row,
printed and written to profiles/r4_dc_packed_probe.jsonl (--out to change); the first line names the card and its power
limit, read in the same run.

For each workload (20 x 256 MiB blocks of C2 = dna seed 1, and of the first C5 block) and each host buffer kind (pinned,
then pageable numpy), two arms are alternated twice on one context:
  items    one dark_bwt_forward_dc_batch call with the four item arrays as its only outputs (the reference's path);
  packed   one dark_bwt_forward_dc_packed_batch call (the stream only).
Block k writes into output set k & 1 of its arm.  A row reports per arm: wall ms per block and input GB/s end to end, the
device ms per block (forward + DC kernels, and the pack kernels in the packed arm: CUDA events), the bytes copied out per
block, and the D2H-only time of those bytes (the same sizes copied from device memory into pinned host buffers by
cudaMemcpyAsync, 20 times, nothing else running).  pack_ms_per_block is the packed arm's DC device time less the items
arm's (both CUDA events on the same blocks).  After every packed run both sets' streams are unpacked by the tests'
reference (tests/dc_pack_ref.c) and the CRC-32s of the four arrays compared with the items arm's.

    python tools/dc_packed_probe.py [--out PATH]
"""
import argparse
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

N, COUNT, REPS = 1 << 28, 20, 2
ITEMS = ("item_pos", "item_dist", "item_sym", "item_rank")
WIDTH = {"item_pos": 4, "item_dist": 4, "item_sym": 1, "item_rank": 1}
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


def host(nbytes, pinned, dt=np.uint8):
    """(keep-alive, numpy view) of a host buffer."""
    if pinned:
        t = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        return t, t.numpy().view(dt)
    return None, np.empty(nbytes // np.dtype(dt).itemsize, dt)


def crc(a):
    return "%08x" % (zlib.crc32(memoryview(np.ascontiguousarray(a)).cast("B")) & 0xFFFFFFFF)


def d2h_only_ms(sizes):
    """COUNT rounds of the same per-array D2H copies, device -> pinned host, on one stream, host clock to a synchronise."""
    dev = [torch.empty(b, dtype=torch.uint8, device="cuda") for b in sizes]
    hst = [torch.empty(b, dtype=torch.uint8).pin_memory() for b in sizes]
    for h, d in zip(hst, dev):  # warm-up
        h.copy_(d, non_blocking=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(COUNT):
        for h, d in zip(hst, dev):
            h.copy_(d, non_blocking=True)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / COUNT
    del dev, hst
    return ms


def med(xs):
    return float(np.median(xs))


def probe(name, kind, seed):
    con = saca.Constructor(N, flags=_ffi.F_DC_BATCH)
    pinned_text = torch.empty(N, dtype=torch.uint8).pin_memory()
    synth.generate(kind, seed, N, out=pinned_text.numpy())
    cap = _ffi.dc_packed_max(N)
    for buffers in ("pinned", "pageable"):
        pinned = buffers == "pinned"
        page_text = None if pinned else pinned_text.numpy().copy()
        text_ptr = pinned_text.data_ptr() if pinned else page_text.ctypes.data
        item_sets = [{a: host(N * WIDTH[a], pinned, np.uint8 if WIDTH[a] == 1 else np.uint32) for a in ITEMS} for _ in range(2)]
        stream_sets = [host(cap, pinned) for _ in range(2)]
        item_ptrs = [[item_sets[k & 1][a][1].ctypes.data for k in range(COUNT)] for a in ITEMS]
        stream_ptrs = [stream_sets[k & 1][1].ctypes.data for k in range(COUNT)]

        def items_arm():
            return con.bwt_dc_batch_into([text_ptr] * COUNT, [N] * COUNT, None, None, *item_ptrs, want_stats=True)

        def packed_arm():
            return con.bwt_dc_packed_batch_into([text_ptr] * COUNT, [N] * COUNT, stream_ptrs, [cap] * COUNT, want_stats=True)

        origins, infos, _ = items_arm()  # warm-up: both slots, the staging lanes, every host page touched
        packed_arm()
        m = int(infos[0].num_items)
        row = {"workload": name, "buffers": buffers, "blocks": COUNT, "block_bytes": N, "num_items": m, "origin": origins[0]}
        item_crcs, ok = None, True
        for rep in range(REPS):
            for arm in ("items", "packed"):
                t0 = time.perf_counter()
                if arm == "items":
                    origins, infos, stats = items_arm()
                else:
                    origins, sizes, infos, stats = packed_arm()
                wall = (time.perf_counter() - t0) * 1e3
                row.setdefault(f"{arm}_ms_per_block", []).append(wall / COUNT)
                row.setdefault(f"{arm}_e2e_GBps", []).append(COUNT * N / (wall / 1e3) / 1e9)
                row.setdefault(f"{arm}_device_ms_per_block", []).append(sum(s["device_ms"] + i.device_ms for s, i in zip(stats, infos)) / COUNT)
                row.setdefault(f"{arm}_dc_ms_per_block", []).append(sum(i.device_ms for i in infos) / COUNT)
                assert all(int(i.num_items) == m for i in infos) and all(o == row["origin"] for o in origins)
                if arm == "items":
                    c = [{a: crc(s[a][1][:m]) for a in ITEMS} for s in item_sets]
                    ok &= item_crcs is None or c == item_crcs
                    item_crcs = c
                else:
                    assert len(set(sizes)) == 1
                    row["stream_bytes_per_block"] = sizes[0]
                    for s, want in zip(stream_sets, item_crcs):
                        got = dc_pack_ref.unpack(s[1][:sizes[0]], m)
                        ok &= {a: crc(x) for a, x in zip(ITEMS, got)} == want
                        del got
        row["items_bytes_out_per_block"] = m * sum(WIDTH.values())
        row["packed_bytes_out_per_block"] = row["stream_bytes_per_block"]
        row["items_d2h_only_pinned_ms_per_block"] = d2h_only_ms([m * WIDTH[a] for a in ITEMS])
        row["packed_d2h_only_pinned_ms_per_block"] = d2h_only_ms([row["stream_bytes_per_block"]])
        row["pack_ms_per_block"] = med(row["packed_dc_ms_per_block"]) - med(row["items_dc_ms_per_block"])
        row["crc_decoded_stream_equals_items"] = "ok" if ok else "MISMATCH"
        row["packed_speedup_over_items"] = med(row["items_ms_per_block"]) / med(row["packed_ms_per_block"])
        for arm in ("items", "packed"):  # overlap: wall near max(device, d2h) = overlapped, near their sum = serial
            dev, d2h = med(row[f"{arm}_device_ms_per_block"]), row[f"{arm}_d2h_only_pinned_ms_per_block"]
            row[f"{arm}_device_plus_d2h_ms"] = dev + d2h
            row[f"{arm}_max_device_d2h_ms"] = max(dev, d2h)
        emit(row)
        del item_sets, stream_sets, page_text
    con.close()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_dc_packed_probe.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("dc_packed_probe.py measures on the GPU: no CUDA device here")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    OUT = open(args.out, "w")
    card()
    probe("c2", "dna", 1)
    probe("c5", *synth.c5_block(0)[:2])
    OUT.close()
