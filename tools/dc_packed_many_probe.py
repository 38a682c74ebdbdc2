#!/usr/bin/env python3
"""The packed item stream for many small blocks, against the four item arrays and against one packed call per block.
One JSON line per row, printed and written to profiles/r4_dc_packed_many_probe.jsonl (--out to change); the first line
names the card and its power limit, read in the same run.

Workloads: 16, 64 and 256 C1-sized text blocks (768,771 bytes, seeds 3 + 100 k as in dc_many_probe.py) and 256 DNA blocks
of 1 MiB (seeds 1 + 100 k).  For each workload and each host buffer kind (pinned, then pageable numpy: texts and outputs),
three arms are alternated REPS times on one context sized to the list:
  items    one dark_bwt_forward_dc_many call with the item offsets and the four item arrays as its only outputs;
  packed   one dark_bwt_forward_dc_packed_many call (the stream and its offsets only);
  single   `count` dark_bwt_forward_dc_packed calls, one per block (the stream only).
A row reports per arm: wall ms of the whole list (host clock around the calls, which return after their copies), device
ms (the forward's CUDA-event time plus the DC pass's, which includes the pack kernels in the packed arms; summed over the
calls of the single arm) and the bytes copied out.  After the timed calls, the packed arm's stream is cut by its offsets,
every block unpacked by the tests' reference (tests/dc_pack_ref.c), and the CRC-32s of the four arrays compared with the
items arm's; the single arm's streams, back to back, must equal the packed arm's stream.

    python tools/dc_packed_many_probe.py [--out PATH] [--reps R]
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
    """(keep-alive, numpy view) of a host buffer, every page touched."""
    if pinned:
        t = torch.zeros(nbytes, dtype=torch.uint8).pin_memory()
        return t, t.numpy().view(dt)
    return None, np.zeros(nbytes // np.dtype(dt).itemsize, dt)


def crc(arrays):
    c = 0
    for a in arrays:
        c = zlib.crc32(memoryview(np.ascontiguousarray(a)).cast("B"), c)
    return "%08x" % (c & 0xFFFFFFFF)


def med(xs):
    return float(np.median(xs))


def probe(name, kind, seed, n, count, reps):
    total = n * count
    con = saca.Constructor(total)
    L, ctx = con._L, con._ctx
    pinned_texts = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(count)]
    for k, t in enumerate(pinned_texts):
        synth.generate(kind, seed + 100 * k, n, out=t.numpy())
    cap = _ffi.dc_packed_max(total)
    ns = (ctypes.c_uint64 * count)(*([n] * count))
    infos = (_ffi.DcInfo * count)()
    origins = (ctypes.c_uint64 * count)()
    stats = _ffi.Stats()
    for buffers in ("pinned", "pageable"):
        pinned = buffers == "pinned"
        texts = pinned_texts if pinned else [t.numpy().copy() for t in pinned_texts]
        tp = (ctypes.c_void_p * count)(*[t.data_ptr() if pinned else t.ctypes.data for t in texts])
        items = {a: host(total * WIDTH[a], pinned, np.uint8 if WIDTH[a] == 1 else np.uint32) for a in ITEMS}
        istarts = host(4 * (count + 1), pinned, np.uint32)
        stream, sstarts = host(cap, pinned), host(8 * (count + 1), pinned, np.uint64)
        one = host(_ffi.dc_packed_max(n), pinned)
        single_streams = [None] * count
        nbytes = ctypes.c_uint64(0)

        def items_arm():
            _ffi.check(L.dark_bwt_forward_dc_many(ctx, tp, ns, count, None, origins, None, istarts[1].ctypes.data,
                                                  *[items[a][1].ctypes.data for a in ITEMS], infos, ctypes.byref(stats)), ctx, "items")
            return stats.device_ms + infos[0].device_ms, int(istarts[1][count]) * sum(WIDTH.values()) + 4 * (count + 1)

        def packed_arm():
            _ffi.check(L.dark_bwt_forward_dc_packed_many(ctx, tp, ns, count, None, origins, stream[1].ctypes.data, cap,
                                                         sstarts[1].ctypes.data, ctypes.byref(nbytes), infos, ctypes.byref(stats)),
                       ctx, "packed many")
            return stats.device_ms + infos[0].device_ms, nbytes.value + 8 * (count + 1)

        def single_arm(keep=False):
            dev, out = 0.0, 0
            o, nb, info = ctypes.c_uint64(0), ctypes.c_uint64(0), _ffi.DcInfo()
            for k in range(count):
                _ffi.check(L.dark_bwt_forward_dc_packed(ctx, tp[k], n, None, ctypes.byref(o), one[1].ctypes.data, one[1].size,
                                                        ctypes.byref(nb), ctypes.byref(info), ctypes.byref(stats)), ctx, "single")
                dev += stats.device_ms + info.device_ms
                out += nb.value
                if keep:
                    single_streams[k] = one[1][:nb.value].copy()
            return dev, out

        arms = {"items": items_arm, "packed_many": packed_arm, "single_packed": single_arm}
        for f in arms.values():  # warm-up: the staging lanes, every host page, the module's kernels
            f()
        row = {"workload": name, "buffers": buffers, "blocks": count, "block_bytes": n, "reps": reps}
        for _ in range(reps):
            for arm, f in arms.items():
                t0 = time.perf_counter()
                dev, out = f()
                wall = (time.perf_counter() - t0) * 1e3
                row.setdefault(f"{arm}_ms", []).append(wall)
                row.setdefault(f"{arm}_device_ms", []).append(dev)
                row[f"{arm}_bytes_out"] = out
        # parity: the packed arm's blocks unpack to the items arm's arrays; the single calls give the same bytes
        items_arm()
        packed_arm()
        single_arm(keep=True)
        its = istarts[1].astype(np.int64)
        offs = sstarts[1].astype(np.int64)
        row["num_items"] = int(its[count])
        row["stream_bytes"] = int(nbytes.value)
        got = [[] for _ in ITEMS]
        for k in range(count):
            u = dc_pack_ref.unpack(stream[1][offs[k]:offs[k + 1]], int(its[k + 1] - its[k]))
            for j, a in enumerate(u):
                got[j].append(a)
        m = int(its[count])
        want = {a: crc([items[a][1][:m]]) for a in ITEMS}
        row["crc_items"] = want
        row["crc_unpacked_stream_equals_items"] = "ok" if {a: crc(g) for a, g in zip(ITEMS, got)} == want else "MISMATCH"
        row["single_streams_equal_packed_many"] = "ok" if np.array_equal(np.concatenate(single_streams), stream[1][:nbytes.value]) \
            else "MISMATCH"
        row["bytes_per_run_packed"] = row["stream_bytes"] / max(m, 1)
        for arm in arms:
            row[f"{arm}_median_ms"] = med(row[f"{arm}_ms"])
            row[f"{arm}_median_device_ms"] = med(row[f"{arm}_device_ms"])
        row["packed_many_speedup_over_items"] = row["items_median_ms"] / row["packed_many_median_ms"]
        row["packed_many_speedup_over_single"] = row["single_packed_median_ms"] / row["packed_many_median_ms"]
        emit(row)
        del items, istarts, stream, sstarts, one, single_streams, got, texts
    con.close()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_dc_packed_many_probe.jsonl"))
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("dc_packed_many_probe.py measures on the GPU: no CUDA device here")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    OUT = open(args.out, "w")
    card()
    kind, seed, n1 = synth.CONFIGS["c1"]
    for count in (16, 64, 256):
        probe("c1x%d" % count, kind, seed, n1, count, args.reps)
    probe("dna_1MiBx256", "dna", 1, 1 << 20, 256, args.reps)
    OUT.close()
