#!/usr/bin/env python3
"""Wall time of the blocking host entries, whose caller-buffer copies go through one copy-in and one copy-out list: the
many-block entries on lists below and above the 1 MiB staging threshold, and the single forward + DC calls on a C2 block.
One JSON line per row, printed and written to profiles/r4_host_frame_probe.jsonl (--out to change); the first line names
the card and its power limit, read in the same run.

Builds: --lib NAME=PATH, once per build (default: the in-tree library as "tree").  The library is loaded once per process,
so each build runs in a child process with DARK_BWT_LIB=PATH, and the builds take turns, --rounds times.

Workloads (texts generated once per child, the same bytes for every build):
  c1x256    256 C1-sized text blocks (768,771 bytes, text seeds 3 + 100 k): every block below the staging threshold
  3MiBx64   64 text blocks of 3 MiB (text seeds 3 + 100 k): every pageable block goes through the staging lanes
            arms, on pinned and on pageable buffers (texts and outputs):
              forward_many     dark_bwt_forward_many (BWTs, origins)
              inverse_many     dark_bwt_inverse_many of those BWTs (texts)
              forward_dc_many  dark_bwt_forward_dc_many (BWTs, origins, item offsets and the four item arrays)
  c2        one 256 MiB C2 block (dna, seed 1), pageable buffers:
              forward_dc         dark_bwt_forward_dc (BWT and the four item arrays)
              forward_dc_packed  dark_bwt_forward_dc_packed (BWT and the packed item stream)
In each child every arm is called once to warm up, then the arms take turns, --reps calls each; a call's wall time is the
host clock around it (the entries return after their copies).  A row gives, per build, the median of each child and of all
its calls, and the CRC-32 of the arm's outputs (the same in every build, or the row says MISMATCH); inverse_many is also
checked against the texts.

    python tools/host_frame_probe.py [--lib NAME=PATH ...] [--rounds R] [--reps K] [--out PATH]
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
ITEMS = ((4, np.uint32), (4, np.uint32), (1, np.uint8), (1, np.uint8))  # item_pos, item_dist, item_sym, item_rank


def host(nbytes, pinned, dt=np.uint8):
    """(keep-alive, numpy view) of a zeroed host buffer."""
    if pinned:
        import torch
        t = torch.zeros(nbytes, dtype=torch.uint8).pin_memory()
        return t, t.numpy().view(dt)
    return None, np.zeros(nbytes // np.dtype(dt).itemsize, dt)


def crc(arrays):
    c = 0
    for a in arrays:
        c = zlib.crc32(memoryview(np.ascontiguousarray(a)).cast("B"), c)
    return "%08x" % (c & 0xFFFFFFFF)


def timed(arms, reps):
    """{arm: [wall ms of each call]} after one warm-up call of each."""
    for f in arms.values():
        f()
    ms = {a: [] for a in arms}
    for _ in range(reps):
        for a, f in arms.items():
            t0 = time.perf_counter()
            f()
            ms[a].append((time.perf_counter() - t0) * 1e3)
    return ms


def many_rows(name, n, count, reps):
    from dark_b200 import _ffi, saca, synth
    total = n * count
    con = saca.Constructor(total + count)  # the inverse's rows: one '$' per block
    L, ctx = con._L, con._ctx
    ns = (ctypes.c_uint64 * count)(*([n] * count))
    origins, infos, stats = (ctypes.c_uint64 * count)(), (_ffi.DcInfo * count)(), _ffi.Stats()
    rows = []
    for buffers in ("pinned", "pageable"):
        pinned = buffers == "pinned"
        texts, bwts, back = ([host(n, pinned) for _ in range(count)] for _ in range(3))
        for k, (_, t) in enumerate(texts):
            synth.generate("text", 3 + 100 * k, n, out=t)
        istarts = host(4 * (count + 1), pinned, np.uint32)
        items = [host(total * w, pinned, dt) for w, dt in ITEMS]
        tp, bp, xp = ((ctypes.c_void_p * count)(*[a.ctypes.data for _, a in arrs]) for arrs in (texts, bwts, back))

        def forward_many():
            _ffi.check(L.dark_bwt_forward_many(ctx, tp, ns, bp, origins, count, ctypes.byref(stats)), ctx, "forward_many")

        def inverse_many():
            _ffi.check(L.dark_bwt_inverse_many(ctx, bp, ns, origins, xp, count, None), ctx, "inverse_many")

        def forward_dc_many():
            _ffi.check(L.dark_bwt_forward_dc_many(ctx, tp, ns, count, bp, origins, None, istarts[1].ctypes.data,
                                                  *[a.ctypes.data for _, a in items], infos, ctypes.byref(stats)), ctx, "forward_dc_many")

        ms = timed({"forward_many": forward_many, "inverse_many": inverse_many, "forward_dc_many": forward_dc_many}, reps)
        m = int(istarts[1][count])
        forward = [b for _, b in bwts] + [np.ctypeslib.as_array(origins)]
        out = {"forward_many": crc(forward),
               "inverse_many": crc([x for _, x in back]) if all(np.array_equal(x, t) for (_, x), (_, t) in zip(back, texts))
               else "NOT THE TEXTS",
               "forward_dc_many": crc(forward + [istarts[1]] + [a[:m] for _, a in items])}
        for arm in ms:
            rows.append({"workload": name, "buffers": buffers, "arm": arm, "blocks": count, "block_bytes": n, "ms": ms[arm],
                         "crc": out[arm]})
        del texts, bwts, back, items
    con.close()
    return rows


def c2_rows(reps):
    from dark_b200 import _ffi, saca, synth
    kind, seed, n = synth.CONFIGS["c2"]
    text = synth.generate(kind, seed, n)
    bwt = np.zeros(n, np.uint8)
    items = [np.zeros(n, dt) for _, dt in ITEMS]
    stream = np.zeros(_ffi.dc_packed_max(n), np.uint8)
    origin, nbytes, info, stats = ctypes.c_uint64(0), ctypes.c_uint64(0), _ffi.DcInfo(), _ffi.Stats()
    with saca.Constructor(n) as con:
        L, ctx = con._L, con._ctx

        def forward_dc():
            _ffi.check(L.dark_bwt_forward_dc(ctx, text.ctypes.data, n, bwt.ctypes.data, ctypes.byref(origin), None,
                                             *[a.ctypes.data for a in items], ctypes.byref(info), ctypes.byref(stats)), ctx, "forward_dc")

        def forward_dc_packed():
            _ffi.check(L.dark_bwt_forward_dc_packed(ctx, text.ctypes.data, n, bwt.ctypes.data, ctypes.byref(origin), stream.ctypes.data,
                                                    stream.size, ctypes.byref(nbytes), ctypes.byref(info), ctypes.byref(stats)),
                       ctx, "forward_dc_packed")

        ms = {}
        out = {}
        for arm, f in (("forward_dc", forward_dc), ("forward_dc_packed", forward_dc_packed)):
            ms.update(timed({arm: f}, reps))
            m = int(info.num_items)
            out[arm] = crc([bwt, np.array([origin.value], np.uint64)] + ([a[:m] for a in items] if arm == "forward_dc"
                                                                          else [stream[:nbytes.value]]))
    return [{"workload": "c2", "buffers": "pageable", "arm": arm, "blocks": 1, "block_bytes": n, "ms": ms[arm], "crc": out[arm]}
            for arm in ms]


def child(reps):
    sys.path.insert(0, ROOT)
    rows = many_rows("c1x256", 768771, 256, reps) + many_rows("3MiBx64", 3 << 20, 64, reps) + c2_rows(reps)
    for r in rows:
        print("ROW " + json.dumps(r), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], metavar="NAME=PATH")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_host_frame_probe.jsonl"))
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        return child(args.reps)
    libs = [tuple(s.split("=", 1)) for s in args.lib] or [("tree", os.path.join(ROOT, "dark_b200", "lib", "libdark_bwt.so"))]
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    if q.returncode != 0 or not q.stdout.strip():
        sys.exit("host_frame_probe.py measures on the GPU: nvidia-smi finds no device here")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    out = open(args.out, "w")

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    emit({"card": q.stdout.strip().splitlines()[0], "builds": dict(libs), "rounds": args.rounds, "reps": args.reps})
    table = {}  # (workload, buffers, arm) -> row
    for rnd in range(args.rounds):
        for name, path in libs:
            env = dict(os.environ, DARK_BWT_LIB=os.path.abspath(path))
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--reps", str(args.reps)], env=env,
                               capture_output=True, text=True)
            if p.returncode != 0:
                sys.exit("build %s, round %d failed:\n%s" % (name, rnd, p.stderr[-3000:]))
            for line in p.stdout.splitlines():
                if not line.startswith("ROW "):
                    continue
                r = json.loads(line[4:])
                row = table.setdefault((r["workload"], r["buffers"], r["arm"]),
                                       {k: r[k] for k in ("workload", "buffers", "arm", "blocks", "block_bytes")})
                row.setdefault(name + "_child_median_ms", []).append(float(np.median(r["ms"])))
                row.setdefault(name + "_all_ms", []).extend(r["ms"])
                row.setdefault("crc", {}).setdefault(name, set()).add(r["crc"])
    for row in table.values():
        for name, _ in libs:
            row[name + "_median_ms"] = float(np.median(row.pop(name + "_all_ms")))
        crcs = set().union(*row["crc"].values())
        row["crc"] = crcs.pop() if len(crcs) == 1 else "MISMATCH %s" % {k: sorted(v) for k, v in row["crc"].items()}
        if len(libs) == 2:
            row["%s_over_%s" % (libs[1][0], libs[0][0])] = row[libs[1][0] + "_median_ms"] / row[libs[0][0] + "_median_ms"]
        emit(row)
    out.close()


if __name__ == "__main__":
    main()
