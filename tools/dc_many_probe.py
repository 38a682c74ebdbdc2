#!/usr/bin/env python3
"""Distance coding of many blocks in one pass, against the single-block calls it replaces.  One JSON line per
measurement; the first line names the card and its power limit, read in the same run.

  many   1, 4, 16, 64, 256 DISTINCT C1-sized text blocks (768,771 bytes, seeds 3 + 100 k as in inverse_many_probe.py):
         - device ms of one dark_bwt_dc_encode_many_device pass over the blocks back to back, against the summed device ms
           of single dark_bwt_dc_encode_device calls on the same blocks;
         - wall ms of one dark_bwt_forward_dc_many call (pinned host buffers), against `count` sequential
           dark_bwt_forward_dc calls;
         - per-block equality of every output with the single calls.
  large  one 256 MiB C2 BWT (dna, seed 1) through dark_bwt_dc_encode_many_device with count = 1, against
         dark_bwt_dc_encode_device, alternated: what the many-block instantiations cost the large single-block case.

    python tools/dc_many_probe.py [many|large|all]
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


def dev_outputs(n, cnt):
    i32 = lambda m: torch.empty(m, dtype=torch.int32, device="cuda")  # noqa: E731
    u8 = lambda m: torch.empty(m, dtype=torch.uint8, device="cuda")  # noqa: E731
    return {"dist": i32(n), "starts": i32(cnt + 1), "pos": i32(n), "idist": i32(n), "sym": u8(n), "rank": u8(n)}


def probe_many():
    kind, seed, n = synth.CONFIGS["c1"]
    for cnt in (1, 4, 16, 64, 256):
        total = cnt * n
        texts = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(cnt)]
        for k in range(cnt):
            synth.generate(kind, seed + 100 * k, n, out=texts[k].numpy())
        con = saca.Constructor(total)
        L, ctx = con._L, con._ctx
        # the BWTs, back to back on the device (the layout forward_many_device writes)
        d_text = torch.cat([t.cuda() for t in texts])
        starts = torch.tensor([k * n for k in range(cnt + 1)], dtype=torch.int32, device="cuda")
        d_bwt = torch.empty(total, dtype=torch.uint8, device="cuda")
        d_org = torch.empty(cnt, dtype=torch.int64, device="cuda")
        con.bwt_many_device(d_text.data_ptr(), starts.data_ptr(), cnt, d_bwt.data_ptr(), d_org.data_ptr())
        del d_text
        o = dev_outputs(total, cnt)
        args = [o[k].data_ptr() for k in ("dist", "starts", "pos", "idist", "sym", "rank")]
        con.dc_encode_many_device(d_bwt.data_ptr(), starts.data_ptr(), cnt, *args)  # warm-up
        reps = max(3, 256 // cnt)
        many_ms = 0.0
        for _ in range(reps):
            infos, ms = con.dc_encode_many_device(d_bwt.data_ptr(), starts.data_ptr(), cnt, *args)
            many_ms += ms
        many_ms /= reps
        h = {k: v.cpu().numpy() for k, v in o.items()}
        its = h["starts"].view(np.uint32)
        # the same blocks one dc_encode_device call each (outputs compared block by block)
        s = dev_outputs(n, 0)
        sargs = [s[k].data_ptr() for k in ("dist", "pos", "idist", "sym", "rank")]
        con.dc_encode_device(d_bwt.data_ptr(), n, *sargs)  # warm-up
        single_ms, parity = 0.0, True
        for k in range(cnt):
            info = con.dc_encode_device(d_bwt.data_ptr() + k * n, n, *sargs)
            single_ms += info.device_ms
            a, e = int(its[k]), int(its[k + 1])
            m = int(info.num_items)
            parity &= m == e - a == int(infos[k].num_items) and info.num_unique == infos[k].num_unique
            parity &= list(info.init) == list(infos[k].init) and list(info.mtf_symbols) == list(infos[k].mtf_symbols)
            parity &= np.array_equal(s["dist"].cpu().numpy(), h["dist"][k * n:(k + 1) * n])
            for key in ("pos", "idist", "sym", "rank"):
                parity &= np.array_equal(s[key].cpu().numpy()[:m], h[key][a:e])
        del o, s
        # host entries: forward_dc_many against count forward_dc calls (pinned text in, pageable outputs as bwt_dc uses)
        tp = [t.data_ptr() for t in texts]
        bwts = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(cnt)]
        out = {"dist": np.empty(total, np.uint32), "starts": np.empty(cnt + 1, np.uint32), "pos": np.empty(total, np.uint32),
               "idist": np.empty(total, np.uint32), "sym": np.empty(total, np.uint8), "rank": np.empty(total, np.uint8)}
        optr = [out[k].ctypes.data for k in ("dist", "starts", "pos", "idist", "sym", "rank")]
        infos_h = (_ffi.DcInfo * cnt)()
        origins = (ctypes.c_uint64 * cnt)()

        def fdm():
            _ffi.check(L.dark_bwt_forward_dc_many(ctx, (ctypes.c_void_p * cnt)(*tp), (ctypes.c_uint64 * cnt)(*([n] * cnt)), cnt,
                                                  (ctypes.c_void_p * cnt)(*[b.data_ptr() for b in bwts]), origins, *optr, infos_h,
                                                  None), ctx, "forward_dc_many")
        single = {"dist": np.empty(n, np.uint32), "pos": np.empty(n, np.uint32), "idist": np.empty(n, np.uint32),
                  "sym": np.empty(n, np.uint8), "rank": np.empty(n, np.uint8)}
        sptr = [single[k].ctypes.data for k in ("dist", "pos", "idist", "sym", "rank")]
        sb = torch.empty(n, dtype=torch.uint8).pin_memory()
        sinfo, sorg = _ffi.DcInfo(), ctypes.c_uint64(0)

        def fdc(k):
            _ffi.check(L.dark_bwt_forward_dc(ctx, tp[k], n, sb.data_ptr(), ctypes.byref(sorg), *sptr, ctypes.byref(sinfo), None), ctx,
                       "forward_dc")
        fdm(), fdc(0)  # warm-up
        reps_h = max(2, 32 // cnt)
        t0 = time.perf_counter()
        for _ in range(reps_h):
            fdm()
        many_wall = (time.perf_counter() - t0) / reps_h * 1e3
        single_wall = 0.0
        fused_parity = True
        for k in range(cnt):
            t0 = time.perf_counter()
            fdc(k)
            single_wall += (time.perf_counter() - t0) * 1e3
            a, e = int(out["starts"][k]), int(out["starts"][k + 1])
            m = int(sinfo.num_items)
            fused_parity &= int(sorg.value) == int(origins[k]) and torch.equal(sb, bwts[k]) and m == e - a
            fused_parity &= list(sinfo.init) == list(infos_h[k].init) and np.array_equal(single["dist"], out["dist"][k * n:(k + 1) * n])
            for key in ("pos", "idist", "sym", "rank"):
                fused_parity &= np.array_equal(single[key][:m], out[key][a:e])
        emit({"many": cnt, "block_bytes": n, "dc_many_device_ms": many_ms, "dc_single_device_ms_sum": single_ms,
              "device_ratio_many_over_single": many_ms / single_ms, "forward_dc_many_wall_ms": many_wall,
              "forward_dc_single_wall_ms_sum": single_wall, "wall_ratio_many_over_single": many_wall / single_wall,
              "dc_many_device_GBps": total / many_ms / 1e6, "calls": reps, "host_calls": reps_h,
              "parity_dc_many_vs_single": "ok" if parity else "MISMATCH",
              "parity_forward_dc_many_vs_single": "ok" if fused_parity else "MISMATCH"})
        con.close()
        del texts, bwts, d_bwt


def probe_large():
    n = 1 << 28
    text = torch.empty(n, dtype=torch.uint8)
    synth.generate("dna", 1, n, out=text.numpy())
    con = saca.Constructor(n)
    d_text = text.cuda()
    d_bwt = torch.empty(n, dtype=torch.uint8, device="cuda")
    con.bwt_device(d_text.data_ptr(), n, d_bwt.data_ptr())
    del d_text
    starts = torch.tensor([0, n], dtype=torch.int32, device="cuda")
    a = dev_outputs(n, 1)
    b = dev_outputs(n, 0)
    margs = [a[k].data_ptr() for k in ("dist", "starts", "pos", "idist", "sym", "rank")]
    sargs = [b[k].data_ptr() for k in ("dist", "pos", "idist", "sym", "rank")]
    con.dc_encode_many_device(d_bwt.data_ptr(), starts.data_ptr(), 1, *margs)
    con.dc_encode_device(d_bwt.data_ptr(), n, *sargs)
    many, single = [], []
    for _ in range(5):  # alternated
        many.append(con.dc_encode_many_device(d_bwt.data_ptr(), starts.data_ptr(), 1, *margs)[1])
        single.append(con.dc_encode_device(d_bwt.data_ptr(), n, *sargs).device_ms)
    info = con.dc_encode_device(d_bwt.data_ptr(), n, *sargs)
    m = int(info.num_items)
    ok = all(torch.equal(a[x][:m], b[y][:m]) for x, y in (("pos", "pos"), ("idist", "idist"), ("sym", "sym"), ("rank", "rank")))
    ok &= torch.equal(a["dist"], b["dist"])
    emit({"large": "c2 dna 256 MiB", "count": 1, "dc_many_device_ms": many, "dc_single_device_ms": single,
          "many_median_ms": float(np.median(many)), "single_median_ms": float(np.median(single)),
          "parity": "ok" if ok else "MISMATCH"})
    con.close()


if not torch.cuda.is_available():
    sys.exit("dc_many_probe.py measures on the GPU: no CUDA device here")
card()
if what in ("many", "all"):
    probe_many()
if what in ("large", "all"):
    probe_large()
