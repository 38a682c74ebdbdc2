#!/usr/bin/env python3
"""Record the control flow of the single-block forward transform (needs a B200).

    python tests/golden/make_forward_fingerprint.py

writes tests/golden/forward_fingerprint.json.  For each case it keeps what the call reports in dark_bwt_stats
except the timings (alphabet, initial symbols, rounds, pairs rounds, radix passes per round, active suffixes per
round, elements sorted, key-generating passes, kernel launches, host round trips), and the origin and CRC-32 of
the BWT.  Two runs of the same driver give the same record, so a refactor of the driver must leave the file as it
is; a change that alters the driver's decisions on purpose regenerates it and says so.

The cases are the test knobs' forced paths of tests/test_gpu_parity.py (one process per environment, the knobs
are read when a context is created), the same inputs with default knobs, the medium golden shapes, the structured,
pairs-mode and sparse-fallback inputs, a context without alphabet packing, and one call each through
dark_bwt_forward_device and dark_bwt_forward_batch.
"""
import ctypes
import json
import os
import subprocess
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.dirname(HERE)):
    if p not in sys.path:
        sys.path.insert(0, p)

OUT = os.path.join(HERE, "forward_fingerprint.json")
BATCH = ["synth:text:3:768771", "synth:dna:1:1048576", "synth:rep17:2:1048576"]


def cases():
    """{case name: (environment, input names, entry)}; entry is host, nopack, device or batch."""
    import test_gpu_parity as P
    out = {}
    for env, kind, seed, n in P.FORCED_PATHS:
        inp = f"synth:{kind}:{seed}:{n}"
        out[",".join(f"{k}={v}" for k, v in sorted(env.items())) + "/" + inp] = (env, [inp], "host")
        out["default/" + inp] = ({}, [inp], "host")
    for key in P.MEDIUM:
        out["default/synth:" + key] = ({}, ["synth:" + key], "host")
    for group, names in (("structured", P._structured_inputs()), ("pairs", P._pairs_inputs()),
                         ("sparse", P._sparse_fallback_inputs())):
        for name in names:
            out[f"default/{group}:{name}"] = ({}, [f"{group}:{name}"], "host")
    out["nopack/synth:mixed:4:1048576"] = ({}, ["synth:mixed:4:1048576"], "nopack")
    out["nopack/pairs:planted_dna"] = ({}, ["pairs:planted_dna"], "nopack")
    out["device/synth:dna:1:1048576"] = ({}, ["synth:dna:1:1048576"], "device")
    out["batch/" + "+".join(BATCH)] = ({}, BATCH, "batch")
    return out


def _input(name):
    import test_gpu_parity as P
    from dark_b200 import synth
    group, rest = name.split(":", 1)
    if group == "synth":
        kind, seed, n = rest.split(":")
        return synth.generate(kind, int(seed), int(n))
    table = {"structured": P._structured_inputs, "pairs": P._pairs_inputs, "sparse": P._sparse_fallback_inputs}[group]()
    t = table[rest]
    return np.frombuffer(t, dtype=np.uint8) if isinstance(t, bytes) else np.ascontiguousarray(t, dtype=np.uint8)


def _record(st, bwt, origin):
    rec = {}
    for field, _ in type(st)._fields_:
        if field.endswith("_ms") or field == "reserved_":
            continue
        v = getattr(st, field)
        rec[field] = [int(x) for x in v] if hasattr(v, "__len__") else int(v)
    rec["origin"] = int(origin)
    rec["bwt_crc32"] = "%08x" % (zlib.crc32(np.ascontiguousarray(bwt).tobytes()) & 0xFFFFFFFF)
    return rec


def run(names):
    """The records of the named cases, in this process (its environment holds their knobs)."""
    from dark_b200 import _ffi, saca
    table = cases()
    res = {}
    for name in names:
        _, inputs, entry = table[name]
        ts = [_input(i) for i in inputs]
        if entry in ("host", "nopack"):
            flags = _ffi.F_NO_ALPHABET_PACKING if entry == "nopack" else _ffi.F_DEFAULT
            with saca.Constructor(ts[0].size, flags=flags) as c:
                bwt, origin = c.bwt(ts[0])
                res[name] = [_record(c.stats, bwt, origin)]
        elif entry == "device":
            import torch
            with saca.Constructor(ts[0].size, flags=_ffi.F_DEVICE_ONLY) as c:
                d_text = torch.from_numpy(ts[0]).cuda()
                d_bwt = torch.empty(ts[0].size, dtype=torch.uint8, device="cuda")
                origin = c.bwt_device(d_text.data_ptr(), ts[0].size, d_bwt.data_ptr())
                res[name] = [_record(c.stats, d_bwt.cpu().numpy(), origin)]
        else:
            outs = [np.empty(t.size, dtype=np.uint8) for t in ts]
            with saca.Constructor(max(t.size for t in ts)) as c:
                stats = (_ffi.Stats * len(ts))()
                origins = (ctypes.c_uint64 * len(ts))()
                T = (ctypes.c_void_p * len(ts))(*[t.ctypes.data for t in ts])
                B = (ctypes.c_void_p * len(ts))(*[o.ctypes.data for o in outs])
                N = (ctypes.c_uint64 * len(ts))(*[t.size for t in ts])
                _ffi.check(c._L.dark_bwt_forward_batch(c._ctx, T, N, B, origins, None, len(ts), stats), c._ctx, "batch")
                res[name] = [_record(stats[k], outs[k], origins[k]) for k in range(len(ts))]
    return res


def collect():
    """Every case's records: one process per environment."""
    groups = {}
    for name, (env, _, _) in cases().items():
        groups.setdefault(json.dumps(env, sort_keys=True), []).append(name)
    res = {}
    for env_key, names in groups.items():
        env = dict(os.environ, **json.loads(env_key))
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--run", json.dumps(names)], env=env, cwd=ROOT,
                             capture_output=True, text=True, timeout=1800)
        if out.returncode != 0:
            raise RuntimeError(f"fingerprint run with {env_key} failed:\n{out.stderr[-3000:]}")
        res.update(json.loads(out.stdout.strip().splitlines()[-1]))
    return res


def main():
    if len(sys.argv) == 3 and sys.argv[1] == "--run":
        print(json.dumps(run(json.loads(sys.argv[2]))))
        return
    res = collect()
    with open(OUT, "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(res[k])}" for k in sorted(res)) + "\n}\n")
    print(f"wrote {len(res)} cases to {OUT}")


if __name__ == "__main__":
    main()
