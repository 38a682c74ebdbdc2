#!/usr/bin/env python3
"""One device-resident forward BWT of a named workload (quick timing).
    python tools/profile_step.py <c1|c2|c3|c4|c5> [reps] [n_override]"""
import json
import os
import sys
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from dark_b200 import saca, synth, _ffi  # noqa: E402

name = sys.argv[1] if len(sys.argv) > 1 else "c2"
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 1
kind, seed, n = synth.CONFIGS.get(name, ("mixed", 1000, 1 << 28))
if len(sys.argv) > 3:
    n = int(sys.argv[3])
flags = _ffi.F_DEVICE_ONLY | (_ffi.F_NO_ALPHABET_PACKING if os.environ.get("CANONICAL") else 0)
text = synth.generate(kind, seed, n)
con = saca.Constructor(n, flags=flags)
dt = torch.from_numpy(text).cuda()
db = torch.empty(n, dtype=torch.uint8, device="cuda")
for _ in range(reps):
    origin = con.bwt_device(dt.data_ptr(), n, db.data_ptr())
    st = con.stats.as_dict()
    print(json.dumps({"workload": name, "n": n, "origin": origin, **{k: st[k] for k in (
        "sigma", "symbols_per_key", "initial_symbols", "rounds", "sort_passes", "kernel_launches", "host_syncs", "device_ms", "init_ms", "sort_ms", "pass_ms",
        "keybuild_ms", "rerank_ms", "emit_ms", "active", "passes")}}))
# the timing is only worth reading if the bytes are right: CRC-32 of the BWT against the committed oracle fixture
gold = json.load(open(os.path.join(ROOT, "tests", "golden", "oracle_golden.json")))
key = "%s:%d:%d" % (kind, seed, n)
if key in gold:
    crc = "%08x" % (zlib.crc32(db.cpu().numpy().tobytes()) & 0xFFFFFFFF)
    ok = crc == gold[key]["bwt_crc32"] and origin == gold[key]["origin"]
    print(json.dumps({"workload": name, "parity": "ok" if ok else "MISMATCH", "bwt_crc32": crc}))
    if not ok:
        sys.exit(3)
con.close()
