#!/usr/bin/env python3
"""bench.py — BWT-forward throughput of the B200-native path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload c2|c3|c5|c1|c4]
                    [--dump-outputs DIR]

A "step" is one forward BWT (suffix sort + BWT emission + origin) of one synthetic block per GPU.
Default workload = BASELINE.json configs[1]: a 256 MiB block of DNA-like 4-symbol text (C2).
N > 1 (launched by torchrun, one rank per GPU): every rank transforms its own block of the same
shape — independent blocks, no data-path collective (SURVEY.md §8e) — weak scaling.

JSON line (rank 0): value = total input MB / max-over-ranks device time; `e2e` = the same metric
through the host-buffer C-ABI call (pinned host -> H2D -> transform -> D2H) timed by wall clock, with the
latency of one isolated call from pinned and from pageable (malloc) buffers beside it;
`roofline` = the radix-pass kernel (dominant) against the measured HBM copy bandwidth, the key-generating
first pass counted at its own 13 B per suffix;
`cpu_baseline` = the oracle (C restatement of the reference's saca.rs + emission) on one host core;
`workloads` = C3 and one C5 block through the same context (device ms, BWT CRC-32 against the committed
oracle fixtures); with N > 1 also `c5` (blocks mixed(1000+b), b = rank, rank+N, ... through the pipelined
batch entry) and `copy_only` (the same H2D/D2H traffic with the transform skipped: the box's copy ceiling).

`--impl reference` times that CPU restatement on all host cores (the reference is Rust and cannot
be compiled in this image; see DESIGN.md), same metric/config/unit.  .dark byte identity and the C1 CLI
round trip of the reference cannot be tested in this image (no rustc/cargo, no golden .dark file).

`--dump-outputs DIR` writes what the last timed step returned to its caller (rank 0's block) as DIR/*.npy, so that
two builds can be compared output for output on the same seeded inputs: see dump_outputs().
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "bwt_forward_throughput"
UNIT = "MB/s"

WORKLOADS = {
    # name: (kind, base_seed, n, description, B_alg per input byte (SURVEY §8d / tests/golden), sum_m/N)
    "c1": ("text", 3, 768771, "C1: 768 KB English-like text block text(seed=3)", 366.437),
    "c2": ("dna", 1, 1 << 28, "C2: 256 MiB synthetic DNA-like 4-symbol block dna(seed=1+rank)", 497.5),
    "c3": ("rep17", 2, 1 << 26, "C3: 64 MiB period-17 block with sparse mutations rep17(seed=2+rank)", 2342.0),
    "c4": ("mixed", 4, 1 << 31, "C4: 2 GiB mixed binary/text block mixed(seed=4+rank)", 461.4),
    "c5": ("mixed", 1000, 1 << 28, "C5 block: 256 MiB mixed binary/text block mixed(seed=1000+rank)", 445.8),
}


def measured_pass_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one radix-pass launch, from the ncu --set full capture committed
    under profiles/ (NOT measured by this run), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ncu_pass_traffic.json")) as f:
            t = json.load(f)
        return {"bytes_per_launch": t["dram__bytes_read.sum"] + t["dram__bytes_write.sum"], "pairs_per_launch": t["pairs_per_launch"],
                "algorithmic_bytes_per_launch": t["algorithmic_bytes_per_launch"],
                "source": "committed ncu capture profiles/r2_ncu_pass_traffic.json (not measured by this run)"}
    except Exception:
        return None


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled in-process every 2 ms (a timed region
    of 20 C2 steps lasts 0.2 s, less than `nvidia-smi` needs to start), `nvidia-smi -lms 20` when NVML cannot be loaded.
    begin() / stop() bracket the timed region; only samples taken between them count."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.rows, self.proc, self.nvml, self.h = [], None, None, None   # rows: (time, sm MHz, max MHz, [reason names])
        self.t0 = self.t1 = None
        self.running = True
        self.how = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
            self.how = "nvml"
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.how = "nvidia-smi"
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _sample_nvml(self):
        n = self.nvml
        sm = float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
        mx = float(n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM))
        try:
            bits = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            bits = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        masks = [getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8), getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20), getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)]
        return (time.perf_counter(), sm, mx, [nm for nm, m in zip(self.NAMES, masks) if bits & m])

    def _poll_nvml(self):
        while self.running:
            try:
                self.rows.append(self._sample_nvml())
            except Exception:
                pass
            time.sleep(0.002)

    def _read_smi(self):
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            if len(r) >= 7 and r[0].replace(".", "").isdigit() and r[1].replace(".", "").isdigit():
                self.rows.append((time.perf_counter(), float(r[0]), float(r[1]),
                                  [nm for k, nm in enumerate(self.NAMES) if r[3 + k].lower() == "active"]))

    def begin(self):
        self.t0 = time.perf_counter()

    def stop(self):
        self.t1 = time.perf_counter()
        if self.how is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML and no nvidia-smi"], "samples": 0}
        self.running = False
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        self.thread.join(timeout=2)
        t0 = self.t0 if self.t0 is not None else 0.0
        inside = [r for r in self.rows if t0 <= r[0] <= self.t1]
        where = "inside the timed region"
        if not inside and self.rows:   # the sampler was slower than the region: the samples nearest to it (warm-up / just after)
            inside = self.rows[-3:]
            where = "nearest to the timed region (none fell inside)"
        sm, mx = [r[1] for r in inside], [r[2] for r in inside]
        reasons = sorted({nm for r in inside for nm in r[3]})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": self.how, "window": where}


def cpu_oracle_rate(kind, seed, sample_n, threads, steps, warmup):
    """MB/s of the oracle (saca.rs restatement + emission) with `threads` host threads, each on
    its own block of sample_n bytes per step.  ctypes drops the GIL during the C call."""
    import numpy as np
    import oracle
    oracle.lib()
    texts = [oracle.gen(kind, seed + t, sample_n) for t in range(threads)]
    arenas = [oracle.Arena(sample_n) for _ in range(threads)]
    per_step = []

    def work(t):
        arenas[t].bwt_forward(texts[t])

    for it in range(warmup + steps):
        ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        t0 = time.perf_counter()
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        dt = time.perf_counter() - t0
        if it >= warmup:
            per_step.append(dt)
    total = sum(per_step)
    return threads * sample_n * len(per_step) / 1e6 / total, total / len(per_step)


def full_size_cpu_figures():
    """One-off CPU timings of the FULL-size configurations on a GPU box's host cores (tools/cpu_full_size.py; committed
    under profiles/ with the command that made them): C2/C3 one thread on the whole block, C5 one wave of nproc blocks."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_cpu_full_size.json")) as f:
            return json.load(f)
    except Exception:
        return None


def run_reference(args, rank):
    """Reference arm: the reference's CPU algorithm (oracle restatement; the Rust original cannot be
    built here) on all host cores.  Rank 0 only."""
    if rank != 0:
        return
    kind, seed, n, desc, _ = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    total_steps = args.steps + args.warmup
    # the largest per-thread sample that keeps the whole run within a few minutes: the oracle sorts about 7 MB/s per
    # thread when every core is busy, so a 32 MiB sample costs ~5 s per step (64 MiB for very short runs)
    sample_n = min(n, (1 << 26) if total_steps <= 8 else (1 << 25) if total_steps <= 30 else (1 << 24))
    rate, step_s = cpu_oracle_rate(kind, seed, sample_n, cores, args.steps, args.warmup)
    sample = f"{cores} threads x one {sample_n}-byte {kind} block per step (prefix-shaped sample of the {n}-byte block)"
    full = full_size_cpu_figures()
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": desc, "block_bytes": n, "sample_bytes": sample_n,
                   "note": "CPU restatement of the reference's saca.rs + TransformIterator (oracle port; Rust reference "
                           "not buildable in this image), all host cores, one bounded sample block per thread and step: "
                           "NOT the same configuration as the GPU arm's single full-size block (a full-size block is "
                           "slower per byte: caches), so the ratio is a floor; the one-off full-size figures are in "
                           "full_size_one_off",
                   "full_size_one_off": full},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def crc32_of(t):
    import zlib
    return "%08x" % (zlib.crc32(t.numpy().tobytes()) & 0xFFFFFFFF)


DUMP_SAMPLE = 1 << 22   # BWT positions --dump-outputs writes: 16 MiB of float32 bytes + 32 MiB of float64 positions
DUMP_SEED = 20261020


def dump_outputs(out_dir, torch, d_bwt, origin):
    """Write what one forward call returns to its caller: origin.npy (the origin, float64[1]), bwt.npy (BWT bytes as
    float32) and bwt_index.npy (the block positions of those bytes, float64).  A block of more than DUMP_SAMPLE bytes
    is sampled at DUMP_SAMPLE distinct positions drawn with a fixed seed, so equal arguments give equal positions;
    the CRC-32 of the whole BWT is `config.bwt_crc32` of the JSON line."""
    import numpy as np
    n = d_bwt.numel()
    if n <= DUMP_SAMPLE:
        idx = np.arange(n, dtype=np.int64)
    else:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_SAMPLE, replace=False))
    vals = d_bwt[torch.from_numpy(idx).to(d_bwt.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "origin.npy"), np.array([origin], dtype=np.float64))
    np.save(os.path.join(out_dir, "bwt.npy"), vals.astype(np.float32))
    np.save(os.path.join(out_dir, "bwt_index.npy"), idx.astype(np.float64))


def golden_fixtures():
    try:
        with open(os.path.join(ROOT, "tests", "golden", "oracle_golden.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def run_side_workload(con, torch, dev, name, steps, gold):
    """A few device-resident steps of another configuration through the same context: device ms, phases, launches,
    and the BWT bytes checked by CRC-32 against the committed oracle fixture."""
    from dark_b200 import synth
    kind, seed, n, desc, balg = WORKLOADS[name]
    h = torch.empty(n, dtype=torch.uint8).pin_memory()
    synth.generate(kind, seed, n, out=h.numpy())
    d_text = h.to(dev)
    d_bwt = torch.empty(n, dtype=torch.uint8, device=dev)
    origin = con.bwt_device(d_text.data_ptr(), n, d_bwt.data_ptr())  # warm
    ms = []
    for _ in range(steps):
        origin = con.bwt_device(d_text.data_ptr(), n, d_bwt.data_ptr())
        ms.append(con.stats.device_ms)
    st = con.stats.as_dict()
    crc = crc32_of(d_bwt.cpu())
    fx = gold.get("%s:%d:%d" % (kind, seed, n))
    peak, _ = measured_peak_gbs()
    best = min(ms)
    return {"workload": desc, "block_bytes": n, "steps": steps, "device_ms": statistics.median(ms), "device_ms_min": best,
            "value": n / 1e6 / (statistics.median(ms) / 1e3), "unit": UNIT, "origin": origin, "bwt_crc32": crc,
            "parity": ("ok" if (fx and fx["bwt_crc32"] == crc and fx["origin"] == origin) else ("MISMATCH" if fx else "no fixture")),
            "rounds": st["rounds"], "sort_passes": st["sort_passes"], "kernel_launches": st["kernel_launches"], "host_syncs": st["host_syncs"],
            "phases_ms": {k: st[k] for k in ("init_ms", "sort_ms", "pass_ms", "gen_pass_ms", "keybuild_ms", "rerank_ms", "emit_ms")},
            "path_b_alg_per_byte": balg, "path_frac_of_measured_peak": balg * n / (best / 1e3) / 1e9 / peak}


def run_native(args, rank, local_rank, world):
    import numpy as np
    import torch
    import torch.distributed as dist
    from dark_b200 import saca, synth, blocks

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the forward BWT has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    kind, base_seed, n, desc, balg_per_byte = WORKLOADS[args.workload]
    seed = base_seed + rank
    # pinned host input/output (the caller's buffers of the host entry point)
    h_text = torch.empty(n, dtype=torch.uint8).pin_memory()
    h_bwt = torch.empty(n, dtype=torch.uint8).pin_memory()
    synth.generate(kind, seed, n, out=h_text.numpy())
    con = saca.Constructor(n, device=local_rank)
    d_text = h_text.to(dev, non_blocking=False)
    d_bwt = torch.empty(n, dtype=torch.uint8, device=dev)
    stream = torch.cuda.ExternalStream(con.stream, device=dev)
    gold = golden_fixtures()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident steps
    sampler = ClockSampler(local_rank) if rank == 0 else None   # started before the warm-up, counted from begin() on
    for _ in range(args.warmup):
        origin = con.bwt_device(d_text.data_ptr(), n, d_bwt.data_ptr())
    # B_alg of THIS block, measured on the GPU from the suffix array (dark_bwt_lcp_profile_device), outside the timed
    # region; it must agree with the oracle profiler's committed figure for the workload
    balg_live = None
    if rank == 0 and n <= (1 << 29):
        d_sa = torch.empty(n, dtype=torch.int32, device=dev)
        con.bwt_device(d_text.data_ptr(), n, d_bwt.data_ptr(), d_sa.data_ptr())
        prof = con.lcp_profile_device(d_text.data_ptr(), n, d_sa.data_ptr())
        balg_live = prof["b_alg"] / n
        del d_sa
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    agg = {"pass_ms": 0.0, "gen_pass_ms": 0.0, "sorted": 0, "gen_sorted": 0, "passes": 0, "gen_passes": 0, "device_ms": 0.0, "init_ms": 0.0,
           "sort_ms": 0.0, "keybuild_ms": 0.0, "rerank_ms": 0.0, "emit_ms": 0.0, "host_syncs": 0}
    if sampler:
        sampler.begin()
    ev0.record(stream)
    for _ in range(args.steps):
        origin = con.bwt_device(d_text.data_ptr(), n, d_bwt.data_ptr())
        s = con.stats
        launches += s.kernel_launches
        agg["pass_ms"] += s.pass_ms
        agg["gen_pass_ms"] += s.gen_pass_ms
        agg["sorted"] += s.sorted_elements
        agg["gen_sorted"] += s.gen_elements
        agg["passes"] += s.sort_passes
        agg["gen_passes"] += s.gen_passes
        agg["host_syncs"] += s.host_syncs
        for k in ("device_ms", "init_ms", "sort_ms", "keybuild_ms", "rerank_ms", "emit_ms"):
            agg[k] += getattr(s, k)
    ev1.record(stream)
    barrier()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, d_bwt, origin)
    ms_total = ev0.elapsed_time(ev1)
    stats = con.stats.as_dict()
    fx = gold.get("%s:%d:%d" % (kind, seed, n))
    main_crc = crc32_of(d_bwt.cpu()) if rank == 0 else None

    # ---- end to end through the host-buffer C-ABI: pinned host blocks in, BWT bytes + origin out, every
    # copy inside the timed region.  Blocks go through the pipelined batch entry (dark_bwt_forward_batch:
    # copy-in of block k+1 / copy-out of block k-1 overlap the transform of block k), which is how a
    # corpus of independent blocks is fed; the latency of one isolated call is reported beside it, from
    # pinned buffers and from plain pageable ones (what the reference's Vec<u8> is: src/main.rs:95).
    e2e_steps = max(4, min(args.steps, 32))  # one pipelined batch of K blocks (the first copy-in and the last copy-out are exposed)
    h_bwt2 = torch.empty(n, dtype=torch.uint8).pin_memory()
    outs = [h_bwt.data_ptr() if i % 2 == 0 else h_bwt2.data_ptr() for i in range(e2e_steps)]
    con.bwt_into(h_text.data_ptr(), n, h_bwt.data_ptr())   # warm
    barrier()
    t0 = time.perf_counter()
    origin_h = con.bwt_into(h_text.data_ptr(), n, h_bwt.data_ptr())
    single_call_s = time.perf_counter() - t0
    assert origin_h == origin
    assert torch.equal(h_bwt[: 1 << 20], d_bwt[: 1 << 20].cpu())
    pageable_s = None
    if rank == 0:
        p_text = np.array(h_text.numpy(), copy=True)           # malloc'ed (pageable) copies of the caller's buffers
        p_bwt = np.empty(n, dtype=np.uint8)
        con.bwt_into(p_text.ctypes.data, n, p_bwt.ctypes.data)  # warm: the staging lanes are pinned on first use
        t0 = time.perf_counter()
        origin_p = con.bwt_into(p_text.ctypes.data, n, p_bwt.ctypes.data)
        pageable_s = time.perf_counter() - t0
        assert origin_p == origin and np.array_equal(p_bwt[-(1 << 20):], h_bwt.numpy()[-(1 << 20):])
        del p_text, p_bwt
    barrier()
    t0 = time.perf_counter()
    origins = con.bwt_batch_into([h_text.data_ptr()] * e2e_steps, [n] * e2e_steps, outs)
    e2e_s = time.perf_counter() - t0
    assert all(o == origin for o in origins)
    assert torch.equal(h_bwt2[-(1 << 20):], d_bwt[-(1 << 20):].cpu())

    # ---- the copy ceiling of this box: the same H2D + D2H traffic on two streams, no transform
    cs_in, cs_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    d_tmp = torch.empty(n, dtype=torch.uint8, device=dev)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        with torch.cuda.stream(cs_in):
            d_tmp.copy_(h_text, non_blocking=True)
        with torch.cuda.stream(cs_out):
            (h_bwt if i % 2 == 0 else h_bwt2).copy_(d_bwt, non_blocking=True)
    cs_in.synchronize()
    cs_out.synchronize()
    copy_s = time.perf_counter() - t0
    del d_tmp

    # ---- C5 (the multi-block configuration): blocks mixed(1000+b), b = rank, rank+N, ..., through the pipelined batch entry
    c5 = None
    if args.workload == "c2" and (world > 1 or args.c5_blocks > 0):
        per_rank = args.c5_blocks if args.c5_blocks > 0 else 4
        ids = blocks.corpus_blocks(rank, world, per_rank)
        texts = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in ids]
        bwts = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in ids]
        for b, t in zip(ids, texts):
            synth.generate("mixed", 1000 + b, n, out=t.numpy())
        con.bwt_batch_into([texts[0].data_ptr()], [n], [bwts[0].data_ptr()])  # warm
        barrier()
        t0 = time.perf_counter()
        origins5, st5 = con.bwt_batch_into([t.data_ptr() for t in texts], [n] * per_rank, [o.data_ptr() for o in bwts], want_stats=True)
        c5_s = time.perf_counter() - t0
        dev_ms5 = sum(x["device_ms"] for x in st5)
        rec = [[b, o, crc32_of(o_t)] for b, o, o_t in zip(ids, origins5, bwts)]
        c5 = {"local": rec, "wall_ms": c5_s * 1e3, "device_ms": dev_ms5, "bytes": n * per_rank}
        del texts, bwts

    # max over ranks of the time, sum over ranks of the work (dark_b200.blocks.aggregate; gloo-tested)
    ms_total, total_bytes = blocks.aggregate(ms_total, n * args.steps)
    e2e_ms, e2e_bytes = blocks.aggregate(e2e_s * 1e3, n * e2e_steps)
    copy_ms, copy_bytes = blocks.aggregate(copy_s * 1e3, n * e2e_steps)
    single_ms, _ = blocks.aggregate(single_call_s * 1e3, 0)
    _, launches = blocks.aggregate(0.0, launches)
    c5_line = None
    if c5 is not None:
        c5_wall, c5_bytes = blocks.aggregate(c5["wall_ms"], c5["bytes"])
        c5_dev, _ = blocks.aggregate(c5["device_ms"], 0)
        flat = blocks.gather_records(c5["local"])
        if rank == 0:
            digest = blocks.corpus_digest(flat)
            checked = {}
            for b, o, crc in flat:
                g = gold.get("mixed:%d:%d" % (1000 + b, n))
                if g:
                    checked[str(b)] = "ok" if (g["bwt_crc32"] == crc and g["origin"] == o) else "MISMATCH"
            c5_line = {"workload": "C5: blocks of %d bytes, mixed(seed=1000+b), b = rank + i*N, %d per rank, dark_bwt_forward_batch on pinned buffers" % (n, len(c5["local"])),
                       "blocks": len(flat), "bytes": c5_bytes, "device_value": c5_bytes / 1e6 / (c5_dev / 1e3), "e2e_value": c5_bytes / 1e6 / (c5_wall / 1e3),
                       "unit": UNIT, "max_rank_device_ms": c5_dev, "max_rank_wall_ms": c5_wall, "digest_crc32_of_block_crcs": digest,
                       "per_block": flat, "fixture_check": checked}

    if rank == 0:
        ms_per_step = ms_total / args.steps
        value = total_bytes / 1e6 / (ms_total / 1e3)
        e2e_value = e2e_bytes / 1e6 / (e2e_ms / 1e3)
        peak, peak_src = measured_peak_gbs()
        # roofline of the dominant kernel = the plain radix pass (12 B read + 12 B written per pair); the key-generating
        # first pass (1 B read + 12 B written per suffix) is accounted on its own
        plain_ms = agg["pass_ms"] - agg["gen_pass_ms"]
        plain_el = agg["sorted"] - agg["gen_sorted"]
        pass_gbs = 24.0 * plain_el / (plain_ms / 1e3) / 1e9 if plain_ms > 0 else 0.0
        gen_gbs = 13.0 * agg["gen_sorted"] / (agg["gen_pass_ms"] / 1e3) / 1e9 if agg["gen_pass_ms"] > 0 else None
        path_gbs = balg_per_byte * n / (ms_per_step / 1e3) / 1e9
        traffic = measured_pass_traffic()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": desc, "block_bytes": n, "blocks_per_step": world, "sharding": "independent blocks, no collective",
                       "l2": "inputs larger than L2 (text %d MiB, working set ~%.1f GiB): no flush between steps" % (n >> 20, 45.0 * n / 2**30),
                       "origin": origin, "bwt_crc32": main_crc,
                       "parity": ("ok" if (fx and fx["bwt_crc32"] == main_crc and fx["origin"] == origin) else ("MISMATCH" if fx else "no fixture")),
                       "sigma": stats["sigma"], "symbols_per_key": stats["symbols_per_key"],
                       "rounds": stats["rounds"], "active_per_round": stats["active"], "passes_per_round": stats["passes"],
                       "kernel_launches_per_step": stats["kernel_launches"], "host_syncs_per_step": agg["host_syncs"] / args.steps,
                       "note": ".dark byte identity and the reference's C1 CLI round trip cannot be tested in this image (no rustc/cargo, "
                               "no golden .dark): parity is SA/BWT/origin against the oracle pinned by the reference's known answers"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n, "d2h_bytes_per_step": n + 8,
                    "steps": e2e_steps, "timer": "host wall clock around dark_bwt_forward_batch (pipelined copies) on pinned host buffers",
                    "single_call_ms": single_ms, "single_call_value": n / 1e6 / (single_ms / 1e3),
                    "pageable_single_call_ms": pageable_s * 1e3 if pageable_s else None,
                    "pageable_single_call_value": n / 1e6 / pageable_s if pageable_s else None,
                    "pageable_vs_pinned": (pageable_s * 1e3 / single_ms) if pageable_s else None},
            "copy_only": {"value": copy_bytes / 1e6 / (copy_ms / 1e3), "unit": UNIT, "blocks": e2e_steps,
                          "what": "the e2e batch's copies alone (H2D of every block on one stream, D2H on another, pinned buffers, no transform): "
                                  "the ceiling the host side of this box puts on e2e"},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_onesweep_tma (radix pass: 12 B read + 12 B written per pair; TMA-staged, scanner CTAs)",
                         "achieved": pass_gbs, "peak": peak, "unit": "GB/s", "frac": pass_gbs / peak, "peak_source": peak_src,
                         "launches_per_step": (agg["passes"] - agg["gen_passes"]) / args.steps,
                         "full_launch_ms": (plain_ms / plain_el * n) if plain_el else None,
                         "full_launch_note": "element-weighted: time of one launch over all %d pairs of the block" % n,
                         "gen_pass": {"what": "key-generating first pass: 1 B of text read + 12 B written per suffix",
                                      "achieved": gen_gbs, "frac": (gen_gbs / peak) if gen_gbs else None,
                                      "launch_ms": agg["gen_pass_ms"] / max(1, agg["gen_passes"]), "launches_per_step": agg["gen_passes"] / args.steps},
                         "all_passes_achieved": (24.0 * plain_el + 13.0 * agg["gen_sorted"]) / (agg["pass_ms"] / 1e3) / 1e9 if agg["pass_ms"] > 0 else None,
                         "traffic": (traffic or {}).get("bytes_per_launch"),
                         "traffic_detail": traffic,
                         "path_b_alg_per_byte": balg_per_byte, "path_b_alg_per_byte_measured_on_gpu": balg_live,
                         "path_note": "B_alg is SURVEY 8(d)'s data-defined byte count of the canonical algorithm; the path moves fewer bytes "
                                      "(alphabet packing, pass pruning), so path_frac is a work-rate figure, not a bandwidth",
                         "path_achieved": path_gbs, "path_frac": path_gbs / peak, "path_frac_of_8TBs": path_gbs / 8000.0},
            "phases_ms_per_step": {k: agg[k] / args.steps for k in ("device_ms", "init_ms", "sort_ms", "pass_ms", "gen_pass_ms", "keybuild_ms",
                                                                    "rerank_ms", "emit_ms")},
        }
        if c5_line:
            line["c5"] = c5_line
        if world == 1 and args.workload == "c2" and not args.no_side_workloads:
            line["workloads"] = {w: run_side_workload(con, torch, dev, w, 3, gold) for w in ("c3", "c5")}
        if world == 1 and not args.no_cpu_baseline:
            sample_n = min(n, 1 << 25)
            rate, step_s = cpu_oracle_rate(kind, base_seed, sample_n, 1, 1, 0)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": 1, "kind": "port",
                                    "sample": f"one {sample_n}-byte {kind}(seed={base_seed}) block, 1 thread, {step_s:.1f} s "
                                              f"(oracle = C restatement of saca.rs + emission)",
                                    "full_size_one_off": full_size_cpu_figures()}
        print(json.dumps(line), flush=True)
    con.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from as it found it
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-workloads", action="store_true", help="skip the c3/c5 sub-records of the 1-GPU run")
    ap.add_argument("--c5-blocks", type=int, default=0, help="C5 blocks per rank for the `c5` sub-record (default: 4 when N > 1, none at N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's BWT (a seeded sample of large blocks) "
                                                          "and origin as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native path (--impl native)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("bench.py: --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    run_native(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
