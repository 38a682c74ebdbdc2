"""Host-side logic on CPU: generators, the emission rule statement, block sharding, and the
multi-rank aggregation of the bench (gloo, world_size 2)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_native_generators_match_oracle_generators(oracle):
    from dark_b200 import synth
    for kind, seed, n in (("dna", 1, 1 << 18), ("rep17", 2, 1 << 18), ("text", 3, 768771), ("mixed", 4, 1 << 21),
                          ("mixed", 1000, (1 << 18) + 77), ("dna", 9, 3), ("text", 8, 2)):
        assert np.array_equal(synth.generate(kind, seed, n), oracle.gen(kind, seed, n)), (kind, seed, n)
    with pytest.raises(Exception):
        synth.generate("nope", 1, 10)
    assert synth.CONFIGS["c2"] == ("dna", 1, 1 << 28)


def test_transform_statement_matches_known_answers_and_oracle(oracle):
    from dark_b200 import saca
    # saca.rs:411-412
    out, origin = saca.transform(b"abracadabra", [10, 7, 0, 3, 5, 8, 1, 4, 6, 9, 2])
    assert (out.tobytes(), origin) == (b"rdarcaaaabb", 2)
    out, origin = saca.transform(b"banana", [5, 3, 1, 0, 4, 2])
    assert (out.tobytes(), origin) == (b"nnbaaa", 3)
    t = oracle.gen("mixed", 4, 50000)
    sa = oracle.saca(t)
    out, origin = saca.transform(t, sa)
    out_o, origin_o = oracle.bwt_emit(t, sa)
    assert origin == origin_o and np.array_equal(out, out_o)
    assert saca.SUF_INVALID == 0xFFFFFFFF and saca.Suffix == np.uint32 and saca.Symbol == np.uint8


def test_block_sharding_partitions_the_corpus():
    from dark_b200 import blocks
    for nb in (0, 1, 7, 128):
        for g in (1, 2, 4, 8):
            shards = blocks.all_shards(nb, g)
            flat = sorted(b for s in shards for b in s)
            assert flat == list(range(nb))
            assert max(len(s) for s in shards) - min(len(s) for s in shards) <= 1
    assert blocks.shard(128, 3, 8) == list(range(3, 128, 8))
    with pytest.raises(ValueError):
        blocks.shard(10, 2, 2)


def _gloo_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from dark_b200 import blocks
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mine = blocks.shard(9, rank, world)
    # every rank "processes" its blocks; time = max over ranks, units = sum over ranks
    ms_local = 10.0 * len(mine) + rank
    total_ms, total_blocks = blocks.aggregate(ms_local, len(mine))
    # block results keyed by block index are identical regardless of the sharding (T6)
    digest = torch.zeros(9, dtype=torch.int64)
    for b in mine:
        digest[b] = (b * 2654435761) % 1000003
    dist.all_reduce(digest)
    # the multi-block bench record: every rank's (block, origin, crc) rows merged in block order, one digest for the set
    ids = blocks.corpus_blocks(rank, world, 3)
    recs = blocks.gather_records([(b, 1000 + b, "%08x" % (b * 40503 + 7)) for b in ids])
    q.put((rank, total_ms, total_blocks, digest.tolist(), recs, blocks.corpus_digest(recs)))
    dist.destroy_process_group()


def test_two_rank_aggregation_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    expect = [(b * 2654435761) % 1000003 for b in range(9)]
    from dark_b200 import blocks
    one_rank = [[b, 1000 + b, "%08x" % (b * 40503 + 7)] for b in range(6)]
    for rank, total_ms, total_blocks, digest, recs, cdig in res:
        assert total_blocks == 9
        assert total_ms == max(10.0 * 5 + 0, 10.0 * 4 + 1)
        assert digest == expect
        assert recs == one_rank                                  # 2 ranks x 3 blocks = blocks 0..5, each exactly once
        assert cdig == blocks.corpus_digest(one_rank)            # the digest does not depend on the sharding
    assert blocks.corpus_blocks(1, 4, 2) == [1, 5] and blocks.gather_records([(3, 1, "aa"), (1, 2, "bb")]) == [[1, 2, "bb"], [3, 1, "aa"]]


def test_bench_reference_arm_prints_contract_line():
    import json
    import subprocess
    env = dict(os.environ)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--workload", "c1"], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "MB/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0


def test_bench_rejects_bad_arguments():
    import subprocess
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=60)
        assert out.returncode == 2 and "error" in out.stderr, (extra, out.stderr[-2000:])


def test_bench_dump_outputs_whole_or_fixed_sample(tmp_path):
    """bench.py --dump-outputs: a small block is written whole; a larger one at DUMP_SAMPLE distinct positions that are
    the same on every run; float32/float64 files only, 64 MB at most."""
    import torch
    import bench
    small = torch.from_numpy(np.random.default_rng(1).integers(0, 256, 1000).astype(np.uint8))
    bench.dump_outputs(str(tmp_path / "small"), torch, small, 7)
    assert np.load(tmp_path / "small" / "origin.npy").tolist() == [7.0]
    assert np.array_equal(np.load(tmp_path / "small" / "bwt.npy"), small.numpy().astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "small" / "bwt_index.npy"), np.arange(1000, dtype=np.float64))
    n = bench.DUMP_SAMPLE + 4099
    big = torch.from_numpy(np.random.default_rng(2).integers(0, 256, n).astype(np.uint8))
    runs = []
    for d in ("run1", "run2"):
        bench.dump_outputs(str(tmp_path / d), torch, big, 123456)
        files = {f: np.load(tmp_path / d / f) for f in ("origin.npy", "bwt.npy", "bwt_index.npy")}
        assert all(a.dtype in (np.float32, np.float64) for a in files.values())
        assert sum(os.path.getsize(tmp_path / d / f) for f in files) <= 64 * 10**6
        runs.append(files)
    idx = runs[0]["bwt_index.npy"]
    assert idx.size == bench.DUMP_SAMPLE and np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < n
    assert np.array_equal(runs[0]["bwt.npy"], big.numpy()[idx.astype(np.int64)].astype(np.float32))
    for f in runs[0]:
        assert np.array_equal(runs[0][f], runs[1][f])


@pytest.mark.gpu
def test_bench_dumps_what_the_timed_steps_computed(oracle, tmp_path):
    """bench.py runs exactly --steps timed steps and --dump-outputs writes the BWT and origin of the last one: on the
    C1 block (written whole) they equal the oracle's."""
    import json
    import subprocess
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", "3", "--warmup", "1",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["gpu_launches"] == 3 * line["config"]["kernel_launches_per_step"]
    bwt_o, origin_o = oracle.bwt_forward(oracle.gen("text", 3, 768771))
    assert np.load(tmp_path / "origin.npy").tolist() == [origin_o]
    assert np.array_equal(np.load(tmp_path / "bwt.npy"), bwt_o.astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "bwt_index.npy"), np.arange(bwt_o.size, dtype=np.float64))
