"""CPU, world_size 2 over gloo: the N>1 plumbing of bench.py -- frame sharding without
overlap, max-over-ranks timing, rank-0-only reference arm."""
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    from ffb6d_b200.dist import frame_shard, split_frames, max_over_ranks, sum_over_ranks
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mine = list(frame_shard(4, rank, world))
    strong = list(split_frames(7, rank, world))
    t = max_over_ranks([10.0 + rank, 5.0 - rank])
    n = sum_over_ranks(100 + rank)
    gathered = [None] * world
    dist.all_gather_object(gathered, (mine, strong))
    dist.barrier()
    dist.destroy_process_group()
    q.put((rank, mine, strong, t, n, gathered))


def test_two_rank_sharding_and_timing_reduce():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (r0, mine0, strong0, t0, n0, g0), (r1, mine1, strong1, t1, n1, g1) = res
    assert mine0 == [0, 1, 2, 3] and mine1 == [4, 5, 6, 7]              # weak scaling: disjoint frames
    assert sorted(strong0 + strong1) == list(range(7)) and abs(len(strong0) - len(strong1)) <= 1
    assert t0 == t1 == [11.0, 5.0]                                      # max over ranks, both see it
    assert n0 == n1 == 201
    assert g0 == g1


def test_reference_arm_prints_on_rank0_only():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0"], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 2 and "--steps" in out.stderr


def test_reference_arm_line_shape():
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--ref-frames", "2", "--n-points", "3072"], env=env,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "points/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["gpu_launches"] == 0
