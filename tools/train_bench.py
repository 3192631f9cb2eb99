#!/usr/bin/env python
"""BASELINE configs 3 and 4: forward + backward (and a full Adam step) of FFB6D's point branch + bidirectional
fusion + heads (ffb6d_b200.model.FFB6DFusionNet: everything of FFB6D.forward except the ResNet/PSPNet image
backbone, whose stage outputs are synthetic leaf tensors) under DistributedDataParallel, one process per GPU,
NCCL gradient all-reduce -- the reference's recipe (train_ycb.py:536-539, 596-599).  BatchNorm statistics are per
GPU by default; --sync-bn converts every BatchNorm with torch.nn.SyncBatchNorm.convert_sync_batchnorm before the DDP
wrap, as the reference converts to SyncBN (train_ycb.py:568): with more than one GPU every BatchNorm layer then
all-reduces its statistics in the forward and in the backward.

    python tools/train_bench.py --config 3                      (1 GPU)
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/train_bench.py --config 3
    ... tools/train_bench.py --config 3 --sync-bn               (global-batch BatchNorm statistics)

Config 3: LineMOD-shaped (2 classes, 8 keypoints + centre), batch 8 per GPU, forward + backward.
Config 4: YCB-shaped (22 classes), batch 4 per GPU, forward + backward + Adam step ("end-to-end train step").
Every step also rebuilds the 22 KNN index tensors on the device from the step's cloud (the reference does this on
the CPU in DataLoader workers).  One JSON line on stdout (rank 0): points/s = GPUs * B * 12288 / t_step, time =
max over ranks of CUDA-event time.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=3, choices=[3, 4])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--sync-bn", action="store_true", help="convert every BatchNorm to torch.nn.SyncBatchNorm")
    ap.add_argument("--profile", action="store_true", help="print the per-kernel GPU time of one step (CUPTI) to stderr")
    args = ap.parse_args()
    import numpy as np
    import torch
    import torch.distributed as dist
    from ffb6d_b200.model import FFB6DFusionNet
    from ffb6d_b200.schedule import build_ffb6d_indices
    from ffb6d_b200.synthetic import make_batch
    from ffb6d_b200.dist import frame_shard, max_over_ranks

    rank, local_rank, world = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("LOCAL_RANK", 0), ("WORLD_SIZE", 1)))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch or (8 if args.config == 3 else 4)
    n_classes, n_kps = (2, 8) if args.config == 3 else (22, 8)
    N0 = 12288
    torch.manual_seed(0)
    model = FFB6DFusionNet(n_classes=n_classes, n_pts=N0, n_kps=n_kps).to(dev).train()
    if args.sync_bn:
        model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(model)
    n_params = sum(p.numel() for p in model.parameters())
    net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank], output_device=local_rank,
                                                    find_unused_parameters=False) if world > 1 else model
    opt = torch.optim.Adam(model.parameters(), lr=1e-4) if args.config == 4 else None

    batch = make_batch(frame_shard(B, rank, world), n_points=N0)
    cld = torch.from_numpy(batch["cld"]).to(dev)
    xyz = torch.from_numpy(batch["dpt_xyz"]).to(dev)
    choose = torch.from_numpy(batch["choose"]).to(dev)
    cld_rgb_nrm = torch.from_numpy(batch["cld_rgb_nrm"]).to(dev)
    g = torch.Generator(device=dev).manual_seed(rank)
    rgb_feats = [torch.randn(s, generator=g, device=dev).requires_grad_(True) for s in FFB6DFusionNet.rgb_feature_shapes(B)]
    # synthetic targets (fixed seed): segmentation labels, keypoint / centre offsets
    labels = torch.randint(0, n_classes, (B, N0), generator=g, device=dev)
    kp_t = torch.randn((B, n_kps, N0, 3), generator=g, device=dev)
    ctr_t = torch.randn((B, 1, N0, 3), generator=g, device=dev)

    def step():
        with torch.no_grad():
            inputs = build_ffb6d_indices(cld, xyz)
        inputs["choose"] = choose
        inputs["cld_rgb_nrm"] = cld_rgb_nrm
        for t in rgb_feats:
            t.grad = None
        if opt is not None:
            opt.zero_grad(set_to_none=True)
        else:
            for p in model.parameters():
                p.grad = None
        out = net(inputs, rgb_feats)
        loss = (torch.nn.functional.cross_entropy(out["pred_rgbd_segs"], labels) * 2.0
                + (out["pred_kp_ofs"] - kp_t).abs().mean() + (out["pred_ctr_ofs"] - ctr_t).abs().mean()
                # the fused image maps feed the (absent) CNN stages: a stand-in term keeps their layers in the graph
                + sum(r.mean() for r in out["fused_rgb"]) * 1e-3)
        loss.backward()
        if opt is not None:
            opt.step()
        return loss

    for _ in range(args.warmup):
        loss = step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    if world > 1:
        dist.barrier()
    ms = max(e0.elapsed_time(e1), wall)
    (ms,) = max_over_ranks([ms], device=dev)
    if args.profile and rank == 0:
        import collections
        import re
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.synchronize()
        agg = collections.OrderedDict()
        for ev in prof.events():
            if ev.device_type is not None and "cuda" in str(ev.device_type).lower():
                name = re.sub(r"\(.*", "", ev.name).replace("void ", "").replace("ffb6d::", "")
                d = agg.setdefault(name, [0, 0.0])
                d[0] += 1
                d[1] += ev.device_time
        tot = sum(v[1] for v in agg.values())
        sys.stderr.write("one step: %.2f ms of kernel time, %d launches (wall %.2f ms/step)\n"
                         % (tot / 1e3, sum(v[0] for v in agg.values()), ms / args.steps))
        for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1])[:25]:
            sys.stderr.write("%-70s n=%4d %9.1f us %5.1f%%\n" % (k[:70], v[0], v[1], 100 * v[1] / tot))
    finite = bool(torch.isfinite(loss).item()) and all(torch.isfinite(p.grad).all().item() for p in model.parameters()
                                                       if p.grad is not None)
    if rank == 0:
        line = {"metric": "FFB6D point branch + fusion + heads, training step, points/s", "config": args.config,
                "what": ("forward + backward" if args.config == 3 else "forward + backward + Adam step")
                + ", DDP gradient all-reduce over NCCL" * (world > 1)
                + ", SyncBatchNorm statistics all-reduce over NCCL" * (world > 1 and args.sync_bn),
                "value": world * B * N0 * args.steps / (ms / 1e3), "unit": "points/s", "n_gpus": world,
                "batch_per_gpu": B, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                "params": n_params, "grad_allreduce_bytes": 4 * n_params if world > 1 else 0, "loss": float(loss.detach()),
                "finite": finite, "sync_bn": args.sync_bn, "dtype": "f32", "data": "synthetic", "scaling": "weak"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
