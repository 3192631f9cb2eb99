#!/usr/bin/env python
"""bench.py -- fused KNN + gather throughput of the FFB6D fusion hot path on B200.

    python bench.py --gpus N --steps K --warmup W          (N>1: launched by torchrun)
    python bench.py --impl reference ...                    (the reference's CPU ops, host cores)

A *step* is one pass of the hot path over one batch of synthetic frames: the 22 KNN index
builds of the dataset schedule + the 23 gathers of FFB6D.forward (BASELINE.md §3), B frames
per GPU (default 32 = BASELINE.json configs[1]).  metric = points/sec = GPUs * B * N0 / t_pass.

One JSON line on stdout (rank 0).  `value`: inputs resident in HBM.  `e2e`: the step's depth maps
and `choose` indices come from pinned host memory (H2D inside the timed region), are back-projected
on the device, and a result digest is read back (D2H inside).  Other flags: --batch, --n-points, --k
(stress sweep), --layout, --streams / --gather-streams (graph branches), --no-graph, --per-op, --dump-outputs DIR
(what the last timed step returned, as .npy files, to compare two builds output for output).  `roofline`: the dominant kernel, per-op CUDA events on the launching stream
inside the timed region, against MEASURED_PEAKS.json.  `cpu_baseline`: the reference's compiled
KNN (oracle/_ref, nanoflann, OpenMP over the batch) + its torch gather expression on the host
cores, bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "fused KNN+gather points/sec at 12288 pts"
UNIT = "points/s"
FALLBACK_HBM_GBS = 6650.0      # /opt/skills/guides/B200_PROFILING.md fallback


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi sampled every 200 ms while the GPU is under load (recipe's clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()            # the exact process we started
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw = [], [], []
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------ CPU reference arm
def _torch_cpu_random_sample(feature, pool_idx):
    """The reference's torch expression (models/ffb6d.py:166-177) restated, on CPU threads."""
    import torch
    if feature.dim() > 3:
        feature = feature.squeeze(3)
    K, d, B = pool_idx.shape[-1], feature.shape[1], pool_idx.shape[0]
    flat = pool_idx.reshape(B, -1)
    g = torch.gather(feature, 2, flat.unsqueeze(1).repeat(1, d, 1)).contiguous()
    return g.reshape(B, d, -1, K).max(dim=3, keepdim=True)[0]


_REF_CACHE = {}


def _reference_inputs(n_points, frames_knn, frames_gather, k):
    """Synthetic inputs of the CPU arm, generated once per process (not part of any timed region)."""
    import numpy as np
    import torch
    from ffb6d_b200.synthetic import make_batch, image_pyramid_np     # plain numpy: does not load the CUDA library
    from ffb6d_b200.tables import gather_schedule
    key = (n_points, frames_knn, frames_gather, k)
    if key not in _REF_CACHE:
        _REF_CACHE.clear()
        batch = make_batch(range(1000, 1000 + frames_knn), n_points=n_points)
        sets = {("cld", i): np.ascontiguousarray(batch["cld"][:, : n_points // 4 ** i]) for i in range(5)}
        pyr = [image_pyramid_np(x) for x in batch["dpt_xyz"]]
        for sr in (2, 4, 8):
            sets[("img", sr)] = np.stack([p[sr] for p in pyr])
        g = torch.Generator().manual_seed(0)
        feats = [torch.randn(frames_gather, C, S, 1, generator=g) for _, _, C, S, _, _ in gather_schedule(n_points)]
        _REF_CACHE[key] = (batch, sets, feats)
    return _REF_CACHE[key]


def cpu_reference_sample(n_points, frames_knn, frames_gather, reps=1, k=16, gather_threads=None, mode="stacked"):
    """Time the reference's CPU implementation of one pass on a bounded sample.

    KNN, `mode`:
      "stacked"   (BASELINE.md C2/C4) the 22-call schedule on `frames_knn` stacked frames through the
                  reference's compiled cpp_knn_batch_omp: OpenMP over the batch is every thread the
                  reference can use (NN/knn_.cxx:108-109);
      "as_called" (C1) what FFB6D's dataset does: 22 x knn_batch(x[None], y[None], k, omp=True) per frame,
                  frames one after the other (ycb_dataset.py:275-308);
      "single"    (C3) the same calls through the non-OpenMP twin cpp_knn_batch: one thread.
    Falls back to the oracle port if oracle/_ref is absent.
    Gathers: the 23 gathers of `frames_gather` frames with the reference's torch expression on host threads.
    Returns dict(sec_per_frame, kind, cores, sample, ...)."""
    import numpy as np
    import torch
    from ffb6d_b200.tables import knn_schedule, gather_schedule
    from oracle import ref_loader as R
    from oracle import cpu_oracle as O

    cores = os.cpu_count() or 1
    kind = "reference" if R.knn_available() else "port"
    fg = min(frames_gather, frames_knn)
    batch, sets, feats = _reference_inputs(n_points, frames_knn, fg, k)
    if kind == "reference":
        def knn(s, q, kk):
            if mode == "stacked":
                return R.knn_batch(s, q, kk, omp=True)
            return np.concatenate([R.knn_batch(s[b:b + 1], q[b:b + 1], kk, omp=(mode == "as_called"))
                                   for b in range(s.shape[0])])
    else:
        knn = O.knn_batch
    t_knn = 1e30
    idx = {}
    for _ in range(max(1, reps)):
        t0 = time.perf_counter()
        for key, s, q, kk in knn_schedule(n_points, k=k):
            idx[key] = knn(sets[s], sets[q], kk).astype(np.int32)       # helper_tool.py:170
        t_knn = min(t_knn, time.perf_counter() - t0)
    # gathers: the reference's torch expression; intra-op threading of torch on a many-core host is far
    # from monotonic, so the thread count that runs it fastest is used (found once, then reused)
    idx["choose"] = batch["choose"]
    for i in range(4):
        idx["cld_sub_idx%d" % i] = idx["cld_nei_idx%d" % i][:, : n_points // 4 ** (i + 1)]
    ops_ = []
    for (op, key, C, S, Q, K), feat in zip(gather_schedule(n_points), feats):
        ii = torch.from_numpy(np.ascontiguousarray(idx[key][:fg])).long()      # train_ycb.py:224-232
        if op == "choose":
            ii = ii.reshape(fg, -1, 1)
        ops_.append((feat, ii))
    candidates = [gather_threads] if gather_threads else sorted(
        {cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True)
    if mode == "single":
        candidates = [1]
    t_g, g_threads = 1e30, candidates[0]
    for nt in candidates:
        torch.set_num_threads(nt)
        for _ in range(max(1, reps)):
            t0 = time.perf_counter()
            for feat, ii in ops_:
                _torch_cpu_random_sample(feat, ii)
            dt = time.perf_counter() - t0
            if dt < t_g:
                t_g, g_threads = dt, nt
    sec_per_frame = t_knn / frames_knn + t_g / fg
    how = {"stacked": "stacked, OpenMP over the batch, %d threads" % cores,
           "as_called": "as FFB6D calls it: B=1 per call, omp=True, frames in sequence",
           "single": "B=1 per call, cpp_knn_batch (no OpenMP): one thread"}[mode]
    sample = ("%d frames x 22 KNN calls via %s (%s), %.2f s; %d frames x 23 gathers via the reference's torch "
              "expression on CPU (%d threads), %.2f s"
              % (frames_knn, "oracle/_ref/libknn_ref.so (unmodified NN/knn_.cxx)" if kind == "reference"
                 else "oracle port (brute force)", how, t_knn, fg, g_threads, t_g))
    return {"sec_per_frame": sec_per_frame, "kind": kind, "cores": cores if mode != "single" else 1, "sample": sample,
            "t_knn": t_knn, "t_gather": t_g, "gather_threads": g_threads,
            "knn_sec_per_frame": t_knn / frames_knn, "gather_sec_per_frame": t_g / fg}


def run_reference_arm(args, rank, emit):
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    fk = args.ref_frames or max(8, cores)          # one frame per core: every thread the reference has is busy
    first = cpu_reference_sample(args.n_points, fk, 2, k=args.k)       # picks the gather thread count (untimed)
    gt = first["gather_threads"]
    for _ in range(max(0, args.warmup - 1)):
        cpu_reference_sample(args.n_points, fk, 2, k=args.k, gather_threads=gt)
    t0 = time.perf_counter()
    per_frame = []
    last = None
    for _ in range(args.steps):
        last = cpu_reference_sample(args.n_points, fk, 2, k=args.k, gather_threads=gt)
        per_frame.append(last["sec_per_frame"])
    wall = time.perf_counter() - t0
    spf = sum(per_frame) / len(per_frame)
    value = args.n_points / spf
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": spf * fk * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "FFB6D fusion pass: 22 KNN index builds + 23 gathers per frame, "
                               "480x640 synthetic RGB-D, %d points, K=%d" % (args.n_points, args.k),
                   "frames_per_step": fk, "note": "CPU arm: each step is a bounded sample of the workload"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": last["cores"], "kind": last["kind"],
                         "sample": last["sample"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------ GPU arm
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def load_ncu_traffic():
    """{kernel family: dram bytes per launch} from the committed ncu summary, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            return json.load(fh)
    except Exception:
        return {}


K1_FAMILY = "K=1 searches (grid_search_k1_tile_kernel for image queries, grid_search_kernel<1>, knn_brute for S<512)"
SELF_FAMILY = "grid_search_group_kernel<SELF> (K=16 self searches)"
NONSELF_FAMILY = "grid_search_group_kernel<non-self> (K=16 cloud -> image searches)"
BUILD_FAMILY = "grid_build_kernel (one cluster launch per grid)"


def kernel_family(op_name):
    """Map a timed op to the kernel (family) that runs it.  Gathers are single kernels and are
    grouped by kernel function; a KNN search op is its search kernel + overflow pass (the search
    kernel is > 90 % of it), a KNN build op is one grid_build_kernel launch."""
    parts = op_name.split(":")
    kind, key = parts[0], parts[1]
    if kind == "gather":
        return parts[2]
    if kind == "knn_build":
        return BUILD_FAMILY
    if "interp" in key or key.startswith("p2r"):
        return K1_FAMILY
    return SELF_FAMILY if key.startswith("cld_nei") else NONSELF_FAMILY


DUMP_BYTES = 60 << 20      # all dumped arrays together, .npy headers aside: under 64 MB


def sample_outputs(inputs, outs, gathers):
    """{name: numpy array} of what one pass returns: every tensor of `inputs` (index tensors, point sets, choose)
    and the gather outputs as ``gather_<index key>``.  Float tensors become float32, integer tensors float64
    (exact).  An array larger than its share of DUMP_BYTES is replaced by its elements (in the logical shape's
    flat order) at positions drawn without replacement by a generator seeded with 0: the same positions for the
    same shape, so that two runs with the same arguments can be compared element for element."""
    import numpy as np
    import torch
    arrays = dict(inputs)
    arrays.update({"gather_%s" % g[1]: t for g, t in zip(gathers, outs)})
    share = DUMP_BYTES // len(arrays)
    res = {}
    for name, t in sorted(arrays.items()):
        dtype = np.dtype(np.float32 if t.is_floating_point() else np.float64)
        cap = share // dtype.itemsize
        if t.numel() > cap:
            pos = np.sort(np.random.default_rng(0).choice(t.numel(), cap, replace=False))
            t = t.reshape(-1)[torch.from_numpy(pos).to(t.device)]
        res[name] = t.cpu().numpy().astype(dtype)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="frames per GPU per step")
    ap.add_argument("--n-points", type=int, default=12288)
    ap.add_argument("--k", type=int, default=16, help="neighbours of the K-NN index builds (stress sweep: 8/16/32)")
    ap.add_argument("--layout", default="nchw", choices=["nchw", "channels_last"])
    ap.add_argument("--ref-frames", type=int, default=0, help="frames per CPU-arm sample (0 = #cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-mlp", action="store_true", help="skip the separately reported fusion-MLP timing")
    ap.add_argument("--streams", type=int, default=2, help="side streams (graph branches) of the index build")
    ap.add_argument("--gather-streams", type=int, default=0, help="side streams of the gathers (0: same number)")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA graph replays")
    ap.add_argument("--per-op", action="store_true", help="also print the per-op table to stderr")
    ap.add_argument("--l2-fetch", type=int, default=0, help="experiment: cudaLimitMaxL2FetchGranularity (32/64/128 bytes)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy, float32 or float64, "
                         "under 64 MB in all: a larger array is a fixed seeded sample of its elements")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    # stdout carries exactly one JSON line: libraries that print to fd 1 (NCCL's version banner)
    # are sent to stderr for the duration of the run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())

    if args.impl == "reference":
        return run_reference_arm(args, rank, emit)

    import numpy as np
    import torch
    from ffb6d_b200 import _lib   # fails loudly if the CUDA library is missing (no CPU fallback)
    from ffb6d_b200.pipeline import FusionPass, OpTimer
    from ffb6d_b200.tables import knn_schedule, set_size
    from ffb6d_b200.synthetic import make_batch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if args.l2_fetch:
        import ctypes
        torch.zeros(1, device=dev)                      # context
        rt = ctypes.CDLL("libcudart.so.12")
        rc_ = rt.cudaDeviceSetLimit(5, ctypes.c_size_t(args.l2_fetch))       # cudaLimitMaxL2FetchGranularity
        got_ = ctypes.c_size_t(0)
        rt.cudaDeviceGetLimit(ctypes.byref(got_), 5)
        sys.stderr.write("bench.py: L2 fetch granularity -> %d (rc %d)\n" % (got_.value, rc_))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()

    B, N0 = args.batch, args.n_points
    # ---- synthetic inputs: distinct frames per rank, pinned on the host + resident on the device
    from ffb6d_b200.dist import frame_shard, max_over_ranks, sum_over_ranks
    batch = make_batch(frame_shard(B, rank, world), n_points=N0)
    cld_h = torch.from_numpy(batch["cld"]).pin_memory()
    xyz_h = torch.from_numpy(batch["dpt_xyz"]).pin_memory()
    cho_h = torch.from_numpy(batch["choose"]).pin_memory()
    cld_d, xyz_d, cho_d = cld_h.to(dev), xyz_h.to(dev), cho_h.to(dev)
    p = FusionPass(B, n_points=N0, k=args.k, device=dev, layout=args.layout, seed=rank, n_streams=args.streams,
                   n_gather_streams=args.gather_streams or None)
    feat_bytes = sum(f.numel() * 4 for f in p.features)

    sampler = ClockSampler(torch.cuda.current_device() if "CUDA_VISIBLE_DEVICES" not in os.environ
                           else os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local_rank]) if rank == 0 else None

    # ---- warm-up (eager), then capture the pass into CUDA graphs: ~200 small launches with
    # static shapes per step; replaying removes the Python/launch overhead from the GPU timeline
    for _ in range(args.warmup):
        p(cld_d, xyz_d, cho_d)
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    p(cld_d, xyz_d, cho_d)
    launches_per_step = _lib.launch_count() - l0
    use_graph = not args.no_graph
    run_resident = None
    if use_graph:
        try:
            run_resident = p.capture(lambda: p(cld_d, xyz_d, cho_d))
        except Exception as e:                      # noqa: BLE001
            sys.stderr.write("bench.py: CUDA graph capture failed (%s); timing eager launches\n" % e)
            use_graph = False
    if run_resident is None:
        def run_resident():
            return p(cld_d, xyz_d, cho_d)
    for _ in range(2):
        run_resident()
    torch.cuda.synchronize()

    # ---- timed region 1: inputs resident in HBM
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.steps):
        last = run_resident()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    launches = launches_per_step * args.steps
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in sample_outputs(*last, p.gathers).items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    resident_res = run_resident()          # untimed: the results the end-to-end path must reproduce
    torch.cuda.synchronize()

    # ---- timed region 2: end to end.  The step's inputs are what the reference's host pipeline
    # holds before its KNN calls: the depth map in metres (`dpt_m`, ycb_dataset.py:194) and the
    # `choose` indices; they are copied from pinned host memory every step (double-buffered: the
    # copy of step i+1 overlaps the pass of step i), back-projected on the device, and a digest of
    # all 45 results is read back into pinned memory.
    from ffb6d_b200.ops import intrinsics_to_device
    from ffb6d_b200.synthetic import INTRINSICS
    digest_h = torch.empty((len(p.gathers) + 22) * 256, dtype=torch.float32).pin_memory()

    def digest_fn(inp, out):
        parts = [o.reshape(-1)[:256] for o in out]
        idx = torch.cat([inp[k].reshape(-1)[:256] for k in sorted(inp) if "idx" in k and "sub" not in k])
        return torch.cat(parts + [idx.float()])   # three small kernels instead of one per result

    ndig = (len(p.gathers) + 22) * 256
    dep_h = torch.from_numpy(batch["depth"]).pin_memory()
    intr_d = intrinsics_to_device(INTRINSICS["linemod"], dev)
    bufs = [(torch.empty_like(dep_h, device=dev), torch.empty_like(cho_d)) for _ in range(2)]
    for dbuf, cbuf in bufs:
        dbuf.copy_(dep_h)
        cbuf.copy_(cho_h)
    torch.cuda.synchronize()
    h2d = dep_h.numel() * 4 + cho_h.numel() * 4
    runs = []
    if use_graph:
        try:
            for i in range(2):
                cur, nxt = bufs[i], bufs[1 - i]
                runs.append(p.capture(lambda cur=cur: p.from_depth(cur[0], intr_d, cur[1]),
                                      prefetch=[(nxt[0], dep_h), (nxt[1], cho_h)], digest=(digest_fn, digest_h)))
        except Exception as e:                      # noqa: BLE001
            sys.stderr.write("bench.py: e2e graph capture failed (%s); eager\n" % e)
            runs = []
    if not runs:
        def eager(i):
            cur, nxt = bufs[i], bufs[1 - i]
            nxt[0].copy_(dep_h, non_blocking=True)
            nxt[1].copy_(cho_h, non_blocking=True)
            res = p.from_depth(cur[0], intr_d, cur[1])
            d = digest_fn(*res)
            digest_h[: d.numel()].copy_(d, non_blocking=True)
            return res
        runs = [lambda: eager(0), lambda: eager(1)]
    for i in range(2):
        runs[i]()
    torch.cuda.synchronize()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    f0.record()
    for i in range(args.steps):
        runs[i & 1]()
    f1.record()
    torch.cuda.synchronize()
    e2e_wall_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    e2e_ms = max(f0.elapsed_time(f1), e2e_wall_ms)
    # the end-to-end path (depth in, back-projection on the device, digest out) must reproduce the
    # resident pass bit for bit, and frame 0 of rank 0 the reference's own index arrays
    digest_ok = bool(torch.equal(digest_h[:ndig], digest_fn(*resident_res).cpu()))
    reference_digest_ok = None
    if rank == 0 and N0 == 12288 and args.k == 16:
        import hashlib
        try:
            with open(os.path.join(ROOT, "tests", "golden", "schedule_digest.json")) as fh:
                gold = json.load(fh)["frames"]["seed0_n12288"]["keys"]
            reference_digest_ok = all(
                hashlib.sha256(np.ascontiguousarray(resident_res[0][key][0].to(torch.int32).cpu().numpy()).tobytes()
                               ).hexdigest() == meta["sha256"] for key, meta in gold.items())
        except (OSError, KeyError):
            reference_digest_ok = None

    # ---- instrumented region: the same launches issued eagerly with a CUDA-event pair around
    # every op, on the launching stream.  A spin kernel in front of each step keeps the GPU
    # behind the CPU so the events bracket kernel time, not Python launch gaps.
    timer = OpTimer()
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    inst_ms, spin_ms, enqueue_ms = 0.0, 0.0, 0.0
    # how long does this box's CPU need to enqueue one instrumented step?  (3 ms ... 25 ms seen on
    # the pool's hosts.)  The spin has to outlast it, or the event pairs measure launch gaps.
    c0 = time.perf_counter()
    p(cld_d, xyz_d, cho_d, OpTimer())
    dry_ms = (time.perf_counter() - c0) * 1e3
    torch.cuda.synchronize()
    spin_cycles = int(min(max(40e6, (1.5 * dry_ms + 5.0) * 2.0e6), 1.2e9))   # cycles at <= 2 GHz
    for _ in range(args.steps):
        s0.record()
        torch.cuda._sleep(spin_cycles)
        s1.record()
        i0.record()
        c0 = time.perf_counter()
        p(cld_d, xyz_d, cho_d, timer)
        enqueue_ms += (time.perf_counter() - c0) * 1e3
        i1.record()
        torch.cuda.synchronize()
        inst_ms += i0.elapsed_time(i1)
        spin_ms += s0.elapsed_time(s1)
    clocks = sampler.stop() if sampler is not None else None

    # ---- max over ranks (device time, never wall clock of one rank)
    ms, e2e_ms = max_over_ranks([ms, e2e_ms], device=dev)
    launches = sum_over_ranks(int(launches), device=dev)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    steps = args.steps
    value = world * B * N0 * steps / (ms / 1e3)
    e2e_value = world * B * N0 * steps / (e2e_ms / 1e3)
    peak, peak_src = load_peaks()

    # ---- roofline of the dominant kernel (per-op events, rank 0)
    fam = {}
    per_op = timer.summary()
    for name, d in per_op.items():
        f = fam.setdefault(kernel_family(name), {"ms": 0.0, "bytes": 0, "n": 0})
        f["ms"] += d["ms"]
        f["bytes"] += d["bytes"]
        f["n"] += d["n"]
    tot_ms = sum(f["ms"] for f in fam.values())
    # `roofline` = the dominant HBM-BOUND kernel family, chosen deterministically: the gather family that
    # moves the most algorithmic bytes (a function of the configuration, not of a timing that flips
    # between runs).  The KNN searches are instruction-issue bound (DRAM < 2 % busy in ncu): they are
    # reported in `compute` with instructions per query instead of a meaningless HBM fraction.
    gfam = [k for k in fam if k.startswith("gather")]
    dom = max(gfam, key=lambda k: (fam[k]["bytes"], k))
    dd = fam[dom]
    achieved = dd["bytes"] / (dd["ms"] / 1e3) / 1e9
    ncu = load_ncu_traffic()
    cap = ncu.get(dom, {}) if isinstance(ncu.get(dom), dict) else {}
    traffic = cap.get("traffic_bytes")
    roofline = {
        "bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic, "traffic_capture": cap or None, "peak_source": peak_src,
        "selection": "gather family with the most algorithmic bytes per step (deterministic)",
        "share_of_step": dd["ms"] / tot_ms, "ops_per_step": dd["n"] // steps,
        "alg_bytes_per_launch": dd["bytes"] / dd["n"], "avg_launch_ms": dd["ms"] / dd["n"],
        "families": {k: {"share": v["ms"] / tot_ms, "ms_per_step": v["ms"] / steps,
                         "GBps": v["bytes"] / (v["ms"] / 1e3) / 1e9,
                         "frac_of_peak": v["bytes"] / (v["ms"] / 1e3) / 1e9 / peak} for k, v in sorted(fam.items())
                     if k.startswith("gather")},
    }
    n_q = {"k1": 0, "k16_self": 0, "k16": 0}
    for key_, s_, q_, kk_ in knn_schedule(N0, k=args.k):
        q_n = set_size(q_, N0)
        n_q["k1" if kk_ == 1 else ("k16_self" if s_ == q_ else "k16")] += q_n * B
    compute = {"note": "KNN index build: integer/fp32 issue bound, HBM traffic ~ algorithmic (12S + 12Q + 4QK per call); "
                       "instructions per query from the committed ncu captures (profiles/ncu_traffic.json)",
               "families": {}}
    for k, v in sorted(fam.items()):
        if k.startswith("gather"):
            continue
        entry = {"share": v["ms"] / tot_ms, "ms_per_step": v["ms"] / steps}
        if k == K1_FAMILY:
            entry["queries_per_step"] = n_q["k1"]
            entry["note"] = ("queries ANSWERED per step; 3 of the 11 searches (p2r_ds_nei_idx0/1/2) are strided pixel subsets of "
                             "p2r_up_nei_idx2/1/0 (image level 2s is every other pixel of level s): copied, not run")
        elif k == SELF_FAMILY:
            entry["queries_per_step"] = n_q["k16_self"]
        elif k == NONSELF_FAMILY:
            entry["queries_per_step"] = n_q["k16"]
            entry["note"] = "4 of the 7 searches are row slices of the other 3 (cloud levels are prefixes): not run"
        if "queries_per_step" in entry and v["ms"] > 0:
            entry["ns_per_query"] = v["ms"] / steps * 1e6 / entry["queries_per_step"]
        cap_k = ncu.get(k)
        if isinstance(cap_k, dict) and "warp_instructions_per_query" in cap_k:
            entry["warp_instructions_per_query"] = cap_k["warp_instructions_per_query"]
        compute["families"][k] = entry
    knn_ms = sum(v["ms"] for k, v in fam.items() if not k.startswith("gather")) / steps
    compute["knn_ms_per_step"] = knn_ms
    compute["gather_ms_per_step"] = sum(v["ms"] for k, v in fam.items() if k.startswith("gather")) / steps
    pass_gbs = p.alg_bytes_per_frame * B * steps / (ms / 1e3) / 1e9
    pass_roofline = {"alg_bytes_per_frame": p.alg_bytes_per_frame, "achieved": pass_gbs, "peak": peak,
                     "unit": "GB/s", "frac": pass_gbs / peak,
                     "note": "whole pass on one GPU: alg_bytes*B / t_pass / HBM peak (BASELINE.md §3)"}
    if args.per_op:
        for name, d in sorted(per_op.items(), key=lambda kv: -kv[1]["ms"]):
            sys.stderr.write("%-28s %8.3f ms/step  %8.1f GB/s\n" % (
                name, d["ms"] / steps, d["bytes"] / (d["ms"] / 1e3) / 1e9))

    # ---- reported separately (BASELINE.md §3): the 28 fusion 1x1 MLPs on the tensor cores
    mlp_line = None
    if not args.no_mlp:
        from ffb6d_b200.pipeline import FusionMLPs
        mlps = FusionMLPs(B, n_points=N0, device=dev, seed=rank)
        for _ in range(2):
            mlps()
        torch.cuda.synchronize()
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = max(2, min(steps, 5))
        m0.record()
        for _ in range(reps):
            mlps()
        m1.record()
        torch.cuda.synchronize()
        mlp_ms = m0.elapsed_time(m1) / reps
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                bf16_peak = float(json.load(fh)["bf16_tflops"])
        except Exception:
            bf16_peak = 1590.0
        tf32_tflops = 3.0 * mlps.flops / (mlp_ms / 1e3) / 1e12          # three TF32 MMAs per fp32 product
        mlp_line = {"layers": len(mlps.layers), "ms_per_step": mlp_ms, "fp32_equiv_tflops": tf32_tflops / 3.0,
                    "tf32_tflops_issued": tf32_tflops,
                    "roofline": {"bound": "tensor", "achieved": tf32_tflops, "peak": bf16_peak / 2.0,
                                 "unit": "TFLOP/s", "frac": tf32_tflops / (bf16_peak / 2.0),
                                 "note": "kind::tf32 peak taken as half the measured bf16 peak; 3xTF32 split for "
                                         "fp32 fidelity (1e-5 contract)"},
                    "note": "28 fused cat+conv1x1+BN(eval)+ReLU layers of the fusion stack (models/ffb6d.py:55-80,"
                            "104-129), frames_per_gpu x 34.1 GFLOP; not part of `value`; weights split into TF32 hi/lo "
                            "tiles once at load (ffb6d_fusion_mlp_pack), activations split in the kernel"}
        del mlps
        torch.cuda.empty_cache()

    # ---- BASELINE configs[1] as ONE chained region: index build + the seven fusion stages (gathers + the 28
    # fusion MLPs, p2r_fuse restructured as W1.rgb + (W2.p)[idx]) + final interpolation + choose gather
    stack_line = None
    if not args.no_mlp:
        try:
            from ffb6d_b200.pipeline import FusionStack
            stack = FusionStack(B, n_points=N0, k=args.k, device=dev, seed=rank)

            def full(restructured):
                return stack(p.build_indices(cld_d, xyz_d, cho_d), restructured)

            res = {}
            for name_, flag in (("restructured", True), ("reference_order", False)):
                run = p.capture(lambda flag=flag: full(flag)) if use_graph else (lambda flag=flag: full(flag))
                for _ in range(2):
                    run()
                torch.cuda.synchronize()
                t0_, t1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                reps = max(3, min(steps, 10))
                t0_.record()
                for _ in range(reps):
                    run()
                t1_.record()
                torch.cuda.synchronize()
                res[name_] = t0_.elapsed_time(t1_) / reps
                del run
            stack_ms = res["restructured"]
            stack_line = {"what": "BASELINE configs[1] chained: 22 KNN index builds + 7 fusion stages (16 gathers, 28 fusion "
                                  "MLPs + 7 small W2.p products, the 7 p2r gathers folded into the p2r_fuse epilogue) + final "
                                  "interpolation + choose gather, one CUDA graph per step",
                          "ms_per_step": stack_ms, "value": world * B * N0 / (stack_ms / 1e3), "unit": UNIT,
                          "reference_order_ms_per_step": res["reference_order"],
                          "mlp_flops_per_step_reference": stack.flops,
                          "note": "reference_order = the same kernels composed as the reference does (materialised "
                                  "interpolated maps, p2r_fuse over 2*C_r channels)"}
            del stack
            torch.cuda.empty_cache()
        except Exception as e:                      # noqa: BLE001
            stack_line = {"error": str(e)[:300]}

    # ---- RandLA local feature aggregation (SURVEY.md §8 a11-a14): the four encoder Dilated_res_blocks of the
    # point branch at FFB6D's widths, inference, on the index tensors of this pass; reported against the
    # survey's LFA gather byte model (56.6 MB/frame at N0 = 12288, K = 16: the three neighbour gathers per block)
    lfa_line = None
    if not args.no_mlp:
        try:
            from ffb6d_b200 import modules as M_
            blocks, feats_ = [], []
            d_in = 8
            gl = torch.Generator(device=dev).manual_seed(rank)
            for i_, d_ in enumerate((32, 64, 128, 256)):
                blk = M_.Dilated_res_block(d_in, d_).to(dev).eval()
                blocks.append(blk)
                feats_.append(torch.randn((B, d_in, N0 // 4 ** i_, 1), generator=gl, device=dev))
                d_in = 2 * d_
            idx_in = resident_res[0]

            def lfa():
                with torch.no_grad():
                    return [blk(f_, idx_in["cld_xyz%d" % i_], idx_in["cld_nei_idx%d" % i_])
                            for i_, (blk, f_) in enumerate(zip(blocks, feats_))]

            for _ in range(2):
                lfa()
            torch.cuda.synchronize()
            t0_, t1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 5
            t0_.record()
            for _ in range(reps):
                lfa()
            t1_.record()
            torch.cuda.synchronize()
            lfa_ms = t0_.elapsed_time(t1_) / reps
            lfa_bytes = sum(4 * (N0 // 4 ** i_) * args.k * (3 + 2 * d_ // 2) for i_, d_ in enumerate((32, 64, 128, 256)))
            lfa_line = {"what": "4 encoder Dilated_res_blocks (relative position encoding, 2 neighbour gathers, 2 attentive "
                                "poolings, 6 conv+BN layers each) on this package's kernels, inference, eager launches",
                        "ms_per_step": lfa_ms, "gather_alg_bytes_per_frame": lfa_bytes,
                        "gather_model_GBps": lfa_bytes * B / (lfa_ms / 1e3) / 1e9,
                        "note": "each attentive pooling is ONE kernel (ffb6d_lfa_att_pool_fused: neighbour gather, position "
                                "MLP, concat, fc, softmax over K, weighted sum, output conv+BN+LeakyReLU in shared memory); "
                                "the [B,C,N,K] neighbour / attention tensors never reach HBM (SURVEY.md §8 f-2)"}
            del blocks, feats_
            torch.cuda.empty_cache()
        except Exception as e:                      # noqa: BLE001
            lfa_line = {"error": str(e)[:300]}

    # ---- the step after the network (SURVEY.md §8 f-4): keypoint voting of one object, 8 keypoints + centre,
    # every one of the object's points voting; timed beside the reference's algorithm in stock torch ops
    # (utils/meanshift_pytorch.py:33-57: N x N matrices, a host sync per iteration, one call per vote set)
    pose_line = None
    if world == 1 and not args.no_mlp:
        try:
            import math as _m
            from ffb6d_b200 import ops as F
            n_obj, n_sets, bw_ = 4096, 9, 0.04
            gp = torch.Generator().manual_seed(0)
            truth = torch.rand(n_sets, 1, 3, generator=gp) * 0.3 + torch.tensor([0.0, 0.0, 0.8])
            votes = truth + torch.randn(n_sets, n_obj, 3, generator=gp) * 0.01
            votes[:, ::7] += torch.rand(n_sets, (n_obj + 6) // 7, 3, generator=gp) * 0.4 - 0.2
            votes = votes.to(dev)

            def torch_fit(A):
                n = A.shape[0]
                C, it = A.clone(), 0
                while True:
                    it += 1
                    dis = torch.norm(C.reshape(1, n, 3) - C.reshape(n, 1, 3), dim=2)
                    w = (torch.exp(-0.5 * (dis / bw_) ** 2) / (bw_ * _m.sqrt(2 * _m.pi))).reshape(n, n, 1)
                    new_C = torch.sum(w * C, dim=1) / torch.sum(w, dim=1)
                    done = torch.max(torch.norm(new_C - C, dim=1)) < bw_ * 1e-3 or it > 300
                    C = new_C
                    if done:
                        break
                dis = torch.norm(C.view(n, 1, 3) - C.view(1, n, 3), dim=2)
                mi = torch.max(torch.sum(dis < bw_, dim=1), 0)[1]
                return C[mi]

            def timed(fn, reps):
                fn()
                torch.cuda.synchronize()
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record()
                for _ in range(reps):
                    fn()
                b_.record()
                torch.cuda.synchronize()
                return a_.elapsed_time(b_) / reps

            ours_ms = timed(lambda: F.mean_shift_fit(votes, None, bw_, 300), 3)
            c_ours, _, it_ours = F.mean_shift_fit(votes, None, bw_, 300)
            torch_ms = timed(lambda: [torch_fit(votes[g_]) for g_ in range(n_sets)], 1)
            c_torch = torch.stack([torch_fit(votes[g_]) for g_ in range(n_sets)])
            rounds = int(it_ours.max().item())
            pose_line = {"what": "keypoint voting of one object: %d vote sets x %d points, Gaussian mean shift (bandwidth 0.04) "
                                 "to the reference's stop rule, one persistent kernel" % (n_sets, n_obj),
                         "ms_per_object": ours_ms, "rounds": rounds,
                         "pair_updates_per_s": float(it_ours.sum().item()) * n_obj * n_obj / (ours_ms / 1e3),
                         "torch_ops_ms_per_object": torch_ms, "speedup_vs_torch_ops": torch_ms / ours_ms,
                         "max_centre_diff_m": float((c_ours - c_torch).abs().max().item()),
                         "note": "exp-bound (one MUFU.EX2 + ~11 FP32 per pair), not HBM-bound: the modes stay in L2; the "
                                 "comparator is the reference's algorithm in stock torch ops on this GPU"}
            del votes
            torch.cuda.empty_cache()
        except Exception as e:                      # noqa: BLE001
            pose_line = {"error": str(e)[:300]}

    # ---- comparators on the same box (BASELINE.md §4).  C5: the reference's own torch expressions
    # (models/ffb6d.py:159-194, restated in _torch_cpu_random_sample) on THIS GPU with the same features and
    # int64 indices (train_ycb.py:224-232 casts them before the forward pass; the cast is not timed).
    gpu_torch = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            idx64 = []
            for op, key, C, Sz, Q, K in p.gathers:
                ii = resident_res[0][key].long()
                idx64.append(ii.reshape(B, -1, 1) if op == "choose" else ii)
            feats = [f if args.layout == "nchw" else f.contiguous() for f in p.features]
            for _ in range(2):
                for f, ii in zip(feats, idx64):
                    _torch_cpu_random_sample(f, ii)
            torch.cuda.synchronize()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 3
            g0.record()
            for _ in range(reps):
                for f, ii in zip(feats, idx64):
                    _torch_cpu_random_sample(f, ii)
            g1.record()
            torch.cuda.synchronize()
            t_ref = g0.elapsed_time(g1) / reps
            gpu_torch = {"what": "C5: the 23 gathers of one step through the reference's torch expression "
                                 "(repeat-expanded int64 index + torch.gather + max) on this GPU",
                         "ms_per_step": t_ref, "alg_GBps": p.gather_alg_bytes_per_frame * B / (t_ref / 1e3) / 1e9,
                         "ours_ms_per_step": compute["gather_ms_per_step"],
                         "speedup_of_ours": t_ref / compute["gather_ms_per_step"]}
            del idx64, feats
            torch.cuda.empty_cache()
        except Exception as e:                      # noqa: BLE001
            gpu_torch = {"error": str(e)[:200]}

    # ---- the actual drop-in boundary: DataProcessing.knn_search(numpy) -> ffb6d_knn_batch_host, called
    # exactly as the datasets call it (22 calls per frame, B = 1, numpy in / numpy int32 out; H2D, search,
    # D2H and a stream synchronise inside every call)
    host_api = None
    if world == 1 and not args.no_cpu_baseline:
        from ffb6d_b200.helper_tool import DataProcessing as DP
        from ffb6d_b200.synthetic import image_pyramid_np
        fr_sets = {("cld", i): batch["cld"][0][: N0 // 4 ** i] for i in range(5)}
        for sr, pts in image_pyramid_np(batch["dpt_xyz"][0]).items():
            fr_sets[("img", sr)] = pts
        best = 1e30
        for _ in range(4):
            t0 = time.perf_counter()
            for key_, s_, q_, kk_ in knn_schedule(N0, k=args.k):
                DP.knn_search(fr_sets[s_][None], fr_sets[q_][None], kk_)
            best = min(best, time.perf_counter() - t0)
        host_api = {"what": "22 x DataProcessing.knn_search(numpy) for one frame through ffb6d_knn_batch_host "
                            "(the reference's call pattern, ycb_dataset.py:275-308)",
                    "ms_per_frame": best * 1e3, "points_per_s_knn_only": N0 / best}

    # ---- CPU baseline (rank 0, N=1 only): the reference's compiled ops on this box's cores
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        r = cpu_reference_sample(N0, args.ref_frames or max(8, cores), 2, reps=2, k=args.k)
        cpu_baseline = {"value": N0 / r["sec_per_frame"], "unit": UNIT, "cores": r["cores"],
                        "kind": r["kind"], "sample": r["sample"],
                        "knn_ms_per_frame": r["knn_sec_per_frame"] * 1e3, "gather_ms_per_frame": r["gather_sec_per_frame"] * 1e3}
        try:
            c1 = cpu_reference_sample(N0, 2, 2, k=args.k, gather_threads=r["gather_threads"], mode="as_called")
            c3 = cpu_reference_sample(N0, 2, 2, k=args.k, mode="single")
            cpu_baseline["C1_as_called"] = {"value": N0 / c1["sec_per_frame"], "unit": UNIT, "cores": c1["cores"],
                                            "knn_ms_per_frame": c1["knn_sec_per_frame"] * 1e3, "sample": c1["sample"]}
            cpu_baseline["C3_single_thread"] = {"value": N0 / c3["sec_per_frame"], "unit": UNIT, "cores": 1,
                                                "knn_ms_per_frame": c3["knn_sec_per_frame"] * 1e3,
                                                "gather_ms_per_frame": c3["gather_sec_per_frame"] * 1e3, "sample": c3["sample"]}
        except Exception as e:                      # noqa: BLE001
            cpu_baseline["comparators_error"] = str(e)[:200]

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
        "warmup": args.warmup, "ms_per_step": ms / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": "BASELINE configs[1]: batch=%d synthetic 480x640 RGB-D frames per GPU, %d sampled "
                        "points, K=%d; one pass = 22 KNN index builds + 11 random_sample + 11 "
                        "nearest_interpolation + choose gather (BASELINE.md §3), fusion MLPs not included"
                        % (B, N0, args.k),
            "frames_per_gpu": B, "n_points": N0, "k": args.k, "feature_layout": args.layout,
            "parallelism": "frames sharded over %d GPU(s), no data-path collective" % world,
            "l2": "per-step inputs (%.1f GB of features + xyz) exceed the 126 MB L2; no flush needed"
                  % ((feat_bytes + xyz_h.numel() * 4) / 1e9),
        },
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms / steps,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(ndig) * 4,
                "note": "per step: H2D of the depth map (f32 metres) + choose from pinned memory (double-buffered, "
                        "overlapping the previous pass), back-projection + 22 KNN + 23 gathers on the device, D2H "
                        "of a 256-element digest of each of the 45 results; gather features are device-resident "
                        "activations as in the reference (the network produces them on the GPU)"},
        "gpu_launches": int(launches), "cuda_graph": bool(use_graph),
        "instrumented_ms_per_step": inst_ms / steps, "sum_of_ops_ms_per_step": tot_ms / steps,
        "instrumented_note": "eager launches + per-op events behind a %.1f ms spin kernel; the CPU needs %.1f ms to "
                             "enqueue a step" % (spin_ms / steps, enqueue_ms / steps),
        "digest_ok": digest_ok, "reference_digest_ok": reference_digest_ok,
        "roofline": roofline, "compute": compute, "pass_roofline": pass_roofline,
        "fusion_mlps": mlp_line, "fusion_stack": stack_line, "lfa_blocks": lfa_line, "pose_voting": pose_line, "cpu_baseline": cpu_baseline, "gpu_torch_reference": gpu_torch,
        "host_api": host_api, "clocks": clocks,
    }
    emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
