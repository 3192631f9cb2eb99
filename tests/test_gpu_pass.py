"""GPU: the path bench.py TIMES is the path that is TESTED.

bench.py times CUDA-graph replays of a 2 + 2-stream, event-ordered pass at B = 32 / 12288 points
(pipeline.FusionPass.capture).  Here that exact object is built with the bench's settings, captured,
replayed several times, and every one of its 22 index tensors and 23 gather outputs is compared
bitwise with (a) a sequential single-stream eager pass over the same inputs and (b) the reference's
own outputs (sha256 digests of tests/golden/schedule_digest.json, frames seed0 / seed1 = frames 0 / 1
of the batch; gathers: closed-form selection by the oracle on sampled channels)."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import cpu_oracle as O

pytestmark = pytest.mark.gpu


def _sha(t):
    return hashlib.sha256(np.ascontiguousarray(t.cpu().numpy()).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def batch32():
    from ffb6d_b200.synthetic import make_batch
    return make_batch(range(32), n_points=12288)      # frames 0 and 1 are the golden frames seed0 / seed1


def _device_inputs(batch, dev):
    return (torch.from_numpy(batch["cld"]).to(dev), torch.from_numpy(batch["dpt_xyz"]).to(dev),
            torch.from_numpy(batch["choose"]).to(dev))


def test_graph_replay_equals_sequential_and_reference(cuda, batch32):
    from ffb6d_b200.pipeline import FusionPass
    B = 32
    cld, xyz, cho = _device_inputs(batch32, cuda)
    p = FusionPass(B, n_points=12288, device=cuda, seed=0, n_streams=2)          # bench.py defaults
    seq = FusionPass(B, n_points=12288, device=cuda, seed=0, n_streams=1)        # one stream, no events
    seq.features = p.features                                                      # same feature tensors
    want_in, want_out = seq(cld, xyz, cho)
    torch.cuda.synchronize()
    replay = p.capture(lambda: p(cld, xyz, cho))
    golden = json.load(open(os.path.join(GOLDEN, "schedule_digest.json")))["frames"]
    for it in range(4):
        # poison the outputs of the previous replay: a replay that skipped a kernel would leave garbage
        got_in, got_out = replay()
        torch.cuda.synchronize()
        for key, w in want_in.items():
            assert torch.equal(got_in[key], w), "replay %d: %s differs from the sequential pass" % (it, key)
        for i, (g, w) in enumerate(zip(got_out, want_out)):
            assert torch.equal(g, w), "replay %d: gather %d (%s) differs" % (it, i, p.gathers[i][1])
        for frame, b in (("seed0_n12288", 0), ("seed1_n12288", 1)):
            for key, meta in golden[frame]["keys"].items():
                assert _sha(got_in[key][b]) == meta["sha256"], "replay %d: %s of frame %d != reference" % (it, key, b)
        for key, t in got_in.items():
            if "idx" in key:
                t.fill_(-7)
        for t in got_out:
            t.fill_(float("nan"))
    # gathers against the closed-form selection (oracle) on the reference's index tensors: frames 0, 1, 31
    got_in, got_out = replay()
    torch.cuda.synchronize()
    rs = np.random.RandomState(0)
    for (op, key, C, S, Q, K), feat, out in zip(p.gathers, p.features, got_out):
        for b in (0, 1, B - 1):
            ch = np.sort(rs.choice(C, size=min(C, 8), replace=False))
            f = feat[b:b + 1, ch].cpu().numpy()
            idx = got_in[key][b:b + 1].cpu().numpy()
            if op == "random_sample":
                want = O.random_sample(f, idx)
            elif op == "nearest_interpolation":
                want = O.nearest_interpolation(f, idx)
            else:
                want = O.choose_gather(f, idx)
            g = out[b:b + 1, ch].cpu().numpy().reshape(want.shape)
            assert np.array_equal(g, want), (key, b)


def test_e2e_graph_from_depth_equals_resident(cuda, batch32):
    """The end-to-end variant (depth + choose in, back-projection on the device) produces the same 45
    results as the resident pass, through its captured graph."""
    from ffb6d_b200.ops import intrinsics_to_device
    from ffb6d_b200.pipeline import FusionPass
    from ffb6d_b200.synthetic import INTRINSICS
    B = 4
    sub = {k: v[:B] for k, v in batch32.items()}
    cld, xyz, cho = _device_inputs(sub, cuda)
    dep = torch.from_numpy(sub["depth"]).to(cuda)
    intr = intrinsics_to_device(INTRINSICS["linemod"], cuda)
    p = FusionPass(B, n_points=12288, device=cuda, seed=3, n_streams=2)
    want_in, want_out = p(cld, xyz, cho)
    torch.cuda.synchronize()
    replay = p.capture(lambda: p.from_depth(dep, intr, cho))
    for _ in range(3):
        got_in, got_out = replay()
        torch.cuda.synchronize()
        for key, w in want_in.items():
            assert torch.equal(got_in[key], w), key
        for g, w in zip(got_out, want_out):
            assert torch.equal(g, w)


def test_bench_dump_outputs_are_the_timed_pass(cuda, tmp_path):
    """bench.py --dump-outputs writes what its timed pass returns: the arrays of a pass over the same frames and
    features run here, sampled the same way, under 64 MB in all."""
    import subprocess
    import sys
    import bench
    from conftest import ROOT
    from ffb6d_b200.pipeline import FusionPass
    from ffb6d_b200.synthetic import make_batch
    B, n = 2, 3072
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--batch", str(B), "--n-points", str(n),
                          "--steps", "2", "--warmup", "1", "--no-mlp", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    p = FusionPass(B, n_points=n, device=cuda, seed=0)
    want = bench.sample_outputs(*p(*_device_inputs(make_batch(range(B), n_points=n), cuda)), p.gathers)
    files = sorted(os.listdir(tmp_path))
    assert files == sorted(name + ".npy" for name in want)
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64 * 10 ** 6
    for name, w in want.items():
        got = np.load(tmp_path / (name + ".npy"))
        assert got.dtype in (np.float32, np.float64) and got.dtype == w.dtype, name
        assert np.array_equal(got, w), name


def test_two_devices_in_one_process():
    """Per-device caches (shared-memory opt-in, SM count): ops on cuda:1 after cuda:0 in the same process."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    import ffb6d_b200 as F
    g = torch.Generator().manual_seed(0)
    feat = torch.randn(2, 64, 12288, 1, generator=g)
    idx = torch.randint(0, 12288, (2, 3072, 16), generator=g)
    outs = []
    for d in (0, 1):
        dev = torch.device("cuda", d)
        outs.append(F.random_sample(feat.to(dev), idx.to(dev)).cpu())      # ~98 KB of dynamic shared memory
    assert torch.equal(outs[0], outs[1])
    assert np.array_equal(outs[0].numpy(), O.random_sample(feat.numpy(), idx.numpy()))


def test_index_validation(cuda):
    """Out-of-range neighbour indices are reported by ffb6d_check_indices (torch.gather raises a device
    assert on them); the backward kernels never write outside grad_feat."""
    import ffb6d_b200 as F
    from ffb6d_b200 import _lib
    from ffb6d_b200.ops import check_indices
    idx = torch.randint(0, 50, (2, 30, 16), device=cuda)
    check_indices(idx, 50)
    bad = idx.clone()
    bad[1, 7, 3] = 50
    bad[0, 0, 0] = -1
    with pytest.raises(_lib.FFB6DError, match="2 of"):
        check_indices(bad, 50)
    feat = torch.randn(2, 8, 50, 1, device=cuda, requires_grad=True)
    out = F.random_sample(feat, idx)
    out.sum().backward()
    assert torch.isfinite(feat.grad).all()


def test_wrap_padded_frame_downstream_features_unchanged(cuda, oracle_ref_golden):
    """The datasets pad frames with fewer valid pixels than points by repeating pixels (np.pad 'wrap',
    ycb_dataset.py:230): the cloud then holds duplicated points and KNN has exact distance ties, where our neighbour
    order (ascending index) differs from the reference's (KD-tree traversal order).  Duplicated points carry identical
    features (same pixel, same network input), so every gather of the forward pass must still produce the reference's
    values: checked with features that are functions of the point coordinates, the reference's KNN (oracle) on one side
    and our index build on the other."""
    import ffb6d_b200 as F
    from ffb6d_b200.schedule import gather_schedule, knn_schedule
    from ffb6d_b200.synthetic import image_pyramid_np, make_frame
    n = 3072
    fr = make_frame(11, n_points=n)
    rs = np.random.RandomState(5)
    keep = fr["choose"][0][: n * 5 // 8]
    choose = np.pad(keep, (0, n - len(keep)), "wrap")
    choose = choose[rs.permutation(n)]
    cld = fr["dpt_xyz"].reshape(-1, 3)[choose]
    assert len(np.unique(choose)) < n                                    # duplicated points exist
    sets = {("cld", i): cld[: n // 4 ** i] for i in range(5)}
    for sr, pts in image_pyramid_np(fr["dpt_xyz"]).items():
        sets[("img", sr)] = pts
    ours = F.build_ffb6d_indices(torch.from_numpy(cld)[None].cuda(), torch.from_numpy(fr["dpt_xyz"])[None].cuda())
    # the reference's own compiled KNN (KD-tree traversal order under ties), stored in tests/golden
    from conftest import reference_knn
    ref = {key: reference_knn(oracle_ref_golden, "wrap_" + key, O.knn_search(sets[s][None], sets[q][None], kk))
           for key, s, q, kk in knn_schedule(n)}
    ref.update({"cld_sub_idx%d" % i: ref["cld_nei_idx%d" % i][:, : n // 4 ** (i + 1)] for i in range(4)})
    n_tied = 0
    for key, s, q, kk in knn_schedule(n):
        got = ours[key].cpu().numpy()
        ok, _, _, msg = O.knn_matches(sets[s][None], sets[q][None], got, ref[key])
        assert ok, (key, msg)
        n_tied += int((got != ref[key]).any(axis=2).sum())
    assert n_tied > 0                                                    # the tie order really differs somewhere
    calls = {key: (s, q) for key, s, q, kk in knn_schedule(n)}
    for op, key, C, S, Q, K in gather_schedule(n):
        if op == "choose":
            continue
        base = key.replace("cld_sub_idx", "cld_nei_idx")
        pts = sets[calls[base][0]]                                       # the gather reads features of the SUPPORT set
        assert pts.shape[0] == S
        cc = min(C, 24)
        w = rs.normal(size=(cc, 3)).astype(np.float32)
        feat = np.sin(pts @ w.T * 7.0).T[None, :, :, None].astype(np.float32).copy()      # [1,cc,S,1], a function of xyz
        idx_ours = ours[key]
        if op == "random_sample":
            got = F.random_sample(torch.from_numpy(feat).cuda(), idx_ours).cpu().numpy()
            want = O.random_sample(feat, ref[key].astype(np.int64))
        else:
            got = F.nearest_interpolation(torch.from_numpy(feat).cuda(), idx_ours).cpu().numpy()
            want = O.nearest_interpolation(feat, ref[key].astype(np.int64))
        assert np.array_equal(got, want), key
