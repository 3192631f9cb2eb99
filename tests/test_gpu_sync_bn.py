"""GPU: synchronised BatchNorm of the 1x1 layers (nn.SyncBatchNorm.convert_sync_batchnorm, the reference's
train_ycb.py:568).

1. The split entry points (ffb6d_bn_train_stats -> _apply, _bwd_stats -> _bwd_apply) at one rank reproduce
   ffb6d_bn_train_fwd / _bwd bit for bit.
2. Virtual ranks: 1-frame shards of the reference's training fixtures (tests/golden/train_cases.npz; the
   one-frame fixture split along its positions) with their fp64 sums added in-process give the reference's
   full-batch outputs, gradients and running statistics;
   an uneven 1 + 2 split of a B = 3 batch matches torch's float64 batch_norm of the whole batch.
3. A real process group: two gloo ranks on one GPU, one frame each, converted modules -> the golden values.
4. No process group, or a group of one: a converted module gives the unconverted module's bits (dW to
   the last bits: its atomics make it differ between any two runs).
5. NCCL on two GPUs (skipped with fewer): as 3, plus FFB6DFusionNet against one process with both frames."""
import copy
import os
import sys
import traceback

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as Fn

from conftest import GOLDEN, ROOT

pytestmark = pytest.mark.gpu

FLAVOURS = ((1e-5, 0.1), (1e-6, 0.99))       # fusion / RandLA BatchNorm (eps, momentum)


def load(name):
    z = np.load(os.path.join(GOLDEN, "train_cases.npz"))
    return {k[len(name) + 1:]: z[k] for k in z.files if k.startswith(name + "/")}


def close(got, want, what, tol=1e-5):
    got = got.detach().cpu().numpy().astype(np.float64) if isinstance(got, torch.Tensor) else np.asarray(got, np.float64)
    want = want.detach().cpu().numpy() if isinstance(want, torch.Tensor) else want
    want = np.asarray(want, np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    scale = max(np.abs(want).max(), 1e-3)
    err = np.abs(got - want).max()
    assert err <= tol * scale, "%s: max abs err %.3e at scale %.3e (%.2e relative)" % (what, err, scale, err / scale)


def sd_of(case, module):
    sd = {k[3:]: torch.from_numpy(v) for k, v in case.items() if k.startswith("sd.")}
    for k in module.state_dict():
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.tensor(0)
    return sd


# ----------------------------------------------------------------------------- thin wrappers of the C ABI
def _lib():
    from ffb6d_b200._lib import lib, check
    from ffb6d_b200.ops import _stream
    return lib, check, _stream


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _ws(C, P, dev):
    lib, _, _ = _lib()
    n = int(lib.ffb6d_bn_workspace_bytes(C, P))
    return torch.empty(n, dtype=torch.uint8, device=dev), n


def bn_fwd(z, gamma, beta, eps, mom, rm, rv, act, slope):
    lib, check, stream = _lib()
    B, C, P = z.shape
    stats, y = torch.empty((C, 4), device=z.device), torch.empty_like(z)
    ws, n = _ws(C, P, z.device)
    check(lib.ffb6d_bn_train_fwd(z.data_ptr(), B, C, P, _ptr(gamma), _ptr(beta), eps, mom, _ptr(rm), _ptr(rv), act,
                                 slope, stats.data_ptr(), y.data_ptr(), ws.data_ptr(), n, stream(z.device)))
    return y, stats


def bn_stats(z):
    lib, check, stream = _lib()
    B, C, P = z.shape
    sums = torch.full((C, 2), float("nan"), dtype=torch.float64, device=z.device)
    ws, n = _ws(C, P, z.device)
    check(lib.ffb6d_bn_train_stats(z.data_ptr(), B, C, P, sums.data_ptr(), ws.data_ptr(), n, stream(z.device)))
    return sums


def bn_apply(z, sums, count, gamma, beta, eps, mom, rm, rv, act, slope):
    lib, check, stream = _lib()
    B, C, P = z.shape
    stats, y = torch.empty((C, 4), device=z.device), torch.empty_like(z)
    check(lib.ffb6d_bn_train_apply(z.data_ptr(), B, C, P, sums.data_ptr(), float(count), _ptr(gamma), _ptr(beta), eps,
                                   mom, _ptr(rm), _ptr(rv), act, slope, stats.data_ptr(), y.data_ptr(), stream(z.device)))
    return y, stats


def bn_bwd(z, gy, stats, act, slope):
    lib, check, stream = _lib()
    B, C, P = z.shape
    dz, gg, gb = torch.empty_like(z), torch.empty(C, device=z.device), torch.empty(C, device=z.device)
    ws, n = _ws(C, P, z.device)
    check(lib.ffb6d_bn_train_bwd(z.data_ptr(), gy.data_ptr(), stats.data_ptr(), B, C, P, act, slope, gg.data_ptr(),
                                 gb.data_ptr(), dz.data_ptr(), ws.data_ptr(), n, stream(z.device)))
    return dz, gg, gb


def bn_bwd_stats(z, gy, stats, act, slope):
    lib, check, stream = _lib()
    B, C, P = z.shape
    sums = torch.full((C, 2), float("nan"), dtype=torch.float64, device=z.device)
    gg, gb = torch.empty(C, device=z.device), torch.empty(C, device=z.device)
    ws, n = _ws(C, P, z.device)
    check(lib.ffb6d_bn_train_bwd_stats(z.data_ptr(), gy.data_ptr(), stats.data_ptr(), B, C, P, act, slope,
                                       sums.data_ptr(), gg.data_ptr(), gb.data_ptr(), ws.data_ptr(), n, stream(z.device)))
    return sums, gg, gb


def bn_bwd_apply(z, gy, stats, sums, count, act, slope):
    lib, check, stream = _lib()
    B, C, P = z.shape
    dz = torch.empty_like(z)
    check(lib.ffb6d_bn_train_bwd_apply(z.data_ptr(), gy.data_ptr(), stats.data_ptr(), sums.data_ptr(), float(count),
                                       B, C, P, act, slope, dz.data_ptr(), stream(z.device)))
    return dz


def bits(t):
    return t.contiguous().view(torch.int32 if t.dtype == torch.float32 else torch.int64)


# ----------------------------------------------------------------------------- 1. one-rank identity
@pytest.mark.parametrize("B,C,P", [(2, 64, 3072), (1, 70, 50), (3, 3, 7), (2, 1024, 600), (8, 64, 19200), (2, 16, 98304),
                                   (2, 64, 1001), (1, 32, 3072)])
def test_split_path_is_bit_identical_at_one_rank(cuda, B, C, P):
    g = torch.Generator().manual_seed(P + C)
    z = (torch.randn(B, C, P, generator=g) * 3 + 0.5).cuda()
    gy = torch.randn(B, C, P, generator=g).cuda()
    gamma, beta = (torch.rand(C, generator=g) + 0.5).cuda(), (torch.randn(C, generator=g) * 0.1).cuda()
    rm0, rv0 = (torch.randn(C, generator=g) * 0.1).cuda(), (torch.rand(C, generator=g) + 0.5).cuda()
    for act, slope in ((0, 0.0), (1, 0.0), (2, 0.2)):
        for eps, mom in FLAVOURS:
            what = "B=%d C=%d P=%d act=%d eps=%g" % (B, C, P, act, eps)
            rm_a, rv_a, rm_b, rv_b = rm0.clone(), rv0.clone(), rm0.clone(), rv0.clone()
            y_a, st_a = bn_fwd(z, gamma, beta, eps, mom, rm_a, rv_a, act, slope)
            sums = bn_stats(z)
            y_b, st_b = bn_apply(z, sums, B * P, gamma, beta, eps, mom, rm_b, rv_b, act, slope)
            for name, a, b in (("y", y_a, y_b), ("stats", st_a, st_b), ("running_mean", rm_a, rm_b),
                               ("running_var", rv_a, rv_b)):
                assert torch.equal(bits(a), bits(b)), "%s: %s differs" % (what, name)
            dz_a, gg_a, gb_a = bn_bwd(z, gy, st_a, act, slope)
            bsums, gg_b, gb_b = bn_bwd_stats(z, gy, st_a, act, slope)
            dz_b = bn_bwd_apply(z, gy, st_a, bsums, B * P, act, slope)
            for name, a, b in (("dz", dz_a, dz_b), ("dgamma", gg_a, gg_b), ("dbeta", gb_a, gb_b)):
                assert torch.equal(bits(a), bits(b)), "%s: %s differs" % (what, name)
            assert torch.equal(gb_b.double(), bsums[:, 0].float().double())


# ----------------------------------------------------------------------------- 2. virtual ranks
def _split(t, dim):
    """Two shards of ``t`` [B, C, P]: 1 + (B - 1) frames (dim 0), or halves of the position axis (dim 2)."""
    if t is None:
        return [None, None]
    k = 1 if dim == 0 else t.shape[2] // 2
    return [t.narrow(dim, 0, k).contiguous(), t.narrow(dim, k, t.shape[dim] - k).contiguous()]


def _shard_layer(x1, x2, w2d, gamma, beta, rm, rv, eps, mom, act, slope, gout, dim):
    """One 1x1 conv + BatchNorm + activation layer on [B, C, P] tensors, run as two ranks holding the shards of
    :func:`_split`; the ranks' fp64 sums are added in-process in place of the all-reduce.  Returns the outputs
    and input gradients reassembled from the shards, each rank's running statistics, and the shard-sums of
    dW / dgamma / dbeta."""
    from ffb6d_b200 import modules as M
    lib, check, stream = _lib()
    C1, Co = x1.shape[1], w2d.shape[0]
    xs = list(zip(_split(x1, dim), _split(x2, dim)))
    zs = [M._gemm(u, v, w2d) for u, v in xs]
    count = sum(z.shape[0] * z.shape[2] for z in zs)
    sums = sum(bn_stats(z) for z in zs)
    outs, runs, sts = [], [], []
    for z in zs:
        rm_r, rv_r = rm.clone(), rv.clone()
        y, st = bn_apply(z, sums, count, gamma, beta, eps, mom, rm_r, rv_r, act, slope)
        outs.append(y)
        runs.append((rm_r, rv_r))
        sts.append(st)
    gys = _split(gout, dim)
    parts = [bn_bwd_stats(z, gy, st, act, slope) for z, gy, st in zip(zs, gys, sts)]
    bsums = sum(p[0] for p in parts)
    ggamma, gbeta = sum(p[1] for p in parts), sum(p[2] for p in parts)
    gw = torch.zeros(Co, w2d.shape[1], device=w2d.device)
    gxs = []
    for (u, v), z, gy, st in zip(xs, zs, gys, sts):
        dz = bn_bwd_apply(z, gy, st, bsums, count, act, slope)
        part = torch.empty_like(gw)
        check(lib.ffb6d_fusion_mlp_wgrad(dz.data_ptr(), u.data_ptr(), C1, _ptr(v), w2d.shape[1] - C1, z.shape[0], Co,
                                         z.shape[2], part.data_ptr(), stream(dz.device)))
        gw += part
        gx1 = M._gemm(dz, None, w2d[:, :C1].t().contiguous())
        gx2 = M._gemm(dz, None, w2d[:, C1:].t().contiguous()) if v is not None else None
        gxs.append((gx1, gx2))
    gx1 = torch.cat([g[0] for g in gxs], dim)
    gx2 = torch.cat([g[1] for g in gxs], dim) if x2 is not None else None
    return torch.cat(outs, dim), gx1, gx2, runs, gw, ggamma, gbeta


@pytest.mark.parametrize("name", ["conv_cat", "conv_pre", "conv_wide"])
def test_virtual_ranks_match_reference_full_batch(cuda, name):
    c = load(name)
    B = c["x1"].shape[0]
    dim = 0 if B > 1 else 2          # 1-frame ranks; a one-frame fixture is split along its positions instead
    cu = lambda k: torch.from_numpy(c[k]).cuda().reshape(B, c[k].shape[1], -1)      # noqa: E731
    w = torch.from_numpy(c["sd.conv.weight"]).cuda()
    w2d = w.reshape(w.shape[0], -1).contiguous()
    x2 = cu("x2") if "x2" in c and c["x2"].shape[1] else None
    bn = {k: torch.from_numpy(c["sd.normlayer.bn." + k]).cuda() for k in ("weight", "bias", "running_mean", "running_var")}
    out, gx1, gx2, runs, gw, gg, gb = _shard_layer(cu("x1"), x2, w2d, bn["weight"], bn["bias"], bn["running_mean"],
                                                   bn["running_var"], 1e-5, 0.1, 1, 0.0, cu("gout"), dim)
    close(out.reshape(c["out"].shape), c["out"], name + " out")
    close(gx1.reshape(c["gx1"].shape), c["gx1"], name + " grad x1")
    if x2 is not None:
        close(gx2.reshape(c["gx2"].shape), c["gx2"], name + " grad x2")
    for r in range(2):
        close(runs[r][0], c["after.normlayer.bn.running_mean"], "%s rank %d running_mean" % (name, r))
        close(runs[r][1], c["after.normlayer.bn.running_var"], "%s rank %d running_var" % (name, r))
        assert torch.equal(runs[r][0], runs[0][0]) and torch.equal(runs[r][1], runs[0][1])
    close(gw.reshape(c["gw"].shape), c["gw"], name + " sum of grad W")
    close(gg, c["ggamma"], name + " sum of grad gamma")
    close(gb, c["gbeta"], name + " sum of grad beta")


def test_uneven_split_matches_float64_whole_batch(cuda):
    B, C1, C2, Co, P = 3, 24, 40, 48, 1001
    g = torch.Generator().manual_seed(5)
    x1, x2 = torch.randn(B, C1, P, generator=g).cuda(), torch.randn(B, C2, P, generator=g).cuda()
    w2d = (torch.randn(Co, C1 + C2, generator=g) * 0.2).cuda()
    gamma, beta = (torch.rand(Co, generator=g) + 0.5).cuda(), (torch.randn(Co, generator=g) * 0.1).cuda()
    rm, rv = (torch.randn(Co, generator=g) * 0.1).cuda(), (torch.rand(Co, generator=g) + 0.5).cuda()
    gout = torch.randn(B, Co, P, generator=g).cuda()
    eps, mom, slope = 1e-6, 0.99, 0.2
    out, gx1, gx2, runs, gw, gg, gb = _shard_layer(x1, x2, w2d, gamma, beta, rm, rv, eps, mom, 2, slope, gout, 0)

    d = lambda t: t.detach().double().requires_grad_(True)      # noqa: E731
    x1d, x2d, wd, gd, bd = d(x1), d(x2), d(w2d), d(gamma), d(beta)
    rmd, rvd = rm.double(), rv.double()
    z = torch.einsum("oc,bcp->bop", wd, torch.cat((x1d, x2d), 1))
    want = Fn.leaky_relu(Fn.batch_norm(z, rmd, rvd, gd, bd, True, mom, eps), slope)
    want.backward(gout.double())
    close(out, want, "uneven out")
    close(gx1, x1d.grad, "uneven grad x1")
    close(gx2, x2d.grad, "uneven grad x2")
    for r in range(2):
        close(runs[r][0], rmd, "uneven rank %d running_mean" % r)
        close(runs[r][1], rvd, "uneven rank %d running_var" % r)
    close(gw, wd.grad, "uneven sum of grad W")
    close(gg, gd.grad, "uneven sum of grad gamma")
    close(gb, bd.grad, "uneven sum of grad beta")


# ----------------------------------------------------------------------------- 3 / 5. real process groups
def _fusion_net_case(dev, frames):
    """FFB6DFusionNet as test_gpu_model.py sets it up (seeded weights, non-trivial BatchNorm), on ``frames`` of
    the two-frame batch; returns (model, inputs, rgb_feats, output-gradient list)."""
    from ffb6d_b200.model import FFB6DFusionNet
    from ffb6d_b200.schedule import build_ffb6d_indices
    from ffb6d_b200.synthetic import make_batch
    B, h, w, n_pts = 2, 120, 160, 4096
    torch.manual_seed(3)
    model = FFB6DFusionNet(n_classes=5, n_pts=n_pts, n_kps=8).to(dev)
    g = torch.Generator().manual_seed(9)
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
                m.weight.copy_(torch.rand(m.weight.shape, generator=g) + 0.5)
                m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.1)
                m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.5)
    batch = make_batch([3 + f for f in frames], n_points=n_pts, h=h, w=w)
    inputs = build_ffb6d_indices(torch.from_numpy(batch["cld"]).to(dev), torch.from_numpy(batch["dpt_xyz"]).to(dev))
    inputs["choose"] = torch.from_numpy(batch["choose"]).to(dev)
    inputs["cld_rgb_nrm"] = torch.from_numpy(batch["cld_rgb_nrm"]).to(dev)
    gg = torch.Generator().manual_seed(1)
    sel = list(frames)
    rgb = [torch.randn(s, generator=gg)[sel].to(dev).requires_grad_(True) for s in FFB6DFusionNet.rgb_feature_shapes(B, h, w)]
    return model.train(), inputs, rgb, gg


def _fusion_net_run(model, inputs, rgb, gg, frames):
    out = model(inputs, rgb)
    flat = [out["pred_rgbd_segs"], out["pred_kp_ofs"], out["pred_ctr_ofs"]] + list(out["fused_rgb"])
    go = [torch.randn((2,) + tuple(v.shape[1:]), generator=gg)[list(frames)].to(v.device) for v in flat]
    sum((v * g_).sum() for v, g_ in zip(flat, go)).backward()
    return ([v.detach().cpu().numpy() for v in flat], {k: p.grad.cpu().numpy() for k, p in model.named_parameters()},
            {k: v.cpu().numpy() for k, v in model.state_dict().items() if "running_" in k})


def _dist_worker(rank, world, port, backend, with_net, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    try:
        from ffb6d_b200 import modules as M
        dev = torch.device("cuda", rank if backend == "nccl" else 0)
        torch.cuda.set_device(dev)
        dist.init_process_group(backend, rank=rank, world_size=world, device_id=dev if backend == "nccl" else None)
        res = {}
        c = load("conv_cat")
        layer = M.Conv2d(64, 48, kernel_size=(1, 1), bn=True)
        layer.load_state_dict(sd_of(c, layer), strict=True)
        layer = torch.nn.SyncBatchNorm.convert_sync_batchnorm(layer).to(dev).train()
        assert isinstance(layer.normlayer.bn, torch.nn.SyncBatchNorm)
        x1 = torch.from_numpy(c["x1"][rank:rank + 1]).to(dev).requires_grad_(True)
        x2 = torch.from_numpy(c["x2"][rank:rank + 1]).to(dev).requires_grad_(True)
        out = layer(x1, x2)
        out.backward(torch.from_numpy(c["gout"][rank:rank + 1]).to(dev))
        bn = layer.normlayer.bn
        res["conv"] = {"out": out, "gx1": x1.grad, "gx2": x2.grad, "gw": layer.conv.weight.grad, "ggamma": bn.weight.grad,
                       "gbeta": bn.bias.grad, "running_mean": bn.running_mean, "running_var": bn.running_var}

        c = load("blk_train_8_16")
        blk = M.Dilated_res_block(8, 16)
        blk.load_state_dict(sd_of(c, blk), strict=True)
        blk = torch.nn.SyncBatchNorm.convert_sync_batchnorm(blk).to(dev).train()
        feature = torch.from_numpy(c["feature"][rank:rank + 1]).to(dev).requires_grad_(True)
        out = blk(feature, torch.from_numpy(c["xyz"][rank:rank + 1]).to(dev), torch.from_numpy(c["idx"][rank:rank + 1]).to(dev))
        out.backward(torch.from_numpy(c["gout"][rank:rank + 1]).to(dev))
        r = {"out": out, "gfeature": feature.grad}
        r.update({"grad." + k: p.grad for k, p in blk.named_parameters()})
        r.update({"after." + k: v for k, v in blk.state_dict().items() if "running_" in k})
        res["blk"] = r
        res = {case: {k: v.detach().cpu().numpy() for k, v in d.items()} for case, d in res.items()}
        if with_net:
            model, inputs, rgb, gg = _fusion_net_case(dev, (rank,))
            model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(model)
            res["net"] = _fusion_net_run(model, inputs, rgb, gg, (rank,))
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, res, None))
    except BaseException:
        q.put((rank, None, traceback.format_exc()))


def _run_ranks(backend, with_net):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() + (7 if backend == "nccl" else 3)) % 2000
    procs = [ctx.Process(target=_dist_worker, args=(r, 2, port, backend, with_net, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        got = sorted((q.get(timeout=600) for _ in procs), key=lambda t: t[0])
    finally:
        for p in procs:
            p.join(timeout=120)
            if p.is_alive():
                p.kill()
                p.join()
    for rank, _, err in got:
        assert err is None, "rank %d failed:\n%s" % (rank, err)
    for p in procs:
        assert p.exitcode == 0
    return [res for _, res, _ in got]


def _check_golden_layers(res):
    c = load("conv_cat")
    for r in range(2):
        g = res[r]["conv"]
        close(g["out"], c["out"][r:r + 1], "conv rank %d out" % r)
        close(g["gx1"], c["gx1"][r:r + 1], "conv rank %d grad x1" % r)
        close(g["gx2"], c["gx2"][r:r + 1], "conv rank %d grad x2" % r)
        close(g["running_mean"], c["after.normlayer.bn.running_mean"], "conv rank %d running_mean" % r)
        close(g["running_var"], c["after.normlayer.bn.running_var"], "conv rank %d running_var" % r)
    for k in ("running_mean", "running_var"):
        assert np.array_equal(res[0]["conv"][k], res[1]["conv"][k]), "conv %s differs across ranks" % k
    for k, want in (("gw", "gw"), ("ggamma", "ggamma"), ("gbeta", "gbeta")):    # DDP would average these
        close(res[0]["conv"][k] + res[1]["conv"][k], c[want], "conv sum over ranks of " + k)

    c = load("blk_train_8_16")
    for r in range(2):
        g = res[r]["blk"]
        close(g["out"], c["out"][r:r + 1], "blk rank %d out" % r, tol=2e-5)
        close(g["gfeature"], c["gfeature"][r:r + 1], "blk rank %d grad feature" % r, tol=5e-5)
    for k in res[0]["blk"]:
        if k.startswith("grad."):
            close(res[0]["blk"][k] + res[1]["blk"][k], c[k], "blk sum over ranks of " + k, tol=5e-5)
        elif k.startswith("after."):
            close(res[0]["blk"][k], c[k], "blk " + k)
            assert np.array_equal(res[0]["blk"][k], res[1]["blk"][k]), "blk %s differs across ranks" % k


def test_gloo_two_ranks_on_one_gpu_match_reference(cuda):
    _check_golden_layers(_run_ranks("gloo", with_net=False))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_nccl_two_gpus_match_one_process(cuda):
    res = _run_ranks("nccl", with_net=True)
    _check_golden_layers(res)
    model, inputs, rgb, gg = _fusion_net_case(cuda, (0, 1))
    outs, grads, runs = _fusion_net_run(model, inputs, rgb, gg, (0, 1))
    for i, want in enumerate(outs):
        for r in range(2):
            close(res[r]["net"][0][i], want[r:r + 1], "net output %d rank %d" % (i, r), tol=5e-5)
    for k, want in runs.items():
        assert np.array_equal(res[0]["net"][2][k], res[1]["net"][2][k]), "net %s differs across ranks" % k
        close(res[0]["net"][2][k], want, "net " + k, tol=5e-5)
    # gradients against the scale of the parameter's conv + BatchNorm unit, as test_gpu_model.py measures them
    def unit(name):
        return name.rsplit(".conv.", 1)[0].rsplit(".normlayer.", 1)[0].rsplit(".bn.bn.", 1)[0].rsplit(".fc.", 1)[0]
    scale = {}
    for k, v in grads.items():
        scale[unit(k)] = max(scale.get(unit(k), 1e-12), float(np.linalg.norm(v)))
    for k, want in grads.items():
        err = np.linalg.norm(res[0]["net"][1][k] + res[1]["net"][1][k] - want) / scale[unit(k)]
        assert err <= 2e-3, "net grad %s: %.3e of its layer's gradient scale" % (k, err)


# ----------------------------------------------------------------------------- 4. nothing to sync with
def _train_step(layer, x1, x2, gout):
    layer.zero_grad(set_to_none=True)
    a, b = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
    out = layer(a, b)
    out.backward(gout)
    bn = layer.normlayer.bn
    return [t.detach().clone() for t in (out, a.grad, b.grad, layer.conv.weight.grad, bn.weight.grad, bn.bias.grad,
                                         bn.running_mean, bn.running_var, bn.num_batches_tracked)]


def _same(got, want, what):
    """Bitwise equal, except dW (index 3): ffb6d_fusion_mlp_wgrad adds its split-K partials with fp32 atomics, so
    dW differs in the last bits between any two runs of the same layer."""
    for i, (a, b) in enumerate(zip(got, want)):
        if i == 3:
            close(a, b, what + ": grad W", tol=1e-6)
        else:
            assert torch.equal(a, b), "%s: tensor %d differs" % (what, i)


def test_converted_module_without_process_group_is_unchanged(cuda):
    from ffb6d_b200 import modules as M
    assert not dist.is_initialized()
    c = load("conv_cat")
    plain = M.Conv2d(64, 48, kernel_size=(1, 1), bn=True)
    plain.load_state_dict(sd_of(c, plain), strict=True)
    synced = torch.nn.SyncBatchNorm.convert_sync_batchnorm(copy.deepcopy(plain))
    assert isinstance(synced.normlayer.bn, torch.nn.SyncBatchNorm)
    synced.load_state_dict(plain.state_dict(), strict=True)       # the reference's keys still load
    plain, synced = plain.cuda().train(), synced.cuda().train()
    x1, x2, gout = (torch.from_numpy(c[k]).cuda() for k in ("x1", "x2", "gout"))
    want = _train_step(plain, x1, x2, gout)
    got = _train_step(synced, x1, x2, gout)
    _same(got, want, "no process group")
    # a process group of one rank: nothing to reduce, the same bits again
    dist.init_process_group("gloo", store=dist.HashStore(), rank=0, world_size=1)
    try:
        again = _train_step(synced, x1, x2, gout)
    finally:
        dist.destroy_process_group()
    want2 = _train_step(plain, x1, x2, gout)
    _same(again, want2, "world size 1")
