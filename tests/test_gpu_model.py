"""GPU: FFB6DFusionNet (the RandLA branch + the 28 fusion layers + the heads of FFB6D.forward, models/ffb6d.py:
203-337, on this package's kernels) against a plain-torch float64 restatement of the same lines built from the
same state dict: forward values and, in training mode, the gradients of every parameter and of the image-branch
inputs.  Index tensors come from build_ffb6d_indices (itself pinned to the reference elsewhere)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

from ffb6d_b200.model import FFB6DFusionNet
from ffb6d_b200.schedule import build_ffb6d_indices
from ffb6d_b200.synthetic import make_batch

pytestmark = pytest.mark.gpu


class TorchRef:
    """The reference's forward with torch ops only (float64), parameters taken from a state dict by the
    reference's names.  ``train``: BatchNorm uses batch statistics."""

    def __init__(self, sd, train, n_kps, dtype=torch.float64):
        self.p = {k: v.detach().to(dtype).requires_grad_(v.dtype.is_floating_point and "running" not in k)
                  for k, v in sd.items() if v.dtype.is_floating_point}
        self.train, self.n_kps, self.dtype = train, n_kps, dtype

    def conv(self, pre, x, bn_name, eps, act, slope=0.2):
        w = self.p[pre + ".conv.weight"]
        y = torch.einsum("oc,bc...->bo...", w.reshape(w.shape[0], -1), x)
        if pre + ".conv.bias" in self.p:
            y = y + self.p[pre + ".conv.bias"].view(1, -1, *([1] * (y.dim() - 2)))
        b = pre + "." + bn_name + ".bn."
        if b + "weight" in self.p:
            y = Fn.batch_norm(y, self.p[b + "running_mean"].clone(), self.p[b + "running_var"].clone(), self.p[b + "weight"],
                              self.p[b + "bias"], self.train, 0.1, eps)
        if act == "relu":
            y = torch.relu(y)
        elif act == "leaky":
            y = Fn.leaky_relu(y, slope)
        return y

    def fconv(self, pre, x):                        # fusion flavour
        return self.conv(pre, x, "normlayer", 1e-5, "relu")

    def rconv(self, pre, x, act="leaky"):           # RandLA flavour
        return self.conv(pre, x, "bn", 1e-6, act)

    @staticmethod
    def random_sample(feature, idx):                # models/ffb6d.py:159-177
        f = feature.squeeze(3) if feature.dim() == 4 else feature
        B, d, K = f.shape[0], f.shape[1], idx.shape[-1]
        g = torch.gather(f, 2, idx.reshape(B, 1, -1).expand(-1, d, -1).long())
        return g.reshape(B, d, -1, K).max(dim=3, keepdim=True)[0]

    @staticmethod
    def nearest(feature, idx):                      # :179-194
        f = feature.squeeze(3)
        B, d = f.shape[0], f.shape[1]
        return torch.gather(f, 2, idx.reshape(B, 1, -1).expand(-1, d, -1).long()).unsqueeze(3)

    def att_pool(self, pre, fs):                    # RandLANet.py:243-250
        w = self.p[pre + ".fc.weight"]
        att = torch.einsum("oc,bcnk->bonk", w.reshape(w.shape[0], -1), fs)
        agg = torch.sum(fs * torch.softmax(att, dim=3), dim=3, keepdim=True)
        return self.rconv(pre + ".mlp", agg)

    def block(self, pre, feature, xyz, idx):        # RandLANet.py:170-234
        B, N, K = idx.shape
        f_pc = self.rconv(pre + ".mlp1", feature)
        nb = torch.gather(xyz, 1, idx.reshape(B, -1, 1).expand(-1, -1, 3).long()).reshape(B, N, K, 3)
        tile = xyz.unsqueeze(2).expand(-1, -1, K, -1)
        rel = tile - nb
        dis = torch.sqrt(torch.sum(rel ** 2, dim=-1, keepdim=True))
        f_xyz = torch.cat([dis, rel, tile, nb], dim=-1).permute(0, 3, 1, 2)
        f_xyz = self.rconv(pre + ".lfa.mlp1", f_xyz)

        def gather_cm(f):
            d = f.shape[1]
            return torch.gather(f.squeeze(3), 2, idx.reshape(B, 1, -1).expand(-1, d, -1).long()).reshape(B, d, N, K)

        agg = self.att_pool(pre + ".lfa.att_pooling_1", torch.cat([gather_cm(f_pc), f_xyz], 1))
        f_xyz = self.rconv(pre + ".lfa.mlp2", f_xyz)
        agg = self.att_pool(pre + ".lfa.att_pooling_2", torch.cat([gather_cm(agg), f_xyz], 1))
        return Fn.leaky_relu(self.rconv(pre + ".mlp2", agg, None) + self.rconv(pre + ".shortcut", feature, None), 0.2)

    def fuse(self, tag, i, rgb0, p0, p2r_idx, r2p_idx):      # models/ffb6d.py:245-263
        bs, c, hr, wr = rgb0.shape
        p2r = self.nearest(self.fconv("%s_fuse_p2r_pre_layers.%d" % (tag, i), p0), p2r_idx).view(bs, -1, hr, wr)
        rgb = self.fconv("%s_fuse_p2r_fuse_layers.%d" % (tag, i), torch.cat((rgb0, p2r), 1))
        r2p = self.random_sample(rgb0.reshape(bs, c, hr * wr, 1), r2p_idx)
        r2p = self.fconv("%s_fuse_r2p_pre_layers.%d" % (tag, i), r2p)
        return rgb, self.fconv("%s_fuse_r2p_fuse_layers.%d" % (tag, i), torch.cat((p0, r2p), 1))

    def forward(self, inp, rgb_feats):
        p_emb = self.rconv("rndla_pre_stages", inp["cld_rgb_nrm"].to(self.dtype)).unsqueeze(3)
        ds_emb, fused = [], []
        for i in range(4):
            f_enc = self.block("rndla_ds_stages.%d" % i, p_emb, inp["cld_xyz%d" % i].to(self.dtype), inp["cld_nei_idx%d" % i])
            p0 = self.random_sample(f_enc, inp["cld_sub_idx%d" % i])
            if i == 0:
                ds_emb.append(f_enc)
            rgb, p_emb = self.fuse("ds", i, rgb_feats[i], p0, inp["p2r_ds_nei_idx%d" % i], inp["r2p_ds_nei_idx%d" % i])
            ds_emb.append(p_emb)
            fused.append(rgb)
        for i in range(3):
            f_interp = self.nearest(p_emb, inp["cld_interp_idx%d" % (3 - i)])
            p0 = self.rconv("rndla_up_stages.%d" % i, torch.cat([ds_emb[-i - 2], f_interp], 1))
            rgb, p_emb = self.fuse("up", i, rgb_feats[4 + i], p0, inp["p2r_up_nei_idx%d" % i], inp["r2p_up_nei_idx%d" % i])
            fused.append(rgb)
        f_interp = self.nearest(p_emb, inp["cld_interp_idx0"])
        p_emb = self.rconv("rndla_up_stages.3", torch.cat([ds_emb[0], f_interp], 1)).squeeze(-1)
        rgb = rgb_feats[7]
        bs, di = rgb.shape[0], rgb.shape[1]
        rgb_c = torch.gather(rgb.view(bs, di, -1), 2, inp["choose"].expand(-1, di, -1).long())
        x0 = torch.cat([rgb_c, p_emb], 1)
        outs = []
        for head in ("rgbd_seg_layer", "kp_ofst_layer", "ctr_ofst_layer"):
            x = x0
            for j in range(3):
                x = self.conv("%s.%d" % (head, j), x, "normlayer", 1e-5, "relu")
            outs.append(self.conv("%s.3" % head, x, "normlayer", 1e-5, None))
        segs, kp, ctr = outs
        kp = kp.view(bs, self.n_kps, 3, -1).permute(0, 1, 3, 2).contiguous()
        ctr = ctr.view(bs, 1, 3, -1).permute(0, 1, 3, 2).contiguous()
        return {"pred_rgbd_segs": segs, "pred_kp_ofs": kp, "pred_ctr_ofs": ctr, "fused_rgb": fused}


def close(got, want, what, tol):
    got, want = got.detach().double().cpu().numpy(), want.detach().double().cpu().numpy()
    scale = max(np.abs(want).max(), 1e-6)
    err = np.abs(got - want).max()
    assert err <= tol * scale, "%s: max abs err %.3e at scale %.3e (%.2e relative)" % (what, err, scale, err / scale)


@pytest.mark.parametrize("train", [False, True], ids=["eval", "train"])
def test_fusion_net_matches_torch_restatement(cuda, train):
    B, h, w, n_pts, n_kps = 2, 120, 160, 4096, 8
    torch.manual_seed(3)
    model = FFB6DFusionNet(n_classes=5, n_pts=n_pts, n_kps=n_kps).cuda()
    g = torch.Generator().manual_seed(9)
    with torch.no_grad():   # non-trivial BatchNorm parameters and statistics
        for m in model.modules():
            if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
                m.weight.copy_(torch.rand(m.weight.shape, generator=g) + 0.5)
                m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.1)
                m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.5)
    model.train(train)
    batch = make_batch([3, 4], n_points=n_pts, h=h, w=w)
    cld = torch.from_numpy(batch["cld"]).cuda()
    xyz = torch.from_numpy(batch["dpt_xyz"]).cuda()
    inputs = build_ffb6d_indices(cld, xyz)
    inputs["choose"] = torch.from_numpy(batch["choose"]).cuda()
    inputs["cld_rgb_nrm"] = torch.from_numpy(batch["cld_rgb_nrm"]).cuda()
    gg = torch.Generator(device="cuda").manual_seed(1)
    rgb_feats = [torch.randn(s, generator=gg, device="cuda").requires_grad_(train)
                 for s in FFB6DFusionNet.rgb_feature_shapes(B, h, w)]
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    ref = TorchRef(sd, train, n_kps)
    rgb64 = [t.detach().double().requires_grad_(train) for t in rgb_feats]
    if train:
        out = model(inputs, rgb_feats)
        want = ref.forward(inputs, rgb64)
    else:
        with torch.no_grad():
            out = model(inputs, rgb_feats)
            want = ref.forward(inputs, rgb64)
    def flat(d):
        return [(k, d[k]) for k in ("pred_rgbd_segs", "pred_kp_ofs", "pred_ctr_ofs")] + \
               [("fused_rgb%d" % i, t) for i, t in enumerate(d["fused_rgb"])]

    for (k, a), (_, b) in zip(flat(out), flat(want)):
        close(a, b, "%s %s" % ("train" if train else "eval", k), 5e-5)
    if not train:
        return
    go = [torch.randn(v.shape, generator=gg, device="cuda") for _, v in flat(out)]
    sum((v * g_).sum() for (_, v), g_ in zip(flat(out), go)).backward()
    sum((v * g_.double()).sum() for (_, v), g_ in zip(flat(want), go)).backward()
    # the same composition through torch in fp32: how far plain fp32 autograd lands from the fp64 gradients.
    # (A 60-layer network with batch-statistics BatchNorm over as few as 32 positions, max-pools and ReLU kinks
    # amplifies fp32 round-off; gradient parity per LAYER is pinned at 1e-5 against the reference's own modules
    # in tests/test_gpu_train.py -- here the whole-network gradients must be as close to fp64 as torch's own.)
    ref32 = TorchRef(sd, train, n_kps, dtype=torch.float32)
    rgb32 = [t.detach().clone().requires_grad_(True) for t in rgb_feats]
    want32 = ref32.forward(inputs, rgb32)
    sum((v * g_).sum() for (_, v), g_ in zip(flat(want32), go)).backward()
    # errors are measured against the gradient scale of the parameter's LAYER (largest gradient norm among the
    # parameters of the same conv + BatchNorm unit): a BatchNorm bias gradient is a sum of terms that nearly
    # cancel behind another BatchNorm, its own norm is no yardstick for round-off
    def unit(name):
        return name.rsplit(".conv.", 1)[0].rsplit(".normlayer.", 1)[0].rsplit(".bn.bn.", 1)[0].rsplit(".fc.", 1)[0]

    scale_of = {}
    for name, _ in model.named_parameters():
        scale_of[unit(name)] = max(scale_of.get(unit(name), 1e-12), ref.p[name].grad.norm().item())
    report = []
    for name, prm in model.named_parameters():
        r, r32 = ref.p[name].grad, ref32.p[name].grad
        assert prm.grad is not None and r is not None, name
        nrm = scale_of[unit(name)]
        e_ours = (prm.grad.double() - r).norm().item() / nrm
        e_t32 = (r32.double() - r).norm().item() / nrm
        report.append((e_ours, e_t32, name))
    report.sort(reverse=True)
    print({"worst": report[:10], "median_ours": sorted(x[0] for x in report)[len(report) // 2],
           "median_torch_fp32": sorted(x[1] for x in report)[len(report) // 2]})
    for e_ours, e_t32, name in report:
        assert e_ours <= max(4 * e_t32, 2e-3), "grad %s: error %.3e of its layer's gradient scale (torch fp32: %.3e); worst: %s" % (
            name, e_ours, e_t32, report[:5])
    for t, r, r32 in zip(rgb_feats, rgb64, rgb32):
        if r.grad is not None:
            nrm = max(r.grad.norm().item(), 1e-12)
            e_ours = (t.grad.double() - r.grad).norm().item() / nrm
            e_t32 = (r32.grad.double() - r.grad).norm().item() / nrm
            assert e_ours <= max(4 * e_t32, 2e-3), (e_ours, e_t32)
