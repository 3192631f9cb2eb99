#!/usr/bin/env python
"""Generate tests/golden/*.npz|json by running THE REFERENCE ITSELF in this container.

Sources of truth (nothing here comes from our own oracle or CUDA code):
  * KNN          oracle/_ref/libknn_ref.so  = unmodified NN/knn_.cxx + nanoflann.hpp
                 (``make -C oracle ref``), called like nearest_neighbors.knn_batch.
  * gathers      FFB6D.random_sample / nearest_interpolation (models/ffb6d.py:159-194) and
                 Building_block.gather_neighbour / relative_pos_encoding
                 (models/RandLA/RandLANet.py:216-234), executed from the reference's own
                 source text (oracle/ref_loader.torch_functions), torch CPU, incl. autograd.
  * grid         oracle/_ref/libgrid_ref.so = unmodified grid_subsampling.cpp + cloud.cpp.

Run:  python tests/golden/make_golden.py      (needs /root/reference; rewrites the fixtures)
The reference has no golden vectors of its own (SURVEY.md §4); these are the pin.
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_loader as R                                   # noqa: E402
from ffb6d_b200.synthetic import make_frame, image_pyramid_np       # noqa: E402
from ffb6d_b200.schedule import knn_schedule                        # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def point_sets(frame, n_points):
    sets = {("cld", i): frame["cld"][: n_points // 4 ** i] for i in range(5)}
    for sr, p in image_pyramid_np(frame["dpt_xyz"]).items():
        sets[("img", sr)] = p
    return sets


def knn_cases():
    """Small KNN problems with full inputs and reference outputs."""
    cases = {}
    fr = make_frame(3, n_points=3072)
    ps = point_sets(fr, 3072)
    # (name, support, query, K)
    probs = [
        ("self_768_k16", ps[("cld", 1)], ps[("cld", 1)], 16),
        ("interp_192_768_k1", ps[("cld", 2)], ps[("cld", 1)], 1),
        ("r2p_4800_192_k16", ps[("img", 8)], ps[("cld", 2)], 16),
        ("p2r_192_4800_k1", ps[("cld", 2)], ps[("img", 8)], 1),
        ("self_48_k16", ps[("cld", 3)], ps[("cld", 3)], 16),
    ]
    rs = np.random.RandomState(11)
    u = rs.rand(1000, 3).astype(np.float32)
    uq = rs.rand(500, 3).astype(np.float32)
    probs += [("uniform_1000_500_k%d" % k, u, uq, k) for k in (1, 8, 32)]
    probs.append(("k_gt_s_10_k16", u[:10], uq[:20], 16))           # trailing slots stay 0
    # exact-distance ties: duplicated support points (the datasets' 'wrap' padding)
    base = rs.rand(192, 3).astype(np.float32)
    dup = np.concatenate([base, base[:64]])[rs.permutation(256)]
    probs.append(("ties_256_k8", dup, dup, 8))
    for name, s, q, k in probs:
        idx = R.knn_batch(s[None], q[None], k, omp=False)[0]
        idx_omp = R.knn_batch(s[None], q[None], k, omp=True)[0]
        assert np.array_equal(idx, idx_omp), name
        cases[name + "/support"] = s
        cases[name + "/query"] = q
        cases[name + "/k"] = np.int32(k)
        cases[name + "/idx"] = idx.astype(np.int32)
    # a batched call (B=3) to pin the batch stride handling
    frames = [make_frame(s, n_points=768) for s in (5, 6, 7)]
    sup = np.stack([f["cld"] for f in frames])
    cases["batch3_768_k16/support"] = sup
    cases["batch3_768_k16/query"] = sup
    cases["batch3_768_k16/k"] = np.int32(16)
    cases["batch3_768_k16/idx"] = R.knn_batch(sup, sup, 16, omp=True).astype(np.int32)
    return cases


def schedule_digest(seed, n_points):
    """sha256 of each of the 22 reference index arrays of one full synthetic frame."""
    fr = make_frame(seed, n_points=n_points)
    ps = point_sets(fr, n_points)
    dig = {}
    for key, s, q, k in knn_schedule(n_points):
        idx = R.knn_search(ps[s][None], ps[q][None], k, omp=False)[0]      # int32 like the dataset
        dig[key] = {"sha256": sha(idx), "shape": list(idx.shape), "S": int(len(ps[s])), "K": k}
    return dig


def gather_cases():
    f = R.torch_functions()
    g = torch.Generator().manual_seed(1234)
    cases = {}

    def rnd(*shape):
        return torch.randn(*shape, generator=g)

    def rint(hi, *shape):
        return torch.randint(0, hi, shape, generator=g)

    for name, (B, Cc, S, Q, K) in {"rs_small": (2, 8, 100, 30, 16), "rs_k8": (1, 5, 77, 41, 8),
                                   "rs_wide": (2, 130, 48, 12, 16)}.items():
        feat = rnd(B, Cc, S, 1).requires_grad_(True)
        idx = rint(S, B, Q, K)
        out = f["random_sample"](feat, idx)
        go = rnd(*out.shape)
        out.backward(go)
        cases.update({name + "/feat": feat.detach().numpy(), name + "/idx": idx.numpy(),
                      name + "/out": out.detach().numpy(), name + "/gout": go.numpy(),
                      name + "/gfeat": feat.grad.numpy()})
    for name, (B, Cc, S, Q) in {"ni_small": (2, 8, 48, 200), "ni_wide": (1, 64, 30, 100)}.items():
        feat = rnd(B, Cc, S, 1).requires_grad_(True)
        idx = rint(S, B, Q, 1)
        out = f["nearest_interpolation"](feat, idx)
        go = rnd(*out.shape)
        out.backward(go)
        cases.update({name + "/feat": feat.detach().numpy(), name + "/idx": idx.numpy(),
                      name + "/out": out.detach().numpy(), name + "/gout": go.numpy(),
                      name + "/gfeat": feat.grad.numpy()})
    for name, (B, N, D, K) in {"gn_xyz": (2, 100, 3, 16), "gn_feat": (2, 60, 16, 16),
                               "gn_odd": (1, 33, 5, 7)}.items():
        pc = rnd(B, N, D).requires_grad_(True)
        idx = rint(N, B, N, K)
        out = f["gather_neighbour"](pc, idx)
        go = rnd(*out.shape)
        out.backward(go)
        cases.update({name + "/pc": pc.detach().numpy(), name + "/idx": idx.numpy(),
                      name + "/out": out.detach().numpy(), name + "/gout": go.numpy(),
                      name + "/gpc": pc.grad.numpy()})
    xyz = rnd(2, 100, 3)
    idx = rint(100, 2, 100, 16)
    cases.update({"rpe/xyz": xyz.numpy(), "rpe/idx": idx.numpy(),
                  "rpe/out": f["relative_pos_encoding"](xyz, idx).numpy()})
    return cases


def grid_cases():
    cases = {}
    rs = np.random.RandomState(21)
    pts = (rs.rand(6000, 3) * np.array([2.0, 1.5, 0.7])).astype(np.float32) - 0.4
    feats = rs.rand(6000, 4).astype(np.float32)
    labels = rs.randint(0, 5, (6000,)).astype(np.int32)
    for name, dl in (("g010", 0.10), ("g004", 0.04)):
        p, fe, la = R.grid_subsampling(pts, feats, labels, dl)
        order = np.lexsort((p[:, 2], p[:, 1], p[:, 0]))
        cases.update({name + "/dl": np.float32(dl), name + "/sub_points": p[order],
                      name + "/sub_features": fe[order], name + "/sub_labels": la[order]})
    (p_only,) = R.grid_subsampling(pts, None, None, 0.1)
    order = np.lexsort((p_only[:, 2], p_only[:, 1], p_only[:, 0]))
    cases["g010/points_only"] = p_only[order]
    cases["points"] = pts
    cases["features"] = feats
    cases["labels"] = labels
    return cases


def backproject_digest():
    """sha256 of float32(dpt_2_pcld(depth)) computed by the reference's own method
    (datasets/ycb/ycb_dataset.py:165-176, executed from its source text) for synthetic depth maps."""
    import ast
    path = os.path.join(R.REF_ROOT, "ffb6d", "datasets", "ycb", "ycb_dataset.py")
    tree = ast.parse(open(path).read())
    fn = None
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name == "dpt_2_pcld":
            ns = {"np": np}
            exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
            fn = ns["dpt_2_pcld"]
    assert fn is not None

    class _Self:   # ycb_dataset.py:31-32
        xmap = np.array([[j for i in range(640)] for j in range(480)])
        ymap = np.array([[i for i in range(640)] for j in range(480)])

    from ffb6d_b200.synthetic import INTRINSICS
    out = {}
    for seed, intr in ((0, "linemod"), (7, "ycb_K1")):
        fr = make_frame(seed, n_points=768, intrinsics=intr)
        xyz = fn(_Self(), fr["depth"], 1.0, INTRINSICS[intr]).astype(np.float32)
        assert np.array_equal(xyz, fr["dpt_xyz"])        # the synthetic generator restates the same lines
        out["seed%d_%s" % (seed, intr)] = {"seed": seed, "intrinsics": intr, "sha256_xyz_f32": sha(xyz),
                                           "sha256_depth": sha(fr["depth"])}
    return out


def lfa_cases():
    """RandLA Dilated_res_block (mlp1 -> Building_block -> mlp2 + shortcut -> leaky_relu; Att_pooling
    inside) executed from the reference's own class source (models/RandLA/RandLANet.py:170-250) with the
    reference's pt_utils (models/RandLA/pytorch_utils.py), eval mode, random BN statistics."""
    import ast
    import importlib.util
    import torch.nn as nn
    import torch.nn.functional as Fn
    rdir = os.path.join(R.REF_ROOT, "ffb6d", "models", "RandLA")
    spec = importlib.util.spec_from_file_location("ref_randla_pt_utils", os.path.join(rdir, "pytorch_utils.py"))
    pt_utils = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(pt_utils)
    path = os.path.join(rdir, "RandLANet.py")
    tree = ast.parse(open(path).read())
    ns = {"torch": torch, "nn": nn, "F": Fn, "pt_utils": pt_utils}
    for node in tree.body:
        if isinstance(node, ast.ClassDef) and node.name in ("Dilated_res_block", "Building_block", "Att_pooling"):
            exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
    cases = {}
    # two toy blocks + the four encoder blocks of FFB6D's RandLA branch at their real widths
    # (d_in -> 2*d_out = 8->64, 64->128, 128->256, 256->512; common.py:26) and point counts N_i / 4
    # (a quarter of the real N keeps the fixture small; channel widths are what select the kernels)
    shapes = {"blk_8_16": (8, 16, 2, 96, 16, 0), "blk_32_32": (32, 32, 1, 40, 16, 1),
              "ffb6d_ds0": (8, 32, 1, 3072, 16, 2), "ffb6d_ds1": (64, 64, 1, 768, 16, 3),
              "ffb6d_ds2": (128, 128, 1, 192, 16, 4), "ffb6d_ds3": (256, 256, 1, 48, 16, 5)}
    for name, (d_in, d_out, B, N, K, seed) in shapes.items():
        torch.manual_seed(seed)
        blk = ns["Dilated_res_block"](d_in, d_out)
        g = torch.Generator().manual_seed(100 + seed)
        with torch.no_grad():
            for m in blk.modules():
                if isinstance(m, nn.BatchNorm2d):
                    m.weight.copy_(torch.rand(m.weight.shape, generator=g) + 0.5)
                    m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
                    m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.2)
                    m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.3)
        blk.eval()
        feature = torch.randn(B, d_in, N, 1, generator=g)
        xyz = torch.randn(B, N, 3, generator=g)
        idx = torch.randint(0, N, (B, N, K), generator=g)
        with torch.no_grad():
            out = blk(feature, xyz, idx)
            f_pc = blk.mlp1(feature)
            lfa = blk.lfa(xyz, f_pc, idx)
        cases.update({name + "/feature": feature.numpy(), name + "/xyz": xyz.numpy(), name + "/idx": idx.numpy(),
                      name + "/out": out.numpy(), name + "/lfa_out": lfa.numpy(), name + "/mlp1_out": f_pc.numpy()})
        for k, v in blk.state_dict().items():
            if v.dtype.is_floating_point:
                cases[name + "/sd." + k] = v.numpy()
    return cases


def _ref_pt_utils():
    """The reference's models/pytorch_utils.py (FFB6D flavour of Conv2d: conv -> BatchNorm2d -> ReLU) as a module."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "ref_ffb6d_pt_utils", os.path.join(R.REF_ROOT, "ffb6d", "models", "pytorch_utils.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _randomise_bn(module, g):
    import torch.nn as nn
    with torch.no_grad():
        for m in module.modules():
            if isinstance(m, nn.BatchNorm2d):
                m.weight.copy_(torch.rand(m.weight.shape, generator=g) + 0.5)
                m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.2)
                m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.3)


def fusion_cases():
    """One bidirectional fusion stage exactly as FFB6D.forward composes it (models/ffb6d.py:245-263): the four
    layers are the reference's own pt_utils.Conv2d instances, the gathers its own random_sample /
    nearest_interpolation (AST-extracted); eval mode, random BatchNorm statistics."""
    pt = _ref_pt_utils()
    f = R.torch_functions()
    cases = {}
    for name, (B, Cr, Cp, h, w, N1, K, seed) in {"stage_64": (2, 64, 64, 30, 40, 192, 16, 0),
                                                 "stage_ragged": (1, 40, 24, 9, 11, 50, 16, 1)}.items():
        torch.manual_seed(seed)
        g = torch.Generator().manual_seed(50 + seed)
        layers = {"r2p_pre": pt.Conv2d(Cr, Cp, kernel_size=(1, 1), bn=True),
                  "r2p_fuse": pt.Conv2d(Cp * 2, Cp, kernel_size=(1, 1), bn=True),
                  "p2r_pre": pt.Conv2d(Cp, Cr, kernel_size=(1, 1), bn=True),
                  "p2r_fuse": pt.Conv2d(Cr * 2, Cr, kernel_size=(1, 1), bn=True)}
        for m in layers.values():
            _randomise_bn(m, g)
            m.eval()
        rgb_emb0 = torch.randn(B, Cr, h, w, generator=g)
        p_emb0 = torch.randn(B, Cp, N1, 1, generator=g)
        p2r_idx = torch.randint(0, N1, (B, h * w, 1), generator=g)
        r2p_idx = torch.randint(0, h * w, (B, N1, K), generator=g)
        with torch.no_grad():
            bs, c, hr, wr = rgb_emb0.size()
            p2r_emb = layers["p2r_pre"](p_emb0)
            p2r_emb = f["nearest_interpolation"](p2r_emb, p2r_idx)
            p2r_emb = p2r_emb.view(bs, -1, hr, wr)
            rgb_emb = layers["p2r_fuse"](torch.cat((rgb_emb0, p2r_emb), dim=1))
            r2p_emb = f["random_sample"](rgb_emb0.reshape(bs, c, hr * wr, 1), r2p_idx).view(bs, c, -1, 1)
            r2p_emb = layers["r2p_pre"](r2p_emb)
            p_emb = layers["r2p_fuse"](torch.cat((p_emb0, r2p_emb), dim=1))
        cases.update({name + "/rgb_emb0": rgb_emb0.numpy(), name + "/p_emb0": p_emb0.numpy(),
                      name + "/p2r_idx": p2r_idx.numpy(), name + "/r2p_idx": r2p_idx.numpy(),
                      name + "/rgb_emb": rgb_emb.numpy(), name + "/p_emb": p_emb.numpy()})
        for lname, m in layers.items():
            for k, v in m.state_dict().items():
                if v.dtype.is_floating_point:
                    cases["%s/sd.%s.%s" % (name, lname, k)] = v.numpy()
    return cases


def train_cases():
    """TRAINING-mode fixtures (batch-statistics BatchNorm, autograd gradients) from the reference's own modules:
    fusion pt_utils.Conv2d layers (models/pytorch_utils.py:75-129) on a concat input, and RandLA's Att_pooling /
    Dilated_res_block (models/RandLA/RandLANet.py:170-250).  Gradients of a fixed upstream gradient `gout`."""
    import ast
    import importlib.util
    import torch.nn as nn
    import torch.nn.functional as Fn
    pt = _ref_pt_utils()
    cases = {}
    for name, (B, C1, C2, Co, tail, seed) in {"conv_cat": (2, 24, 40, 48, (12, 10), 0), "conv_pre": (2, 64, 0, 32, (50, 1), 1),
                                              "conv_wide": (1, 256, 256, 128, (192, 1), 2)}.items():
        torch.manual_seed(seed)
        g = torch.Generator().manual_seed(70 + seed)
        layer = pt.Conv2d(C1 + C2, Co, kernel_size=(1, 1), bn=True)
        _randomise_bn(layer, g)
        layer.train()
        x1 = torch.randn((B, C1) + tail, generator=g).requires_grad_(True)
        x2 = torch.randn((B, C2) + tail, generator=g).requires_grad_(True) if C2 else None
        before = {k: v.clone() for k, v in layer.state_dict().items()}
        x = torch.cat((x1, x2), dim=1) if C2 else x1
        out = layer(x)
        gout = torch.randn(out.shape, generator=g)
        out.backward(gout)
        cases.update({name + "/x1": x1.detach().numpy(), name + "/out": out.detach().numpy(), name + "/gout": gout.numpy(),
                      name + "/gx1": x1.grad.numpy(), name + "/gw": layer.conv.weight.grad.numpy(),
                      name + "/ggamma": layer.normlayer.bn.weight.grad.numpy(),
                      name + "/gbeta": layer.normlayer.bn.bias.grad.numpy()})
        if C2:
            cases.update({name + "/x2": x2.detach().numpy(), name + "/gx2": x2.grad.numpy()})
        for k, v in before.items():
            if v.dtype.is_floating_point:
                cases["%s/sd.%s" % (name, k)] = v.numpy()
        for k in ("normlayer.bn.running_mean", "normlayer.bn.running_var"):
            cases["%s/after.%s" % (name, k)] = layer.state_dict()[k].numpy()
    # RandLA block in training mode
    rdir = os.path.join(R.REF_ROOT, "ffb6d", "models", "RandLA")
    spec = importlib.util.spec_from_file_location("ref_randla_pt_utils", os.path.join(rdir, "pytorch_utils.py"))
    rpt = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(rpt)
    path = os.path.join(rdir, "RandLANet.py")
    tree = ast.parse(open(path).read())
    ns = {"torch": torch, "nn": nn, "F": Fn, "pt_utils": rpt}
    for node in tree.body:
        if isinstance(node, ast.ClassDef) and node.name in ("Dilated_res_block", "Building_block", "Att_pooling"):
            exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
    for name, (d_in, d_out, B, N, K, seed) in {"blk_train_8_16": (8, 16, 2, 96, 16, 0),
                                               "blk_train_64_64": (64, 64, 1, 192, 16, 1)}.items():
        torch.manual_seed(seed)
        blk = ns["Dilated_res_block"](d_in, d_out)
        g = torch.Generator().manual_seed(200 + seed)
        _randomise_bn(blk, g)
        blk.train()
        feature = torch.randn(B, d_in, N, 1, generator=g).requires_grad_(True)
        xyz = torch.randn(B, N, 3, generator=g)
        idx = torch.randint(0, N, (B, N, K), generator=g)
        before = {k: v.clone() for k, v in blk.state_dict().items()}
        out = blk(feature, xyz, idx)
        gout = torch.randn(out.shape, generator=g)
        out.backward(gout)
        cases.update({name + "/feature": feature.detach().numpy(), name + "/xyz": xyz.numpy(), name + "/idx": idx.numpy(),
                      name + "/out": out.detach().numpy(), name + "/gout": gout.numpy(), name + "/gfeature": feature.grad.numpy()})
        for k, v in before.items():
            if v.dtype.is_floating_point:
                cases["%s/sd.%s" % (name, k)] = v.numpy()
        for k, prm in blk.named_parameters():
            cases["%s/grad.%s" % (name, k)] = prm.grad.numpy()
        for k, v in blk.state_dict().items():
            if "running_" in k:
                cases["%s/after.%s" % (name, k)] = v.numpy()
    return cases


def pose_vote_sets(seed, n, n_sets=3):
    """Synthetic keypoint votes: a dense cluster around the true keypoint, a smaller decoy cluster and
    uniform outliers (what per-point offset predictions look like on a partly mis-segmented object)."""
    g = np.random.RandomState(seed)
    sets = []
    for s in range(n_sets):
        centre = g.uniform(-0.2, 0.2, 3) + np.array([0.0, 0.0, 0.9])
        n_main = int(n * 0.7)
        n_decoy = int(n * 0.2)
        main = centre + g.normal(0, 0.008 + 0.004 * s, (n_main, 3))
        decoy = centre + np.array([0.09, -0.03, 0.02]) + g.normal(0, 0.01, (n_decoy, 3))
        out = centre + g.uniform(-0.3, 0.3, (n - n_main - n_decoy, 3))
        v = np.concatenate((main, decoy, out)).astype(np.float32)
        sets.append(v[g.permutation(n)])
    return np.stack(sets)


def pose_cases():
    """Outputs of the reference's MeanShiftTorch.fit / best_fit_transform (executed from its source on the CPU)."""
    P = R.pose_functions()
    out = {}
    for name, seed, n, bw, max_iter in (("small", 0, 64, 0.04, 300), ("mid", 1, 700, 0.04, 300), ("wide", 2, 1500, 0.05, 300),
                                        ("capped", 3, 400, 0.04, 5), ("single", 4, 1, 0.04, 300)):
        votes = pose_vote_sets(seed, n)
        out[name + "_votes"] = votes
        out[name + "_params"] = np.array([bw, max_iter], np.float64)
        ms = P["MeanShiftTorch"](bandwidth=bw, max_iter=max_iter)
        ctrs, labs = [], []
        for g in range(votes.shape[0]):
            c, lab = ms.fit(torch.from_numpy(votes[g]))
            ctrs.append(c.numpy())
            labs.append(lab.numpy())
        out[name + "_centres"] = np.stack(ctrs).astype(np.float32)
        out[name + "_labels"] = np.stack(labs).astype(np.uint8)
    g = np.random.RandomState(11)
    A = g.uniform(-0.1, 0.1, (6, 9, 3))
    Bs = []
    for k in range(6):
        q, _ = np.linalg.qr(g.normal(size=(3, 3)))
        if np.linalg.det(q) < 0:
            q[:, 0] *= -1
        Bs.append(A[k] @ q.T + g.uniform(-0.5, 0.5, 3) + g.normal(0, 0.002, (9, 3)))
    A[4, :, 2] = 0.0                                         # coplanar mesh keypoints
    Bs[5] = Bs[5] * np.array([1.0, 1.0, -1.0])               # a mirrored target: the reflection branch
    B = np.stack(Bs)
    A32, B32 = A.astype(np.float32), B.astype(np.float32)
    out["fit_A"], out["fit_B"] = A32, B32
    out["fit_T"] = np.stack([P["best_fit_transform"](A32[k].astype(np.float64), B32[k].astype(np.float64)) for k in range(6)])
    return out


def wrap_padded_frame(n):
    """A frame padded with repeated pixels (np.pad 'wrap', ycb_dataset.py:230): duplicated points, exact KNN ties."""
    fr = make_frame(11, n_points=n)
    rs = np.random.RandomState(5)
    keep = fr["choose"][0][: n * 5 // 8]
    choose = np.pad(keep, (0, n - len(keep)), "wrap")[rs.permutation(n)]
    return dict(fr, cld=fr["dpt_xyz"].reshape(-1, 3)[choose])


def oracle_ref_cases():
    """The reference's results on the seeded inputs of tests/test_oracle_vs_ref.py (and of the wrap-padded frame
    of tests/test_gpu_pass.py).  Results those tests compare exactly are stored as sha256 digests.  A KNN result
    is stored as the rows where it differs from the oracle's result on the same inputs (tie order), plus the
    sha256 of the whole int64 array: the test rebuilds the reference's array from the oracle's and checks it."""
    from oracle import cpu_oracle as O
    cases = {}

    def knn(name, sup, qry, k, want):
        want = want.astype(np.int64)
        got = O.knn_batch(sup, qry, k).astype(np.int64)
        rows = np.argwhere((got != want).any(axis=2)).astype(np.int32)
        cases[name + "/rows"] = rows
        cases[name + "/vals"] = want[rows[:, 0], rows[:, 1]].astype(np.int32)
        cases[name + "/sha256"] = np.array(sha(want))

    for seed, S, Q, K in ((0, 500, 300, 16), (1, 2000, 100, 1), (2, 64, 64, 32), (3, 5, 9, 8), (4, 3000, 700, 4)):
        rs = np.random.RandomState(seed)
        sup = rs.randn(2, S, 3).astype(np.float32)
        qry = rs.randn(2, Q, 3).astype(np.float32)
        knn("random%d" % seed, sup, qry, K, R.knn_batch(sup, qry, K, omp=True))
    cld = make_frame(9, n_points=3072)["cld"][None]
    knn("surface", cld, cld, 16, R.knn_batch(cld, cld, 16))
    for n in (4096, 40960, 131072):
        fr = make_frame(21, n_points=n)
        lvl1 = fr["cld"][None, : n // 4]
        lvl2 = fr["cld"][None, : n // 16]
        img = np.ascontiguousarray(fr["dpt_xyz"][::4, ::4].reshape(1, -1, 3))
        for j, (sup, qry, k) in enumerate(((lvl1, lvl1, 16), (lvl2, img, 1), (img, lvl2, 32))):
            knn("stress%d_%d" % (n, j), sup, qry, k, R.knn_batch(sup, qry, k))
    n = 3072
    sets = point_sets(wrap_padded_frame(n), n)
    for key, s, q, k in knn_schedule(n):
        knn("wrap_" + key, sets[s][None], sets[q][None], k, R.knn_search(sets[s][None], sets[q][None], k))

    f = R.torch_functions()
    g = torch.Generator().manual_seed(7)
    feat = torch.randn(3, 17, 211, 1, generator=g)
    idx = torch.randint(0, 211, (3, 50, 16), generator=g)
    cases["torch/random_sample"] = np.array(sha(f["random_sample"](feat, idx).numpy()))
    idx1 = torch.randint(0, 211, (3, 400, 1), generator=g)
    cases["torch/nearest_interpolation"] = np.array(sha(f["nearest_interpolation"](feat, idx1).numpy()))
    pc = torch.randn(2, 90, 6, generator=g)
    nidx = torch.randint(0, 90, (2, 90, 16), generator=g)
    cases["torch/gather_neighbour"] = np.array(sha(f["gather_neighbour"](pc, nidx).numpy()))

    rs = np.random.RandomState(5)
    pts = (rs.randn(4000, 3) * 0.5).astype(np.float32)
    feats = rs.rand(4000, 3).astype(np.float32)
    rp, rf = R.grid_subsampling(pts, feats, None, 0.07)
    o = np.lexsort((rp[:, 2], rp[:, 1], rp[:, 0]))
    cases["grid/points"] = np.array(sha(rp[o]))
    cases["grid/features"] = np.array(sha(rf[o]))
    return cases


def main():
    if not R.reference_sources_present():
        raise SystemExit("needs /root/reference")
    R.build_ref()
    if len(sys.argv) > 2 and sys.argv[1] == "--only":      # regenerate one fixture file
        which = sys.argv[2]
        fn = {"lfa": lfa_cases, "knn": knn_cases, "gather": gather_cases, "grid": grid_cases, "train": train_cases,
              "fusion": fusion_cases, "pose": pose_cases, "oracle_ref": oracle_ref_cases}[which]
        np.savez_compressed(os.path.join(OUT, which + "_cases.npz"), **fn())
        print("rewrote", which + "_cases.npz")
        return
    np.savez_compressed(os.path.join(OUT, "knn_cases.npz"), **knn_cases())
    np.savez_compressed(os.path.join(OUT, "gather_cases.npz"), **gather_cases())
    np.savez_compressed(os.path.join(OUT, "grid_cases.npz"), **grid_cases())
    np.savez_compressed(os.path.join(OUT, "lfa_cases.npz"), **lfa_cases())
    np.savez_compressed(os.path.join(OUT, "fusion_cases.npz"), **fusion_cases())
    np.savez_compressed(os.path.join(OUT, "train_cases.npz"), **train_cases())
    np.savez_compressed(os.path.join(OUT, "pose_cases.npz"), **pose_cases())
    np.savez_compressed(os.path.join(OUT, "oracle_ref_cases.npz"), **oracle_ref_cases())
    dig = {"generator": "ffb6d_b200.synthetic.make_frame", "frames": {}}
    for seed, n in ((0, 12288), (1, 12288), (2, 3072)):
        dig["frames"]["seed%d_n%d" % (seed, n)] = {"seed": seed, "n_points": n,
                                                    "keys": schedule_digest(seed, n)}
    with open(os.path.join(OUT, "schedule_digest.json"), "w") as fh:
        json.dump(dig, fh, indent=1, sort_keys=True)
    with open(os.path.join(OUT, "backproject_digest.json"), "w") as fh:
        json.dump(backproject_digest(), fh, indent=1, sort_keys=True)
    print("golden fixtures written to", OUT)


if __name__ == "__main__":
    main()
