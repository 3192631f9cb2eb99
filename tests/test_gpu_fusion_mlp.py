"""GPU: the fused cat + 1x1 conv + BatchNorm(eval) + ReLU tensor-core kernel against a float64
evaluation of the reference layer (models/pytorch_utils.py:75-129: conv(bias=False) -> BatchNorm2d
-> ReLU) and against torch's own fp32 path.  Floating-point kernel: tolerance 1e-5 of the output
scale (BASELINE.json "fused features within 1e-5 fp32")."""
import numpy as np
import pytest
import torch
import torch.nn as nn

import ffb6d_b200 as F

pytestmark = pytest.mark.gpu


def _record(name, err_of_scale, rel, rel32):
    """Print the measured errors (DESIGN.md quotes them; shown by ``pytest -s``)."""
    import json
    print(json.dumps({"layer": name, "max_abs_err_over_scale": err_of_scale, "max_rel_err_above_floor": rel,
                      "torch_fp32_rel": rel32}))


def reference_layer(x1, x2, conv, bn, relu=True, dtype=torch.float64):
    x = torch.cat((x1, x2), dim=1) if x2 is not None else x1
    y = nn.functional.conv2d(x.to(dtype), conv.weight.to(dtype))
    y = nn.functional.batch_norm(y, bn.running_mean.to(dtype), bn.running_var.to(dtype), bn.weight.to(dtype),
                                 bn.bias.to(dtype), training=False, eps=bn.eps)
    return torch.relu(y) if relu else y


def make_layer(cin, cout, seed):
    g = torch.Generator().manual_seed(seed)
    conv = nn.Conv2d(cin, cout, (1, 1), bias=False)
    bn = nn.BatchNorm2d(cout)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / cin ** 0.5)
        bn.weight.copy_(torch.rand(cout, generator=g) + 0.5)
        bn.bias.copy_(torch.randn(cout, generator=g) * 0.1)
        bn.running_mean.copy_(torch.randn(cout, generator=g) * 0.2)
        bn.running_var.copy_(torch.rand(cout, generator=g) + 0.3)
    return conv.cuda().eval(), bn.cuda().eval()


# (B, C1, C2, Co, trailing shape): fusion layers of models/ffb6d.py (SURVEY.md App. A.3) + ragged shapes
CASES = [
    (2, 64, 64, 64, (3072, 1)),        # ds0 r2p_fuse
    (2, 64, 64, 64, (120, 160)),       # ds0 p2r_fuse on the image map
    (1, 512, 512, 256, (192, 1)),      # ds2 r2p_fuse
    (1, 1024, 1024, 1024, (60, 80)),   # ds3 p2r_fuse (20 GFLOP / frame)
    (2, 256, 0, 256, (192, 1)),        # *_pre layers: no concat
    (1, 36, 8, 70, (50, 1)),           # ragged: Ci % 32 != 0, Co % 128 != 0, P % 128 != 0
    (1, 5, 0, 3, (7, 1)),              # nothing aligned (scalar path)
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "B%d_%d+%d->%d_%s" % (c[0], c[1], c[2], c[3], "x".join(map(str, c[4]))))
def test_fusion_mlp_matches_reference_layer(cuda, case):
    B, C1, C2, Co, tail = case
    g = torch.Generator().manual_seed(C1 + Co)
    x1 = torch.randn((B, C1) + tail, generator=g).cuda()
    x2 = torch.randn((B, C2) + tail, generator=g).cuda() if C2 else None
    conv, bn = make_layer(C1 + C2, Co, seed=Co)
    scale, shift = F.fold_batchnorm(bn)
    got = F.fusion_mlp(x1, x2, conv.weight, scale, shift)
    want = reference_layer(x1, x2, conv, bn)
    assert got.shape == want.shape and got.dtype == torch.float32
    ref_scale = want.abs().max().item()
    err = (got.double() - want).abs().max().item()
    assert err <= 1e-5 * max(ref_scale, 1.0), "max abs err %.3e (output scale %.3e)" % (err, ref_scale)
    # no worse than torch's own fp32 path (TF32 disabled) by more than a small factor
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        fp32 = reference_layer(x1, x2, conv, bn, dtype=torch.float32)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    err32 = (fp32.double() - want).abs().max().item()
    assert err <= max(8 * err32, 2e-6 * max(ref_scale, 1.0)), (err, err32)
    # element-wise relative error above an absolute floor of 10 % of the output scale (outputs near zero
    # are sums of K cancelling fp32 products: their error scales with the terms, not with the result);
    # 1e-5, or what torch's own fp32 path shows on the same elements if that is larger
    big = want.abs() > 0.1 * max(ref_scale, 1.0)
    if big.any():
        rel = ((got.double() - want).abs()[big] / want.abs()[big]).max().item()
        rel32 = ((fp32.double() - want).abs()[big] / want.abs()[big]).max().item()
        _record("%d+%d->%d x%d" % (C1, C2, Co, int(np.prod(tail))), err / max(ref_scale, 1.0), rel, rel32)
        assert rel <= max(1e-5, 4 * rel32), "element-wise relative err %.3e (torch fp32: %.3e)" % (rel, rel32)
    # without ReLU
    got_lin = F.fusion_mlp(x1, x2, conv.weight, scale, shift, relu=False)
    want_lin = reference_layer(x1, x2, conv, bn, relu=False)
    assert (got_lin.double() - want_lin).abs().max().item() <= 1e-5 * max(want_lin.abs().max().item(), 1.0)


@pytest.mark.parametrize("case", [CASES[0], CASES[3], CASES[5]], ids=["ds0", "ds3", "ragged"])
def test_fusion_mlp_packed_weights_bit_identical(cuda, case):
    """Weights split once (ffb6d_fusion_mlp_pack) give the same bits as the per-call split, and the
    pack survives many calls."""
    B, C1, C2, Co, tail = case
    g = torch.Generator().manual_seed(7)
    x1 = torch.randn((B, C1) + tail, generator=g).cuda()
    x2 = torch.randn((B, C2) + tail, generator=g).cuda() if C2 else None
    conv, bn = make_layer(C1 + C2, Co, seed=3)
    scale, shift = F.fold_batchnorm(bn)
    packed = F.fusion_mlp_pack(conv.weight)
    assert packed.Co == Co and packed.Ci == C1 + C2
    want = F.fusion_mlp(x1, x2, conv.weight, scale, shift)
    for _ in range(3):
        got = F.fusion_mlp(x1, x2, packed, scale, shift)
        assert torch.equal(got, want)
    with pytest.raises(ValueError):
        F.fusion_mlp(x1[:, :-1], x2, packed, scale, shift)
