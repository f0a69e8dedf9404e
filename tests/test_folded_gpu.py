"""GPU tests of the folded pack block (packnet_sfm_b200/folded.py, csrc/fold_kernels.cu).

The fold is the default path of pack1..pack3 since round 2 (B200: 37.9 -> 30.9 ms per step); the un-folded path (feature
stencil + convolution over the inflated channel count) still serves pack4 / pack5 and stays covered by tests/test_layers_gpu.py
and the `unfolded` parameter of tests/test_packnet_gpu.py."""
import os

import pytest
import torch
import torch.nn.functional as F

from conftest import assert_golden_close, load_golden, rel_l2
from oracle import packnet_oracle as PO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def nchw(x):
    return x.permute(0, 3, 1, 2).contiguous()


@pytest.mark.parametrize("case", [(4, 8, 3), (3, 33, 3), (2, 6, 5), (16, 64, 5), (64, 64, 3), (5, 40, 5)])
def test_fold_kernels_match_the_pytorch_definition(case):
    """pn_pack_fold_forward / backward (nine windows) against conv_transpose3d in float64, values and gradients."""
    from packnet_sfm_b200 import folded
    co, C, k = case
    n = 4 * C
    torch.manual_seed(co + C + k)
    w2 = ((torch.rand(co, 8 * n, k, k, device=DEV) - 0.5)).requires_grad_(True)
    w3 = (torch.rand(8, 1, 3, 3, 3, device=DEV) - 0.5).requires_grad_(True)
    outs = folded.fold_set(w2, w3)
    gs = [torch.rand_like(o) - 0.5 for o in outs]
    torch.autograd.backward(outs, gs)
    torch.cuda.synchronize()
    w2d, w3d = (t.detach().double().requires_grad_(True) for t in (w2, w3))
    refs = folded.fold_set_torch(w2d, w3d)
    torch.autograd.backward(refs, [g.double() if i in (0, 9) else g.double().permute(0, 3, 1, 2) for i, g in enumerate(gs)])
    for name, a, b in zip(folded.FOLD_ORDER + ("S",), outs, refs):
        if name not in ("main", "S"):
            b = b.permute(0, 2, 3, 1)            # the kernels emit the frame weights channels-last
        assert a.shape == b.shape, name
        assert rel_l2(a, b) < 1e-6, (name, rel_l2(a, b))
    assert rel_l2(w2.grad, w2d.grad) < 1e-6, rel_l2(w2.grad, w2d.grad)
    assert rel_l2(w3.grad, w3d.grad) < 1e-5, rel_l2(w3.grad, w3d.grad)


@pytest.mark.parametrize("case", [(2, 16, 24, 32, 16, 3), (1, 16, 24, 40, 16, 5), (4, 64, 12, 40, 128, 3), (2, 64, 48, 64, 64, 5)])
def test_folded_pack_conv_on_the_engine(case):
    """space-to-depth + folds + tcgen05 convolution + frame strips against the reference composition in float64."""
    from packnet_sfm_b200 import folded, functional as PF
    B, C, H, W, Co, k = case
    torch.manual_seed(B + C + H + k)
    x = (torch.rand(B, H, W, C, device=DEV) - 0.5).requires_grad_(True)
    w2 = ((torch.rand(Co, 32 * C, k, k, device=DEV) - 0.5) * (2.0 / (32 * C * k * k) ** 0.5)).requires_grad_(True)
    b2 = (torch.rand(Co, device=DEV) - 0.5).requires_grad_(True)
    w3 = (torch.rand(8, 1, 3, 3, 3, device=DEV) - 0.5).requires_grad_(True)
    b3 = (torch.rand(8, device=DEV) - 0.5).requires_grad_(True)
    z = folded.pack_conv_folded(x, w2, b2, w3, b3, PF.conv2d)
    gz = torch.rand_like(z) - 0.5
    z.backward(gz)
    torch.cuda.synchronize()
    xd, w2d, b2d, w3d, b3d = (t.detach().double().cpu().requires_grad_(True) for t in (x, w2, b2, w3, b3))
    t = PO.conv3d_features(PO.packing(xd.permute(0, 3, 1, 2)), w3d, b3d)
    zr = F.conv2d(F.pad(t, [k // 2] * 4), w2d, b2d).permute(0, 2, 3, 1)
    zr.backward(gz.double().cpu())
    assert rel_l2(z.cpu(), zr) < 1e-4, rel_l2(z.cpu(), zr)
    # the frame must be as good as the interior (the strips are exact fp32)
    m = k // 2
    assert rel_l2(z[:, :m].cpu(), zr[:, :m]) < 1e-4 and rel_l2(z[:, :, -m:].cpu(), zr[:, :, -m:]) < 1e-4
    assert rel_l2(x.grad.cpu(), xd.grad) < 1e-4, rel_l2(x.grad.cpu(), xd.grad)
    assert rel_l2(w2.grad.cpu(), w2d.grad) < 1e-3, rel_l2(w2.grad.cpu(), w2d.grad)
    assert rel_l2(w3.grad.cpu(), w3d.grad) < 1e-3, rel_l2(w3.grad.cpu(), w3d.grad)
    assert rel_l2(b2.grad.cpu(), b2d.grad) < 1e-5 and rel_l2(b3.grad.cpu(), b3d.grad) < 1e-3


@pytest.mark.parametrize("case", [(2, 8, 12, 16, 8, 3), (1, 8, 14, 20, 16, 5), (3, 40, 8, 20, 24, 3)])
def test_fold_and_frame_kernels_with_a_pytorch_convolution(case):
    """pn_pack_fold_* and pn_pack_frame_* alone: the O(area) convolution is PyTorch's (fp32, TF32 off), so a failure here
    is in the fold / frame kernels and one only in test_folded_pack_conv_on_the_engine is in the engine's new shapes."""
    from packnet_sfm_b200 import folded
    B, C, H, W, Co, k = case
    torch.manual_seed(B + C + H + k)

    def conv(xs, w, b):
        with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
            return F.conv2d(xs.permute(0, 3, 1, 2), w, b, padding=w.shape[-1] // 2).permute(0, 2, 3, 1).contiguous()

    x = (torch.rand(B, H, W, C, device=DEV) - 0.5).requires_grad_(True)
    w2 = ((torch.rand(Co, 32 * C, k, k, device=DEV) - 0.5) * (2.0 / (32 * C * k * k) ** 0.5)).requires_grad_(True)
    b2 = (torch.rand(Co, device=DEV) - 0.5).requires_grad_(True)
    w3 = (torch.rand(8, 1, 3, 3, 3, device=DEV) - 0.5).requires_grad_(True)
    b3 = (torch.rand(8, device=DEV) - 0.5).requires_grad_(True)
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        z = folded.pack_conv_folded(x, w2, b2, w3, b3, conv)
        gz = torch.rand_like(z) - 0.5
        z.backward(gz)
    torch.cuda.synchronize()
    xd, w2d, b2d, w3d, b3d = (t.detach().double().cpu().requires_grad_(True) for t in (x, w2, b2, w3, b3))
    t = PO.conv3d_features(PO.packing(xd.permute(0, 3, 1, 2)), w3d, b3d)
    zr = F.conv2d(F.pad(t, [k // 2] * 4), w2d, b2d).permute(0, 2, 3, 1)
    zr.backward(gz.double().cpu())
    for name, a, b in (("z", z, zr), ("gx", x.grad, xd.grad), ("gw2", w2.grad, w2d.grad), ("gb2", b2.grad, b2d.grad),
                       ("gw3", w3.grad, w3d.grad), ("gb3", b3.grad, b3d.grad)):
        assert rel_l2(a.detach().cpu(), b.detach()) < 2e-5, (name, rel_l2(a.detach().cpu(), b.detach()))


BLOCKS = [("pack_k3", 32, 3, 21), ("pack_k5", 16, 5, 22)]


@pytest.mark.parametrize("tag,cin,k,seed", BLOCKS, ids=[b[0] for b in BLOCKS])
def test_folded_pack_block_matches_reference_golden(tag, cin, k, seed):
    from packnet_sfm_b200 import functional as PF, networks as N
    z = load_golden("blocks")
    mod = N.PackLayerConv3d(cin, k)
    mod.load_state_dict(PO.block_state_dict("pack", cin, k=k, seed=seed), strict=True)
    mod = mod.to(DEV)
    PF.set_pack_fold(True, min_pixels=0)
    try:
        x = nhwc(z[tag + "_x"].to(DEV)).requires_grad_(True)
        y = mod(x)
        y.backward(nhwc(z[tag + "_gy"].to(DEV)))
        torch.cuda.synchronize()
    finally:
        PF.set_pack_fold(True, min_pixels=1920)     # the default policy
    assert rel_l2(nchw(y).cpu(), z[tag + "_y"]) < 1e-4, rel_l2(nchw(y).cpu(), z[tag + "_y"])
    assert rel_l2(nchw(x.grad).cpu(), z[tag + "_gx"]) < 1e-3
    for name, p in mod.named_parameters():
        assert_golden_close(p.grad, z, tag + "_g_" + name, 1e-3, 5e-5)


def test_packnet01_with_folded_pack_layers_matches_reference_golden():
    from packnet_sfm_b200 import functional as PF
    from packnet_sfm_b200.networks import PackNet01
    z = load_golden("packnet01_64x96")
    net = PackNet01(version="1A")
    net.load_state_dict(PO.packnet01_state_dict(seed=42, randomize_affine=True), strict=True)
    net = net.to(DEV).train()
    PF.set_pack_fold(True, min_pixels=0)
    try:
        with torch.no_grad():
            out = net(z["rgb"].to(DEV))["inv_depths"]
    finally:
        PF.set_pack_fold(True, min_pixels=1920)     # the default policy
    for i, d in enumerate(out):
        ref = z["disp%d" % (i + 1)]
        rel = ((d.cpu() - ref).abs() / ref.abs()).max().item()
        print("folded disp%d max-rel %.3e" % (i + 1, rel))
        assert rel < 1e-3
