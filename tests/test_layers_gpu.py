"""GPU parity tests of the layer kernels through the C-ABI: tcgen05 convolution (forward, data gradient,
weight gradient), Conv3d feature stencils, GroupNorm+ELU, and the assembled pack / unpack / Conv2D /
ResidualConv blocks against the golden vectors generated from the live reference."""
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


def _trunc(x):
    return (x.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


CONV_CASES = [
    # B, H, W, Cin, Cout, k
    (1, 16, 8, 32, 16, 1),
    (2, 40, 36, 64, 48, 3),
    (1, 32, 24, 96, 64, 5),
    (4, 6, 20, 64, 128, 3),      # batch-folded small map (pack5-like)
    (1, 16, 16, 40, 32, 3),      # ragged K (Cin not a multiple of the 32/64-channel chunk)
    (1, 16, 16, 64, 512, 3),     # several N tiles
    (1, 32, 24, 64, 64, 7),
    (2, 96, 160, 64, 64, 3),     # 240 work items: persistent tile loop, two accumulator sets in TMEM
    (2, 64, 96, 32, 256, 3),     # 192 work items over 2 N blocks of 128: persistent, one accumulator set
]


@pytest.mark.parametrize("case", CONV_CASES)
@pytest.mark.parametrize("precision", [1, 3, 4])
def test_conv2d_forward_backward(case, precision):
    from packnet_sfm_b200 import functional as PF
    B, H, W, Cin, Cout, k = case
    torch.manual_seed(B * 1000 + H + Cin + k)
    PF.set_precision(precision)
    try:
        x = (torch.rand(B, H, W, Cin, device=DEV) - 0.5).requires_grad_(True)
        w = ((torch.rand(Cout, Cin, k, k, device=DEV) - 0.5) * (2.0 / (Cin * k * k) ** 0.5)).requires_grad_(True)
        b = (torch.rand(Cout, device=DEV) - 0.5).requires_grad_(True)
        gy = torch.rand(B, H, W, Cout, device=DEV) - 0.5
        y = PF.conv2d(x, w, b)
        y.backward(gy)
        torch.cuda.synchronize()
        xd, wd, bd = (t.detach().double().requires_grad_(True) for t in (x, w, b))
        yr = F.conv2d(xd.permute(0, 3, 1, 2), wd, bd, padding=k // 2).permute(0, 2, 3, 1)
        yr.backward(gy.double())
        # tf32x3: the TMEM accumulator adds with truncation, the error grows ~3e-9 per accumulated K element
        # (measured, profiles/r01_conv_probe.txt); tf32x1: 2^-11 operand truncation
        # bf16x3: 16 mantissa bits kept per operand -> ~1e-5 per product, random accumulation
        kred = Cin * k * k
        tol = {1: 3e-3, 3: 1e-5 + 1e-8 * max(kred, B * H * W), 4: 6e-5 + 1e-8 * max(kred, B * H * W)}[precision]
        assert rel_l2(y, yr) < tol, ("y", rel_l2(y, yr))
        assert rel_l2(x.grad, xd.grad) < tol, ("gx", rel_l2(x.grad, xd.grad))
        assert rel_l2(w.grad, wd.grad) < tol, ("gw", rel_l2(w.grad, wd.grad))
        assert rel_l2(b.grad, bd.grad) < 1e-5
        if precision == 1:
            # tf32x1 is exactly "fp32 accumulate of tf32-truncated operands"
            ye = F.conv2d(_trunc(x.detach()).permute(0, 3, 1, 2).double(), _trunc(w.detach()).double(), b.detach().double(),
                          padding=k // 2).permute(0, 2, 3, 1)
            assert rel_l2(y, ye) < 2e-5
    finally:
        PF.set_precision(PF.PRECISION_BF16X3)


@pytest.mark.parametrize("mode", [1, 2])
def test_conv2d_staging_modes_agree(mode):
    """PER_TAP (reload per tap) and HALO (patch reuse through shifted descriptors) give the same numbers."""
    import conv_helpers as ops
    torch.manual_seed(5)
    x = torch.rand(2, 48, 40, 64, device=DEV) - 0.5
    w = (torch.rand(64, 64, 5, 5, device=DEV) - 0.5) * 0.05
    for prec, tol in ((ops.PRECISION_TF32X3, 3e-5), (ops.PRECISION_BF16X3, 8e-5)):
        y = ops.conv2d_nhwc(x, w, None, prec, mode)
        yr = F.conv2d(x.permute(0, 3, 1, 2).double(), w.double(), padding=2).permute(0, 2, 3, 1)
        assert rel_l2(y, yr) < tol, (prec, rel_l2(y, yr))


def test_feature_stencils_and_groupnorm():
    from packnet_sfm_b200 import functional as PF
    torch.manual_seed(3)
    shapes = ((True, (2, 16, 24, 32)), (False, (2, 6, 20, 32)), (True, (1, 12, 8, 512)),
              (True, (1, 10, 14, 8)),       # odd low-res height, ragged width (masked rows / columns)
              (False, (1, 5, 7, 24)), (False, (2, 9, 33, 128)), (True, (2, 4, 4, 64)),
              (True, (1, 8, 8, 5)))         # depth 20 is not a multiple of 8: generic kernels
    for pack, shape in shapes:
        x = (torch.rand(*shape, device=DEV) - 0.5).requires_grad_(True)
        w3 = ((torch.rand(8, 1, 3, 3, 3, device=DEV) - 0.5)).requires_grad_(True)
        b3 = (torch.rand(8, device=DEV) - 0.5).requires_grad_(True)
        y = PF.pack_features(x, w3, b3) if pack else PF.unpack_features(x, w3, b3)
        gy = torch.rand_like(y) - 0.5
        y.backward(gy)
        xd, wd, bd = (t.detach().double().requires_grad_(True) for t in (x, w3, b3))
        xn = xd.permute(0, 3, 1, 2)
        if pack:
            yr = PO.conv3d_features(PO.packing(xn), wd, bd).permute(0, 2, 3, 1)
        else:
            yr = F.pixel_shuffle(PO.conv3d_features(xn, wd, bd), 2).permute(0, 2, 3, 1)
        yr.backward(gy.double())
        assert rel_l2(y, yr) < 1e-6
        assert rel_l2(x.grad, xd.grad) < 1e-5
        assert rel_l2(w3.grad, wd.grad) < 1e-4
        assert rel_l2(b3.grad, bd.grad) < 1e-4
    for C in (16, 64, 512):
        x = (torch.rand(2, 12, 20, C, device=DEV) * 2 - 0.7).requires_grad_(True)
        x2 = (torch.rand(2, 12, 20, C, device=DEV) - 0.5).requires_grad_(True)
        g = (torch.rand(C, device=DEV) + 0.5).requires_grad_(True)
        bt = (torch.rand(C, device=DEV) - 0.5).requires_grad_(True)
        for second in (None, x2):
            for t in (x, x2, g, bt):
                t.grad = None
            y = PF.groupnorm_elu(x, g, bt, 1e-5, x2=second)
            gy = torch.rand_like(y) - 0.5
            y.backward(gy)
            xd, x2d, gd, bd = (t.detach().double().requires_grad_(True) for t in (x, x2, g, bt))
            inp = xd if second is None else xd + x2d
            yr = F.elu(F.group_norm(inp.permute(0, 3, 1, 2), 16, gd, bd, 1e-5)).permute(0, 2, 3, 1)
            yr.backward(gy.double())
            assert rel_l2(y, yr) < 1e-6
            assert rel_l2(x.grad, xd.grad) < 1e-5
            assert rel_l2(g.grad, gd.grad) < 1e-5 and rel_l2(bt.grad, bd.grad) < 1e-5
            if second is not None:
                assert rel_l2(x2.grad, x2d.grad) < 1e-5


def _load_block(module, sd):
    module.load_state_dict(sd, strict=True)
    return module.to(DEV)


def test_head_conv_matches_fp64_conv2d():
    """Conv2d(C->1, 3x3, pad 1) of InvDepth (layers01.py:110-116): exact-fp32 kernel vs float64 F.conv2d."""
    from packnet_sfm_b200 import functional as PF
    torch.manual_seed(11)
    for B, H, W, C in ((2, 24, 40, 64), (1, 9, 13, 128), (1, 6, 20, 256), (1, 16, 8, 4)):
        x = (torch.rand(B, H, W, C, device=DEV) - 0.5).requires_grad_(True)
        w = ((torch.rand(1, C, 3, 3, device=DEV) - 0.5) * 0.2).requires_grad_(True)
        b = (torch.rand(1, device=DEV) - 0.5).requires_grad_(True)
        y = PF.head_conv(x, w, b)
        gy = torch.rand_like(y) - 0.5
        y.backward(gy)
        xd, wd, bd = (t.detach().double().requires_grad_(True) for t in (x, w, b))
        yr = F.conv2d(xd.permute(0, 3, 1, 2), wd, bd, padding=1)[:, 0]
        yr.backward(gy.double())
        assert rel_l2(y, yr) < 1e-6
        assert rel_l2(x.grad, xd.grad) < 1e-6
        assert rel_l2(w.grad, wd.grad) < 1e-5
        assert rel_l2(b.grad, bd.grad) < 1e-5


BLOCKS = [
    ("pack_k3", lambda N: N.PackLayerConv3d(32, 3), lambda: PO.block_state_dict("pack", 32, k=3, seed=21)),
    ("pack_k5", lambda N: N.PackLayerConv3d(16, 5), lambda: PO.block_state_dict("pack", 16, k=5, seed=22)),
    ("unpack", lambda N: N.UnpackLayerConv3d(64, 32, 3), lambda: PO.block_state_dict("unpack", 64, 32, 3, seed=23)),
    ("conv2d_k7", lambda N: N.Conv2D(32, 32, 7, 1), lambda: PO.block_state_dict("conv2d", 32, 32, 7, seed=24)),
    ("residual", lambda N: N.ResidualConv(32, 64, 1), lambda: PO.block_state_dict("residual", 32, 64, seed=25)),
]


@pytest.mark.parametrize("tag,make,sd", BLOCKS, ids=[b[0] for b in BLOCKS])
def test_blocks_match_reference_golden(tag, make, sd):
    """Same class names, parameters and outputs as the reference layers (golden from the live reference)."""
    from packnet_sfm_b200 import networks as N
    z = load_golden("blocks")
    mod = _load_block(make(N), sd())
    x = nhwc(z[tag + "_x"].to(DEV)).requires_grad_(True)
    y = mod(x)
    y.backward(nhwc(z[tag + "_gy"].to(DEV)))
    torch.cuda.synchronize()
    assert rel_l2(nchw(y).cpu(), z[tag + "_y"]) < 1e-4, rel_l2(nchw(y).cpu(), z[tag + "_y"])
    assert rel_l2(nchw(x.grad).cpu(), z[tag + "_gx"]) < 1e-3
    for k, p in mod.named_parameters():
        assert_golden_close(p.grad, z, tag + "_g_" + k, 1e-3, 5e-5)
