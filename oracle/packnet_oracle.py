"""CPU oracle: a plain-PyTorch (fp32, CPU) restatement of the reference hot path.

TEST INFRASTRUCTURE ONLY -- never imported by the product path (packnet_sfm_b200/).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may use it.

Every function cites the reference file:line it restates (paths relative to /root/reference).
The restatement is pinned two ways (SURVEY.md §8c -- the reference ships no tests or golden vectors):
  * tests/test_oracle_vs_reference.py holds it to the unmodified reference module's state-dict names,
    shapes and depth maps (stored by oracle/gen_golden.py), and
  * tests/golden/*.npz hold input/output vectors generated from the live reference by
    oracle/gen_golden.py; tests/test_oracle_golden.py checks the restatement against them everywhere.

State dict keys follow the reference module tree (PackNet01.py:25-104), so the same tensors drive the
reference module, this oracle and the CUDA path.
"""
import math

import torch
import torch.nn.functional as F


# ---------------------------------------------------------------------------------------------------
# optional TF32 emulation (used only for the precision study in DESIGN.md; default off = fp32 oracle)
# ---------------------------------------------------------------------------------------------------
def _tf32_trunc(x):
    """Drop the low 13 mantissa bits (what a tf32 tensor-core operand read keeps)."""
    return (x.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


def _tf32_rn(x):
    """Round-to-nearest-even to 10 explicit mantissa bits."""
    i = x.contiguous().view(torch.int32)
    lsb = (i >> 13) & 1
    i = i + 0xFFF + lsb
    return (i & ~0x1FFF).view(torch.float32)


class Precision:
    FP32 = "fp32"
    TF32_TRUNC = "tf32_trunc"
    TF32_RN = "tf32_rn"


def _q(x, precision):
    if precision == Precision.FP32:
        return x
    if precision == Precision.TF32_TRUNC:
        return _tf32_trunc(x)
    if precision == Precision.TF32_RN:
        return _tf32_rn(x)
    raise ValueError(precision)


def _conv2d(x, w, b, precision):
    return F.conv2d(_q(x, precision), _q(w, precision), b)


# ---------------------------------------------------------------------------------------------------
# layers (packnet_sfm/networks/layers/packnet/layers01.py)
# ---------------------------------------------------------------------------------------------------
def packing(x, r=2):
    """space-to-depth, layers01.py:126-148: out[b, c*4 + i*2 + j, h, w] = x[b, c, 2h+i, 2w+j]."""
    b, c, h, w = x.shape
    x = x.contiguous().view(b, c, h // r, r, w // r, r)
    return x.permute(0, 1, 3, 5, 2, 4).contiguous().view(b, c * r * r, h // r, w // r)


def conv2d_gn_elu(x, sd, prefix, k, precision=Precision.FP32):
    """Conv2D, layers01.py:10-37: zero-pad k//2 -> Conv2d -> GroupNorm(16, eps 1e-5) -> ELU."""
    w = sd[prefix + ".conv_base.weight"]
    b = sd[prefix + ".conv_base.bias"]
    x = _conv2d(F.pad(x, [k // 2] * 4), w, b, precision)
    x = F.group_norm(x, 16, sd[prefix + ".normalize.weight"], sd[prefix + ".normalize.bias"], 1e-5)
    return F.elu(x)


def residual_conv(x, sd, prefix, precision=Precision.FP32):
    """ResidualConv, layers01.py:40-72 (dropout=None): conv1(3x3) -> conv2(3x3) + 1x1 shortcut -> GN -> ELU."""
    y = conv2d_gn_elu(x, sd, prefix + ".conv1", 3, precision)
    y = conv2d_gn_elu(y, sd, prefix + ".conv2", 3, precision)
    s = _conv2d(x, sd[prefix + ".conv3.weight"], sd[prefix + ".conv3.bias"], precision)
    y = F.group_norm(y + s, 16, sd[prefix + ".normalize.weight"], sd[prefix + ".normalize.bias"], 1e-5)
    return F.elu(y)


def residual_block(x, sd, prefix, num_blocks, precision=Precision.FP32):
    """ResidualBlock, layers01.py:75-95."""
    for i in range(num_blocks):
        x = residual_conv(x, sd, "%s.%d" % (prefix, i), precision)
    return x


def inv_depth_head(x, sd, prefix, min_depth=0.5, precision=Precision.FP32):
    """InvDepth, layers01.py:98-122: pad 1 -> Conv2d(C->1, 3x3) -> sigmoid / min_depth."""
    y = _conv2d(F.pad(x, [1] * 4), sd[prefix + ".conv1.weight"], sd[prefix + ".conv1.bias"], precision)
    return torch.sigmoid(y) / min_depth


def conv3d_features(x, w3, b3):
    """The Conv3d(1->8, 3x3x3, pad 1) of the pack/unpack layers (layers01.py:236-237,243-246):
    [B,C,H,W] -> unsqueeze -> conv3d -> view [B, 8*C, H, W] with channel index f*C + c."""
    b, c, h, w = x.shape
    y = F.conv3d(x.unsqueeze(1), w3, b3, padding=1)
    return y.view(b, y.shape[1] * c, h, w)


def pack_layer(x, sd, prefix, k, precision=Precision.FP32):
    """PackLayerConv3d.forward, layers01.py:239-247."""
    x = packing(x)
    x = conv3d_features(x, sd[prefix + ".conv3d.weight"], sd[prefix + ".conv3d.bias"])
    return conv2d_gn_elu(x, sd, prefix + ".conv", k, precision)


def unpack_layer(x, sd, prefix, k=3, precision=Precision.FP32):
    """UnpackLayerConv3d.forward, layers01.py:278-286."""
    x = conv2d_gn_elu(x, sd, prefix + ".conv", k, precision)
    x = conv3d_features(x, sd[prefix + ".conv3d.weight"], sd[prefix + ".conv3d.bias"])
    return F.pixel_shuffle(x, 2)


# ---------------------------------------------------------------------------------------------------
# PackNet01 (packnet_sfm/networks/depth/PackNet01.py)
# ---------------------------------------------------------------------------------------------------
def packnet01_forward(rgb, sd, version="A", precision=Precision.FP32, return_features=False):
    """PackNet01.forward in train mode, PackNet01.py:106-185 -> [disp1, disp2, disp3, disp4]."""
    p = precision
    feats = {}
    x = conv2d_gn_elu(rgb, sd, "pre_calc", 5, p)
    x1 = conv2d_gn_elu(x, sd, "conv1", 7, p)
    x1p = pack_layer(x1, sd, "pack1", 5, p)
    x2 = residual_block(x1p, sd, "conv2", 2, p)
    x2p = pack_layer(x2, sd, "pack2", 3, p)
    x3 = residual_block(x2p, sd, "conv3", 2, p)
    x3p = pack_layer(x3, sd, "pack3", 3, p)
    x4 = residual_block(x3p, sd, "conv4", 3, p)
    x4p = pack_layer(x4, sd, "pack4", 3, p)
    x5 = residual_block(x4p, sd, "conv5", 3, p)
    x5p = pack_layer(x5, sd, "pack5", 3, p)
    skip1, skip2, skip3, skip4, skip5 = x, x1p, x2p, x3p, x4p
    cat = (lambda a, b: torch.cat((a, b), 1)) if version == "A" else (lambda a, b: a + b)

    unpack5 = unpack_layer(x5p, sd, "unpack5", 3, p)
    iconv5 = conv2d_gn_elu(cat(unpack5, skip5), sd, "iconv5", 3, p)

    unpack4 = unpack_layer(iconv5, sd, "unpack4", 3, p)
    iconv4 = conv2d_gn_elu(cat(unpack4, skip4), sd, "iconv4", 3, p)
    disp4 = inv_depth_head(iconv4, sd, "disp4_layer", precision=p)
    udisp4 = F.interpolate(disp4, scale_factor=2, mode="nearest")

    unpack3 = unpack_layer(iconv4, sd, "unpack3", 3, p)
    iconv3 = conv2d_gn_elu(torch.cat((cat(unpack3, skip3), udisp4), 1), sd, "iconv3", 3, p)
    disp3 = inv_depth_head(iconv3, sd, "disp3_layer", precision=p)
    udisp3 = F.interpolate(disp3, scale_factor=2, mode="nearest")

    unpack2 = unpack_layer(iconv3, sd, "unpack2", 3, p)
    iconv2 = conv2d_gn_elu(torch.cat((cat(unpack2, skip2), udisp3), 1), sd, "iconv2", 3, p)
    disp2 = inv_depth_head(iconv2, sd, "disp2_layer", precision=p)
    udisp2 = F.interpolate(disp2, scale_factor=2, mode="nearest")

    unpack1 = unpack_layer(iconv2, sd, "unpack1", 3, p)
    iconv1 = conv2d_gn_elu(torch.cat((cat(unpack1, skip1), udisp2), 1), sd, "iconv1", 3, p)
    disp1 = inv_depth_head(iconv1, sd, "disp1_layer", precision=p)
    if return_features:
        feats.update(x=x, x1=x1, x1p=x1p, x2=x2, x2p=x2p, x5p=x5p, unpack5=unpack5, iconv5=iconv5,
                     iconv1=iconv1)
        return [disp1, disp2, disp3, disp4], feats
    return [disp1, disp2, disp3, disp4]


def packnet01_state_dict(seed=42, version="A", randomize_affine=False):
    """Random PackNet01 weights with the reference's shapes, names and init distribution
    (Xavier-uniform conv weights, zero conv biases, GroupNorm affine = (1, 0); PackNet01.py:98-104).
    Not bit-identical to the reference's RNG stream -- tests that need identical weights pass the
    reference module's own state_dict instead.  randomize_affine=True additionally perturbs every
    bias and GroupNorm affine parameter (a trained-like state; zero biases would hide bias bugs)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}

    def conv(name, cout, cin, *ks):
        fan_in = cin * math.prod(ks)
        fan_out = cout * math.prod(ks)
        bound = math.sqrt(6.0 / (fan_in + fan_out))
        sd[name + ".weight"] = (torch.rand(cout, cin, *ks, generator=g) * 2 - 1) * bound
        sd[name + ".bias"] = torch.zeros(cout)

    def gn(name, c):
        sd[name + ".weight"] = torch.ones(c)
        sd[name + ".bias"] = torch.zeros(c)

    def conv2d_block(name, cin, cout, k):
        conv(name + ".conv_base", cout, cin, k, k)
        gn(name + ".normalize", cout)

    def res_block(name, cin, cout, n):
        for i in range(n):
            ci = cin if i == 0 else cout
            conv2d_block("%s.%d.conv1" % (name, i), ci, cout, 3)
            conv2d_block("%s.%d.conv2" % (name, i), cout, cout, 3)
            conv("%s.%d.conv3" % (name, i), cout, ci, 1, 1)
            gn("%s.%d.normalize" % (name, i), cout)

    ni, no = 64, 1
    n1, n2, n3, n4, n5 = 64, 64, 128, 256, 512
    if version == "A":
        n1o, n1i = n1, n1 + ni + no
        n2o, n2i = n2, n2 + n1 + no
        n3o, n3i = n3, n3 + n2 + no
        n4o, n4i = n4, n4 + n3
        n5o, n5i = n5, n5 + n4
    else:
        n1o, n1i = n1, n1 + no
        n2o, n2i = n2, n2 + no
        n3o, n3i = n3 // 2, n3 // 2 + no
        n4o, n4i = n4 // 2, n4 // 2
        n5o, n5i = n5 // 2, n5 // 2
    conv2d_block("pre_calc", 3, ni, 5)
    for name, c, k in (("pack1", n1, 5), ("pack2", n2, 3), ("pack3", n3, 3), ("pack4", n4, 3), ("pack5", n5, 3)):
        conv2d_block(name + ".conv", c * 32, c, k)
        conv(name + ".conv3d", 8, 1, 3, 3, 3)
    conv2d_block("conv1", ni, n1, 7)
    res_block("conv2", n1, n2, 2)
    res_block("conv3", n2, n3, 2)
    res_block("conv4", n3, n4, 3)
    res_block("conv5", n4, n5, 3)
    for name, cin, cout in (("unpack5", n5, n5o), ("unpack4", n5, n4o), ("unpack3", n4, n3o),
                            ("unpack2", n3, n2o), ("unpack1", n2, n1o)):
        conv2d_block(name + ".conv", cin, cout * 4 // 8, 3)
        conv(name + ".conv3d", 8, 1, 3, 3, 3)
    for name, cin, cout in (("iconv5", n5i, n5), ("iconv4", n4i, n4), ("iconv3", n3i, n3),
                            ("iconv2", n2i, n2), ("iconv1", n1i, n1)):
        conv2d_block(name, cin, cout, 3)
    for name, c in (("disp4_layer", n4), ("disp3_layer", n3), ("disp2_layer", n2), ("disp1_layer", n1)):
        conv(name + ".conv1", 1, c, 3, 3)
    if randomize_affine:
        randomize_affine_(sd, g)
    return sd


def randomize_affine_(sd, g):
    """In place: biases ~ U(-0.1, 0.1); GroupNorm weight ~ U(0.5, 1.5), GroupNorm bias ~ U(-0.2, 0.2)."""
    for k in sorted(sd):
        if k.endswith(".normalize.weight"):
            sd[k] = 0.5 + torch.rand(sd[k].shape, generator=g)
        elif k.endswith(".normalize.bias"):
            sd[k] = (torch.rand(sd[k].shape, generator=g) * 2 - 1) * 0.2
        elif k.endswith(".bias"):
            sd[k] = (torch.rand(sd[k].shape, generator=g) * 2 - 1) * 0.1
    return sd


def block_state_dict(kind, cin, cout=None, k=3, seed=7):
    """Seeded weights for ONE pack / unpack / conv2d / residual block with the reference's key names
    (prefix-free), non-zero biases and non-trivial GroupNorm affine.
      kind='pack'   : PackLayerConv3d(cin, k)            layers01.py:213-237
      kind='unpack' : UnpackLayerConv3d(cin, cout, k)    layers01.py:250-276
      kind='conv2d' : Conv2D(cin, cout, k, 1)            layers01.py:10-32
      kind='residual': ResidualConv(cin, cout, 1)        layers01.py:40-65"""
    g = torch.Generator().manual_seed(seed)
    sd = {}

    def conv(name, co, ci, *ks):
        bound = math.sqrt(6.0 / ((ci + co) * math.prod(ks)))
        sd[name + ".weight"] = (torch.rand(co, ci, *ks, generator=g) * 2 - 1) * bound
        sd[name + ".bias"] = torch.zeros(co)

    def gn(name, c):
        sd[name + ".weight"] = torch.ones(c)
        sd[name + ".bias"] = torch.zeros(c)

    if kind == "pack":
        conv("conv.conv_base", cin, cin * 32, k, k)
        gn("conv.normalize", cin)
        conv("conv3d", 8, 1, 3, 3, 3)
    elif kind == "unpack":
        conv("conv.conv_base", cout * 4 // 8, cin, k, k)
        gn("conv.normalize", cout * 4 // 8)
        conv("conv3d", 8, 1, 3, 3, 3)
    elif kind == "conv2d":
        conv("conv_base", cout, cin, k, k)
        gn("normalize", cout)
    elif kind == "residual":
        for nm, ci in (("conv1", cin), ("conv2", cout)):
            conv(nm + ".conv_base", cout, ci, 3, 3)
            gn(nm + ".normalize", cout)
        conv("conv3", cout, cin, 1, 1)
        gn("normalize", cout)
    else:
        raise ValueError(kind)
    return randomize_affine_(sd, g)
