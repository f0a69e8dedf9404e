"""The drop-in registration (packnet_sfm_b200/dropin.py) and the self-supervised forward built from the drop-in classes,
against what the unmodified reference's own SelfSupModel computed (oracle/gen_golden.py: selfsup_flip_case)."""
import importlib
import importlib.util
import sys

from conftest import load_golden


def _purge(prefixes):
    for name in list(sys.modules):
        if any(name == p or name.startswith(p + ".") for p in prefixes):
            del sys.modules[name]


def test_reference_models_pick_up_the_dropin_classes():
    """The reference resolves its networks by module path + class name through importlib (packnet_sfm/utils/load.py
    load_class: find_spec, import_module, getattr) and hard-imports the loss (SelfSupModel.py:4).  After dropin.install()
    both resolve to this package's classes."""
    from packnet_sfm_b200 import dropin, losses, networks
    dropin.install()
    try:
        path = "packnet_sfm.networks.depth.PackNet01"
        assert importlib.util.find_spec(path) is not None
        cls = getattr(importlib.import_module(path), "PackNet01")
        assert cls is networks.PackNet01
        from packnet_sfm.losses.multiview_photometric_loss import MultiViewPhotometricLoss
        assert MultiViewPhotometricLoss is losses.MultiViewPhotometricLoss
        layers = importlib.import_module("packnet_sfm.networks.layers.packnet.layers01")
        for name in ("Conv2D", "ResidualConv", "ResidualBlock", "InvDepth", "PackLayerConv3d", "UnpackLayerConv3d"):
            assert getattr(layers, name) is getattr(networks, name)
        net = cls(version="1A", dropout=0.0)
        assert len(net.state_dict()) == 216
    finally:
        _purge(["packnet_sfm"])


def test_selfsup_forward_with_dropin_classes_matches_reference_golden(emulated_kernels, monkeypatch):
    """The reference's own SelfSupModel.forward (flip forced, maps upsampled) with its PackNet01, PoseNet and loss produced the
    fixture.  Here the same weights and batch run through this package's SelfSupModel glue with PackNet01 and
    MultiViewPhotometricLoss, the classes the drop-in registers -- their SIMT kernels (feature stencils, GroupNorm+ELU, head
    convolution, fused loss) execute from their real source under the host emulation; only the tcgen05 convolution is stood
    in by PyTorch's fp32 conv2d.  Same loss, same metrics, same depth maps."""
    import torch
    import torch.nn.functional as F
    from oracle import packnet_oracle as PO
    from oracle.step_oracle import posenet_state_dict
    from packnet_sfm_b200 import functional as PF, models, networks
    z = load_golden("selfsup_flip_1x32x64")
    batch = {"rgb": z["rgb"], "rgb_context": [z["ctx0"], z["ctx1"]], "rgb_original": z["rgb"],
             "rgb_context_original": [z["ctx0"], z["ctx1"]], "intrinsics": z["K"]}

    def conv2d(x, w, b=None):       # stand-in for the tensor-core engine (NHWC, zero pad k//2, weight padded to the activation)
        if w.shape[1] != x.shape[3]:
            w = torch.cat([w, torch.zeros(w.shape[0], x.shape[3] - w.shape[1], w.shape[2], w.shape[3])], 1)
        return F.conv2d(x.permute(0, 3, 1, 2), w, b, padding=w.shape[-1] // 2).permute(0, 2, 3, 1).contiguous()

    monkeypatch.setattr(PF, "conv2d", conv2d)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", torch.backends.cudnn.allow_tf32)   # SelfSupModel sets it
    depth = networks.PackNet01(version="1A")
    depth.load_state_dict(PO.packnet01_state_dict(seed=42, randomize_affine=True), strict=True)
    pose = models.PoseNet(nb_ref_imgs=2, rotation_mode="euler")
    pose.load_state_dict(posenet_state_dict(43), strict=True)
    model = models.SelfSupModel(depth_net=depth, pose_net=pose, num_scales=4, ssim_loss_weight=0.85, smooth_loss_weight=0.001,
                                photometric_reduce_op="min", clip_loss=0.0, automask_loss=True, rotation_mode="euler",
                                flip_lr_prob=1.0, upsample_depth_maps=True, fuse_upsample=False).train()
    with torch.no_grad():
        out = model(batch)
    want, got = float(z["loss"]), float(out["loss"])
    assert abs(got - want) <= 1e-5 * abs(want), (got, want)
    for key in ("photometric_loss", "smoothness_loss"):
        assert abs(float(out["metrics"][key]) - float(z[key])) <= 1e-4 * abs(float(z[key])) + 1e-9
    for i, a in enumerate(out["inv_depths"]):
        b = z["inv%d" % i]
        assert a.shape == b.shape and float(((a - b).abs() / b.abs()).max()) < 1e-4
