"""Generate tests/golden/*.npz from the LIVE, UNMODIFIED reference (build container only).

TEST INFRASTRUCTURE ONLY.  Run:  python oracle/gen_golden.py
/root/reference cannot travel to the GPU box, so the vectors it produces are committed as small
fixtures together with this script (the reference has no golden vectors of its own, SURVEY.md §0.2).

Every output array comes from reference classes:
  packnet_sfm.losses.multiview_photometric_loss.MultiViewPhotometricLoss  (+ autograd for the gradients)
  packnet_sfm.geometry.camera.Camera.reconstruct / project                 (normalised warp coordinates)
  packnet_sfm.networks.layers.packnet.layers01.{PackLayerConv3d,UnpackLayerConv3d,Conv2D,ResidualConv}
  packnet_sfm.networks.depth.PackNet01.PackNet01
Inputs and weights are regenerated from seeds (packnet_sfm_b200/synthetic.py, oracle/packnet_oracle.py);
the inputs are stored too (the block inputs as their seed and shape, the large ones as a checksum) so an RNG
change cannot silently invalidate a fixture.  No fixture file exceeds 1 MB: large gradients are stored as a
seeded sample plus their norm, the larger depth maps of the full-size cases at a pixel stride.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shims  # noqa: E402

ref_shims.install()
from oracle import packnet_oracle as PO  # noqa: E402
from packnet_sfm_b200 import synthetic  # noqa: E402
from oracle.loss_oracle import pose_from_vec, upsample_output  # noqa: E402

from packnet_sfm.losses.multiview_photometric_loss import MultiViewPhotometricLoss  # noqa: E402
from packnet_sfm.geometry.camera import Camera  # noqa: E402
from packnet_sfm.geometry.pose import Pose  # noqa: E402
from packnet_sfm.networks.layers.packnet import layers01 as L  # noqa: E402
from packnet_sfm.networks.depth.PackNet01 import PackNet01  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
YACS_LOSS_DEFAULTS = dict(num_scales=4, ssim_loss_weight=0.85, occ_reg_weight=0.1, smooth_loss_weight=0.001,
                          C1=1e-4, C2=9e-4, photometric_reduce_op="min", disp_norm=True, clip_loss=0.0,
                          progressive_scaling=0.0, padding_mode="zeros", automask_loss=True)


def loss_case(name, B, H, W, full_res, **overrides):
    frames = synthetic.make_frames(B, H, W, seed=11)
    inv = synthetic.make_inv_depths(B, H, W, seed=12, full_res=full_res)
    vec = synthetic.make_pose_vecs(B, seed=13)
    if overrides.pop("big_motion", False):
        vec = vec * 8.0  # push many samples out of bounds / behind the camera
    inv = [d.clone().requires_grad_(True) for d in inv]
    mats = [pose_from_vec(vec[:, j]).clone().requires_grad_(True) for j in range(vec.shape[1])]
    poses = [Pose(m) for m in mats]
    kw = dict(YACS_LOSS_DEFAULTS)
    kw.update(overrides)
    loss_fn = MultiViewPhotometricLoss(**kw)
    K = frames["intrinsics"]
    out = loss_fn(frames["rgb"], frames["rgb_context"], inv, K, K, poses)
    out["loss"].backward()
    arrays = {
        "rgb": frames["rgb"], "ctx0": frames["rgb_context"][0], "ctx1": frames["rgb_context"][1],
        "K": K, "loss": out["loss"].detach(),
        "photometric_loss": out["metrics"]["photometric_loss"], "smoothness_loss": out["metrics"]["smoothness_loss"],
    }
    for i, d in enumerate(inv):
        arrays["inv%d" % i] = d.detach()
        arrays["ginv%d" % i] = d.grad
    for j, m in enumerate(mats):
        arrays["pose%d" % j] = m.detach()
        arrays["gpose%d" % j] = m.grad
    # normalised warp coordinates straight from the reference camera classes (scale 0)
    with torch.no_grad():
        for j in range(2):
            cam = Camera(K=K.float())
            ref_cam = Camera(K=K.float(), Tcw=Pose(mats[j].detach()))
            depth = 1.0 / inv[0].detach().clamp(min=1e-6)
            arrays["grid%d" % j] = ref_cam.project(cam.reconstruct(depth, frame="w"), frame="w")
    meta = {k: v for k, v in kw.items()}
    np.savez_compressed(os.path.join(OUT, name + ".npz"), meta=np.array(repr(meta)),
                        **{k: np.asarray(v.detach().numpy() if torch.is_tensor(v) else v) for k, v in arrays.items()})
    print(name, float(out["loss"]))


def _load(module, sd):
    missing = module.load_state_dict(sd, strict=True)
    return module


def seeded_input(arrays, key, shape, seed):
    """A uniform(-0.5, 0.5) input, stored as its seed and shape (tests/conftest.py:load_golden regenerates it)."""
    arrays[key + "/seed"] = np.int64(seed)
    arrays[key + "/shape"] = np.array(shape, dtype=np.int64)
    return torch.rand(shape, generator=torch.Generator().manual_seed(seed)) - 0.5


def store_sampled(arrays, key, t, n=4096, seed=0):
    """A tensor of more than 8n elements is stored as n seeded random elements (`key/idx` flat positions, `key/samp`) and
    the whole tensor's float64 norm (`key/norm`); keeps every fixture file under 1 MB."""
    flat = t.detach().reshape(-1)
    if flat.numel() <= 8 * n:
        arrays[key] = t.detach()
        return
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:n].sort().values
    arrays[key + "/idx"] = idx.to(torch.int32)
    arrays[key + "/samp"] = flat[idx]
    arrays[key + "/norm"] = np.float64(flat.double().norm().item())


def block_cases():
    arrays = {}

    def run(i, tag, module, sd, shape):
        _load(module, sd)
        x = seeded_input(arrays, tag + "_x", shape, 50 + 2 * i).requires_grad_(True)
        y = module(x)
        gy = seeded_input(arrays, tag + "_gy", tuple(y.shape), 51 + 2 * i)
        y.backward(gy)
        arrays[tag + "_y"] = y.detach()
        arrays[tag + "_gx"] = x.grad
        for k, p in module.named_parameters():
            store_sampled(arrays, tag + "_g_" + k, p.grad, seed=i)

    run(0, "pack_k3", L.PackLayerConv3d(32, 3), PO.block_state_dict("pack", 32, k=3, seed=21), (2, 32, 16, 24))
    run(1, "pack_k5", L.PackLayerConv3d(16, 5), PO.block_state_dict("pack", 16, k=5, seed=22), (1, 16, 12, 40))
    run(2, "unpack", L.UnpackLayerConv3d(64, 32, 3), PO.block_state_dict("unpack", 64, 32, 3, seed=23), (2, 64, 6, 20))
    run(3, "conv2d_k7", L.Conv2D(32, 32, 7, 1), PO.block_state_dict("conv2d", 32, 32, 7, seed=24), (1, 32, 12, 20))
    run(4, "residual", L.ResidualConv(32, 64, 1), PO.block_state_dict("residual", 32, 64, seed=25), (2, 32, 8, 12))
    np.savez_compressed(os.path.join(OUT, "blocks.npz"),
                        **{k: v.numpy() if torch.is_tensor(v) else v for k, v in arrays.items()})
    print("blocks", len(arrays))


def restatement_case():
    """The reference's PackNet01 as a module: its state-dict names and shapes, and its depth maps for the oracle's default
    weights (Xavier-uniform convolutions, zero biases, GroupNorm affine (1, 0))."""
    net = PackNet01(version="1A").train()
    arrays = {"keys": np.array(list(net.state_dict()))}
    for k, v in net.state_dict().items():
        arrays["shape/" + k] = np.array(v.shape, dtype=np.int64)
    _load(net, PO.packnet01_state_dict())
    x = synthetic.make_frames(1, 64, 96, seed=3)["rgb"]
    with torch.no_grad():
        out = net(x)["inv_depths"]
    arrays["rgb"] = x.numpy()
    for i, d in enumerate(out):
        arrays["disp%d" % (i + 1)] = d.numpy()
    np.savez_compressed(os.path.join(OUT, "packnet01_restatement_64x96.npz"), **arrays)
    print("packnet01_restatement", len(arrays["keys"]), float(out[0].mean()))


def loss_restatement_case():
    """The reference's MultiViewPhotometricLoss with the training defaults on four full-resolution maps."""
    B, H, W = 2, 24, 48
    fr = synthetic.make_frames(B, H, W, seed=5)
    inv = synthetic.make_inv_depths(B, H, W, seed=6)
    mats = [pose_from_vec(synthetic.make_pose_vecs(B, seed=7)[:, j]) for j in range(2)]
    loss_fn = MultiViewPhotometricLoss(num_scales=4, ssim_loss_weight=0.85, smooth_loss_weight=0.001,
                                       photometric_reduce_op="min", clip_loss=0.0, automask_loss=True)
    K = fr["intrinsics"]
    out = loss_fn(fr["rgb"], fr["rgb_context"], inv, K, K, [Pose(m.clone()) for m in mats])
    arrays = {"rgb": fr["rgb"], "ctx0": fr["rgb_context"][0], "ctx1": fr["rgb_context"][1], "K": K,
              "loss": out["loss"]}
    arrays.update({"inv%d" % i: d for i, d in enumerate(inv)})
    arrays.update({"pose%d" % j: m for j, m in enumerate(mats)})
    np.savez_compressed(os.path.join(OUT, "loss_restatement_2x24x48.npz"), **{k: v.detach().numpy() for k, v in arrays.items()})
    print("loss_restatement", float(out["loss"]))


def selfsup_flip_case():
    """The reference's own SelfSupModel.forward (left-right flip forced, maps upsampled) with its PackNet01, PoseNet and
    loss: loss, metrics and the four depth maps of one training-mode forward."""
    from oracle.step_oracle import posenet_state_dict
    from packnet_sfm.models.SelfSupModel import SelfSupModel
    from packnet_sfm.networks.pose.PoseNet import PoseNet
    H, W = 32, 64
    fr = synthetic.make_frames(1, H, W, seed=3)
    batch = {"rgb": fr["rgb"], "rgb_context": fr["rgb_context"], "rgb_original": fr["rgb"],
             "rgb_context_original": fr["rgb_context"], "intrinsics": fr["intrinsics"]}
    depth = _load(PackNet01(version="1A"), PO.packnet01_state_dict(seed=42, randomize_affine=True))
    pose = _load(PoseNet(nb_ref_imgs=2, rotation_mode="euler"), posenet_state_dict(43))
    model = SelfSupModel(depth_net=depth, pose_net=pose, num_scales=4, ssim_loss_weight=0.85, smooth_loss_weight=0.001,
                         photometric_reduce_op="min", clip_loss=0.0, automask_loss=True, rotation_mode="euler",
                         flip_lr_prob=1.0, upsample_depth_maps=True).train()
    with torch.no_grad():
        out = model(batch)
    arrays = {"rgb": fr["rgb"], "ctx0": fr["rgb_context"][0], "ctx1": fr["rgb_context"][1], "K": fr["intrinsics"],
              "loss": out["loss"], "photometric_loss": out["metrics"]["photometric_loss"],
              "smoothness_loss": out["metrics"]["smoothness_loss"]}
    arrays.update({"inv%d" % i: d for i, d in enumerate(out["inv_depths"])})
    np.savez_compressed(os.path.join(OUT, "selfsup_flip_1x32x64.npz"), **{k: v.numpy() for k, v in arrays.items()})
    print("selfsup_flip", float(out["loss"]))


def packnet_case():
    sd = PO.packnet01_state_dict(seed=42, randomize_affine=True)
    net = PackNet01(version="1A")
    _load(net, sd)
    net.train()
    x = synthetic.make_frames(1, 64, 96, seed=31)["rgb"]
    with torch.no_grad():
        out = net(x)["inv_depths"]
    arrays = {"rgb": x.numpy()}
    for i, d in enumerate(out):
        arrays["disp%d" % (i + 1)] = d.numpy()
    np.savez_compressed(os.path.join(OUT, "packnet01_64x96.npz"), **arrays)
    print("packnet01", [tuple(d.shape) for d in out], float(out[0].mean()))


def strided_index(numel, n):
    """n evenly spaced flat indices (integer arithmetic: the tests rebuild exactly the same ones)."""
    n = min(n, numel)
    return (torch.arange(n, dtype=torch.int64) * (numel - 1)) // max(n - 1, 1)


def _grad_samples(named_grads, arrays, prefix, n=64):
    """Per parameter: float64 L2 norm and `n` evenly strided elements of the flattened gradient (keeps a 128 M-parameter
    gradient in a fixture of a few hundred KB while still touching every tensor)."""
    for k, g in named_grads:
        flat = g.detach().reshape(-1)
        idx = strided_index(flat.numel(), n)
        arrays[prefix + "norm/" + k] = np.float64(flat.double().norm().item())
        arrays[prefix + "samp/" + k] = flat[idx].numpy()


def packnet_baseline_case(B=4, H=192, W=640, name="packnet01_192x640_b4", strides=(2, 2, 1, 1)):
    """PackNet01 at BASELINE configs[1] (B=4, 192x640): the engine paths that the 64x96 fixture cannot reach (persistent
    tile loop, batch folding, split-K thresholds).  Depth maps (fp32; map i at every strides[i]-th pixel), the gradient of sum_i <disp_i, gy_i> for a
    seeded gy as per-parameter norms + strided samples.  The input is regenerated from its seed by the test; a checksum
    guards against an RNG change."""
    sd = PO.packnet01_state_dict(seed=42, randomize_affine=True)
    net = PackNet01(version="1A")
    _load(net, sd)
    net.train()
    x = synthetic.make_frames(B, H, W, seed=77)["rgb"]
    out = net(x)["inv_depths"]
    g = torch.Generator().manual_seed(78)
    arrays = {"seed_rgb": np.int64(77), "seed_gy": np.int64(78), "rgb_sum": np.float64(x.double().sum().item()),
              "rgb_probe": x.reshape(-1)[::100003].numpy()}
    obj = 0.0
    for i, d in enumerate(out):
        gy = torch.rand(d.shape, generator=g) - 0.5
        obj = obj + (d * gy).sum()
        # the larger maps are stored at every strides[i]-th pixel in both directions (fixture size)
        arrays["disp%d" % (i + 1)] = d.detach()[..., ::strides[i], ::strides[i]].numpy()
        arrays["disp%d_stride" % (i + 1)] = np.int64(strides[i])
    obj.backward()
    _grad_samples([(k, p.grad) for k, p in net.named_parameters()], arrays, "g")
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrays)
    print(name, [tuple(d.shape) for d in out], float(out[0].mean()))


def packnet_config3_case():
    """BASELINE configs[2]'s per-GPU shape: B=2, 384x1280."""
    packnet_baseline_case(B=2, H=384, W=1280, name="packnet01_384x1280_b2", strides=(4, 2, 1, 1))


def step_case(B=2, H=64, W=96, name="step_2x64x96"):
    """Two optimizer steps of the reference's own SelfSupModel (models/SelfSupModel.py:63-97 over SfmModel.py:81-127) with
    the reference's PackNet01 / PoseNet / loss, Adam(lr 2e-4) as model_wrapper.py:128-166: step 0 without the left-right
    flip, step 1 with it.  Stored: both losses and metrics, the depth / pose outputs of step 0, per-parameter gradient
    norms + samples of step 0, and strided parameter samples after each step (8 depth-net tensors + all of PoseNet)."""
    from oracle.step_oracle import posenet_state_dict
    from packnet_sfm.models.SelfSupModel import SelfSupModel
    from packnet_sfm.networks.pose.PoseNet import PoseNet
    depth = PackNet01(version="1A")
    _load(depth, PO.packnet01_state_dict(seed=42, randomize_affine=True))
    pose = PoseNet(nb_ref_imgs=2, rotation_mode="euler")
    _load(pose, posenet_state_dict(43))
    model = SelfSupModel(depth_net=depth, pose_net=pose, rotation_mode="euler", flip_lr_prob=0.0, upsample_depth_maps=True,
                         **YACS_LOSS_DEFAULTS)
    model.train()
    opt = torch.optim.Adam([{"params": depth.parameters(), "lr": 2e-4}, {"params": pose.parameters(), "lr": 2e-4}])
    fr = synthetic.make_frames(B, H, W, seed=91)
    batch = {"rgb": fr["rgb"], "rgb_context": fr["rgb_context"], "rgb_original": fr["rgb"],
             "rgb_context_original": fr["rgb_context"], "intrinsics": fr["intrinsics"]}
    arrays = {"seed_frames": np.int64(91), "B": np.int64(B), "H": np.int64(H), "W": np.int64(W)}
    watch = ["pre_calc.conv_base.weight", "conv1.conv_base.weight", "pack1.conv3d.weight", "pack1.conv.conv_base.weight",
             "pack5.conv.conv_base.weight", "conv5.2.conv3.weight", "unpack3.conv.normalize.weight", "disp1_layer.conv1.weight"]
    for step, flip in enumerate((0.0, 1.0)):
        model.flip_lr_prob = flip
        opt.zero_grad(set_to_none=True)
        out = model(batch)
        out["loss"].backward()
        arrays["loss%d" % step] = out["loss"].detach().numpy()
        arrays["photometric_loss%d" % step] = out["metrics"]["photometric_loss"].numpy()
        arrays["smoothness_loss%d" % step] = out["metrics"]["smoothness_loss"].numpy()
        if step == 0:
            arrays["inv_depth0_step0"] = out["inv_depths"][0].detach().numpy()
            for j, pz in enumerate(out["poses"]):
                arrays["pose%d_step0" % j] = pz.mat.detach().numpy()
            _grad_samples([("depth." + k, p.grad) for k, p in depth.named_parameters()] +
                          [("pose." + k, p.grad) for k, p in pose.named_parameters()], arrays, "g0")
        opt.step()
        named = dict(depth.named_parameters())
        for k in watch:
            flat = named[k].detach().reshape(-1)
            idx = strided_index(flat.numel(), 4096)
            arrays["p%d/depth.%s" % (step, k)] = flat[idx].numpy().copy()
        for k, p_ in pose.named_parameters():
            flat = p_.detach().reshape(-1)
            idx = strided_index(flat.numel(), 512)
            arrays["p%d/pose.%s" % (step, k)] = flat[idx].numpy().copy()
        print(name, "step", step, "flip", flip, float(out["loss"]))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrays)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    only = sys.argv[1:]
    if only:            # python oracle/gen_golden.py step_case packnet_baseline_case
        for fn in only:
            globals()[fn]()
        sys.exit(0)
    loss_case("loss_fullres", 2, 32, 64, True)
    loss_case("loss_multires", 2, 32, 64, False)
    loss_case("loss_mean_noautomask", 1, 24, 40, True, photometric_reduce_op="mean", automask_loss=False,
              smooth_loss_weight=0.1)
    loss_case("loss_bigmotion", 2, 32, 64, True, big_motion=True)
    loss_case("loss_progressive", 1, 32, 64, False, progressive_scaling=0.2)
    block_cases()
    restatement_case()
    loss_restatement_case()
    selfsup_flip_case()
    packnet_case()
    step_case()
    packnet_baseline_case()
    packnet_config3_case()
