"""CPU oracle for the photometric view-synthesis loss (fp32, plain PyTorch + numpy).

TEST INFRASTRUCTURE ONLY -- never imported by the product path (packnet_sfm_b200/).

Restates, with file:line citations into /root/reference/packnet_sfm:
  geometry/pose_utils.py:8-60      euler2mat / pose_vec2mat / invert_pose
  geometry/camera_utils.py:16-59   scale_intrinsics / view_synthesis
  geometry/camera.py:71-191        Kinv / scaled / reconstruct / project
  utils/image.py:85-113,178-282    gradient_x/y, match_scales, image_grid
  utils/depth.py:103-198           inv2depth, inv_depths_normalize, calc_smoothness
  losses/multiview_photometric_loss.py:14-53,127-344   SSIM + MultiViewPhotometricLoss
  losses/loss_base.py:9-48         ProgressiveScaling
  models/model_utils.py:152-180    upsample_output (nearest)

Pinned against tests/golden/loss_*.npz, generated from the live reference by oracle/gen_golden.py
(tests/test_oracle_vs_reference.py, tests/test_oracle_golden.py).

`warp_tap_indices` is the integer oracle for the "warp pixel indices bit-exact" bar: it spells out the
reference's fp32 operation chain one rounding at a time in numpy (numpy never contracts a*b+c into an
FMA), then applies ATen's documented unnormalisation `((g + 1) / 2) * (size - 1)`
(torch/include/ATen/native/GridSampler.h, grid_sampler_unnormalize, align_corners=True) and floor.
"""
import numpy as np
import torch
import torch.nn.functional as F


# ---------------------------------------------------------------------------------------------------
# pose (geometry/pose_utils.py, geometry/pose.py)
# ---------------------------------------------------------------------------------------------------
def euler2mat(angle):
    """pose_utils.py:8-37 -- R = Rx @ Ry @ Rz."""
    B = angle.size(0)
    x, y, z = angle[:, 0], angle[:, 1], angle[:, 2]
    cosz, sinz = torch.cos(z), torch.sin(z)
    zeros = z.detach() * 0
    ones = zeros.detach() + 1
    zmat = torch.stack([cosz, -sinz, zeros, sinz, cosz, zeros, zeros, zeros, ones], dim=1).view(B, 3, 3)
    cosy, siny = torch.cos(y), torch.sin(y)
    ymat = torch.stack([cosy, zeros, siny, zeros, ones, zeros, -siny, zeros, cosy], dim=1).view(B, 3, 3)
    cosx, sinx = torch.cos(x), torch.sin(x)
    xmat = torch.stack([ones, zeros, zeros, zeros, cosx, -sinx, zeros, sinx, cosx], dim=1).view(B, 3, 3)
    return xmat.bmm(ymat).bmm(zmat)


def pose_from_vec(vec):
    """Pose.from_vec(vec, 'euler'), pose.py:39-46 + pose_utils.py:41-51 -> [B,4,4]."""
    trans, rot = vec[:, :3].unsqueeze(-1), vec[:, 3:]
    mat = torch.cat([euler2mat(rot), trans], dim=2)
    pose = torch.eye(4, dtype=vec.dtype, device=vec.device).repeat([len(vec), 1, 1])
    pose[:, :3, :3] = mat[:, :3, :3]
    pose[:, :3, -1] = mat[:, :3, -1]
    return pose


# ---------------------------------------------------------------------------------------------------
# camera (geometry/camera.py, geometry/camera_utils.py)
# ---------------------------------------------------------------------------------------------------
def scale_intrinsics(K, x_scale, y_scale):
    """camera_utils.py:16-22 (on a clone, as Camera.scaled does, camera.py:107)."""
    K = K.clone()
    K[..., 0, 0] *= x_scale
    K[..., 1, 1] *= y_scale
    K[..., 0, 2] = (K[..., 0, 2] + 0.5) * x_scale - 0.5
    K[..., 1, 2] = (K[..., 1, 2] + 0.5) * y_scale - 0.5
    return K


def scaled_K(K, scale):
    """Camera.scaled, camera.py:84-108: scale == 1 returns the same camera."""
    return K if scale == 1.0 else scale_intrinsics(K, scale, scale)


def K_inverse(K):
    """Camera.Kinv, camera.py:71-80."""
    Kinv = K.clone()
    Kinv[:, 0, 0] = 1.0 / K[:, 0, 0]
    Kinv[:, 1, 1] = 1.0 / K[:, 1, 1]
    Kinv[:, 0, 2] = -1.0 * K[:, 0, 2] / K[:, 0, 0]
    Kinv[:, 1, 2] = -1.0 * K[:, 1, 2] / K[:, 1, 1]
    return Kinv


def image_grid(B, H, W, dtype, device=None):
    """image.py:218-282 -- [B,3,H,W] of (x, y, 1) with x in 0..W-1."""
    xs = torch.linspace(0, W - 1, W, dtype=dtype, device=device)
    ys = torch.linspace(0, H - 1, H, dtype=dtype, device=device)
    ys, xs = torch.meshgrid([ys, xs], indexing="ij")
    xs, ys = xs.repeat([B, 1, 1]), ys.repeat([B, 1, 1])
    return torch.stack([xs, ys, torch.ones_like(xs)], dim=1)


def reconstruct(depth, K):
    """Camera.reconstruct(depth, 'w') for the identity-pose target camera, camera.py:112-148.
    Twc of the identity pose is the identity, and R=I, t=0 leaves Xc bit-identical."""
    B, _, H, W = depth.shape
    flat_grid = image_grid(B, H, W, depth.dtype, depth.device).view(B, 3, -1)
    xnorm = K_inverse(K).bmm(flat_grid).view(B, 3, H, W)
    return xnorm * depth


def project(X, K, pose):
    """Camera.project(X, 'w'), camera.py:150-191 with Tcw = pose (pose.py:80-86)."""
    B, _, H, W = X.shape
    Xw = pose[:, :3, :3].bmm(X.view(B, 3, -1)) + pose[:, :3, -1].unsqueeze(-1)
    Xc = K.bmm(Xw)
    Xx, Yy = Xc[:, 0], Xc[:, 1]
    Z = Xc[:, 2].clamp(min=1e-5)
    Xnorm = 2 * (Xx / Z) / (W - 1) - 1.0
    Ynorm = 2 * (Yy / Z) / (H - 1) - 1.0
    return torch.stack([Xnorm, Ynorm], dim=-1).view(B, H, W, 2)


def view_synthesis(ref_image, depth, K, ref_K, pose, padding_mode="zeros"):
    """camera_utils.py:27-59."""
    world_points = reconstruct(depth, K)
    ref_coords = project(world_points, ref_K, pose)
    return F.grid_sample(ref_image, ref_coords, mode="bilinear", padding_mode=padding_mode, align_corners=True)


# ---------------------------------------------------------------------------------------------------
# helpers (utils/image.py, utils/depth.py, models/model_utils.py)
# ---------------------------------------------------------------------------------------------------
def inv2depth(inv_depth):
    """depth.py:103-120."""
    return 1.0 / inv_depth.clamp(min=1e-6)


def match_scales(image, targets, num_scales):
    """image.py:178-214 -- bilinear align_corners=True resize; identity when shapes are equal."""
    out = []
    for i in range(num_scales):
        shape = targets[i].shape[-2:]
        if tuple(image.shape[-2:]) == tuple(shape):
            out.append(image)
        else:
            out.append(F.interpolate(image, size=shape, mode="bilinear", align_corners=True))
    return out


def upsample_output(inv_depths):
    """model_utils.py:152-180 via SfmModel.py:87-88: nearest-upsample every scale to scale 0's shape."""
    shape = inv_depths[0].shape[-2:]
    return [F.interpolate(d, shape, mode="nearest") for d in inv_depths]


def calc_smoothness(inv_depths, images, num_scales):
    """depth.py:146-198."""
    sx, sy = [], []
    for i in range(num_scales):
        d = inv_depths[i]
        mean = d.mean(2, True).mean(3, True)
        dn = d / mean.clamp(min=1e-6)
        gx = dn[:, :, :, :-1] - dn[:, :, :, 1:]
        gy = dn[:, :, :-1, :] - dn[:, :, 1:, :]
        im = images[i]
        igx = im[:, :, :, :-1] - im[:, :, :, 1:]
        igy = im[:, :, :-1, :] - im[:, :, 1:, :]
        wx = torch.exp(-torch.mean(torch.abs(igx), 1, keepdim=True))
        wy = torch.exp(-torch.mean(torch.abs(igy), 1, keepdim=True))
        sx.append(gx * wx)
        sy.append(gy * wy)
    return sx, sy


def ssim(x, y, C1=1e-4, C2=9e-4):
    """SSIM(), multiview_photometric_loss.py:14-53 (3x3 box, reflection pad 1)."""
    x, y = F.pad(x, [1] * 4, mode="reflect"), F.pad(y, [1] * 4, mode="reflect")
    mu_x, mu_y = F.avg_pool2d(x, 3, 1), F.avg_pool2d(y, 3, 1)
    mu_x_mu_y = mu_x * mu_y
    mu_x_sq, mu_y_sq = mu_x.pow(2), mu_y.pow(2)
    sigma_x = F.avg_pool2d(x.pow(2), 3, 1) - mu_x_sq
    sigma_y = F.avg_pool2d(y.pow(2), 3, 1) - mu_y_sq
    sigma_xy = F.avg_pool2d(x * y, 3, 1) - mu_x_mu_y
    v1 = 2 * sigma_xy + C2
    v2 = sigma_x + sigma_y + C2
    return ((2 * mu_x_mu_y + C1) * v1) / ((mu_x_sq + mu_y_sq + C1) * v2)


def progressive_num_scales(progressive_scaling, num_scales, progress):
    """ProgressiveScaling, loss_base.py:9-48."""
    if progressive_scaling > 0.0:
        marks = np.float32([progressive_scaling * (i + 1) for i in range(num_scales - 1)] + [1.0])
        return int(num_scales - np.searchsorted(marks, progress))
    return num_scales


# ---------------------------------------------------------------------------------------------------
# MultiViewPhotometricLoss.forward (losses/multiview_photometric_loss.py:287-344)
# ---------------------------------------------------------------------------------------------------
def photometric_loss_maps(t_est, images, n, ssim_loss_weight, C1, C2, clip_loss):
    """calc_photometric_loss, multiview_photometric_loss.py:188-223."""
    l1 = [torch.abs(t_est[i] - images[i]) for i in range(n)]
    if ssim_loss_weight > 0.0:
        sl = [torch.clamp((1.0 - ssim(t_est[i], images[i], C1, C2)) / 2.0, 0.0, 1.0) for i in range(n)]
        out = [ssim_loss_weight * sl[i].mean(1, True) + (1 - ssim_loss_weight) * l1[i].mean(1, True)
               for i in range(n)]
    else:
        out = l1
    if clip_loss > 0.0:
        for i in range(n):
            mean, std = out[i].mean(), out[i].std()
            out[i] = torch.clamp(out[i], max=float(mean + clip_loss * std))
    return out


def multiview_photometric_loss(image, context, inv_depths, K, ref_K, poses, num_scales=4,
                               ssim_loss_weight=0.85, smooth_loss_weight=0.001, C1=1e-4, C2=9e-4,
                               photometric_reduce_op="min", clip_loss=0.0, progressive_scaling=0.0,
                               padding_mode="zeros", automask_loss=True, progress=0.0,
                               return_maps=False):
    """`poses` is a list of [B,4,4] matrices (Pose.mat).  Defaults are the yacs training defaults
    (configs/default_config.py:88-103), not the constructor defaults (SURVEY.md §0.4)."""
    n = progressive_num_scales(progressive_scaling, num_scales, progress)
    W = image.shape[-1]
    photometric_losses = [[] for _ in range(n)]
    images = match_scales(image, inv_depths, n)
    warped_all = []
    for ref_image, pose in zip(context, poses):
        # warp_ref_image, :127-165
        ref_images = match_scales(ref_image, inv_depths, n)
        ref_warped = []
        for i in range(n):
            scale = inv_depths[i].shape[-1] / float(W)
            ref_warped.append(view_synthesis(ref_images[i], inv2depth(inv_depths[i]),
                                             scaled_K(K.float(), scale), scaled_K(ref_K.float(), scale),
                                             pose, padding_mode))
        warped_all.append(ref_warped)
        pl = photometric_loss_maps(ref_warped, images, n, ssim_loss_weight, C1, C2, clip_loss)
        for i in range(n):
            photometric_losses[i].append(pl[i])
        if automask_loss:
            ul = photometric_loss_maps(ref_images, images, n, ssim_loss_weight, C1, C2, clip_loss)
            for i in range(n):
                photometric_losses[i].append(ul[i])

    # reduce_photometric_loss, :225-253
    def reduce_fn(losses):
        if photometric_reduce_op == "mean":
            return sum([l.mean() for l in losses]) / len(losses)
        if photometric_reduce_op == "min":
            return torch.cat(losses, 1).min(1, True)[0].mean()
        raise NotImplementedError(photometric_reduce_op)

    photometric = sum([reduce_fn(photometric_losses[i]) for i in range(n)]) / n
    loss = photometric
    photometric_metric = photometric.detach()
    smoothness = torch.zeros((), device=loss.device)
    if smooth_loss_weight > 0.0:
        # calc_smoothness_loss, :257-283
        sx, sy = calc_smoothness(inv_depths, images, n)
        smoothness = sum([(sx[i].abs().mean() + sy[i].abs().mean()) / 2 ** i for i in range(n)]) / n
        smoothness = smooth_loss_weight * smoothness
        loss = loss + smoothness
        # Reference quirk, kept on purpose: `loss += smoothness` (:338) is IN PLACE on the tensor whose
        # detached alias was stored by add_metric('photometric_loss', ...) (:252, loss_base.py:72-74),
        # so the reported 'photometric_loss' metric includes the smoothness term.
        photometric_metric = loss.detach()
    out = {"loss": loss.unsqueeze(0),
           "metrics": {"photometric_loss": photometric_metric, "smoothness_loss": smoothness.detach()}}
    if return_maps:
        out["warped"] = warped_all
        out["photometric_maps"] = photometric_losses
    return out


# ---------------------------------------------------------------------------------------------------
# integer oracle for the warp tap indices
# ---------------------------------------------------------------------------------------------------
def warp_tap_indices(inv_depth, K, ref_K, pose, full_width=None):
    """Integer bilinear tap origin (x0, y0) = floor(ix), floor(iy) for every pixel, as int32 [B,H,W,2],
    plus the unnormalised float coordinates [B,H,W,2] (for the knife-edge report).

    One fp32 rounding per reference op, in the reference's order:
      camera.py:136       xnorm = Kinv.bmm(grid)       -> (k00*u + k01*v) + k02*1   (left-to-right, no FMA)
      camera.py:138       Xc = xnorm * depth
      pose.py:84-85       Xw = R.bmm(Xc) + t           (target cam: R=I,t=0 exact; ref cam: the pose)
      camera.py:173       P  = K.bmm(Xw)
      camera.py:178-182   Z = clamp(Pz,1e-5); xn = 2*(Px/Z)/(W-1) - 1
      GridSampler.h       ix = ((xn + 1) / 2) * (W - 1); x0 = floor(ix)
    """
    f32 = np.float32
    inv = inv_depth.detach().numpy().astype(f32)
    B, _, H, W = inv.shape
    scale = 1.0 if full_width is None else W / float(full_width)
    Kt = scaled_K(K.float(), scale)
    Kr = scaled_K(ref_K.float(), scale).numpy().astype(f32)
    Kinv = K_inverse(Kt).numpy().astype(f32)
    T = pose.detach().numpy().astype(f32)
    depth = (f32(1.0) / np.maximum(inv, f32(1e-6))).astype(f32)[:, 0]          # depth.py:120
    u = np.arange(W, dtype=f32)[None, None, :].repeat(H, 1)
    v = np.arange(H, dtype=f32)[None, :, None].repeat(W, 2)
    one = f32(1.0)

    def mat3(M, b, x, y, z):
        rows = []
        for r in range(3):
            acc = (M[b, r, 0] * x).astype(f32)
            acc = (acc + (M[b, r, 1] * y).astype(f32)).astype(f32)
            acc = (acc + (M[b, r, 2] * z).astype(f32)).astype(f32)
            rows.append(acc)
        return rows

    idx = np.zeros((B, H, W, 2), np.int32)
    coords = np.zeros((B, H, W, 2), f32)
    for b in range(B):
        rx, ry, rz = mat3(Kinv, b, u[0], v[0], np.full((H, W), one, f32))
        X, Y, Zc = (rx * depth[b]).astype(f32), (ry * depth[b]).astype(f32), (rz * depth[b]).astype(f32)
        R = T[:, :3, :3]
        wx, wy, wz = mat3(R, b, X, Y, Zc)
        wx = (wx + T[b, 0, 3]).astype(f32)
        wy = (wy + T[b, 1, 3]).astype(f32)
        wz = (wz + T[b, 2, 3]).astype(f32)
        px, py, pz = mat3(Kr, b, wx, wy, wz)
        Z = np.maximum(pz, f32(1e-5))
        xn = (((f32(2.0) * (px / Z).astype(f32)).astype(f32) / f32(W - 1)).astype(f32) - one).astype(f32)
        yn = (((f32(2.0) * (py / Z).astype(f32)).astype(f32) / f32(H - 1)).astype(f32) - one).astype(f32)
        ix = (((xn + one).astype(f32) / f32(2.0)).astype(f32) * f32(W - 1)).astype(f32)
        iy = (((yn + one).astype(f32) / f32(2.0)).astype(f32) * f32(H - 1)).astype(f32)
        coords[b, ..., 0], coords[b, ..., 1] = ix, iy
        # clip before the int cast only to keep the cast defined; the CUDA side applies the same window
        idx[b, ..., 0] = np.floor(np.clip(ix, -2.0e9, 2.0e9)).astype(np.int64).clip(-2**31, 2**31 - 1)
        idx[b, ..., 1] = np.floor(np.clip(iy, -2.0e9, 2.0e9)).astype(np.int64).clip(-2**31, 2**31 - 1)
    return idx, coords


def knife_edge_mask(coords, tol=1e-4):
    """Pixels whose unnormalised coordinate lies within `tol` of an integer (BASELINE.md §2)."""
    return (np.abs(coords - np.round(coords)) < tol).any(-1)
