"""Host-side mirror of the reference's operator interface around the rasteriser -- same
names, argument meaning and error behaviour as the reference functions, device-agnostic
(the reference hard-codes .cuda(); these follow the input tensors' device so the host logic
is testable on CPU), with the rasteriser / fused kernels reached through the C ABI.

    build_rotation                         reference utils/slam_external.py:25-42
    calc_ssim                              utils/slam_external.py:54-97
    l1_loss_v1, l1_loss_v1_mask            utils/slam_helpers.py:5-9
    setup_camera                           utils/recon_helpers.py:4-27
    transform_to_frame                     utils/slam_helpers.py:323-385
    transformed_params2rendervar           utils/slam_helpers.py:127-160
    get_depth_and_silhouette               utils/slam_helpers.py:217-234
    transformed_params2depthplussilhouette utils/slam_helpers.py:255-287
    initialize_optimizer                   src/vtgaussian_slam.py:180-187
    get_loss                               src/vtgaussian_slam.py:407-689
"""
from __future__ import annotations

from math import exp

import torch
import torch.nn.functional as F

from .rasterizer import GaussianRasterizationSettings as Camera
from .rasterizer import GaussianRasterizer as Renderer
from .rasterizer import run_fitting


# ---------------------------------------------------------------------------- small ops
def build_rotation(q):
    """[M,4] quaternions (w,x,y,z), normalised here -> [M,3,3] rotation matrices."""
    w, x, y, z = (q / q.norm(dim=1, keepdim=True)).unbind(dim=1)
    rows = (1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
            2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
            2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y))
    return torch.stack(rows, dim=1).reshape(-1, 3, 3)


def l1_loss_v1(x, y):
    return (x - y).abs().mean()


def l1_loss_v1_mask(x, y, mask):
    return ((x - y).abs() * mask).mean()


def quat_mult(q1, q2):
    """Hamilton product of [M,4] (w,x,y,z) quaternions."""
    a, b, c, d = q1.unbind(dim=1)
    e, f, g, h = q2.unbind(dim=1)
    return torch.stack((a * e - b * f - c * g - d * h,
                        a * f + b * e + c * h - d * g,
                        a * g - b * h + c * e + d * f,
                        a * h + b * g - c * f + d * e), dim=1)


def _ssim_window(size, sigma, channels, like):
    k = torch.arange(size, dtype=torch.float32) - size // 2
    g = torch.tensor([exp(-float(v) ** 2 / (2.0 * sigma ** 2)) for v in k])
    g = (g / g.sum()).unsqueeze(1)
    w2d = (g @ g.t()).float()
    return w2d.expand(channels, 1, size, size).contiguous().to(like.device).type_as(like)


def calc_ssim(img1, img2, window_size=11, size_average=True):
    """SSIM with an 11x11 Gaussian window (sigma 1.5), zero padding, c1 = 0.01^2, c2 = 0.03^2."""
    ch = img1.size(-3)
    win = _ssim_window(window_size, 1.5, ch, img1)
    blur = lambda t: F.conv2d(t, win, padding=window_size // 2, groups=ch)
    mu1, mu2 = blur(img1), blur(img2)
    var1 = blur(img1 * img1) - mu1.pow(2)
    var2 = blur(img2 * img2) - mu2.pow(2)
    cov = blur(img1 * img2) - mu1 * mu2
    c1, c2 = 0.01 ** 2, 0.03 ** 2
    ssim_map = ((2 * mu1 * mu2 + c1) * (2 * cov + c2)) / ((mu1.pow(2) + mu2.pow(2) + c1) * (var1 + var2 + c2))
    return ssim_map.mean() if size_average else ssim_map.mean(1).mean(1).mean(1)


# ---------------------------------------------------------------------------- camera
def setup_camera(w, h, k, w2c, near=0.01, far=100, device="cuda"):
    """The 11 raster settings for intrinsics k and world-to-camera w2c (matrices in the rasteriser's row-vector
    convention: viewmatrix = w2c^T, projmatrix = (P w2c)^T)."""
    fx, fy, cx, cy = k[0][0], k[1][1], k[0][2], k[1][2]
    world2cam = torch.tensor(w2c).to(device).float()
    proj = torch.zeros(4, 4, device=device)
    proj[0, 0], proj[0, 2] = 2 * fx / w, -(w - 2 * cx) / w
    proj[1, 1], proj[1, 2] = 2 * fy / h, -(h - 2 * cy) / h
    proj[2, 2], proj[2, 3] = far / (far - near), -(far * near) / (far - near)
    proj[3, 2] = 1.0
    view_t = world2cam.t().unsqueeze(0)
    return Camera(image_height=h, image_width=w, tanfovx=w / (2 * fx), tanfovy=h / (2 * fy),
                  bg=torch.zeros(3, dtype=torch.float32, device=device), scale_modifier=1.0,
                  viewmatrix=view_t, projmatrix=view_t.bmm(proj.t().unsqueeze(0)), sh_degree=0,
                  campos=torch.inverse(world2cam)[:3, 3], prefiltered=False)


# ---------------------------------------------------------------------------- render variables
def _frame_pose(params, time_idx, camera_grad, opt_cam_rot, opt_cam_trans):
    if camera_grad and opt_cam_rot is not None and opt_cam_trans is not None:
        return F.normalize(opt_cam_rot[None]), opt_cam_trans
    q, t = params['cam_unnorm_rots'][..., time_idx], params['cam_trans'][..., time_idx]
    if not camera_grad:
        q, t = q.detach(), t.detach()
    return F.normalize(q), t


def transform_to_frame(params, time_idx, gaussians_grad, camera_grad, opt_cam_rot=None, opt_cam_trans=None, latest_w2c=None):
    """World -> camera frame `time_idx`: means3D through [R(q)|t] (optionally pre-multiplied by latest_w2c);
    anisotropic Gaussians (log_scales [N,3]) also get their quaternions rotated."""
    cam_rot, cam_tran = _frame_pose(params, time_idx, camera_grad, opt_cam_rot, opt_cam_trans)
    pts, unnorm_rots = params['means3D'], params['unnorm_rotations']
    if not gaussians_grad:
        pts, unnorm_rots = pts.detach(), unnorm_rots.detach()
    rel_w2c = torch.eye(4, device=pts.device, dtype=pts.dtype)
    rel_w2c[:3, :3] = build_rotation(cam_rot)
    rel_w2c[:3, 3] = cam_tran
    if latest_w2c is not None:
        rel_w2c = latest_w2c @ rel_w2c
    homog = torch.cat((pts, torch.ones_like(pts[:, :1])), dim=1)
    out = {'means3D': (rel_w2c @ homog.T).T[:, :3]}
    if params['log_scales'].shape[1] == 1:                 # isotropic: rotations pass through
        out['unnorm_rotations'] = unnorm_rots
    else:
        out['unnorm_rotations'] = quat_mult(cam_rot, F.normalize(unnorm_rots))
    return out


def _activated(params, transformed_gaussians, colors):
    ls = params['log_scales']
    return {
        'means3D': transformed_gaussians['means3D'],
        'colors_precomp': colors,
        'rotations': F.normalize(transformed_gaussians['unnorm_rotations']),
        'opacities': torch.sigmoid(params['logit_opacities']),
        'scales': torch.exp(ls.expand(-1, 3) if ls.shape[1] == 1 else ls),
        'means2D': torch.zeros_like(params['means3D'], requires_grad=True) + 0,
    }


def transformed_params2rendervar(params, transformed_gaussians):
    return _activated(params, transformed_gaussians, params['rgb_colors'])


def get_depth_and_silhouette(pts_3D, w2c):
    """Per-Gaussian 'colours' (z, 1, z^2) with z the depth of the centre in the frame w2c."""
    z = pts_3D @ w2c[2, :3] + w2c[2, 3]
    return torch.stack((z, torch.ones_like(z), z * z), dim=1)


def transformed_params2depthplussilhouette(params, w2c, transformed_gaussians):
    return _activated(params, transformed_gaussians, get_depth_and_silhouette(transformed_gaussians['means3D'], w2c))


class Adam(torch.optim.Optimizer):
    """torch.optim.Adam(betas, eps, weight_decay=0, amsgrad=False) for CUDA float32 tensors through `vtgs_adam`: one
    library launch per tensor that has a gradient, no foreach / dispatcher work on the host (a third of the host time of
    a reference-style tracking iteration went into the Python of torch's Adam.step()).  Parameter groups, `defaults` and
    the per-parameter state (`step`, `exp_avg`, `exp_avg_sq`) are laid out as torch.optim.Adam lays them out, so code
    that edits `optimizer.state[p]` / `param_groups` (the reference's densification helpers, utils/slam_external.py)
    keeps working."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=0, amsgrad=False, maximize=False))

    @torch.no_grad()
    def step(self, closure=None):
        from .fused import adam_step
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        for group in self.param_groups:
            b1, b2 = group['betas']
            for prm in group['params']:
                g = prm.grad
                if g is None:
                    continue
                if not (prm.is_cuda and prm.dtype == torch.float32 and prm.is_contiguous()):
                    raise ValueError("slam_ops.Adam updates contiguous float32 CUDA tensors")
                st = self.state[prm]
                if len(st) == 0:
                    st['step'] = torch.tensor(0.0)
                    st['exp_avg'] = torch.zeros_like(prm, memory_format=torch.preserve_format)
                    st['exp_avg_sq'] = torch.zeros_like(prm, memory_format=torch.preserve_format)
                st['step'] += 1
                if g.dtype != torch.float32 or not g.is_contiguous():
                    g = g.float().contiguous()
                adam_step(prm, g, st['exp_avg'], st['exp_avg_sq'], group['lr'], step=int(st['step']), beta1=b1, beta2=b2,
                          eps=group['eps'])
        return loss


def initialize_optimizer(params, lrs_dict, tracking):
    """Adam over one parameter group per tensor (reference src/vtgaussian_slam.py:180-187: eps 1e-8 for tracking, lr 0 /
    eps 1e-15 defaults for mapping).  CUDA float32 parameters get `slam_ops.Adam` (the same update through the library's
    Adam kernel); anything else torch.optim.Adam."""
    param_groups = [{'params': [v], 'name': k, 'lr': lrs_dict[k]} for k, v in params.items()]
    native = all(isinstance(v, torch.Tensor) and v.is_cuda and v.dtype == torch.float32 for v in params.values())
    cls = Adam if native else torch.optim.Adam
    if tracking:
        return cls(param_groups)
    return cls(param_groups, lr=0.0, eps=1e-15)


# ---------------------------------------------------------------------------- the loss
REPLICA_SIL_LADDER = [0.990, 0.993, 0.995, 0.997, 0.999]


def _masks_and_losses(im, depth_sil, curr_data, loss_weights, use_sil_for_loss, sil_thres, use_l1,
                      ignore_outlier_depth_loss, tracking, additional_mask, dataset_name, tracking_iteration,
                      presence_sil_mask_mse_ls, sil_thres_ls, far_depth_filter_thres, vis_mask):
    """The part of get_loss after the two renders (reference :467-612,:678-679), pure torch."""
    losses = {}
    depth = depth_sil[0, :, :].unsqueeze(0)
    silhouette = depth_sil[1, :, :]
    presence_sil_mask = None
    if dataset_name == 'replica':
        if tracking and use_sil_for_loss:
            if tracking_iteration == 0 and presence_sil_mask_mse_ls is not None:
                mse_ls = []
                for thr in REPLICA_SIL_LADDER:          # :476-508 pick the threshold with the smallest masked MSE
                    m = (silhouette > thr) & (curr_data['depth'] > 0)
                    cm = torch.tile(m, (3, 1, 1)).detach()
                    mse_ls.append(torch.mean((curr_data['im'] - im)[cm] ** 2).item())
                min_mse = min(mse_ls)
                presence_sil_mask_mse_ls.append(min_mse)
                sil_thres_ls.append(REPLICA_SIL_LADDER[mse_ls.index(min_mse)])
                presence_sil_mask = (silhouette > sil_thres_ls[-1])
            elif sil_thres_ls:
                presence_sil_mask = (silhouette > sil_thres_ls[-1])
            else:
                presence_sil_mask = (silhouette > sil_thres)
    else:
        presence_sil_mask = (silhouette > sil_thres)

    depth_sq = depth_sil[2, :, :].unsqueeze(0)
    uncertainty = (depth_sq - depth ** 2).detach()
    nan_mask = (~torch.isnan(depth)) & (~torch.isnan(uncertainty))
    if ignore_outlier_depth_loss:
        depth_error = torch.abs(curr_data['depth'] - depth) * (curr_data['depth'] > 0)
        mask = (depth_error < 50 * depth_error.median())
        mask = mask & (curr_data['depth'] > 0)
    else:
        mask = (curr_data['depth'] > 0)
    mask = mask & nan_mask
    if tracking and use_sil_for_loss:
        mask = mask & presence_sil_mask
    if tracking and vis_mask is not None and dataset_name != 'replica':
        mask = mask & vis_mask
    if tracking and far_depth_filter_thres is not None and dataset_name not in ('replica', 'scannetpp'):
        mask = mask & (curr_data['depth'] < far_depth_filter_thres)

    if use_l1:
        mask = mask.detach()
        if tracking:
            losses['depth'] = torch.abs(curr_data['depth'] - depth)[mask].sum()
        else:
            losses['depth'] = torch.abs(curr_data['depth'] - depth)[mask].mean()
    if tracking and (use_sil_for_loss or ignore_outlier_depth_loss):
        color_mask = torch.tile(mask, (3, 1, 1)).detach()
        losses['im'] = torch.abs(curr_data['im'] - im)[color_mask].sum()
    elif tracking:
        losses['im'] = torch.abs(curr_data['im'] - im).sum()
    else:
        if additional_mask is None:
            losses['im'] = 0.8 * l1_loss_v1(im, curr_data['im']) + 0.2 * (1.0 - calc_ssim(im, curr_data['im']))
        else:
            am = 10 * additional_mask.to(im.device).float() + 0.8 * torch.ones_like(additional_mask).to(im.device).float()
            losses['im'] = l1_loss_v1_mask(im, curr_data['im'], am) + 0.2 * (1.0 - calc_ssim(im, curr_data['im']))
    weighted_losses = {k: v * loss_weights[k] for k, v in losses.items()}
    loss = sum(weighted_losses.values())
    weighted_losses['loss'] = loss
    return loss, weighted_losses


def _give_grad(means2D, grad):
    """The reference reads variables['means2D'].grad after loss.backward() (utils/slam_external.py:100-102): the leaf
    handed out by get_loss receives the screen-space gradient here (accumulated, like autograd would)."""
    if means2D is None:
        return
    if means2D.grad is None:
        means2D.grad = grad
    else:
        means2D.grad += grad


def _poll_due(renderer, tracking_iteration=None):
    """Poll the overflow counter on a renderer's first use, at the first tracking iteration of a frame, and every 16th
    call otherwise."""
    renderer.polls += 1
    return renderer.polls == 1 or tracking_iteration == 0 or renderer.polls % 16 == 0


class _FusedRender(torch.autograd.Function):
    """im, depth_sil, radii = both rasteriser passes of get_loss as one fused six-plane pass,
    differentiable w.r.t. the Gaussian parameters and the frame's pose slices."""

    @staticmethod
    def forward(ctx, renderer, means3D, rgb, unnorm_rot, logit_op, log_scales, cam_q, cam_t, want_gauss, want_pose, means2D):
        params = dict(means3D=means3D.detach().contiguous(), rgb_colors=rgb.detach().contiguous(),
                      unnorm_rotations=unnorm_rot.detach().contiguous(), logit_opacities=logit_op.detach().contiguous(),
                      log_scales=log_scales.detach().contiguous())
        q, t = cam_q.detach().contiguous().reshape(4), cam_t.detach().contiguous().reshape(3)
        img, radii = run_fitting(lambda: renderer.forward(params, q, t), [renderer], poll=_poll_due(renderer))
        renderer.pending_backward = any(ctx.needs_input_grad)
        ctx.renderer, ctx.params, ctx.q, ctx.t = renderer, params, q, t
        ctx.want = (want_gauss, want_pose)
        ctx.pose_shapes = (cam_q.shape, cam_t.shape)
        out = img.clone()
        ctx.means2D = means2D              # a leaf the caller keeps in variables['means2D']: receives .grad in backward
        radii = radii.clone()
        ctx.mark_non_differentiable(radii)
        return out[:3], out[3:6], radii

    @staticmethod
    def backward(ctx, g_im, g_ds, _g_radii):
        r, params = ctx.renderer, ctx.params
        H, W = r.H, r.W
        dL4 = torch.zeros((4, H, W), dtype=torch.float32, device=g_im.device)
        if g_im is not None:
            dL4[:3] = g_im
        if g_ds is not None:
            if float(g_ds[1:].abs().max()) != 0.0:
                raise NotImplementedError("the fused backward carries gradients for r,g,b and depth only "
                                          "(the reference never differentiates silhouette / depth^2, SURVEY A.7)")
            dL4[3] = g_ds[0]
        want_gauss, want_pose = ctx.want
        pg = {k: torch.zeros_like(params[k]) for k in params} if want_gauss else None
        pose = (torch.zeros(4, device=g_im.device), torch.zeros(3, device=g_im.device)) if want_pose else None
        m2d = torch.zeros_like(params["means3D"])
        r.backward(params, ctx.q, ctx.t, dL_dimage4=dL4, param_grads=pg, pose_grads=pose, means2D_grad=m2d)
        r.pending_backward = False
        _give_grad(ctx.means2D, m2d)
        gq = pose[0].reshape(ctx.pose_shapes[0]) if want_pose else None
        gt = pose[1].reshape(ctx.pose_shapes[1]) if want_pose else None
        if want_gauss:
            return (None, pg["means3D"], pg["rgb_colors"], pg["unnorm_rotations"], pg["logit_opacities"], pg["log_scales"],
                    gq, gt, None, None, None)
        return (None, None, None, None, None, None, gq, gt, None, None, None)


class _FusedTrackingLoss(torch.autograd.Function):
    """loss, loss_terms, radii = get_loss(tracking=True) in three library calls: fused six-plane render,
    masked-L1 tracking loss + dL/dplanes (vtgs_loss), and -- in backward -- the reduction straight to the
    frame's 7 pose numbers (vtgs_fused_backward).  Gaussians are frozen in tracking (their LRs are 0 and
    transform_to_frame detaches them, reference :432-436)."""

    @staticmethod
    def forward(ctx, renderer, params, cam_q, cam_t, gt_rgb, gt_depth, cfg, thres_fn, poll, book, seen_box):
        p = {k: params[k].detach().contiguous() for k in ("means3D", "rgb_colors", "unnorm_rotations", "logit_opacities", "log_scales")}
        q, t = cam_q.detach().contiguous().reshape(4), cam_t.detach().contiguous().reshape(3)
        ctx.pose_shapes = (cam_q.shape, cam_t.shape)
        # A tracking iteration always back-propagates to the pose (reference :1886-1889), so when a pose gradient is
        # wanted the whole iteration -- render, loss, backward, radius bookkeeping -- goes down in ONE library call and
        # backward() only hands the stored gradient over: the host side of a reference-style step is what paces it.
        ctx.eager = thres_fn is None and (ctx.needs_input_grad[2] or ctx.needs_input_grad[3])
        if ctx.eager:
            rgb, dep = gt_rgb.contiguous(), gt_depth.contiguous()
            # (the bookkeeping only reads the radii: repeatable)
            terms, radii, g7, seen = run_fitting(lambda: renderer.tracking_step_cached(p, q, t, rgb, dep, max_2D_radius=book, **cfg),
                                                 [renderer], poll=poll)
            ctx.g7 = g7.clone()                     # the renderer's entry is overwritten by its next step
            terms = terms.clone()
            seen_box.append(seen)
            ctx.mark_non_differentiable(radii, terms)
            return terms[0].clone(), terms, radii
        img, radii = run_fitting(lambda: renderer.forward(p, q, t), [renderer], poll=poll)
        cfg = dict(cfg)
        if thres_fn is not None:
            cfg["sil_thres"] = thres_fn(renderer, gt_rgb.contiguous(), gt_depth.contiguous())
        terms = renderer.tracking_loss(gt_rgb.contiguous(), gt_depth.contiguous(), **cfg).clone()
        renderer.pending_backward = any(ctx.needs_input_grad)
        ctx.renderer, ctx.p, ctx.q, ctx.t = renderer, p, q, t
        ctx.dL4 = renderer.dL_dimage4          # valid until the renderer's next loss call
        if book is not None:
            from .fused import book_radii
            seen_box.append(book_radii(radii, book))
        # radii: the renderer's own buffer (valid until its next forward; get_loss books it at once): no N-sized copy
        ctx.mark_non_differentiable(radii, terms)
        return terms[0].clone(), terms, radii

    @staticmethod
    def backward(ctx, g_loss, _g_terms, _g_radii):
        if ctx.eager:
            g7 = ctx.g7 * g_loss.detach().to(torch.float32)
            return (None, None, g7[:4].reshape(ctx.pose_shapes[0]), g7[4:].reshape(ctx.pose_shapes[1]), None, None, None, None,
                    None, None, None)
        # the backward overwrites both (no zero fill) and multiplies the incoming dL/dloss in its final reduction
        dq = torch.empty(4, dtype=torch.float32, device=g_loss.device)
        dt = torch.empty(3, dtype=torch.float32, device=g_loss.device)
        scale = g_loss.detach().to(torch.float32).contiguous()
        ctx.renderer.backward(ctx.p, ctx.q, ctx.t, dL_dimage4=ctx.dL4, pose_grads=(dq, dt), pose_scale=scale,
                              dl_bound=ctx.renderer.loss_terms[6:7])
        ctx.renderer.pending_backward = False
        return (None, None, dq.reshape(ctx.pose_shapes[0]), dt.reshape(ctx.pose_shapes[1]), None, None, None, None, None, None, None)


class _FusedMappingLoss(torch.autograd.Function):
    """loss, loss_terms, radii = get_loss(mapping=True) on the device: fused six-plane render, the mapping loss
    with its SSIM forward/backward kernels, and the backward to the Gaussian parameters (and the pose if do_ba)."""

    @staticmethod
    def forward(ctx, renderer, means3D, rgb, unnorm_rot, logit_op, log_scales, cam_q, cam_t, gt_rgb, gt_depth, w_im, w_depth,
                want_pose, means2D):
        p = dict(means3D=means3D.detach().contiguous(), rgb_colors=rgb.detach().contiguous(),
                 unnorm_rotations=unnorm_rot.detach().contiguous(), logit_opacities=logit_op.detach().contiguous(),
                 log_scales=log_scales.detach().contiguous())
        q, t = cam_q.detach().contiguous().reshape(4), cam_t.detach().contiguous().reshape(3)
        _, radii = run_fitting(lambda: renderer.forward(p, q, t), [renderer], poll=_poll_due(renderer))
        terms = renderer.mapping_loss(gt_rgb.contiguous(), gt_depth.contiguous(), w_im=w_im, w_depth=w_depth).clone()
        renderer.pending_backward = any(ctx.needs_input_grad)
        ctx.renderer, ctx.p, ctx.q, ctx.t, ctx.want_pose = renderer, p, q, t, want_pose
        ctx.pose_shapes = (cam_q.shape, cam_t.shape)
        ctx.means2D = means2D              # a leaf the caller keeps in variables['means2D']: receives .grad in backward
        radii = radii.clone()
        ctx.mark_non_differentiable(radii, terms)
        return terms[0].clone(), terms, radii

    @staticmethod
    def backward(ctx, g_loss, _g_terms, _g_radii):
        p = ctx.p
        pg = {k: torch.zeros_like(v) for k, v in p.items()}
        pose = None
        if ctx.want_pose:
            pose = (torch.zeros(4, dtype=torch.float32, device=g_loss.device), torch.zeros(3, dtype=torch.float32, device=g_loss.device))
        m2d = torch.zeros_like(p["means3D"])
        ctx.renderer.backward(p, ctx.q, ctx.t, param_grads=pg, pose_grads=pose, means2D_grad=m2d)
        ctx.renderer.pending_backward = False
        _give_grad(ctx.means2D, m2d * g_loss)
        gq = (pose[0] * g_loss).reshape(ctx.pose_shapes[0]) if pose else None
        gt = (pose[1] * g_loss).reshape(ctx.pose_shapes[1]) if pose else None
        return (None, pg["means3D"] * g_loss, pg["rgb_colors"] * g_loss, pg["unnorm_rotations"] * g_loss,
                pg["logit_opacities"] * g_loss, pg["log_scales"] * g_loss, gq, gt, None, None, None, None, None, None)


def _book_radii(variables, radius):
    """reference :681-683: seen = radius > 0; max_2D_radius[seen] = max(radius[seen], max_2D_radius[seen]) -- without the
    boolean-index gathers (one library launch on CUDA, two elementwise torch ops otherwise; radii are >= 0, so unseen
    entries keep their value)."""
    m = variables['max_2D_radius']
    if radius.is_cuda and radius.dtype == torch.int32 and m.dtype == torch.float32 and m.is_contiguous() and radius.is_contiguous():
        from .fused import book_radii
        variables['seen'] = book_radii(radius, m)              # one launch; max_2D_radius updated in place
        return
    variables['seen'] = radius > 0
    variables['max_2D_radius'] = torch.maximum(m, radius.to(m.dtype))


_RENDERERS: dict = {}
_DEPTH_ROWS: dict = {}


def _depth_row_of(w2c):
    """Third row of curr_data['w2c'] as host floats (get_depth_and_silhouette's z).  The device->host read is
    cached per tensor (the reference keeps one first-frame w2c for the whole run, src/vtgaussian_slam.py:209)."""
    key = (id(w2c), getattr(w2c, "_version", 0))
    hit = _DEPTH_ROWS.get(key)
    if hit is None:
        if len(_DEPTH_ROWS) > 64:
            _DEPTH_ROWS.clear()
        row = tuple(float(v) for v in torch.as_tensor(w2c).detach().float().cpu()[2])
        hit = _DEPTH_ROWS[key] = (row, w2c)          # keep the tensor alive so its id stays unique
    return hit[0]


RENDERER_POOL_BYTES = 24 << 30      # device memory the get_loss renderer pool may hold (B200: 180 GB of HBM)


def _renderer_for(cam, n, device):
    """A FusedRenderer for (camera, N) whose buffers are free: a renderer that still holds the state of a forward
    whose backward has not run yet (e.g. the reference's all-keyframes mapping branch sums several get_loss calls
    before one backward, src/vtgaussian_slam.py:2609-2666) is never handed out again.  The pool is bounded by bytes
    and evicts the least recently used idle renderers (N changes at every base frame and differs between tracking and
    mapping)."""
    from .fused import FusedRenderer
    key = (id(cam), n, str(device))
    pool = _RENDERERS.pop(key, None)
    if pool is None:
        pool = ([], cam)                # the camera object is kept alive so that its id stays unique
    _RENDERERS[key] = pool              # (re-)insert as most recently used
    for r in pool[0]:
        if not getattr(r, "pending_backward", False):
            return r
    r = FusedRenderer(cam, n, device=device)
    pool[0].append(r)
    total = sum(x.nbytes for p_ in _RENDERERS.values() for x in p_[0])
    for k in list(_RENDERERS):
        if total <= RENDERER_POOL_BYTES:
            break
        if k == key:
            continue
        idle = [x for x in _RENDERERS[k][0] if not getattr(x, "pending_backward", False)]
        total -= sum(x.nbytes for x in idle)
        keep = [x for x in _RENDERERS[k][0] if getattr(x, "pending_backward", False)]
        if keep:
            _RENDERERS[k] = (keep, _RENDERERS[k][1])
        else:
            del _RENDERERS[k]
    return r


def get_loss(params, curr_data, variables, iter_time_idx, loss_weights, use_sil_for_loss,
             sil_thres, use_l1, ignore_outlier_depth_loss, tracking=False,
             mapping=False, do_ba=False, plot_dir=None, visualize_tracking_loss=False,
             tracking_iteration=None, additional_mask=None, dataset_name=None,
             presence_sil_mask_mse_ls=None, sil_thres_ls=None, far_depth_filter_thres=None, vis_mask_thres=0.05,
             curr_w2c=None, overlap_w2c=None, overlap_gtdepth=None, overlap_last_w2c=None, overlap_last_gtdepth=None,
             overlap_mid_w2c=None, overlap_mid_gtdepth=None, vis_mask=None, backend="fused"):
    """Compute loss for mapping and tracking -- signature and return values of the reference's
    get_loss (src/vtgaussian_slam.py:407-689).  `backend="dropin"` follows the reference
    literally (two Renderer calls); `backend="fused"` (default) renders the six planes in one
    pass with the front end and the pose / parameter chain inside the CUDA kernels.  The
    overlap-visibility mask the reference derives from neighbouring keyframes (:536-583) is
    SLAM policy outside this path: pass it precomputed as `vis_mask`, or pass the reference's own
    `curr_w2c` / `overlap_*` arguments and it is computed here (keyframes.tracking_vis_mask: one keyframe for
    TUM, first | mid | last for ScanNet(++), none for Replica -- reference :536-583)."""
    if vis_mask is None and tracking and overlap_w2c is not None and dataset_name != 'replica':
        from .keyframes import tracking_vis_mask
        overlaps = [(overlap_w2c, overlap_gtdepth)]
        if dataset_name in ('scannet', 'scannetpp'):
            overlaps += [(overlap_mid_w2c, overlap_mid_gtdepth), (overlap_last_w2c, overlap_last_gtdepth)]
        dev_ = curr_data['depth'].device
        overlaps = [(w.to(dev_), d.to(dev_)) for w, d in overlaps]
        vis_mask = tracking_vis_mask(curr_data['depth'], curr_data['intrinsics'].to(dev_), curr_w2c.to(dev_), overlaps, vis_mask_thres)
    for k, v in params.items():
        if not isinstance(v, torch.Tensor):
            params[k] = torch.tensor(v).float().contiguous()
    gaussians_grad = not tracking
    camera_grad = tracking or (mapping and do_ba)

    if backend == "dropin":
        transformed_gaussians = transform_to_frame(params, iter_time_idx, gaussians_grad=gaussians_grad, camera_grad=camera_grad)
        rendervar = transformed_params2rendervar(params, transformed_gaussians)
        depth_sil_rendervar = transformed_params2depthplussilhouette(params, curr_data['w2c'], transformed_gaussians)
        rendervar['means2D'].retain_grad()
        im, radius, _, = Renderer(raster_settings=curr_data['cam'])(**rendervar)
        variables['means2D'] = rendervar['means2D']
        depth_sil, _, _, = Renderer(raster_settings=curr_data['cam'])(**depth_sil_rendervar)
    elif backend == "fused":
        if params['log_scales'].shape[1] != 1:
            raise NotImplementedError("fused backend: isotropic Gaussians only; use backend='dropin'")
        dev = params['means3D'].device
        r = _renderer_for(curr_data['cam'], params['means3D'].shape[0], dev)
        r.depth_row = _depth_row_of(curr_data['w2c'])
        cam_q = params['cam_unnorm_rots'][0, :, iter_time_idx]
        cam_t = params['cam_trans'][0, :, iter_time_idx]
        if not camera_grad:
            cam_q, cam_t = cam_q.detach(), cam_t.detach()
        fused_loss_ok = (tracking and use_l1 and additional_mask is None and set(loss_weights) == {'im', 'depth'})
        if fused_loss_ok:
            # whole tracking loss on the device: no boolean-index gathers, no host synchronisation
            thres, thres_fn = sil_thres, None
            far = 0.0
            if dataset_name == 'replica' and use_sil_for_loss:
                if tracking_iteration == 0 and presence_sil_mask_mse_ls is not None:
                    def thres_fn(renderer, gt_rgb, gt_depth):       # :476-508 threshold ladder, one kernel + one host read
                        res = renderer.sil_ladder(gt_rgb, gt_depth).cpu()
                        presence_sil_mask_mse_ls.append(float(res[11]))
                        sil_thres_ls.append(min(REPLICA_SIL_LADDER, key=lambda v: abs(v - float(res[10]))))
                        return sil_thres_ls[-1]
                elif sil_thres_ls:
                    thres = sil_thres_ls[-1]
            if far_depth_filter_thres is not None and dataset_name not in ('replica', 'scannetpp'):     # reference :586
                far = float(far_depth_filter_thres)
            cfg = dict(w_im=float(loss_weights['im']), w_depth=float(loss_weights['depth']),
                       use_sil_for_loss=bool(use_sil_for_loss), sil_thres=float(thres), far_depth_thres=far,
                       ignore_outlier_depth_loss=bool(ignore_outlier_depth_loss),
                       pixel_mask=(None if (vis_mask is None or dataset_name == 'replica')
                                   else vis_mask.reshape(curr_data['depth'].shape[-2:])))
            # radius bookkeeping (:681-683) inside the same library call when the buffers allow it
            m2r = variables['max_2D_radius']
            book = m2r if (m2r.is_cuda and m2r.dtype == torch.float32 and m2r.is_contiguous() and m2r.shape[0] == r.N) else None
            seen_box = []
            loss, terms, radius = _FusedTrackingLoss.apply(r, params, cam_q, cam_t, curr_data['im'], curr_data['depth'], cfg, thres_fn,
                                                           _poll_due(r, tracking_iteration), book, seen_box)
            weighted_losses = {'depth': terms[2], 'im': terms[1], 'loss': loss}
            if book is not None:
                variables['seen'] = seen_box[0]        # (the renderer's buffer: valid until its next tracking step)
            else:
                _book_radii(variables, radius)
            if presence_sil_mask_mse_ls is not None:
                return loss, variables, weighted_losses, presence_sil_mask_mse_ls, sil_thres_ls
            return loss, variables, weighted_losses
        fused_map_ok = (mapping and not tracking and use_l1 and not ignore_outlier_depth_loss and additional_mask is None
                        and set(loss_weights) == {'im', 'depth'})
        if fused_map_ok:
            means2D = torch.zeros_like(params['means3D'], requires_grad=True)        # leaf: .grad is filled by the backward
            loss, terms, radius = _FusedMappingLoss.apply(
                r, params['means3D'], params['rgb_colors'], params['unnorm_rotations'], params['logit_opacities'],
                params['log_scales'], cam_q, cam_t, curr_data['im'], curr_data['depth'], float(loss_weights['im']),
                float(loss_weights['depth']), camera_grad, means2D)
            variables['means2D'] = means2D
            weighted_losses = {'depth': terms[2], 'im': terms[1], 'loss': loss}
            _book_radii(variables, radius)
            return loss, variables, weighted_losses
        g = (lambda t: t) if gaussians_grad else (lambda t: t.detach())
        means2D = torch.zeros_like(params['means3D'], requires_grad=True)            # leaf: .grad is filled by the backward
        im, depth_sil, radius = _FusedRender.apply(
            r, g(params['means3D']), g(params['rgb_colors']), g(params['unnorm_rotations']), g(params['logit_opacities']),
            g(params['log_scales']), cam_q, cam_t, gaussians_grad, camera_grad, means2D)
        variables['means2D'] = means2D
    else:
        raise ValueError(f"unknown backend {backend!r}")

    loss, weighted_losses = _masks_and_losses(
        im, depth_sil, curr_data, loss_weights, use_sil_for_loss, sil_thres, use_l1, ignore_outlier_depth_loss, tracking,
        additional_mask, dataset_name, tracking_iteration, presence_sil_mask_mse_ls, sil_thres_ls, far_depth_filter_thres,
        vis_mask)

    _book_radii(variables, radius)
    if presence_sil_mask_mse_ls is not None:
        return loss, variables, weighted_losses, presence_sil_mask_mse_ls, sil_thres_ls
    return loss, variables, weighted_losses


def mapping_loss_and_grad(image6, kf, w_im=1.0, w_depth=1.0):
    """Mapping loss of get_loss (:597,:608: mean-L1 depth on depth>0, 0.8 L1 + 0.2 (1-SSIM) colour)
    and its gradient w.r.t. the r,g,b,depth planes, for MappingSolver."""
    img = image6.detach().clone().requires_grad_(True)
    data = dict(im=kf["gt_rgb"], depth=kf["gt_depth"].reshape(1, *image6.shape[1:]))
    loss, _ = _masks_and_losses(img[:3], img[3:6], data, dict(im=w_im, depth=w_depth), False, 0.5, True, False, False,
                                None, None, None, None, None, None, None)
    (g,) = torch.autograd.grad(loss, img)
    return loss.detach(), g[:4].contiguous()
