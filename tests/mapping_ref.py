"""fp64 reference of the mapping iteration (test infrastructure): the reference's own front end (slam_ops host mirrors),
the tiled torch_ref render of the six planes and the mapping branch of get_loss, all through torch autograd on the CPU.

Only the non-differentiable selections come from the oracle's forward: the tile rects and the blend order (its fp32 view
depths, which the kernels reproduce bit for bit).  Every alpha >= 1/255 and T >= 1e-4 decision is the reference's own.
"""
import numpy as np
import torch

import oracle
import torch_ref
from helpers import cam_dict, oracle_camera
from vtgaussian_slam_b200 import slam_ops

F64 = torch.float64
PARAM_KEYS = ("means3D", "rgb_colors", "unnorm_rotations", "logit_opacities", "log_scales")


def mapping_loss(image6, gt_rgb, gt_depth, w_im=1.0, w_depth=1.0):
    """The mapping loss of get_loss (reference :597,:608, slam_ops._masks_and_losses with mapping=True) on fp64 planes
    image6[6,H,W] -> (loss, terms[7]) with terms = loss, w_im*im, w_depth*depth, mask count, L1 mean, SSIM, depth mean:
    the layout of FusedRenderer.mapping_loss's loss_terms.

    calc_ssim runs in fp64 for fp64 planes: its window is built in fp32 (each tap exp() rounded to fp32, normalised in
    fp32, the outer product rounded to fp32) and then converted.  The kernels' make_window builds the same fp32 taps; the
    two windows differ only by that fp32 rounding (a few 1e-8 relative per tap), far below what the comparisons resolve."""
    H, W = image6.shape[1:]
    gt_rgb = torch.as_tensor(gt_rgb, dtype=F64, device=image6.device).reshape(3, H, W)
    gt_depth = torch.as_tensor(gt_depth, dtype=F64, device=image6.device).reshape(1, H, W)
    data = dict(im=gt_rgb, depth=gt_depth)
    loss, wl = slam_ops._masks_and_losses(image6[:3], image6[3:6], data, dict(im=w_im, depth=w_depth), False, 0.5, True, False,
                                          False, None, None, None, None, None, None, None)
    with torch.no_grad():
        d, dsq = image6[3:4], image6[5:6]
        mask = (gt_depth > 0) & ~torch.isnan(d) & ~torch.isnan(dsq - d * d)
        terms = [loss.detach(), wl["im"], wl["depth"], mask.sum().to(F64), (image6[:3] - gt_rgb).abs().mean(),
                 slam_ops.calc_ssim(image6[:3], gt_rgb), (gt_depth - d).abs()[mask].mean()]
    return loss, np.array([float(x.detach()) for x in terms])


def planes_grad(image6, gt_rgb, gt_depth, w_im=1.0, w_depth=1.0, device="cpu"):
    """-> (terms[7], dL/d(r, g, b, depth)[4,H,W]) of mapping_loss for fp32 planes, in fp64 torch on `device` (full frames
    take tens of seconds on the CPU)."""
    img = torch.as_tensor(np.asarray(image6), dtype=F64, device=device).clone().requires_grad_(True)
    loss, terms = mapping_loss(img, gt_rgb, gt_depth, w_im, w_depth)
    (g,) = torch.autograd.grad(loss, img)
    assert float(g[4:].abs().max()) == 0.0            # silhouette and depth^2 carry no gradient
    return terms, g[:4].cpu().numpy()


def iteration(p, q, t, W, H, K, gt_rgb, gt_depth, depth_row=(0.0, 0.0, 1.0, 0.0), w_im=1.0, w_depth=1.0):
    """One render + mapping loss + backward of the view-tied Gaussians `p` (numpy, the reference's parameter layout) seen
    at the pose (cam_unnorm_rot q[4], cam_trans t[3]), in fp64.  The frame's settings are setup_camera(W, H, K, I); the
    depth plane is depth_row . (x_cam, 1) (curr_data['w2c'][2]).
    -> dict(loss, terms[7], grads: the five parameters + cam_unnorm_rots[4] + cam_trans[3] + means2D[N,3],
            n_contrib[H,W] of the fp64 blend, image6[6,H,W])."""
    cam_o, s = oracle_camera(W, H, K)
    fe = oracle.frontend(p["means3D"], p["rgb_colors"], p["unnorm_rotations"], p["logit_opacities"], p["log_scales"], q, t,
                         depth_row=depth_row)
    sel = oracle.Oracle().forward(cam_o, *fe)
    P = {k: torch.tensor(p[k], dtype=F64, requires_grad=True) for k in PARAM_KEYS}
    P["cam_unnorm_rots"] = torch.tensor(np.asarray(q, np.float64)).reshape(1, 4, 1).requires_grad_(True)
    P["cam_trans"] = torch.tensor(np.asarray(t, np.float64)).reshape(1, 3, 1).requires_grad_(True)
    tg = slam_ops.transform_to_frame(P, 0, gaussians_grad=True, camera_grad=True)
    rv = slam_ops.transformed_params2rendervar(P, tg)
    w2c = torch.eye(4, dtype=F64)
    w2c[2] = torch.tensor(depth_row, dtype=F64)
    dsc = slam_ops.get_depth_and_silhouette(tg["means3D"], w2c)
    m2d = torch.zeros(P["means3D"].shape[0], 3, dtype=F64, requires_grad=True)
    out = torch_ref.render(cam_dict(s), rv["means3D"], rv["scales"], rv["rotations"], rv["opacities"][:, 0],
                           torch.cat([rv["colors_precomp"], dsc], 1), sel["rects"], means2D=m2d, tiled=True,
                           sort_depths=sel["depths"])
    loss, terms = mapping_loss(out["color"], gt_rgb, gt_depth, w_im, w_depth)
    loss.backward()
    grads = {k: P[k].grad.numpy() for k in PARAM_KEYS}
    grads["cam_unnorm_rots"] = P["cam_unnorm_rots"].grad.numpy().reshape(4)
    grads["cam_trans"] = P["cam_trans"].grad.numpy().reshape(3)
    grads["means2D"] = m2d.grad.numpy()
    return dict(loss=float(loss.detach()), terms=terms, grads=grads, n_contrib=out["n_contrib"].numpy(),
                image6=out["color"].detach().numpy())


def errors(got, want, scale=None):
    """-> (normwise relative error |g - g64|_2 / |g64|_2, max error / max |g64|).  `scale` (default: want) supplies both
    denominators instead: the gradient of an analytically zero quantity is measured against a related nonzero one."""
    got, want = np.asarray(got, np.float64).reshape(-1), np.asarray(want, np.float64).reshape(-1)
    scale = want if scale is None else np.asarray(scale, np.float64).reshape(-1)
    d = got - want
    return float(np.linalg.norm(d) / max(np.linalg.norm(scale), 1e-300)), float(np.abs(d).max() / max(np.abs(scale).max(), 1e-300))
