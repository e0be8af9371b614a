"""Rendered-sequence evaluation (SURVEY.md 8(f) row N4): the reference's `eval` (utils/eval_helpers.py:339-602) over the
fused renderer -- per evaluated frame ONE forward-only six-plane render of the frame's section(s) at its estimated pose
(the reference: transform_to_frame, two render-variable builders, two rasteriser passes) and ONE metrics kernel
(`vtgs_eval_metrics`: PSNR of the valid-depth-weighted images, depth L1 / "RMSE"), MS-SSIM on the device, then the
Horn-aligned trajectory error.  LPIPS needs the AlexNet weights of the `lpips` package (not available offline): reported
as None.  CUDA only, like everything that renders."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib, metrics
from .fused import FusedRenderer
from .rasterizer import _ptr, _stream_ptr, run_fitting
from .slam_loop import quat_from_matrix


class FrameEvaluator:
    """Renders sections at a pose and reduces the reference's per-frame numbers on the device."""

    def __init__(self, settings, device="cuda:0"):
        self.settings, self.device = settings, torch.device(device)
        self._renderers = {}
        self._scratch = torch.zeros(int(_lib.lib().vtgs_eval_scratch_floats()), dtype=torch.float32, device=self.device)

    def renderer(self, n):
        if n not in self._renderers:
            if len(self._renderers) >= 4:
                self._renderers.pop(next(iter(self._renderers)))
            self._renderers[n] = FusedRenderer(self.settings, n, device=self.device)
        return self._renderers[n]

    def render(self, params, w2c):
        """-> image6[6,H,W] (r, g, b, depth, silhouette, depth^2) of `params` seen from the 4x4 `w2c`."""
        M = np.asarray(torch.as_tensor(w2c).detach().cpu(), np.float64)
        q = torch.as_tensor(quat_from_matrix(M[:3, :3]), dtype=torch.float32, device=self.device)
        t = torch.as_tensor(M[:3, 3], dtype=torch.float32, device=self.device)
        r = self.renderer(int(params["means3D"].shape[0]))
        image6, _ = run_fitting(lambda: r.forward(params, q, t), [r])
        return image6

    def frame_metrics(self, image6, gt_rgb, gt_depth, sil_thres, use_presence=False, want_ssim=True):
        """-> dict(psnr, depth_l1, depth_rmse, ms_ssim, valid) of one rendered frame (reference :431-477).
        use_presence: weight by the presence mask too (the reference's `mapping_iters == 0 and not add_new_gaussians`)."""
        r = next(iter(self._renderers.values()))
        out = torch.zeros(8, dtype=torch.float32, device=self.device)
        gt_rgb = gt_rgb.to(self.device, torch.float32).contiguous()
        gt_depth = gt_depth.to(self.device, torch.float32).reshape(r.H, r.W).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().vtgs_eval_metrics(C.byref(r.cam), _ptr(image6), _ptr(gt_rgb), _ptr(gt_depth), float(sil_thres),
                                                    int(bool(use_presence)), _ptr(out), _ptr(self._scratch), _stream_ptr(self.device)))
        ssim = None
        if want_ssim and min(r.H, r.W) > 160:
            w = (gt_depth > 0)
            if use_presence:
                w = w & (image6[4] > sil_thres)
            ssim = metrics.ms_ssim((image6[:3] * w)[None], (gt_rgb * w)[None], data_range=1.0, size_average=True)
        o = out.cpu()
        return dict(psnr=float(o[5]), depth_l1=float(o[6]), depth_rmse=float(o[7]), valid=float(o[4]),
                    ms_ssim=None if ssim is None else float(ssim))


def eval_sequence(frames, store, w2c_list, settings, baseframe_every, sil_thres=0.5, mapping_iters=1, add_new_gaussians=True,
                  eval_every=1, baseframe_corr_list=None, gt_c2w=None, want_ssim=True, device="cuda:0"):
    """The reference's `eval`: frame t is rendered from section int(t / baseframe_every) -- or, with
    `baseframe_corr_list`, from the concatenation of the sections of the listed frames (:386-394) -- at w2c_list[t].
    frames: indexable of dicts with 'im'[3,H,W], 'depth'[1,H,W] (and 'c2w' when gt_c2w is not given);
    store: slam_loop.SectionStore (e.g. import_params_ls).  -> dict of per-frame lists, their means and the ATE."""
    ev = FrameEvaluator(settings, device)
    use_presence = mapping_iters == 0 and not add_new_gaussians
    res = dict(frame=[], psnr=[], depth_rmse=[], depth_l1=[], ms_ssim=[], lpips=None)
    gts = []
    n = min(len(frames), len(w2c_list))
    for t in range(n):
        fr = frames[t]
        if gt_c2w is None and "c2w" in fr:
            gts.append(np.asarray(fr["c2w"], np.float64))
        if t != 0 and t % eval_every != 0:
            continue
        base = int(t / baseframe_every)
        if baseframe_corr_list is None or base == 0:
            secs = [min(base, len(store) - 1)]
        else:
            secs = [int(i / baseframe_every) for i in baseframe_corr_list[base - 1]]
        params = store.gather(secs)
        image6 = ev.render(params, w2c_list[t])
        m = ev.frame_metrics(image6, torch.as_tensor(fr["im"]), torch.as_tensor(fr["depth"]), sil_thres, use_presence, want_ssim)
        res["frame"].append(t)
        for k_, key in (("psnr", "psnr"), ("depth_rmse", "depth_rmse"), ("depth_l1", "depth_l1"), ("ms_ssim", "ms_ssim")):
            res[k_].append(m[key])
    gt = gt_c2w if gt_c2w is not None else (gts if len(gts) == n else None)
    if gt is not None:
        ok = [i for i in range(n) if np.isfinite(np.asarray(gt[i])).all()]
        res["ate_rmse"] = metrics.ate_after_alignment([gt[i] for i in ok], [np.linalg.inv(np.asarray(w2c_list[i], np.float64)) for i in ok])
    for k_ in ("psnr", "depth_rmse", "depth_l1", "ms_ssim"):
        vals = [v for v in res[k_] if v is not None]
        res["avg_" + k_] = float(np.mean(vals)) if vals else None
    return res
