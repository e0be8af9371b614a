"""Fused view-tied render -> loss -> backward -> Adam iteration (the hot loops of
reference src/vtgaussian_slam.py:1794-1891 (tracking) and :2525-2702 (mapping)).

One six-plane pass replaces the two rasteriser passes of get_loss (:461,:466), the front end
(transform_to_frame, the two render-variable builders) runs inside the preprocess kernel,
the masked-L1 loss and its gradient are one kernel, the backward reduces straight to the
7 pose numbers (tracking) and/or the Gaussian parameter gradients (mapping), and Adam is one
kernel per tensor.  Nothing here synchronises with the host, so `TrackingSolver` /
`MappingSolver` capture a whole iteration in a CUDA graph.

All compute is in libvtgs_cuda.so (include/vtgs.h); no CPU path.
"""
from __future__ import annotations

import ctypes as C
import operator
import os

import torch

from . import _lib
from .rasterizer import (Workspace, _ptr, _require_cuda, _stream_ptr, _tensor_bytes, camera_struct, grown_pair_capacity,
                         initial_pair_capacity, run_fitting)

PARAM_KEYS = ("means3D", "rgb_colors", "unnorm_rotations", "logit_opacities", "log_scales")
BA_RECORDS_PER_RANK = 8         # keyframes one rank may step with do_ba in a sharded mapping iteration (its record table)


class FusedRenderer:
    """Persistent buffers for rendering N view-tied Gaussians into a W x H frame.

    pair_capacity bounds R = sum(tiles_touched); the library never reads R back.  Run the work
    through `run_fitting` with a poll when a blocking read is cheap -- e.g. once per frame --
    and it is repeated with grown pair buffers if a render was truncated."""

    def __init__(self, settings, num_gaussians, device="cuda:0", pair_capacity=None, tile_rows=(0, 0),
                 depth_row=(0.0, 0.0, 1.0, 0.0), deterministic=None):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("FusedRenderer needs a CUDA device: vtgaussian_slam_b200 has no CPU fallback")
        self.cam = camera_struct(settings, tile_rows=tile_rows)
        self.W, self.H, self.N = self.cam.image_width, self.cam.image_height, int(num_gaussians)
        if pair_capacity is None:
            pair_capacity = initial_pair_capacity(self.device, self.N)
        # deterministic: fixed-point gradient accumulation (rasterizer.set_deterministic is the default when None)
        self.ws = Workspace(self.device, self.W, self.H, self.N, pair_capacity, deterministic=deterministic)
        self.ws.ensure_grad_geom()
        self.depth_row = tuple(float(v) for v in depth_row)
        L = _lib.lib()
        f32 = dict(dtype=torch.float32, device=self.device)
        self.image6 = torch.zeros((6, self.H, self.W), **f32)
        self.radii = torch.zeros(max(self.N, 1), dtype=torch.int32, device=self.device)
        self.dL_dimage4 = torch.zeros((4, self.H, self.W), **f32)
        self.loss_terms = torch.zeros(8, **f32)
        self._loss_scratch = torch.zeros(int(L.vtgs_loss_scratch_floats(self.W, self.H, 0)), **f32)
        self._pose_scratch = torch.zeros(int(L.vtgs_pose_scratch_floats(self.N)), **f32)
        self._map_scratch = None
        self._median_state = None
        self._sil = None                    # [0:10] ladder sums, [10] chosen threshold, [11] its MSE
        self._bufs, self._bufs_generation = self.ws.struct(), self.ws.generation
        self.polls = 0
        self._step_graphs = {}              # tracking_step_cached: pointer set -> captured launch sequence
        self._cap_stream = None

    # -- helpers ---------------------------------------------------------------------------
    def _buffers(self):
        """The workspace's VtgsBuffers.  When the pair buffers have been reallocated since it was built, it is rebuilt
        and the step graphs, whose launches point into the old buffers, are dropped."""
        if self._bufs_generation != self.ws.generation:
            self._bufs, self._bufs_generation = self.ws.struct(), self.ws.generation
            self._step_graphs.clear()
        return self._bufs

    def overflowed(self):
        R, overflow, _ = self.ws.read_counters()
        return bool(overflow), R

    def ensure_capacity(self):
        """One blocking read of the device counters.  -> True if the last forward overflowed the pair buffers: they
        have been enlarged and the forward (and everything derived from it) must be repeated."""
        return self.ws.ensure_capacity()

    @property
    def nbytes(self):
        """Device memory held by this renderer's tensors and its workspace's (pool accounting in slam_ops)."""
        return self.ws.nbytes + _tensor_bytes(self)

    def median_state(self, image6=None, gt_depth=None, process_group=None, num_pixels_total=None):
        """Radix-select state of median(|gt - depth| (gt > 0)) over the frame (reference :525-527, :757-758) for the
        last forward.  With a process group every rank histograms its tile-row band and the histograms are
        all-reduced between the two kernels of each pass, so all ranks pick the same (frame-wide) median."""
        L = _lib.lib()
        if self._median_state is None:
            self._median_state = torch.zeros(_lib.MEDIAN_STATE_WORDS, dtype=torch.int32, device=self.device)
        st = self._median_state
        st.zero_()
        img = self.image6 if image6 is None else image6
        P = self.W * self.H if num_pixels_total is None else int(num_pixels_total)
        with torch.cuda.device(self.device):
            for ps in range(4):
                _lib.check(L.vtgs_median_hist(C.byref(self.cam), _ptr(img[3]), _ptr(gt_depth), ps, _ptr(st), _stream_ptr(self.device)))
                if process_group is not None:
                    torch.distributed.all_reduce(st[:_lib.MEDIAN_SUMMABLE_WORDS], group=process_group)
                _lib.check(L.vtgs_median_pick(P, ps, _ptr(st), _stream_ptr(self.device)))
        return st

    def sil_ladder(self, gt_rgb, gt_depth, image6=None, process_group=None):
        """Replica's iteration-0 threshold search (reference :472-510) on the last forward, on the device.
        -> tensor[12]: ten sums, the chosen threshold [10] and its MSE [11]; [10:11] can be handed to tracking_loss as
        `sil_thres_dev`.  With a process group the ten band sums are all-reduced before the choice."""
        L = _lib.lib()
        if self._sil is None:
            self._sil = torch.zeros(12, dtype=torch.float32, device=self.device)
        img = self.image6 if image6 is None else image6
        with torch.cuda.device(self.device):
            _lib.check(L.vtgs_sil_ladder(C.byref(self.cam), _ptr(img), _ptr(gt_rgb), _ptr(gt_depth), _ptr(self._sil),
                                         _ptr(self._loss_scratch), _stream_ptr(self.device)))
            if process_group is not None:
                torch.distributed.all_reduce(self._sil[:10], group=process_group)
            _lib.check(L.vtgs_sil_select(_ptr(self._sil), _ptr(self._sil[10:]), _ptr(self._sil[11:]), _stream_ptr(self.device)))
        return self._sil

    def nonpresence_mask(self, gt_depth, sil_thres=0.5, image6=None):
        """Non-presence mask of the reference's silhouette-driven Gaussian addition (add_new_gaussians_base_frame,
        src/vtgaussian_slam.py:747-760) for the last forward: -> (mask[H,W] uint8, count[1] int32), both on the device."""
        img = self.image6 if image6 is None else image6
        st = self.median_state(img, gt_depth)
        mask = torch.empty((self.H, self.W), dtype=torch.uint8, device=self.device)
        count = torch.zeros(1, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().vtgs_nonpresence_mask(C.byref(self.cam), _ptr(img), _ptr(gt_depth), float(sil_thres), _ptr(st),
                                                        _ptr(mask), _ptr(count), _stream_ptr(self.device)))
        return mask, count

    def _params_struct(self, params):
        p = _lib.VtgsParams()
        for k in PARAM_KEYS:
            t = params[k]
            _require_cuda(k, t)
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError(f"params['{k}'] must be contiguous float32")
            setattr(p, k, t.data_ptr())
        ls = params["log_scales"]
        p.log_scales_dim = 1 if ls.dim() == 1 else int(ls.shape[1])
        p.num_gaussians = self.N
        if params["means3D"].shape[0] != self.N:
            raise ValueError("number of Gaussians differs from the renderer's")
        return p

    def _pose_struct(self, cam_q, cam_t):
        for n, t, k in (("cam_q", cam_q, 4), ("cam_t", cam_t, 3)):
            _require_cuda(n, t)
            if t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != k:
                raise ValueError(f"{n} must be a contiguous float32 tensor of {k} elements")
        ps = _lib.VtgsPose()
        ps.cam_unnorm_rot = cam_q.data_ptr()
        ps.cam_trans = cam_t.data_ptr()
        ps.depth_row[:] = self.depth_row
        return ps

    # -- the three stages ------------------------------------------------------------------
    def forward(self, params, cam_q, cam_t):
        """-> image6[6,H,W] = (r, g, b, depth, silhouette, depth^2), radii[N].  Buffers are reused."""
        p, ps = self._params_struct(params), self._pose_struct(cam_q, cam_t)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().vtgs_fused_forward(C.byref(self.cam), C.byref(p), C.byref(ps), _ptr(self.image6),
                                                     _ptr(self.radii), C.byref(self._buffers()), _stream_ptr(self.device)))
        return self.image6, self.radii[:self.N]

    def tracking_loss(self, gt_rgb, gt_depth, w_im=0.5, w_depth=0.025, use_sil_for_loss=True, sil_thres=0.99,
                      far_depth_thres=0.0, image6=None, ignore_outlier_depth_loss=False, pixel_mask=None,
                      sil_thres_dev=None, median_state=None):
        """Masked-L1 tracking loss (reference get_loss :513-605,:678-679) of the last forward.
        ignore_outlier_depth_loss: also drop pixels whose depth error is >= 50x its frame median (:525-528);
        pixel_mask: optional [H,W] uint8 / bool CUDA tensor, 0 = masked out (the overlap-visibility mask, :536-583).
        sil_thres_dev: optional device float overriding sil_thres (sil_ladder()[10:11]); median_state: a finished
        median_state() (needed with a tile-row band, where the median is a frame-wide quantity).
        -> loss_terms[8] (device): loss, w_im*im, w_depth*depth, mask count, ...; fills dL_dimage4."""
        pm = None
        if pixel_mask is not None:
            _require_cuda("pixel_mask", pixel_mask)
            pm = pixel_mask.reshape(self.H, self.W)
            pm = (pm if pm.dtype == torch.uint8 else pm.to(torch.uint8)).contiguous()
            self._pixel_mask = pm               # keep alive until the kernel has run
        cfg = _lib.VtgsLossConfig(0, int(bool(use_sil_for_loss)), int(bool(ignore_outlier_depth_loss)), 1, float(sil_thres),
                                  float(w_im), float(w_depth), float(far_depth_thres), _ptr(pm), _ptr(sil_thres_dev),
                                  _ptr(median_state))
        img = self.image6 if image6 is None else image6
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().vtgs_loss(C.byref(self.cam), C.byref(cfg), _ptr(img), _ptr(gt_rgb), _ptr(gt_depth),
                                            _ptr(self.dL_dimage4), _ptr(self.loss_terms), _ptr(self._loss_scratch),
                                            _stream_ptr(self.device)))
        return self.loss_terms

    def tracking_step(self, params, cam_q, cam_t, gt_rgb, gt_depth, pose_grads, w_im=0.5, w_depth=0.025, use_sil_for_loss=True,
                      sil_thres=0.99, far_depth_thres=0.0, ignore_outlier_depth_loss=False, pixel_mask=None,
                      max_2D_radius=None, seen=None):
        """forward + tracking_loss + backward (to the 7 pose numbers, unscaled) [+ book_radii] in ONE library call
        (`vtgs_fused_tracking_step`): what get_loss(tracking=True) followed by loss.backward() launches, with one
        Python / ctypes crossing instead of four.  -> (loss_terms[8], radii[N]); fills pose_grads = (d_cam_q[4], d_cam_t[3])."""
        p, ps = self._params_struct(params), self._pose_struct(cam_q, cam_t)
        pm = None
        if pixel_mask is not None:
            _require_cuda("pixel_mask", pixel_mask)
            pm = pixel_mask.reshape(self.H, self.W)
            pm = (pm if pm.dtype == torch.uint8 else pm.to(torch.uint8)).contiguous()
            self._pixel_mask = pm
        cfg = _lib.VtgsLossConfig(0, int(bool(use_sil_for_loss)), int(bool(ignore_outlier_depth_loss)), 1, float(sil_thres),
                                  float(w_im), float(w_depth), float(far_depth_thres), _ptr(pm), None, None)
        g = _lib.VtgsParamGrads()
        g.cam_unnorm_rot, g.cam_trans = pose_grads[0].data_ptr(), pose_grads[1].data_ptr()
        g.pose_scratch = self._pose_scratch.data_ptr()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().vtgs_fused_tracking_step(
                C.byref(self.cam), C.byref(p), C.byref(ps), C.byref(cfg), _ptr(gt_rgb), _ptr(gt_depth), _ptr(self.image6),
                _ptr(self.radii), _ptr(self.dL_dimage4), _ptr(self.loss_terms), _ptr(self._loss_scratch), C.byref(g),
                _ptr(max_2D_radius), _ptr(seen), C.byref(self._buffers()), _stream_ptr(self.device)))
        return self.loss_terms, self.radii[:self.N]

    STEP_GRAPHS_MAX = 8

    def tracking_step_cached(self, params, cam_q, cam_t, gt_rgb, gt_depth, max_2D_radius=None, **cfg):
        """tracking_step for callers that step from a host loop with the SAME buffers (the reference's tracking loop: 40-200
        iterations per frame on one pose slice and one frame): the second call with a given set of pointers and loss
        settings captures the launch sequence in a CUDA graph, later ones replay it (one launch, and back-to-back kernels
        overlap their tails as in TrackingSolver).  The entry owns the outputs that must not move: -> (loss_terms, radii,
        pose_grad[7] = d_cam_q | d_cam_t, seen or None), valid until the entry's next call."""
        self._buffers()                     # (drops the graphs of reallocated pair buffers)
        pm = cfg.get("pixel_mask")
        key = (tuple(params[k].data_ptr() for k in PARAM_KEYS), cam_q.data_ptr(), cam_t.data_ptr(), gt_rgb.data_ptr(), gt_depth.data_ptr(),
               0 if pm is None else pm.data_ptr(), 0 if max_2D_radius is None else max_2D_radius.data_ptr(),
               tuple(sorted((k, v) for k, v in cfg.items() if k != "pixel_mask")))
        ent = self._step_graphs.pop(key, None)
        if ent is None:
            if len(self._step_graphs) >= self.STEP_GRAPHS_MAX:
                self._step_graphs.pop(next(iter(self._step_graphs)))          # least recently used
            ent = dict(calls=0, graph=None, g7=torch.empty(7, dtype=torch.float32, device=self.device),
                       seen=None if max_2D_radius is None else torch.empty(self.N, dtype=torch.bool, device=self.device))
        self._step_graphs[key] = ent
        ent["calls"] += 1
        run = lambda: self.tracking_step(params, cam_q, cam_t, gt_rgb, gt_depth, (ent["g7"][:4], ent["g7"][4:]),
                                         max_2D_radius=max_2D_radius, seen=ent["seen"], **cfg)
        pm_stable = pm is None or (pm.dtype == torch.uint8 and pm.is_contiguous())
        if (ent["graph"] is None and ent["calls"] == 2 and pm_stable and os.environ.get("VTGS_STEP_GRAPH", "1") != "0"
                and not torch.cuda.is_current_stream_capturing()):          # (a caller capturing its own graph keeps plain launches)
            if self._cap_stream is None:
                self._cap_stream = torch.cuda.Stream(self.device)
            cur = torch.cuda.current_stream(self.device)
            self._cap_stream.wait_stream(cur)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(self._cap_stream):
                g.capture_begin(capture_error_mode="thread_local")      # (a frame-prefetch worker may be allocating)
                run()
                g.capture_end()
            cur.wait_stream(self._cap_stream)
            ent["graph"] = g
        if ent["graph"] is not None:
            ent["graph"].replay()
        else:
            run()
        return self.loss_terms, self.radii[:self.N], ent["g7"], ent["seen"]

    def mapping_loss(self, gt_rgb, gt_depth, w_im=1.0, w_depth=1.0, image6=None):
        """Mapping loss of get_loss (reference :597,:608): w_depth * mean|gt-d|[gt>0] + w_im * (0.8 L1mean +
        0.2 (1 - SSIM)) of the last forward, SSIM forward+backward in hand-written kernels.
        -> loss_terms[8] (device): loss, w_im*im, w_depth*depth, mask count, L1 mean, SSIM, depth L1 mean; fills dL_dimage4."""
        if self._map_scratch is None:
            n = int(_lib.lib().vtgs_loss_scratch_floats(self.W, self.H, 1))
            self._map_scratch = torch.zeros(n, dtype=torch.float32, device=self.device)
        cfg = _lib.VtgsLossConfig(1, 0, 0, 1, 0.0, float(w_im), float(w_depth), 0.0)
        img = self.image6 if image6 is None else image6
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().vtgs_loss(C.byref(self.cam), C.byref(cfg), _ptr(img), _ptr(gt_rgb), _ptr(gt_depth),
                                            _ptr(self.dL_dimage4), _ptr(self.loss_terms), _ptr(self._map_scratch),
                                            _stream_ptr(self.device)))
        return self.loss_terms

    def backward(self, params, cam_q, cam_t, dL_dimage4=None, param_grads=None, pose_grads=None, means2D_grad=None,
                 accumulate=False, pose_scale=None, dl_bound=None):
        """param_grads: dict key -> tensor to receive dL/dparams[key] (any subset of PARAM_KEYS).
        pose_grads: (d_cam_q[4], d_cam_t[3]) tensors or None; pose_scale: optional device scalar multiplied into them."""
        p, ps = self._params_struct(params), self._pose_struct(cam_q, cam_t)
        g = _lib.VtgsParamGrads()
        for k in PARAM_KEYS:
            t = None if param_grads is None else param_grads.get(k)
            if t is not None:
                if t.shape != params[k].shape or t.dtype != torch.float32 or not t.is_contiguous():
                    raise ValueError(f"gradient buffer for '{k}' must match the parameter")
                setattr(g, k, t.data_ptr())
        if means2D_grad is not None:
            g.means2D = means2D_grad.data_ptr()
        if pose_grads is not None:
            g.cam_unnorm_rot, g.cam_trans = pose_grads[0].data_ptr(), pose_grads[1].data_ptr()
            g.pose_scratch = self._pose_scratch.data_ptr()
            if pose_scale is not None:
                g.pose_scale = pose_scale.data_ptr()
        if dl_bound is not None:            # deterministic mode: a device scalar >= max |dL_dimage4| (else it is measured)
            g.dL_abs_bound = dl_bound.data_ptr()
        dL = self.dL_dimage4 if dL_dimage4 is None else dL_dimage4
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().vtgs_fused_backward(C.byref(self.cam), C.byref(p), C.byref(ps), _ptr(dL), int(bool(accumulate)),
                                                      C.byref(g), C.byref(self._buffers()), _stream_ptr(self.device)))


def book_radii(radii, max_2D_radius, seen=None):
    """get_loss's radius bookkeeping (reference src/vtgaussian_slam.py:681-683) in one launch: -> seen (bool[N]);
    max_2D_radius (float[N]) is updated in place."""
    n = int(radii.shape[0])
    if seen is None:
        seen = torch.empty(n, dtype=torch.bool, device=radii.device)
    with torch.cuda.device(radii.device):
        _lib.check(_lib.lib().vtgs_book_radii(n, _ptr(radii), _ptr(max_2D_radius), _ptr(seen), _stream_ptr(radii.device)))
    return seen


def retie(means3D, w2c_old, cam_q, cam_t):
    """In place: means3D <- inv([R(cam_q)|cam_t]) (w2c_old means3D) -- the reference's re-tie of a section's newest
    Gaussians to the pose the mapping step just optimised (src/vtgaussian_slam.py:2706-2727).  `means3D` may be a
    contiguous row slice (e.g. params['means3D'][-num_gs_curr:])."""
    _require_cuda("means3D", means3D)
    if not means3D.is_contiguous() or means3D.dtype != torch.float32:
        raise ValueError("means3D must be a contiguous float32 tensor (a row slice is fine)")
    m = torch.as_tensor(w2c_old).detach().float().cpu().reshape(4, 4)[:3].reshape(-1).tolist()
    arr = (C.c_float * 12)(*m)
    with torch.cuda.device(means3D.device):
        _lib.check(_lib.lib().vtgs_retie(_ptr(means3D), means3D.shape[0], C.byref(arr), _ptr(cam_q), _ptr(cam_t),
                                         _stream_ptr(means3D.device)))
    return means3D


def adam_step(param, grad, exp_avg, exp_avg_sq, lr, step=None, step_dev=None, beta1=0.9, beta2=0.999, eps=1e-8):
    """torch.optim.Adam's update of one tensor (reference initialize_optimizer,
    src/vtgaussian_slam.py:180-187: eps 1e-8 tracking, 1e-15 mapping)."""
    _require_cuda("param", param)
    with torch.cuda.device(param.device):
        _lib.check(_lib.lib().vtgs_adam(_ptr(param), _ptr(grad), _ptr(exp_avg), _ptr(exp_avg_sq), param.numel(), float(lr),
                                        float(beta1), float(beta2), float(eps), int(step or 0), _ptr(step_dev),
                                        _stream_ptr(param.device)))


def retie_dev(means3D, old_q, old_t, cam_q, cam_t):
    """retie() with the old pose on the device (un-normalised quaternion [4] + translation [3]): no host round trip."""
    _require_cuda("means3D", means3D)
    if not means3D.is_contiguous() or means3D.dtype != torch.float32:
        raise ValueError("means3D must be a contiguous float32 tensor (a row slice is fine)")
    with torch.cuda.device(means3D.device):
        _lib.check(_lib.lib().vtgs_retie_dev(_ptr(means3D), means3D.shape[0], _ptr(old_q), _ptr(old_t), _ptr(cam_q), _ptr(cam_t),
                                             _stream_ptr(means3D.device)))
    return means3D


def ba_record_table(keyframes, num_gaussians):
    """This rank's record table of a keyframe-sharded bundle-adjustment iteration (`vtgs_retie_records`, include/vtgs.h),
    on the host: [BA_RECORDS_PER_RANK, BA_RECORD_WORDS] int32 with one record per keyframe in list order -- valid = 1, the
    keyframe's "id", its `retie_last` -- and the pose words and the unused slots zero.  Raises ValueError when a keyframe
    has no integer "id", two keyframes share one, there are more keyframes than records or `retie_last` is not in 0..N."""
    if len(keyframes) > BA_RECORDS_PER_RANK:
        raise ValueError(f"do_ba under keyframe sharding steps at most {BA_RECORDS_PER_RANK} keyframes per rank and iteration, "
                         f"got {len(keyframes)}")
    table = torch.zeros((BA_RECORDS_PER_RANK, _lib.BA_RECORD_WORDS), dtype=torch.int32)
    ids = set()
    for s, kf in enumerate(keyframes):
        try:
            k = operator.index(kf["id"])
        except (KeyError, TypeError):
            raise ValueError("do_ba under keyframe sharding needs an integer 'id' on every keyframe") from None
        if not -2 ** 31 <= k < 2 ** 31 or k in ids:
            raise ValueError(f"keyframe id {k} is repeated or does not fit 32 bits")
        ids.add(k)
        n_last = int(kf.get("retie_last", 0))
        if not 0 <= n_last <= num_gaussians:
            raise ValueError(f"retie_last = {n_last} of keyframe {k} is not in 0..{num_gaussians}")
        table[s, 0], table[s, 1], table[s, 2] = 1, k, n_last
    return table


def decode_ba_poses(tables):
    """{id: (cam_q[4], cam_t[3])}: the stepped poses of the valid records of host tables [..., BA_RECORD_WORDS] int32.
    Raises ValueError when an id appears twice."""
    words = tables.reshape(-1, _lib.BA_RECORD_WORDS)
    floats = words.view(torch.float32)
    poses = {}
    for rec, f in zip(words.tolist(), floats):
        if rec[0] == 0:
            continue
        if rec[1] in poses:
            raise ValueError(f"keyframe id {rec[1]} appears in two bundle-adjustment records")
        poses[rec[1]] = (f[11:15].clone(), f[15:18].clone())
    return poses


class TrackingSolver:
    """The reference's per-frame tracking loop (src/vtgaussian_slam.py:1794-1970) for one frame:
    num_iters x (get_loss(tracking=True) -> backward -> Adam on the 7 pose numbers), keeping
    the best pose by loss.  Gaussians are frozen (their tracking LRs are 0, configs/replica/room0.py:78-86).

    One iteration = 9 kernel launches, no host synchronisation; with use_graph the iteration is
    captured once and replayed.

    replica_sil_search: the reference's Replica branch (:472-510) -- at the FIRST iteration of a frame the silhouette
        threshold is chosen among {0.990 .. 0.999} by the masked colour MSE, on the device (one ladder kernel + a
        one-thread choice; 10 floats all-reduced when sharded), and kept for the frame's other iterations.
    ignore_outlier_depth_loss: the frame-wide median mask (:525-528); with a process group the radix-select
        histograms are all-reduced, so every rank uses the same median.
    book_post_step: keep the pose AFTER the step whose loss was the smallest (what the reference does, :1888-1970);
        False keeps the pose the loss was evaluated at."""

    LAUNCHES_PER_ITER = 9          # K1', scan, scatter, sort, K5', loss, K6', K7', update (+8 median launches with ignore_outlier_depth_loss)

    def __init__(self, settings, params, device="cuda:0", lr_rot=4e-4, lr_trans=2e-3, w_im=0.5, w_depth=0.025,
                 use_sil_for_loss=True, sil_thres=0.99, tile_rows=(0, 0), pair_capacity=None, use_graph=True,
                 process_group=None, ignore_outlier_depth_loss=False, far_depth_thres=0.0, replica_sil_search=False,
                 book_post_step=True, deterministic=None):
        self.device = torch.device(device)
        self.params = {k: params[k].detach().to(self.device).float().contiguous() for k in PARAM_KEYS}
        N = self.params["means3D"].shape[0]
        self.r = FusedRenderer(settings, N, device=self.device, tile_rows=tile_rows, pair_capacity=pair_capacity,
                               deterministic=deterministic)
        self.cfg = dict(w_im=w_im, w_depth=w_depth, use_sil_for_loss=use_sil_for_loss, sil_thres=sil_thres,
                        ignore_outlier_depth_loss=ignore_outlier_depth_loss, far_depth_thres=far_depth_thres)
        self.replica_sil_search = bool(replica_sil_search) and bool(use_sil_for_loss)
        self.flags = _lib.TRACK_BOOK_POST_STEP if book_post_step else 0
        self.lr_rot, self.lr_trans = lr_rot, lr_trans
        f32 = dict(dtype=torch.float32, device=self.device)
        self.cam_q = torch.tensor([1.0, 0, 0, 0], **f32)
        self.cam_t = torch.zeros(3, **f32)
        # gradient message of one iteration: d_q[4] d_t[3] pad loss_terms[8] -> 16 floats (all-reduced when sharded)
        self.msg = torch.zeros(16, **f32)
        self.d_q, self.d_t = self.msg[0:4], self.msg[4:7]
        self.r.loss_terms = self.msg[8:16]          # the loss kernel writes straight into the message
        self.adam = torch.zeros(14, **f32)                 # m_q[4] v_q[4] m_t[3] v_t[3]
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.best = torch.zeros(8, **f32)                  # best_loss, best_q[4], best_t[3]
        self.best[0] = float("inf")
        self.best_loss, self.best_q, self.best_t = self.best[0:1], self.best[1:5], self.best[5:8]
        self.gt_rgb = torch.zeros((3, self.r.H, self.r.W), **f32)
        self.gt_depth = torch.zeros((1, self.r.H, self.r.W), **f32)
        self.pg = process_group
        self.use_graph = use_graph
        self._graph = None
        self._graph0 = None              # the frame's first iteration when it differs (replica_sil_search)
        self._graph_generation = None    # the renderer's workspace generation the graphs were captured on
        self._it = 0                     # iterations since set_frame
        self._init = None

    def set_frame(self, gt_rgb, gt_depth, cam_q, cam_t):
        """New frame: targets, initial pose (e.g. constant-velocity propagated) and a fresh Adam
        state -- the reference re-creates its optimiser every frame (:1678-1758)."""
        self.gt_rgb.copy_(gt_rgb, non_blocking=True)
        self.gt_depth.copy_(gt_depth.reshape(self.gt_depth.shape), non_blocking=True)
        self._init = (torch.as_tensor(cam_q, dtype=torch.float32).reshape(4).clone(), torch.as_tensor(cam_t, dtype=torch.float32).reshape(3).clone())
        self._reset_pose()

    def _reset_pose(self):
        self.cam_q.copy_(self._init[0], non_blocking=True)
        self.cam_t.copy_(self._init[1], non_blocking=True)
        self.adam.zero_()
        self.step_dev.zero_()
        self.best.zero_()
        self.best[0] = float("inf")
        self._it = 0

    def _iteration(self, first=False):
        r = self.r
        r.forward(self.params, self.cam_q, self.cam_t)
        extra = {}
        if self.cfg["ignore_outlier_depth_loss"] and self.pg is not None:
            extra["median_state"] = r.median_state(gt_depth=self.gt_depth, process_group=self.pg)
        if self.replica_sil_search:
            if first:
                r.sil_ladder(self.gt_rgb, self.gt_depth, process_group=self.pg)
            extra["sil_thres_dev"] = r._sil[10:11]
        r.tracking_loss(self.gt_rgb, self.gt_depth, **self.cfg, **extra)
        r.backward(self.params, self.cam_q, self.cam_t, pose_grads=(self.d_q, self.d_t), dl_bound=r.loss_terms[6:7])
        if self.pg is not None:
            # tile-band sharding: every rank holds its band's partial sums; one 16-float all-reduce
            torch.distributed.all_reduce(self.msg, group=self.pg)
        # best-candidate bookkeeping (reference :1961-1970) + Adam on the 7 pose numbers, one launch
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().vtgs_tracking_update(_ptr(self.cam_q), _ptr(self.cam_t), _ptr(self.msg), _ptr(self.adam),
                                                       _ptr(self.step_dev), _ptr(self.best), float(self.lr_rot),
                                                       float(self.lr_trans), 1e-8, int(self.flags), _stream_ptr(self.device)))

    def _capture(self, first):
        # warm-up on a side stream, then capture; the solver state is restored around both
        s = torch.cuda.Stream(self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        state = (self.cam_q, self.cam_t, self.adam, self.step_dev, self.best)
        snap = [t.clone() for t in state]
        with torch.cuda.stream(s):
            self._iteration(first)
        torch.cuda.current_stream(self.device).wait_stream(s)
        for t, v in zip(state, snap):
            t.copy_(v)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._iteration(first)
        for t, v in zip(state, snap):
            t.copy_(v)
        return g

    def step(self):
        first = self._it == 0 and self.replica_sil_search
        self._it += 1
        if not self.use_graph:
            self._iteration(first)
            return
        if self._graph_generation != self.r.ws.generation:          # captured launches point into the pair buffers
            self._graph = self._graph0 = None
            self._graph_generation = self.r.ws.generation
        if first:
            if self._graph0 is None:
                self._graph0 = self._capture(True)
            self._graph0.replay()
            return
        if self._graph is None:
            if self.replica_sil_search and self.r._sil is None:
                self.r.sil_ladder(self.gt_rgb, self.gt_depth, process_group=self.pg)      # allocates the threshold the graph reads
            self._graph = self._capture(False)
        self._graph.replay()

    def loss_terms(self):
        return self.msg[8:16]

    def check(self, grow=True, raise_on_overflow=True):
        """One blocking read of the device counters (call once per frame, not per iteration).  If the pair buffers
        overflowed (R > pair_capacity: the renders of this frame were truncated) they are enlarged (grow=True; the
        captured graphs follow them at the next step); then either raises or returns None so that the caller re-runs the
        frame (`run_frame` does).  -> R otherwise."""
        overflow, R = self.r.overflowed()
        if overflow:
            if grow:
                self.r.ws.reserve_pairs(grown_pair_capacity(R))
            if raise_on_overflow:
                raise _lib.VtgsError(f"pair buffer overflow: R = {R} > capacity; buffers "
                                     f"{'were grown -- re-run the frame' if grow else 'unchanged'}")
            return None
        return R

    def run_frame(self, num_iters):
        """num_iters iterations from the pose given to set_frame, one blocking read of the result, and -- if the pair
        buffers turned out too small for this frame -- a transparent re-run with larger ones.
        -> best[8] on the host: (best loss, best cam_unnorm_rot[4], best cam_trans[3])."""
        return self.run_frame_with_metric(num_iters, None)

    def run_frame_with_metric(self, num_iters, metric_fn):
        """run_frame with the reference's `choose_metric` of a section's base frame (:1891-1970): after every Adam step
        `metric_fn(cam_unnorm_rot[4], cam_trans[3])` (host tensors of the POST-step pose; e.g. the point-to-plane distance
        to the overlapping keyframe, keyframes.point2plane_dist) ranks the candidate, and the pose with the smallest
        metric is kept.  One blocking pose read per iteration -- the reference runs an Open3D KD-tree there.
        -> best[8] on the host: (best metric, cam_unnorm_rot[4], cam_trans[3])."""
        def frame():
            best = torch.full((8,), float("inf"))
            for _ in range(num_iters):
                self.step()
                if metric_fn is not None:
                    q, t = self.cam_q.cpu(), self.cam_t.cpu()
                    m = float(metric_fn(q, t))
                    if m < float(best[0]):
                        best[0] = m
                        best[1:5], best[5:8] = q, t
            return self.best.cpu() if metric_fn is None else best
        return run_fitting(frame, [self.r], on_regrow=self._reset_pose)


class MappingSolver:
    """The reference's mapping iteration (src/vtgaussian_slam.py:2525-2752) over a set of
    keyframes with the semantics of its all-keyframes branch (:2609-2666): sum of the
    per-keyframe losses, one backward, one Adam step over rgb / logit-opacity / log-scale
    (mapping LRs, configs/replica/room0.py:99-107; means3D and rotations have LR 0).

    Parameters that are already contiguous float32 CUDA tensors are updated IN PLACE (no copy is made).
    The mapping loss (0.8 L1 + 0.2 (1-SSIM) + depth L1 mean) runs in the library's SSIM kernels; an optional
    `loss_fn(image6, kf) -> (loss, dL_dimage4)` can replace it (e.g. slam_ops.mapping_loss_and_grad, the
    torch-autograd restatement used to check it).

    global_params: the reference's frozen-section term (`loss_global`, :2552, :2600, :2645): a second render of the same
        keyframe over the frozen earlier sections PLUS the trainable ones, added to the loss.  Pass the parameter
        tensors of that union with the trainable Gaussians LAST; when those last rows alias `params` (row views of one
        SectionStore arena) nothing is copied, otherwise the trainable rows are refreshed before every global render.
        The frozen rows get no update (their `fixed_lrs` are 0, configs/replica/room0.py:108-116).
    do_ba (per iteration): the keyframes' poses get gradients and an Adam step of their own (`do_ba`, :2545-2548; LRs
        `cam_unnorm_rots` / `cam_trans` of `lrs`); a keyframe carrying `retie_last=n` has the newest n Gaussians re-tied
        to its pose after the step (:2706-2727).
    do_ba with a process group: every keyframe needs an "id", an int unique across the ranks (e.g. its frame index); a
        rank steps at most BA_RECORDS_PER_RANK keyframes per iteration.  The owner of a keyframe steps its pose and writes
        a record (id, retie_last, old and new pose); the ranks exchange the records after the parameter step and every
        rank applies every re-tie, in (rank, keyframe) order, to its replica of means3D, so the replicas stay bitwise
        equal.  `ba_poses()` returns the poses all ranks stepped in the last such iteration."""

    def __init__(self, settings, params, device="cuda:0", lrs=None, eps=1e-15, pair_capacity=None, process_group=None,
                 global_params=None, poll_every=16, deterministic=None, sharded_step="auto"):
        self.device = torch.device(device)
        self.params = {k: params[k].detach().to(self.device).float().contiguous() for k in PARAM_KEYS}
        N = self.params["means3D"].shape[0]
        self.settings = settings
        self.deterministic = deterministic
        self.r = FusedRenderer(settings, N, device=self.device, pair_capacity=pair_capacity, deterministic=deterministic)
        self.lrs = dict(rgb_colors=0.0025, logit_opacities=0.05, log_scales=0.005) if lrs is None else dict(lrs)
        self.pose_lrs = (float(self.lrs.pop("cam_unnorm_rots", 0.0)), float(self.lrs.pop("cam_trans", 0.0)))
        self.lrs = {k: v for k, v in self.lrs.items() if k in PARAM_KEYS and v != 0.0}
        self.eps = eps
        # one flat gradient message (all learnable parameter gradients + the loss): a single all-reduce per step
        sizes = {k: self.params[k].numel() for k in self.lrs}
        self.flat = torch.zeros(sum(sizes.values()) + 1, dtype=torch.float32, device=self.device)
        self.grads, off = {}, 0
        for k, n in sizes.items():
            self.grads[k] = self.flat[off:off + n].view(self.params[k].shape)
            off += n
        self.m = {k: torch.zeros_like(self.params[k]) for k in self.lrs}
        self.v = {k: torch.zeros_like(self.params[k]) for k in self.lrs}
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.pg = process_group
        self.total_loss = self.flat[-1:]
        # keyframe shards: the step after the backward is ONE kernel over NVLink peer memory (reduce-scatter + Adam on
        # this rank's slice + all-gather of the new parameters, `vtgs_sharded_adam`) when torch's symmetric memory can
        # map the ranks' blocks into each other; otherwise one NCCL all-reduce followed by a replicated Adam
        self.sharded = None
        self.sharded_error = None
        world = torch.distributed.get_world_size(process_group) if process_group is not None else 1
        if world > 1 and sharded_step and os.environ.get("VTGS_SHARDED_STEP", "1") != "0":
            try:
                self._setup_sharded(sizes, world)
            except Exception as e:             # no peer mapping on this box: NCCL path
                if sharded_step is True:
                    raise
                self.sharded, self.sharded_error = None, repr(e)[:300]
        self.poll_every = int(poll_every)
        self._iters = 0
        self._ba_iters = 0                  # keyframe-sharded do_ba iterations: their parity picks the fused step's record table
        self._ba_mine = self._ba_tables = None
        self.gparams = self.r_global = self.ggrads = None
        if global_params is not None:
            self.set_global(global_params)

    @staticmethod
    def sharded_slices(n_pad, world):
        """Element ranges [begin, end) of the flat vectors that each rank owns in `vtgs_sharded_adam` (whole float4s,
        ceil-divided; trailing ranks may own less or nothing): the kernel's partition, restated for the host (sizing of
        the sharded moments, the 2-rank gloo test of the step's algorithm)."""
        n4 = n_pad // 4
        per = (n4 + world - 1) // world
        return [(4 * min(n4, per * r), 4 * min(n4, per * (r + 1))) for r in range(world)]

    def _setup_sharded(self, sizes, world):
        import torch.distributed._symmetric_memory as symm
        if world > 8:
            raise RuntimeError("vtgs_sharded_adam supports up to 8 ranks")
        n = sum(sizes.values())
        n_pad = (n + 3) // 4 * 4
        tab = BA_RECORDS_PER_RANK * _lib.BA_RECORD_WORDS
        block = symm.empty(2 * n_pad + 4 + 2 * tab, dtype=torch.float32, device=self.device)
        hdl = symm.rendezvous(block, self.pg)
        block.zero_()
        pflat, gflat = block[:n_pad], block[n_pad:2 * n_pad]
        off, seg_end = 0, []
        for k, cnt in sizes.items():
            view = pflat[off:off + cnt].view(self.params[k].shape)
            view.copy_(self.params[k])
            self.params[k] = view                       # the learnable parameters now live in the symmetric block
            self.grads[k] = gflat[off:off + cnt].view(self.params[k].shape)
            off += cnt
            seg_end.append(off)
        seg_end[-1] = n_pad
        rank = torch.distributed.get_rank(self.pg)
        per = max(e - b for b, e in self.sharded_slices(n_pad, world))
        self.flat = gflat                               # (kept for callers that time the plain all-reduce of the message)
        self.total_loss = block[2 * n_pad:2 * n_pad + 1]
        nseg = len(seg_end)
        self.sharded = dict(
            hdl=hdl, block=block, n=n_pad, world=world, rank=rank, nseg=nseg,
            mc=(int(getattr(hdl, "multicast_ptr", 0) or 0) if os.environ.get("VTGS_SHARDED_MULTICAST", "0") == "1" else 0),
            bases=(C.c_uint64 * world)(*[int(p_) for p_ in hdl.buffer_ptrs]),
            seg_end=(C.c_int64 * nseg)(*seg_end), lr=(C.c_float * nseg)(*[float(self.lrs[k]) for k in sizes]),
            m=torch.zeros(per, dtype=torch.float32, device=self.device), v=torch.zeros(per, dtype=torch.float32, device=self.device),
            loss=torch.zeros(1, dtype=torch.float32, device=self.device),
            # the bundle-adjustment record tables, double-buffered by the parity of the do_ba iteration.  A rank writes its
            # table before the step's first barrier and the peers read it after the second, with nothing ordering those
            # reads against the rank's next write; with two tables that write goes to the other one, and the write after
            # it comes behind the next step's barriers, which no peer reaches before its re-tie from this table is done
            ba=block[2 * n_pad + 4:].view(torch.int32).view(2, BA_RECORDS_PER_RANK, _lib.BA_RECORD_WORDS))
        self.m = self.v = None                          # the moments are sharded: this rank keeps its slice only
        torch.cuda.synchronize(self.device)
        hdl.barrier(channel=0)

    def _sharded_step(self):
        sh = self.sharded
        sh["hdl"].barrier(channel=0)                    # every rank's gradients are complete
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().vtgs_sharded_adam(sh["world"], sh["rank"], sh["bases"], sh["mc"], 0, sh["n"], 2 * sh["n"], _ptr(sh["m"]),
                                                    _ptr(sh["v"]), sh["n"], sh["nseg"], sh["seg_end"], sh["lr"], 0.9, 0.999,
                                                    float(self.eps), _ptr(self.step_dev), _ptr(sh["loss"]),
                                                    _stream_ptr(self.device)))
        sh["hdl"].barrier(channel=0)                    # every rank's new parameters have landed

    def _ba_step(self, keyframes, header):
        """Keyframe sharding, do_ba: the pose Adam steps of this rank's keyframes, each recorded (old and new pose) in this
        rank's table -> that table on the device."""
        if self.sharded is not None:
            table = self.sharded["ba"][self._ba_iters % 2]
        else:
            if self._ba_mine is None:
                self._ba_mine = torch.empty(header.shape, dtype=torch.int32, device=self.device)
            table = self._ba_mine
        table.copy_(header, non_blocking=True)
        poses = table.view(torch.float32)
        for s, kf in enumerate(keyframes):
            st = kf["_ba"]
            poses[s, 4:8].copy_(kf["cam_q"])
            poses[s, 8:11].copy_(kf["cam_t"])
            st["step"].add_(1)
            if self.pose_lrs[0] != 0.0:
                adam_step(kf["cam_q"], st["d_q"], st["m_q"], st["v_q"], self.pose_lrs[0], step_dev=st["step"], eps=self.eps)
            if self.pose_lrs[1] != 0.0:
                adam_step(kf["cam_t"], st["d_t"], st["m_t"], st["v_t"], self.pose_lrs[1], step_dev=st["step"], eps=self.eps)
            poses[s, 11:15].copy_(kf["cam_q"])
            poses[s, 15:18].copy_(kf["cam_t"])
        return table

    def _ba_retie(self, table):
        """Keyframe sharding, do_ba, after the parameter step: every rank's records reach every rank -- read from the peers'
        symmetric blocks (fused step) or one all-gather -- and `vtgs_retie_records` applies all their re-ties to this
        rank's means3D in (rank, slot) order, leaving the gathered tables in `_ba_tables`."""
        world = torch.distributed.get_world_size(self.pg)
        if self._ba_tables is None:
            self._ba_tables = torch.empty((world,) + tuple(table.shape), dtype=torch.int32, device=self.device)
        if self.sharded is not None:
            off = table.data_ptr() - self.sharded["block"].data_ptr()           # the same offset in every rank's block
            bases, out = (C.c_uint64 * world)(*[b + off for b in self.sharded["bases"]]), self._ba_tables
        else:
            torch.distributed.all_gather_into_tensor(self._ba_tables.view(-1, table.shape[1]), table, group=self.pg)
            bases, out = (C.c_uint64 * world)(*[self._ba_tables[r].data_ptr() for r in range(world)]), None
        means3D = self.params["means3D"]
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().vtgs_retie_records(world, bases, table.shape[0], _ptr(means3D), means3D.shape[0], _ptr(out),
                                                     _stream_ptr(self.device)))
        self._ba_iters += 1

    def ba_poses(self):
        """{id: (cam_q[4], cam_t[3])} on the host: the pose every rank's keyframe got in the last bundle-adjustment iteration
        under keyframe sharding, from this rank's gathered tables (one blocking read).  Raises ValueError if an id appears
        twice among the ranks."""
        if self._ba_tables is None:
            raise RuntimeError("ba_poses: no do_ba iteration has run under a process group")
        return decode_ba_poses(self._ba_tables.cpu())

    def set_global(self, global_params):
        gp = {k: global_params[k].detach().to(self.device).float().contiguous() for k in PARAM_KEYS}
        N, Ng = self.params["means3D"].shape[0], gp["means3D"].shape[0]
        if Ng < N:
            raise ValueError("global_params must hold the frozen sections followed by the trainable Gaussians")
        self.gparams = gp
        self._global_aliases = all(gp[k][Ng - N:].data_ptr() == self.params[k].data_ptr() for k in PARAM_KEYS)
        self.r_global = FusedRenderer(self.settings, Ng, device=self.device, deterministic=self.deterministic)
        self.ggrads = {k: torch.zeros_like(gp[k]) for k in self.lrs}

    def _render_backward(self, r, params, kf, grads, accumulate, loss_fn, w_im, w_depth, pose):
        img, _ = r.forward(params, kf["cam_q"], kf["cam_t"])
        if loss_fn is None:
            loss, dL4 = r.mapping_loss(kf["gt_rgb"], kf["gt_depth"], w_im=w_im, w_depth=w_depth)[0:1], None
        else:
            loss, dL4 = loss_fn(img, kf)
        self.total_loss += loss
        r.backward(params, kf["cam_q"], kf["cam_t"], dL_dimage4=dL4, param_grads=grads, pose_grads=pose, accumulate=accumulate)

    def _gradients(self, keyframes, loss_fn, w_im, w_depth, do_ba):
        """Loss and gradients of one iteration over `keyframes`, nothing updated yet: repeatable."""
        self.total_loss.zero_()
        first = True
        for kf in keyframes:
            pose = None
            if do_ba:
                st = kf.setdefault("_ba", None)
                if st is None:
                    z = lambda n: torch.zeros(n, dtype=torch.float32, device=self.device)
                    st = kf["_ba"] = dict(d_q=z(4), d_t=z(3), m_q=z(4), v_q=z(4), m_t=z(3), v_t=z(3), old_q=z(4), old_t=z(3),
                                          step=torch.zeros(1, dtype=torch.int32, device=self.device))
                pose = (st["d_q"], st["d_t"])
            self._render_backward(self.r, self.params, kf, self.grads, not first, loss_fn, w_im, w_depth, pose)
            first = False
            if self.r_global is not None and kf.get("global", True):
                N = self.params["means3D"].shape[0]
                if not self._global_aliases:
                    for k in PARAM_KEYS:
                        self.gparams[k][-N:].copy_(self.params[k])
                gpose = None
                if do_ba:
                    st = kf["_ba"]
                    gpose = (st.setdefault("gd_q", torch.zeros_like(st["d_q"])), st.setdefault("gd_t", torch.zeros_like(st["d_t"])))
                self._render_backward(self.r_global, self.gparams, kf, self.ggrads, False, loss_fn, w_im, w_depth, gpose)
                for k in self.lrs:
                    self.grads[k] += self.ggrads[k][-N:]
                if do_ba:
                    st["d_q"] += st["gd_q"]
                    st["d_t"] += st["gd_t"]
        if first:
            for g in self.grads.values():
                g.zero_()

    def iteration(self, keyframes, loss_fn=None, w_im=1.0, w_depth=1.0, do_ba=False):
        """keyframes: list of dict(cam_q, cam_t, gt_rgb, gt_depth[, global=True][, retie_last=n][, id]) owned by THIS rank
        ("id" is required with do_ba and a process group).  loss_fn=None uses the fused mapping loss kernels
        (FusedRenderer.mapping_loss)."""
        # (a sharded do_ba iteration's keyframes are checked before anything is updated)
        ba_header = ba_record_table(keyframes, self.params["means3D"].shape[0]) if do_ba and self.pg is not None else None
        poll = self.poll_every > 0 and self._iters % self.poll_every == 0
        # the overflow check (one blocking read every `poll_every` iterations) comes before anything is updated
        run_fitting(lambda: self._gradients(keyframes, loss_fn, w_im, w_depth, do_ba),
                    [self.r] if self.r_global is None else [self.r, self.r_global], poll=poll)
        self._iters += 1
        self.step_dev.add_(1)
        # keyframe sharding: the pose steps come before the parameter step (they touch disjoint tensors), so that the fused
        # step's barriers publish the records
        ba_table = self._ba_step(keyframes, ba_header) if ba_header is not None else None
        if self.sharded is not None:
            self._sharded_step()
        else:
            if self.pg is not None:
                # keyframe sharding: ONE all-reduce (SUM) of the flat gradient message over NVLink (5 N fp32 + loss)
                torch.distributed.all_reduce(self.flat, group=self.pg)
            for k, lr in self.lrs.items():
                adam_step(self.params[k], self.grads[k], self.m[k], self.v[k], lr, step_dev=self.step_dev, eps=self.eps)
        if ba_table is not None:
            self._ba_retie(ba_table)
        elif do_ba:
            for kf in keyframes:
                st = kf["_ba"]
                n_last = int(kf.get("retie_last", 0))
                if n_last > 0:
                    st["old_q"].copy_(kf["cam_q"])
                    st["old_t"].copy_(kf["cam_t"])
                st["step"].add_(1)
                if self.pose_lrs[0] != 0.0:
                    adam_step(kf["cam_q"], st["d_q"], st["m_q"], st["v_q"], self.pose_lrs[0], step_dev=st["step"], eps=self.eps)
                if self.pose_lrs[1] != 0.0:
                    adam_step(kf["cam_t"], st["d_t"], st["m_t"], st["v_t"], self.pose_lrs[1], step_dev=st["step"], eps=self.eps)
                if n_last > 0:
                    # the section's newest Gaussians stay tied to the keyframe: pts <- c2w_new (w2c_old pts), :2706-2727
                    retie_dev(self.params["means3D"][-n_last:], st["old_q"], st["old_t"], kf["cam_q"], kf["cam_t"])
        return self.total_loss if self.sharded is None else self.sharded["loss"]
