"""A compact view-tied SLAM loop over the fused solvers: the caller side of the hot path (SURVEY.md 8(f) rows
N1/N2 in embryo, BASELINE config "TUM fr1_desk-shaped full tracking+mapping loop over synthetic frames").

What it mirrors of the reference's `rgbd_slam` (src/vtgaussian_slam.py:1574-2876), and what it leaves out:

  * sections ("base frames", :1620-1760): every `baseframe_every` frames a new set of view-tied Gaussians is
    built from that frame's RGB-D at its tracked pose -- `section_from_frame` follows get_pointcloud (:76-128:
    one Gaussian per valid pixel at ((x-cx+0.5)/fx z, (y-cy+0.5)/fy z, z), z = 1.005 depth, isotropic
    scale z / ((fx+fy)/2)) and initialize_params (:132-177: identity quaternions, logit opacity 0);
  * pose initialisation (:817-885): constant velocity, init_c2w = c2w[t-1] inv(c2w[t-2]) c2w[t-1];
  * tracking (:1794-1970): `track_iters` x (render -> masked L1 -> backward to the pose -> Adam), best pose by
    loss kept -- TrackingSolver, one CUDA graph replay per iteration;
  * mapping (:2525-2702): `map_iters` x (sum of keyframe losses -> backward -> Adam over rgb / opacity / scale of
    the current section) over the section's most recent keyframes -- MappingSolver.
  * section choice at a section's base frame (:1526-1553, :1891-1970; LoopConfig.section_selection = "overlap"): the
    earliest sections that still overlap the new frame (keyframes.keyframe_selection_overlap_visbased_earliest_dynamic_
    new_topkbase) are rendered together with the newest one, candidates ranked by the device point-to-plane metric;
  * silhouette-driven Gaussian addition (:732-813): add_missing_gaussians.
  Left out (not on the hot path, SURVEY.md 8 "out of scope" / later rows): edge-mask densification on the 2x grid inside
  the loop (densified_section builds such a section), the frozen-section loss inside the loop (MappingSolver has it),
  checkpoints.

Everything on the device runs through the CUDA library; there is no CPU fallback.
"""
from __future__ import annotations

import time
from dataclasses import dataclass, field

import numpy as np
import torch

from .fused import MappingSolver, TrackingSolver
from .rasterizer import GaussianRasterizationSettings, run_fitting
from . import synthetic


@dataclass
class LoopConfig:
    track_iters: int = 40                 # configs/replica/room0.py:62 uses 60 (BASELINE quotes 40); fr1_config.py:63 uses 200
    map_iters: int = 15                   # room0.py:89 100, fr1_config.py:80 30
    baseframe_every: int = 10             # fr1_config.py:36 30
    map_every: int = 5
    keyframes_per_map: int = 4
    track_sections: int = 1               # track against the newest k sections (consecutive rows of the SectionStore);
                                          # k > 1 renders overlapping sections together and tracks less tightly
    lr_rot: float = 4e-4                  # room0.py:78-86
    lr_trans: float = 2e-3
    track_w_im: float = 0.5
    track_w_depth: float = 1.0            # fr1_config.py:66 (Replica: 0.025... see DESIGN.md)
    sil_thres: float = 0.99
    map_w_im: float = 1.0
    map_w_depth: float = 1.0
    map_lrs: dict = field(default_factory=lambda: dict(rgb_colors=0.0025, logit_opacities=0.05, log_scales=0.005))
    use_graph: bool = True
    # -- section choice at a section's base frame (reference :1526-1553, :1891-1970; `onlybase_overlap` configs) --
    section_selection: str = "latest"     # "overlap": the first frame of a new section is tracked against the EARLIEST
                                          # sections that still overlap it (visibility-based, dynamic threshold) plus
                                          # the newest one, which ties the new section to old geometry instead of
                                          # chaining it to the drift of its predecessor
    overlap_every: int = 5                # a keyframe (pose + depth) is kept every this many frames (fr1_config.py:38)
    kf_depth_thresh: float = 0.01         # fr1_config.py tracking.kf_depth_thresh
    earliest_thres: float = 0.5
    lower_earliest_thres_percent: float = 0.8
    topk_base: int = 3
    base_metric: str = "loss"             # "p2p": rank the base frame's candidate poses by the point-to-plane distance
                                          # to the earliest overlapping section's base frame (reference choose_metric)
    p2p_method: str = "sum"


def quat_from_matrix(R):
    """Unit quaternion (w, x, y, z) of a 3x3 rotation (numerically safe branch selection)."""
    R = np.asarray(R, np.float64)
    tr = np.trace(R)
    if tr > 0:
        s = np.sqrt(tr + 1.0) * 2
        q = [0.25 * s, (R[2, 1] - R[1, 2]) / s, (R[0, 2] - R[2, 0]) / s, (R[1, 0] - R[0, 1]) / s]
    else:
        i = int(np.argmax(np.diag(R)))
        j, k = (i + 1) % 3, (i + 2) % 3
        s = np.sqrt(1.0 + R[i, i] - R[j, j] - R[k, k]) * 2
        q = [0.0] * 4
        q[0] = (R[k, j] - R[j, k]) / s
        q[1 + i] = 0.25 * s
        q[1 + j] = (R[j, i] + R[i, j]) / s
        q[1 + k] = (R[k, i] + R[i, k]) / s
    q = np.asarray(q)
    return q / np.linalg.norm(q) * (1.0 if q[0] >= 0 else -1.0)


def matrix_from_quat(q, t):
    """4x4 [R(q/|q|) | t] (the reference's build_rotation, utils/slam_external.py:25-42)."""
    w, x, y, z = np.asarray(q, np.float64) / np.linalg.norm(q)
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                  [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                  [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
    M = np.eye(4)
    M[:3, :3] = R
    M[:3, 3] = np.asarray(t, np.float64)
    return M


def propagate_pose(w2c_prev1, w2c_prev2):
    """Constant-velocity initial guess (reference initialize_camera_pose, :838-875)."""
    c1, c2 = np.linalg.inv(w2c_prev1), np.linalg.inv(w2c_prev2)
    return np.linalg.inv(c1 @ np.linalg.inv(c2) @ c1)


def geometric_edge_mask(image_hwc, dilate=True, rgb=True):
    """uint8[H,W] edge mask (255 on edges) of an HxWx3 image in 0..255: Canny (50 / 200, aperture 3, L2 gradient) on
    the grey image cast to uint8, optionally dilated 3x3 -- the reference's densification mask
    (src/vtgaussian_slam.py:1022-1041, computed once from the first frame, :1287-1289)."""
    import cv2
    grey = cv2.cvtColor(np.asarray(image_hwc), cv2.COLOR_RGB2GRAY if rgb else cv2.COLOR_BGR2GRAY)
    if grey.dtype != np.uint8:
        grey = grey.astype(np.uint8)
    edges = cv2.Canny(grey, threshold1=50, threshold2=200, apertureSize=3, L2gradient=True)
    return cv2.dilate(edges, np.ones((3, 3), np.uint8), iterations=1) if dilate else edges


def densified_section(rgb, depth, K, rgb_dense, depth_dense, K_dense, c2w, edge_mask, device, factor=1.005):
    """A section as the reference builds it at a base frame when a densification dataset is configured
    (initialize_params_base_timestep, :285-345): every valid pixel of the tracking-resolution frame, followed by the
    pixels of the denser frame (the same view at 2x resolution) that lie on `edge_mask` (any resolution: resized
    with nearest neighbour to the dense grid) and have valid depth.  The dense Gaussians are half as wide
    (scale = z / f of the dense intrinsics)."""
    import cv2
    Hd, Wd = depth_dense.shape[-2:]
    m = cv2.resize(np.asarray(edge_mask), (Wd, Hd), interpolation=cv2.INTER_NEAREST).astype(np.bool_)
    base = section_from_frame(rgb, depth, K, c2w, device, factor)
    dense = section_from_frame(rgb_dense, depth_dense, K_dense, c2w, device, factor,
                               pixel_mask=torch.as_tensor(m.reshape(-1), device=device))
    return {k: torch.cat((base[k], dense[k]), dim=0).contiguous() for k in base}


def section_from_frame(rgb, depth, K, c2w, device, factor=1.005, pixel_mask=None):
    """View-tied Gaussians of one RGB-D frame in the world frame (reference get_pointcloud + initialize_params).
    rgb[3,H,W], depth[1,H,W] tensors; pixels with depth <= 0 (and, if given, outside the flat bool `pixel_mask`)
    are dropped."""
    H, W = depth.shape[-2:]
    fx, fy, cx, cy = float(K[0][0]), float(K[1][1]), float(K[0][2]), float(K[1][2])
    f32 = dict(dtype=torch.float32, device=device)
    xx = ((torch.arange(W, **f32) - cx + 0.5) / fx).repeat(H)
    yy = ((torch.arange(H, **f32) - cy + 0.5) / fy).repeat_interleave(W)
    z = depth.reshape(-1).to(**f32) * factor
    keep = z > 0
    if pixel_mask is not None:
        keep = keep & pixel_mask.reshape(-1).to(device)
    pts = torch.stack((xx * z, yy * z, z), -1)
    M = torch.as_tensor(np.asarray(c2w, np.float32), device=device)
    pts = pts @ M[:3, :3].T + M[:3, 3]
    cols = rgb.to(**f32).reshape(3, -1).T
    scale = z / ((fx + fy) / 2.0)
    n = int(keep.sum().item())
    rots = torch.zeros((n, 4), **f32)
    rots[:, 0] = 1.0
    return dict(means3D=pts[keep].contiguous(), rgb_colors=cols[keep].contiguous(), unnorm_rotations=rots,
                logit_opacities=torch.zeros((n, 1), **f32), log_scales=torch.log(scale[keep])[:, None].contiguous())


class SectionStore:
    """Device arena of view-tied sections: one SoA buffer per parameter, every section a contiguous row range.
    Consecutive sections are therefore rendered, tracked against and optimised IN PLACE through row-slice views --
    the reference concatenates the selected sections' tensors on every iteration and splits them back afterwards
    (src/vtgaussian_slam.py:2734, :2832-2839)."""

    KEYS = dict(means3D=3, rgb_colors=3, unnorm_rotations=4, logit_opacities=1, log_scales=1)

    def __init__(self, capacity, device="cuda:0"):
        self.device = torch.device(device)
        self.capacity = int(capacity)
        self.buf = {k: torch.empty((self.capacity, c), dtype=torch.float32, device=self.device) for k, c in self.KEYS.items()}
        self.offsets = [0]                 # section i owns rows [offsets[i], offsets[i + 1])

    def __len__(self):
        return len(self.offsets) - 1

    @property
    def num_gaussians(self):
        return self.offsets[-1]

    def _grow(self, need):
        cap = max(need, 2 * self.capacity)
        for k, c in self.KEYS.items():
            nb = torch.empty((cap, c), dtype=torch.float32, device=self.device)
            nb[:self.offsets[-1]] = self.buf[k][:self.offsets[-1]]
            self.buf[k] = nb
        self.capacity = cap

    def append(self, params):
        """Copy a section's parameters to the end of the arena -> its index.  (Views handed out before a growth of
        the arena keep pointing at the old storage: take them again after appending.)"""
        n = int(params["means3D"].shape[0])
        a = self.offsets[-1]
        if a + n > self.capacity:
            self._grow(a + n)
        for k in self.KEYS:
            self.buf[k][a:a + n] = params[k].to(self.device, torch.float32).reshape(n, self.KEYS[k])
        self.offsets.append(a + n)
        return len(self) - 1

    def extend_last(self, params):
        """Append Gaussians to the NEWEST section (it ends the arena, so its row range simply grows): the
        silhouette-driven additions of the reference's add_new_gaussians_base_frame (src/vtgaussian_slam.py:791-798
        concatenates them to the current parameter tensors).  Views taken before must be taken again."""
        n = int(params["means3D"].shape[0])
        a = self.offsets[-1]
        if a + n > self.capacity:
            self._grow(a + n)
        for k in self.KEYS:
            self.buf[k][a:a + n] = params[k].to(self.device, torch.float32).reshape(n, self.KEYS[k])
        self.offsets[-1] = a + n
        return n

    def rows(self, first, last=None):
        """Contiguous row-slice views (no copy) of sections first..last inclusive."""
        last = first if last is None else last
        a, b = self.offsets[first], self.offsets[last + 1]
        return {k: v[a:b] for k, v in self.buf.items()}


    def gather(self, indices):
        """Parameters of the listed sections as one contiguous set: row-slice views when the sections are consecutive
        (no copy), otherwise one concatenated copy (what the reference does on every iteration, :2734)."""
        idx = sorted(set(int(i) for i in indices))
        if not idx:
            raise ValueError("no section selected")
        if idx == list(range(idx[0], idx[-1] + 1)):
            return self.rows(idx[0], idx[-1])
        return {k: torch.cat([v[self.offsets[i]:self.offsets[i + 1]] for i in idx], dim=0) for k, v in self.buf.items()}


def ate_rmse(est_c2w, gt_c2w):
    """Translation RMSE between two trajectories that share their first pose (no alignment: both are relative to frame 0)."""
    e = np.asarray(est_c2w)[:, :3, 3] - np.asarray(gt_c2w)[:, :3, 3]
    return float(np.sqrt((e ** 2).sum(-1).mean()))


class ViewTiedSLAM:
    """frames: dicts with 'im'[3,H,W], 'depth'[1,H,W] (numpy or tensors), optional 'c2w' ground truth."""

    def __init__(self, W, H, K, cfg: LoopConfig | None = None, device="cuda:0"):
        self.W, self.H, self.K = int(W), int(H), np.asarray(K, np.float64)
        self.cfg = cfg or LoopConfig()
        self.device = torch.device(device)
        s = synthetic.setup_camera(self.W, self.H, self.K, np.eye(4))
        t = lambda a: torch.as_tensor(a, dtype=torch.float32, device=self.device)
        self.settings = GaussianRasterizationSettings(
            image_height=s["image_height"], image_width=s["image_width"], tanfovx=s["tanfovx"], tanfovy=s["tanfovy"],
            bg=t(s["bg"]), scale_modifier=s["scale_modifier"], viewmatrix=t(s["viewmatrix"]), projmatrix=t(s["projmatrix"]),
            sh_degree=0, campos=t(s["campos"]), prefiltered=False)
        self.w2c = []                      # estimated poses, one 4x4 per frame
        self.sections = []                 # dict(params (arena views), index, base, keyframes=[(idx, rgb, depth)])
        self.store = None                  # SectionStore, created with the first section
        self.tracker = None
        self.mapper = None
        if self.cfg.section_selection == "overlap" and self.cfg.baseframe_every % self.cfg.overlap_every != 0:
            raise ValueError("overlap-driven section choice needs baseframe_every to be a multiple of overlap_every")
        self.keyframe_list = []            # every `overlap_every` frames: dict(id, est_w2c, depth) for the section choice
        self.section_choices = []          # per base frame: the sections it was tracked against
        self.stats = dict(track_iters=0, map_iters=0, track_s=0.0, map_s=0.0, track_loss=[])

    # -- sections -------------------------------------------------------------------------------------------
    def _new_section(self, idx, rgb, depth):
        c2w = np.linalg.inv(self.w2c[idx])
        fresh = section_from_frame(rgb, depth, self.K, c2w, self.device)
        if self.store is None:
            self.store = SectionStore(4 * fresh["means3D"].shape[0], self.device)
        k = self.store.append(fresh)
        sec = dict(params=self.store.rows(k), index=k, base=idx, keyframes=[])
        self.sections.append(sec)
        for s_ in self.sections:                         # the arena may have moved: refresh every view
            s_["params"] = self.store.rows(s_["index"])
        c = self.cfg
        # the solvers alias the arena rows (contiguous float32 CUDA row slices are used in place): mapping updates the
        # newest section where it lives, and the tracker -- over the newest `track_sections` consecutive sections --
        # sees them without a copy
        self.mapper = MappingSolver(self.settings, sec["params"], device=self.device, lrs=c.map_lrs)
        first = max(0, k - max(1, c.track_sections) + 1)
        self.tracker = TrackingSolver(self.settings, self.store.rows(first, k), device=self.device, lr_rot=c.lr_rot,
                                      lr_trans=c.lr_trans, w_im=c.track_w_im, w_depth=c.track_w_depth,
                                      sil_thres=c.sil_thres, use_graph=c.use_graph)
        return sec

    def add_missing_gaussians(self, idx, rgb, depth, sil_thres=0.5):
        """Silhouette-driven Gaussian addition (reference add_new_gaussians_base_frame, src/vtgaussian_slam.py:732-813):
        a forward-only fused render of the tracked sections from frame idx's pose, the non-presence mask
        (silhouette < sil_thres, or rendered depth behind the measurement by more than 50x the median depth error) in one
        kernel, and one new view-tied Gaussian per masked valid-depth pixel appended to the newest section.
        -> number of Gaussians added.  (The reference's second, 2x-resolution pass over the Canny edge mask is what
        densified_section builds at a section start.)"""
        tr = self.tracker
        M = self.w2c[idx]
        q = torch.as_tensor(quat_from_matrix(M[:3, :3]), dtype=torch.float32, device=self.device)
        t = torch.as_tensor(M[:3, 3], dtype=torch.float32, device=self.device)
        run_fitting(lambda: tr.r.forward(tr.params, q, t), [tr.r])
        mask, count = tr.r.nonpresence_mask(depth, sil_thres=sil_thres)
        if int(count.item()) == 0:
            return 0
        keep = mask.bool() & (depth[0] > 0)
        if not bool(keep.any()):
            return 0
        fresh = section_from_frame(rgb, depth, self.K, np.linalg.inv(M), self.device, pixel_mask=keep)
        n = self.store.extend_last(fresh)
        k = len(self.store) - 1
        for s_ in self.sections:
            s_["params"] = self.store.rows(s_["index"])
        c = self.cfg
        self.mapper = MappingSolver(self.settings, self.sections[-1]["params"], device=self.device, lrs=c.map_lrs)
        first = max(0, k - max(1, c.track_sections) + 1)
        self.tracker = TrackingSolver(self.settings, self.store.rows(first, k), device=self.device, lr_rot=c.lr_rot,
                                      lr_trans=c.lr_trans, w_im=c.track_w_im, w_depth=c.track_w_depth,
                                      sil_thres=c.sil_thres, use_graph=c.use_graph)
        return n

    def _keyframe(self, sec, idx, rgb, depth):
        sec["keyframes"].append((idx, rgb, depth))

    def _map(self, sec):
        c = self.cfg
        kfs = []
        chosen = [sec["keyframes"][0]] + sec["keyframes"][1:][-(c.keyframes_per_map - 1):] if c.keyframes_per_map > 1 else sec["keyframes"][-1:]
        for idx, rgb, depth in chosen:
            M = self.w2c[idx]
            kfs.append(dict(cam_q=torch.as_tensor(quat_from_matrix(M[:3, :3]), dtype=torch.float32, device=self.device),
                            cam_t=torch.as_tensor(M[:3, 3], dtype=torch.float32, device=self.device),
                            gt_rgb=rgb, gt_depth=depth))
        t0 = time.perf_counter()
        for _ in range(c.map_iters):
            self.mapper.iteration(kfs, w_im=c.map_w_im, w_depth=c.map_w_depth)
        torch.cuda.synchronize(self.device)
        self.stats["map_s"] += time.perf_counter() - t0
        self.stats["map_iters"] += c.map_iters * len(kfs)

    # -- tracking -------------------------------------------------------------------------------------------
    def _track(self, idx, rgb, depth):
        c = self.cfg
        init = propagate_pose(self.w2c[idx - 1], self.w2c[idx - 2]) if idx >= 2 else self.w2c[idx - 1].copy()
        tr = self.tracker
        tr.set_frame(rgb, depth, quat_from_matrix(init[:3, :3]).astype(np.float32), init[:3, 3].astype(np.float32))
        t0 = time.perf_counter()
        # the +1 evaluates (and books) the pose of the last Adam step; one blocking read per frame; a frame whose pair
        # buffers turned out too small is re-run with larger ones (TrackingSolver.run_frame)
        best = tr.run_frame(c.track_iters + 1).numpy()
        self.stats["track_s"] += time.perf_counter() - t0
        self.stats["track_iters"] += c.track_iters + 1
        self.stats["track_loss"].append(float(best[0]))
        return matrix_from_quat(best[1:5], best[5:8])

    def _track_base_frame(self, idx, rgb, depth):
        """First frame of a new section with section_selection == "overlap": choose the sections to track against by
        their visibility-based overlap with this frame at its propagated pose (reference :1526-1553:
        keyframe_selection_overlap_visbased_earliest_dynamic_new_topkbase over the keyframes of all finished sections but
        the tail of the newest; the earliest one alone while there are at most two sections), render them together
        (zero-copy when consecutive, one gather otherwise) and, with base_metric == "p2p", keep the candidate pose
        with the smallest point-to-plane distance to the earliest chosen section's base frame (:1891-1970)."""
        from . import keyframes as kfsel
        c = self.cfg
        init = propagate_pose(self.w2c[idx - 1], self.w2c[idx - 2]) if idx >= 2 else self.w2c[idx - 1].copy()
        per_section = max(1, int(c.baseframe_every / c.overlap_every))
        n_sections = len(self.store)
        kfs = self.keyframe_list[:len(self.keyframe_list) - per_section + 1] if per_section > 1 else self.keyframe_list
        Kt = torch.as_tensor(self.K[:3, :3], dtype=torch.float32, device=self.device)
        w2c_t = torch.as_tensor(init, dtype=torch.float32, device=self.device)
        chosen = kfsel.keyframe_selection_overlap_visbased_earliest_dynamic_new_topkbase(
            depth, w2c_t, Kt, kfs, c.topk_base, dict(baseframe_every=c.baseframe_every, overlap_every=c.overlap_every),
            kf_depth_thresh=c.kf_depth_thresh, earliest_thres=c.earliest_thres,
            lower_earliest_thres_percent=c.lower_earliest_thres_percent, topk_base=None if n_sections <= 2 else c.topk_base)
        chosen = [s_ for s_ in chosen if s_ < n_sections]
        sel = sorted(set(chosen) | {n_sections - 1})
        self.section_choices.append((idx, sel))
        tr = TrackingSolver(self.settings, self.store.gather(sel), device=self.device, lr_rot=c.lr_rot, lr_trans=c.lr_trans,
                            w_im=c.track_w_im, w_depth=c.track_w_depth, sil_thres=c.sil_thres, use_graph=c.use_graph)
        tr.set_frame(rgb, depth, quat_from_matrix(init[:3, :3]).astype(np.float32), init[:3, 3].astype(np.float32))
        t0 = time.perf_counter()
        if c.base_metric == "p2p":
            anchor = next(k for k in self.keyframe_list if k["id"] == self.sections[sel[0]]["base"])
            metric = lambda q, t: kfsel.point2plane_dist(anchor["depth"], depth, self.K[:3, :3], anchor["est_w2c"],
                                                         matrix_from_quat(q.numpy(), t.numpy()), method=c.p2p_method)
            best = tr.run_frame_with_metric(c.track_iters, metric).numpy()
        else:
            best = tr.run_frame(c.track_iters + 1).numpy()
        self.stats["track_s"] += time.perf_counter() - t0
        self.stats["track_iters"] += c.track_iters + (0 if c.base_metric == "p2p" else 1)
        self.stats["track_loss"].append(float(best[0]))
        return matrix_from_quat(best[1:5], best[5:8])

    # -- driver ---------------------------------------------------------------------------------------------
    def process(self, frame):
        idx = len(self.w2c)
        rgb = torch.as_tensor(frame["im"], dtype=torch.float32).to(self.device, non_blocking=True).contiguous()
        depth = torch.as_tensor(frame["depth"], dtype=torch.float32).to(self.device, non_blocking=True).reshape(1, self.H, self.W).contiguous()
        c = self.cfg
        if idx == 0:
            self.w2c.append(np.eye(4))
        elif c.section_selection == "overlap" and idx % c.baseframe_every == 0 and self.keyframe_list:
            self.w2c.append(self._track_base_frame(idx, rgb, depth))
        else:
            self.w2c.append(self._track(idx, rgb, depth))
        if c.section_selection == "overlap" and idx % c.overlap_every == 0:
            self.keyframe_list.append(dict(id=idx, est_w2c=torch.as_tensor(self.w2c[idx], dtype=torch.float32, device=self.device),
                                           depth=depth))
        if idx % c.baseframe_every == 0:
            sec = self._new_section(idx, rgb, depth)
            self._keyframe(sec, idx, rgb, depth)
            self._map(sec)
        elif idx % c.map_every == 0:
            sec = self.sections[-1]
            self._keyframe(sec, idx, rgb, depth)
            self._map(sec)
        return self.w2c[-1]

    def run(self, frames):
        for fr in frames:
            self.process(fr)
        return np.stack([np.linalg.inv(m) for m in self.w2c])


# ---- results in the reference's on-disk form (src/vtgaussian_slam.py:2868-2876: np.save of the list of per-section
# parameter dicts, an object array of CPU tensors) -- so the reference's evaluation scripts can read a run of this loop
def export_params_ls(path, store, w2c_list):
    """Write `params_ls.npy`: one dict per section with the five Gaussian tensors plus the whole estimated
    trajectory as cam_unnorm_rots[1,4,T] / cam_trans[1,3,T] (relative w2c per frame, as initialize_params lays
    them out, :166-170)."""
    T = len(w2c_list)
    rots = torch.zeros((1, 4, T), dtype=torch.float32)
    trans = torch.zeros((1, 3, T), dtype=torch.float32)
    for i, M in enumerate(w2c_list):
        M = np.asarray(M, np.float64)
        rots[0, :, i] = torch.as_tensor(quat_from_matrix(M[:3, :3]), dtype=torch.float32)
        trans[0, :, i] = torch.as_tensor(M[:3, 3], dtype=torch.float32)
    out = []
    for k in range(len(store)):
        d = {name: t.detach().cpu().clone() for name, t in store.rows(k).items()}
        d["cam_unnorm_rots"], d["cam_trans"] = rots.clone(), trans.clone()
        out.append(d)
    np.save(path, np.array(out, dtype=object), allow_pickle=True)
    return path


def import_params_ls(path, device="cpu"):
    """Read a `params_ls.npy` (this loop's or the reference's) -> (SectionStore, list of 4x4 w2c of the trajectory
    stored with the LAST section)."""
    sections = list(np.load(path, allow_pickle=True))
    if not sections:
        raise ValueError(f"{path}: no sections")
    as_t = lambda v: v if isinstance(v, torch.Tensor) else torch.as_tensor(np.asarray(v))
    total = sum(int(as_t(s["means3D"]).shape[0]) for s in sections)
    store = SectionStore(max(total, 1), device)
    for s in sections:
        p = {k: as_t(s[k]).float() for k in SectionStore.KEYS}
        if p["log_scales"].dim() == 1:
            p["log_scales"] = p["log_scales"][:, None]
        if p["log_scales"].shape[1] != 1:
            raise NotImplementedError("anisotropic sections (log_scales [N,3]) are not stored by SectionStore")
        if p["logit_opacities"].dim() == 1:
            p["logit_opacities"] = p["logit_opacities"][:, None]
        store.append(p)
    last = sections[-1]
    rots, trans = as_t(last["cam_unnorm_rots"]).float(), as_t(last["cam_trans"]).float()
    w2c = [matrix_from_quat(rots[0, :, i].numpy(), trans[0, :, i].numpy()) for i in range(rots.shape[-1])]
    return store, w2c
