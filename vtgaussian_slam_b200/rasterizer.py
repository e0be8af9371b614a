"""Drop-in replacement of the reference's `diff_gaussian_rasterization` Python surface.

Mirrors what VTGaussian-SLAM imports and calls (reference src/vtgaussian_slam.py:38,461,466,747;
utils/recon_helpers.py:2,14-26; utils/eval_helpers.py:17,240,247,431,443):

    GaussianRasterizationSettings(image_height, image_width, tanfovx, tanfovy, bg, scale_modifier,
                                  viewmatrix, projmatrix, sh_degree, campos, prefiltered)
    GaussianRasterizer(raster_settings)(means3D, means2D, opacities, shs=None, colors_precomp=None,
                                        scales=None, rotations=None, cov3D_precomp=None)
        -> (color[3,H,W], radii[N] int32, depth[1,H,W])

Gradients flow to means3D, means2D (screen space), colors_precomp, opacities, scales, rotations;
none through radii / depth -- as in the reference's "-w-depth" rasteriser.  All compute is in
libvtgs_cuda.so through the C ABI of include/vtgs.h; there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import NamedTuple

import torch
from torch import nn

from . import _lib

_RADIUS_SIGMA_MULT = float(os.environ.get("VTGS_RADIUS_SIGMA_MULT", "3.0"))


def set_radius_sigma_mult(v: float):
    """The 3-sigma splat radius multiplier (the reference fork's 'smallerGSradii' delta is
    unknown offline; upstream value 3.0 is the default)."""
    global _RADIUS_SIGMA_MULT
    _RADIUS_SIGMA_MULT = float(v)
    _CAM_CACHE.clear()


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool


_CAM_CACHE: dict = {}


def camera_struct(s, tile_rows=(0, 0)) -> _lib.VtgsCamera:
    """VtgsCamera for a settings tuple (or a dict with the same keys).  The device->host read
    of the two matrices is cached per settings object (the reference builds its camera once
    per run, src/vtgaussian_slam.py:209)."""
    get = (lambda k: s[k]) if isinstance(s, dict) else (lambda k: getattr(s, k))
    vm, pm, bg = get("viewmatrix"), get("projmatrix"), get("bg")
    key = (id(vm), id(pm), id(bg), getattr(vm, "_version", 0), getattr(pm, "_version", 0), getattr(bg, "_version", 0),
           int(get("image_width")), int(get("image_height")), float(get("tanfovx")), float(get("tanfovy")),
           float(get("scale_modifier")), tuple(tile_rows), _RADIUS_SIGMA_MULT)
    hit = _CAM_CACHE.get(key)
    if hit is not None:
        return hit[0]
    cam = _lib.VtgsCamera()
    cam.image_width, cam.image_height = int(get("image_width")), int(get("image_height"))
    cam.tanfovx, cam.tanfovy = float(get("tanfovx")), float(get("tanfovy"))
    vmh = torch.as_tensor(vm).detach().float().reshape(-1).cpu().tolist()
    pmh = torch.as_tensor(pm).detach().float().reshape(-1).cpu().tolist()
    bgh = torch.as_tensor(bg).detach().float().reshape(-1).cpu().tolist()
    if len(vmh) != 16 or len(pmh) != 16 or len(bgh) != 3:
        raise ValueError("viewmatrix/projmatrix must have 16 elements and bg 3")
    cam.viewmatrix[:] = vmh
    cam.projmatrix[:] = pmh
    cam.bg[:] = bgh
    cam.scale_modifier = float(get("scale_modifier"))
    cam.radius_sigma_mult = _RADIUS_SIGMA_MULT
    cam.tile_row_begin, cam.tile_row_end = int(tile_rows[0]), int(tile_rows[1])
    if len(_CAM_CACHE) > 64:
        _CAM_CACHE.clear()
    _CAM_CACHE[key] = (cam, vm, pm, bg)      # keep the tensors alive so ids stay unique
    return cam


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


_DETERMINISTIC = os.environ.get("VTGS_DETERMINISTIC", "0") not in ("", "0")


def set_deterministic(on: bool):
    """Process-wide default of the backward's gradient accumulation (VTGS_BUF_DETERMINISTIC, include/vtgs.h): partial
    sums split onto exact power-of-two grids, bitwise reproducible run to run and across ranks, instead of plain fp32
    atomics whose result depends on their arrival order.
    Takes effect for workspaces whose own `deterministic` is None, at their next forward (captured CUDA graphs keep
    what they were captured with).  Also settable with the environment variable VTGS_DETERMINISTIC=1."""
    global _DETERMINISTIC
    _DETERMINISTIC = bool(on)


def _tensor_bytes(obj):
    return sum(t.nbytes for t in vars(obj).values() if isinstance(t, torch.Tensor))


class Workspace:
    """Device buffers of one forward (VtgsBuffers), owned as torch tensors and sized by `vtgs_workspace_query`.
    `generation` counts the reallocations of the pair buffers: what holds their addresses (a VtgsBuffers struct, a
    captured CUDA graph) is stale when it changes.  `grad_geom` must be zero on entry to a backward and is left zeroed by it."""

    def __init__(self, device, width, height, n, pair_capacity, deterministic=None):
        self.device, self.W, self.H, self.N = device, int(width), int(height), int(n)
        self.deterministic = deterministic                 # None: follow set_deterministic()
        sz = self._query(pair_capacity)
        u8 = dict(dtype=torch.uint8, device=device)
        self.tiles = (sz.tiles_x, sz.tiles_y)
        self.geom = torch.empty(sz.geom_bytes, **u8)
        self.tiles_touched = torch.empty(sz.tiles_touched_bytes // 4, dtype=torch.int32, device=device)
        self.tile_counts = torch.empty(sz.tile_counts_bytes // 4, dtype=torch.int32, device=device)
        self.tile_ranges = torch.empty((sz.tile_ranges_bytes // 8, 2), dtype=torch.int32, device=device)
        self.final_T = torch.empty((self.H, self.W), dtype=torch.float32, device=device)
        self.n_contrib = torch.empty((self.H, self.W), dtype=torch.int32, device=device)
        self.grad_geom = None
        self.counters = torch.zeros(sz.counters_bytes // 4, dtype=torch.int32, device=device)
        self.region_cnt = torch.zeros(sz.region_cnt_bytes // 4, dtype=torch.int32, device=device)
        self.region_done = torch.zeros(sz.region_done_bytes // 4, dtype=torch.int32, device=device)
        self.band_flags = torch.zeros(max(int(sz.band_flags_bytes), 1), dtype=torch.uint8, device=device)
        self.band_cand = torch.zeros(max(int(sz.band_cand_bytes) // 4, 1), dtype=torch.int32, device=device)
        self.tile_order = torch.zeros(max(int(sz.tile_order_bytes) // 4, 1), dtype=torch.int32, device=device)
        self.pair_keys = self.point_list = self.region_pairs = self.region_masks = None
        self.pair_capacity = self.generation = 0
        self.num_rendered = None                            # R of the last read_counters()
        self.reserve_pairs(pair_capacity)

    def _query(self, pair_capacity):
        sz = _lib.VtgsWorkspaceSizes()
        _lib.check(_lib.lib().vtgs_workspace_query(self.W, self.H, self.N, int(pair_capacity), C.byref(sz)))
        return sz

    def reserve_pairs(self, cap):
        cap = max(int(cap), 1)
        if cap > self.pair_capacity:
            sz = self._query(cap)
            self.pair_keys = torch.empty(sz.pair_keys_bytes // 8, dtype=torch.int64, device=self.device)
            self.point_list = torch.empty(sz.point_list_bytes // 4, dtype=torch.int32, device=self.device)
            self.region_pairs = torch.empty((sz.region_pairs_bytes // 8, 2), dtype=torch.int32, device=self.device)
            self.region_masks = torch.empty(sz.region_masks_bytes // 4, dtype=torch.int32, device=self.device)
            self.pair_capacity = cap
            self.generation += 1

    @property
    def nbytes(self):
        """Memory held by the workspace's tensors (a shared grad_geom included)."""
        return _tensor_bytes(self)

    def ensure_grad_geom(self):
        if self.grad_geom is None:
            self.grad_geom = torch.zeros((max(self.N, 1), _lib.GRAD_GEOM_FLOATS), dtype=torch.float32, device=self.device)
        return self.grad_geom

    def struct(self) -> _lib.VtgsBuffers:
        b = _lib.VtgsBuffers()
        b.geom = self.geom.data_ptr()
        b.tiles_touched = self.tiles_touched.data_ptr()
        b.tile_counts = self.tile_counts.data_ptr()
        b.tile_ranges = self.tile_ranges.data_ptr()
        b.pair_keys = self.pair_keys.data_ptr()
        b.point_list = self.point_list.data_ptr()
        b.final_T = self.final_T.data_ptr()
        b.n_contrib = self.n_contrib.data_ptr()
        b.grad_geom = self.ensure_grad_geom().data_ptr()
        b.counters = self.counters.data_ptr()
        b.region_pairs = self.region_pairs.data_ptr()
        b.region_cnt = self.region_cnt.data_ptr()
        b.region_masks = self.region_masks.data_ptr()
        b.region_done = self.region_done.data_ptr()
        b.pair_capacity = self.pair_capacity
        b.band_flags = self.band_flags.data_ptr()
        b.band_cand = self.band_cand.data_ptr()
        b.tile_order = self.tile_order.data_ptr()
        det = _DETERMINISTIC if self.deterministic is None else self.deterministic
        b.flags = _lib.BUF_DETERMINISTIC if det else 0
        return b

    def read_counters(self):
        """Blocking D2H read of (num_rendered, overflow, max_tile_pairs).  R / N also raises the device's estimate that
        sizes new pair buffers (initial_pair_capacity)."""
        c = self.counters[:3].cpu().tolist()
        R = self.num_rendered = int(c[0]) & 0xFFFFFFFF
        if self.N > 0:
            _PAIR_RATIO[self.device] = max(_PAIR_RATIO.get(self.device, 0.0), R / self.N)
        return R, int(c[1]), int(c[2])

    def ensure_capacity(self):
        """One blocking read of the device counters.  -> True if the last forward overflowed the pair buffers: they
        have been enlarged and the forward (and everything derived from it) must be repeated."""
        R, overflow, _ = self.read_counters()
        if overflow:
            self.reserve_pairs(grown_pair_capacity(R))
        return bool(overflow)


# grad_geom scratch is left zeroed by every backward: share one per (device, N)
_GRAD_GEOM_CACHE: dict = {}
# largest pairs-per-Gaussian ratio R / N read back on each device so far (it never decreases)
_PAIR_RATIO: dict = {}


def initial_pair_capacity(device, n):
    """Pair capacity of a new workspace for n Gaussians: the device's R / N estimate (view-tied sections: ~2 tiles per
    Gaussian) with head room.  A forward that still overflows is grown by ensure_capacity() and repeated."""
    return int(n * max(6.0, 1.5 * _PAIR_RATIO.get(torch.device(device), 0.0))) + 65536


def grown_pair_capacity(R):
    """Pair capacity after a forward that needed R pairs."""
    return int(R * 1.5) + 65536


def run_fitting(work, renderers, poll=True, on_regrow=None, attempts=3):
    """-> work(), run until its renders fit (a truncated render gives a wrong loss and wrong gradients without any
    error).  With `poll` each of `renderers` (a Workspace, a fused.FusedRenderer) reads its counters once after the run;
    if any overflowed, they grow, on_regrow() resets what the run advanced and work() runs again; VtgsError after `attempts`."""
    for _ in range(attempts):
        out = work()
        if not poll or not any([r.ensure_capacity() for r in renderers]):
            return out
        if on_regrow is not None:
            on_regrow()
    raise _lib.VtgsError("pair buffer overflow persisted after regrowing")


def _require_cuda(name, t):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: vtgaussian_slam_b200 has no CPU fallback")


def rasterize_forward(cam: _lib.VtgsCamera, means3D, scales, rotations, opacities, colors):
    """Raw (non-autograd) forward through the C ABI.  Returns (color, depth, radii, workspace)."""
    for n, t in (("means3D", means3D), ("scales", scales), ("rotations", rotations), ("opacities", opacities), ("colors", colors)):
        _require_cuda(n, t)
    dev = means3D.device
    N = means3D.shape[0]
    W, H = cam.image_width, cam.image_height
    f32 = lambda t: t.detach().contiguous().float()
    means3D, scales, rotations, opacities, colors = map(f32, (means3D, scales, rotations, opacities, colors))
    ws = Workspace(dev, W, H, N, initial_pair_capacity(dev, N))
    key = (dev, N)
    gg = _GRAD_GEOM_CACHE.get(key)
    if gg is None:
        if len(_GRAD_GEOM_CACHE) > 8:
            _GRAD_GEOM_CACHE.clear()
        gg = _GRAD_GEOM_CACHE[key] = torch.zeros((max(N, 1), _lib.GRAD_GEOM_FLOATS), dtype=torch.float32, device=dev)
    ws.grad_geom = gg
    color = torch.empty((3, H, W), dtype=torch.float32, device=dev)
    depth = torch.empty((1, H, W), dtype=torch.float32, device=dev)
    radii = torch.zeros(N, dtype=torch.int32, device=dev)
    L = _lib.lib()

    def forward():
        _lib.check(L.vtgs_forward(C.byref(cam), N, _ptr(means3D), _ptr(scales), _ptr(rotations), _ptr(opacities),
                                  _ptr(colors), _ptr(color), _ptr(depth), _ptr(radii), C.byref(ws.struct()), _stream_ptr(dev)))
    with torch.cuda.device(dev):
        # like the reference binding (one blocking D2H of num_rendered per forward): the drop-in API
        # polls every forward.  The fused path (fused.py) never synchronises inside an iteration.
        run_fitting(forward, [ws])
    ws.saved_inputs = (means3D, scales, rotations, opacities, colors)
    return color, depth, radii, ws


def rasterize_backward(cam: _lib.VtgsCamera, ws: Workspace, dL_dcolor):
    means3D, scales, rotations, opacities, colors = ws.saved_inputs
    dev, N = means3D.device, means3D.shape[0]
    dL = dL_dcolor.detach().contiguous().float()
    z = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
    g_m2d, g_col, g_op = z(N, 3), z(N, 3), z(N, 1)
    g_m3d, g_sc, g_rot = z(N, 3), z(N, 3), z(N, 4)
    b = ws.struct()
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().vtgs_backward(C.byref(cam), N, _ptr(means3D), _ptr(scales), _ptr(rotations), _ptr(opacities),
                                            _ptr(colors), _ptr(dL), _ptr(g_m2d), _ptr(g_col), _ptr(g_op), _ptr(g_m3d),
                                            _ptr(g_sc), _ptr(g_rot), C.byref(b), _stream_ptr(dev)))
    return g_m3d, g_m2d, g_col, g_op, g_sc, g_rot


class _RasterizeGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, colors_precomp, opacities, scales, rotations, raster_settings):
        cam = camera_struct(raster_settings)
        color, depth, radii, ws = rasterize_forward(cam, means3D, scales, rotations, opacities, colors_precomp)
        ctx.cam, ctx.ws = cam, ws
        ctx.shapes = (opacities.shape,)
        ctx.mark_non_differentiable(radii, depth)
        return color, radii, depth

    @staticmethod
    def backward(ctx, grad_color, _grad_radii, _grad_depth):
        g_m3d, g_m2d, g_col, g_op, g_sc, g_rot = rasterize_backward(ctx.cam, ctx.ws, grad_color)
        ctx.ws = None
        return g_m3d, g_m2d, g_col, g_op.reshape(ctx.shapes[0]), g_sc, g_rot, None


class GaussianRasterizer(nn.Module):
    def __init__(self, raster_settings):
        super().__init__()
        self.raster_settings = raster_settings

    def markVisible(self, positions):
        _require_cuda("positions", positions)
        with torch.no_grad():
            cam = camera_struct(self.raster_settings)
            p = positions.detach().contiguous().float()
            out = torch.zeros(p.shape[0], dtype=torch.uint8, device=p.device)
            with torch.cuda.device(p.device):
                _lib.check(_lib.lib().vtgs_mark_visible(C.byref(cam), p.shape[0], _ptr(p), _ptr(out), _stream_ptr(p.device)))
        return out.bool()

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                cov3D_precomp=None):
        if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
            raise Exception('Please provide excatly one of either SHs or precomputed colors!')
        if ((scales is None or rotations is None) and cov3D_precomp is None) or \
                ((scales is not None or rotations is not None) and cov3D_precomp is not None):
            raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')
        if shs is not None:
            raise NotImplementedError("SH colours are not on VTGaussian-SLAM's path (sh_degree=0, colors_precomp only)")
        if cov3D_precomp is not None:
            raise NotImplementedError("cov3D_precomp is not on VTGaussian-SLAM's path (scales + rotations only)")
        if colors_precomp.shape[-1] != 3:
            raise RuntimeError("colors_precomp must be [N,3] (NUM_CHANNELS = 3)")
        return _RasterizeGaussians.apply(means3D, means2D, colors_precomp, opacities, scales, rotations, self.raster_settings)
