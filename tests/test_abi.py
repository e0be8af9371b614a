"""CPU tests of the drop-in boundary: the C-ABI library loads without a GPU, exports every
symbol include/vtgs.h declares, struct layouts agree, argument validation works, and the
Python surface mirrors the reference's (no compute without a GPU)."""
import ctypes as C
import os
import re

import pytest
import torch

from vtgaussian_slam_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    _lib.build()
    return _lib.lib()


def test_every_declared_symbol_is_exported(L):
    hdr = open(os.path.join(ROOT, "include", "vtgs.h")).read()
    declared = set(re.findall(r"VTGS_API\s+[\w\s\*]+?\b(vtgs_\w+)\s*\(", hdr))
    assert len(declared) >= 15
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(L, name)
    assert L.vtgs_abi_version() == _lib.ABI_VERSION == 4
    assert b"sm_100a" in L.vtgs_build_info()


def test_struct_layouts_match_the_header(L):
    assert C.sizeof(_lib.VtgsCamera) == 4 * (2 + 2 + 16 + 16 + 3 + 1 + 1 + 2)
    assert C.sizeof(_lib.VtgsCounters) == 4 * (4 + 9 + 3 + 4 + 2 + 10)
    assert C.sizeof(_lib.VtgsBuffers) == 8 * 19            # 18 pointers / sizes + flags, reserved
    assert C.sizeof(_lib.VtgsParams) == 8 * 5 + 8 + 8
    assert C.sizeof(_lib.VtgsPose) == 16 + 16
    assert C.sizeof(_lib.VtgsLossConfig) == 32 + 8 + 8 + 8
    assert C.sizeof(_lib.VtgsParamGrads) == 88


def test_workspace_query_and_validation(L):
    sz = _lib.VtgsWorkspaceSizes()
    assert L.vtgs_workspace_query(1200, 680, 1000000, 4000000, C.byref(sz)) == 0
    assert (sz.tiles_x, sz.tiles_y) == (75, 43)
    assert sz.geom_bytes == 64 * 1000000 and sz.pair_keys_bytes == 8 * 4000000
    assert sz.final_T_bytes == 1200 * 680 * 4
    assert L.vtgs_workspace_query(0, 680, 1, 1, C.byref(sz)) == -1
    assert b"bad dimensions" in L.vtgs_last_error()
    cam = _lib.VtgsCamera()
    assert L.vtgs_mark_visible(C.byref(cam), 0, None, None, None) == -1     # zero-sized image
    assert L.vtgs_pose_scratch_floats(1000) >= 12 * 4


# Argument checks of every entry point.  Each case breaks exactly one check that returns before any CUDA call, so the
# call fails the same way with or without a GPU.  _D stands for a device address: no check dereferences it.
_D = 16
_NO_CAM = C.POINTER(_lib.VtgsCamera)()


def _cam(**kw):
    c = _lib.VtgsCamera(image_width=64, image_height=48, tanfovx=0.5, tanfovy=0.5, scale_modifier=1.0, radius_sigma_mult=3.0)
    for k, v in kw.items():
        setattr(c, k, v)
    return C.byref(c)


def _buf(**kw):
    b = _lib.VtgsBuffers(pair_capacity=1024)
    for name, t in _lib.VtgsBuffers._fields_:
        if t is C.c_void_p:
            setattr(b, name, _D)
    for k, v in kw.items():
        setattr(b, k, v)
    return C.byref(b)


def _params(**kw):
    p = _lib.VtgsParams(_D, _D, _D, _D, _D, log_scales_dim=1, num_gaussians=10)
    for k, v in kw.items():
        setattr(p, k, v)
    return C.byref(p)


def _pose(**kw):
    p = _lib.VtgsPose(_D, _D)
    for k, v in kw.items():
        setattr(p, k, v)
    return C.byref(p)


def _cfg(**kw):
    c = _lib.VtgsLossConfig(mode=0, use_l1=1, w_im=0.5, w_depth=1.0)
    for k, v in kw.items():
        setattr(c, k, v)
    return C.byref(c)


def _grads(**kw):
    g = _lib.VtgsParamGrads()
    for k, v in kw.items():
        setattr(g, k, v)
    return C.byref(g)


def _forward(L, cam=None, N=10, ins=(_D,) * 5, outs=(_D, _D), radii=_D, buf=None):
    return L.vtgs_forward(_cam() if cam is None else cam, N, *ins, *outs, radii, buf or _buf(), None)


def _backward(L, cam=None, N=10, ptr=(_D,) * 12, buf=None):
    return L.vtgs_backward(_cam() if cam is None else cam, N, *ptr, buf or _buf(), None)


def _fused_forward(L, cam=None, params=None, pose=None, out=_D, radii=_D, buf=None):
    return L.vtgs_fused_forward(_cam() if cam is None else cam, params or _params(), pose or _pose(), out, radii, buf or _buf(), None)


def _fused_backward(L, params=None, pose=None, dl=_D, grads=None):
    return L.vtgs_fused_backward(_cam(), params or _params(), pose or _pose(), dl, 0, grads or _grads(), _buf(), None)


def _loss(L, cam=None, cfg=None, scratch=_D):
    return L.vtgs_loss(_cam() if cam is None else cam, cfg or _cfg(), _D, _D, _D, _D, _D, scratch, None)


def _sharded_adam(L, world=2, rank=0, bases=None, mc=0, n=8, nseg=1):
    bases = (C.c_uint64 * 8)(*([256] * 8)) if bases is None else bases
    seg_end, lr = (C.c_int64 * 4)(8), (C.c_float * 4)(1e-3)
    return L.vtgs_sharded_adam(world, rank, bases, mc, 0, 8, 16, _D, _D, n, nseg, seg_end, lr, 0.9, 0.999, 1e-8, _D, _D, None)


def _p2p_match(L, n_tgt=4, tgt_nrm=_D, n_src=4, max_dist=0.1, table_size=64, out_dist=_D):
    return L.vtgs_p2p_match(n_tgt, _D, tgt_nrm, _D, n_src, _D, _D, max_dist, _D, table_size, _D, out_dist, None, None)


_INVALID, _UNSUPPORTED = -1, -3
_ARG_CASES = {
    # the camera and workspace checks every rendering entry point shares
    "forward/cam_null": (lambda L: _forward(L, cam=_NO_CAM), _INVALID, "cam is NULL"),
    "forward/image_size": (lambda L: _forward(L, cam=_cam(image_height=0)), _INVALID, "image size must be positive"),
    "forward/tanfov": (lambda L: _forward(L, cam=_cam(tanfovy=0.0)), _INVALID, "tanfov must be positive"),
    "forward/sigma_mult": (lambda L: _forward(L, cam=_cam(radius_sigma_mult=0.0)), _INVALID, "radius_sigma_mult must be positive"),
    "forward/buffers_null": (lambda L: L.vtgs_forward(_cam(), 10, *[_D] * 8, None, None), _INVALID, "buffers is NULL"),
    "forward/workspace_null": (lambda L: _forward(L, buf=_buf(final_T=None)), _INVALID, "workspace pointer is NULL"),
    "forward/per_gaussian_null": (lambda L: _forward(L, buf=_buf(grad_geom=None)), _INVALID, "per-Gaussian workspace pointer is NULL"),
    "forward/pair_null": (lambda L: _forward(L, buf=_buf(region_pairs=None)), _INVALID, "pair workspace pointer is NULL"),
    "forward/pair_capacity": (lambda L: _forward(L, buf=_buf(pair_capacity=1 << 32)), _INVALID, "pair_capacity must fit 32 bits"),
    "forward/negative_n": (lambda L: _forward(L, N=-1), _INVALID, "num_gaussians < 0"),
    "forward/output_null": (lambda L: _forward(L, outs=(_D, None)), _INVALID, "output pointer is NULL"),
    "forward/input_null": (lambda L: _forward(L, ins=(_D, _D, None, _D, _D)), _INVALID, "input pointer is NULL"),
    "forward/image_too_large": (lambda L: _forward(L, cam=_cam(image_width=16 * 65536, image_height=16)), _INVALID,
                                "image too large for packed tile rects"),
    "forward/too_many_gaussians": (lambda L: _forward(L, N=1 << 32), _UNSUPPORTED, "at most 2^32 - 1 Gaussians"),
    "backward/cam_null": (lambda L: _backward(L, cam=_NO_CAM), _INVALID, "cam is NULL"),
    "backward/buffers_null": (lambda L: L.vtgs_backward(_cam(), 10, *[_D] * 12, None, None), _INVALID, "buffers is NULL"),
    "backward/negative_n": (lambda L: _backward(L, N=-1), _INVALID, "num_gaussians < 0"),
    "backward/pointer_null": (lambda L: _backward(L, ptr=(_D,) * 11 + (None,)), _INVALID, "pointer is NULL"),
    "mark_visible/cam_null": (lambda L: L.vtgs_mark_visible(None, 10, _D, _D, None), _INVALID, "cam is NULL"),
    "mark_visible/pointer_null": (lambda L: L.vtgs_mark_visible(_cam(), 10, _D, None, None), _INVALID, "pointer is NULL"),
    "export_sorted_keys/cam_null": (lambda L: L.vtgs_export_sorted_keys(None, 10, _buf(), _D, 64, None), _INVALID, "cam is NULL"),
    "export_sorted_keys/pointer_null": (lambda L: L.vtgs_export_sorted_keys(_cam(), 10, _buf(), None, 64, None), _INVALID,
                                        "pointer is NULL"),
    "export_geometry/buffers_null": (lambda L: L.vtgs_export_geometry(10, None, _D, _D, _D, None), _INVALID, "buffers is NULL"),
    "fused_forward/cam_null": (lambda L: _fused_forward(L, cam=_NO_CAM), _INVALID, "cam is NULL"),
    "fused_forward/params_null": (lambda L: L.vtgs_fused_forward(_cam(), None, _pose(), _D, _D, _buf(), None), _INVALID,
                                  "params / pose is NULL"),
    "fused_forward/buffers_null": (lambda L: L.vtgs_fused_forward(_cam(), _params(), _pose(), _D, _D, None, None), _INVALID,
                                   "buffers is NULL"),
    "fused_forward/negative_n": (lambda L: _fused_forward(L, params=_params(num_gaussians=-1)), _INVALID, "num_gaussians < 0"),
    "fused_forward/param_null": (lambda L: _fused_forward(L, params=_params(log_scales=None)), _INVALID, "param pointer is NULL"),
    "fused_forward/pose_null": (lambda L: _fused_forward(L, pose=_pose(cam_trans=None)), _INVALID, "pose pointer is NULL"),
    "fused_forward/anisotropic": (lambda L: _fused_forward(L, params=_params(log_scales_dim=3)), _UNSUPPORTED,
                                  "isotropic Gaussians only"),
    "fused_forward/out_null": (lambda L: _fused_forward(L, out=None), _INVALID, "out_image6 is NULL"),
    "fused_forward/radii_null": (lambda L: _fused_forward(L, radii=None), _INVALID, "radii is NULL"),
    "fused_forward/image_too_large": (lambda L: _fused_forward(L, cam=_cam(image_width=16 * 65536, image_height=16)), _INVALID,
                                      "image too large for packed tile rects"),
    "fused_backward/pose_null": (lambda L: L.vtgs_fused_backward(_cam(), _params(), None, _D, 0, _grads(), _buf(), None),
                                 _INVALID, "params / pose is NULL"),
    "fused_backward/anisotropic": (lambda L: _fused_backward(L, params=_params(log_scales_dim=3)), _UNSUPPORTED,
                                   "isotropic Gaussians only"),
    "fused_backward/pointer_null": (lambda L: _fused_backward(L, dl=None), _INVALID, "pointer is NULL"),
    "fused_backward/pose_scratch": (lambda L: _fused_backward(L, grads=_grads(cam_unnorm_rot=_D, cam_trans=_D)), _INVALID,
                                    "pose gradients need pose_scratch"),
    "fused_tracking_step/mapping_cfg": (lambda L: L.vtgs_fused_tracking_step(_cam(), _params(), _pose(), _cfg(mode=1), *[_D] * 7,
                                                                              _grads(), None, None, _buf(), None),
                                        _INVALID, "needs a tracking-mode loss configuration"),
    "fused_tracking_step/radius_pair": (lambda L: L.vtgs_fused_tracking_step(_cam(), _params(), _pose(), _cfg(), *[_D] * 7,
                                                                              _grads(), _D, None, _buf(), None),
                                        _INVALID, "max_2D_radius and seen come as a pair"),
    "fused_tracking_step/anisotropic": (lambda L: L.vtgs_fused_tracking_step(_cam(), _params(log_scales_dim=3), _pose(), _cfg(),
                                                                              *[_D] * 7, _grads(), None, None, _buf(), None),
                                        _UNSUPPORTED, "isotropic Gaussians only"),
    "loss/cam_null": (lambda L: _loss(L, cam=_NO_CAM), _INVALID, "cam is NULL"),
    "loss/pointer_null": (lambda L: _loss(L, scratch=None), _INVALID, "pointer is NULL"),
    "loss/outlier_in_mapping": (lambda L: _loss(L, cfg=_cfg(mode=1, ignore_outlier_depth=1)), _UNSUPPORTED,
                                "ignore_outlier_depth_loss is a tracking option"),
    "loss/outlier_band_without_median": (lambda L: _loss(L, cam=_cam(tile_row_begin=1, tile_row_end=2),
                                                         cfg=_cfg(ignore_outlier_depth=1)), _UNSUPPORTED,
                                         "needs VtgsLossConfig.median_state"),
    "loss/no_l1": (lambda L: _loss(L, cfg=_cfg(use_l1=0)), _UNSUPPORTED, "use_l1 = False is not supported"),
    "loss/mapping_band": (lambda L: _loss(L, cam=_cam(tile_row_begin=1, tile_row_end=2), cfg=_cfg(mode=1)), _INVALID,
                          "mapping loss is not band-sharded"),
    "loss/unknown_mode": (lambda L: _loss(L, cfg=_cfg(mode=2)), _INVALID, "unknown loss mode"),
    "retie/negative_n": (lambda L: L.vtgs_retie(_D, -1, C.byref((C.c_float * 12)()), _D, _D, None), _INVALID, "n < 0"),
    "retie/pointer_null": (lambda L: L.vtgs_retie(_D, 10, None, _D, _D, None), _INVALID, "pointer is NULL"),
    "retie_dev/negative_n": (lambda L: L.vtgs_retie_dev(_D, -1, _D, _D, _D, _D, None), _INVALID, "n < 0"),
    "retie_dev/pointer_null": (lambda L: L.vtgs_retie_dev(_D, 10, _D, None, _D, _D, None), _INVALID, "pointer is NULL"),
    "adam/negative_n": (lambda L: L.vtgs_adam(_D, _D, _D, _D, -1, 1e-3, 0.9, 0.999, 1e-8, 1, None, None), _INVALID, "n < 0"),
    "adam/pointer_null": (lambda L: L.vtgs_adam(_D, None, _D, _D, 8, 1e-3, 0.9, 0.999, 1e-8, 1, None, None), _INVALID,
                          "pointer is NULL"),
    "adam/step_zero": (lambda L: L.vtgs_adam(_D, _D, _D, _D, 8, 1e-3, 0.9, 0.999, 1e-8, 0, None, None), _INVALID,
                       "step must be >= 1"),
    "sharded_adam/world": (lambda L: _sharded_adam(L, world=9), _INVALID, "world must be 1..8"),
    "sharded_adam/rank": (lambda L: _sharded_adam(L, rank=2), _INVALID, "world must be 1..8 and rank inside it"),
    "sharded_adam/pointer_null": (lambda L: L.vtgs_sharded_adam(2, 0, None, 0, 0, 8, 16, _D, _D, 8, 1, _D, _D, 0.9, 0.999, 1e-8,
                                                                 _D, _D, None), _INVALID, "pointer is NULL"),
    "sharded_adam/multiple_of_4": (lambda L: _sharded_adam(L, n=6), _INVALID, "multiples of 4 floats"),
    "sharded_adam/segments": (lambda L: _sharded_adam(L, nseg=5), _INVALID, "1..4 segments"),
    "sharded_adam/peer_alignment": (lambda L: _sharded_adam(L, bases=(C.c_uint64 * 8)(256, 264)), _INVALID,
                                    "peer base must be a 16-byte aligned address"),
    "sharded_adam/multicast_alignment": (lambda L: _sharded_adam(L, mc=264), _INVALID, "multicast base must be 16-byte aligned"),
    "tracking_update/pointer_null": (lambda L: L.vtgs_tracking_update(_D, _D, _D, _D, _D, None, 1e-3, 1e-3, 1e-8, 0, None),
                                     _INVALID, "pointer is NULL"),
    "median_hist/cam_null": (lambda L: L.vtgs_median_hist(None, _D, _D, 0, _D, None), _INVALID, "cam is NULL"),
    "median_hist/pointer_null": (lambda L: L.vtgs_median_hist(_cam(), _D, _D, 0, None, None), _INVALID, "pointer is NULL"),
    "median_hist/pass": (lambda L: L.vtgs_median_hist(_cam(), _D, _D, 4, _D, None), _INVALID, "pass must be 0..3"),
    "median_pick/bad_argument": (lambda L: L.vtgs_median_pick(0, 0, _D, None), _INVALID, "bad argument"),
    "median_pick/pass": (lambda L: L.vtgs_median_pick(100, -1, _D, None), _INVALID, "pass must be 0..3"),
    "sil_ladder/cam_null": (lambda L: L.vtgs_sil_ladder(None, _D, _D, _D, _D, _D, None), _INVALID, "cam is NULL"),
    "sil_ladder/pointer_null": (lambda L: L.vtgs_sil_ladder(_cam(), _D, _D, _D, _D, None, None), _INVALID, "pointer is NULL"),
    "sil_select/pointer_null": (lambda L: L.vtgs_sil_select(_D, None, _D, None), _INVALID, "pointer is NULL"),
    "nonpresence_mask/cam_null": (lambda L: L.vtgs_nonpresence_mask(None, _D, _D, 0.5, _D, _D, None, None), _INVALID,
                                  "cam is NULL"),
    "nonpresence_mask/pointer_null": (lambda L: L.vtgs_nonpresence_mask(_cam(), _D, _D, 0.5, _D, None, None, None), _INVALID,
                                      "pointer is NULL"),
    "eval_metrics/cam_null": (lambda L: L.vtgs_eval_metrics(None, _D, _D, _D, 0.5, 0, _D, _D, None), _INVALID, "cam is NULL"),
    "eval_metrics/pointer_null": (lambda L: L.vtgs_eval_metrics(_cam(), _D, _D, _D, 0.5, 0, None, _D, None), _INVALID,
                                  "pointer is NULL"),
    "p2p_prepare/image_size": (lambda L: L.vtgs_p2p_prepare(0, 48, C.byref((C.c_float * 4)()), C.byref((C.c_float * 12)()),
                                                            None, _D, None, _D, None, _D, None), _INVALID, "bad image size"),
    "p2p_prepare/pointer_null": (lambda L: L.vtgs_p2p_prepare(64, 48, C.byref((C.c_float * 4)()), C.byref((C.c_float * 12)()),
                                                              None, None, None, _D, None, _D, None), _INVALID, "pointer is NULL"),
    "p2p_match/point_count": (lambda L: _p2p_match(L, n_tgt=-1), _INVALID, "bad point count"),
    "p2p_match/max_dist": (lambda L: _p2p_match(L, max_dist=0.0), _INVALID, "max_dist must be positive"),
    "p2p_match/table_size": (lambda L: _p2p_match(L, table_size=48), _INVALID, "table_size must be a power of two"),
    "p2p_match/target_null": (lambda L: _p2p_match(L, tgt_nrm=None), _INVALID, "pointer is NULL"),
    "p2p_match/source_null": (lambda L: _p2p_match(L, out_dist=None), _INVALID, "pointer is NULL"),
    "frame_convert/image_size": (lambda L: L.vtgs_frame_convert(0, 48, 64, 48, _D, _D, 1000.0, _D, _D, None), _INVALID,
                                 "bad image size"),
    "frame_convert/pairs": (lambda L: L.vtgs_frame_convert(64, 48, 64, 48, _D, _D, 1000.0, None, _D, None), _INVALID,
                            "input / output pointers must come in pairs"),
    "frame_convert/depth_scale": (lambda L: L.vtgs_frame_convert(64, 48, 64, 48, _D, _D, 0.0, _D, _D, None), _INVALID,
                                  "png_depth_scale must be positive"),
    "book_radii/negative_n": (lambda L: L.vtgs_book_radii(-1, _D, _D, _D, None), _INVALID, "n < 0"),
    "book_radii/pointer_null": (lambda L: L.vtgs_book_radii(10, _D, _D, None, None), _INVALID, "pointer is NULL"),
    "ffma_probe/bad_argument": (lambda L: L.vtgs_ffma_probe(0, _D, None, None), _INVALID, "bad argument"),
    "workspace_query/sizes_null": (lambda L: L.vtgs_workspace_query(64, 48, 10, 1024, None), _INVALID, "sizes is NULL"),
    "profile_summary/buffer_null": (lambda L: L.vtgs_profile_summary(None, 64), _INVALID, "buffer is NULL"),
}


@pytest.mark.parametrize("case", sorted(_ARG_CASES))
def test_entry_point_argument_checks(L, case):
    call, code, message = _ARG_CASES[case]
    assert call(L) == code
    assert message.encode() in L.vtgs_last_error()


def test_python_surface_mirrors_the_reference():
    import diff_gaussian_rasterization as dgr
    fields = dgr.GaussianRasterizationSettings._fields
    assert fields == ("image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix",
                      "projmatrix", "sh_degree", "campos", "prefiltered")       # utils/recon_helpers.py:14-26
    s = dgr.GaussianRasterizationSettings(4, 4, 1.0, 1.0, torch.zeros(3), 1.0, torch.eye(4)[None], torch.eye(4)[None], 0,
                                          torch.zeros(3), False)
    r = dgr.GaussianRasterizer(raster_settings=s)
    z3, z4, z1 = torch.zeros(2, 3), torch.zeros(2, 4), torch.zeros(2, 1)
    with pytest.raises(Exception, match="excatly one"):
        r(means3D=z3, means2D=z3, opacities=z1, scales=z3, rotations=z4)
    with pytest.raises(NotImplementedError):
        r(means3D=z3, means2D=z3, opacities=z1, shs=torch.zeros(2, 1, 3), scales=z3, rotations=z4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        r(means3D=z3, means2D=z3, opacities=z1, colors_precomp=z3, scales=z3, rotations=z4)


def test_product_never_imports_the_oracle():
    for pkg in ("vtgaussian_slam_b200", "diff_gaussian_rasterization"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, pkg)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    src = open(os.path.join(dirpath, f)).read()
                    assert not re.search(r"^\s*(import|from)\s+oracle\b", src, re.M), f
                    assert "libvtgs_oracle" not in src, f
