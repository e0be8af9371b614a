"""CPU: host side of the section-start alignment of the SLAM loop (LoopConfig.align_sections): which sections a base
frame is aligned against, and the configurations the loop refuses."""
import pytest

from vtgaussian_slam_b200 import synthetic
from vtgaussian_slam_b200.slam_loop import LoopConfig, ViewTiedSLAM, base_frame_sections

POSE_LRS = dict(rgb_colors=0.0025, logit_opacities=0.05, log_scales=0.005, cam_unnorm_rots=4e-4, cam_trans=2e-3)


@pytest.mark.parametrize("align, frozen", [(0, []), (1, [3]), (2, [2, 3]), (3, [1, 2, 3]), (7, [1, 2, 3])])
def test_latest_mode_aligns_against_the_last_tracked_sections(align, frozen):
    # section 4's base frame was tracked against the newest 3 sections before it: rows 1..3
    assert base_frame_sections(4, 3, align) == ([1, 2, 3], frozen)


def test_latest_mode_at_the_start_of_the_sequence():
    assert base_frame_sections(0, 1, 2) == ([], [])                      # frame 0: tracked against nothing, never aligned
    assert base_frame_sections(1, 3, 2) == ([0], [0])                    # fewer sections exist than track_sections
    assert base_frame_sections(2, 1, 2) == ([1], [1])
    assert base_frame_sections(2, 0, 1) == ([1], [1])                    # track_sections below 1 tracks the newest one


@pytest.mark.parametrize("align, frozen", [(0, []), (1, [5]), (2, [2, 5]), (3, [0, 2, 5]), (4, [0, 2, 5])])
def test_overlap_mode_aligns_against_the_last_selected_sections(align, frozen):
    # "overlap": the earliest overlapping sections plus the newest one, whatever track_sections says
    assert base_frame_sections(6, 1, align, selected=[0, 2, 5]) == ([0, 2, 5], frozen)
    assert base_frame_sections(6, 1, align, selected=(5, 2, 0)) == ([0, 2, 5], frozen)


def _slam(**cfg):
    W, H, K = synthetic.intrinsics("tum_fr1", 64, 48)
    return ViewTiedSLAM(W, H, K, LoopConfig(**cfg), device="cpu")


def test_defaults_leave_alignment_off():
    assert LoopConfig().align_sections == 0
    assert _slam().cfg.align_sections == 0


@pytest.mark.parametrize("cfg", [
    dict(align_sections=-1),
    dict(align_sections=-1, map_lrs=POSE_LRS),
    dict(align_sections=1),                                                          # default map_lrs: no pose LRs
    dict(align_sections=2, map_lrs=dict(POSE_LRS, cam_unnorm_rots=0.0, cam_trans=0.0)),
    dict(align_sections=1, map_lrs=dict(rgb_colors=0.0025, cam_trans=0.0)),
])
def test_refused_configurations(cfg):
    with pytest.raises(ValueError):
        _slam(**cfg)


@pytest.mark.parametrize("lrs", [POSE_LRS, dict(rgb_colors=0.0025, cam_trans=2e-3), dict(cam_unnorm_rots=4e-4)])
def test_accepted_configurations(lrs):
    assert _slam(align_sections=2, map_lrs=lrs).cfg.align_sections == 2
    assert _slam(align_sections=0, map_lrs=lrs).cfg.align_sections == 0
