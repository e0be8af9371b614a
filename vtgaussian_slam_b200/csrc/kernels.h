// kernels.h -- what the translation units of libvtgs_cuda.so share on the host: the argument checks of the C entry
// points and the internal calls one file makes into another.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace vtgs {

#define VTGS_REQUIRE(cond, msg)                           \
    do {                                                  \
        if (!(cond)) {                                    \
            vtgs::set_error("invalid argument: %s", msg); \
            return VTGS_E_INVALID;                        \
        }                                                 \
    } while (0)

inline int check_cam(const VtgsCamera* cam) {
    VTGS_REQUIRE(cam != nullptr, "cam is NULL");
    VTGS_REQUIRE(cam->image_width > 0 && cam->image_height > 0, "image size must be positive");
    VTGS_REQUIRE(cam->tanfovx > 0.f && cam->tanfovy > 0.f, "tanfov must be positive");
    VTGS_REQUIRE(cam->radius_sigma_mult > 0.f, "radius_sigma_mult must be positive");
    return VTGS_OK;
}

inline int check_buf(const VtgsBuffers* b, int64_t N) {
    VTGS_REQUIRE(b != nullptr, "buffers is NULL");
    VTGS_REQUIRE(b->tile_counts && b->tile_ranges && b->final_T && b->n_contrib && b->counters && b->region_cnt && b->region_masks && b->region_done, "workspace pointer is NULL");
    if (N > 0) VTGS_REQUIRE(b->geom && b->tiles_touched && b->grad_geom, "per-Gaussian workspace pointer is NULL");
    VTGS_REQUIRE(b->pair_capacity == 0 || (b->pair_keys && b->point_list && b->region_pairs), "pair workspace pointer is NULL");
    VTGS_REQUIRE(b->pair_capacity < 0xffffffffull, "pair_capacity must fit 32 bits");
    return VTGS_OK;
}

inline int check_fused(const VtgsCamera* cam, const VtgsParams* p, const VtgsPose* pose, const VtgsBuffers* buf) {
    if (int e = check_cam(cam)) return e;
    VTGS_REQUIRE(p && pose, "params / pose is NULL");
    if (int e = check_buf(buf, p->num_gaussians)) return e;
    VTGS_REQUIRE(p->num_gaussians >= 0, "num_gaussians < 0");
    if (p->num_gaussians > 0)
        VTGS_REQUIRE(p->means3D && p->rgb_colors && p->unnorm_rotations && p->logit_opacities && p->log_scales, "param pointer is NULL");
    VTGS_REQUIRE(pose->cam_unnorm_rot && pose->cam_trans, "pose pointer is NULL");
    if (p->log_scales_dim != 1) {
        set_error("fused path supports isotropic Gaussians only (log_scales [N,1]); use vtgs_forward/backward for anisotropic");
        return VTGS_E_UNSUPPORTED;
    }
    return VTGS_OK;
}

// backward.cu: publishes the frame's pose for the backward when the fused forward has no Gaussian to preprocess.
int launch_pose_matrix(const VtgsPose* pose, VtgsCounters* counters, cudaStream_t stream);

}  // namespace vtgs
