// forward.cu -- K1' preprocess, K2'-K5a' tile binning, K5' front-to-back blend (sm_100a).
//
// Replaces the forward half of the reference's external rasteriser
// (`_C.rasterize_gaussians`, called at reference src/vtgaussian_slam.py:461,466,747):
// upstream preprocessCUDA / InclusiveSum / duplicateWithKeys / DeviceRadixSort /
// identifyTileRanges / renderCUDA (SURVEY.md 2.3 K1-K5, Appendix A.1-A.3).
//
// Design (DESIGN.md):
//  * binning is an MSD radix sort on the 64-bit (tile | depth) key: the tile digit is a
//    counting sort (per-tile histogram in preprocess, a one-block scan that also yields the
//    tile ranges, an atomic-cursor scatter), the 32 depth bits (+ Gaussian id as the
//    stable tie-break) are sorted per tile in shared memory.  The sorted order is
//    (tile, depth bits, Gaussian index) -- exactly what the reference's stable LSD sort
//    of its duplicateWithKeys output produces.
//  * the blend kernel culls each staged batch against its eight 8x4-pixel warp regions
//    with one ballot per region, so a warp only evaluates splats whose alpha >= 1/255
//    ellipse can touch its pixels (view-tied splats are ~1 px wide: ~70% of the
//    upstream pair tests disappear) while list positions (n_contrib) stay exact.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>

#include "blend_common.cuh"
#include "kernels.h"

namespace vtgs {

// Front end of the fused path (transform_to_frame + activations); unused in API mode.
struct FrontEnd {
    const float* cam_unnorm_rot;   // device [4]: the frame's un-normalised pose quaternion
    const float* cam_trans;        // device [3]
    VtgsCounters* counters;        // device: receives pose_R / pose_t / pose_q / pose_qnorm for the backward
    float depth_row[4];
    int log_scales_dim;
};

// Warp-collective walk over every lane's tile rect [minx,maxx) x [miny,maxy).  Each step all lanes
// present their current tile (or none); lanes presenting the same tile are grouped with
// match.any so that the callback can issue ONE atomic per distinct tile:
//   f(tile, tile_x, tile_y, peers_mask, rank_in_group, is_leader).  Must be called by all 32 lanes.
template <typename F>
__device__ __forceinline__ void warp_tile_walk(int minx, int miny, int maxx, int maxy, int gx, F f) {
    const int lane = threadIdx.x & 31;
    int tx = minx, ty = miny;
    bool have = (maxx > minx) && (maxy > miny);
    while (__any_sync(VTGS_FULL_MASK, have)) {
        const int tile = have ? ty * gx + tx : -1 - lane;      // distinct negative ids: never grouped
        const uint32_t peers = __match_any_sync(VTGS_FULL_MASK, tile);
        if (have) {
            const int rank = __popc(peers & ((1u << lane) - 1u));
            f(tile, tx, ty, peers, rank, rank == 0);
            if (++tx >= maxx) { tx = minx; if (++ty >= maxy) have = false; }
        }
    }
}

// =============================== K0': band candidate blocks ================================
// Tile-band sharding (multi-GPU tracking): every rank holds all N Gaussians but renders only its band of tile rows.
// Per iteration, one fully parallel pass over (position, log-scale) -- 16 bytes per Gaussian -- marks the 256-Gaussian
// BLOCKS that hold at least one splat able to reach the band at the CURRENT pose (the same conservative screen-space
// bound K1' applies per splat) and zeroes radii / tiles_touched of the others.  K1', the scatter and K7' then skip the
// unmarked blocks outright, so their cost follows the band, not N: a view-tied section is ordered like its image, so a
// band of rows is a few contiguous runs of blocks.  Nothing is cached across iterations: no staleness to bound.
__global__ void __launch_bounds__(256)
band_flags_kernel(const __grid_constant__ CamConst cam, int64_t N, FrontEnd fe, const float* __restrict__ means3D,
                  const float* __restrict__ log_scales, int32_t* __restrict__ radii, uint32_t* __restrict__ tiles_touched,
                  uint8_t* __restrict__ flags, uint32_t* __restrict__ cand, uint32_t* __restrict__ n_cand) {
    VTGS_PDL_PROLOGUE();
    // one block = 4 candidate blocks of 256 Gaussians: all 16 loads of a thread are in flight together
    __shared__ float s_Rt[12];
    __shared__ uint32_t s_any[4];
    const int tid = threadIdx.x;
    if (tid == 0) {
        float Rt[12], qn[4], nrm2[2];
        pose_from_quat(fe.cam_unnorm_rot, fe.cam_trans, Rt, qn, nrm2);
#pragma unroll
        for (int k = 0; k < 12; ++k) s_Rt[k] = Rt[k];
    }
    if (tid < 4) s_any[tid] = 0u;
    float px[4], py[4], pz[4], ls[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int64_t i = ((int64_t)blockIdx.x * 4 + j) * 256 + tid;
        px[j] = py[j] = pz[j] = ls[j] = 0.0f;
        if (i < N) {
            px[j] = means3D[3 * i]; py[j] = means3D[3 * i + 1]; pz[j] = means3D[3 * i + 2];
            if (fe.log_scales_dim == 1) ls[j] = log_scales[i];
            else ls[j] = fmaxf(log_scales[3 * i], fmaxf(log_scales[3 * i + 1], log_scales[3 * i + 2]));
        }
    }
    __syncthreads();
    const float kx = cam.focal_x * cam.focal_x * (1.0f + cam.limx * cam.limx) + cam.focal_y * cam.focal_y * (1.0f + cam.limy * cam.limy);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int64_t i = ((int64_t)blockIdx.x * 4 + j) * 256 + tid;
        bool reach = false;
        if (i < N) {
            const float X = s_Rt[0] * px[j] + s_Rt[1] * py[j] + s_Rt[2] * pz[j] + s_Rt[9];
            const float Y = s_Rt[3] * px[j] + s_Rt[4] * py[j] + s_Rt[5] * pz[j] + s_Rt[10];
            const float Z = s_Rt[6] * px[j] + s_Rt[7] * py[j] + s_Rt[8] * pz[j] + s_Rt[11];
            const float tz_ = xform_row(cam.view, 2, X, Y, Z);
            if (tz_ > VTGS_NEAR_CULL) {                  // (behind the near plane: K1' would cull it anyway)
                const float smax = __expf(ls[j]) * 1.001f * cam.scale_modifier;
                const float hy_ = xform_row(cam.proj, 1, X, Y, Z), hw_ = xform_row(cam.proj, 3, X, Y, Z);
                const float py_ = ((__fdividef(hy_, hw_ + VTGS_EPS_W) + 1.0f) * (float)cam.H - 1.0f) * 0.5f;
                const float itz = __fdividef(1.0f, tz_);
                const float tr = smax * smax * itz * itz * kx + 2.0f * VTGS_LOWPASS;
                const float rb = cam.sigma_mult * sqrtf(tr) * 1.02f + 4.0f;      // a little wider than K1's own test
                reach = !((py_ - rb > (float)(cam.row1 * 16)) || (py_ + rb + 16.0f < (float)(cam.row0 * 16)));
            }
        }
        if (__any_sync(VTGS_FULL_MASK, reach) && (tid & 31) == 0) s_any[j] = 1u;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int64_t blk = (int64_t)blockIdx.x * 4 + j;
        const int64_t i = blk * 256 + tid;
        const bool any = s_any[j] != 0u;
        if (tid == 0 && blk * 256 < N) {
            flags[blk] = any ? 1 : 0;
            if (any) cand[atomicAdd(n_cand, 1u)] = (uint32_t)blk;       // (order is arbitrary: nothing downstream depends on it)
        }
        if (!any && i < N) { radii[i] = 0; tiles_touched[i] = 0u; }
    }
}

// =============================== K1': preprocess =========================================
// Persistent grid-stride kernel, one Gaussian per thread per trip; the loads of the NEXT Gaussian are
// in flight while the current one is projected (the math is ~1000 instructions of IEEE div / sqrt /
// fp64 ndc2Pix per Gaussian, the loads ~48 B, the stores one 64-byte record).
struct K1Item {
    float x, y, z, c0, c1, c2, s0, s1, s2, op;
    float4 q;
};

__device__ __forceinline__ void k1_load_rest(K1Item& it, int64_t i, bool rot_aligned, const float* __restrict__ rotations,
                                             const float* __restrict__ opacities, const float* __restrict__ colors) {
    it.c0 = colors[3 * i]; it.c1 = colors[3 * i + 1]; it.c2 = colors[3 * i + 2];
    it.op = opacities[i];
    it.q = rot_aligned ? reinterpret_cast<const float4*>(rotations)[i]
                       : make_float4(rotations[4 * i], rotations[4 * i + 1], rotations[4 * i + 2], rotations[4 * i + 3]);
}

template <bool FUSED>
__device__ __forceinline__ void k1_load(K1Item& it, int64_t i, int ls_dim, bool rot_aligned,
                                        const float* __restrict__ means3D, const float* __restrict__ scales,
                                        const float* __restrict__ rotations, const float* __restrict__ opacities,
                                        const float* __restrict__ colors, bool position_only = false) {
    it.x = means3D[3 * i]; it.y = means3D[3 * i + 1]; it.z = means3D[3 * i + 2];
    if (FUSED && ls_dim == 1) { it.s0 = scales[i]; it.s1 = it.s0; it.s2 = it.s0; }
    else { it.s0 = scales[3 * i]; it.s1 = scales[3 * i + 1]; it.s2 = scales[3 * i + 2]; }
    if (position_only) return;          // tile-band mode: the other 32 bytes are fetched only for splats that reach the band
    k1_load_rest(it, i, rot_aligned, rotations, opacities, colors);
}

// LITE (fused, narrow tile bands: most splats are rejected): only position and scale are fetched before the band test.
template <bool FUSED, bool LITE = false>
__global__ void __launch_bounds__(256, 3)
preprocess_kernel(const __grid_constant__ CamConst cam, int64_t N, FrontEnd fe,
                  const float* __restrict__ means3D, const float* __restrict__ scales,
                  const float* __restrict__ rotations, const float* __restrict__ opacities,
                  const float* __restrict__ colors,
                  GeomRecord* __restrict__ geom, int32_t* __restrict__ radii,
                  uint32_t* __restrict__ tiles_touched, uint32_t* __restrict__ tile_counts,
                  const uint32_t* __restrict__ cand, const uint32_t* __restrict__ n_cand, uint32_t* __restrict__ colour_max_bits) {
    VTGS_PDL_PROLOGUE();
    // Persistent loop over 256-Gaussian blocks: all of them, or (tile bands) the candidate blocks K0' listed.
    float cmax = 0.0f;          // max |colour| over the splats this thread emitted (deterministic backward: bound of c . dL/dpixel)
    const int tid = threadIdx.x;
    const int64_t nblk = cand != nullptr ? (int64_t)*n_cand : (N + 255) / 256;
    const bool rot_aligned = (reinterpret_cast<uintptr_t>(rotations) & 15) == 0;
    const bool band_active = cam.row0 > 0 || cam.row1 < cam.gy;
    float Rt[12];
    if (FUSED) {
        // every thread derives the pose matrix itself (a few dozen instructions, once per persistent thread);
        // thread 0 publishes it for the backward (K7' and the pose chain)
        float qn[4], nrm2[2];
        pose_from_quat(fe.cam_unnorm_rot, fe.cam_trans, Rt, qn, nrm2);
        if (blockIdx.x == 0 && tid == 0) {
#pragma unroll
            for (int k = 0; k < 9; ++k) fe.counters->pose_R[k] = Rt[k];
#pragma unroll
            for (int k = 0; k < 3; ++k) fe.counters->pose_t[k] = Rt[9 + k];
#pragma unroll
            for (int k = 0; k < 4; ++k) fe.counters->pose_q[k] = qn[k];
            fe.counters->pose_qnorm[0] = nrm2[0]; fe.counters->pose_qnorm[1] = nrm2[1];
        }
    }
    auto gaussian_of = [&](int64_t trip) -> int64_t {       // index handled by this thread in list trip `trip`
        if (trip >= nblk) return N;
        const int64_t blk = cand != nullptr ? (int64_t)cand[trip] : trip;
        return blk * 256 + tid;
    };
    int64_t trip = blockIdx.x;
    int64_t i = gaussian_of(trip);
    K1Item nxt;
    constexpr bool lite = LITE;
    if (i < N) k1_load<FUSED>(nxt, i, fe.log_scales_dim, rot_aligned, means3D, scales, rotations, opacities, colors, lite);
    // whole blocks loop together (the tile walk below is warp-collective)
    for (; trip < nblk; trip += gridDim.x) {
        const int64_t i_next = gaussian_of(trip + gridDim.x);
        int w_minx = 0, w_maxx = 0, w_miny = 0, w_maxy = 0;       // tile rect to count (empty when culled / out of range)
        if (i < N) {
            K1Item it = nxt;
            if (i_next < N) k1_load<FUSED>(nxt, i_next, fe.log_scales_dim, rot_aligned, means3D, scales, rotations, opacities, colors, lite);
            float x = it.x, y = it.y, z = it.z;
            float sx, sy, sz, qr = it.q.x, qx = it.q.y, qy = it.q.z, qz = it.q.w, op, c3;
            if (FUSED) {
                // transform_to_frame + activations (reference utils/slam_helpers.py:323-385,127-160):
                // p' = R p + t, scales = exp(log_scales), opacity = sigmoid(logit), q = normalize(q)
                const float X = fadd(ffma(Rt[2], z, ffma(Rt[1], y, fmul(Rt[0], x))), Rt[9]);
                const float Y = fadd(ffma(Rt[5], z, ffma(Rt[4], y, fmul(Rt[3], x))), Rt[10]);
                const float Z = fadd(ffma(Rt[8], z, ffma(Rt[7], y, fmul(Rt[6], x))), Rt[11]);
                x = X; y = Y; z = Z;
                if (fe.log_scales_dim == 3) { sx = vexpf(it.s0); sy = vexpf(it.s1); sz = vexpf(it.s2); }
                else { sx = sy = sz = vexpf(it.s0); }
            } else {
                sx = it.s0; sy = it.s1; sz = it.s2;
            }
            SplatGeom g;
            bool outside_band = false;
            if (FUSED && band_active) {
                // Tile-band sharding: a conservative bound of the splat's screen-space extent decides in ~40
                // instructions that it cannot reach this rank's rows, skipping the activations and the
                // ~900-instruction projection, and the 64-byte record (nothing reads it when tiles_touched = 0).
                // (radius <= sigma_mult * sqrt(trace(cov2D)), trace <= s^2 (|J0|^2 + |J1|^2) + 2 * lowpass with the
                // clamped Jacobian; 1 % + 3 px of slack cover the approximate arithmetic and the ceil.)
                const float tz_ = xform_row(cam.view, 2, x, y, z);
                if (tz_ > VTGS_NEAR_CULL) {
                    const float hy_ = xform_row(cam.proj, 1, x, y, z), hw_ = xform_row(cam.proj, 3, x, y, z);
                    const float py_ = ((__fdividef(hy_, hw_ + VTGS_EPS_W) + 1.0f) * (float)cam.H - 1.0f) * 0.5f;
                    const float smax = fmaxf(sx, fmaxf(sy, sz)) * cam.scale_modifier, itz = __fdividef(1.0f, tz_);
                    const float tr = smax * smax * itz * itz * (cam.focal_x * cam.focal_x * (1.0f + cam.limx * cam.limx) +
                                                                 cam.focal_y * cam.focal_y * (1.0f + cam.limy * cam.limy)) + 2.0f * VTGS_LOWPASS;
                    const float rb = cam.sigma_mult * sqrtf(tr) * 1.01f + 3.0f;
                    outside_band = (py_ - rb > (float)(cam.row1 * 16)) || (py_ + rb + 16.0f < (float)(cam.row0 * 16));
                }
            }
            if (outside_band) {
                radii[i] = 0;
                tiles_touched[i] = 0;
            } else {
            if (lite) {                                   // (band mode) now that the splat is known to matter
                k1_load_rest(it, i, rot_aligned, rotations, opacities, colors);
                qr = it.q.x; qx = it.q.y; qy = it.q.z; qz = it.q.w;
            }
            if (FUSED) {
                const float nrm = __fsqrt_rn(ffma(qz, qz, ffma(qy, qy, ffma(qx, qx, fmul(qr, qr)))));
                const float d = fmaxf(nrm, 1e-12f);
                if (d != 1.0f) {         // x / 1 = x: view-tied Gaussians keep the unit quaternion they were created with
                    qr = __fdiv_rn(qr, d); qx = __fdiv_rn(qx, d); qy = __fdiv_rn(qy, d); qz = __fdiv_rn(qz, d);
                }
                op = __fdiv_rn(1.0f, fadd(1.0f, vexpf(-it.op)));
                // get_depth_and_silhouette (reference utils/slam_helpers.py:217-234): z of w2c * p'
                c3 = fadd(ffma(fe.depth_row[2], z, ffma(fe.depth_row[1], y, fmul(fe.depth_row[0], x))), fe.depth_row[3]);
            } else {
                op = it.op;
                c3 = 0.0f;
            }
            splat_geometry(cam, x, y, z, sx, sy, sz, qr, qx, qy, qz, g);
            if (!FUSED) c3 = g.depth;

            GeomRecord rec;
            uint32_t tiles = 0;
            if (g.radius > 0) {
                const int miny = max(g.miny, cam.row0), maxy = min(g.maxy, cam.row1);
                const int hgt = max(0, maxy - miny);
                tiles = (uint32_t)((g.maxx - g.minx) * hgt);
                float pthr, hx, hy;
                cull_bounds(op, g.cov_a, g.cov_c, pthr, hx, hy);
                rec.q0 = make_float4(g.px, g.py, hx, hy);
                rec.q1 = make_float4(g.A, g.B, g.C, op);
                rec.q2 = make_float4(it.c0, it.c1, it.c2, c3);
                rec.q3 = make_float4(g.depth, pthr, __uint_as_float((uint32_t)g.minx | ((uint32_t)miny << 16)),
                                     __uint_as_float((uint32_t)g.maxx | ((uint32_t)(hgt > 0 ? maxy : miny) << 16)));
                w_minx = g.minx; w_maxx = g.maxx; w_miny = miny; w_maxy = hgt > 0 ? maxy : miny;
                cmax = fmaxf(cmax, fmaxf(fmaxf(fabsf(it.c0), fabsf(it.c1)), fmaxf(fabsf(it.c2), fabsf(c3))));
            } else {
                rec.q0 = make_float4(0.f, 0.f, -1e30f, -1e30f);
                rec.q1 = make_float4(0.f, 0.f, 0.f, 0.f);
                rec.q2 = make_float4(0.f, 0.f, 0.f, 0.f);
                rec.q3 = make_float4(g.depth, 1.0f, __uint_as_float(0u), __uint_as_float(0u));
            }
            geom[i] = rec;
            radii[i] = g.radius;
            tiles_touched[i] = tiles;
            }
        }
        // per-tile histogram, warp-aggregated: neighbouring Gaussians (neighbouring pixels of a view-tied
        // section) touch the same tiles, so one atomic per distinct tile per warp step instead of one per lane
        {
            // lanes with the SAME rect (one match per Gaussian, not per walk step) elect a leader that adds the group's
            // size to every tile of the rect
            const bool have = (w_maxx > w_minx) && (w_maxy > w_miny);
            if (__any_sync(VTGS_FULL_MASK, have)) {          // (a warp of culled / out-of-band splats skips the match)
                // lanes without a rect share one signature (they never act on it): the match costs per DISTINCT value
                const uint32_t sig_lo = have ? ((uint32_t)w_minx | ((uint32_t)w_miny << 16)) : 0xffffffffu;
                const uint32_t sig_hi = have ? ((uint32_t)w_maxx | ((uint32_t)w_maxy << 16)) : 0xffffffffu;
                const uint32_t peers = __match_any_sync(VTGS_FULL_MASK, ((unsigned long long)sig_hi << 32) | sig_lo);
                if (have && (peers & ((1u << (tid & 31)) - 1u)) == 0u) {
                    const uint32_t cnt = (uint32_t)__popc(peers);
                    for (int ty = w_miny; ty < w_maxy; ++ty)
                        for (int tx = w_minx; tx < w_maxx; ++tx) atomicAdd(&tile_counts[ty * cam.gx + tx], cnt);
                }
            }
        }
        i = i_next;
    }
    if (colour_max_bits != nullptr) {                     // non-negative floats order like their bit patterns
        uint32_t b = __float_as_uint(cmax);
        b = __reduce_max_sync(VTGS_FULL_MASK, b);
        if ((tid & 31) == 0 && b != 0u) atomicMax(colour_max_bits, b);
    }
}

// =============================== K2'/K5a': tile scan = tile ranges =========================
// One block.  Exclusive scan of the per-tile counts gives each tile's [begin, end) in the
// sorted list directly (identifyTileRanges for free); counts are re-zeroed to serve as the
// scatter cursors.  Empty tiles get (0,0) like the reference's memset.
__global__ void __launch_bounds__(1024)
tile_scan_kernel(uint32_t* __restrict__ tile_counts, uint32_t* __restrict__ ranges, int num_tiles,
                 uint64_t capacity, VtgsCounters* __restrict__ counters, uint32_t* __restrict__ tile_order) {
    VTGS_PDL_PROLOGUE();
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_carry;
    __shared__ uint32_t s_max[32];
    __shared__ uint32_t s_hist[32], s_cur[32], s_vmax;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    uint32_t vmax = 0;
    // the counts of up to 8 chunks of 1024 tiles are fetched before the first dependent use (one L2 round trip for
    // any image up to 8192 tiles instead of one per chunk)
    constexpr int PRE = 8;
    uint32_t pre[PRE];
#pragma unroll
    for (int k = 0; k < PRE; ++k) {
        const int t = k * 1024 + tid;
        pre[k] = t < num_tiles ? tile_counts[t] : 0u;
    }
    __syncthreads();
    int chunk = 0;
    for (int base = 0; base < num_tiles; base += 1024, ++chunk) {
        const int t = base + tid;
        uint32_t c = 0u;
        if (chunk < PRE) {
#pragma unroll
            for (int k = 0; k < PRE; ++k) if (k == chunk) c = pre[k];
        } else if (t < num_tiles) {
            c = tile_counts[t];
        }
        vmax = max(vmax, c);
        uint32_t incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t n = __shfl_up_sync(VTGS_FULL_MASK, incl, o);
            if (lane >= o) incl += n;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t n = __shfl_up_sync(VTGS_FULL_MASK, w, o);
                if (lane >= o) w += n;
            }
            s_warp[lane] = w;     // inclusive over warps
        }
        __syncthreads();
        const uint32_t carry = s_carry;
        const uint32_t excl = carry + (warp > 0 ? s_warp[warp - 1] : 0u) + incl - c;
        if (t < num_tiles) {
            uint64_t b = excl, e = (uint64_t)excl + c;
            if (b > capacity) b = capacity;
            if (e > capacity) e = capacity;
            if (c == 0) { b = 0; e = 0; }
            ranges[2 * t] = (uint32_t)b;
            ranges[2 * t + 1] = (uint32_t)e;
            tile_counts[t] = 0;
        }
        __syncthreads();
        if (tid == 1023) s_carry = carry + s_warp[31];
        __syncthreads();
    }
    vmax = max(vmax, __shfl_xor_sync(VTGS_FULL_MASK, vmax, 16));
    vmax = max(vmax, __shfl_xor_sync(VTGS_FULL_MASK, vmax, 8));
    vmax = max(vmax, __shfl_xor_sync(VTGS_FULL_MASK, vmax, 4));
    vmax = max(vmax, __shfl_xor_sync(VTGS_FULL_MASK, vmax, 2));
    vmax = max(vmax, __shfl_xor_sync(VTGS_FULL_MASK, vmax, 1));
    if (lane == 0) s_max[warp] = vmax;
    __syncthreads();
    if (tid == 0) {
        uint32_t m = 0;
        for (int w = 0; w < 32; ++w) m = max(m, s_max[w]);
        const uint32_t total = s_carry;
        counters->num_rendered = total;
        counters->overflow = (uint64_t)total > capacity ? 1u : 0u;
        counters->max_tile_pairs = m;
        s_vmax = m;
    }
    if (tile_order == nullptr) return;
    // Longest lists first: a 32-bucket counting sort of the tiles by list length (descending).  Blocks are handed to the
    // SMs in index order, so the sort / blend kernels, which take their tile from this order, start the heaviest tiles
    // first and fill the tail of the launch with light ones (order inside a bucket is arbitrary: no output depends on it).
    if (tid < 32) { s_hist[tid] = 0u; s_cur[tid] = 0u; }
    __syncthreads();
    const uint32_t denom = s_vmax + 1u;
    if (num_tiles > PRE * 1024) {                        // larger images than the prefetch covers: raster order
        for (int t = tid; t < num_tiles; t += 1024) tile_order[t] = (uint32_t)t;
        return;
    }
    uint32_t bk[PRE];
#pragma unroll
    for (int k = 0; k < PRE; ++k) {
        const int t = k * 1024 + tid;
        bk[k] = 31u - min(31u, (uint32_t)(((uint64_t)pre[k] * 32u) / denom));
        if (t < num_tiles) atomicAdd(&s_hist[bk[k]], 1u);
    }
    __syncthreads();
    if (warp == 0) {
        const uint32_t h = s_hist[lane];
        uint32_t incl = h;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t n = __shfl_up_sync(VTGS_FULL_MASK, incl, o);
            if (lane >= o) incl += n;
        }
        s_cur[lane] = incl - h;                          // bucket starts; bumped below as slots are claimed
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < PRE; ++k) {
        const int t = k * 1024 + tid;
        if (t < num_tiles) tile_order[atomicAdd(&s_cur[bk[k]], 1u)] = (uint32_t)t;
    }
}

// =============================== K3': scatter (duplicateWithKeys) ==========================
// One thread per Gaussian: for every touched tile claim a slot in that tile's segment and
// store (depth_bits << 32 | id).  Slot order inside a segment is arbitrary; the per-tile
// sort on the composite key makes the final order deterministic.
// WIDE (N >= 2^24): the low word is the full 32-bit Gaussian index, as in the reference's keys; the region mask that
// otherwise rides in the low byte is re-derived from the record when the tile's region lists are built.
template <bool WIDE>
__device__ __forceinline__ uint32_t key_id(uint32_t lo) { return WIDE ? lo : lo >> 8; }

template <bool WIDE>
__global__ void __launch_bounds__(256)
scatter_kernel(int64_t N, int gx, const GeomRecord* __restrict__ geom, const uint32_t* __restrict__ tiles_touched,
               const uint32_t* __restrict__ ranges, uint32_t* __restrict__ tile_cursor,
               uint64_t* __restrict__ pair_keys, const uint32_t* __restrict__ cand, const uint32_t* __restrict__ n_cand) {
    VTGS_PDL_PROLOGUE();
    // blocks of 256 Gaussians: all of them (one per CUDA block), or the candidate blocks of a tile band (persistent loop)
    const int64_t nblk = cand != nullptr ? (int64_t)*n_cand : (N + 255) / 256;
    for (int64_t trip = blockIdx.x; trip < nblk; trip += gridDim.x) {
    const int64_t i = (cand != nullptr ? (int64_t)cand[trip] : trip) * 256 + threadIdx.x;
    int minx = 0, miny = 0, maxx = 0, maxy = 0;
    uint64_t key = 0;
    float4 q0 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < N && tiles_touched[i] != 0) {
        const float4 q3 = geom[i].q3;
        q0 = geom[i].q0;
        const uint32_t rmin = __float_as_uint(q3.z), rmax = __float_as_uint(q3.w);
        minx = rmin & 0xffff; miny = rmin >> 16; maxx = rmax & 0xffff; maxy = rmax >> 16;
        key = ((uint64_t)__float_as_uint(q3.x) << 32) | (WIDE ? (uint64_t)(uint32_t)i : ((uint64_t)(uint32_t)i << 8));
    }
    warp_tile_walk(minx, miny, maxx, maxy, gx, [&](int tile, int tx, int ty, uint32_t peers, int rank, bool leader) {
        uint32_t base = 0;
        if (leader) base = ranges[2 * tile] + atomicAdd(&tile_cursor[tile], (uint32_t)__popc(peers));
        base = __shfl_sync(peers, base, __ffs(peers) - 1);
        const uint32_t pos = base + (uint32_t)rank;
        // low 8 bits: which of this tile's 8 warp regions the splat's alpha >= 1/255 box touches (ids are unique, so
        // these bits never decide the order; the sort kernel reads them back instead of gathering the record again)
        const uint32_t rmask = WIDE ? 0u : region_mask(q0, (float)(tx * 16), (float)(ty * 16));
        if (pos < ranges[2 * tile + 1]) pair_keys[pos] = key | rmask;
    });
    }
}

// =============================== K4': per-tile sort ========================================
// One block per tile.  Normalised bitonic network (every compare-exchange ascending, the
// first sub-step of each merge mirrors the index) so that indices >= n act as +inf padding
// without being stored.  It serves the tie fall-back of the radix sorts below (shared or global memory).
constexpr int SORT_SMEM_ELEMS = 2048;

__device__ __forceinline__ void bitonic_network(uint64_t* __restrict__ s, int n, int npad) {
    const int pairs = npad >> 1;
    for (int lk = 1; (1 << lk) <= npad; ++lk) {
        const int k = 1 << lk;
        // flip step: partner is the mirror inside the block of k
        {
            const int lh = lk - 1, hm = (1 << lh) - 1;
            for (int t = threadIdx.x; t < pairs; t += blockDim.x) {
                const int blk = t >> lh, off = t & hm;
                const int i = (blk << lk) + off, p = (blk << lk) + (k - 1 - off);
                if (p < n) {
                    const uint64_t a = s[i], b = s[p];
                    if (a > b) { s[i] = b; s[p] = a; }
                }
            }
            __syncthreads();
        }
        for (int lj = lk - 2; lj >= 0; --lj) {
            const int j = 1 << lj;
            for (int t = threadIdx.x; t < pairs; t += blockDim.x) {
                const int i = ((t >> lj) << (lj + 1)) | (t & (j - 1)), p = i + j;
                if (p < n) {
                    const uint64_t a = s[i], b = s[p];
                    if (a > b) { s[i] = b; s[p] = a; }
                }
            }
            __syncthreads();
        }
    }
}

// Register-resident bitonic sort of up to 256*E keys by one 256-thread block: thread t holds the E
// consecutive elements [t*E, t*E+E).  Exchange distance j < E stays inside a thread, E <= j < 32E is
// a warp shuffle, only the three largest distances go through shared memory (6 barriers-pairs for
// 1024 keys instead of 55).  Unused slots hold ~0 (sorts last).
template <int E>
__device__ __forceinline__ void bitonic_regs(uint64_t (&v)[E], uint64_t* __restrict__ s_x, int tid, int npad) {
    for (int k = 2; k <= npad; k <<= 1) {
        const bool asc_t = ((tid * E) & k) == 0;                         // direction of this thread's run when k >= E
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j < E) {
#pragma unroll
                for (int jj = E / 2; jj >= 1; jj >>= 1) {               // compile-time distance: registers stay registers
                    if (j != jj) continue;
#pragma unroll
                    for (int e = 0; e < E; ++e) {
                        if ((e & jj) == 0) {
                            const bool asc = k >= E ? asc_t : ((e & k) == 0);
                            const uint64_t a = v[e], b = v[e | jj];
                            const bool sw = (a > b) == asc;
                            v[e] = sw ? b : a;
                            v[e | jj] = sw ? a : b;
                        }
                    }
                }
            } else if (j < 32 * E) {
                const int tm = j / E;                                   // lane bit
                const bool lower = (tid & tm) == 0;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const uint64_t o = __shfl_xor_sync(VTGS_FULL_MASK, v[e], tm);
                    const bool take_min = lower == asc_t;
                    v[e] = ((o < v[e]) == take_min) ? o : v[e];
                }
            } else {
                const int tm = j / E;                                   // warp bit
                const bool lower = (tid & tm) == 0;
                __syncthreads();
#pragma unroll
                for (int e = 0; e < E; ++e) s_x[e * 256 + tid] = v[e];   // [e][tid]: conflict-free
                __syncthreads();
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const uint64_t o = s_x[e * 256 + (tid ^ tm)];
                    const bool take_min = lower == asc_t;
                    v[e] = ((o < v[e]) == take_min) ? o : v[e];
                }
            }
        }
    }
}

template <int E, bool WIDE>
__device__ __forceinline__ void sort_segment_regs(uint64_t* __restrict__ s_x, uint64_t* __restrict__ keys, uint32_t* __restrict__ ids,
                                                  int n, int tid) {
    uint64_t v[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int i = tid * E + e;
        v[e] = i < n ? keys[i] : ~0ull;
    }
    int npad = 2 * E;                       // at least one cross-thread stage keeps the code uniform
    while (npad < n) npad <<= 1;
    bitonic_regs<E>(v, s_x, tid, npad);
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int i = tid * E + e;
        if (i < n) { keys[i] = v[e]; ids[i] = key_id<WIDE>((uint32_t)v[e]); }
    }
}

// Stable LSD radix sort of a tile's segment (256 < n <= SORT_SMEM_ELEMS) on the DEPTH word of the keys, 8 bits per
// pass, only over the bits in which the tile's depths actually differ (a tile sees a narrow depth range: usually
// 3 passes).  Warp w owns the contiguous chunk [32 E w, 32 E (w + 1)), element (round e, lane l) = chunk + 32 e + l,
// so that (warp, round, lane) order IS list order: ranks come from __match_any_sync inside a round, running
// per-warp digit counters across rounds and one block scan over (digit, warp) per pass -- ~1/5 of the bitonic
// network's instructions.  The scatter's slot order is arbitrary, so equal depths (rare) would come out in arbitrary
// order: a tile that holds any tie re-sorts its (already depth-ordered) keys with the full 64-bit network.
template <int E>
__device__ __forceinline__ void sort_segment_radix(uint64_t* __restrict__ s_keys, uint32_t (*__restrict__ wh)[256],
                                                   uint32_t* __restrict__ s_red, const uint64_t* __restrict__ keys_in, int n, int tid) {
    const int lane = tid & 31, warp = tid >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    const int cbase = warp * 32 * E + lane;
    uint64_t v[E];
    uint32_t dmin = 0xffffffffu, dmax = 0u;
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int i = cbase + 32 * e;
        v[e] = ~0ull;
        if (i < n) {
            v[e] = keys_in[i];
            const uint32_t hi = (uint32_t)(v[e] >> 32);
            dmin = min(dmin, hi);
            dmax = max(dmax, hi);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        dmin = min(dmin, __shfl_xor_sync(VTGS_FULL_MASK, dmin, o));
        dmax = max(dmax, __shfl_xor_sync(VTGS_FULL_MASK, dmax, o));
    }
    if (lane == 0) { s_red[warp] = dmin; s_red[8 + warp] = dmax; }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < 8; ++w) { dmin = min(dmin, s_red[w]); dmax = max(dmax, s_red[8 + w]); }
    const int hb = 32 - __clz((int)(dmin ^ dmax));            // low bits in which the depths differ (0: all equal)
    __syncthreads();                                           // s_red is reused by the scans below
    for (int shift = 0; shift < hb; shift += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) wh[warp][lane + 32 * k] = 0u;
        __syncwarp();
        uint32_t off[E];
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const bool valid = cbase + 32 * e < n;
            const uint32_t vm = __ballot_sync(VTGS_FULL_MASK, valid);
            uint32_t d = 0u, peers = 0u, prev = 0u;
            if (valid) {
                d = (uint32_t)(v[e] >> (32 + shift)) & 0xffu;
                peers = __match_any_sync(vm, d);
                prev = wh[warp][d];
            }
            __syncwarp();
            const uint32_t rank = __popc(peers & lt);
            if (valid && rank == 0u) wh[warp][d] = prev + (uint32_t)__popc(peers);
            __syncwarp();
            off[e] = prev + rank;
        }
        __syncthreads();
        {   // exclusive scan over (digit, warp): thread b owns digit b
            uint32_t run = 0u;
#pragma unroll
            for (int w = 0; w < 8; ++w) { const uint32_t c = wh[w][tid]; wh[w][tid] = run; run += c; }
            uint32_t incl = run;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(VTGS_FULL_MASK, incl, o);
                if (lane >= o) incl += t;
            }
            if (lane == 31) s_red[warp] = incl;
            __syncthreads();
            uint32_t dbase = incl - run;
#pragma unroll
            for (int w = 0; w < 8; ++w) if (w < warp) dbase += s_red[w];
#pragma unroll
            for (int w = 0; w < 8; ++w) wh[w][tid] += dbase;
        }
        __syncthreads();
#pragma unroll
        for (int e = 0; e < E; ++e)
            if (cbase + 32 * e < n) s_keys[wh[warp][(uint32_t)(v[e] >> (32 + shift)) & 0xffu] + off[e]] = v[e];
        __syncthreads();
#pragma unroll
        for (int e = 0; e < E; ++e)
            if (cbase + 32 * e < n) v[e] = s_keys[cbase + 32 * e];
    }
    if (hb == 0) {
#pragma unroll
        for (int e = 0; e < E; ++e)
            if (cbase + 32 * e < n) s_keys[cbase + 32 * e] = v[e];
        __syncthreads();
    }
    // Equal depths: with ~10^3 floats from a narrow range per tile a coincidence somewhere is likely (birthday
    // bound), but runs are short.  Every member of a run finds its place by counting the run's smaller ids
    // (low words: id << 8 | mask, ids are unique); runs longer than TIE_RUN_MAX fall back to the 64-bit network.
    constexpr int TIE_RUN_MAX = 48;
    bool moved = false, too_long = false;
    int newpos[E];
    // the list is depth-sorted: equal depths TIE_RUN_MAX apart mean a longer run -- one load decides it for everyone
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int i = cbase + 32 * e;
        if (i < n && i >= TIE_RUN_MAX) too_long |= (uint32_t)(s_keys[i - TIE_RUN_MAX] >> 32) == (uint32_t)(v[e] >> 32);
    }
    const bool any_long = __syncthreads_or(too_long) != 0;
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int i = cbase + 32 * e;
        newpos[e] = i;
        if (i < n && !any_long) {
            const uint32_t hi = (uint32_t)(v[e] >> 32), lo = (uint32_t)v[e];
            int shiftpos = 0, steps = 0;
            for (int j = i - 1; j >= 0; --j) {
                const uint64_t o = s_keys[j];
                if ((uint32_t)(o >> 32) != hi) break;
                if ((uint32_t)o > lo) --shiftpos;
                if (++steps > TIE_RUN_MAX) { too_long = true; break; }
            }
            for (int j = i + 1; j < n; ++j) {
                const uint64_t o = s_keys[j];
                if ((uint32_t)(o >> 32) != hi) break;
                if ((uint32_t)o < lo) ++shiftpos;
                if (++steps > TIE_RUN_MAX) { too_long = true; break; }
            }
            newpos[e] = i + shiftpos;
            moved |= shiftpos != 0;
        }
    }
    const bool any_moved = __syncthreads_or(moved) != 0;          // (a barrier: every read of s_keys above is done)
    if (any_long) {
        // long runs (e.g. a fronto-parallel wall seen from the pose its quantised depths were measured at): full
        // 64-bit sort of the tile with the register / shuffle bitonic network (3x cheaper than the shared-memory one)
        constexpr int E2 = E <= 2 ? 2 : (E <= 4 ? 4 : 8);
        uint64_t w[E2];
#pragma unroll
        for (int e = 0; e < E2; ++e) w[e] = tid * E2 + e < n ? s_keys[tid * E2 + e] : ~0ull;
        int npad = 2 * E2;
        while (npad < n) npad <<= 1;
        bitonic_regs<E2>(w, s_keys, tid, npad);          // s_keys doubles as the exchange buffer (barriers inside)
        __syncthreads();
#pragma unroll
        for (int e = 0; e < E2; ++e)
            if (tid * E2 + e < n) s_keys[tid * E2 + e] = w[e];
        __syncthreads();
    } else if (any_moved) {
#pragma unroll
        for (int e = 0; e < E; ++e)
            if (cbase + 32 * e < n && newpos[e] != cbase + 32 * e) s_keys[newpos[e]] = v[e];
        __syncthreads();
    }
}

// The same radix sort for long segments (n > SORT_SMEM_ELEMS: several overlapping sections in one view): keys
// stream from / to global memory (L1 / L2 resident: a tile's segment is a few tens of KB), ping-ponging between the
// segment and `scratch` (the tile's still unused slice of the region-list arena, 8 n entries).  Nothing is held in
// registers, so any n works: every pass reads its keys twice (count, then rank + scatter).
__device__ __noinline__ void sort_segment_radix_long(uint64_t* keys, uint64_t* scratch, uint32_t (*wh)[256], uint32_t* s_red,
                                                     int n, int tid) {
    const int lane = tid & 31, warp = tid >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    const int chunk = ((n + 255) >> 8) << 5;                 // keys per warp (a multiple of 32), list order = (warp, round, lane)
    const int wbeg = min(n, warp * chunk), wend = min(n, wbeg + chunk);
    uint32_t dmin = 0xffffffffu, dmax = 0u;
    for (int i = tid; i < n; i += 256) {
        const uint32_t hi = (uint32_t)(keys[i] >> 32);
        dmin = min(dmin, hi);
        dmax = max(dmax, hi);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        dmin = min(dmin, __shfl_xor_sync(VTGS_FULL_MASK, dmin, o));
        dmax = max(dmax, __shfl_xor_sync(VTGS_FULL_MASK, dmax, o));
    }
    if (lane == 0) { s_red[warp] = dmin; s_red[8 + warp] = dmax; }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < 8; ++w) { dmin = min(dmin, s_red[w]); dmax = max(dmax, s_red[8 + w]); }
    const int hb = 32 - __clz((int)(dmin ^ dmax));
    __syncthreads();
    uint64_t* src = keys;
    uint64_t* dst = scratch;
    for (int shift = 0; shift < hb; shift += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) wh[warp][lane + 32 * k] = 0u;
        __syncwarp();
        for (int base = wbeg; base < wend; base += 32) {
            const bool valid = base + lane < wend;
            const uint32_t vm = __ballot_sync(VTGS_FULL_MASK, valid);
            if (valid) {
                const uint32_t d = (uint32_t)(src[base + lane] >> (32 + shift)) & 0xffu;
                const uint32_t peers = __match_any_sync(vm, d);
                if ((peers & lt) == 0u) wh[warp][d] += (uint32_t)__popc(peers);       // one lane per distinct digit
            }
            __syncwarp();
        }
        __syncthreads();
        {
            uint32_t run = 0u;
#pragma unroll
            for (int w = 0; w < 8; ++w) { const uint32_t c = wh[w][tid]; wh[w][tid] = run; run += c; }
            uint32_t incl = run;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(VTGS_FULL_MASK, incl, o);
                if (lane >= o) incl += t;
            }
            if (lane == 31) s_red[warp] = incl;
            __syncthreads();
            uint32_t dbase = incl - run;
#pragma unroll
            for (int w = 0; w < 8; ++w) if (w < warp) dbase += s_red[w];
#pragma unroll
            for (int w = 0; w < 8; ++w) wh[w][tid] += dbase;
        }
        __syncthreads();
        for (int base = wbeg; base < wend; base += 32) {
            const bool valid = base + lane < wend;
            const uint32_t vm = __ballot_sync(VTGS_FULL_MASK, valid);
            uint64_t k = 0ull;
            uint32_t d = 0u, peers = 0u, prev = 0u;
            if (valid) {
                k = src[base + lane];
                d = (uint32_t)(k >> (32 + shift)) & 0xffu;
                peers = __match_any_sync(vm, d);
                prev = wh[warp][d];
            }
            __syncwarp();
            if (valid) {
                const uint32_t rank = __popc(peers & lt);
                if (rank == 0u) wh[warp][d] = prev + (uint32_t)__popc(peers);
                dst[prev + rank] = k;
            }
            __syncwarp();
        }
        __syncthreads();
        uint64_t* t = src; src = dst; dst = t;
    }
    if (src != keys) {
        for (int i = tid; i < n; i += 256) keys[i] = src[i];
        __syncthreads();
    }
    // equal-depth runs: order by id (see sort_segment_radix); the repaired list is assembled in `scratch`
    constexpr int TIE_RUN_MAX = 48;
    bool moved = false, too_long = false;
    for (int i = tid + TIE_RUN_MAX; i < n; i += 256)
        too_long |= (uint32_t)(keys[i - TIE_RUN_MAX] >> 32) == (uint32_t)(keys[i] >> 32);
    const bool any_long = __syncthreads_or(too_long) != 0;
    for (int i = tid; i < n && !any_long; i += 256) {
        const uint64_t k = keys[i];
        const uint32_t hi = (uint32_t)(k >> 32), lo = (uint32_t)k;
        int shiftpos = 0, steps = 0;
        for (int j = i - 1; j >= 0; --j) {
            const uint64_t o = keys[j];
            if ((uint32_t)(o >> 32) != hi) break;
            if ((uint32_t)o > lo) --shiftpos;
            if (++steps > TIE_RUN_MAX) { too_long = true; break; }
        }
        for (int j = i + 1; j < n; ++j) {
            const uint64_t o = keys[j];
            if ((uint32_t)(o >> 32) != hi) break;
            if ((uint32_t)o < lo) ++shiftpos;
            if (++steps > TIE_RUN_MAX) { too_long = true; break; }
        }
        scratch[i + shiftpos] = k;
        moved |= shiftpos != 0;
    }
    const bool any_moved = __syncthreads_or(moved) != 0;
    if (any_long) {
        int npad = 2;
        while (npad < n) npad <<= 1;
        bitonic_network(keys, n, npad);
    } else if (any_moved) {
        for (int i = tid; i < n; i += 256) keys[i] = scratch[i];
        __syncthreads();
    }
}

// After a tile's list is sorted: per-region lists.  Every (sorted) entry is tested once against the
// tile's 8 warp regions (box of its alpha >= 1/255 ellipse) and appended, in list order, to the list of
// every region it may touch as (Gaussian id, 1-based position in the tile list).  The blend kernels then
// walk only their own region's list: the culling is done once per (tile, splat) here instead of once per
// (warp, splat) in each of the two blend kernels.
// Arena: region r of a tile with list [rb, re) owns slots [8 rb + r (re - rb), 8 rb + (r + 1)(re - rb)).
template <bool WIDE>
__device__ __forceinline__ void build_region_lists(const uint64_t* keys, int n, uint32_t rb, int tile, const GeomRecord* __restrict__ geom,
                                                   float tox, float toy, uint2* __restrict__ region_pairs, uint32_t* __restrict__ region_cnt) {
    // warp r compacts region r's entries of the whole (sorted) list: ballot + prefix popcount keep the list order,
    // the running base lives in a register -- no shared counters, no block barriers between chunks
    const int tid = threadIdx.x, lane = tid & 31, r = tid >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    __syncthreads();                                   // the sorted keys written by other threads are visible
    uint2* __restrict__ out = region_pairs + (size_t)8 * rb + (size_t)r * n;
    uint32_t base = 0u;
    int i0 = 0;
    for (; i0 + 64 <= n; i0 += 64) {                   // two chunks per trip: independent loads
        const uint32_t lo0 = (uint32_t)keys[i0 + lane], lo1 = (uint32_t)keys[i0 + 32 + lane];
        const uint32_t rm0 = WIDE ? region_mask(geom[lo0].q0, tox, toy) : lo0, rm1 = WIDE ? region_mask(geom[lo1].q0, tox, toy) : lo1;
        const bool h0 = (rm0 >> r) & 1u, h1 = (rm1 >> r) & 1u;
        const uint32_t b0 = __ballot_sync(VTGS_FULL_MASK, h0), b1 = __ballot_sync(VTGS_FULL_MASK, h1);
        const uint32_t base1 = base + (uint32_t)__popc(b0);
        if (h0) out[base + __popc(b0 & lt)] = make_uint2(key_id<WIDE>(lo0), (uint32_t)(i0 + lane) + 1u);
        if (h1) out[base1 + __popc(b1 & lt)] = make_uint2(key_id<WIDE>(lo1), (uint32_t)(i0 + 32 + lane) + 1u);
        base = base1 + (uint32_t)__popc(b1);
    }
    for (; i0 < n; i0 += 32) {
        const int i = i0 + lane;
        const uint32_t lo = i < n ? (uint32_t)keys[i] : 0u;
        const uint32_t rm = WIDE ? (i < n ? region_mask(geom[lo].q0, tox, toy) : 0u) : lo;
        const bool h = (rm >> r) & 1u;
        const uint32_t bal = __ballot_sync(VTGS_FULL_MASK, h);
        if (h) out[base + __popc(bal & lt)] = make_uint2(key_id<WIDE>(lo), (uint32_t)i + 1u);
        base += (uint32_t)__popc(bal);
    }
    if (lane == 0) region_cnt[(size_t)tile * 8 + r] = base;
}

template <bool WIDE>
__global__ void __launch_bounds__(256, 4)
tile_sort_kernel(const __grid_constant__ CamConst cam, const uint32_t* __restrict__ ranges, int tile0,
                 uint64_t* __restrict__ pair_keys, uint32_t* __restrict__ point_list, const GeomRecord* __restrict__ geom,
                 uint2* __restrict__ region_pairs, uint32_t* __restrict__ region_cnt, const uint32_t* __restrict__ tile_order) {
    VTGS_PDL_PROLOGUE();
    extern __shared__ __align__(16) uint64_t s_keys[];
    __shared__ uint32_t s_wh[8][256];
    __shared__ uint32_t s_cnt[64];
    const int tile = tile0 + (tile_order ? (int)tile_order[blockIdx.x] : (int)blockIdx.x);
    const uint32_t b = ranges[2 * tile], e = ranges[2 * tile + 1];
    const int n = (int)(e - b);
    if (n <= 0) {
        if (threadIdx.x < 8) region_cnt[(size_t)tile * 8 + threadIdx.x] = 0;
        return;
    }
    const uint64_t* sorted = pair_keys + b;
    if (n <= 256) sort_segment_regs<2, WIDE>(s_keys, pair_keys + b, point_list + b, n, threadIdx.x);
    else if (n <= 2048) {
        const uint64_t* in = pair_keys + b;
        const int tid = threadIdx.x;
        if (n <= 512) sort_segment_radix<2>(s_keys, s_wh, s_cnt, in, n, tid);
        else if (n <= 768) sort_segment_radix<3>(s_keys, s_wh, s_cnt, in, n, tid);
        else if (n <= 1024) sort_segment_radix<4>(s_keys, s_wh, s_cnt, in, n, tid);
        else if (n <= 1536) sort_segment_radix<6>(s_keys, s_wh, s_cnt, in, n, tid);
        else sort_segment_radix<8>(s_keys, s_wh, s_cnt, in, n, tid);
        for (int i = tid; i < n; i += 256) {
            const uint64_t k = s_keys[i];
            pair_keys[b + i] = k;
            point_list[b + i] = key_id<WIDE>((uint32_t)k);
        }
        sorted = s_keys;
    } else {
        sort_segment_radix_long(pair_keys + b, reinterpret_cast<uint64_t*>(region_pairs + (size_t)8 * b), s_wh, s_cnt, n, threadIdx.x);
        for (int i = threadIdx.x; i < n; i += 256) point_list[b + i] = key_id<WIDE>((uint32_t)pair_keys[b + i]);
    }
    build_region_lists<WIDE>(sorted, n, b, tile, geom, (float)((tile % cam.gx) * 16), (float)((tile / cam.gx) * 16), region_pairs, region_cnt);
}

// =============================== K5': forward blend ========================================
// Block = FWD_WARPS INDEPENDENT warps (no block barrier); a warp owns one 8x4-pixel region of a tile and walks that
// region's list (built by the sort kernel) in CHUNKS of FWD_GC groups of 32 splats (blend_common.cuh):
//   stage  lane = splat : software-prefetched gathers of the 64-byte records -> shared memory (40 B per splat);
//   P1     lane = splat : row-interval test of the region's 32 pixels, masks transposed to pixel lanes;
//   P2     lane = pixel : every lane walks ITS OWN masks of the whole chunk front to back without re-converging at
//                         group boundaries -- exact power / alpha / T tests and the blend in list order, so
//                         n_contrib, final_T and the planes are bit-identical to the one-splat-at-a-time oracle;
//                         the masks are reduced in place to the splats actually blended (consumed by K6').
// Planes: API mode 3 colours (+ depth plane), fused mode r,g,b,z,sil,z^2.
// Cold path of the pixel walk: the pixel saturated at `bit` of word gg -- that splat and every later one of the chunk
// were not applied.  col = &pm[0][lane] (words are 32 apart).
__device__ __noinline__ void clear_mask_bit(uint32_t* word, uint32_t bit) { *word &= ~bit; }
__device__ __noinline__ void truncate_masks(uint32_t* col, int gg, int gc, uint32_t bit) {
    col[gg * 32] &= bit - 1u;
    for (int g2 = gg + 1; g2 < gc; ++g2) col[g2 * 32] = 0u;
}

#ifndef VTGS_FWD_WARPS
#define VTGS_FWD_WARPS 4
#endif
#ifndef VTGS_FWD_GC
#define VTGS_FWD_GC 6
#endif
#ifndef VTGS_FWD_NZ
#define VTGS_FWD_NZ 1                       // 1: per-pixel bitmap of the chunk's non-empty mask words instead of the sentinel search
#endif
constexpr int FWD_WARPS = VTGS_FWD_WARPS;   // warps (regions) per block: a tile is covered by 8 / FWD_WARPS blocks
constexpr int FWD_GC = VTGS_FWD_GC;         // groups per chunk: 1408 B of shared memory per group and warp
#ifndef VTGS_FWD_BLOCKS
#define VTGS_FWD_BLOCKS ((FWD_GC <= 6 ? 24 : 20) / FWD_WARPS)
#endif
template <bool FUSED>
__global__ void __launch_bounds__(32 * FWD_WARPS, VTGS_FWD_BLOCKS)
blend_forward_kernel(const __grid_constant__ CamConst cam, const uint32_t* __restrict__ ranges,
                     const uint2* __restrict__ region_pairs, const uint32_t* __restrict__ region_cnt,
                     uint32_t* __restrict__ region_masks, uint32_t* __restrict__ region_done,
                     const GeomRecord* __restrict__ geom,
                     float* __restrict__ out_color, float* __restrict__ out_depth,
                     float* __restrict__ final_T, uint32_t* __restrict__ n_contrib, const uint32_t* __restrict__ tile_order) {
    VTGS_PDL_PROLOGUE();
    __shared__ ChunkSmem<FWD_GC> Ws[FWD_WARPS];

    constexpr int BPT = 8 / FWD_WARPS;                                  // blocks per tile
    const int tile = cam.row0 * cam.gx + (tile_order ? (int)tile_order[blockIdx.x / BPT] : (int)(blockIdx.x / BPT));
    const int tile_x = tile % cam.gx, tile_y = tile / cam.gx;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = (blockIdx.x % BPT) * FWD_WARPS + (tid >> 5);       // region index inside the tile
    ChunkSmem<FWD_GC>& S = Ws[tid >> 5];
    const int rx0 = tile_x * 16 + (warp % REGIONS_X) * REGION_W, ry0 = tile_y * 16 + (warp / REGIONS_X) * REGION_H;
    const int pix_x = rx0 + (lane % REGION_W), pix_y = ry0 + (lane / REGION_W);
    const bool inside = pix_x < cam.W && pix_y < cam.H;
    const float pxf = (float)pix_x, pyf = (float)pix_y;
    const float x0f = (float)rx0, y0f = (float)ry0;

    const uint32_t rb = ranges[2 * tile], re = ranges[2 * tile + 1];
    const int n = (int)region_cnt[(size_t)tile * 8 + warp];
    const uint2* __restrict__ list = region_pairs + (size_t)8 * rb + (size_t)warp * (re - rb);
    uint32_t* __restrict__ masks = region_masks + mask_arena_base(rb, re, tile, warp);
    const int ngroups = (n + 31) >> 5;

    float T = 1.0f;
    float C0 = 0.f, C1 = 0.f, C2 = 0.f, C3 = 0.f, C4 = 0.f, C5 = 0.f;
    int last_k = -1;                    // region-list index of the last splat this pixel blended
    bool done = !inside;

    // software pipeline: list entries two groups ahead, records one group ahead
    uint2 ent_next = lane < n ? list[lane] : make_uint2(0u, 0u);
    uint2 ent_next2 = (32 + lane) < n ? list[32 + lane] : make_uint2(0u, 0u);
    SplatRegs nxt;
    load_splat(nxt, lane < n, geom, ent_next);
    bool all_done = __all_sync(VTGS_FULL_MASK, done);
    int g0 = 0;
    for (; g0 < ngroups && !all_done; g0 += FWD_GC) {
        const int gc = min(FWD_GC, ngroups - g0);
        __syncwarp();                                   // the previous chunk's reads of S are complete
        // ---- stage + P1, lane = splat
#if VTGS_FWD_NZ
        uint32_t nz = 0u;                               // groups of the chunk in which this pixel has a candidate
#endif
        for (int gg = 0; gg < gc; ++gg) {
            const SplatRegs cur = nxt;
            const int k = (g0 + gg) * 32 + lane;
            const bool have = k < n;
            ent_next = ent_next2;
            ent_next2 = (k + 64) < n ? list[k + 64] : make_uint2(0u, 0u);
            load_splat(nxt, (k + 32) < n, geom, ent_next);
            uint32_t em = 0u;
            if (have) {
                S.r0[gg * 32 + lane] = make_float4(cur.a.x, cur.a.y, cur.b.x, cur.b.y);
                S.r1[gg * 32 + lane] = make_float4(cur.b.z, cur.a.w, cur.c.x, cur.c.y);
                S.r2[gg * 32 + lane] = make_float2(cur.c.z, cur.c.w);
                em = p1_rows(cur.a.x, cur.a.y, cur.b.x, cur.b.y, cur.b.z, cur.b.w, x0f, y0f);
            }
            const uint32_t m = warp_transpose_bits(em, lane);
            S.pm[gg][lane] = done ? 0u : m;
#if VTGS_FWD_NZ
            nz |= (m != 0u && !done) ? (1u << gg) : 0u;
#endif
        }
#if !VTGS_FWD_NZ
        S.pm[gc][lane] = 0xffffffffu;                   // sentinel: the search for a lane's next non-empty word stops here
#endif
        __syncwarp();
        // ---- P2, lane = pixel: one pass over the chunk's masks, no re-convergence between groups.  The mask corrections
        // (P1's superset / the T test rejecting a splat) are cold and kept out of line.
        if (!done) {
            int gg = 0, lk = -1;
#if VTGS_FWD_NZ
            uint32_t m = 0u;
            for (;;) {
                if (m == 0u) {                             // next group with a candidate for this pixel: one step, whatever the gap
                    if (nz == 0u) break;
                    gg = __ffs(nz) - 1;
                    nz &= nz - 1u;
                    m = S.pm[gg][lane];
                }
#else
            uint32_t m = S.pm[0][lane];
            for (;;) {
                while (m == 0u) m = S.pm[++gg][lane];      // (the sentinel row bounds it)
                if (gg >= gc) break;
#endif
                const uint32_t bit = m & (0u - m);
                m ^= bit;
                const int idx = gg * 32 + msb_index(bit);
                const float4 q0 = S.r0[idx], q1 = S.r1[idx];
                const float power = power_of(q0.z, q0.w, q1.x, fsub(q0.x, pxf), fsub(q0.y, pyf));
                // fused mode: opacity = sigmoid(.) < 1 and power >= pthr - margins ~ -5.6: no clamp needed (same bits)
                const float alpha = fminf(VTGS_ALPHA_MAX, fmul(q1.y, vexpf<!FUSED>(power)));
                if (power > 0.0f || alpha < VTGS_ALPHA_MIN) {        // P1 is a superset: drop the pair from the mask
                    clear_mask_bit(&S.pm[gg][lane], bit);
                    continue;
                }
                const float test_T = fmul(T, fsub(1.0f, alpha));
                if (test_T < VTGS_T_MIN) {                           // saturated: this and all later splats are not applied
                    truncate_masks(&S.pm[0][lane], gg, gc, bit);
                    done = true;
                    break;
                }
                const float2 q2 = S.r2[idx];
                C0 = ffma(fmul(q1.z, alpha), T, C0);
                C1 = ffma(fmul(q1.w, alpha), T, C1);
                C2 = ffma(fmul(q2.x, alpha), T, C2);
                C3 = ffma(fmul(q2.y, alpha), T, C3);
                if (FUSED) {
                    C4 = ffma(alpha, T, C4);                               // 1.0 * alpha * T
                    C5 = ffma(fmul(fmul(q2.y, q2.y), alpha), T, C5);       // z^2 channel
                }
                T = test_T;
                lk = idx;
            }
            if (lk >= 0) last_k = g0 * 32 + lk;
        }
        __syncwarp();
        for (int gg = 0; gg < gc; ++gg) masks[(g0 + gg) * 32 + lane] = S.pm[gg][lane];      // coalesced, for K6'
        all_done = __all_sync(VTGS_FULL_MASK, done);
    }
    if (lane == 0) region_done[(size_t)tile * 8 + warp] = (uint32_t)min(g0, ngroups);

    if (inside) {
        const size_t P = (size_t)cam.W * cam.H;
        const size_t pid = (size_t)pix_y * cam.W + pix_x;
        final_T[pid] = T;
        n_contrib[pid] = last_k >= 0 ? list[last_k].y : 0u;         // 1-based position in the TILE list
        out_color[pid] = ffma(T, cam.bg[0], C0);
        out_color[P + pid] = ffma(T, cam.bg[1], C1);
        out_color[2 * P + pid] = ffma(T, cam.bg[2], C2);
        if (FUSED) {
            out_color[3 * P + pid] = C3;
            out_color[4 * P + pid] = C4;
            out_color[5 * P + pid] = C5;
        } else {
            out_depth[pid] = C3;
        }
    }
}

// Rows outside the band keep the background (multi-GPU tracking: each rank owns a band).
__global__ void fill_outside_band_kernel(const __grid_constant__ CamConst cam, int planes,
                                         float* __restrict__ out_color, float* __restrict__ out_depth,
                                         float* __restrict__ final_T, uint32_t* __restrict__ n_contrib) {
    VTGS_PDL_PROLOGUE();
    const size_t P = (size_t)cam.W * cam.H;
    const size_t pid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (pid >= P) return;
    const int y = (int)(pid / cam.W);
    if (y >= cam.row0 * 16 && y < cam.row1 * 16) return;
    final_T[pid] = 1.0f;
    n_contrib[pid] = 0;
    for (int ch = 0; ch < planes; ++ch) out_color[ch * P + pid] = ch < 3 ? cam.bg[ch] : 0.0f;
    if (out_depth) out_depth[pid] = 0.0f;
}

// =============================== host orchestration ======================================
// The forward of both paths: API mode (vtgs_forward) and the fused path (vtgs_fused_forward: `fused`, front end `fe`).
static int launch_forward(const VtgsCamera* camera, int64_t N, bool fused, const FrontEnd& fe,
                          const float* means3D, const float* scales, const float* rotations,
                          const float* opacities, const float* colors,
                          float* out_color, float* out_depth, int32_t* radii, VtgsBuffers* buf,
                          cudaStream_t stream) {
    const CamConst cam = make_cam_const(*camera);
    const int num_tiles = cam.gx * cam.gy;
    if (cam.gx > 0xffff || cam.gy > 0xffff) { set_error("image too large for packed tile rects"); return VTGS_E_INVALID; }
    if (N > (int64_t)0xffffffffll) { set_error("at most 2^32 - 1 Gaussians per render (32-bit id in the sort key, as in the reference)"); return VTGS_E_UNSUPPORTED; }
    const bool wide = N >= ((int64_t)1 << 24);          // the compact key (id << 8 | region mask) holds 24-bit ids
    GeomRecord* geom = reinterpret_cast<GeomRecord*>(buf->geom);
    VTGS_CUDA_CHECK(cudaMemsetAsync(buf->tile_counts, 0, sizeof(uint32_t) * (num_tiles + 3), stream));     // + the candidate-list counter, max |colour|, max |dL/dpixel|
    const int blocks = (int)((N + 255) / 256);
    const int k1_blocks = blocks < 148 * 6 ? blocks : 148 * 6;          // persistent: 3 resident blocks per SM x 2 waves
    const bool band_active = cam.row0 > 0 || cam.row1 < cam.gy;
    // tile bands: candidate blocks (K0').  The list's counter is the word after the per-tile counts (zeroed with them).
    const bool use_cand = fused && band_active && N > 0 && buf->band_flags != nullptr && buf->band_cand != nullptr;
    const uint32_t* cand = use_cand ? buf->band_cand : nullptr;
    uint32_t* n_cand = buf->tile_counts + num_tiles;
    uint32_t* cmax_bits = (buf->flags & VTGS_BUF_DETERMINISTIC) ? buf->tile_counts + num_tiles + 1 : nullptr;
    const int persistent = 148 * 3;
    if (N > 0) {
        const bool narrow_band = (cam.row1 - cam.row0) * 5 < cam.gy * 2;
        if (use_cand)
            if (int e = launch_k("band_flags_kernel", Launch::pdl, band_flags_kernel, dim3((blocks + 3) / 4), dim3(256), 0, stream,
                                 cam, N, fe, means3D, scales, radii, buf->tiles_touched, buf->band_flags, buf->band_cand, n_cand)) return e;
        const int k1_grid = use_cand ? std::min(blocks, persistent) : k1_blocks;
        auto k1 = fused ? (narrow_band ? preprocess_kernel<true, true> : preprocess_kernel<true, false>) : preprocess_kernel<false, false>;
        if (int e = launch_k("preprocess_kernel", Launch::pdl, k1, dim3(k1_grid), dim3(256), 0, stream, cam, N, fe, means3D, scales, rotations,
                             opacities, colors, geom, radii, buf->tiles_touched, buf->tile_counts, cand, fused ? n_cand : nullptr, cmax_bits)) return e;
    }
    // only the band's tiles hold counts (tile-band sharding: K1' clips every rect to the band); the fused solvers never
    // look at another tile's range, so they scan the band alone -- API mode keeps (0,0) ranges for the other tiles
    const int band_tiles = (cam.row1 - cam.row0) * cam.gx;
    const int scan0 = fused ? cam.row0 * cam.gx : 0, scan_n = fused ? band_tiles : num_tiles;
    // the tile order is relative to the scanned range: usable when that is exactly what the sort / blend kernels cover
    // (worth its ~4 us in the scan only when a launch is about one wave of blocks: tile bands)
    uint32_t* order = (fused && band_active) ? buf->tile_order : nullptr;
    if (int e = launch_k("tile_scan_kernel", Launch::pdl, tile_scan_kernel, dim3(1), dim3(1024), 0, stream, buf->tile_counts + scan0,
                         buf->tile_ranges + 2 * (size_t)scan0, scan_n, buf->pair_capacity, buf->counters, order)) return e;
    if (N > 0 && band_tiles > 0) {
        const int sb = use_cand ? std::min(blocks, 148 * 8) : blocks;
        if (int e = launch_k("scatter_kernel", Launch::pdl, wide ? scatter_kernel<true> : scatter_kernel<false>, dim3(sb), dim3(256), 0, stream,
                             N, cam.gx, geom, buf->tiles_touched, buf->tile_ranges, buf->tile_counts, buf->pair_keys, cand, n_cand)) return e;
        static std::atomic<uint64_t> sort_attr{0};
        if (first_call_on_device(sort_attr)) {
            VTGS_CUDA_CHECK(cudaFuncSetAttribute(tile_sort_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SORT_SMEM_ELEMS * 8));
            VTGS_CUDA_CHECK(cudaFuncSetAttribute(tile_sort_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SORT_SMEM_ELEMS * 8));
        }
        if (int e = launch_k("tile_sort_kernel", Launch::pdl, wide ? tile_sort_kernel<true> : tile_sort_kernel<false>, dim3(band_tiles), dim3(256),
                             SORT_SMEM_ELEMS * 8, stream, cam, buf->tile_ranges, cam.row0 * cam.gx, buf->pair_keys, buf->point_list, geom,
                             reinterpret_cast<uint2*>(buf->region_pairs), buf->region_cnt, order)) return e;
    }
    if (N <= 0) VTGS_CUDA_CHECK(cudaMemsetAsync(buf->region_cnt, 0, sizeof(uint32_t) * 8 * num_tiles, stream));
    if (band_tiles > 0) {
        static std::atomic<uint64_t> fwd_attr{0};
        if (first_call_on_device(fwd_attr)) {        // 6 blocks x 33 KB of static shared memory per SM
            VTGS_CUDA_CHECK(cudaFuncSetAttribute(blend_forward_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
            VTGS_CUDA_CHECK(cudaFuncSetAttribute(blend_forward_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        }
        if (int e = launch_k("blend_forward_kernel", Launch::pdl, fused ? blend_forward_kernel<true> : blend_forward_kernel<false>,
                             dim3(band_tiles * (8 / FWD_WARPS)), dim3(32 * FWD_WARPS), 0, stream, cam, buf->tile_ranges,
                             reinterpret_cast<const uint2*>(buf->region_pairs), buf->region_cnt, buf->region_masks, buf->region_done, geom,
                             out_color, out_depth, buf->final_T, buf->n_contrib, order)) return e;
    }
    if (band_tiles < num_tiles && !fused) {       // API mode returns complete planes; the fused solvers only ever read their band
        const size_t P = (size_t)cam.W * cam.H;
        if (int e = launch_k("fill_outside_band_kernel", Launch::pdl, fill_outside_band_kernel, dim3((unsigned)((P + 255) / 256)), dim3(256), 0,
                             stream, cam, fused ? 6 : 3, out_color, out_depth, buf->final_T, buf->n_contrib)) return e;
    }
    return VTGS_OK;
}

// ---- parity / debug exports ---------------------------------------------------------------
__global__ void export_keys_kernel(const uint32_t* __restrict__ ranges, int num_tiles, const uint64_t* __restrict__ pair_keys,
                                   uint64_t* __restrict__ out, uint64_t cap) {
    const int tile = blockIdx.x;
    if (tile >= num_tiles) return;
    const uint32_t b = ranges[2 * tile], e = ranges[2 * tile + 1];
    for (uint32_t i = b + threadIdx.x; i < e; i += blockDim.x)
        if (i < cap) out[i] = ((uint64_t)tile << 32) | (pair_keys[i] >> 32);
}

__global__ void export_geom_kernel(int64_t N, const GeomRecord* __restrict__ geom, float* means2D, float* depths, float* conic_opacity) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const GeomRecord r = geom[i];
    if (means2D) { means2D[2 * i] = r.q0.x; means2D[2 * i + 1] = r.q0.y; }
    if (depths) depths[i] = r.q3.x;
    if (conic_opacity) { conic_opacity[4 * i] = r.q1.x; conic_opacity[4 * i + 1] = r.q1.y; conic_opacity[4 * i + 2] = r.q1.z; conic_opacity[4 * i + 3] = r.q1.w; }
}

__global__ void mark_visible_kernel(const __grid_constant__ CamConst cam, int64_t N, const float* __restrict__ means3D, uint8_t* __restrict__ present) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    present[i] = xform_row(cam.view, 2, means3D[3 * i], means3D[3 * i + 1], means3D[3 * i + 2]) > VTGS_NEAR_CULL ? 1 : 0;
}

}  // namespace vtgs

// =============================== C entry points (include/vtgs.h) ===========================
using namespace vtgs;

int vtgs_forward(const VtgsCamera* cam, int64_t N, const float* means3D, const float* scales,
                 const float* rotations, const float* opacities, const float* colors,
                 float* out_color, float* out_depth, int32_t* radii, VtgsBuffers* buf, void* stream) {
    if (int e = check_cam(cam)) return e;
    if (int e = check_buf(buf, N)) return e;
    VTGS_REQUIRE(N >= 0, "num_gaussians < 0");
    VTGS_REQUIRE(out_color && out_depth, "output pointer is NULL");
    if (N > 0) VTGS_REQUIRE(means3D && scales && rotations && opacities && colors && radii, "input pointer is NULL");
    FrontEnd fe{};
    return launch_forward(cam, N, false, fe, means3D, scales, rotations, opacities, colors, out_color, out_depth, radii, buf,
                          (cudaStream_t)stream);
}

int vtgs_fused_forward(const VtgsCamera* cam, const VtgsParams* p, const VtgsPose* pose, float* out_image6, int32_t* radii,
                       VtgsBuffers* buf, void* stream) {
    if (int e = check_fused(cam, p, pose, buf)) return e;
    VTGS_REQUIRE(out_image6 != nullptr, "out_image6 is NULL");
    if (p->num_gaussians > 0) VTGS_REQUIRE(radii != nullptr, "radii is NULL");
    FrontEnd fe{};
    fe.cam_unnorm_rot = pose->cam_unnorm_rot;
    fe.cam_trans = pose->cam_trans;
    fe.counters = buf->counters;
    if (p->num_gaussians <= 0)          // nothing to preprocess: still publish the pose for the backward
        if (int e = launch_pose_matrix(pose, buf->counters, (cudaStream_t)stream)) return e;
    for (int k = 0; k < 4; ++k) fe.depth_row[k] = pose->depth_row[k];
    fe.log_scales_dim = p->log_scales_dim;
    return launch_forward(cam, p->num_gaussians, true, fe, p->means3D, p->log_scales, p->unnorm_rotations, p->logit_opacities,
                          p->rgb_colors, out_image6, nullptr, radii, buf, (cudaStream_t)stream);
}

int vtgs_export_sorted_keys(const VtgsCamera* camera, int64_t N, const VtgsBuffers* buf, uint64_t* keys_out,
                            uint64_t keys_capacity, void* stream) {
    (void)N;
    if (int e = check_cam(camera)) return e;
    VTGS_REQUIRE(buf && keys_out, "pointer is NULL");
    const CamConst cam = make_cam_const(*camera);
    const int num_tiles = cam.gx * cam.gy;
    return launch_k("export_keys_kernel", Launch::plain, export_keys_kernel, dim3(num_tiles), dim3(128), 0, (cudaStream_t)stream,
                    buf->tile_ranges, num_tiles, buf->pair_keys, keys_out, keys_capacity);
}

int vtgs_export_geometry(int64_t N, const VtgsBuffers* buf, float* means2D, float* depths, float* conic_opacity, void* stream) {
    VTGS_REQUIRE(buf != nullptr, "buffers is NULL");
    if (N <= 0) return VTGS_OK;
    return launch_k("export_geom_kernel", Launch::plain, export_geom_kernel, dim3((unsigned)((N + 255) / 256)), dim3(256), 0,
                    (cudaStream_t)stream, N, reinterpret_cast<const GeomRecord*>(buf->geom), means2D, depths, conic_opacity);
}

int vtgs_mark_visible(const VtgsCamera* camera, int64_t N, const float* means3D, uint8_t* present, void* stream) {
    if (int e = check_cam(camera)) return e;
    if (N > 0) VTGS_REQUIRE(means3D && present, "pointer is NULL");
    if (N <= 0) return VTGS_OK;
    const CamConst cam = make_cam_const(*camera);
    return launch_k("mark_visible_kernel", Launch::plain, mark_visible_kernel, dim3((unsigned)((N + 255) / 256)), dim3(256), 0,
                    (cudaStream_t)stream, cam, N, means3D, present);
}
