// caller.cu -- kernels of the rows either side of the hot path (SURVEY.md 8(f) N3 / N4): the per-frame evaluation
// metrics of the reference's `eval` (utils/eval_helpers.py:431-477) on the fused six-plane render, and a device
// point-to-plane metric replacing the Open3D / kornia CPU round trip of `compute_point2plane_dist`
// (src/vtgaussian_slam.py:1070-1155) that the reference runs inside its tracking loop (:1929, :1956).
#include "common.cuh"
#include "kernels.h"

namespace vtgs {

// =============================== evaluation metrics ==========================================
// One pass over the frame: per-channel squared error of the weighted images, masked depth L1, valid count; the last
// block reduces the per-block partials in a fixed order (fp64) and derives PSNR / depth L1.
constexpr int EVAL_BLOCKS = 592;          // 4 blocks per SM
constexpr int EVAL_TERMS = 8;             // 5 used

__global__ void __launch_bounds__(256)
eval_metrics_kernel(size_t P, const float* __restrict__ image6, const float* __restrict__ gt_rgb, const float* __restrict__ gt_depth,
                    float sil_thres, int use_presence, float* __restrict__ partials, unsigned int* __restrict__ ticket,
                    float* __restrict__ out8) {
    __shared__ float s_part[8][EVAL_TERMS];
    __shared__ double s_sum[EVAL_TERMS][32];
    __shared__ bool s_last;
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (size_t pid = (size_t)blockIdx.x * 256 + threadIdx.x; pid < P; pid += (size_t)gridDim.x * 256) {
        const float gd = __ldg(gt_depth + pid);
        const bool valid = gd > 0.0f;
        const bool presence = __ldcs(image6 + 4 * P + pid) > sil_thres;
        const float w = (valid && (!use_presence || presence)) ? 1.0f : 0.0f;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            // weighted_im - weighted_gt_im = (im - gt) * w, w in {0, 1}
            const float e = (__ldcs(image6 + c * P + pid) - __ldg(gt_rgb + c * P + pid)) * w;
            acc[c] = fmaf(e, e, acc[c]);
        }
        if (valid) {
            // rastered_depth * valid - gt, times the presence mask in the tracking-only configuration
            float e = fabsf(__ldcs(image6 + 3 * P + pid) - gd);
            if (use_presence && !presence) e = 0.0f;
            acc[3] += e;
            acc[4] += 1.0f;
        }
    }
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int k = 0; k < 5; ++k) acc[k] = warp_sum(acc[k]);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < EVAL_TERMS; ++k) s_part[warp][k] = k < 5 ? acc[k] : 0.0f;
    }
    __syncthreads();
    if (tid < EVAL_TERMS) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += s_part[w][tid];
        partials[(size_t)blockIdx.x * EVAL_TERMS + tid] = s;
        __threadfence();
    }
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int term = tid & (EVAL_TERMS - 1), sl = tid >> 3;            // 32 slices of blocks
    double a = 0.0;
    for (int b = sl; b < (int)gridDim.x; b += 32) a += (double)__ldcg(&partials[(size_t)b * EVAL_TERMS + term]);
    s_sum[term][sl] = a;
    __syncthreads();
    if (tid == 0) {
        double tot[5];
        for (int k = 0; k < 5; ++k) {
            double t = 0.0;
            for (int i = 0; i < 32; ++i) t += s_sum[k][i];
            tot[k] = t;
        }
        double psnr = 0.0;
        for (int c = 0; c < 3; ++c) {
            out8[c] = (float)tot[c];
            psnr += 20.0 * log10(1.0 / sqrt(tot[c] / (double)P));      // calc_psnr (utils/slam_external.py), then .mean()
        }
        out8[3] = (float)tot[3];
        out8[4] = (float)tot[4];
        out8[5] = (float)(psnr / 3.0);
        out8[6] = (float)(tot[3] / tot[4]);                            // depth L1
        out8[7] = out8[6];                                             // the reference's "rmse": sqrt(x^2) = |x|, same sum
        *ticket = 0u;
    }
}

// =============================== point-to-plane metric =======================================
struct P2PFrame {
    int W, H;
    float fx, fy, cx, cy;
    float c2w[12];          // rows of the 3x4 camera-to-world matrix of THIS frame
    float other_w2c[12];    // rows of the 3x4 world-to-camera matrix of the OTHER frame (frustum test)
    int frustum;
};

// Per pixel of one frame: world point (the reference's get_pointcloud with factor 1: pixel centres at +0.5), optional
// world normal (kornia.geometry.depth_to_normals: Sobel gradients /8 with replicated borders of the points unprojected
// at integer pixel coordinates, cross product, normalised; then rotated by c2w as trans_normal_c2w does) and validity
// (depth > 0, optional mask, inside the other view's image with positive depth -- get_frustum_mask).
__global__ void __launch_bounds__(256)
p2p_prepare_kernel(const __grid_constant__ P2PFrame f, const float* __restrict__ depth, const uint8_t* __restrict__ mask,
                   float* __restrict__ pts, float* __restrict__ nrm, uint8_t* __restrict__ valid) {
    const int pid = blockIdx.x * 256 + threadIdx.x;
    if (pid >= f.W * f.H) return;
    const int u = pid % f.W, v = pid / f.W;
    const float z = depth[pid];
    const float xc = ((float)u - f.cx + 0.5f) / f.fx * z, yc = ((float)v - f.cy + 0.5f) / f.fy * z;
    const float* M = f.c2w;
    const float X = M[0] * xc + M[1] * yc + M[2] * z + M[3];
    const float Y = M[4] * xc + M[5] * yc + M[6] * z + M[7];
    const float Z = M[8] * xc + M[9] * yc + M[10] * z + M[11];
    pts[3 * pid] = X; pts[3 * pid + 1] = Y; pts[3 * pid + 2] = Z;
    bool ok = z > 0.0f && (!mask || mask[pid] != 0);
    if (f.frustum) {
        const float* O = f.other_w2c;
        const float a = O[0] * X + O[1] * Y + O[2] * Z + O[3];
        const float b = O[4] * X + O[5] * Y + O[6] * Z + O[7];
        const float c = O[8] * X + O[9] * Y + O[10] * Z + O[11];
        const float zz = c + 1e-8f;
        const float uu = (f.fx * a + f.cx * c) / zz, vv = (f.fy * b + f.cy * c) / zz;
        ok = ok && uu < (float)f.W && uu > 0.0f && vv < (float)f.H && vv > 0.0f && zz > 0.0f;
    }
    valid[pid] = ok ? 1 : 0;
    if (!nrm) return;
    float gx[3] = {0.f, 0.f, 0.f}, gy[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int dv = -1; dv <= 1; ++dv) {
#pragma unroll
        for (int du = -1; du <= 1; ++du) {
            const int uu = min(max(u + du, 0), f.W - 1), vv = min(max(v + dv, 0), f.H - 1);
            const float zn = depth[vv * f.W + uu];
            const float p[3] = {((float)uu - f.cx) / f.fx * zn, ((float)vv - f.cy) / f.fy * zn, zn};
            const float wx = (float)(du * (dv == 0 ? 2 : 1)) * 0.125f;      // Sobel x: [-1 0 1; -2 0 2; -1 0 1] / 8
            const float wy = (float)(dv * (du == 0 ? 2 : 1)) * 0.125f;      // Sobel y: its transpose
#pragma unroll
            for (int k = 0; k < 3; ++k) { gx[k] = fmaf(wx, p[k], gx[k]); gy[k] = fmaf(wy, p[k], gy[k]); }
        }
    }
    float n[3] = {gx[1] * gy[2] - gx[2] * gy[1], gx[2] * gy[0] - gx[0] * gy[2], gx[0] * gy[1] - gx[1] * gy[0]};
    const float inv = 1.0f / fmaxf(sqrtf(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]), 1e-12f);     // F.normalize eps
    n[0] *= inv; n[1] *= inv; n[2] *= inv;
    nrm[3 * pid] = M[0] * n[0] + M[1] * n[1] + M[2] * n[2];
    nrm[3 * pid + 1] = M[4] * n[0] + M[5] * n[1] + M[6] * n[2];
    nrm[3 * pid + 2] = M[8] * n[0] + M[9] * n[1] + M[10] * n[2];
}

__device__ __forceinline__ uint32_t cell_hash(int cx, int cy, int cz, uint32_t mask) {
    return ((uint32_t)cx * 73856093u ^ (uint32_t)cy * 19349663u ^ (uint32_t)cz * 83492791u) & mask;
}

// Uniform hash grid over the target cloud, cell edge = the search radius: every bucket heads a linked list of the points
// whose cell hashes to it (cells that collide share a list; the query tests real distances, so that only costs work).
__global__ void __launch_bounds__(256)
p2p_insert_kernel(int64_t n, const float* __restrict__ pts, const uint8_t* __restrict__ valid, float inv_cell,
                  int32_t* __restrict__ head, uint32_t mask, int32_t* __restrict__ next) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n || !valid[i]) return;
    const int cx = (int)floorf(pts[3 * i] * inv_cell), cy = (int)floorf(pts[3 * i + 1] * inv_cell), cz = (int)floorf(pts[3 * i + 2] * inv_cell);
    next[i] = atomicExch(&head[cell_hash(cx, cy, cz, mask)], (int32_t)i);
}

// Nearest target point within max_dist of every valid source point (Open3D evaluate_registration: a hybrid
// radius / 1-NN KD-tree query per source point); ties go to the lower target index, so the result does not depend on
// the insertion order.  out_dist[j] = n_target . (p_source - p_target), NaN without a correspondence.
__global__ void __launch_bounds__(128)
p2p_query_kernel(int64_t n_src, const float* __restrict__ src, const uint8_t* __restrict__ src_valid,
                 const float* __restrict__ tgt, const float* __restrict__ tgt_nrm, float inv_cell, float max_d2,
                 const int32_t* __restrict__ head, uint32_t mask, const int32_t* __restrict__ next,
                 float* __restrict__ out_dist, int32_t* __restrict__ out_idx) {
    const int64_t j = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (j >= n_src) return;
    float res = __int_as_float(0x7fc00000);
    int32_t best_i = -1;
    if (src_valid[j]) {
        const float x = src[3 * j], y = src[3 * j + 1], z = src[3 * j + 2];
        const int cx = (int)floorf(x * inv_cell), cy = (int)floorf(y * inv_cell), cz = (int)floorf(z * inv_cell);
        float best = max_d2;
        uint32_t seen[27];
        int ns = 0;
        for (int dz = -1; dz <= 1; ++dz)
            for (int dy = -1; dy <= 1; ++dy)
                for (int dx = -1; dx <= 1; ++dx) {
                    const uint32_t h = cell_hash(cx + dx, cy + dy, cz + dz, mask);
                    bool dup = false;
                    for (int k = 0; k < ns; ++k) dup = dup || seen[k] == h;
                    if (dup) continue;                        // two of the 27 cells share a bucket: walk its list once
                    seen[ns++] = h;
                    for (int32_t i = head[h]; i >= 0; i = next[i]) {
                        const float ex = x - tgt[3 * i], ey = y - tgt[3 * i + 1], ez = z - tgt[3 * i + 2];
                        const float d2 = ex * ex + ey * ey + ez * ez;
                        if (d2 < best || (d2 == best && best_i >= 0 && i < best_i) || (d2 == best && best_i < 0)) { best = d2; best_i = i; }
                    }
                }
        if (best_i >= 0) {
            const int32_t i = best_i;
            res = tgt_nrm[3 * i] * (x - tgt[3 * i]) + tgt_nrm[3 * i + 1] * (y - tgt[3 * i + 1]) + tgt_nrm[3 * i + 2] * (z - tgt[3 * i + 2]);
        }
    }
    out_dist[j] = res;
    if (out_idx) out_idx[j] = best_i;
}

// =============================== frame conversion on the device ==============================
// What the reference's dataset does to a decoded frame on the CPU before every use (datasets/gradslam_datasets/
// basedataset.py:215-272 + src/vtgaussian_slam.py:198-202): colour uint8 HWC -> float64 -> cv2.resize(INTER_LINEAR) ->
// float32 CHW / 255; depth uint16 -> float64 -> cv2.resize(INTER_NEAREST) -> / png_depth_scale -> float32.  Done here
// from the RAW decoded bytes, so a frame crosses PCIe as 3 + 2 bytes per pixel instead of 16, and the arithmetic follows
// OpenCV's generic path for CV_64F (double coefficients and accumulation, horizontal pass first: checked against
// cv2 4.13 to 1e-13 before the float32 cast) so the planes agree with the CPU loader's to the last bit of the float32 result.
struct ResizeGeom { int sw, sh, dw, dh; double scale_x, scale_y; };

__device__ __forceinline__ void linear_tap(int d, double scale, int ssize, int& s0, double& f, bool& edge) {
    f = ((double)d + 0.5) * scale - 0.5;
    s0 = (int)floor(f);
    f -= (double)s0;
    edge = false;
    if (s0 < 0) { f = 0.0; s0 = 0; }
    if (s0 + 1 >= ssize) { edge = true; if (s0 >= ssize - 1) { f = 0.0; s0 = ssize - 1; } }
}

__global__ void __launch_bounds__(256)
frame_convert_kernel(const __grid_constant__ ResizeGeom g, const uint8_t* __restrict__ rgb, const uint16_t* __restrict__ depth,
                     double depth_scale, float* __restrict__ im, float* __restrict__ depth_out) {
    const int pid = blockIdx.x * 256 + threadIdx.x;
    if (pid >= g.dw * g.dh) return;
    const int x = pid % g.dw, y = pid / g.dw;
    if (rgb) {
        int sx; double fx; bool xedge;
        linear_tap(x, g.scale_x, g.sw, sx, fx, xedge);
        // vertical taps: rows sy, sy + 1 clipped, weights (1 - fy, fy) kept as they are (cv::resizeGeneric_Invoker)
        double fy = ((double)y + 0.5) * g.scale_y - 0.5;
        const int sy = (int)floor(fy);
        fy -= (double)sy;
        const int r0 = min(max(sy, 0), g.sh - 1), r1 = min(max(sy + 1, 0), g.sh - 1);
        const double a0 = 1.0 - fx, a1 = fx, b0 = 1.0 - fy, b1 = fy;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            double h[2];
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const uint8_t* row = rgb + ((size_t)(k ? r1 : r0) * g.sw) * 3;
                const double s0 = (double)row[sx * 3 + c];
                // past xmax OpenCV copies the source sample (x 1); before it, both taps
                h[k] = xedge ? s0 : __dadd_rn(__dmul_rn(s0, a0), __dmul_rn((double)row[(sx + 1) * 3 + c], a1));
            }
            const double v = __dadd_rn(__dmul_rn(h[0], b0), __dmul_rn(h[1], b1));
            im[(size_t)c * g.dw * g.dh + pid] = __fdiv_rn((float)v, 255.0f);
        }
    }
    if (depth) {
        const int sx = min((int)floor((double)x * g.scale_x), g.sw - 1), sy = min((int)floor((double)y * g.scale_y), g.sh - 1);
        depth_out[pid] = (float)((double)depth[(size_t)sy * g.sw + sx] / depth_scale);
    }
}

// ---- radius bookkeeping of get_loss (reference src/vtgaussian_slam.py:681-683) ---------------------------------------
__global__ void __launch_bounds__(256)
book_radii_kernel(int64_t n, const int32_t* __restrict__ radii, float* __restrict__ max_radius, uint8_t* __restrict__ seen) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const int32_t r = radii[i];
    seen[i] = r > 0 ? 1 : 0;
    const float m = max_radius[i], rf = (float)r;
    if (rf > m) max_radius[i] = rf;
}

}  // namespace vtgs

// =============================== C entry points (include/vtgs.h) ===========================
using namespace vtgs;

uint64_t vtgs_eval_scratch_floats(void) { return (uint64_t)EVAL_BLOCKS * EVAL_TERMS + 4; }

int vtgs_eval_metrics(const VtgsCamera* cam, const float* image6, const float* gt_rgb, const float* gt_depth, float sil_thres,
                      int32_t use_presence, float* out8, float* scratch, void* stream_) {
    if (int e = check_cam(cam)) return e;
    VTGS_REQUIRE(image6 && gt_rgb && gt_depth && out8 && scratch, "pointer is NULL");
    const cudaStream_t stream = (cudaStream_t)stream_;
    const size_t P = (size_t)cam->image_width * cam->image_height;
    unsigned int* ticket = reinterpret_cast<unsigned int*>(scratch + (size_t)EVAL_BLOCKS * EVAL_TERMS);
    VTGS_CUDA_CHECK(cudaMemsetAsync(ticket, 0, sizeof(unsigned int), stream));
    return launch_k("eval_metrics_kernel", Launch::plain, eval_metrics_kernel, dim3(EVAL_BLOCKS), dim3(256), 0, stream, P, image6, gt_rgb, gt_depth,
                    sil_thres, use_presence, scratch, ticket, out8);
}

int vtgs_p2p_prepare(int32_t W, int32_t H, const float* intr4, const float* c2w12, const float* other_w2c12, const float* depth,
                     const uint8_t* mask, float* pts, float* nrm, uint8_t* valid, void* stream) {
    VTGS_REQUIRE(W > 0 && H > 0 && (int64_t)W * H < (int64_t)1 << 31, "bad image size");
    VTGS_REQUIRE(intr4 && c2w12 && depth && pts && valid, "pointer is NULL");
    P2PFrame f{};
    f.W = W; f.H = H;
    f.fx = intr4[0]; f.fy = intr4[1]; f.cx = intr4[2]; f.cy = intr4[3];
    for (int k = 0; k < 12; ++k) { f.c2w[k] = c2w12[k]; f.other_w2c[k] = other_w2c12 ? other_w2c12[k] : 0.0f; }
    f.frustum = other_w2c12 != nullptr;
    const int P = W * H;
    return launch_k("p2p_prepare_kernel", Launch::plain, p2p_prepare_kernel, dim3((P + 255) / 256), dim3(256), 0, (cudaStream_t)stream, f, depth,
                    mask, pts, nrm, valid);
}

int vtgs_p2p_match(int64_t n_tgt, const float* tgt_pts, const float* tgt_nrm, const uint8_t* tgt_valid, int64_t n_src,
                   const float* src_pts, const uint8_t* src_valid, float max_dist, int32_t* table, int64_t table_size,
                   int32_t* next, float* out_dist, int32_t* out_idx, void* stream_) {
    VTGS_REQUIRE(n_tgt >= 0 && n_src >= 0 && n_tgt < (int64_t)1 << 31, "bad point count");
    VTGS_REQUIRE(max_dist > 0.0f, "max_dist must be positive");
    VTGS_REQUIRE(table && table_size > 0 && (table_size & (table_size - 1)) == 0 && table_size <= (int64_t)1 << 31, "table_size must be a power of two");
    if (n_tgt > 0) VTGS_REQUIRE(tgt_pts && tgt_nrm && tgt_valid && next, "pointer is NULL");
    if (n_src > 0) VTGS_REQUIRE(src_pts && src_valid && out_dist, "pointer is NULL");
    const cudaStream_t stream = (cudaStream_t)stream_;
    VTGS_CUDA_CHECK(cudaMemsetAsync(table, 0xFF, sizeof(int32_t) * (size_t)table_size, stream));
    const float inv_cell = 1.0f / max_dist;
    const uint32_t mask = (uint32_t)(table_size - 1);
    if (n_tgt > 0)
        if (int e = launch_k("p2p_insert_kernel", Launch::plain, p2p_insert_kernel, dim3((unsigned)((n_tgt + 255) / 256)), dim3(256), 0, stream,
                             n_tgt, tgt_pts, tgt_valid, inv_cell, table, mask, next)) return e;
    if (n_src > 0)
        return launch_k("p2p_query_kernel", Launch::plain, p2p_query_kernel, dim3((unsigned)((n_src + 127) / 128)), dim3(128), 0, stream, n_src,
                        src_pts, src_valid, tgt_pts, tgt_nrm, inv_cell, max_dist * max_dist, table, mask, next, out_dist, out_idx);
    return VTGS_OK;
}

int vtgs_frame_convert(int32_t src_w, int32_t src_h, int32_t dst_w, int32_t dst_h, const uint8_t* rgb_hwc, const uint16_t* depth_u16,
                       double png_depth_scale, float* im_chw, float* depth_out, void* stream) {
    VTGS_REQUIRE(src_w > 0 && src_h > 0 && dst_w > 0 && dst_h > 0, "bad image size");
    VTGS_REQUIRE((rgb_hwc == nullptr) == (im_chw == nullptr) && (depth_u16 == nullptr) == (depth_out == nullptr), "input / output pointers must come in pairs");
    VTGS_REQUIRE(depth_u16 == nullptr || png_depth_scale > 0.0, "png_depth_scale must be positive");
    ResizeGeom g{src_w, src_h, dst_w, dst_h, 1.0 / ((double)dst_w / (double)src_w), 1.0 / ((double)dst_h / (double)src_h)};   // cv::resize: 1 / inv_scale
    return launch_k("frame_convert_kernel", Launch::plain, frame_convert_kernel, dim3((dst_w * dst_h + 255) / 256), dim3(256), 0, (cudaStream_t)stream,
                    g, rgb_hwc, depth_u16, png_depth_scale, im_chw, depth_out);
}

int vtgs_book_radii(int64_t n, const int32_t* radii, float* max_2D_radius, uint8_t* seen, void* stream) {
    VTGS_REQUIRE(n >= 0, "n < 0");
    if (n > 0) VTGS_REQUIRE(radii && max_2D_radius && seen, "pointer is NULL");
    if (n <= 0) return VTGS_OK;
    return launch_k("book_radii_kernel", Launch::plain, book_radii_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, n,
                    radii, max_2D_radius, seen);
}
