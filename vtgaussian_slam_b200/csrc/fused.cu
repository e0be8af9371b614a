// fused.cu -- the per-iteration work the reference does in PyTorch around the rasteriser:
// the tracking / mapping loss of get_loss (reference src/vtgaussian_slam.py:513-612,678-679)
// with its gradient w.r.t. the rendered planes, and the Adam update
// (torch.optim.Adam as configured at src/vtgaussian_slam.py:180-187).
#include <algorithm>
#include <cstdlib>
#include "common.cuh"
#include "kernels.h"

namespace vtgs {

constexpr int LOSS_PX_PER_THREAD = 4;  // 1024 pixels per block: 4x fewer partials for the in-kernel final reduction
constexpr int LOSS_TERMS = 4;      // per-block partials: depth L1, rgb L1, mask count, spare

__device__ __forceinline__ float sgn(float v) { return v > 0.0f ? 1.0f : (v < 0.0f ? -1.0f : 0.0f); }

// ---- exact median of depth_error = |gt - d| * (gt > 0) over the frame (reference :525-527, torch.median = the
// LOWER median, element (P - 1) / 2 of the sorted values) by radix select: four passes, each a 256-bin histogram of
// the next byte of the float bits (non-negative floats order like their bit patterns; NaN sorts last and, as in
// torch, makes the median NaN) among the values matching the prefix selected so far, then one block picks the bin
// holding the target rank.  The histogram pass covers the camera's tile-row band, so a sharded frame all-reduces the
// first VTGS_MEDIAN_SUMMABLE_WORDS words between the two kernels.
// state: hist[0..255], nan_count[256] | prefix[257], rank[258], result bits[259].
constexpr int MEDIAN_STATE_WORDS = VTGS_MEDIAN_STATE_WORDS;
__global__ void __launch_bounds__(256)
median_hist_kernel(const float* __restrict__ depth_plane, const float* __restrict__ gt_depth, size_t pix_begin, size_t pix_end,
                   int pass, unsigned int* __restrict__ st) {
    VTGS_PDL_PROLOGUE();
    __shared__ unsigned int sh[256];
    const int tid = threadIdx.x;
    sh[tid] = 0u;
    __syncthreads();
    const unsigned int prefix = st[257];
    unsigned int nan_local = 0u;
    for (size_t i = pix_begin + (size_t)blockIdx.x * 256 + tid; i < pix_end; i += (size_t)gridDim.x * 256) {
        const float gd = gt_depth[i], d = depth_plane[i];
        const float e = fabsf(gd - d) * (gd > 0.0f ? 1.0f : 0.0f);
        unsigned int key = __float_as_uint(e);
        if (e != e) { key = 0xffffffffu; if (pass == 0) ++nan_local; }
        if (pass == 0 || (key >> (32 - 8 * pass)) == prefix) atomicAdd(&sh[(key >> (24 - 8 * pass)) & 0xffu], 1u);
    }
    __syncthreads();
    if (sh[tid]) atomicAdd(st + tid, sh[tid]);
    if (nan_local) atomicAdd(st + 256, nan_local);
}

__global__ void __launch_bounds__(256)
median_pick_kernel(unsigned long long P_total, int pass, unsigned int* __restrict__ st) {
    VTGS_PDL_PROLOGUE();
    __shared__ unsigned int sh[256];
    const int tid = threadIdx.x;
    sh[tid] = st[tid];
    st[tid] = 0u;                                        // clean histogram for the next pass / call
    __syncthreads();
    if (tid == 0) {
        const unsigned int prefix = st[257];
        unsigned int rank = pass == 0 ? (unsigned int)((P_total - 1) / 2) : st[258];
        unsigned int cum = 0u;
        int b = 0;
        for (; b < 255; ++b) {
            if (rank < cum + sh[b]) break;
            cum += sh[b];
        }
        const unsigned int np = (prefix << 8) | (unsigned int)b;
        st[257] = pass == 3 ? 0u : np;
        st[258] = rank - cum;
        if (pass == 3) {
            st[259] = st[256] > 0u ? 0x7fc00000u : np;
            st[256] = 0u;
        }
    }
}

static int launch_median_hist(const VtgsCamera* camera, const float* depth_plane, const float* gt_depth, int pass, uint32_t* state,
                              cudaStream_t stream) {
    const CamConst cam = make_cam_const(*camera);
    size_t b, e;
    band_pixel_range(cam, b, e);
    if (e <= b) return VTGS_OK;
    const int mb = (int)std::min<size_t>((e - b + 1023) / 1024, 148 * 4);
    return launch_k("median_hist_kernel", Launch::pdl, median_hist_kernel, dim3(mb), dim3(256), 0, stream, depth_plane, gt_depth, b, e, pass, state);
}

static int launch_median_pick(int64_t P_total, int pass, uint32_t* state, cudaStream_t stream) {
    return launch_k("median_pick_kernel", Launch::pdl, median_pick_kernel, dim3(1), dim3(256), 0, stream, (unsigned long long)P_total, pass, state);
}

// ---- Replica iteration-0 silhouette-threshold search (reference src/vtgaussian_slam.py:472-510) --------------------
// The five masks are nested (0.990 < 0.993 < ... < 0.999), so a pixel is binned by the number of thresholds its
// silhouette exceeds and the per-threshold sums are suffix sums of the bins.
constexpr int LADDER_N = 5;
__device__ __constant__ float c_sil_ladder[LADDER_N] = {0.990f, 0.993f, 0.995f, 0.997f, 0.999f};
__global__ void __launch_bounds__(256)
sil_ladder_kernel(const __grid_constant__ CamConst cam, const float* __restrict__ image6, const float* __restrict__ gt_rgb,
                  const float* __restrict__ gt_depth, float* __restrict__ partials, unsigned int* __restrict__ ticket,
                  float* __restrict__ sums10) {
    __shared__ LastBlockSum<2 * LADDER_N> red;
    const size_t P = (size_t)cam.W * cam.H;
    size_t row_begin, row_end;
    band_pixel_range(cam, row_begin, row_end);
    float sq[LADDER_N], cnt[LADDER_N];
#pragma unroll
    for (int k = 0; k < LADDER_N; ++k) { sq[k] = 0.f; cnt[k] = 0.f; }
    for (int rep = 0; rep < 4; ++rep) {
        const size_t pid = row_begin + ((size_t)blockIdx.x * 4 + rep) * 256 + threadIdx.x;
        if (pid >= row_end) break;
        const float sil = image6[4 * P + pid];
        if (!(gt_depth[pid] > 0.0f)) continue;
        const float er = gt_rgb[pid] - image6[pid], eg = gt_rgb[P + pid] - image6[P + pid], eb = gt_rgb[2 * P + pid] - image6[2 * P + pid];
        const float e2 = er * er + eg * eg + eb * eb;
#pragma unroll
        for (int k = 0; k < LADDER_N; ++k)
            if (sil > c_sil_ladder[k]) { sq[k] += e2; cnt[k] += 1.0f; }
    }
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int k = 0; k < LADDER_N; ++k) { sq[k] = warp_sum(sq[k]); cnt[k] = warp_sum(cnt[k]); }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < LADDER_N; ++k) { red.part[warp][k] = sq[k]; red.part[warp][LADDER_N + k] = cnt[k]; }
    }
    if (!red.reduce(partials, ticket)) return;
    if (tid < 2 * LADDER_N) sums10[tid] = (float)red.total(tid);
}

__global__ void sil_select_kernel(const float* __restrict__ sums10, float* __restrict__ thr_out, float* __restrict__ mse_out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int best = 0;
    float best_mse = 0.0f;
    bool have = false;
    for (int k = 0; k < LADDER_N; ++k) {
        const float c = sums10[LADDER_N + k];
        if (!(c > 0.0f)) continue;                       // torch.mean of an empty selection is nan: never the minimum
        const float mse = sums10[k] / (3.0f * c);
        if (!have || mse < best_mse) { best = k; best_mse = mse; have = true; }
    }
    *thr_out = c_sil_ladder[best];
    if (mse_out) *mse_out = have ? best_mse : __uint_as_float(0x7fc00000u);
}

// ---- non-presence mask of the silhouette-driven Gaussian addition (reference src/vtgaussian_slam.py:747-760) ----
__global__ void __launch_bounds__(256)
nonpresence_mask_kernel(size_t P, const float* __restrict__ image6, const float* __restrict__ gt_depth, float sil_thres,
                        const unsigned int* __restrict__ median_state, uint8_t* __restrict__ mask_out, unsigned int* __restrict__ count) {
    const size_t pid = (size_t)blockIdx.x * 256 + threadIdx.x;
    const float thr = 50.0f * __uint_as_float(median_state[259]);
    bool m = false;
    if (pid < P) {
        const float d = image6[3 * P + pid], sil = image6[4 * P + pid], gd = gt_depth[pid];
        const float err = fabsf(gd - d) * (gd > 0.0f ? 1.0f : 0.0f);
        m = (sil < sil_thres) || ((d > gd) && (err > thr));
        mask_out[pid] = m ? 1 : 0;
    }
    if (count) {
        const unsigned int b = __ballot_sync(VTGS_FULL_MASK, m);
        if ((threadIdx.x & 31) == 0 && b) atomicAdd(count, (unsigned int)__popc(b));
    }
}

// ---- FP32 FMA throughput probe ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
ffma_probe_kernel(long long iters, float* __restrict__ sink) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float m = 0.999f, c = 1e-4f;
#pragma unroll 16
    for (long long i = 0; i < iters; ++i) {
        a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
        a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
    }
    const float r = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (r == 123456.789f) *sink = r;                     // never true: keeps the loop alive
}

// Tracking loss (mode 0): sums of masked absolute differences; dL/dplane = w * sign * mask.
__global__ void __launch_bounds__(256)
tracking_loss_kernel(const __grid_constant__ CamConst cam, VtgsLossConfig cfg, const float* __restrict__ image6,
                     const float* __restrict__ gt_rgb, const float* __restrict__ gt_depth,
                     float* __restrict__ dL_dimage4, float* __restrict__ partials, unsigned int* __restrict__ ticket,
                     float* __restrict__ loss_terms, const unsigned int* __restrict__ median_state) {
    VTGS_PDL_PROLOGUE();
    __shared__ LastBlockSum<LOSS_TERMS> red;
    const size_t P = (size_t)cam.W * cam.H;
    size_t row_begin, row_end;
    band_pixel_range(cam, row_begin, row_end);
    // outlier mask: depth_error < 50 * median(depth_error) (NaN median: nothing passes)
    const float outlier_thr = median_state ? 50.0f * __uint_as_float(__ldcg(median_state + 259)) : 0.0f;
    const float sil_thres = cfg.sil_thres_dev ? __ldcg(cfg.sil_thres_dev) : cfg.sil_thres;
    float ld = 0.f, li = 0.f, cnt = 0.f;
    // all of a thread's loads are issued before the first dependent use (10 planes x LOSS_PX_PER_THREAD pixels in flight)
    float in[LOSS_PX_PER_THREAD][10];
    const size_t pid0 = row_begin + (size_t)blockIdx.x * LOSS_PX_PER_THREAD * 256 + threadIdx.x;
#pragma unroll
    for (int rep = 0; rep < LOSS_PX_PER_THREAD; ++rep) {
        const size_t pid = pid0 + (size_t)rep * 256;
        if (pid < row_end) {
#pragma unroll
            for (int k = 0; k < 6; ++k) in[rep][k] = __ldcs(image6 + (size_t)k * P + pid);
#pragma unroll
            for (int k = 0; k < 3; ++k) in[rep][6 + k] = __ldg(gt_rgb + (size_t)k * P + pid);
            in[rep][9] = __ldg(gt_depth + pid);
        }
    }
#pragma unroll
    for (int rep = 0; rep < LOSS_PX_PER_THREAD; ++rep) {
        const size_t pid = pid0 + (size_t)rep * 256;
        if (pid >= row_end) break;
        const float r = in[rep][0], g = in[rep][1], b = in[rep][2];
        const float d = in[rep][3], sil = in[rep][4], dsq = in[rep][5];
        const float gd = in[rep][9];
        const float unc = dsq - d * d;
        bool mask = gd > 0.0f && !(d != d) && !(unc != unc);
        if (cfg.use_sil_for_loss) mask = mask && sil > sil_thres;
        if (cfg.far_depth_thres > 0.0f) mask = mask && gd < cfg.far_depth_thres;
        if (median_state) mask = mask && (fabsf(gd - d) * (gd > 0.0f ? 1.0f : 0.0f) < outlier_thr);
        if (cfg.pixel_mask) mask = mask && cfg.pixel_mask[pid] != 0;
        // reference :600-605: the colour term is masked only with use_sil_for_loss / outlier masks
        const bool mask_im = (cfg.use_sil_for_loss || cfg.ignore_outlier_depth) ? mask : true;
        const float er = r - in[rep][6], eg = g - in[rep][7], eb = b - in[rep][8];
        const float ed = d - gd;
        if (mask) { ld += fabsf(ed); cnt += 1.0f; }
        if (mask_im) li += fabsf(er) + fabsf(eg) + fabsf(eb);
        dL_dimage4[pid] = mask_im ? cfg.w_im * sgn(er) : 0.0f;
        dL_dimage4[P + pid] = mask_im ? cfg.w_im * sgn(eg) : 0.0f;
        dL_dimage4[2 * P + pid] = mask_im ? cfg.w_im * sgn(eb) : 0.0f;
        dL_dimage4[3 * P + pid] = mask ? cfg.w_depth * sgn(ed) : 0.0f;
    }
    ld = warp_sum(ld); li = warp_sum(li); cnt = warp_sum(cnt);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (lane == 0) { red.part[warp][0] = ld; red.part[warp][1] = li; red.part[warp][2] = cnt; red.part[warp][3] = 0.f; }
    if (!red.reduce(partials, ticket)) return;
    if (tid == 0) {
        double tot[LOSS_TERMS];
        for (int k = 0; k < LOSS_TERMS; ++k) tot[k] = red.total(k);
        const double wim = (double)cfg.w_im * tot[1], wd = (double)cfg.w_depth * tot[0];
        loss_terms[0] = (float)(wim + wd);
        loss_terms[1] = (float)wim;
        loss_terms[2] = (float)wd;
        loss_terms[3] = (float)tot[2];
        loss_terms[4] = (float)tot[1];
        loss_terms[5] = 0.0f;
        loss_terms[6] = fmaxf(fabsf(cfg.w_im), fabsf(cfg.w_depth));      // >= |dL/dplane| everywhere: VtgsParamGrads.dL_abs_bound
        loss_terms[7] = 0.0f;
    }
}

// =============================== mapping loss (mode 1) =========================================
// Reference get_loss, mapping branch (src/vtgaussian_slam.py:597,608): depth = mean |gt - d| over
// (gt > 0 & ~nan); im = 0.8 * mean|im - gt| + 0.2 * (1 - SSIM), SSIM = calc_ssim
// (utils/slam_external.py:54-97: 11x11 Gaussian window sigma 1.5, zero padding, c1 = 0.01^2, c2 = 0.03^2).
// Three kernels: stats + SSIM forward (per 16x16 tile and channel, separable window in shared memory,
// also emits the three derivative maps), a deterministic finalize, and the SSIM backward that
// convolves the derivative maps and assembles dL/d(r,g,b,depth).
constexpr int SSIM_R = 5;                 // window radius
constexpr int SSIM_T = 32;                // output tile edge: 32 x 32 pixels per block of 256 threads
constexpr int SSIM_H = SSIM_T + 2 * SSIM_R;
constexpr int SSIM_HS = 8;                // horizontal pass: one thread filters a strip of 8 outputs of one row
constexpr int SSIM_VS = 4;                // vertical pass: one thread filters 4 outputs of one column
constexpr int MAP_TERMS = 4;              // per-block partials: rgb L1 sum, depth L1 sum, mask count, ssim sum
static_assert(SSIM_H * (SSIM_T / SSIM_HS) <= 256 && SSIM_T * (SSIM_T / SSIM_VS) == 256, "SSIM strip decomposition");

struct SsimWindow { float g[2 * SSIM_R + 1]; };

static SsimWindow make_window() {
    SsimWindow w;
    float sum = 0.f;
    for (int k = 0; k <= 2 * SSIM_R; ++k) {
        w.g[k] = (float)exp(-(double)((k - SSIM_R) * (k - SSIM_R)) / (2.0 * 1.5 * 1.5));
        sum += w.g[k];
    }
    for (int k = 0; k <= 2 * SSIM_R; ++k) w.g[k] /= sum;
    return w;
}

// grid (ceil(W/32), ceil(H/32), 3 channels); block 256.  Separable 11-tap window over a 42 x 42 halo in shared
// memory; both passes are register-tiled (a thread slides the window over a strip it holds in registers: 18 loads
// feed 8 outputs horizontally, 14 loads feed 4 outputs vertically), which is what bounds this kernel -- shared
// memory loads, not FMAs or HBM.
__global__ void __launch_bounds__(256)
ssim_forward_kernel(int W, int H, const SsimWindow win, const float* __restrict__ image6, const float* __restrict__ gt_rgb,
                    const float* __restrict__ gt_depth, float* __restrict__ maps /* [3 ch][3 maps][P] */,
                    float* __restrict__ partials) {
    VTGS_PDL_PROLOGUE();
    __shared__ float sx[SSIM_H][SSIM_H + 1], sy[SSIM_H][SSIM_H + 1];
    __shared__ float hb[5][SSIM_H][SSIM_T + 1];
    __shared__ float s_part[8][MAP_TERMS];
    const int ch = blockIdx.z;
    const size_t P = (size_t)W * H;
    const float* X = image6 + (size_t)ch * P;
    const float* Y = gt_rgb + (size_t)ch * P;
    const int tid = threadIdx.x;
    const int ox = blockIdx.x * SSIM_T - SSIM_R, oy = blockIdx.y * SSIM_T - SSIM_R;
    for (int k = tid; k < SSIM_H * SSIM_H; k += 256) {
        const int r = k / SSIM_H, c = k % SSIM_H;
        const int gx = ox + c, gy = oy + r;
        const bool in = gx >= 0 && gx < W && gy >= 0 && gy < H;          // zero padding
        sx[r][c] = in ? X[(size_t)gy * W + gx] : 0.0f;
        sy[r][c] = in ? Y[(size_t)gy * W + gx] : 0.0f;
    }
    __syncthreads();
    // horizontal pass: 42 rows x 32 columns of the five fields, strips of 8 columns
    if (tid < SSIM_H * (SSIM_T / SSIM_HS)) {
        const int r = tid / (SSIM_T / SSIM_HS), c0 = (tid % (SSIM_T / SSIM_HS)) * SSIM_HS;
        float xv[SSIM_HS + 2 * SSIM_R], yv[SSIM_HS + 2 * SSIM_R];
#pragma unroll
        for (int i = 0; i < SSIM_HS + 2 * SSIM_R; ++i) { xv[i] = sx[r][c0 + i]; yv[i] = sy[r][c0 + i]; }
#pragma unroll
        for (int o = 0; o < SSIM_HS; ++o) {
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f;
#pragma unroll
            for (int j = 0; j <= 2 * SSIM_R; ++j) {
                const float x = xv[o + j], y = yv[o + j], g = win.g[j];
                a0 = fmaf(g, x, a0); a1 = fmaf(g, y, a1); a2 = fmaf(g, x * x, a2); a3 = fmaf(g, y * y, a3); a4 = fmaf(g, x * y, a4);
            }
            hb[0][r][c0 + o] = a0; hb[1][r][c0 + o] = a1; hb[2][r][c0 + o] = a2; hb[3][r][c0 + o] = a3; hb[4][r][c0 + o] = a4;
        }
    }
    __syncthreads();
    // vertical pass: thread = (group of 4 rows, column)
    const int tx = tid & 31, ty0 = (tid >> 5) * SSIM_VS;
    float f[5][SSIM_VS];
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        float v[SSIM_VS + 2 * SSIM_R];
#pragma unroll
        for (int i = 0; i < SSIM_VS + 2 * SSIM_R; ++i) v[i] = hb[k][ty0 + i][tx];
#pragma unroll
        for (int o = 0; o < SSIM_VS; ++o) {
            float a = 0.f;
#pragma unroll
            for (int j = 0; j <= 2 * SSIM_R; ++j) a = fmaf(win.g[j], v[o + j], a);
            f[k][o] = a;
        }
    }
    const int px = blockIdx.x * SSIM_T + tx;
    float l1 = 0.f, ld = 0.f, cnt = 0.f, ss = 0.f;
#pragma unroll
    for (int o = 0; o < SSIM_VS; ++o) {
        const int ty = ty0 + o, py = blockIdx.y * SSIM_T + ty;
        if (px < W && py < H) {
            const float m1 = f[0][o], m2 = f[1][o], X2 = f[2][o], Y2 = f[3][o], XY = f[4][o];
            const float c1 = 0.0001f, c2 = 0.0009f;
            const float s11 = X2 - m1 * m1, s22 = Y2 - m2 * m2, s12 = XY - m1 * m2;
            const float A1 = 2.f * m1 * m2 + c1, A2 = 2.f * s12 + c2, B1 = m1 * m1 + m2 * m2 + c1, B2 = s11 + s22 + c2;
            const float inv = 1.0f / (B1 * B2);
            const float S = A1 * A2 * inv;
            ss += S;
            const size_t pid = (size_t)py * W + px;
            float* mp = maps + (size_t)ch * 3 * P;
            mp[pid] = (2.f * m2 * (A2 - A1) - 2.f * m1 * S * (B2 - B1)) * inv;      // dS/dmu1 (X2, XY held)
            mp[P + pid] = -S / B2;                                                 // dS/dconv(x^2)
            mp[2 * P + pid] = 2.f * A1 * inv;                                      // dS/dconv(xy)
            l1 += fabsf(sx[ty + SSIM_R][tx + SSIM_R] - sy[ty + SSIM_R][tx + SSIM_R]);
            if (ch == 0) {
                const float d = image6[3 * P + pid], dsq = image6[5 * P + pid], gd = gt_depth[pid];
                const float unc = dsq - d * d;
                if (gd > 0.0f && !(d != d) && !(unc != unc)) { ld += fabsf(gd - d); cnt += 1.0f; }
            }
        }
    }
    l1 = warp_sum(l1); ld = warp_sum(ld); cnt = warp_sum(cnt); ss = warp_sum(ss);
    const int lane = tid & 31, warp = tid >> 5;
    if (lane == 0) { s_part[warp][0] = l1; s_part[warp][1] = ld; s_part[warp][2] = cnt; s_part[warp][3] = ss; }
    __syncthreads();
    if (tid < MAP_TERMS) {
        const size_t b = ((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
        partials[b * MAP_TERMS + tid] = warp_order_sum(s_part, tid);
    }
}

// The slice stage of the fixed-order sum (common.cuh) over ssim_forward_kernel's partials, then the loss terms.
__global__ void __launch_bounds__(1024)
mapping_finalize_kernel(const float* __restrict__ partials, int nblocks, int W, int H, VtgsLossConfig cfg, float* __restrict__ loss_terms) {
    VTGS_PDL_PROLOGUE();
    __shared__ double s_sum[MAP_TERMS][256];
    __shared__ double s_tot[MAP_TERMS];
    const int tid = threadIdx.x;
    slice_sums<MAP_TERMS, 1024, false>(partials, nblocks, s_sum);
    __syncthreads();
    if (tid < MAP_TERMS) s_tot[tid] = slices_total(s_sum, tid);
    __syncthreads();
    if (tid == 0) {
        const double n3 = 3.0 * (double)W * (double)H;
        const double l1_mean = s_tot[0] / n3, ssim = s_tot[3] / n3;
        const double cnt = s_tot[2];
        const double depth_mean = cnt > 0.0 ? s_tot[1] / cnt : 0.0 / 0.0;      // torch: mean of an empty selection is nan
        const double im = 0.8 * l1_mean + 0.2 * (1.0 - ssim);
        loss_terms[0] = (float)((double)cfg.w_im * im + (double)cfg.w_depth * depth_mean);
        loss_terms[1] = (float)((double)cfg.w_im * im);
        loss_terms[2] = (float)((double)cfg.w_depth * depth_mean);
        loss_terms[3] = (float)cnt;
        loss_terms[4] = (float)l1_mean;
        loss_terms[5] = (float)ssim;
        loss_terms[6] = (float)depth_mean;
        loss_terms[7] = 0.0f;
    }
}

// dL/dx = conv(gS * a) + 2 x conv(gS * b) + y conv(gS * c), gS = -0.2 w_im / (3P); plus the L1 terms.
// Same tiling as the forward: 32 x 32 outputs per block, register-tiled separable passes.
__global__ void __launch_bounds__(256)
ssim_backward_kernel(int W, int H, const SsimWindow win, VtgsLossConfig cfg, const float* __restrict__ image6,
                     const float* __restrict__ gt_rgb, const float* __restrict__ gt_depth, const float* __restrict__ maps,
                     const float* __restrict__ loss_terms, float* __restrict__ dL_dimage4) {
    VTGS_PDL_PROLOGUE();
    __shared__ float sm[3][SSIM_H][SSIM_H + 1];
    __shared__ float hb[3][SSIM_H][SSIM_T + 1];
    const int ch = blockIdx.z;
    const size_t P = (size_t)W * H;
    const float* mp = maps + (size_t)ch * 3 * P;
    const int tid = threadIdx.x;
    const int ox = blockIdx.x * SSIM_T - SSIM_R, oy = blockIdx.y * SSIM_T - SSIM_R;
    for (int k = tid; k < SSIM_H * SSIM_H; k += 256) {
        const int r = k / SSIM_H, c = k % SSIM_H;
        const int gx = ox + c, gy = oy + r;
        const bool in = gx >= 0 && gx < W && gy >= 0 && gy < H;
        const size_t pid = (size_t)gy * W + gx;
        sm[0][r][c] = in ? mp[pid] : 0.0f;
        sm[1][r][c] = in ? mp[P + pid] : 0.0f;
        sm[2][r][c] = in ? mp[2 * P + pid] : 0.0f;
    }
    __syncthreads();
    if (tid < SSIM_H * (SSIM_T / SSIM_HS)) {
        const int r = tid / (SSIM_T / SSIM_HS), c0 = (tid % (SSIM_T / SSIM_HS)) * SSIM_HS;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            float v[SSIM_HS + 2 * SSIM_R];
#pragma unroll
            for (int i = 0; i < SSIM_HS + 2 * SSIM_R; ++i) v[i] = sm[k][r][c0 + i];
#pragma unroll
            for (int o = 0; o < SSIM_HS; ++o) {
                float a = 0.f;
#pragma unroll
                for (int j = 0; j <= 2 * SSIM_R; ++j) a = fmaf(win.g[j], v[o + j], a);
                hb[k][r][c0 + o] = a;
            }
        }
    }
    __syncthreads();
    const int tx = tid & 31, ty0 = (tid >> 5) * SSIM_VS;
    float f[3][SSIM_VS];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float v[SSIM_VS + 2 * SSIM_R];
#pragma unroll
        for (int i = 0; i < SSIM_VS + 2 * SSIM_R; ++i) v[i] = hb[k][ty0 + i][tx];
#pragma unroll
        for (int o = 0; o < SSIM_VS; ++o) {
            float a = 0.f;
#pragma unroll
            for (int j = 0; j <= 2 * SSIM_R; ++j) a = fmaf(win.g[j], v[o + j], a);
            f[k][o] = a;
        }
    }
    const int px = blockIdx.x * SSIM_T + tx;
    if (px >= W) return;
    const float n3 = 3.0f * (float)W * (float)H;
#pragma unroll
    for (int o = 0; o < SSIM_VS; ++o) {
        const int py = blockIdx.y * SSIM_T + ty0 + o;
        if (py >= H) break;
        const size_t pid = (size_t)py * W + px;
        const float x = image6[(size_t)ch * P + pid], y = gt_rgb[(size_t)ch * P + pid];
        const float dssim = f[0][o] + 2.0f * x * f[1][o] + y * f[2][o];
        dL_dimage4[(size_t)ch * P + pid] = cfg.w_im * (0.8f * sgn(x - y) - 0.2f * dssim) / n3;
        if (ch == 0) {
            const float d = image6[3 * P + pid], dsq = image6[5 * P + pid], gd = gt_depth[pid];
            const float unc = dsq - d * d;
            const bool mask = gd > 0.0f && !(d != d) && !(unc != unc);
            const float cnt = loss_terms[3];
            dL_dimage4[3 * P + pid] = mask ? cfg.w_depth * sgn(d - gd) / cnt : 0.0f;
        }
    }
}

// ---- re-tie a section's Gaussians to its optimised pose (reference src/vtgaussian_slam.py:2706-2727) ----
// pts <- inv([R(q)|t]) * (w2c_old * pts), q/t read from the device (the pose the optimiser just updated).
// R of an unnormalised pose quaternion: F.normalize, then build_rotation's second normalisation.  Plain fp32 that the
// compiler may contract, so not pose_from_quat's spec'd order: the two give different bits.
__device__ __forceinline__ void retie_rotation(const float* __restrict__ q_un, float* R) {
    const float u0 = q_un[0], u1 = q_un[1], u2 = q_un[2], u3 = q_un[3];
    const float n1 = fmaxf(sqrtf(u0 * u0 + u1 * u1 + u2 * u2 + u3 * u3), 1e-12f);
    const float q0 = u0 / n1, q1 = u1 / n1, q2 = u2 / n1, q3 = u3 / n1;
    const float n2 = sqrtf(q0 * q0 + q1 * q1 + q2 * q2 + q3 * q3);
    quat_to_R(q0 / n2, q1 / n2, q2 / n2, q3 / n2, R);
}

struct Mat34 { float m[12]; };
__global__ void __launch_bounds__(256)
retie_kernel(float* __restrict__ means3D, int64_t n, const Mat34 old, const float* __restrict__ q_un, const float* __restrict__ t) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    float R[9];
    retie_rotation(q_un, R);
    const float x = means3D[3 * i], y = means3D[3 * i + 1], z = means3D[3 * i + 2];
    const float cx = old.m[0] * x + old.m[1] * y + old.m[2] * z + old.m[3] - t[0];
    const float cy = old.m[4] * x + old.m[5] * y + old.m[6] * z + old.m[7] - t[1];
    const float cz = old.m[8] * x + old.m[9] * y + old.m[10] * z + old.m[11] - t[2];
    means3D[3 * i] = R[0] * cx + R[3] * cy + R[6] * cz;          // R^T (p_cam - t)
    means3D[3 * i + 1] = R[1] * cx + R[4] * cy + R[7] * cz;
    means3D[3 * i + 2] = R[2] * cx + R[5] * cy + R[8] * cz;
}

// The same with the OLD pose on the device too (the mapping step snapshots the pose before its Adam update): no host
// round trip, so the mapping iteration stays free of synchronisation.  retie_row re-ties row i; retie_dev_kernel and
// retie_records_kernel both go through it, so their results agree bit for bit.
__device__ __forceinline__ void retie_row(float* __restrict__ means3D, int64_t i, const float* __restrict__ q_old,
                                          const float* __restrict__ t_old, const float* __restrict__ q_un, const float* __restrict__ t) {
    float Ro[9], Rn[9];
    retie_rotation(q_old, Ro);
    retie_rotation(q_un, Rn);
    const float x = means3D[3 * i], y = means3D[3 * i + 1], z = means3D[3 * i + 2];
    const float cx = Ro[0] * x + Ro[1] * y + Ro[2] * z + t_old[0] - t[0];
    const float cy = Ro[3] * x + Ro[4] * y + Ro[5] * z + t_old[1] - t[1];
    const float cz = Ro[6] * x + Ro[7] * y + Ro[8] * z + t_old[2] - t[2];
    means3D[3 * i] = Rn[0] * cx + Rn[3] * cy + Rn[6] * cz;          // R_new^T (p_cam - t_new)
    means3D[3 * i + 1] = Rn[1] * cx + Rn[4] * cy + Rn[7] * cz;
    means3D[3 * i + 2] = Rn[2] * cx + Rn[5] * cy + Rn[8] * cz;
}

__global__ void __launch_bounds__(256)
retie_dev_kernel(float* __restrict__ means3D, int64_t n, const float* __restrict__ q_old, const float* __restrict__ t_old,
                 const float* __restrict__ q_un, const float* __restrict__ t) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    retie_row(means3D, i, q_old, t_old, q_un, t);
}

// ---- the re-ties of a keyframe-sharded bundle-adjustment iteration, every rank's records in one launch ----------------
// Record (VTGS_BA_RECORD_WORDS 32-bit words, include/vtgs.h): valid, id, n_last, reserved | old_q[4] old_t[3] |
// new_q[4] new_t[3] | pad[2].  Each block stages the records in shared memory, RECORD_CHUNK at a time, and walks the
// rows from the lowest one a staged record re-ties.  A row always belongs to the same thread (its index modulo the grid's
// thread count), so the chunks reach it in (rank, slot) order: the order of the unsharded solver's retie_dev calls.
constexpr int RECORD_WORDS = VTGS_BA_RECORD_WORDS;
constexpr int RECORD_CHUNK = 64;                  // 8 ranks x 8 records: the mapping solver's whole exchange in one chunk
constexpr int RECORDS_MAX_WORLD = 8;
static_assert(RECORD_WORDS % 4 == 0, "records are read as 16-byte vectors");
struct RecordTables { uint64_t base[RECORDS_MAX_WORLD]; };

__global__ void __launch_bounds__(256)
retie_records_kernel(const __grid_constant__ RecordTables tabs, int world, int records_per_rank, float* __restrict__ means3D,
                     int64_t n_rows, uint32_t* __restrict__ table_out) {
    __shared__ uint4 s_rec[RECORD_CHUNK * RECORD_WORDS / 4];
    const uint32_t* rec = reinterpret_cast<const uint32_t*>(s_rec);
    const int64_t total = (int64_t)world * records_per_rank, stride = (int64_t)gridDim.x * 256;
    for (int64_t c0 = 0; c0 < total; c0 += RECORD_CHUNK) {
        const int nrec = (int)min((int64_t)RECORD_CHUNK, total - c0);
        for (int k = threadIdx.x; k < nrec * (RECORD_WORDS / 4); k += 256) {
            const int64_t r = (c0 + k / (RECORD_WORDS / 4)) / records_per_rank, s = (c0 + k / (RECORD_WORDS / 4)) % records_per_rank;
            const uint4 w = reinterpret_cast<const uint4*>(tabs.base[r])[s * (RECORD_WORDS / 4) + k % (RECORD_WORDS / 4)];
            s_rec[k] = w;
            if (table_out != nullptr && blockIdx.x == 0) {
                uint32_t* o = table_out + c0 * RECORD_WORDS + 4 * (int64_t)k;
                o[0] = w.x; o[1] = w.y; o[2] = w.z; o[3] = w.w;
            }
        }
        __syncthreads();
        int64_t lo = n_rows;
        for (int j = 0; j < nrec; ++j) {
            const int32_t n_last = (int32_t)rec[j * RECORD_WORDS + 2];
            if (rec[j * RECORD_WORDS] != 0u && n_last > 0) lo = min(lo, n_rows - min((int64_t)n_last, n_rows));
        }
        for (int64_t i = lo / stride * stride + (int64_t)blockIdx.x * 256 + threadIdx.x; i < n_rows; i += stride) {
            for (int j = 0; j < nrec; ++j) {
                const uint32_t* R = rec + j * RECORD_WORDS;
                const int32_t n_last = (int32_t)R[2];
                if (R[0] == 0u || n_last <= 0 || i < n_rows - min((int64_t)n_last, n_rows)) continue;
                const float* f = reinterpret_cast<const float*>(R);
                retie_row(means3D, i, f + 4, f + 8, f + 11, f + 15);
            }
        }
        __syncthreads();
    }
}

// ---- Adam -----------------------------------------------------------------------------------
// beta^t by repeated squaring in fp64: a dozen DMULs (pow() is microseconds of serial fp64 on this part,
// paid as a prologue by every block).
__device__ __forceinline__ double ipow(double b, int t) {
    double r = 1.0;
    for (int e = t; e > 0; e >>= 1) {
        if (e & 1) r *= b;
        b *= b;
    }
    return r;
}

// torch.optim.Adam's update of one element; step_size = lr / (1 - b1^t), bc2s = sqrt(1 - b2^t)
__device__ __forceinline__ void adam_update(float& p, const float g, float& m, float& v, float step_size, float bc2s, float b1,
                                            float b2, float eps) {
    const float mi = m + (1.0f - b1) * (g - m);                 // exp_avg.lerp_(grad, 1 - beta1)
    const float vi = b2 * v + (1.0f - b2) * g * g;              // exp_avg_sq.mul_(b2).addcmul_(g, g, 1 - b2)
    m = mi; v = vi;
    const float denom = sqrtf(vi) / bc2s + eps;
    p = p - step_size * (mi / denom);
}

__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int64_t n,
            float lr, float b1, float b2, float eps, int step, const int32_t* __restrict__ step_dev, int vec4) {
    VTGS_PDL_PROLOGUE();
    __shared__ float s_c[2];
    if (threadIdx.x == 0) {
        const int t = step_dev ? *step_dev : step;
        const double bc1 = 1.0 - ipow((double)b1, t);
        const double bc2 = 1.0 - ipow((double)b2, t);
        s_c[0] = (float)((double)lr / bc1);
        s_c[1] = (float)sqrt(bc2);
    }
    __syncthreads();
    const float step_size = s_c[0], bc2s = s_c[1];
    auto upd = [&](float& pi, const float gi, float& mi, float& vi) { adam_update(pi, gi, mi, vi, step_size, bc2s, b1, b2, eps); };
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (vec4) {                                                      // four elements per thread, 16-byte accesses
        if (4 * i >= n) return;
        float4 p4 = reinterpret_cast<float4*>(p)[i], m4 = reinterpret_cast<float4*>(m)[i], v4 = reinterpret_cast<float4*>(v)[i];
        const float4 g4 = reinterpret_cast<const float4*>(g)[i];
        upd(p4.x, g4.x, m4.x, v4.x); upd(p4.y, g4.y, m4.y, v4.y); upd(p4.z, g4.z, m4.z, v4.z); upd(p4.w, g4.w, m4.w, v4.w);
        reinterpret_cast<float4*>(p)[i] = p4; reinterpret_cast<float4*>(m)[i] = m4; reinterpret_cast<float4*>(v)[i] = v4;
        return;
    }
    if (i >= n) return;
    float pi = p[i], mi = m[i], vi = v[i];
    upd(pi, g[i], mi, vi);
    p[i] = pi; m[i] = mi; v[i] = vi;
}

// ---- keyframe-sharded mapping step: reduce-scatter + Adam + all-gather in ONE kernel over NVLink peer memory ----------
// Every rank holds the same symmetric block [params | gradients | loss] (torch symmetric memory: each rank's block is
// mapped into every other rank's address space).  Rank r owns the r-th slice of the flat vectors: it reads that slice of
// the gradients from ALL ranks (peer loads over NVLink, summed in rank order: a fixed order), applies Adam with ITS
// slice of the moments (the optimiser state is sharded: 1 / world of the memory and of the work), and stores the
// updated parameters into every rank's block (peer stores).  Per rank and step: n floats in, n floats out over NVLink,
// against the all-reduce's 2 n (world - 1) / world each way plus a replicated Adam over all n.
// The caller brackets the launch with two cross-device barriers (gradients complete before / parameters landed after).
constexpr int SHARD_MAX_WORLD = 8;
struct ShardedAdamArgs {
    uint64_t base[SHARD_MAX_WORLD];   // peer base pointers of the symmetric block
    uint64_t pbase[SHARD_MAX_WORLD];  // (the same blocks: where the new parameters are stored)
    int64_t seg_end[4];               // flat layout: segment s = [seg_end[s-1], seg_end[s]) elements, learning rate lr[s]
    float lr[4];
    int nseg, world, rank;
};

// The sharded kernels' step constants (thread 0 of each block): lr[s] / (1 - b1^t) per segment s, and sqrt(1 - b2^t)
__device__ __forceinline__ void sharded_adam_consts(const ShardedAdamArgs& a, float b1, float b2, int t, float (&step)[4], float& bc2s) {
    const double bc1 = 1.0 - ipow((double)b1, t);
    for (int k = 0; k < a.nseg; ++k) step[k] = (float)((double)a.lr[k] / bc1);
    bc2s = (float)sqrt(1.0 - ipow((double)b2, t));
}
// the segment of flat element e, whose learning rate it takes
__device__ __forceinline__ int segment_of(const ShardedAdamArgs& a, int64_t e) {
    int sg = 0;
    while (sg + 1 < a.nseg && e >= a.seg_end[sg]) ++sg;
    return sg;
}

// W: ranks (compile-time: the peer loads of one element are issued together), U: float4 per thread and trip, so that
// about eight remote 16-byte loads are in flight per thread whatever the world size (an NVLink round trip is ~3 us)
template <int W, int U>
__global__ void __launch_bounds__(256)
sharded_adam_kernel(const __grid_constant__ ShardedAdamArgs a, int64_t param_off, int64_t grad_off, int64_t loss_off,
                    float* __restrict__ m, float* __restrict__ v, int64_t n4, float b1, float b2, float eps,
                    const int32_t* __restrict__ step_dev, float* __restrict__ loss_out) {
    __shared__ float s_step[4], s_bc2s;
    if (threadIdx.x == 0) {
        sharded_adam_consts(a, b1, b2, *step_dev, s_step, s_bc2s);
        if (blockIdx.x == 0) {
            float L = 0.0f;
            for (int k = 0; k < a.world; ++k) L += reinterpret_cast<const float*>(a.base[k])[loss_off];
            *loss_out = L;
        }
    }
    __syncthreads();
    const float bc2s = s_bc2s;
    const int64_t per = (n4 + a.world - 1) / a.world;
    const int64_t begin = per * a.rank, end = min(n4, begin + per);
    const float4* gsrc[W];
    float4* pdst[W];
#pragma unroll
    for (int k = 0; k < W; ++k) {
        const int kk = k < a.world ? k : a.rank;          // (W > world: the spare slots alias this rank and are skipped)
        gsrc[k] = reinterpret_cast<const float4*>(a.base[kk]) + grad_off / 4;
        pdst[k] = reinterpret_cast<float4*>(a.pbase[kk]) + param_off / 4;
    }
    const float4* my_p = reinterpret_cast<const float4*>(a.base[a.rank]) + param_off / 4;   // identical everywhere: local copy
    auto upd = [&](float& pi, const float gi, float& mi, float& vi, int64_t e) {
        adam_update(pi, gi, mi, vi, s_step[segment_of(a, e)], bc2s, b1, b2, eps);
    };
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t j0 = begin + (int64_t)blockIdx.x * 256 + threadIdx.x; j0 < end; j0 += stride * U) {
        float4 g[U][W];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t j = j0 + u * stride;
#pragma unroll
            for (int k = 0; k < W; ++k)
                if (k < a.world && j < end) g[u][k] = gsrc[k][j];
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t j = j0 + u * stride;
            if (j >= end) break;
            float4 gs = g[u][0];
#pragma unroll
            for (int k = 1; k < W; ++k)
                if (k < a.world) { gs.x += g[u][k].x; gs.y += g[u][k].y; gs.z += g[u][k].z; gs.w += g[u][k].w; }
            float4 p4 = my_p[j], m4 = reinterpret_cast<float4*>(m)[j - begin], v4 = reinterpret_cast<float4*>(v)[j - begin];
            upd(p4.x, gs.x, m4.x, v4.x, 4 * j); upd(p4.y, gs.y, m4.y, v4.y, 4 * j + 1);
            upd(p4.z, gs.z, m4.z, v4.z, 4 * j + 2); upd(p4.w, gs.w, m4.w, v4.w, 4 * j + 3);
            reinterpret_cast<float4*>(m)[j - begin] = m4; reinterpret_cast<float4*>(v)[j - begin] = v4;
#pragma unroll
            for (int k = 0; k < W; ++k)
                if (k < a.world) pdst[k][j] = p4;
        }
    }
}

// The same step through the NVSwitch's multicast object (NVLS), when torch's symmetric memory could bind one: ONE
// multimem.ld_reduce pulls the sum of a 16-byte vector over all ranks (reduced inside the switch: the rank receives its
// slice once instead of `world` times) and ONE multimem.st pushes the new parameters to every rank.
__global__ void __launch_bounds__(256)
sharded_adam_mc_kernel(const __grid_constant__ ShardedAdamArgs a, uint64_t mc_base, int64_t param_off, int64_t grad_off,
                       int64_t loss_off, float* __restrict__ m, float* __restrict__ v, int64_t n4, float b1, float b2, float eps,
                       const int32_t* __restrict__ step_dev, float* __restrict__ loss_out) {
    __shared__ float s_step[4], s_bc2s;
    if (threadIdx.x == 0) {
        sharded_adam_consts(a, b1, b2, *step_dev, s_step, s_bc2s);
        if (blockIdx.x == 0) {
            float L;
            asm volatile("multimem.ld_reduce.relaxed.sys.global.add.f32 %0, [%1];" : "=f"(L) : "l"(reinterpret_cast<const float*>(mc_base) + loss_off) : "memory");
            *loss_out = L;
        }
    }
    __syncthreads();
    const float bc2s = s_bc2s;
    const int64_t per = (n4 + a.world - 1) / a.world;
    const int64_t begin = per * a.rank, end = min(n4, begin + per);
    const float4* mc_g = reinterpret_cast<const float4*>(mc_base) + grad_off / 4;
    float4* mc_p = reinterpret_cast<float4*>(mc_base) + param_off / 4;
    const float4* my_p = reinterpret_cast<const float4*>(a.base[a.rank]) + param_off / 4;
    auto upd = [&](float& pi, const float gi, float& mi, float& vi, int64_t e) {
        adam_update(pi, gi, mi, vi, s_step[segment_of(a, e)], bc2s, b1, b2, eps);
    };
    constexpr int U = 4;
    const int64_t stride = (int64_t)gridDim.x * 256;
    for (int64_t j0 = begin + (int64_t)blockIdx.x * 256 + threadIdx.x; j0 < end; j0 += stride * U) {
        float4 gs[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t j = j0 + u * stride;
            if (j < end)
                asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
                             : "=f"(gs[u].x), "=f"(gs[u].y), "=f"(gs[u].z), "=f"(gs[u].w) : "l"(mc_g + j) : "memory");
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t j = j0 + u * stride;
            if (j >= end) break;
            float4 p4 = my_p[j], m4 = reinterpret_cast<float4*>(m)[j - begin], v4 = reinterpret_cast<float4*>(v)[j - begin];
            upd(p4.x, gs[u].x, m4.x, v4.x, 4 * j); upd(p4.y, gs[u].y, m4.y, v4.y, 4 * j + 1);
            upd(p4.z, gs[u].z, m4.z, v4.z, 4 * j + 2); upd(p4.w, gs[u].w, m4.w, v4.w, 4 * j + 3);
            reinterpret_cast<float4*>(m)[j - begin] = m4; reinterpret_cast<float4*>(v)[j - begin] = v4;
            asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};"
                         :: "l"(mc_p + j), "f"(p4.x), "f"(p4.y), "f"(p4.z), "f"(p4.w) : "memory");
        }
    }
}

// ---- tracking pose update: best-candidate bookkeeping + Adam on the 7 pose numbers, one launch ----
// Reference src/vtgaussian_slam.py:1890 (optimizer.step) and :1961-1970 (keep the candidate pose with
// the smallest loss; the loss of an iteration belongs to the pose BEFORE that iteration's step).
__global__ void tracking_update_kernel(float* __restrict__ cam_q, float* __restrict__ cam_t, const float* __restrict__ msg,
                                       float* __restrict__ adam, int32_t* __restrict__ step_dev, float* __restrict__ best,
                                       float lr_rot, float lr_trans, float b1, float b2, float eps, int flags) {
    VTGS_PDL_PROLOGUE();
    const int k = threadIdx.x;           // 0..3 quaternion, 4..6 translation
    __shared__ int s_step;
    __shared__ bool s_better;
    if (k == 0) {
        s_step = *step_dev + 1;
        *step_dev = s_step;
        const float metric = (flags & VTGS_TRACK_CALLER_METRIC) ? msg[15] : msg[8];
        s_better = metric < best[0];
        if (s_better) best[0] = metric;
    }
    __syncthreads();
    if (k >= 7) return;
    float* p = k < 4 ? cam_q + k : cam_t + (k - 4);
    if (s_better && !(flags & VTGS_TRACK_BOOK_POST_STEP)) best[1 + k] = *p;
    const float g = msg[k];
    float* m = adam + (k < 4 ? k : 8 + (k - 4));
    float* v = adam + (k < 4 ? 4 + k : 11 + (k - 4));
    const double bc1 = 1.0 - ipow((double)b1, s_step), bc2 = 1.0 - ipow((double)b2, s_step);
    const float step_size = (float)((double)(k < 4 ? lr_rot : lr_trans) / bc1);
    float pn = *p, mi = *m, vi = *v;
    adam_update(pn, g, mi, vi, step_size, (float)sqrt(bc2), b1, b2, eps);
    *m = mi; *v = vi; *p = pn;
    if (s_better && (flags & VTGS_TRACK_BOOK_POST_STEP)) best[1 + k] = pn;
}

}  // namespace vtgs

// =============================== C entry points (include/vtgs.h) ===========================
using namespace vtgs;

uint64_t vtgs_loss_scratch_floats(int32_t W, int32_t H, int32_t mode) {
    const uint64_t P = (uint64_t)W * H;
    if (mode == 1) return 9 * P + ((uint64_t)((W + 15) / 16) * ((H + 15) / 16) * 3 + 1) * 4;
    /* [tracking loss: 4 floats per 1024-pixel block + ticket + the radix-select state of the outlier median (320 words)
     *  | silhouette ladder: 10 floats per block + ticket] */
    return ((P + 1023) / 1024) * 14 + 320 + 16;
}

int vtgs_loss(const VtgsCamera* camera, const VtgsLossConfig* cfg, const float* image6, const float* gt_rgb,
              const float* gt_depth, float* dL_dimage4, float* loss_terms, float* scratch, void* stream_) {
    if (int e = check_cam(camera)) return e;
    VTGS_REQUIRE(cfg && image6 && gt_rgb && gt_depth && dL_dimage4 && loss_terms && scratch, "pointer is NULL");
    const cudaStream_t stream = (cudaStream_t)stream_;
    const CamConst cam = make_cam_const(*camera);
    if (cfg->ignore_outlier_depth && cfg->mode != 0) { set_error("ignore_outlier_depth_loss is a tracking option"); return VTGS_E_UNSUPPORTED; }
    if (cfg->ignore_outlier_depth && cfg->median_state == nullptr && (cam.row0 != 0 || cam.row1 != cam.gy)) {
        set_error("ignore_outlier_depth_loss with a tile-row band needs VtgsLossConfig.median_state (vtgs_median_hist / all-reduce / vtgs_median_pick)");
        return VTGS_E_UNSUPPORTED;
    }
    if (!cfg->use_l1) { set_error("use_l1 = False is not supported"); return VTGS_E_UNSUPPORTED; }
    if (cfg->mode == 1) {
        if (cam.row0 != 0 || cam.row1 != cam.gy) { set_error("mapping loss is not band-sharded"); return VTGS_E_INVALID; }
        static const SsimWindow win = make_window();
        const size_t P = (size_t)cam.W * cam.H;
        const dim3 grid((cam.W + SSIM_T - 1) / SSIM_T, (cam.H + SSIM_T - 1) / SSIM_T, 3), block(256);
        const int nb = (int)(grid.x * grid.y * grid.z);
        float* maps = scratch;                      // 9 P floats
        float* partials = scratch + 9 * P;          // nb * 4
        if (int e = launch_k("ssim_forward_kernel", Launch::pdl, ssim_forward_kernel, grid, block, 0, stream, cam.W, cam.H, win, image6, gt_rgb,
                             gt_depth, maps, partials)) return e;
        if (int e = launch_k("mapping_finalize_kernel", Launch::pdl, mapping_finalize_kernel, dim3(1), dim3(1024), 0, stream, partials, nb, cam.W,
                             cam.H, *cfg, loss_terms)) return e;
        return launch_k("ssim_backward_kernel", Launch::pdl, ssim_backward_kernel, grid, block, 0, stream, cam.W, cam.H, win, *cfg, image6, gt_rgb,
                        gt_depth, maps, loss_terms, dL_dimage4);
    }
    if (cfg->mode != 0) { set_error("unknown loss mode"); return VTGS_E_INVALID; }
    size_t pix_b, pix_e;
    band_pixel_range(cam, pix_b, pix_e);
    const int nblocks = (int)((pix_e - pix_b + 256 * LOSS_PX_PER_THREAD - 1) / (256 * LOSS_PX_PER_THREAD));
    if (nblocks > 0) {
        unsigned int* ticket = reinterpret_cast<unsigned int*>(scratch + (size_t)nblocks * LOSS_TERMS);
        const unsigned int* median_state = nullptr;
        if (cfg->ignore_outlier_depth && cfg->median_state != nullptr) {
            median_state = cfg->median_state;
        } else if (cfg->ignore_outlier_depth) {
            unsigned int* st = ticket + 16;
            const size_t P = (size_t)cam.W * cam.H;
            VTGS_CUDA_CHECK(cudaMemsetAsync(st, 0, MEDIAN_STATE_WORDS * sizeof(unsigned int), stream));
            for (int pass = 0; pass < 4; ++pass) {
                if (int e = launch_median_hist(camera, image6 + 3 * P, gt_depth, pass, st, stream)) return e;
                if (int e = launch_median_pick((int64_t)P, pass, st, stream)) return e;
            }
            median_state = st;
        }
        return launch_k("tracking_loss_kernel", Launch::pdl, tracking_loss_kernel, dim3(nblocks), dim3(256), 0, stream, cam, *cfg, image6, gt_rgb,
                        gt_depth, dL_dimage4, scratch, ticket, loss_terms, median_state);
    }
    VTGS_CUDA_CHECK(cudaMemsetAsync(loss_terms, 0, 8 * sizeof(float), stream));
    return VTGS_OK;
}

int vtgs_median_hist(const VtgsCamera* cam, const float* depth_plane, const float* gt_depth, int32_t pass, uint32_t* state, void* stream) {
    if (int e = check_cam(cam)) return e;
    VTGS_REQUIRE(depth_plane && gt_depth && state, "pointer is NULL");
    VTGS_REQUIRE(pass >= 0 && pass < 4, "pass must be 0..3");
    return launch_median_hist(cam, depth_plane, gt_depth, pass, state, (cudaStream_t)stream);
}

int vtgs_median_pick(int64_t num_pixels_total, int32_t pass, uint32_t* state, void* stream) {
    VTGS_REQUIRE(state != nullptr && num_pixels_total > 0, "bad argument");
    VTGS_REQUIRE(pass >= 0 && pass < 4, "pass must be 0..3");
    return launch_median_pick(num_pixels_total, pass, state, (cudaStream_t)stream);
}

int vtgs_sil_ladder(const VtgsCamera* camera, const float* image6, const float* gt_rgb, const float* gt_depth, float* sums10,
                    float* scratch, void* stream_) {
    if (int e = check_cam(camera)) return e;
    VTGS_REQUIRE(image6 && gt_rgb && gt_depth && sums10 && scratch, "pointer is NULL");
    const cudaStream_t stream = (cudaStream_t)stream_;
    const CamConst cam = make_cam_const(*camera);
    size_t b, e;
    band_pixel_range(cam, b, e);
    const int nblocks = (int)((e - b + 1023) / 1024);
    if (nblocks <= 0) { VTGS_CUDA_CHECK(cudaMemsetAsync(sums10, 0, 10 * sizeof(float), stream)); return VTGS_OK; }
    // the loss scratch (vtgs_loss_scratch_floats, mode 0) = [tracking-loss region: 4 floats per 1024-pixel block of the
    // whole frame, its ticket, the median state | ladder region: 10 floats per block, its ticket]: the two never overlap,
    // so the tracking loss's self-resetting ticket stays intact
    const size_t nb_full = ((size_t)cam.W * cam.H + 1023) / 1024;
    float* part = scratch + nb_full * 4 + 320;
    unsigned int* ticket = reinterpret_cast<unsigned int*>(part + nb_full * 2 * LADDER_N);
    VTGS_CUDA_CHECK(cudaMemsetAsync(ticket, 0, sizeof(unsigned int), stream));
    return launch_k("sil_ladder_kernel", Launch::plain, sil_ladder_kernel, dim3(nblocks), dim3(256), 0, stream, cam, image6, gt_rgb, gt_depth,
                    part, ticket, sums10);
}

int vtgs_sil_select(const float* sums10, float* sil_thres_dev, float* min_mse_dev, void* stream) {
    VTGS_REQUIRE(sums10 && sil_thres_dev, "pointer is NULL");
    return launch_k("sil_select_kernel", Launch::plain, sil_select_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, sums10, sil_thres_dev,
                    min_mse_dev);
}

int vtgs_nonpresence_mask(const VtgsCamera* camera, const float* image6, const float* gt_depth, float sil_thres,
                          const uint32_t* median_state, uint8_t* mask_out, uint32_t* count_dev, void* stream_) {
    if (int e = check_cam(camera)) return e;
    VTGS_REQUIRE(image6 && gt_depth && median_state && mask_out, "pointer is NULL");
    const cudaStream_t stream = (cudaStream_t)stream_;
    const size_t P = (size_t)camera->image_width * camera->image_height;
    if (count_dev) VTGS_CUDA_CHECK(cudaMemsetAsync(count_dev, 0, sizeof(uint32_t), stream));
    return launch_k("nonpresence_mask_kernel", Launch::plain, nonpresence_mask_kernel, dim3((unsigned)((P + 255) / 256)), dim3(256), 0, stream,
                    P, image6, gt_depth, sil_thres, median_state, mask_out, count_dev);
}

int vtgs_ffma_probe(int64_t iters, float* sink, uint64_t* threads_out, void* stream) {
    VTGS_REQUIRE(iters > 0 && sink != nullptr, "bad argument");
    const int blocks = 148 * 8;                          // 8 resident blocks of 256 threads per SM: 64 warps / SM
    if (threads_out) *threads_out = (uint64_t)blocks * 256;
    return launch_k("ffma_probe_kernel", Launch::plain, ffma_probe_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, (long long)iters, sink);
}

int vtgs_retie(float* means3D, int64_t n, const float* w2c_old, const float* cam_unnorm_rot, const float* cam_trans, void* stream) {
    VTGS_REQUIRE(n >= 0, "n < 0");
    VTGS_REQUIRE(w2c_old && cam_unnorm_rot && cam_trans && (n == 0 || means3D), "pointer is NULL");
    if (n <= 0) return VTGS_OK;
    Mat34 m;
    for (int k = 0; k < 12; ++k) m.m[k] = w2c_old[k];
    return launch_k("retie_kernel", Launch::plain, retie_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, means3D, n,
                    m, cam_unnorm_rot, cam_trans);
}

int vtgs_retie_dev(float* means3D, int64_t n, const float* old_unnorm_rot, const float* old_trans, const float* cam_unnorm_rot,
                   const float* cam_trans, void* stream) {
    VTGS_REQUIRE(n >= 0, "n < 0");
    VTGS_REQUIRE(old_unnorm_rot && old_trans && cam_unnorm_rot && cam_trans && (n == 0 || means3D), "pointer is NULL");
    if (n <= 0) return VTGS_OK;
    return launch_k("retie_kernel", Launch::plain, retie_dev_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream,
                    means3D, n, old_unnorm_rot, old_trans, cam_unnorm_rot, cam_trans);
}

int vtgs_retie_records(int32_t world, const uint64_t* table_bases, int32_t records_per_rank, float* means3D, int64_t n_rows,
                       uint32_t* table_out, void* stream) {
    VTGS_REQUIRE(world >= 1 && world <= RECORDS_MAX_WORLD, "world must be 1..8");
    VTGS_REQUIRE(records_per_rank >= 1, "records_per_rank must be >= 1");
    VTGS_REQUIRE(n_rows >= 0, "n_rows < 0");
    VTGS_REQUIRE(table_bases && (n_rows == 0 || means3D), "pointer is NULL");
    for (int k = 0; k < world; ++k) VTGS_REQUIRE(table_bases[k] != 0 && (table_bases[k] & 15) == 0, "table base must be a 16-byte aligned address");
    if (n_rows == 0 && table_out == nullptr) return VTGS_OK;
    RecordTables tabs{};
    for (int k = 0; k < world; ++k) tabs.base[k] = table_bases[k];
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n_rows + 255) / 256, 148 * 2));
    return launch_k("retie_records_kernel", Launch::plain, retie_records_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, tabs, (int)world,
                    (int)records_per_rank, means3D, n_rows, table_out);
}

int vtgs_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
              float beta2, float eps, int32_t step, const int32_t* step_dev, void* stream) {
    VTGS_REQUIRE(n >= 0, "n < 0");
    if (n > 0) VTGS_REQUIRE(param && grad && exp_avg && exp_avg_sq, "pointer is NULL");
    VTGS_REQUIRE(step_dev != nullptr || step >= 1, "step must be >= 1");
    if (n <= 0) return VTGS_OK;
    const bool vec4 = (n % 4 == 0) && (((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0;
    const int64_t threads = vec4 ? n / 4 : n;
    return launch_k("adam_kernel", Launch::pdl, adam_kernel, dim3((unsigned)((threads + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, param,
                    grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, step_dev, vec4 ? 1 : 0);
}

int vtgs_sharded_adam(int32_t world, int32_t rank, const uint64_t* peer_bases, uint64_t multicast_base, int64_t param_off, int64_t grad_off, int64_t loss_off,
                      float* exp_avg, float* exp_avg_sq, int64_t n, int32_t nseg, const int64_t* seg_end, const float* lr, float beta1,
                      float beta2, float eps, const int32_t* step_dev, float* loss_out, void* stream) {
    VTGS_REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world, "world must be 1..8 and rank inside it");
    VTGS_REQUIRE(peer_bases && exp_avg && exp_avg_sq && seg_end && lr && step_dev && loss_out, "pointer is NULL");
    VTGS_REQUIRE(n >= 0 && n % 4 == 0 && param_off % 4 == 0 && grad_off % 4 == 0, "flat vectors must be multiples of 4 floats");
    VTGS_REQUIRE(nseg >= 1 && nseg <= 4, "1..4 segments");
    for (int k = 0; k < world; ++k) VTGS_REQUIRE(peer_bases[k] != 0 && (peer_bases[k] & 15) == 0, "peer base must be a 16-byte aligned address");
    VTGS_REQUIRE((multicast_base & 15) == 0, "multicast base must be 16-byte aligned");
    ShardedAdamArgs a{};
    a.nseg = nseg; a.world = world; a.rank = rank;
    for (int k = 0; k < world; ++k) a.base[k] = peer_bases[k];
    for (int k = 0; k < world; ++k) a.pbase[k] = peer_bases[k];
    for (int k = 0; k < nseg; ++k) { a.seg_end[k] = seg_end[k]; a.lr[k] = lr[k]; }
    const int64_t n4 = n / 4;
    int blocks = 148 * 4;
    if (const char* e = getenv("VTGS_SHARD_BLOCKS")) blocks = std::max(1, atoi(e));      // tools/bench_sharded_step.py (8 B200: flat from 296 blocks on)
    if (multicast_base != 0)
        return launch_k("sharded_adam_kernel", Launch::plain, sharded_adam_mc_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, a,
                        multicast_base, param_off, grad_off, loss_off, exp_avg, exp_avg_sq, n4, beta1, beta2, eps, step_dev, loss_out);
    auto k = world <= 2 ? sharded_adam_kernel<2, 4> : world <= 4 ? sharded_adam_kernel<4, 2> : sharded_adam_kernel<8, 1>;
    return launch_k("sharded_adam_kernel", Launch::plain, k, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, a, param_off, grad_off, loss_off,
                    exp_avg, exp_avg_sq, n4, beta1, beta2, eps, step_dev, loss_out);
}

int vtgs_tracking_update(float* cam_unnorm_rot, float* cam_trans, const float* msg, float* adam_state, int32_t* step_dev,
                         float* best, float lr_rot, float lr_trans, float eps, int32_t flags, void* stream) {
    VTGS_REQUIRE(cam_unnorm_rot && cam_trans && msg && adam_state && step_dev && best, "pointer is NULL");
    return launch_k("tracking_update_kernel", Launch::pdl, tracking_update_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, cam_unnorm_rot,
                    cam_trans, msg, adam_state, step_dev, best, lr_rot, lr_trans, 0.9f, 0.999f, eps, flags);
}
