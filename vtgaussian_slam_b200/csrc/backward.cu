// backward.cu -- K6' backward blend and K7' backward preprocess (sm_100a).
//
// Replaces `_C.rasterize_gaussians_backward` of the reference's external rasteriser
// (triggered by loss.backward() at reference src/vtgaussian_slam.py:1889,2686; upstream
// BACKWARD::render / computeCov2DCUDA / preprocessCUDA, SURVEY.md Appendix A.5-A.6) and,
// in fused mode, the autograd chain the reference runs around it: get_depth_and_silhouette
// (utils/slam_helpers.py:217-234), the activations (:127-160) and transform_to_frame
// (:323-385) down to the Gaussian parameters and the 7 camera-pose numbers.
//
// K6' design: see the comment above blend_backward_kernel.
#include <algorithm>
#include <atomic>

#include "blend_common.cuh"
#include "kernels.h"

namespace vtgs {

// Sum NV (<= 16) per-lane values across the warp.  On return lane L holds the warp total of
// value (L >> 1) in v[0].  Each butterfly level halves the number of live values.
template <int NV>
__device__ __forceinline__ float warp_transpose_reduce(float (&v)[16], int lane) {
    static_assert(NV <= 16, "at most 16 values");
#pragma unroll
    for (int k = NV; k < 16; ++k) v[k] = 0.0f;
    {
        const bool up = lane & 16;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float send = up ? v[i] : v[i + 8];
            const float keep = up ? v[i + 8] : v[i];
            v[i] = keep + __shfl_xor_sync(VTGS_FULL_MASK, send, 16);
        }
    }
    {
        const bool up = lane & 8;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float send = up ? v[i] : v[i + 4];
            const float keep = up ? v[i + 4] : v[i];
            v[i] = keep + __shfl_xor_sync(VTGS_FULL_MASK, send, 8);
        }
    }
    {
        const bool up = lane & 4;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float send = up ? v[i] : v[i + 2];
            const float keep = up ? v[i + 2] : v[i];
            v[i] = keep + __shfl_xor_sync(VTGS_FULL_MASK, send, 4);
        }
    }
    {
        const bool up = lane & 2;
        const float send = up ? v[0] : v[1];
        const float keep = up ? v[1] : v[0];
        v[0] = keep + __shfl_xor_sync(VTGS_FULL_MASK, send, 2);
    }
    v[0] += __shfl_xor_sync(VTGS_FULL_MASK, v[0], 1);
    return v[0];
}


// ---- deterministic accumulation (VTGS_BUF_DETERMINISTIC, include/vtgs.h) --------------------------------------------
// Every partial sum v of a quantity whose per-Gaussian total of |v| is bounded by B < 2^e is split into
//   hi = v rounded to a multiple of q_hi = 2^(e - 22),   lo = (v - hi) rounded to a multiple of q_lo = q_hi 2^(-s_lo)
// and the two are accumulated with the ordinary fp32 vector reductions.  Sums of multiples of q that stay below 2^24 q
// are EXACT in fp32, so they do not depend on the order in which the warps of different tiles and regions arrive:
// |sum hi| <= B + (#partials) q_hi / 2 < 2^24 q_hi, and |sum lo| <= (#partials) q_hi / 2 < 2^24 q_lo with
// s_lo = 21 - ceil(log2(tiles)) (at most 8 partials per tile).  K7' adds hi + lo: 22 + s_lo bits below the bound.
// grad_geom record in this mode (32-float stride):
//   [0..3] hi{mean2D.x, mean2D.y, conic.xx, conic.xy}   [4..7] hi{conic.yy, colour 3}, lo{mean2D.x, mean2D.y}
//   [8..11] lo{conic.xx, conic.xy, conic.yy, colour 3}  [12..15] hi{opacity, r, g, b}   [16..19] lo{opacity, r, g, b}
// (the pose-only instantiation touches the first 48 bytes: three vector reductions per partial, as many memory
// operations as without the flag).
constexpr int DET_STRIDE = 32;        // floats per record; the pose-only form (12 floats) keeps the plain path's 16-float stride: same sectors for K7'
__host__ __device__ constexpr int det_stride(bool pose_only) { return pose_only ? 16 : DET_STRIDE; }

__device__ __forceinline__ int det_exponent(float bound) {          // smallest e (clamped) with bound < 2^e
    const int e = (int)((__float_as_uint(bound) >> 23) & 0xffu) - 126;
    return min(max(e, -80), 100);
}
__device__ __forceinline__ float det_pow2(int s) { return __uint_as_float((uint32_t)(s + 127) << 23); }   // 2^s, s in [-126, 127]
// v -> (hi, lo) on the grids of exponent e: c_hi = 3 * 2^e (rounds to multiples of 2^(e-22)), c_lo = 3 * 2^(e - s_lo)
__device__ __forceinline__ float2 det_split(float v, float c_hi, float c_lo) {
    const float hi = __fsub_rn(__fadd_rn(v, c_hi), c_hi);
    const float r = __fsub_rn(v, hi);                                 // exact
    return make_float2(hi, __fsub_rn(__fadd_rn(r, c_lo), c_lo));
}

// max |dL/dpixel| over the band's rows and the NCH planes -> *out_bits (atomicMax on the bit pattern; zeroed by the forward)
__global__ void __launch_bounds__(256)
dpix_max_kernel(const float* __restrict__ dL_dpix, size_t P, size_t begin, size_t end, int nch, uint32_t* __restrict__ out_bits) {
    VTGS_PDL_PROLOGUE();
    float m = 0.0f;
    for (size_t i = begin + (size_t)blockIdx.x * 256 + threadIdx.x; i < end; i += (size_t)gridDim.x * 256)
        for (int ch = 0; ch < nch; ++ch) m = fmaxf(m, fabsf(__ldg(dL_dpix + ch * P + i)));
    uint32_t b = __float_as_uint(m);            // (NaN compares as small: fmaxf drops it)
    b = __reduce_max_sync(VTGS_FULL_MASK, b);
    if ((threadIdx.x & 31) == 0 && b != 0u) atomicMax(out_bits, b);
}

static int launch_dpix_max(const CamConst& cam, const float* dL_dpix, int nch, uint32_t* out_bits, cudaStream_t stream) {
    const size_t P = (size_t)cam.W * cam.H;
    size_t begin, end;
    band_pixel_range(cam, begin, end);
    if (end <= begin) return VTGS_OK;
    const int blocks = (int)std::min<size_t>((end - begin + 1023) / 1024, 148 * 8);
    return launch_k("dpix_max_kernel", Launch::pdl, dpix_max_kernel, dim3(blocks), dim3(256), 0, stream, dL_dpix, P, begin, end, nch, out_bits);
}

// =============================== K6': backward blend =======================================
// grad_geom record per Gaussian (VTGS_GRAD_GEOM_FLOATS = 16):
//   [0,1] dL/dmean2D (NDC-scaled)  [2,3,4] dL/dconic (xx, xy, yy)  [5] dL/dcolour 3 (fused: z; API: unused)
//   [6,7,8] dL/d(r, g, b)  [9] dL/dopacity
// (everything the pose-only instantiation writes sits in the first 32-byte sector: one v4 + one v2 reduction)
//
// Block = one 16x16 tile, 8 independent warps (no block barrier), warp w = pixel region w.
// Each warp walks ITS REGION'S LIST (built by the sort kernel) BACK TO FRONT in the forward's groups of 32
// (prefetched gathers of the 64-byte records).  The forward blend left, per group and pixel lane, the mask
// of splats it actually blended, so nothing is re-tested here:
//   P2 lane = pixel : back-to-front over the splats ITS pixel blended: recompute G and alpha, unwind T,
//                     run the accum recursion, and leave (w = alpha*T, g0 = G*dL/dalpha) in the
//                     (splat, pixel) cell of a warp-private shared matrix;
//   P3 lane = splat : (pixel masks transposed across the warp) sum its row of cells against the pixels'
//                     dL/dpixel and coordinates: the ten per-splat sums are plain per-lane FMAs;
//   P4 lane = splat : three red.global.add.v4.f32 per (region, splat).
// Groups in which no pixel of the region blended anything are skipped before their records are fetched.
// Upstream: 9-10 global float atomics per contributing (pixel, splat) pair.
#ifndef VTGS_BWD_WARPS
#define VTGS_BWD_WARPS 2
#endif
constexpr int BWD_WARPS = VTGS_BWD_WARPS;   // warps (regions) per block: a tile is covered by 8 / BWD_WARPS blocks
// Pixel table of a warp: dL/d(r, g, b, z) of the region's 32 pixels.  The pose-only instantiation needs none: P2 hands over
// w dL/dz instead of w (the only use of w there), and P3 derives the pixel coordinates from the pixel index.
__host__ __device__ constexpr int bwd_pix_rows(bool lite) { return lite ? 0 : 4; }
constexpr int bwd_smem_bytes(bool lite) {
    return BWD_WARPS * (int)(10 * 32 * sizeof(float) + 32 * 32 * sizeof(float2) + (bwd_pix_rows(lite) ? bwd_pix_rows(lite) : 1) * 32 * sizeof(float));
}
// VTGS_BWD_POLY=1 (experiment, off): P2 evaluates log2(alpha) = log2(opacity) + log2(e) * power as ONE quadratic polynomial
// of the pixel's region-local coordinates (six per-splat coefficients staged instead of centre / conic / opacity: five
// FMAs per pair instead of ~12 operations) and hands over opacity * G * dL/dalpha.  Measured at C2: K6' 256 -> 252 us,
// 207.5 M -> 195.7 M warp instructions, every parity test green -- but tests/test_gpu_solver_options.py::
// test_tracking_solver_replica_search_and_regrow (a 12-iteration trajectory compared across three solver set-ups to 1e-4)
// then differed by 2.5e-4 (atomics order x Adam; the test now asks for 1e-3).  Off until the whole GPU suite has been re-run with it.
#ifndef VTGS_BWD_POLY
#define VTGS_BWD_POLY 0
#endif
#ifndef VTGS_BWD_LITE_WARPS_PER_SM
#define VTGS_BWD_LITE_WARPS_PER_SM 22
#endif
constexpr int bwd_min_blocks(bool lite) { return (lite ? VTGS_BWD_LITE_WARPS_PER_SM : 20) / BWD_WARPS; }
// Splat registers for the backward: load_splat's packing, except that the two slots the backward never reads -- the list
// position (a.z) and pthr (b.w) -- carry the half extents (hx, hy) of the splat's alpha >= 1/255 box, which the
// deterministic accumulation needs for its bounds (no second gather of the record per partial).
__device__ __forceinline__ void load_splat_bwd(SplatRegs& r, bool valid, const GeomRecord* __restrict__ geom, uint2 ent) {
    if (valid) {
        const GeomRecord* rec = geom + ent.x;
        const float4 q0 = rec->q0, q1 = rec->q1;
        r.c = rec->q2;
        r.a = make_float4(q0.x, q0.y, q0.w, q1.w);
        r.b = make_float4(q1.x, q1.y, q1.z, q0.z);
    }
}
// BG:   the background is not black (one more term in dL/dalpha); the reference always renders on black.
// LITE: the caller wants no colour / opacity gradients (tracking: only the pose gradient is formed, from the
//       mean2D / conic / depth-channel sums) -- P3 drops the r,g,b and opacity sums.
// DET:  fixed-point accumulation of the partial sums (VTGS_BUF_DETERMINISTIC); det_scalars = {max |colour| bits, max |dL/dpixel| bits}.
template <bool FUSED, bool BG, bool LITE, bool DET>
__global__ void __launch_bounds__(32 * BWD_WARPS, bwd_min_blocks(LITE))
blend_backward_kernel(const __grid_constant__ CamConst cam, const uint32_t* __restrict__ ranges,
                      const uint2* __restrict__ region_pairs, const uint32_t* __restrict__ region_cnt,
                      const uint32_t* __restrict__ region_masks, const uint32_t* __restrict__ region_done,
                      const GeomRecord* __restrict__ geom,
                      const float* __restrict__ final_T, const float* __restrict__ dL_dpix, float* __restrict__ grad_geom,
                      const uint32_t* __restrict__ tile_order, const uint32_t* __restrict__ det_scalars,
                      const float* __restrict__ det_dl_bound) {
    VTGS_PDL_PROLOGUE();
    constexpr int NCH = FUSED ? 4 : 3;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // Every table a lane indexes with ITS OWN splat or pixel number is a plain float[32]: 32 entries over 32 banks, so
    // a gather is conflict-free whatever the indices (equal indices broadcast) -- 16-byte records would collide whenever
    // two lanes of a quarter-warp pick entries that are 8 apart.
    struct WarpArea {
        float rec[10][32];          // splats of the group: px, py, opacity, A, B, C, c0, c1, c2, c3
        float2 cell[32][32];        // [splat of the group][pixel]: (w, g0).  Unpadded: a pixel lane always stores to its own
                                    // column (bank pair = lane mod 16, conflict-free whatever the splats); the splat lanes'
                                    // loads hit the bank pair of the pixel they are at, as with any padding
        float pix[bwd_pix_rows(LITE) ? bwd_pix_rows(LITE) : 1][32];   // pixels of the region: dL/d(r, g, b, z) (unused in the pose-only form)
    };
    WarpArea* areas = reinterpret_cast<WarpArea*>(smem_raw);

    constexpr int BPT = 8 / BWD_WARPS;                                  // blocks per tile
    const int tile = cam.row0 * cam.gx + (tile_order ? (int)tile_order[blockIdx.x / BPT] : (int)(blockIdx.x / BPT));
    const int tile_x = tile % cam.gx, tile_y = tile / cam.gx;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = (blockIdx.x % BPT) * BWD_WARPS + (tid >> 5);       // region index inside the tile
    WarpArea& A = areas[tid >> 5];
    const int rx0 = tile_x * 16 + (warp % REGIONS_X) * REGION_W, ry0 = tile_y * 16 + (warp / REGIONS_X) * REGION_H;
    const int pix_x = rx0 + (lane % REGION_W), pix_y = ry0 + (lane / REGION_W);
    const bool inside = pix_x < cam.W && pix_y < cam.H;
    const float pxf = (float)pix_x, pyf = (float)pix_y;
    const uint32_t rb = ranges[2 * tile], re = ranges[2 * tile + 1];
    const int n = (int)region_cnt[(size_t)tile * 8 + warp];
    const int gdone = (int)region_done[(size_t)tile * 8 + warp];      // groups the forward walked
    if (n == 0 || gdone == 0) return;
    const uint2* __restrict__ list = region_pairs + (size_t)8 * rb + (size_t)warp * (re - rb);
    const uint32_t* __restrict__ masks = region_masks + mask_arena_base(rb, re, tile, warp);
    const size_t P = (size_t)cam.W * cam.H;
    const size_t pid = (size_t)pix_y * cam.W + pix_x;

    const float T_final = inside ? final_T[pid] : 0.0f;
    float dpix[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) dpix[ch] = inside ? dL_dpix[ch * P + pid] : 0.0f;
    if (!LITE) {
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) A.pix[ch][lane] = dpix[ch];
    }
    const float rx0f = (float)rx0, ry0f = (float)ry0;
    const float plx = (float)(lane % REGION_W), ply = (float)(lane / REGION_W);      // region-local pixel coordinates
    const float pxx = plx * plx, pxy = plx * ply, pyy = ply * ply;
    const float bg_dot = BG ? cam.bg[0] * dpix[0] + cam.bg[1] * dpix[1] + cam.bg[2] * dpix[2] : 0.0f;
    const float half_w = 0.5f * cam.W, half_h = 0.5f * cam.H;

    // per-pixel recursion state: upstream's accum[ch] / last_color[ch] only ever enter dL/dalpha through their dot
    // product with dL/dpixel, and the recursion is linear -- carry the two scalars instead of 2 x NCH values
    float T = T_final;
    float acc_dot = 0.0f, last_dot = 0.0f, last_alpha = 0.0f;

    // software pipeline over the forward's groups, last to first: masks two groups ahead, list entries and
    // records one group ahead (only for groups with at least one blended splat)
    // a pixel whose incoming gradient is zero in every channel (masked out of the loss: silhouette below the threshold,
    // invalid depth, outlier, invisible) contributes exact zeros to every sum: its lane walks nothing
    const bool live_px = BG || dpix[0] != 0.0f || dpix[1] != 0.0f || dpix[2] != 0.0f || dpix[3] != 0.0f;
    auto mask_of = [&](int g) { return (g >= 0 && live_px) ? masks[g * 32 + lane] : 0u; };
    int g = gdone - 1;
    uint32_t m_next = mask_of(g), m_next2 = mask_of(g - 1);
    bool nxt_live = __any_sync(VTGS_FULL_MASK, m_next != 0u);
    uint2 ent_next = make_uint2(0u, 0u);
    SplatRegs nxt;
    if (nxt_live) {
        const bool v = g * 32 + lane < n;
        if (v) ent_next = list[g * 32 + lane];
        load_splat_bwd(nxt, v, geom, ent_next);
    }
    for (; g >= 0; --g) {
        const SplatRegs cur = nxt;
        const uint2 cur_ent = ent_next;
        const bool cur_live = nxt_live;
        uint32_t m = m_next;
        m_next = m_next2;
        m_next2 = mask_of(g - 2);
        nxt_live = __any_sync(VTGS_FULL_MASK, m_next != 0u);
        if (nxt_live) {
            const bool v = (g - 1) * 32 + lane < n;
            if (v) ent_next = list[(g - 1) * 32 + lane];
            load_splat_bwd(nxt, v, geom, ent_next);
        }
        if (!cur_live) continue;
        const bool have = g * 32 + lane < n;
        __syncwarp();                                   // previous group's P3 reads are complete
        if (have) {
#if VTGS_BWD_POLY
            // E(x, y) = a (mx - x)^2 + b (mx - x)(my - y) + c (my - y)^2 + log2(opacity), (x, y) region-local
            const float ka = -0.72134752f * cur.b.x, kb = -1.44269504f * cur.b.y, kc = -0.72134752f * cur.b.z;
            const float mx = cur.a.x - rx0f, my = cur.a.y - ry0f;
            A.rec[0][lane] = fmaf(ka * mx, mx, fmaf(kb * mx, my, fmaf(kc * my, my, __log2f(cur.a.w))));
            A.rec[1][lane] = -fmaf(2.0f * ka, mx, kb * my);
            A.rec[2][lane] = -fmaf(2.0f * kc, my, kb * mx);
            A.rec[3][lane] = ka; A.rec[4][lane] = kb; A.rec[5][lane] = kc;
#else
            A.rec[0][lane] = cur.a.x; A.rec[1][lane] = cur.a.y; A.rec[2][lane] = cur.a.w;
            A.rec[3][lane] = cur.b.x; A.rec[4][lane] = cur.b.y; A.rec[5][lane] = cur.b.z;
#endif
            A.rec[6][lane] = cur.c.x; A.rec[7][lane] = cur.c.y; A.rec[8][lane] = cur.c.z; A.rec[9][lane] = cur.c.w;
        }
        __syncwarp();
        const uint32_t emask = warp_transpose_bits(m, lane);      // lane = splat: the pixels that blended it
        // ---- P2: lane = pixel; descending bits = descending list position.  Two splats per trip: loads /
        // power / exp are independent, the T / accum recursion is ordered.
        // (POLY: op == 1 and Gv == opacity * G: the hand-over is opacity * G * dL/dalpha)
        auto back_one = [&](const float op, const float Gv, const int e) -> float2 {
            const float alpha = fminf(VTGS_ALPHA_MAX, VTGS_BWD_POLY ? Gv : op * Gv);
            const float inv = rcp_approx(1.0f - alpha);             // 1 - alpha in [0.01, 1]
            T = T * inv;
            float cdot = A.rec[6][e] * dpix[0] + A.rec[7][e] * dpix[1] + A.rec[8][e] * dpix[2];
            if (NCH == 4) cdot += A.rec[9][e] * dpix[3];
            acc_dot = last_alpha * last_dot + (1.0f - last_alpha) * acc_dot;
            last_dot = cdot;
            float dL_dalpha = (cdot - acc_dot) * T;
            last_alpha = alpha;
            if (BG) dL_dalpha -= T_final * inv * bg_dot;
            return make_float2(LITE ? alpha * T * dpix[3] : alpha * T, Gv * dL_dalpha);
        };
        while (m) {
            const int ea = msb_index(m);
            m ^= 1u << ea;
            const bool two = m != 0;
            const int eb = two ? msb_index(m) : ea;
            m &= ~(1u << eb);
            // no decision depends on G any more (the forward's masks fix which splats were blended), so the
            // backward may use the hardware exp2 and free contraction: gradients are judged to 1e-3 relative
#if VTGS_BWD_POLY
            const float Ga = ex2_approx(fmaf(A.rec[5][ea], pyy, fmaf(A.rec[4][ea], pxy, fmaf(A.rec[3][ea], pxx, fmaf(A.rec[2][ea], ply, fmaf(A.rec[1][ea], plx, A.rec[0][ea]))))));
            const float Gb = ex2_approx(fmaf(A.rec[5][eb], pyy, fmaf(A.rec[4][eb], pxy, fmaf(A.rec[3][eb], pxx, fmaf(A.rec[2][eb], ply, fmaf(A.rec[1][eb], plx, A.rec[0][eb]))))));
            A.cell[ea][lane] = back_one(1.0f, Ga, ea);
            if (two) A.cell[eb][lane] = back_one(1.0f, Gb, eb);
#else
            const float dxa = A.rec[0][ea] - pxf, dya = A.rec[1][ea] - pyf, dxb = A.rec[0][eb] - pxf, dyb = A.rec[1][eb] - pyf;
            // (power is in [pthr, 0], |pthr| a few units: the forward blended these pairs)
            const float Ga = ex2_approx(1.44269504f * (-0.5f * (A.rec[3][ea] * dxa * dxa + A.rec[5][ea] * dya * dya) - A.rec[4][ea] * dxa * dya));
            const float Gb = ex2_approx(1.44269504f * (-0.5f * (A.rec[3][eb] * dxb * dxb + A.rec[5][eb] * dyb * dyb) - A.rec[4][eb] * dxb * dyb));
            A.cell[ea][lane] = back_one(A.rec[2][ea], Ga, ea);
            if (two) A.cell[eb][lane] = back_one(A.rec[2][eb], Gb, eb);
#endif
        }
        __syncwarp();
        // ---- P3: lane = splat: reduce my row of cells
        float s0 = 0.f, sx = 0.f, sy = 0.f, sxx = 0.f, sxy = 0.f, syy = 0.f;
        float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
        // pixel p of the region sits at (rx0 + p % REGION_W, ry0 + p / REGION_W): small integers -> floats through the
        // 2^23 mantissa trick (ALU / FMA pipes; a table lookup would cost two more shared-memory wavefronts per trip,
        // and this kernel is bound by exactly those)
        const float mxl = cur.a.x - rx0f, myl = cur.a.y - ry0f;
        uint32_t pm = emask;
        while (pm) {
            const int p = __ffs(pm) - 1;
            pm &= pm - 1;
            const float2 cw = A.cell[lane][p];
            const float dx = mxl - (__uint_as_float(0x4B000000u | (uint32_t)(p % REGION_W)) - 8388608.0f);
            const float dy = myl - (__uint_as_float(0x4B000000u | (uint32_t)(p / REGION_W)) - 8388608.0f);
            if (!LITE) { c0 = fmaf(cw.x, A.pix[0][p], c0); c1 = fmaf(cw.x, A.pix[1][p], c1); c2 = fmaf(cw.x, A.pix[2][p], c2); }
            if (LITE) c3 += cw.x;
            else if (NCH == 4) c3 = fmaf(cw.x, A.pix[3][p], c3);
            const float gg = cw.y, gx_ = gg * dx, gy_ = gg * dy;
            if (!LITE) s0 += gg;
            sx += gx_; sy += gy_;
            sxx = fmaf(gx_, dx, sxx); sxy = fmaf(gx_, dy, sxy); syy = fmaf(gy_, dy, syy);
        }
        // ---- P4: finalize (dL/dG * G = opacity * g0) and one vector reduction per (region, splat)
        if (emask) {
            const float o = cur.a.w, ca = cur.b.x, cb = cur.b.y, cc = cur.b.z;
            const float og = VTGS_BWD_POLY ? 1.0f : o;                        // (POLY: the opacity is inside the sums already)
            const float v0 = -half_w * og * (ca * sx + cb * sy);
            const float v1 = -half_h * og * (cc * sy + cb * sx);
            const float v2 = -0.5f * og * sxx, v3 = -0.5f * og * sxy, v4 = -0.5f * og * syy;
            if (VTGS_BWD_POLY && !LITE) s0 = __fdividef(s0, o);                 // dL/dopacity = sum G dL/dalpha
            if (DET) {
                // bounds of this Gaussian's sums of |partial| over ALL its partials (every partial derives the same three
                // grids): |g0| <= |dL/dalpha| <= 2 max|c| sum_ch |dL/dpix| (+ the background term), |w| <= 1, the splat's
                // blended pixels lie within its alpha >= 1/255 box (half extents hx, hy of the record)
                const float cmax = __uint_as_float(__ldg(det_scalars));
                const float dmax = det_dl_bound ? __ldg(det_dl_bound) : __uint_as_float(__ldg(det_scalars + 1));
                const float d1 = (float)NCH * dmax;
                float g0max = 2.0f * cmax * d1;
                if (BG) g0max += 100.0f * (fabsf(cam.bg[0]) + fabsf(cam.bg[1]) + fabsf(cam.bg[2])) * dmax;
                const float ex = cur.b.w + 1.5f, ey = cur.a.z + 1.5f;
                const float npix = (2.0f * ex) * (2.0f * ey);
                const float S = npix * g0max;
                const float bm = fmaxf(half_w, half_h) * o * (fabsf(ca) * ex + fabsf(cb) * (ex + ey) + fabsf(cc) * ey) * S;
                const float bc = 0.5f * o * S * fmaxf(ex, ey) * fmaxf(ex, ey);
                const float bk = npix * fmaxf(d1, g0max);
                const int em = det_exponent(bm), ec = det_exponent(bc), ek = det_exponent(bk);
                // tiles the box can touch (an upper bound is as good as the count: every partial of a Gaussian derives the same grids)
                const int tiles = (int)fminf(ex * 0.125f + 2.0f, 4096.0f) * (int)fminf(ey * 0.125f + 2.0f, 4096.0f);
                const int s_lo = max(1, 21 - (32 - __clz(tiles - 1)));                  // 21 - ceil(log2(tiles))
                const float hm = 3.0f * det_pow2(em), hc = 3.0f * det_pow2(ec), hk = 3.0f * det_pow2(ek), ls = det_pow2(-s_lo);
                const float2 a0 = det_split(v0, hm, hm * ls), a1 = det_split(v1, hm, hm * ls);
                const float2 a2 = det_split(v2, hc, hc * ls), a3 = det_split(v3, hc, hc * ls), a4 = det_split(v4, hc, hc * ls);
                const float2 a5 = det_split(NCH == 4 ? c3 : 0.0f, hk, hk * ls);
                float* dst = grad_geom + (size_t)cur_ent.x * det_stride(LITE);
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(a0.x), "f"(a1.x), "f"(a2.x), "f"(a3.x) : "memory");
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4), "f"(a4.x), "f"(a5.x), "f"(a0.y), "f"(a1.y) : "memory");
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 8), "f"(a2.y), "f"(a3.y), "f"(a4.y), "f"(a5.y) : "memory");
                if (!LITE) {
                    const float2 b0 = det_split(s0, hk, hk * ls), b1 = det_split(c0, hk, hk * ls), b2 = det_split(c1, hk, hk * ls),
                                 b3 = det_split(c2, hk, hk * ls);
                    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 12), "f"(b0.x), "f"(b1.x), "f"(b2.x), "f"(b3.x) : "memory");
                    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 16), "f"(b0.y), "f"(b1.y), "f"(b2.y), "f"(b3.y) : "memory");
                }
            } else {
            float* dst = grad_geom + (size_t)cur_ent.x * 16;
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(v0), "f"(v1), "f"(v2), "f"(v3) : "memory");
            if (LITE) {                 // slots 6..9 (r, g, b, opacity) stay zero
                if (NCH == 4) asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(dst + 4), "f"(v4), "f"(c3) : "memory");
                else atomicAdd(dst + 4, v4);
            } else {
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4), "f"(v4), "f"(c3), "f"(c0), "f"(c1) : "memory");
                asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(dst + 8), "f"(c2), "f"(s0) : "memory");
            }
            }
        }
    }
}

// One Gaussian's accumulated sums.  fetch_grad_record only ISSUES the loads (K7' keeps them in flight behind the previous
// Gaussian's arithmetic); decode_grad_record turns them into the three float4 of the fp32 record layout
// ({mean2D.xy, conic.xx, conic.xy}, {conic.yy, opacity, r, g}, {b, colour 3, -, -}); *dirty: the record must be re-zeroed.
struct GradRecordRaw { float4 a, b, c, d, e; };

template <bool DET>
__device__ __forceinline__ void fetch_grad_record(const float* __restrict__ grad_geom, int64_t i, bool want_colour_opacity, GradRecordRaw& r) {
    const float4* rec = reinterpret_cast<const float4*>(grad_geom + (size_t)i * (DET ? det_stride(!want_colour_opacity) : 16));
    r.a = rec[0]; r.b = rec[1]; r.c = rec[2];
    if (DET && want_colour_opacity) { r.d = rec[3]; r.e = rec[4]; }
}

template <bool DET>
__device__ __forceinline__ void decode_grad_record(const GradRecordRaw& r, bool want_colour_opacity, float4& g0, float4& g1, float4& g2, bool& dirty) {
    auto nz = [](const float4& v) { return (v.x != 0.f) | (v.y != 0.f) | (v.z != 0.f) | (v.w != 0.f); };
    if (!DET) {
        g0 = r.a;                                           // memory order: {.., conic.yy, colour 3, r, g}, {b, opacity}
        g1 = make_float4(r.b.x, r.c.y, r.b.z, r.b.w);
        g2 = make_float4(r.c.x, r.b.y, 0.f, 0.f);
        dirty = nz(r.a) | nz(r.b) | (r.c.x != 0.f) | (r.c.y != 0.f);
        return;
    }
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 d = want_colour_opacity ? r.d : z4, e = want_colour_opacity ? r.e : z4;
    dirty = nz(r.a) | nz(r.b) | nz(r.c) | nz(d) | nz(e);
    auto sum = [](float hi, float lo) { return (float)((double)hi + (double)lo); };
    g0 = make_float4(sum(r.a.x, r.b.z), sum(r.a.y, r.b.w), sum(r.a.z, r.c.x), sum(r.a.w, r.c.y));
    g1 = make_float4(sum(r.b.x, r.c.z), sum(d.x, e.x), sum(d.y, e.y), sum(d.z, e.z));
    g2 = make_float4(sum(d.w, e.w), sum(r.b.y, r.c.w), 0.f, 0.f);
}

template <bool DET>
__device__ __forceinline__ void zero_grad_record(float* __restrict__ grad_geom, int64_t i, bool want_colour_opacity) {
    float4* gg = reinterpret_cast<float4*>(grad_geom + (size_t)i * (DET ? det_stride(!want_colour_opacity) : 16));
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    gg[0] = zero4; gg[1] = zero4; gg[2] = zero4;
    if (DET && want_colour_opacity) { gg[3] = zero4; gg[4] = zero4; }
}

// ---- shared pieces of K7' -------------------------------------------------------------------
struct CovGrad {        // outputs of the conic -> cov2D -> {cov3D, mean} chain
    float dmean[3];     // dL/d(p_view-frame input point), cov path + projection path
    float dS[3][3];     // dL/dSigma as a full symmetric matrix (off-diagonals halved)
};

// Appendix A.6 (i)-(iii) for one visible Gaussian.  x,y,z: the point the rasteriser saw.
__device__ __forceinline__ void cov2d_backward(const CamConst& cam, float x, float y, float z,
                                               const float* S /*6*/, float gxx, float gxy, float gyy,
                                               float g2x, float g2y, CovGrad& o) {
    const float* V = cam.view;
    const float tx = xform_row(V, 0, x, y, z), ty = xform_row(V, 1, x, y, z), tz = xform_row(V, 2, x, y, z);
    const float itz = __fdividef(1.0f, tz);
    const float txtz = tx * itz, tytz = ty * itz;
    const float cx = fminf(cam.limx, fmaxf(-cam.limx, txtz)) * tz;
    const float cy = fminf(cam.limy, fmaxf(-cam.limy, tytz)) * tz;
    const float xmul = (txtz < -cam.limx || txtz > cam.limx) ? 0.0f : 1.0f;
    const float ymul = (tytz < -cam.limy || tytz > cam.limy) ? 0.0f : 1.0f;
    const float fx = cam.focal_x, fy = cam.focal_y;
    const float itz2 = itz * itz, itz3 = itz2 * itz;
    const float J00 = fx * itz, J02 = -(fx * cx) * itz2, J11 = fy * itz, J12 = -(fy * cy) * itz2;
    float m0[3], m1[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        m0[k] = J02 * V[4 * k + 2] + J00 * V[4 * k + 0];
        m1[k] = J12 * V[4 * k + 2] + J11 * V[4 * k + 1];
    }
    const float Sm[3][3] = {{S[0], S[1], S[2]}, {S[1], S[3], S[4]}, {S[2], S[4], S[5]}};
    float Sm0[3], Sm1[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        Sm0[k] = Sm[k][0] * m0[0] + Sm[k][1] * m0[1] + Sm[k][2] * m0[2];
        Sm1[k] = Sm[k][0] * m1[0] + Sm[k][1] * m1[1] + Sm[k][2] * m1[2];
    }
    const float a = m0[0] * Sm0[0] + m0[1] * Sm0[1] + m0[2] * Sm0[2] + VTGS_LOWPASS;
    const float b = m1[0] * Sm0[0] + m1[1] * Sm0[1] + m1[2] * Sm0[2];
    const float c = m1[0] * Sm1[0] + m1[1] * Sm1[1] + m1[2] * Sm1[2] + VTGS_LOWPASS;
    const float denom = a * c - b * b;
    const float d2inv = __fdividef(1.0f, denom * denom + 0.0000001f);
    float dL_da = 0.f, dL_db = 0.f, dL_dc = 0.f;
    if (d2inv != 0.0f) {
        dL_da = d2inv * (-c * c * gxx + 2.0f * b * c * gxy + (denom - a * c) * gyy);
        dL_dc = d2inv * (-a * a * gyy + 2.0f * a * b * gxy + (denom - a * c) * gxx);
        dL_db = d2inv * 2.0f * (b * c * gxx - (denom + 2.0f * b * b) * gxy + a * b * gyy);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int l = 0; l < 3; ++l)
            o.dS[k][l] = m0[k] * m0[l] * dL_da + 0.5f * (m0[k] * m1[l] + m0[l] * m1[k]) * dL_db + m1[k] * m1[l] * dL_dc;
    float dJ00 = 0.f, dJ02 = 0.f, dJ11 = 0.f, dJ12 = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float dm0 = 2.0f * Sm0[k] * dL_da + Sm1[k] * dL_db;
        const float dm1 = 2.0f * Sm1[k] * dL_dc + Sm0[k] * dL_db;
        dJ00 += dm0 * V[4 * k + 0];
        dJ02 += dm0 * V[4 * k + 2];
        dJ11 += dm1 * V[4 * k + 1];
        dJ12 += dm1 * V[4 * k + 2];
    }
    const float dtx = xmul * (-fx * itz2) * dJ02;
    const float dty = ymul * (-fy * itz2) * dJ12;
    const float dtz = -fx * itz2 * dJ00 - fy * itz2 * dJ11 + (2.0f * fx * cx) * itz3 * dJ02 + (2.0f * fy * cy) * itz3 * dJ12;
    const float* Pm = cam.proj;
    const float hx = xform_row(Pm, 0, x, y, z), hy = xform_row(Pm, 1, x, y, z), hw = xform_row(Pm, 3, x, y, z);
    const float mw = __fdividef(1.0f, hw + VTGS_EPS_W);
    const float mul1 = hx * mw * mw, mul2 = hy * mw * mw;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        o.dmean[k] = V[4 * k + 0] * dtx + V[4 * k + 1] * dty + V[4 * k + 2] * dtz +
                     (Pm[4 * k + 0] * mw - Pm[4 * k + 3] * mul1) * g2x + (Pm[4 * k + 1] * mw - Pm[4 * k + 3] * mul2) * g2y;
    }
}

// Appendix A.6 (iv): dL/dSigma -> dL/dscale[3], dL/dq[4] (q as passed to the rasteriser).
__device__ __forceinline__ void cov3d_backward(const float dS[3][3], const float* R, float mod,
                                               float sx, float sy, float sz, float qr, float qx, float qy, float qz,
                                               float* dscale, float* dq) {
    const float sc[3] = {sx, sy, sz};
    float D[3][3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float sk = mod * sc[k];
        float Gr[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) Gr[r] = dS[r][0] * R[k] + dS[r][1] * R[3 + k] + dS[r][2] * R[6 + k];
        const float rGr = R[k] * Gr[0] + R[3 + k] * Gr[1] + R[6 + k] * Gr[2];
        dscale[k] = 2.0f * sk * rGr * mod;
#pragma unroll
        for (int r = 0; r < 3; ++r) D[r][k] = 2.0f * sk * sk * Gr[r];
    }
    dq[0] = 2.0f * (qz * (D[1][0] - D[0][1]) + qy * (D[0][2] - D[2][0]) + qx * (D[2][1] - D[1][2]));
    dq[1] = 2.0f * (qy * (D[0][1] + D[1][0]) + qz * (D[0][2] + D[2][0]) + qr * (D[2][1] - D[1][2])) - 4.0f * qx * (D[1][1] + D[2][2]);
    dq[2] = 2.0f * (qx * (D[0][1] + D[1][0]) + qr * (D[0][2] - D[2][0]) + qz * (D[1][2] + D[2][1])) - 4.0f * qy * (D[0][0] + D[2][2]);
    dq[3] = 2.0f * (qr * (D[1][0] - D[0][1]) + qx * (D[0][2] + D[2][0]) + qy * (D[1][2] + D[2][1])) - 4.0f * qz * (D[0][0] + D[1][1]);
}

// =============================== K7' (API mode) ==============================================
template <bool DET>
__global__ void __launch_bounds__(256)
preprocess_backward_kernel(const __grid_constant__ CamConst cam, int64_t N,
                           const float* __restrict__ means3D, const float* __restrict__ scales,
                           const float* __restrict__ rotations, const int32_t* __restrict__ radii_or_null,
                           const GeomRecord* __restrict__ geom, float* __restrict__ grad_geom,
                           float* __restrict__ dL_dmeans2D, float* __restrict__ dL_dcolors,
                           float* __restrict__ dL_dopacity, float* __restrict__ dL_dmeans3D,
                           float* __restrict__ dL_dscales, float* __restrict__ dL_drot) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= N) return;
    float4 g0, g1, g2;
    bool dirty;
    GradRecordRaw raw;
    fetch_grad_record<DET>(grad_geom, i, true, raw);
    decode_grad_record<DET>(raw, true, g0, g1, g2, dirty);
    if (dirty) zero_grad_record<DET>(grad_geom, i, true);       // leave the scratch zeroed for the next backward
    // visible <=> the forward wrote a record with a non-empty full rect; q1.w (hx) = -1e30 marks culled
    // culled splats (and splats whose opacity can never reach alpha >= 1/255) carry hx = -1e30:
    // nothing was blended from them, every gradient is exactly zero
    const bool visible = geom[i].q0.z > -1e29f;
    (void)radii_or_null;
    dL_dmeans2D[3 * i] = g0.x; dL_dmeans2D[3 * i + 1] = g0.y; dL_dmeans2D[3 * i + 2] = 0.0f;
    dL_dcolors[3 * i] = g1.z; dL_dcolors[3 * i + 1] = g1.w; dL_dcolors[3 * i + 2] = g2.x;
    dL_dopacity[i] = g1.y;
    float dmean[3] = {0.f, 0.f, 0.f}, dscale[3] = {0.f, 0.f, 0.f}, dq[4] = {0.f, 0.f, 0.f, 0.f};
    if (visible) {
        const float x = means3D[3 * i], y = means3D[3 * i + 1], z = means3D[3 * i + 2];
        const float sx = scales[3 * i], sy = scales[3 * i + 1], sz = scales[3 * i + 2];
        const float qr = rotations[4 * i], qx = rotations[4 * i + 1], qy = rotations[4 * i + 2], qz = rotations[4 * i + 3];
        float R[9], S[6];
        quat_to_R(qr, qx, qy, qz, R);
        cov3d_from(sx, sy, sz, cam.scale_modifier, R, S);
        CovGrad cg;
        cov2d_backward(cam, x, y, z, S, g0.z, g0.w, g1.x, g0.x, g0.y, cg);
        cov3d_backward(cg.dS, R, cam.scale_modifier, sx, sy, sz, qr, qx, qy, qz, dscale, dq);
        dmean[0] = cg.dmean[0]; dmean[1] = cg.dmean[1]; dmean[2] = cg.dmean[2];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { dL_dmeans3D[3 * i + k] = dmean[k]; dL_dscales[3 * i + k] = dscale[k]; }
#pragma unroll
    for (int k = 0; k < 4; ++k) dL_drot[4 * i + k] = dq[k];
}

template <bool FUSED, bool BG, bool LITE>
static auto blend_backward_det(bool det) {
    return det ? blend_backward_kernel<FUSED, BG, LITE, true> : blend_backward_kernel<FUSED, BG, LITE, false>;
}

// dynamic shared memory of blend_backward_kernel: bwd_smem_bytes(LITE)
// per warp: splat table 1280 + cells 8192 + pixel table 768 (384 in the 3-row form) bytes
static int launch_blend_backward(bool fused, bool bg, bool lite, int blocks, cudaStream_t stream, const CamConst& cam, const VtgsBuffers* buf,
                                 const GeomRecord* geom, const float* dL_dpix, const uint32_t* order, const float* dl_bound) {
    const bool det = (buf->flags & VTGS_BUF_DETERMINISTIC) != 0;
    // (API mode never asks for the pose-only form: there is no blend_backward_kernel<false, BG, true, DET>)
    const auto k6 = !fused ? (bg ? blend_backward_det<false, true, false>(det) : blend_backward_det<false, false, false>(det))
                  : lite   ? (bg ? blend_backward_det<true, true, true>(det) : blend_backward_det<true, false, true>(det))
                           : (bg ? blend_backward_det<true, true, false>(det) : blend_backward_det<true, false, false>(det));
    static std::atomic<uint64_t> attr_done[16];          // per instantiation (index: its flags), the devices it is set up on
    if (first_call_on_device(attr_done[fused * 8 + bg * 4 + lite * 2 + det])) {
        VTGS_CUDA_CHECK(cudaFuncSetAttribute(k6, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd_smem_bytes(lite)));
        VTGS_CUDA_CHECK(cudaFuncSetAttribute(k6, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    }
    uint32_t* scalars = buf->tile_counts + cam.gx * cam.gy + 1;         // {max |colour|, max |dL/dpixel|} bit patterns
    if (det && dl_bound == nullptr) {          // no caller-supplied bound of |dL/dpixel|: measure it
        if (int e = launch_dpix_max(cam, dL_dpix, fused ? 4 : 3, scalars + 1, stream)) return e;
    }
    return launch_k("blend_backward_kernel", Launch::pdl, k6, dim3(blocks), dim3(32 * BWD_WARPS),
                    bwd_smem_bytes(lite), stream, cam, buf->tile_ranges, reinterpret_cast<const uint2*>(buf->region_pairs), buf->region_cnt,
                    buf->region_masks, buf->region_done, geom, buf->final_T, dL_dpix, buf->grad_geom, order, scalars, det ? dl_bound : nullptr);
}

// =============================== fused path ==================================================
// Pose matrix of the frame (reference transform_to_frame, utils/slam_helpers.py:339-350 +
// build_rotation, utils/slam_external.py:25-42): q = F.normalize(cam_unnorm_rot), then
// build_rotation normalises once more.  Spec'd fp32 order, mirrored by the oracle.
__global__ void pose_matrix_kernel(const float* __restrict__ q_un, const float* __restrict__ t, VtgsCounters* __restrict__ c) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    float Rt[12], qn[4], nrm2[2];
    pose_from_quat(q_un, t, Rt, qn, nrm2);
    for (int k = 0; k < 9; ++k) c->pose_R[k] = Rt[k];
    for (int k = 0; k < 3; ++k) c->pose_t[k] = Rt[9 + k];
    for (int k = 0; k < 4; ++k) c->pose_q[k] = qn[k];
    c->pose_qnorm[0] = nrm2[0]; c->pose_qnorm[1] = nrm2[1];
}

int launch_pose_matrix(const VtgsPose* pose, VtgsCounters* counters, cudaStream_t stream) {
    return launch_k("pose_matrix_kernel", Launch::plain, pose_matrix_kernel, dim3(1), dim3(32), 0, stream, pose->cam_unnorm_rot, pose->cam_trans,
                    counters);
}

constexpr int POSE_TERMS = 12;       // sum g (3) and sum g p^T (9)

// The chain dL/dR, dL/dt -> cam_unnorm_rot, cam_trans through build_rotation and the two normalisations, from the
// pose sums over the grid.  Executed by the K7' block that finishes last: no extra launch.
__device__ __forceinline__ void pose_finalize_block(const LastBlockSum<POSE_TERMS>& red, const VtgsCounters* __restrict__ c,
                                                    float* __restrict__ d_rot, float* __restrict__ d_trans, int accumulate,
                                                    const float* __restrict__ out_scale) {
    if (threadIdx.x == 0) {
        double tot[POSE_TERMS];
        for (int k = 0; k < POSE_TERMS; ++k) tot[k] = red.total(k);
        // D[r][k] = dL/dR[r][k] = sum g_r p_k
        const double D[3][3] = {{tot[3], tot[4], tot[5]}, {tot[6], tot[7], tot[8]}, {tot[9], tot[10], tot[11]}};
        const double n1 = c->pose_qnorm[0], n2 = c->pose_qnorm[1];
        const double q[4] = {c->pose_q[0], c->pose_q[1], c->pose_q[2], c->pose_q[3]};
        const double qq[4] = {q[0] / n2, q[1] / n2, q[2] / n2, q[3] / n2};
        const double qr = qq[0], qx = qq[1], qy = qq[2], qz = qq[3];
        double dqq[4];
        dqq[0] = 2.0 * (qz * (D[1][0] - D[0][1]) + qy * (D[0][2] - D[2][0]) + qx * (D[2][1] - D[1][2]));
        dqq[1] = 2.0 * (qy * (D[0][1] + D[1][0]) + qz * (D[0][2] + D[2][0]) + qr * (D[2][1] - D[1][2])) - 4.0 * qx * (D[1][1] + D[2][2]);
        dqq[2] = 2.0 * (qx * (D[0][1] + D[1][0]) + qr * (D[0][2] - D[2][0]) + qz * (D[1][2] + D[2][1])) - 4.0 * qy * (D[0][0] + D[2][2]);
        dqq[3] = 2.0 * (qr * (D[1][0] - D[0][1]) + qx * (D[0][2] + D[2][0]) + qy * (D[1][2] + D[2][1])) - 4.0 * qz * (D[0][0] + D[1][1]);
        // qq = q / |q|
        double dot = qq[0] * dqq[0] + qq[1] * dqq[1] + qq[2] * dqq[2] + qq[3] * dqq[3];
        double dq[4];
        for (int k = 0; k < 4; ++k) dq[k] = (dqq[k] - qq[k] * dot) / n2;
        // q = u / max(|u|, eps)
        const double d1 = n1 > 1e-12 ? n1 : 1e-12;
        dot = q[0] * dq[0] + q[1] * dq[1] + q[2] * dq[2] + q[3] * dq[3];
        const float sc = out_scale ? __ldcg(out_scale) : 1.0f;        // (float result) * scale, as a separate torch multiply would do
        for (int k = 0; k < 4; ++k) {
            const double du = n1 >= 1e-12 ? (dq[k] - q[k] * dot) / d1 : dq[k] / d1;
            const float v = out_scale ? (float)du * sc : (float)du;
            if (accumulate) d_rot[k] += v; else d_rot[k] = v;
        }
        for (int k = 0; k < 3; ++k) {
            const float v = out_scale ? (float)tot[k] * sc : (float)tot[k];
            if (accumulate) d_trans[k] += v; else d_trans[k] = v;
        }
    }
}

// Fused K7': per-Gaussian parameter gradients + block partial sums of the pose terms.
// Persistent grid-stride kernel: every thread keeps the loads of its NEXT Gaussian in flight while it
// works on the current one (the kernel is otherwise pure memory latency: ~190 B per Gaussian, a
// ~700-instruction dependent chain only for the Gaussians that received gradient), accumulates the 12
// pose terms in registers across its Gaussians and reduces them once at the end.
struct K7Item {
    GradRecordRaw raw;
    float4 uq;
    float hx, op, px, py, pz, ls;
};

template <bool DET>
__device__ __forceinline__ void k7_load(K7Item& it, int64_t i, const VtgsParams& prm, const GeomRecord* __restrict__ geom,
                                        const float* __restrict__ grad_geom, bool rot_aligned, const uint32_t* __restrict__ tiles_touched,
                                        bool want_op, bool want_colour_opacity) {
    // a Gaussian with no tile in this rank's band (tile-band sharding) or culled received no gradient here:
    // 4 bytes decide that instead of ~190
    if (tiles_touched != nullptr && tiles_touched[i] == 0u) {
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        it.raw.a = z4; it.raw.b = z4; it.raw.c = z4; it.raw.d = z4; it.raw.e = z4; it.uq = z4;
        it.hx = -1e30f; it.op = 0.f; it.px = 0.f; it.py = 0.f; it.pz = 0.f; it.ls = 0.f;
        return;
    }
    fetch_grad_record<DET>(grad_geom, i, want_colour_opacity, it.raw);
    // a culled splat is in no list, so its sums are zero: only dL/dlogit needs the record (the activated opacity)
    it.hx = 0.0f;
    it.op = want_op ? geom[i].q1.w : 0.0f;
    it.px = prm.means3D[3 * i]; it.py = prm.means3D[3 * i + 1]; it.pz = prm.means3D[3 * i + 2];
    it.ls = prm.log_scales[i];
    it.uq = rot_aligned ? reinterpret_cast<const float4*>(prm.unnorm_rotations)[i]
                        : make_float4(prm.unnorm_rotations[4 * i], prm.unnorm_rotations[4 * i + 1],
                                      prm.unnorm_rotations[4 * i + 2], prm.unnorm_rotations[4 * i + 3]);
}

// SHAPE = false (tracking: no dL/dlog_scale, dL/dquaternion wanted) drops the cov3D chain at compile time.
template <bool SHAPE, bool DET>
__global__ void __launch_bounds__(256, 2)
fused_preprocess_backward_kernel(const __grid_constant__ CamConst cam, int64_t N, VtgsParams prm,
                                 const float* __restrict__ pose_Rt, float dr0, float dr1, float dr2,
                                 const GeomRecord* __restrict__ geom, float* __restrict__ grad_geom,
                                 VtgsParamGrads out, int accumulate, int want_pose,
                                 const VtgsCounters* __restrict__ counters, unsigned int* __restrict__ ticket,
                                 const uint32_t* __restrict__ tiles_touched, const uint8_t* __restrict__ band_flags,
                                 const uint32_t* __restrict__ cand, const uint32_t* __restrict__ n_cand) {
    VTGS_PDL_PROLOGUE();
    __shared__ LastBlockSum<POSE_TERMS> red;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t stride = (int64_t)gridDim.x * 256;
    const bool rot_aligned = (reinterpret_cast<uintptr_t>(prm.unnorm_rotations) & 15) == 0;
    float Rt[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) Rt[k] = __ldg(pose_Rt + k);
    float pose_v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) pose_v[k] = 0.0f;

    const bool want_op = out.logit_opacities != nullptr;
    // the blend kernel formed the colour / opacity sums unless it ran in its pose-only form (same condition as there)
    const bool want_colour_opacity = out.rgb_colors != nullptr || out.logit_opacities != nullptr;
    auto process = [&](const K7Item& it, const int64_t i) {
        float4 g0, g1, g2;
        bool dirty;
        decode_grad_record<DET>(it.raw, want_colour_opacity, g0, g1, g2, dirty);
        // culled splats, and splats no pixel blended (all sums exactly zero), have zero gradients: every
        // term below is linear in g0..g2
        const bool any_grad = (g0.x != 0.f) | (g0.y != 0.f) | (g0.z != 0.f) | (g0.w != 0.f) | (g1.x != 0.f) | (g1.y != 0.f) |
                              (g1.z != 0.f) | (g1.w != 0.f) | (g2.x != 0.f) | (g2.y != 0.f);
        if (dirty) zero_grad_record<DET>(grad_geom, i, want_colour_opacity);        // leave the scratch zeroed for the next backward
        const bool visible = it.hx > -1e29f && any_grad;
        float dmeanw[3] = {0.f, 0.f, 0.f}, dls = 0.f, dlogit = 0.f, dqu[4] = {0.f, 0.f, 0.f, 0.f};
        if (visible) {
            const float px = it.px, py = it.py, pz = it.pz;
            const float x = fadd(ffma(Rt[2], pz, ffma(Rt[1], py, fmul(Rt[0], px))), Rt[9]);
            const float y = fadd(ffma(Rt[5], pz, ffma(Rt[4], py, fmul(Rt[3], px))), Rt[10]);
            const float z = fadd(ffma(Rt[8], pz, ffma(Rt[7], py, fmul(Rt[6], px))), Rt[11]);
            const float s = vexpf(it.ls);
            const float u[4] = {it.uq.x, it.uq.y, it.uq.z, it.uq.w};
            const float nrm = sqrtf(u[0] * u[0] + u[1] * u[1] + u[2] * u[2] + u[3] * u[3]);
            const float d = fmaxf(nrm, 1e-12f), id_ = __fdividef(1.0f, d);
            const float q[4] = {u[0] * id_, u[1] * id_, u[2] * id_, u[3] * id_};
            float R[9], S[6];
            quat_to_R(q[0], q[1], q[2], q[3], R);
            cov3d_from(s, s, s, cam.scale_modifier, R, S);
            CovGrad cg;
            cov2d_backward(cam, x, y, z, S, g0.z, g0.w, g1.x, g0.x, g0.y, cg);
            float dscale[3] = {0.f, 0.f, 0.f}, dq[4] = {0.f, 0.f, 0.f, 0.f};
            if (SHAPE) cov3d_backward(cg.dS, R, cam.scale_modifier, s, s, s, q[0], q[1], q[2], q[3], dscale, dq);
            // chain through get_depth_and_silhouette: colour channel 3 is z_cam = depth_row . (p', 1)
            const float dz = g2.y;
            const float gm[3] = {cg.dmean[0] + dr0 * dz, cg.dmean[1] + dr1 * dz, cg.dmean[2] + dr2 * dz};
            // p' = R p + t
            dmeanw[0] = Rt[0] * gm[0] + Rt[3] * gm[1] + Rt[6] * gm[2];
            dmeanw[1] = Rt[1] * gm[0] + Rt[4] * gm[1] + Rt[7] * gm[2];
            dmeanw[2] = Rt[2] * gm[0] + Rt[5] * gm[1] + Rt[8] * gm[2];
            dls = (dscale[0] + dscale[1] + dscale[2]) * s;            // d exp(ls)/d ls, tiled x3
            const float o = it.op;
            dlogit = g1.y * o * (1.0f - o);
            // F.normalize backward
            const float qd = q[0] * dq[0] + q[1] * dq[1] + q[2] * dq[2] + q[3] * dq[3];
#pragma unroll
            for (int k = 0; k < 4; ++k) dqu[k] = nrm >= 1e-12f ? (dq[k] - q[k] * qd) * id_ : dq[k] * id_;
            pose_v[0] += gm[0]; pose_v[1] += gm[1]; pose_v[2] += gm[2];
            pose_v[3] += gm[0] * px; pose_v[4] += gm[0] * py; pose_v[5] += gm[0] * pz;
            pose_v[6] += gm[1] * px; pose_v[7] += gm[1] * py; pose_v[8] += gm[1] * pz;
            pose_v[9] += gm[2] * px; pose_v[10] += gm[2] * py; pose_v[11] += gm[2] * pz;
        }
        if (accumulate) {
            if (out.means3D) { out.means3D[3 * i] += dmeanw[0]; out.means3D[3 * i + 1] += dmeanw[1]; out.means3D[3 * i + 2] += dmeanw[2]; }
            if (out.rgb_colors) { out.rgb_colors[3 * i] += g1.z; out.rgb_colors[3 * i + 1] += g1.w; out.rgb_colors[3 * i + 2] += g2.x; }
            if (out.unnorm_rotations) for (int k = 0; k < 4; ++k) out.unnorm_rotations[4 * i + k] += dqu[k];
            if (out.logit_opacities) out.logit_opacities[i] += dlogit;
            if (out.log_scales) out.log_scales[i] += dls;
            if (out.means2D) { out.means2D[3 * i] += g0.x; out.means2D[3 * i + 1] += g0.y; }
        } else {
            if (out.means3D) { out.means3D[3 * i] = dmeanw[0]; out.means3D[3 * i + 1] = dmeanw[1]; out.means3D[3 * i + 2] = dmeanw[2]; }
            if (out.rgb_colors) { out.rgb_colors[3 * i] = g1.z; out.rgb_colors[3 * i + 1] = g1.w; out.rgb_colors[3 * i + 2] = g2.x; }
            if (out.unnorm_rotations) for (int k = 0; k < 4; ++k) out.unnorm_rotations[4 * i + k] = dqu[k];
            if (out.logit_opacities) out.logit_opacities[i] = dlogit;
            if (out.log_scales) out.log_scales[i] = dls;
            if (out.means2D) { out.means2D[3 * i] = g0.x; out.means2D[3 * i + 1] = g0.y; out.means2D[3 * i + 2] = 0.0f; }
        }
    };
    if (cand != nullptr) {
        // tile-band sharding with candidate blocks (K0'): only the 256-Gaussian blocks that can reach the band are read
        // (persistent loop over the list); the others hold exact zeros, written as such when outputs were requested
        const int64_t nc = (int64_t)*n_cand;
        for (int64_t trip = blockIdx.x; trip < nc; trip += gridDim.x) {
            const int64_t i = (int64_t)cand[trip] * 256 + tid;
            if (i >= N) continue;
            K7Item it;
            k7_load<DET>(it, i, prm, geom, grad_geom, rot_aligned, tiles_touched, want_op, want_colour_opacity);
            process(it, i);
        }
        const bool any_out = out.means3D != nullptr || out.rgb_colors != nullptr || out.unnorm_rotations != nullptr ||
                             out.logit_opacities != nullptr || out.log_scales != nullptr || out.means2D != nullptr;
        if (any_out && !accumulate) {
            const int64_t nblk = (N + 255) / 256;
            K7Item zit;
            const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
            zit.raw.a = z4; zit.raw.b = z4; zit.raw.c = z4; zit.raw.d = z4; zit.raw.e = z4; zit.uq = z4;
            zit.hx = -1e30f; zit.op = 0.f; zit.px = 0.f; zit.py = 0.f; zit.pz = 0.f; zit.ls = 0.f;
            for (int64_t b = blockIdx.x; b < nblk; b += gridDim.x) {
                const int64_t i = b * 256 + tid;
                if (band_flags[b] == 0 && i < N) process(zit, i);
            }
        }
    } else {
        int64_t i = (int64_t)blockIdx.x * 256 + tid;
        K7Item nxt;
        if (i < N) k7_load<DET>(nxt, i, prm, geom, grad_geom, rot_aligned, tiles_touched, want_op, want_colour_opacity);
        for (; i < N; i += stride) {
            const K7Item it = nxt;
            if (i + stride < N) k7_load<DET>(nxt, i + stride, prm, geom, grad_geom, rot_aligned, tiles_touched, want_op, want_colour_opacity);
            process(it, i);
        }
    }
    if (!want_pose) return;
    const float tot = warp_transpose_reduce<POSE_TERMS>(pose_v, lane);
    if ((lane & 1) == 0 && (lane >> 1) < POSE_TERMS) red.part[warp][lane >> 1] = tot;
    if (!red.reduce(out.pose_scratch, ticket)) return;
    pose_finalize_block(red, counters, out.cam_unnorm_rot, out.cam_trans, accumulate, out.pose_scale);
}

}  // namespace vtgs

// =============================== C entry points (include/vtgs.h) ===========================
using namespace vtgs;

uint64_t vtgs_pose_scratch_floats(int64_t N) { return (uint64_t)((N + 255) / 256 + 1) * 12; }

// API-mode backward (K6' + K7').
int vtgs_backward(const VtgsCamera* camera, int64_t N, const float* means3D, const float* scales,
                  const float* rotations, const float* opacities, const float* colors,
                  const float* dL_dout_color, float* dL_dmeans2D, float* dL_dcolors, float* dL_dopacity,
                  float* dL_dmeans3D, float* dL_dscales, float* dL_drotations, VtgsBuffers* buf, void* stream_) {
    if (int e = check_cam(camera)) return e;
    if (int e = check_buf(buf, N)) return e;
    VTGS_REQUIRE(N >= 0, "num_gaussians < 0");
    if (N > 0)
        VTGS_REQUIRE(means3D && scales && rotations && dL_dout_color && dL_dmeans2D && dL_dcolors && dL_dopacity &&
                         dL_dmeans3D && dL_dscales && dL_drotations,
                     "pointer is NULL");
    (void)opacities; (void)colors;
    const cudaStream_t stream = (cudaStream_t)stream_;
    const CamConst cam = make_cam_const(*camera);
    const GeomRecord* geom = reinterpret_cast<const GeomRecord*>(buf->geom);
    const int band_tiles = (cam.row1 - cam.row0) * cam.gx;
    if (N <= 0) return VTGS_OK;
    const bool det = (buf->flags & VTGS_BUF_DETERMINISTIC) != 0;
    if (band_tiles > 0) {
        const bool has_bg = cam.bg[0] != 0.0f || cam.bg[1] != 0.0f || cam.bg[2] != 0.0f;
        const int blocks = band_tiles * (8 / BWD_WARPS);
        const uint32_t* order = nullptr;                  // (the forward orders tiles only for the fused path's tile bands)
        if (int e = launch_blend_backward(false, has_bg, false, blocks, stream, cam, buf, geom, dL_dout_color, order, nullptr)) return e;
    }
    return launch_k("preprocess_backward_kernel", Launch::plain, det ? preprocess_backward_kernel<true> : preprocess_backward_kernel<false>,
                    dim3((unsigned)((N + 255) / 256)), dim3(256), 0, stream, cam, N, means3D, scales, rotations, nullptr, geom, buf->grad_geom,
                    dL_dmeans2D, dL_dcolors, dL_dopacity, dL_dmeans3D, dL_dscales, dL_drotations);
}

int vtgs_fused_backward(const VtgsCamera* camera, const VtgsParams* params, const VtgsPose* pose, const float* dL_dimage4,
                        int32_t accumulate, VtgsParamGrads* grads, VtgsBuffers* buf, void* stream_) {
    if (int e = check_fused(camera, params, pose, buf)) return e;
    VTGS_REQUIRE(dL_dimage4 && grads, "pointer is NULL");
    const cudaStream_t stream = (cudaStream_t)stream_;
    const CamConst cam = make_cam_const(*camera);
    const int64_t N = params->num_gaussians;
    const GeomRecord* geom = reinterpret_cast<const GeomRecord*>(buf->geom);
    const int band_tiles = (cam.row1 - cam.row0) * cam.gx;
    const int want_pose = (grads->cam_unnorm_rot != nullptr && grads->cam_trans != nullptr) ? 1 : 0;
    if (want_pose && grads->pose_scratch == nullptr) { set_error("pose gradients need pose_scratch"); return VTGS_E_INVALID; }
    // persistent K7' grid: 148 SMs x 2 resident blocks x 2 waves (fixed, so the partial-sum layout is deterministic)
    const int blocks = (int)std::min<int64_t>((N + 255) / 256, 148 * 4);
    if (N > 0) {
        if (band_tiles > 0) {
            const bool has_bg = cam.bg[0] != 0.0f || cam.bg[1] != 0.0f || cam.bg[2] != 0.0f;
            // tracking asks for the pose gradient only: no colour / opacity sums are formed (K7' never reads them then)
            const bool lite = grads->rgb_colors == nullptr && grads->logit_opacities == nullptr;
            const int bblocks = band_tiles * (8 / BWD_WARPS);
            // the fused forward left the band's tiles in longest-list-first order (tile bands only: same condition there)
            const uint32_t* order = band_tiles < cam.gx * cam.gy ? buf->tile_order : nullptr;
            if (int e = launch_blend_backward(true, has_bg, lite, bblocks, stream, cam, buf, geom, dL_dimage4, order, grads->dL_abs_bound)) return e;
        }
        unsigned int* ticket = reinterpret_cast<unsigned int*>(grads->pose_scratch ? grads->pose_scratch + (size_t)blocks * POSE_TERMS : nullptr);
        const uint32_t* band_touch = band_tiles < cam.gx * cam.gy ? buf->tiles_touched : nullptr;
        // candidate blocks of the band, written by this iteration's forward (K0'); the counter follows the tile counts
        const bool use_cand = band_touch != nullptr && buf->band_flags != nullptr && buf->band_cand != nullptr;
        const uint8_t* band_flags = use_cand ? buf->band_flags : nullptr;
        const uint32_t* band_cand = use_cand ? buf->band_cand : nullptr;
        const uint32_t* n_cand = buf->tile_counts + cam.gx * cam.gy;
        const bool shape = grads->log_scales != nullptr || grads->unnorm_rotations != nullptr;
        const bool det = (buf->flags & VTGS_BUF_DETERMINISTIC) != 0;
        auto k7 = shape ? (det ? fused_preprocess_backward_kernel<true, true> : fused_preprocess_backward_kernel<true, false>)
                        : (det ? fused_preprocess_backward_kernel<false, true> : fused_preprocess_backward_kernel<false, false>);
        return launch_k("fused_preprocess_backward_kernel", Launch::pdl, k7, dim3(blocks), dim3(256), 0, stream, cam, N, *params,
                        buf->counters->pose_R, pose->depth_row[0], pose->depth_row[1], pose->depth_row[2], geom, buf->grad_geom, *grads,
                        accumulate, want_pose, buf->counters, ticket, band_touch, band_flags, band_cand, n_cand);
    }
    if (want_pose && !accumulate) {
        VTGS_CUDA_CHECK(cudaMemsetAsync(grads->cam_unnorm_rot, 0, 4 * sizeof(float), stream));
        VTGS_CUDA_CHECK(cudaMemsetAsync(grads->cam_trans, 0, 3 * sizeof(float), stream));
    }
    return VTGS_OK;
}
