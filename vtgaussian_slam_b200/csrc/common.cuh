// common.cuh -- shared device helpers of the sm_100a splatting kernels.
//
// Arithmetic spec (DESIGN.md "Arithmetic spec"): the forward is IEEE fp32 in a fixed
// operation order; products and sums are only fused where the code says __fmaf_rn.
// __fmul_rn / __fadd_rn / __fsub_rn are never contracted by nvcc, so the result does not
// depend on -fmad.  Every function here that feeds an integer output (radii, tile rects,
// sort keys, n_contrib) is written with these intrinsics.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/vtgs.h"

#define VTGS_FULL_MASK 0xffffffffu

namespace vtgs {

// ---- error plumbing (host) -------------------------------------------------------------
void set_error(const char* fmt, ...);
#define VTGS_CUDA_CHECK(expr)                                                        \
    do {                                                                             \
        cudaError_t _e = (expr);                                                     \
        if (_e != cudaSuccess) {                                                     \
            vtgs::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),  \
                            __FILE__, __LINE__);                                     \
            return VTGS_E_CUDA;                                                      \
        }                                                                            \
    } while (0)

// RAII event bracket around one kernel launch (only when vtgs_profile_enable(1) was called).
struct ProfScope {
    ProfScope(const char* name, cudaStream_t stream);
    ~ProfScope();
    int slot;
    cudaStream_t stream;
};

// ---- programmatic dependent launch (PDL) ------------------------------------------------------------------------
// The kernels of an iteration form a chain in one stream / CUDA graph, and several of them are short.  Launched with
// the programmatic-stream-serialization attribute, a kernel's launch and block scheduling overlap the drain of its
// predecessor; its blocks then sit in pdl_wait() until the predecessor grid has completed and its memory is visible.
// Every kernel launched with Launch::pdl therefore starts with pdl_wait() BEFORE it touches global memory: the
// ordering is that of a plain stream.  (Without the attribute the instruction is a no-op.)  Measured at C2 on one
// B200 (graph replay): +0.5 %; with an early `griddepcontrol.launch_dependents` in every kernel (dependent blocks
// resident behind the predecessor's last wave) -0.4 %, so the trigger stays implicit.  VTGS_PDL=0 turns the attribute off.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#define VTGS_PDL_PROLOGUE() vtgs::pdl_wait()

bool pdl_enabled();        // api.cu: environment VTGS_PDL (default on)

// Launch::plain is for kernels without pdl_wait(): a launch with no attributes, the same as <<<>>>.
enum class Launch { plain, pdl };

// Every kernel launch of the library: `kernel` runs under the profile name `name` (vtgs_profile_summary; bench.py's
// per_kernel_us keys on these names).  Returns VTGS_OK, or VTGS_E_CUDA when the launch failed.
template <typename... KArgs, typename... Args>
inline int launch_k(const char* name, Launch mode, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                    cudaStream_t stream, Args&&... args) {
    {
        ProfScope prof(name, stream);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid;
        cfg.blockDim = block;
        cfg.dynamicSmemBytes = smem;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = (mode == Launch::pdl && pdl_enabled()) ? 1 : 0;
        (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);      // its error is also cudaGetLastError()'s
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("launch of %s failed: %s", name, cudaGetErrorString(e));
        return VTGS_E_CUDA;
    }
    return VTGS_OK;
}

// One-time kernel attribute setup PER DEVICE (a process may drive several GPUs): true for the first caller on the
// current device.  `mask` is a function-local static std::atomic<uint64_t>.
template <typename AtomicU64>
inline bool first_call_on_device(AtomicU64& mask) {
    int d = 0;
    cudaGetDevice(&d);
    const uint64_t bit = 1ull << (d & 63);
    return (mask.fetch_or(bit) & bit) == 0;
}

// ---- packed per-Gaussian render record (VTGS_GEOM_RECORD_BYTES = 64) ---------------------
//   q0 = {px, py, hx, hy}            pixel centre and the half extents of the alpha >= 1/255 ellipse's box
//   q1 = {A, B, C, opacity}          conic and opacity
//   q2 = {c0, c1, c2, c3}            colours; c3 = view depth (API mode) / z channel (fused mode)
//   q3 = {depth, pthr, rect_min, rect_max}   pthr: conservative lower bound of `power` for alpha >= 1/255;
//                                    rect packed as x | y << 16 (band-clipped in y)
// Culled splats carry hx = hy = -1e30 and pthr = 1 (never pass any test).
struct __align__(16) GeomRecord {
    float4 q0, q3, q1, q2;          // memory order: {q0, q3} (what the scatter reads) share one 32-byte sector
};
static_assert(sizeof(GeomRecord) == VTGS_GEOM_RECORD_BYTES, "record size");

struct CamConst {
    float view[16];
    float proj[16];
    float bg[3];
    float tanfovx, tanfovy;
    float focal_x, focal_y;
    float limx, limy;
    float scale_modifier;
    float sigma_mult;
    int W, H;
    int gx, gy;
    int row0, row1;
};

inline CamConst make_cam_const(const VtgsCamera& c) {
    CamConst k;
    for (int i = 0; i < 16; ++i) { k.view[i] = c.viewmatrix[i]; k.proj[i] = c.projmatrix[i]; }
    for (int i = 0; i < 3; ++i) k.bg[i] = c.bg[i];
    k.tanfovx = c.tanfovx; k.tanfovy = c.tanfovy;
    k.W = c.image_width; k.H = c.image_height;
    // host fp32 arithmetic (IEEE, no contraction possible in these single operations)
    k.focal_x = (float)c.image_width / (2.0f * c.tanfovx);
    k.focal_y = (float)c.image_height / (2.0f * c.tanfovy);
    k.limx = VTGS_FRUSTUM_MULT * c.tanfovx;
    k.limy = VTGS_FRUSTUM_MULT * c.tanfovy;
    k.scale_modifier = c.scale_modifier;
    k.sigma_mult = c.radius_sigma_mult;
    k.gx = (c.image_width + VTGS_TILE - 1) / VTGS_TILE;
    k.gy = (c.image_height + VTGS_TILE - 1) / VTGS_TILE;
    k.row0 = 0; k.row1 = k.gy;
    if (c.tile_row_end > c.tile_row_begin) {
        k.row0 = c.tile_row_begin < 0 ? 0 : c.tile_row_begin;
        k.row1 = c.tile_row_end > k.gy ? k.gy : c.tile_row_end;
    }
    return k;
}

// Pixels [b, e) of the camera's tile-row band, clamped to the frame (b <= e; the whole frame without a band).
__host__ __device__ __forceinline__ void band_pixel_range(const CamConst& cam, size_t& b, size_t& e) {
    const size_t P = (size_t)cam.W * cam.H;
    b = (size_t)cam.row0 * 16 * cam.W;
    e = (size_t)cam.row1 * 16 * cam.W;
    if (e > P) e = P;
    if (b > e) b = e;
}

// ---- spec'd elementary functions (device) -------------------------------------------------
__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float ffma(float a, float b, float c) { return __fmaf_rn(a, b, c); }

// exp(x): Cody-Waite reduction + Cephes degree-5 polynomial, scaling by exponent add.
// Bit-identical to vexpf() of the CPU oracle.
// CLAMP = false: the caller guarantees x in [-87, 88] (the clamp is then the identity; same bits).
template <bool CLAMP = true>
__device__ __forceinline__ float vexpf(float x) {
    if (CLAMP) x = fminf(fmaxf(x, -87.0f), 88.0f);
    const float t = ffma(x, 1.44269504088896341f, 12582912.0f);
    const float n = fsub(t, 12582912.0f);
    float r = ffma(n, -0.693145751953125f, x);
    r = ffma(n, -1.428606765330187045e-06f, r);
    float p = 1.9875691500e-4f;
    p = ffma(p, r, 1.3981999507e-3f);
    p = ffma(p, r, 8.3334519073e-3f);
    p = ffma(p, r, 4.1665795894e-2f);
    p = ffma(p, r, 1.6666665459e-1f);
    p = ffma(p, r, 5.0000001201e-1f);
    const float r2 = fmul(r, r);
    float e = ffma(p, r2, r);
    e = fadd(e, 1.0f);
    // n (|n| <= 128) sits in the low mantissa bits of t = 1.5 * 2^23 + n, whose other low 22 bits are zero:
    // bits(t) << 23 == (int)n << 23 (mod 2^32) -- the exponent add without a float -> int conversion
    return __uint_as_float(__float_as_uint(e) + (__float_as_uint(t) << 23));
}

// Bare MUFU approximations for arguments known to be far from the denormal / overflow guards that __expf and
// __fdividef wrap around them (3 and 5 extra instructions): gradients only (judged to 1e-3), never decisions.
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ float sqrt_approx(float x) {
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// index of the most significant set bit (x != 0): one FLO instead of 31 - (31 - FLO)
__device__ __forceinline__ int msb_index(uint32_t x) {
    int r;
    asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(x));
    return r;
}

__device__ __forceinline__ float xform_row(const float* __restrict__ m, int r, float x, float y, float z) {
    return fadd(ffma(m[8 + r], z, ffma(m[4 + r], y, fmul(m[r], x))), m[12 + r]);
}
__device__ __forceinline__ float dot3(float a0, float a1, float a2, float b0, float b1, float b2) {
    return ffma(a2, b2, ffma(a1, b1, fmul(a0, b0)));
}

__device__ __forceinline__ void quat_to_R(float r, float x, float y, float z, float* R) {
    R[0] = fsub(1.0f, fmul(2.0f, ffma(z, z, fmul(y, y))));
    R[1] = fmul(2.0f, ffma(x, y, -fmul(r, z)));
    R[2] = fmul(2.0f, ffma(x, z, fmul(r, y)));
    R[3] = fmul(2.0f, ffma(x, y, fmul(r, z)));
    R[4] = fsub(1.0f, fmul(2.0f, ffma(z, z, fmul(x, x))));
    R[5] = fmul(2.0f, ffma(y, z, -fmul(r, x)));
    R[6] = fmul(2.0f, ffma(x, z, -fmul(r, y)));
    R[7] = fmul(2.0f, ffma(y, z, fmul(r, x)));
    R[8] = fsub(1.0f, fmul(2.0f, ffma(y, y, fmul(x, x))));
}

// Sigma = R diag((mod*s)^2) R^T, upper triangle {xx, xy, xz, yy, yz, zz}.
__device__ __forceinline__ void cov3d_from(float sx, float sy, float sz, float mod, const float* R, float* S) {
    const float s0 = fmul(mod, sx), s1 = fmul(mod, sy), s2 = fmul(mod, sz);
    const float a0 = fmul(s0, s0), a1 = fmul(s1, s1), a2 = fmul(s2, s2);
#define VTGS_SIG(i, j) ffma(fmul(a2, R[3 * i + 2]), R[3 * j + 2], ffma(fmul(a1, R[3 * i + 1]), R[3 * j + 1], fmul(fmul(a0, R[3 * i]), R[3 * j])))
    S[0] = VTGS_SIG(0, 0); S[1] = VTGS_SIG(0, 1); S[2] = VTGS_SIG(0, 2);
    S[3] = VTGS_SIG(1, 1); S[4] = VTGS_SIG(1, 2); S[5] = VTGS_SIG(2, 2);
#undef VTGS_SIG
}

// power = -0.5 (A dx^2 + C dy^2) - B dx dy in the spec'd order.
__device__ __forceinline__ float power_of(float A, float B, float C, float dx, float dy) {
    const float q = ffma(fmul(A, dx), dx, fmul(fmul(C, dy), dy));
    return ffma(-0.5f, q, -fmul(fmul(B, dx), dy));
}

__device__ __forceinline__ int clampi(int v, int hi) { return min(hi, max(0, v)); }

// Tile rect of a splat (upstream getRect) in the spec'd float order; casts saturate (cvt.rzi).
__device__ __forceinline__ void tile_rect(float px, float py, int radius, int gx, int gy,
                                          int& minx, int& miny, int& maxx, int& maxy) {
    const float rf = (float)radius;
    minx = clampi(__float2int_rz(__fdiv_rn(fsub(px, rf), 16.0f)), gx);
    miny = clampi(__float2int_rz(__fdiv_rn(fsub(py, rf), 16.0f)), gy);
    maxx = clampi(__float2int_rz(__fdiv_rn(fsub(fadd(fadd(px, rf), 16.0f), 1.0f), 16.0f)), gx);
    maxy = clampi(__float2int_rz(__fdiv_rn(fsub(fadd(fadd(py, rf), 16.0f), 1.0f), 16.0f)), gy);
}

struct SplatGeom {      // what preprocess computes for one Gaussian
    float px, py, depth;
    float A, B, C;      // conic
    float cov_a, cov_b, cov_c;
    int radius;         // 0 = culled
    int minx, miny, maxx, maxy;   // full-image tile rect
};

// SURVEY.md Appendix A.1 in the spec'd operation order (mirrors oracle preprocess_one).
__device__ __forceinline__ void splat_geometry(const CamConst& cam, float x, float y, float z,
                                               float sx, float sy, float sz,
                                               float qr, float qx, float qy, float qz, SplatGeom& g) {
    g.radius = 0;
    const float* V = cam.view;
    const float tx = xform_row(V, 0, x, y, z);
    const float ty = xform_row(V, 1, x, y, z);
    const float tz = xform_row(V, 2, x, y, z);
    g.depth = tz;
    if (tz <= VTGS_NEAR_CULL) return;
    const float hx = xform_row(cam.proj, 0, x, y, z);
    const float hy = xform_row(cam.proj, 1, x, y, z);
    const float hw = xform_row(cam.proj, 3, x, y, z);
    const float pw = __fdiv_rn(1.0f, fadd(hw, VTGS_EPS_W));
    const float ndcx = fmul(hx, pw), ndcy = fmul(hy, pw);

    float R[9], S[6];
    quat_to_R(qr, qx, qy, qz, R);
    cov3d_from(sx, sy, sz, cam.scale_modifier, R, S);

    const float cx = fmul(fminf(cam.limx, fmaxf(-cam.limx, __fdiv_rn(tx, tz))), tz);
    const float cy = fmul(fminf(cam.limy, fmaxf(-cam.limy, __fdiv_rn(ty, tz))), tz);
    const float tz2 = fmul(tz, tz);
    const float J00 = __fdiv_rn(cam.focal_x, tz);
    const float J02 = __fdiv_rn(-fmul(cam.focal_x, cx), tz2);
    const float J11 = __fdiv_rn(cam.focal_y, tz);
    const float J12 = __fdiv_rn(-fmul(cam.focal_y, cy), tz2);
    float m0[3], m1[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        m0[k] = ffma(J02, V[4 * k + 2], fmul(J00, V[4 * k + 0]));
        m1[k] = ffma(J12, V[4 * k + 2], fmul(J11, V[4 * k + 1]));
    }
    const float u0 = dot3(S[0], S[1], S[2], m0[0], m0[1], m0[2]);
    const float u1 = dot3(S[1], S[3], S[4], m0[0], m0[1], m0[2]);
    const float u2 = dot3(S[2], S[4], S[5], m0[0], m0[1], m0[2]);
    const float v0 = dot3(S[0], S[1], S[2], m1[0], m1[1], m1[2]);
    const float v1 = dot3(S[1], S[3], S[4], m1[0], m1[1], m1[2]);
    const float v2 = dot3(S[2], S[4], S[5], m1[0], m1[1], m1[2]);
    const float a = fadd(dot3(m0[0], m0[1], m0[2], u0, u1, u2), VTGS_LOWPASS);
    const float b = dot3(m1[0], m1[1], m1[2], u0, u1, u2);
    const float c = fadd(dot3(m1[0], m1[1], m1[2], v0, v1, v2), VTGS_LOWPASS);

    const float det = ffma(a, c, -fmul(b, b));
    if (det == 0.0f) return;
    const float inv = __fdiv_rn(1.0f, det);
    const float mid = fmul(0.5f, fadd(a, c));
    const float sq = __fsqrt_rn(fmaxf(VTGS_LAMBDA_FLOOR, ffma(mid, mid, -det)));
    const float lam = fmaxf(fadd(mid, sq), fsub(mid, sq));
    const int radius = __float2int_rz(ceilf(fmul(cam.sigma_mult, __fsqrt_rn(lam))));
    // ndc2Pix: fp64, rounded once (upstream writes it with double literals)
    const float px = (float)((((double)ndcx + 1.0) * (double)cam.W - 1.0) * 0.5);
    const float py = (float)((((double)ndcy + 1.0) * (double)cam.H - 1.0) * 0.5);
    int minx, miny, maxx, maxy;
    tile_rect(px, py, radius, cam.gx, cam.gy, minx, miny, maxx, maxy);
    if ((maxx - minx) * (maxy - miny) == 0) return;
    g.px = px; g.py = py;
    g.A = fmul(c, inv); g.B = fmul(-b, inv); g.C = fmul(a, inv);
    g.cov_a = a; g.cov_b = b; g.cov_c = c;
    g.radius = radius;
    g.minx = minx; g.miny = miny; g.maxx = maxx; g.maxy = maxy;
}

// Conservative blend-culling data for one splat: pthr (lower bound of power for which
// alpha >= 1/255 is possible) and the half extents of that ellipse's bounding box.
// These only ever REMOVE pair tests that would fail the exact alpha test, so they need no
// bit-parity with the oracle, only safety margins.
__device__ __forceinline__ void cull_bounds(float opacity, float cov_a, float cov_c, float& pthr, float& hx, float& hy) {
    pthr = logf(VTGS_ALPHA_MIN / opacity) - 1e-3f;      // NaN / +inf when opacity <= 0: never passes
    if (!(pthr <= 0.0f)) { pthr = 1.0f; hx = -1e30f; hy = -1e30f; return; }
    const float two_tau = -2.0f * pthr;
    hx = sqrtf(two_tau * cov_a) * 1.0001f + 0.01f;
    hy = sqrtf(two_tau * cov_c) * 1.0001f + 0.01f;
    if (!(hx == hx) || !(hy == hy)) { hx = 1e30f; hy = 1e30f; }
}

// Pose of the frame (reference transform_to_frame, utils/slam_helpers.py:339-350 + build_rotation,
// utils/slam_external.py:25-42): q = F.normalize(cam_unnorm_rot), then build_rotation normalises once
// more.  Spec'd fp32 order, mirrored by the oracle (vtgso_pose_matrix).  Rt = R (row-major 9) then t (3).
__device__ __forceinline__ void pose_from_quat(const float* __restrict__ q_un, const float* __restrict__ t,
                                               float* Rt, float* q_norm1 /*4*/, float* norms /*2*/) {
    const float u0 = q_un[0], u1 = q_un[1], u2 = q_un[2], u3 = q_un[3];
    const float n1 = __fsqrt_rn(ffma(u3, u3, ffma(u2, u2, ffma(u1, u1, fmul(u0, u0)))));
    const float d1 = fmaxf(n1, 1e-12f);
    const float q0 = __fdiv_rn(u0, d1), q1 = __fdiv_rn(u1, d1), q2 = __fdiv_rn(u2, d1), q3 = __fdiv_rn(u3, d1);
    const float n2 = __fsqrt_rn(ffma(q3, q3, ffma(q2, q2, ffma(q1, q1, fmul(q0, q0)))));
    quat_to_R(__fdiv_rn(q0, n2), __fdiv_rn(q1, n2), __fdiv_rn(q2, n2), __fdiv_rn(q3, n2), Rt);
    Rt[9] = t[0]; Rt[10] = t[1]; Rt[11] = t[2];
    q_norm1[0] = q0; q_norm1[1] = q1; q_norm1[2] = q2; q_norm1[3] = q3;
    norms[0] = n1; norms[1] = n2;
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(VTGS_FULL_MASK, v, o);
    return v;
}

// ---- fixed-order sum of T terms over the blocks of a grid -------------------------------------------------------------
// Each block leaves one fp32 partial per term, its warps' values summed in warp order.  SLICES = THREADS / T threads
// per term then form fp64 slice sums: slice s sums the blocks b = s (mod SLICES) in ascending order, and a term's total
// sums its slices in ascending order.  The result is the same whatever order the blocks ran in.
template <int T, int WARPS>
__device__ __forceinline__ float warp_order_sum(const float (&part)[WARPS][T], int term) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) s += part[w][term];
    return s;
}

// SAME_GRID: the partials were written by other blocks of the running grid, so they are read from L2 (__ldcg), not
// through this SM's L1; otherwise an earlier launch wrote them.
template <int T, int THREADS, bool SAME_GRID = true>
__device__ __forceinline__ void slice_sums(const float* partials, int nblocks, double (&slice)[T][THREADS / T]) {
    constexpr int SLICES = THREADS / T;
    const int tid = threadIdx.x;
    if (tid < T * SLICES) {
        const int term = tid % T, sl = tid / T;          // consecutive threads read consecutive partials
        double acc = 0.0;
        for (int b = sl; b < nblocks; b += SLICES) {
            const float* p = &partials[(size_t)b * T + term];
            acc += (double)(SAME_GRID ? __ldcg(p) : *p);
        }
        slice[term][sl] = acc;
    }
}

template <int T, int SLICES>
__device__ __forceinline__ double slices_total(const double (&slice)[T][SLICES], int term) {
    double a = 0.0;
    for (int s = 0; s < SLICES; ++s) a += slice[term][s];
    return a;
}

// The same in one launch: the block whose ticket comes last sums every block's partials.  Declared __shared__ by the
// kernel, which leaves each warp's values in part[warp][term] and calls reduce() with all its threads.  reduce()
// returns true in the last block only, with the slice sums formed and the ticket (zero on entry) reset to zero;
// total(term) is then the term's sum over the grid.
template <int T, int THREADS = 256>
struct LastBlockSum {
    float part[THREADS / 32][T];
    double slice[T][THREADS / T];
    bool last;

    __device__ __forceinline__ bool reduce(float* partials, unsigned int* ticket) {
        const int tid = threadIdx.x;
        __syncthreads();
        if (tid < T) {
            partials[(size_t)blockIdx.x * T + tid] = warp_order_sum(part, tid);
            __threadfence();                             // the partial is visible before the ticket is taken
        }
        __syncthreads();
        if (tid == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
        __syncthreads();
        if (!last) return false;
        if (tid == 0) *ticket = 0u;                      // every block has taken its ticket
        __threadfence();
        slice_sums<T, THREADS>(partials, gridDim.x, slice);
        __syncthreads();
        return true;
    }
    __device__ __forceinline__ double total(int term) const { return slices_total(slice, term); }
};

}  // namespace vtgs
