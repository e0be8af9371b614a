// api.cu -- the library-wide part of the extern "C" boundary declared in include/vtgs.h: errors, build info, workspace
// sizes, PDL and profiling switches, and the composed tracking step.  Every other entry point is defined in the .cu
// file that owns its kernels.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"
#include "kernels.h"

namespace vtgs {
static thread_local char g_err[512] = "";
bool pdl_enabled() {
    static const bool on = [] { const char* e = getenv("VTGS_PDL"); return !(e && e[0] == '0'); }();
    return on;
}

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// ---- optional per-kernel event timing ----------------------------------------------------------
struct ProfRec { const char* name; cudaEvent_t a, b; };
static bool g_prof_on = false;
static std::vector<ProfRec> g_prof;
static std::mutex g_prof_mu;

ProfScope::ProfScope(const char* name, cudaStream_t st) : slot(-1), stream(st) {
    if (!g_prof_on) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    ProfRec r{name, nullptr, nullptr};
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
    cudaEventRecord(r.a, st);
    g_prof.push_back(r);
    slot = (int)g_prof.size() - 1;
}
ProfScope::~ProfScope() {
    if (slot < 0) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    cudaEventRecord(g_prof[slot].b, stream);
}
}  // namespace vtgs

using namespace vtgs;

#pragma GCC visibility push(default)
extern "C" {

int vtgs_abi_version(void) { return VTGS_ABI_VERSION; }
const char* vtgs_last_error(void) { return g_err; }
const char* vtgs_build_info(void) {
    return "libvtgs_cuda sm_100a (compute_100a) nvcc " VTGS_STR_NVCC " -lineinfo; hand-written CUDA, no CUB/Thrust";
}

int vtgs_workspace_query(int32_t W, int32_t H, int64_t N, uint64_t pair_capacity, VtgsWorkspaceSizes* s) {
    VTGS_REQUIRE(s != nullptr, "sizes is NULL");
    VTGS_REQUIRE(W > 0 && H > 0 && N >= 0, "bad dimensions");
    const uint64_t gx = (W + VTGS_TILE - 1) / VTGS_TILE, gy = (H + VTGS_TILE - 1) / VTGS_TILE;
    const uint64_t n = (uint64_t)(N > 0 ? N : 1), P = (uint64_t)W * H;
    s->geom_bytes = n * VTGS_GEOM_RECORD_BYTES;
    s->tiles_touched_bytes = n * 4;
    s->tile_counts_bytes = (gx * gy + 3) * 4;
    s->tile_ranges_bytes = gx * gy * 8;
    s->pair_keys_bytes = (pair_capacity > 0 ? pair_capacity : 1) * 8;
    s->point_list_bytes = (pair_capacity > 0 ? pair_capacity : 1) * 4;
    s->final_T_bytes = P * 4;
    s->n_contrib_bytes = P * 4;
    s->grad_geom_bytes = n * VTGS_GRAD_GEOM_FLOATS * 4;
    s->counters_bytes = sizeof(VtgsCounters);
    s->region_pairs_bytes = (pair_capacity > 0 ? pair_capacity : 1) * 8 * 8;
    s->region_cnt_bytes = gx * gy * 8 * 4;
    s->region_masks_bytes = ((pair_capacity > 0 ? pair_capacity : 1) + 32 * gx * gy) * 8 * 4;
    s->region_done_bytes = gx * gy * 8 * 4;
    s->band_flags_bytes = (n + 255) / 256;
    s->band_cand_bytes = ((n + 255) / 256) * 4;
    s->tile_order_bytes = gx * gy * 4;
    s->tiles_x = (uint32_t)gx;
    s->tiles_y = (uint32_t)gy;
    return VTGS_OK;
}

int vtgs_fused_tracking_step(const VtgsCamera* cam, const VtgsParams* p, const VtgsPose* pose, const VtgsLossConfig* cfg,
                             const float* gt_rgb, const float* gt_depth, float* out_image6, int32_t* radii, float* dL_dimage4,
                             float* loss_terms, float* loss_scratch, VtgsParamGrads* grads, float* max_2D_radius, uint8_t* seen,
                             VtgsBuffers* buf, void* stream) {
    VTGS_REQUIRE(cfg && cfg->mode == 0, "vtgs_fused_tracking_step needs a tracking-mode loss configuration");
    VTGS_REQUIRE((max_2D_radius == nullptr) == (seen == nullptr), "max_2D_radius and seen come as a pair");
    if (int e = vtgs_fused_forward(cam, p, pose, out_image6, radii, buf, stream)) return e;
    if (int e = vtgs_loss(cam, cfg, out_image6, gt_rgb, gt_depth, dL_dimage4, loss_terms, loss_scratch, stream)) return e;
    VtgsParamGrads g = *grads;
    if (g.dL_abs_bound == nullptr) g.dL_abs_bound = loss_terms + 6;     // the tracking loss's own bound of |dL/dplane|
    if (int e = vtgs_fused_backward(cam, p, pose, dL_dimage4, 0, &g, buf, stream)) return e;
    if (max_2D_radius != nullptr)
        if (int e = vtgs_book_radii(p->num_gaussians, radii, max_2D_radius, seen, stream)) return e;
    return VTGS_OK;
}

int vtgs_profile_enable(int32_t on) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (on) {
        for (auto& r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
        g_prof.clear();
    }
    g_prof_on = on != 0;
    return VTGS_OK;
}

int vtgs_profile_summary(char* buf, uint64_t capacity) {
    VTGS_REQUIRE(buf != nullptr && capacity > 0, "buffer is NULL");
    std::lock_guard<std::mutex> lk(g_prof_mu);
    std::map<std::string, std::pair<int, double>> agg;
    std::vector<std::string> order;
    for (auto& r : g_prof) {
        if (cudaEventSynchronize(r.b) != cudaSuccess) continue;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) continue;
        if (!agg.count(r.name)) order.push_back(r.name);
        auto& e = agg[r.name];
        e.first += 1;
        e.second += ms;
    }
    std::string out;
    for (auto& n : order) {
        char line[256];
        snprintf(line, sizeof(line), "%s %d %.6f\n", n.c_str(), agg[n].first, agg[n].second);
        out += line;
    }
    if (out.size() + 1 > capacity) { set_error("profile buffer too small"); return VTGS_E_INVALID; }
    memcpy(buf, out.c_str(), out.size() + 1);
    return VTGS_OK;
}

}  // extern "C"
#pragma GCC visibility pop
