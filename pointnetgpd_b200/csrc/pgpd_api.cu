// pgpd_api.cu -- extern "C" entry points of libpgpd.so (see include/pgpd.h) and the model-level
// orchestration: STN3d (tower + regression head), PointNetfeat (+ transform + trunk tower) and
// PointNetCls (+ classifier head + log_softmax), forward and backward.
#include "common.cuh"
#include "tower.cuh"
#include "head.cuh"
#include "prep.cuh"
#include "project.cuh"
#include "gpd.cuh"
#include "dual.cuh"

#include <string>

namespace pgpd {

static thread_local std::string g_err;

static int fail(int code, const char* msg) {
    g_err = msg;
    return code;
}

static int check_cuda(const char* where) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        g_err = std::string(where) + ": " + cudaGetErrorString(e);
        return PGPD_E_CUDA;
    }
    return PGPD_OK;
}

struct ModelWs {
    TowerWs stn_t, trunk_t;
    HeadWs stn_h, cls_h;
    float* g_stn;    // [B][1024] pooled feature of the T-Net tower
    float* G;        // [B][1024] global feature (trunk)
    float* logp;     // [B][k]
    float* dG;       // [B][1024]
    float* dg_stn;   // [B][1024]
    float* dT;       // [B][9]
    size_t bytes;
};

static void plan_model(void* base, int what, int B, int N, int k, int flags, ModelWs& w) {
    Carver c(base);
    const bool save = (flags & PGPD_F_SAVE) != 0;
    plan_tower(c, w.stn_t, B, N);
    if (what >= PGPD_FEAT) {
        if (save) plan_tower(c, w.trunk_t, B, N);
        else static_cast<TowerKeep&>(w.trunk_t) = static_cast<TowerKeep&>(w.stn_t);   // inference: reuse
    }
    plan_tower_scratch(c, w.stn_t, B, N, save);
    static_cast<TowerScratch&>(w.trunk_t) = static_cast<TowerScratch&>(w.stn_t);
    plan_head(c, w.stn_h, B, 9, save);
    w.g_stn = c.take<float>((size_t)B * C3);
    w.G = c.take<float>((size_t)B * C3);
    w.logp = nullptr;
    if (what == PGPD_CLS) {
        plan_head(c, w.cls_h, B, k, save);
        w.logp = c.take<float>((size_t)B * k);
    }
    if (save) {
        w.dG = c.take<float>((size_t)B * C3);
        w.dg_stn = c.take<float>((size_t)B * C3);
        w.dT = c.take<float>((size_t)B * 9);
    }
    w.bytes = (c.off + 255) & ~(size_t)255;
}

static int check_common(int what, const void* m, const float* x, int B, int N, int k, const void* ws, size_t ws_bytes, size_t need) {
    if (what != PGPD_STN && what != PGPD_FEAT && what != PGPD_CLS) return fail(PGPD_E_ARG, "what must be PGPD_STN, PGPD_FEAT or PGPD_CLS");
    if (!m || !x) return fail(PGPD_E_ARG, "null model or input pointer");
    if (B < 1 || N < 1) return fail(PGPD_E_ARG, "B and N must be >= 1");
    if (what == PGPD_CLS && (k < 1 || k > 1024)) return fail(PGPD_E_ARG, "k must be in [1,1024]");
    if ((long long)B * N > 0x7fffffffLL / 128) return fail(PGPD_E_ARG, "B*N too large for this build (B*N*128 must fit in int32)");
    if (!ws || ((uintptr_t)ws & 255)) return fail(PGPD_E_WORKSPACE, "workspace is null or not 256-byte aligned");
    if (ws_bytes < need) return fail(PGPD_E_WORKSPACE, "workspace too small (see pgpd_workspace_bytes)");
    {
        // weights are read with 16-byte vector loads
        const pgpd_model* mm = static_cast<const pgpd_model*>(m);
        bool ok = true;
        auto chk_t = [&](const pgpd_tower& t) { for (int i = 0; i < 3; ++i) ok = ok && !((uintptr_t)t.conv[i].w & 15); };
        auto chk_h = [&](const pgpd_head& h) { for (int i = 0; i < 3; ++i) ok = ok && !((uintptr_t)h.fc[i].w & 15); };
        chk_t(mm->stn_tower); chk_h(mm->stn_head);
        if (what >= PGPD_FEAT) chk_t(mm->trunk);
        if (what == PGPD_CLS) chk_h(mm->cls_head);
        if (!ok || ((uintptr_t)x & 3)) return fail(PGPD_E_ARG, "conv / fc weight pointers must be 16-byte aligned");
    }
    return PGPD_OK;
}

__global__ void k_add_opt(const float* a, const float* b, float* out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = a[i] + (b ? b[i] : 0.f);
}

static bool want_tc(int flags) {
#ifdef PGPD_EMU
    (void)flags;
    return false;
#else
    return !(flags & PGPD_F_SIMT) && tc::available();
#endif
}

static bool head_tc(int flags) { return want_tc(flags); }

static void run_tower_fwd(const TowerArgs& a, TowerWs& w, float* pooled, int) { tower_forward(a, w, pooled); }

static void run_tower_bwd(const TowerArgs& a, TowerWs& w, const pgpd_tower_grad& g, const float* dpooled, float* dtrans, int) {
    tower_backward(a, w, g, dpooled, dtrans);
}

}  // namespace pgpd

using namespace pgpd;

extern "C" {

int pgpd_version(void) { return PGPD_VERSION; }

const char* pgpd_last_error(void) { return g_err.c_str(); }

int pgpd_has_tensor_core_path(void) {
#ifdef PGPD_EMU
    return 0;
#else
    return tc::available() ? 1 : 0;
#endif
}

unsigned long long pgpd_launch_count(void) { return launch_counter(); }

int pgpd_profile_enable(int on) {
    Profiler& pr = profiler();
    pr.reset();
    pr.on = on != 0;
    pr.sticky = on == 2;
    return PGPD_OK;
}

int pgpd_profile_read(int* launches, float* total_ms) {
    if (!launches || !total_ms) return fail(PGPD_E_ARG, "null pointer");
    if (profiler().read(launches, total_ms) != 0) return fail(PGPD_E_CUDA, "event timing failed");
    return PGPD_OK;
}

#ifdef PGPD_DEBUG
/* tuning aid (not part of the documented ABI): copies the [256][8] pipeline cycle counters written by the
 * layer-3 kernel when PGPD_L3_DEBUG is set */
int pgpd_debug_l3_counters(long long* host_out) {
#ifdef PGPD_EMU
    (void)host_out; return PGPD_E_UNSUPPORTED;
#else
    cudaDeviceSynchronize();
    return cudaMemcpy(host_out, tc::l3_debug_buffer(), 512 * 8 * sizeof(long long), cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : PGPD_E_CUDA;
#endif
}

/* tuning aid: route the streaming kernels' cycle counters to the same debug buffer (on != 0) or switch them off */
int pgpd_debug_stream_counters(int on) {
#ifdef PGPD_EMU
    (void)on; return PGPD_E_UNSUPPORTED;
#else
    long long* ptr = on ? tc::l3_debug_buffer() : nullptr;
    cudaDeviceSynchronize();
    if (on) cudaMemset(ptr, 0, 512 * 8 * sizeof(long long));
    return cudaMemcpyToSymbol(tc::g_stream_dbg, &ptr, sizeof(ptr)) == cudaSuccess ? 0 : PGPD_E_CUDA;
#endif
}
#endif  /* PGPD_DEBUG */

size_t pgpd_workspace_bytes(int what, int B, int N, int k, int flags) {
    if (B < 1 || N < 1) return 0;
    ModelWs w;
    plan_model(nullptr, what, B, N, k < 1 ? 1 : k, flags, w);
    return w.bytes;
}

int pgpd_forward(int what, const pgpd_model* m, const float* x, int B, int N, int k, int flags,
                 float* out, float* trans, void* workspace, size_t workspace_bytes, void* stream) {
    ModelWs w;
    plan_model(nullptr, what, B < 1 ? 1 : B, N < 1 ? 1 : N, k < 1 ? 1 : k, flags, w);
    int rc = check_common(what, m, x, B, N, k, workspace, workspace_bytes, w.bytes);
    if (rc) return rc;
    if (!trans) return fail(PGPD_E_ARG, "trans output pointer is null");
    if (what != PGPD_STN && !out) return fail(PGPD_E_ARG, "out pointer is null");
    const bool train = (flags & PGPD_F_TRAIN) != 0;
    if (train && B == 1)
        return fail(PGPD_E_BATCH1, "Expected more than 1 value per channel when training (BatchNorm over a batch of 1)");
    plan_model(workspace, what, B, N, k, flags, w);
    cudaStream_t s = (cudaStream_t)stream;
    const bool save = (flags & PGPD_F_SAVE) != 0;

    // ---- STN3d (pointnet.py:27-45)
    TowerArgs ta{&m->stn_tower, x, nullptr, B, N, true, train, save, s, want_tc(flags)};
    run_tower_fwd(ta, w.stn_t, w.g_stn, flags);
    HeadArgs ha{&m->stn_head, w.g_stn, B, 9, train, true, s, head_tc(flags)};
    head_forward(ha, w.stn_h, trans, nullptr);
    if (what >= PGPD_FEAT) {
        // ---- transform + trunk tower (pointnet.py:140-149); the pooled feature goes straight to the caller for PGPD_FEAT
        TowerArgs tb{&m->trunk, x, w.stn_h.out, B, N, false, train, save, s, want_tc(flags)};
        run_tower_fwd(tb, w.trunk_t, what == PGPD_FEAT ? out : w.G, flags);
        if (what == PGPD_CLS) {
            // ---- classifier head (pointnet.py:191-194)
            HeadArgs hb{&m->cls_head, w.G, B, k, train, false, s, head_tc(flags)};
            head_forward(hb, w.cls_h, out, w.logp);
        }
    }
    return check_cuda("pgpd_forward");
}

int pgpd_backward(int what, const pgpd_model* m, const pgpd_model_grad* g, const float* x,
                  int B, int N, int k, int flags, const float* dout, const float* dtrans,
                  void* workspace, size_t workspace_bytes, void* stream) {
    ModelWs w;
    flags |= PGPD_F_SAVE;
    plan_model(nullptr, what, B < 1 ? 1 : B, N < 1 ? 1 : N, k < 1 ? 1 : k, flags, w);
    int rc = check_common(what, m, x, B, N, k, workspace, workspace_bytes, w.bytes);
    if (rc) return rc;
    if (!g) return fail(PGPD_E_ARG, "null gradient struct");
    if (!(flags & PGPD_F_TRAIN)) return fail(PGPD_E_UNSUPPORTED, "backward through eval-mode BatchNorm is not implemented");
    if (what != PGPD_STN && !dout && !((flags & PGPD_F_BWD_STN) && !(flags & PGPD_F_BWD_HEAD))) return fail(PGPD_E_ARG, "dout is null");
    if (what == PGPD_STN && !dtrans) return fail(PGPD_E_ARG, "dtrans is null");
    if (B == 1) return fail(PGPD_E_BATCH1, "batch of 1 in training mode");
    plan_model(workspace, what, B, N, k, flags, w);
    cudaStream_t s = (cudaStream_t)stream;

    const bool split = what >= PGPD_FEAT && ((flags & PGPD_F_BWD_HEAD) != 0) != ((flags & PGPD_F_BWD_STN) != 0);
    const bool do_head = !split || (flags & PGPD_F_BWD_HEAD), do_stn = !split || (flags & PGPD_F_BWD_STN);
    if (what >= PGPD_FEAT) {
        if (do_head) {
            const float* dG = dout;
            if (what == PGPD_CLS) {
                launch(k_log_softmax_bwd, grid1d(B, 128), dim3(128), 0, s, (const float*)w.logp, dout, B, k, w.cls_h.dO);
                HeadArgs hb{&m->cls_head, w.G, B, k, true, false, s, head_tc(flags)};
                head_backward(hb, w.cls_h, g->cls_head, w.dG);
                dG = w.dG;
            }
            TowerArgs tb{&m->trunk, x, w.stn_h.out, B, N, false, true, true, s, want_tc(flags)};
            run_tower_bwd(tb, w.trunk_t, g->trunk, dG, w.dT, flags);
            launch(k_add_opt, grid1d((size_t)B * 9, 128), dim3(128), 0, s, (const float*)w.dT, dtrans, w.stn_h.dO, (size_t)B * 9);
        }
    } else {
        cudaMemcpyAsync(w.stn_h.dO, dtrans, (size_t)B * 9 * sizeof(float), cudaMemcpyDeviceToDevice, s);
    }
    if (do_stn) {
        HeadArgs ha{&m->stn_head, w.g_stn, B, 9, true, true, s, head_tc(flags)};
        head_backward(ha, w.stn_h, g->stn_head, w.dg_stn);
        TowerArgs ta{&m->stn_tower, x, nullptr, B, N, true, true, true, s, want_tc(flags)};
        run_tower_bwd(ta, w.stn_t, g->stn_tower, w.dg_stn, nullptr, flags);
    }
    return check_cuda("pgpd_backward");
}

// ---- tower-level entry points -------------------------------------------------------------------------
static void plan_tower_only(void* base, int B, int N, int flags, TowerWs& w, size_t& bytes) {
    Carver c(base);
    plan_tower(c, w, B, N);
    plan_tower_scratch(c, w, B, N, (flags & PGPD_F_SAVE) != 0);
    bytes = (c.off + 255) & ~(size_t)255;
}

size_t pgpd_tower_workspace_bytes(int B, int N, int flags) {
    if (B < 1 || N < 1) return 0;
    TowerWs w; size_t bytes;
    plan_tower_only(nullptr, B, N, flags, w, bytes);
    return bytes;
}

int pgpd_tower_forward(const pgpd_tower* t, const float* x, const float* trans, int B, int N,
                       int relu_last, int flags, float* pooled,
                       void* workspace, size_t workspace_bytes, void* stream) {
    if (!t || !x || !pooled) return fail(PGPD_E_ARG, "null pointer");
    for (int i = 0; i < 3; ++i) if ((uintptr_t)t->conv[i].w & 15) return fail(PGPD_E_ARG, "conv weight pointers must be 16-byte aligned");
    if (B < 1 || N < 1) return fail(PGPD_E_ARG, "B and N must be >= 1");
    if ((long long)B * N > 0x7fffffffLL / 128) return fail(PGPD_E_ARG, "B*N too large");
    const bool train = (flags & PGPD_F_TRAIN) != 0;
    if (train && (long long)B * N == 1) return fail(PGPD_E_BATCH1, "one value per channel in training mode");
    TowerWs w; size_t need;
    plan_tower_only(nullptr, B, N, flags, w, need);
    if (!workspace || ((uintptr_t)workspace & 255)) return fail(PGPD_E_WORKSPACE, "workspace null or misaligned");
    if (workspace_bytes < need) return fail(PGPD_E_WORKSPACE, "workspace too small");
    plan_tower_only(workspace, B, N, flags, w, need);
    TowerArgs a{t, x, trans, B, N, relu_last != 0, train, (flags & PGPD_F_SAVE) != 0, (cudaStream_t)stream, want_tc(flags)};
    run_tower_fwd(a, w, pooled, flags);
    return check_cuda("pgpd_tower_forward");
}

int pgpd_tower_backward(const pgpd_tower* t, const pgpd_tower_grad* g, const float* x,
                        const float* trans, int B, int N, int relu_last, int flags,
                        const float* dpooled, float* dtrans_out,
                        void* workspace, size_t workspace_bytes, void* stream) {
    if (!t || !g || !x || !dpooled) return fail(PGPD_E_ARG, "null pointer");
    for (int i = 0; i < 3; ++i) if ((uintptr_t)t->conv[i].w & 15) return fail(PGPD_E_ARG, "conv weight pointers must be 16-byte aligned");
    if (B < 1 || N < 1) return fail(PGPD_E_ARG, "B and N must be >= 1");
    if ((long long)B * N > 0x7fffffffLL / 128) return fail(PGPD_E_ARG, "B*N too large for this build (B*N*128 must fit in int32)");
    if (!(flags & PGPD_F_TRAIN)) return fail(PGPD_E_UNSUPPORTED, "backward through eval-mode BatchNorm is not implemented");
    if (trans && !dtrans_out) return fail(PGPD_E_ARG, "dtrans_out is null but trans is given");
    flags |= PGPD_F_SAVE;
    TowerWs w; size_t need;
    plan_tower_only(nullptr, B, N, flags, w, need);
    if (!workspace || ((uintptr_t)workspace & 255)) return fail(PGPD_E_WORKSPACE, "workspace null or misaligned");
    if (workspace_bytes < need) return fail(PGPD_E_WORKSPACE, "workspace too small");
    plan_tower_only(workspace, B, N, flags, w, need);
    TowerArgs a{t, x, trans, B, N, relu_last != 0, true, true, (cudaStream_t)stream, want_tc(flags)};
    run_tower_bwd(a, w, *g, dpooled, dtrans_out, flags);
    return check_cuda("pgpd_tower_backward");
}

// ---- GPDClassifier (SURVEY.md section 8f row 4) ---------------------------------------------------------------------
size_t pgpd_gpd_workspace_bytes(int B, int C, int flags) {
    if (B < 1 || C < 1) return 0;
    GpdWs w;
    plan_gpd(nullptr, B, (flags & PGPD_F_SAVE) != 0, w);
    return w.bytes;
}

static int gpd_check(const pgpd_gpd* m, const float* x, int B, int C, const void* ws, size_t ws_bytes, size_t need) {
    if (!m || !x) return fail(PGPD_E_ARG, "null model or input pointer");
    if (B < 1 || C < 1 || C > 64) return fail(PGPD_E_ARG, "B must be >= 1 and C in [1,64]");
    if ((long long)B * GPD_FLAT > 0x7fffffffLL) return fail(PGPD_E_ARG, "B too large");
    if (!m->conv1.w || !m->conv2.w || !m->fc1.w || !m->fc2.w || !m->conv1.b || !m->conv2.b || !m->fc1.b || !m->fc2.b)
        return fail(PGPD_E_ARG, "null weight pointer");
    if ((uintptr_t)m->fc1.w & 15) return fail(PGPD_E_ARG, "fc1 weight pointer must be 16-byte aligned");
    if (!ws || ((uintptr_t)ws & 255)) return fail(PGPD_E_WORKSPACE, "workspace is null or not 256-byte aligned");
    if (ws_bytes < need) return fail(PGPD_E_WORKSPACE, "workspace too small (see pgpd_gpd_workspace_bytes)");
    return PGPD_OK;
}

int pgpd_gpd_forward(const pgpd_gpd* m, const float* x, int B, int C, int flags, float* logp,
                     void* workspace, size_t workspace_bytes, void* stream) {
    GpdWs w;
    plan_gpd(nullptr, B < 1 ? 1 : B, (flags & PGPD_F_SAVE) != 0, w);
    int rc = gpd_check(m, x, B, C, workspace, workspace_bytes, w.bytes);
    if (rc) return rc;
    if (!logp) return fail(PGPD_E_ARG, "logp output pointer is null");
    plan_gpd(workspace, B, (flags & PGPD_F_SAVE) != 0, w);
    GpdArgs a{m, x, B, C, (cudaStream_t)stream, want_tc(flags)};
    gpd_forward(a, w, logp);
    return check_cuda("pgpd_gpd_forward");
}

int pgpd_gpd_backward(const pgpd_gpd* m, const pgpd_gpd_grad* g, const float* x, int B, int C, int flags,
                      const float* dlogp, void* workspace, size_t workspace_bytes, void* stream) {
    GpdWs w;
    plan_gpd(nullptr, B < 1 ? 1 : B, true, w);
    int rc = gpd_check(m, x, B, C, workspace, workspace_bytes, w.bytes);
    if (rc) return rc;
    if (!g || !dlogp) return fail(PGPD_E_ARG, "null gradient struct or dlogp");
    plan_gpd(workspace, B, true, w);
    GpdArgs a{m, x, B, C, (cudaStream_t)stream, want_tc(flags)};
    gpd_backward(a, w, *g, dlogp);
    return check_cuda("pgpd_gpd_backward");
}

// ---- the dual-cloud network (SURVEY.md section 8f row 4; csrc/dual.cuh) ----------------------------------------------------------
static int dual_check(int what, const pgpd_dual* m, const float* x, int B, int N, int k, const void* ws, size_t ws_bytes, size_t need) {
    if (what != PGPD_DUAL_STN && what != PGPD_DUAL_FEAT && what != PGPD_DUAL_CLS)
        return fail(PGPD_E_ARG, "what must be PGPD_DUAL_STN, PGPD_DUAL_FEAT or PGPD_DUAL_CLS");
    if (!m || !x) return fail(PGPD_E_ARG, "null model or input pointer");
    if (B < 1 || N < 1) return fail(PGPD_E_ARG, "B and N must be >= 1");
    if (what == PGPD_DUAL_CLS && (k < 1 || k > 1024)) return fail(PGPD_E_ARG, "k must be in [1,1024]");
    if ((long long)B * N > 0x7fffffffLL / 1024) return fail(PGPD_E_ARG, "B*N too large for this build (B*N*1024 must fit in int32)");
    if (!ws || ((uintptr_t)ws & 255)) return fail(PGPD_E_WORKSPACE, "workspace is null or not 256-byte aligned");
    if (ws_bytes < need) return fail(PGPD_E_WORKSPACE, "workspace too small (see pgpd_dual_workspace_bytes)");
    return PGPD_OK;
}

size_t pgpd_dual_workspace_bytes(int what, int B, int N, int k, int flags) {
    if (B < 1 || N < 1) return 0;
    dual::DualWs w;
    dual::plan_dual(nullptr, what, B, N, k < 1 ? 1 : k, (flags & PGPD_F_SAVE) != 0, w);
    return w.bytes;
}

int pgpd_dual_forward(int what, const pgpd_dual* m, const float* x, int B, int N, int k, int flags,
                      float* out, float* trans, void* workspace, size_t workspace_bytes, void* stream) {
    dual::DualWs w;
    const bool save = (flags & PGPD_F_SAVE) != 0;
    dual::plan_dual(nullptr, what, B < 1 ? 1 : B, N < 1 ? 1 : N, k < 1 ? 1 : k, save, w);
    int rc = dual_check(what, m, x, B, N, k, workspace, workspace_bytes, w.bytes);
    if (rc) return rc;
    if (!trans) return fail(PGPD_E_ARG, "trans output pointer is null");
    if (what != PGPD_DUAL_STN && !out) return fail(PGPD_E_ARG, "out pointer is null");
    const bool train = (flags & PGPD_F_TRAIN) != 0;
    if (train && B == 1)
        return fail(PGPD_E_BATCH1, "Expected more than 1 value per channel when training (BatchNorm over a batch of 1)");
    dual::plan_dual(workspace, what, B, N, k, save, w);
    dual::dual_forward(what, *m, x, B, N, k, train, out, trans, w, (cudaStream_t)stream);
    return check_cuda("pgpd_dual_forward");
}

int pgpd_dual_backward(int what, const pgpd_dual* m, const pgpd_dual_grad* g, const float* x, int B, int N, int k, int flags,
                       const float* dout, const float* dtrans, void* workspace, size_t workspace_bytes, void* stream) {
    dual::DualWs w;
    dual::plan_dual(nullptr, what, B < 1 ? 1 : B, N < 1 ? 1 : N, k < 1 ? 1 : k, true, w);
    int rc = dual_check(what, m, x, B, N, k, workspace, workspace_bytes, w.bytes);
    if (rc) return rc;
    if (!g) return fail(PGPD_E_ARG, "null gradient struct");
    if (!(flags & PGPD_F_TRAIN)) return fail(PGPD_E_UNSUPPORTED, "backward through eval-mode BatchNorm is not implemented");
    if (what != PGPD_DUAL_STN && !dout) return fail(PGPD_E_ARG, "dout is null");
    if (what == PGPD_DUAL_STN && !dtrans) return fail(PGPD_E_ARG, "dtrans is null");
    if (B == 1) return fail(PGPD_E_BATCH1, "batch of 1 in training mode");
    dual::plan_dual(workspace, what, B, N, k, true, w);
    dual::dual_backward(what, *m, *g, x, B, N, k, dout, dtrans, w, (cudaStream_t)stream);
    return check_cuda("pgpd_dual_backward");
}

// ---- data preparation in front of the model (SURVEY.md section 8f rows 1-2) ---------------------------------------
int pgpd_crop_box(const float* pc, int P, const double* frames, int G, const int* offsets, int* counts,
                  float* out_pts, int* out_idx, void* stream) {
    if (!pc || !frames || P < 0 || G < 1) return fail(PGPD_E_ARG, "bad argument");
    if (!counts && !(out_pts && out_idx && offsets)) return fail(PGPD_E_ARG, "need counts, or offsets + out_pts + out_idx");
    if ((out_pts == nullptr) != (out_idx == nullptr)) return fail(PGPD_E_ARG, "out_pts and out_idx go together");
    launch(k_crop_box, dim3(G), dim3(256), 0, (cudaStream_t)stream, pc, P, frames, offsets, counts, out_pts, out_idx);
    return check_cuda("pgpd_crop_box");
}

int pgpd_resample(const float* pts, const int* offsets, int C, int N, int repeat, unsigned long long seed,
                  float* out_x, int* out_idx, void* stream) {
    if (!pts || !offsets || !out_x || C < 1 || N < 1 || repeat < 1) return fail(PGPD_E_ARG, "bad argument");
    launch(k_resample, dim3(C, repeat), dim3(256), 0, (cudaStream_t)stream, pts, offsets, N, seed, out_x, out_idx);
    return check_cuda("pgpd_resample");
}

size_t pgpd_gpd_project_workspace_bytes(int P, int G, int total_in_box, int chann) {
    if (P < 0 || G < 1 || total_in_box < 0 || (chann != 3 && chann != 12)) return 0;
    proj::ProjWs w;
    proj::plan_project(nullptr, P, total_in_box, chann, w);
    return w.bytes;
}

int pgpd_gpd_project(const float* pc, int P, const double* frames, int G, const int* offsets, const int* idx, int chann,
                     float* out, unsigned char* valid, void* workspace, size_t workspace_bytes, void* stream) {
    if (!pc || !frames || !offsets || !out || !valid || P < 0 || G < 1) return fail(PGPD_E_ARG, "bad argument");
    if (chann != 3 && chann != 12) return fail(PGPD_E_ARG, "chann must be 3 or 12");
    if (!workspace || ((uintptr_t)workspace & 255)) return fail(PGPD_E_WORKSPACE, "workspace is null or not 256-byte aligned");
    const int cap = proj::project_capacity(workspace_bytes, P, chann);
    if (cap < 0) return fail(PGPD_E_WORKSPACE, "workspace too small (see pgpd_gpd_project_workspace_bytes)");
    if (cap > 0 && !idx) return fail(PGPD_E_ARG, "idx is null");
    proj::ProjWs w;
    proj::plan_project(workspace, P, cap, chann, w);
    proj::project(pc, P, frames, G, offsets, idx, cap, chann, out, valid, w, (cudaStream_t)stream);
    return check_cuda("pgpd_gpd_project");
}

}  // extern "C"
