// capi.cu -- extern "C" entry points of libomni_b200.so (declared in include/omni_b200.h).
#include <stdlib.h>
#include "omni_internal.cuh"
#include "fast_kernels.cuh"
#include "fast_device.cuh"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

static thread_local char g_err[512] = "";

void omni_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *omni_last_error_string(void) { return g_err; }
extern "C" int omni_version(void) { return OMNI_ABI_VERSION; }

extern "C" int omni_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ---- context -----------------------------------------------------------------------------------
extern "C" int omni_ctx_create(int device, omni_ctx **out)
{
    OMNI_REQUIRE(out != nullptr, "omni_ctx_create: out is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        omni_set_error("no CUDA device available (%s); libomni_b200 has no CPU fallback",
                       e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        cudaGetLastError();
        return OMNI_ERR_CUDA;
    }
    OMNI_REQUIRE(device >= 0 && device < n, "omni_ctx_create: device %d out of range [0,%d)", device, n);
    OMNI_CUDA(cudaSetDevice(device));
    omni_ctx *c = new omni_ctx();
    c->device = device;
    {   // A/B switch for measurements only: both edge kernels are bit-identical (tests run both)
        const char *ev = getenv("OMNI_B200_EDGE_DENSE");
        c->edge_sparse = (ev && ev[0] == '1') ? 0 : 1;
        ev = getenv("OMNI_B200_ASSIGN_LABCELL");
        c->assign_rgbcell = (ev && ev[0] == '1') ? 0 : 1;
        ev = getenv("OMNI_B200_DENSE_PIPELINE");
        c->pipeline = (ev && ev[0] == '1') ? 0 : 1;
    }
    OMNI_CUDA(cudaMalloc(&c->d_flags, 64 * sizeof(int)));
    OMNI_CUDA(cudaMemset(c->d_flags, 0, 64 * sizeof(int)));
    OMNI_CUDA(cudaMalloc(&c->d_counts, 4 * OMNI_MAX_K * sizeof(unsigned long long)));
    OMNI_CUDA(cudaHostAlloc(&c->h_flags, 64 * sizeof(int), cudaHostAllocDefault));
    OMNI_CUDA(cudaHostAlloc(&c->h_counts, 4 * OMNI_MAX_K * sizeof(unsigned long long), cudaHostAllocDefault));
    OMNI_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    OMNI_CUDA(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device));
    *out = c;
    return OMNI_OK;
}

extern "C" int omni_ctx_destroy(omni_ctx *c)
{
    if (!c) return OMNI_OK;
    cudaSetDevice(c->device);
    for (int i = 0; i < OMNI_WS_SLOTS; i++) if (c->ws[i]) cudaFree(c->ws[i]);
    for (auto &kv : c->resize_tabs) if (kv.second.d_blob) cudaFree(kv.second.d_blob);
    if (c->d_flags) cudaFree(c->d_flags);
    if (c->d_rgb_boxes) cudaFree(c->d_rgb_boxes);
    if (c->d_rgb_boxes3) cudaFree(c->d_rgb_boxes3);
    if (c->d_counts) cudaFree(c->d_counts);
    if (c->h_flags) cudaFreeHost(c->h_flags);
    if (c->h_counts) cudaFreeHost(c->h_counts);
    if (c->stream) cudaStreamDestroy(c->stream);
    for (auto &r : c->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto e : c->ev_pool) cudaEventDestroy(e);
    fast_ctx_release(c);
    if (c->pk_ready) {
        cudaStreamDestroy(c->pk_in); cudaStreamDestroy(c->pk_out);
        for (auto e : c->pk_ev) cudaEventDestroy(e);
    }
    if (c->pk_counts) cudaFreeHost(c->pk_counts);
    if (c->bd_ready) { for (auto e : c->bd_ev) cudaEventDestroy(e); cudaStreamDestroy(c->bd_tail); }
    if (c->band_helper) omni_ctx_destroy(c->band_helper);
    delete c;
    return OMNI_OK;
}

extern "C" int omni_set_fast_path(omni_ctx *ctx, int enable)
{
    OMNI_REQUIRE(ctx != nullptr, "omni_set_fast_path: ctx is NULL");
    ctx->fast = enable ? 1 : 0;
    if (enable) {
        ctx->edge_sparse = ctx->assign_rgbcell = (enable == 2) ? 0 : 1;
        ctx->pipeline = (enable == 1) ? 1 : 0;
    }
    return OMNI_OK;
}

extern "C" int omni_set_assume_binary_masks(omni_ctx *ctx, int enable)
{
    OMNI_REQUIRE(ctx != nullptr, "omni_set_assume_binary_masks: ctx is NULL");
    ctx->assume_binary = enable ? 1 : 0;
    return OMNI_OK;
}

extern "C" int omni_set_table_cache(omni_ctx *ctx, int enable)
{
    OMNI_REQUIRE(ctx != nullptr, "omni_set_table_cache: ctx is NULL");
    ctx->table_cache = enable ? 1 : 0;
    if (!enable) ctx->cells_valid = ctx->cells3_valid = 0;
    return OMNI_OK;
}

extern "C" int omni_set_host_bands(omni_ctx *ctx, int mode)
{
    OMNI_REQUIRE(ctx != nullptr, "ctx is NULL");
    OMNI_REQUIRE(mode >= 0 && mode <= 2, "omni_set_host_bands: mode must be 0, 1 or 2");
    ctx->host_bands = mode;
    return OMNI_OK;
}

extern "C" int omni_last_band_resends(omni_ctx *ctx) { return ctx ? ctx->last_band_resends : -1; }

extern "C" int omni_host_alloc(size_t bytes, void **out)
{
    OMNI_REQUIRE(out != nullptr, "omni_host_alloc: out is NULL");
    OMNI_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return OMNI_OK;
}

extern "C" int omni_host_free(void *p)
{
    if (p) OMNI_CUDA(cudaFreeHost(p));
    return OMNI_OK;
}

extern "C" int omni_last_hysteresis_passes(omni_ctx *ctx)
{
    if (!ctx) return 0;
    if (ctx->last_hyst_passes < 0) {              // the bit-plane kernel leaves its round count in d_flags[0]
        // read on the stream the kernel ran on, then wait for it (the legacy stream does not order against non-blocking streams)
        cudaStream_t st = ctx->last_hyst_stream;
        if (cudaSetDevice(ctx->device) != cudaSuccess ||
            cudaMemcpyAsync(ctx->h_flags + 9, ctx->d_flags, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess) {
            cudaGetLastError();
            return 0;
        }
        ctx->last_hyst_passes = ctx->h_flags[9];
    }
    return ctx->last_hyst_passes;
}

// ---- launch accounting / per-kernel timing ----------------------------------------------------------
KScope::KScope(omni_ctx *ctx, const char *name, cudaStream_t s) : c(ctx), st(s)
{
    if (!c) return;                       // unscoped launch (the caller brackets it)
    c->launches++;
    if (!c->prof_on) return;
    cudaEvent_t a = nullptr;
    for (cudaEvent_t *e : {&a, &b}) {
        if (!c->ev_pool.empty()) { *e = c->ev_pool.back(); c->ev_pool.pop_back(); }
        else if (cudaEventCreate(e) != cudaSuccess) { cudaGetLastError(); *e = nullptr; }
    }
    if (!a || !b) { b = nullptr; return; }
    cudaEventRecord(a, st);
    c->prof.push_back({name, a, b});
}
KScope::~KScope() { if (b) cudaEventRecord(b, st); }

extern "C" long long omni_launch_count(omni_ctx *ctx) { return ctx ? ctx->launches : 0; }

static void prof_recycle(omni_ctx *ctx)
{
    for (auto &r : ctx->prof) { ctx->ev_pool.push_back(r.a); ctx->ev_pool.push_back(r.b); }
    ctx->prof.clear();
}

extern "C" int omni_profile_enable(omni_ctx *ctx, int on)
{
    OMNI_REQUIRE(ctx != nullptr, "omni_profile_enable: ctx is NULL");
    OMNI_CUDA(cudaSetDevice(ctx->device));
    OMNI_CUDA(cudaDeviceSynchronize());
    prof_recycle(ctx);
    ctx->prof_on = on ? 1 : 0;
    return OMNI_OK;
}

// Text table "name\tlaunches\ttotal_ms\n" per kernel name, in first-launch order; clears the records.
extern "C" int omni_profile_summary(omni_ctx *ctx, char *buf, size_t buflen)
{
    OMNI_REQUIRE(ctx != nullptr && buf != nullptr && buflen > 0, "omni_profile_summary: bad arguments");
    OMNI_CUDA(cudaSetDevice(ctx->device));
    OMNI_CUDA(cudaDeviceSynchronize());
    std::vector<std::tuple<const char *, long, double>> agg;
    for (auto &r : ctx->prof) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) { cudaGetLastError(); ms = 0.f; }
        size_t i = 0;
        for (; i < agg.size(); i++) if (!strcmp(std::get<0>(agg[i]), r.name)) break;
        if (i == agg.size()) agg.emplace_back(r.name, 0L, 0.0);
        std::get<1>(agg[i])++; std::get<2>(agg[i]) += ms;
    }
    prof_recycle(ctx);
    size_t o = 0; buf[0] = 0;
    for (auto &a : agg) {
        int n = snprintf(buf + o, buflen - o, "%s\t%ld\t%.6f\n", std::get<0>(a), std::get<1>(a), std::get<2>(a));
        if (n < 0 || (size_t)n >= buflen - o) break;
        o += (size_t)n;
    }
    return OMNI_OK;
}

int omni_ws_reserve(omni_ctx *ctx, int slot, size_t bytes)
{
    if (ctx->ws_bytes[slot] >= bytes) return OMNI_OK;
    // the candidate tables of both cache generations live in slot 5: a new allocation holds none of them (it may even come back
    // at the old address, so no pointer comparison can tell)
    if (slot == 5) ctx->cells_valid = ctx->cells3_valid = 0;
    if (ctx->ws[slot]) { OMNI_CUDA(cudaFree(ctx->ws[slot])); ctx->ws[slot] = nullptr; ctx->ws_bytes[slot] = 0; }
    size_t want = bytes + bytes / 8;
    cudaError_t e = cudaMalloc(&ctx->ws[slot], want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        omni_set_error("workspace slot %d: cudaMalloc(%zu) failed: %s", slot, want, cudaGetErrorString(e));
        return OMNI_ERR_NOMEM;
    }
    ctx->ws_bytes[slot] = want;
    return OMNI_OK;
}

// ---- host-side parameter preparation --------------------------------------------------------------
// cv2.getStructuringElement(MORPH_RECT | MORPH_ELLIPSE, (k,k)) as one span per row (SURVEY A.0).
void omni_build_se(int shape_ellipse, int k, MorphSE *se)
{
    int r = k / 2, c = k / 2, a = k / 2;
    double inv_r2 = r ? 1.0 / ((double)r * r) : 0.0;
    se->k = k;
    for (int i = 0; i < k; i++) {
        int j1 = 0, j2 = 0;
        if (!shape_ellipse) j2 = k;
        else {
            int dy = i - r;
            if (abs(dy) <= r) {
                int dx = (int)lrint(c * sqrt((r * r - dy * dy) * inv_r2));
                j1 = c - dx > 0 ? c - dx : 0;
                j2 = c + dx + 1 < k ? c + dx + 1 : k;
            }
        }
        se->x0[i] = (int8_t)(j1 - a);                  // |j - a| <= 127 for k <= 255
        se->x1[i] = (int8_t)(j2 - 1 - a);
    }
}

// OpenCV's computeResizeAreaTab (double arithmetic on the host, float weights) -- SURVEY A.1(iii).
static void area_tab(int ssize, int dsize, double scale, std::vector<int> &ofs, std::vector<int> &si, std::vector<float> &al)
{
    ofs.assign(1, 0);
    for (int dx = 0; dx < dsize; dx++) {
        double fsx1 = dx * scale, fsx2 = fsx1 + scale;
        double cw = scale < ssize - fsx1 ? scale : ssize - fsx1;
        int sx1 = (int)ceil(fsx1), sx2 = (int)floor(fsx2);
        if (sx2 > ssize - 1) sx2 = ssize - 1;
        if (sx1 > sx2) sx1 = sx2;
        if (sx1 - fsx1 > 1e-3) { si.push_back(sx1 - 1); al.push_back((float)((sx1 - fsx1) / cw)); }
        for (int sx = sx1; sx < sx2; sx++) { si.push_back(sx); al.push_back((float)(1.0 / cw)); }
        if (fsx2 - sx2 > 1e-3) {
            double a = fsx2 - sx2; if (a > 1.0) a = 1.0; if (a > cw) a = cw;
            si.push_back(sx2); al.push_back((float)(a / cw));
        }
        ofs.push_back((int)si.size());
    }
}

const ResizeTab *omni_get_resize_tab(omni_ctx *ctx, int sh, int sw, int dh, int dw, cudaStream_t st)
{
    auto key = std::make_tuple(sh, sw, dh, dw);
    auto it = ctx->resize_tabs.find(key);
    if (it != ctx->resize_tabs.end()) return &it->second;
    std::vector<int> xo, xs, yo, ys;
    std::vector<float> xa, ya;
    area_tab(sw, dw, (double)sw / dw, xo, xs, xa);
    area_tab(sh, dh, (double)sh / dh, yo, ys, ya);
    size_t n_int = xo.size() + xs.size() + yo.size() + ys.size(), n_f = xa.size() + ya.size();
    std::vector<int> blob(n_int + n_f);
    size_t o = 0, o_xo = o; memcpy(&blob[o], xo.data(), xo.size() * 4); o += xo.size();
    size_t o_xs = o; memcpy(&blob[o], xs.data(), xs.size() * 4); o += xs.size();
    size_t o_yo = o; memcpy(&blob[o], yo.data(), yo.size() * 4); o += yo.size();
    size_t o_ys = o; memcpy(&blob[o], ys.data(), ys.size() * 4); o += ys.size();
    size_t o_xa = o; memcpy(&blob[o], xa.data(), xa.size() * 4); o += xa.size();
    size_t o_ya = o; memcpy(&blob[o], ya.data(), ya.size() * 4); o += ya.size();
    ResizeTab t;
    if (cudaMalloc(&t.d_blob, blob.size() * 4) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    // synchronous copy from pageable memory (tables are built once per geometry and cached); the device-wide wait makes the
    // bytes visible to `st` whatever its flags (the legacy stream does not order against non-blocking streams)
    if (cudaMemcpy(t.d_blob, blob.data(), blob.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {
        cudaGetLastError(); cudaFree(t.d_blob); return nullptr;
    }
    (void)st;
    const int *b = (const int *)t.d_blob;
    t.dev.xofs = b + o_xo; t.dev.xsi = b + o_xs; t.dev.yofs = b + o_yo; t.dev.ysi = b + o_ys;
    t.dev.xal = (const float *)(b + o_xa); t.dev.yal = (const float *)(b + o_ya);
    auto ins = ctx->resize_tabs.emplace(key, t);
    return &ins.first->second;
}

static int set_device(omni_ctx *ctx)
{
    OMNI_REQUIRE(ctx != nullptr, "ctx is NULL");
    OMNI_CUDA(cudaSetDevice(ctx->device));
    return OMNI_OK;
}
#define OMNI_TRY(expr) do { int rc__ = (expr); if (rc__ != OMNI_OK) return rc__; } while (0)

// slots the fused device-resident calls use for this geometry, before the growth slack of omni_ws_reserve
static void fused_ws_plan(int h, int w, int K, int ksize, int nf, size_t out[OMNI_WS_SLOTS])
{
    for (int i = 0; i < OMNI_WS_SLOTS; i++) out[i] = 0;
    label_ws_bytes(h, w, K, nf, out);
    dense_ws_bytes(h, w, K, nf, ksize, out);
}

extern "C" size_t omni_workspace_bytes(int h, int w, int K, int ksize, int n_frames)
{
    if (h <= 0 || w <= 0 || K < 1 || K > OMNI_MAX_K || n_frames < 1 || n_frames * K > OMNI_MAX_K) return 0;
    size_t plan[OMNI_WS_SLOTS], total = 0;
    fused_ws_plan(h, w, K, ksize, n_frames, plan);
    for (int i = 0; i < OMNI_WS_SLOTS; i++) total += plan[i] + plan[i] / 8;
    return total;
}

extern "C" int omni_ctx_reserve(omni_ctx *ctx, int h, int w, int K, int ksize, int n_frames)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(h > 0 && w > 0 && K >= 1 && K <= OMNI_MAX_K && n_frames >= 1 && n_frames * K <= OMNI_MAX_K,
                 "omni_ctx_reserve: bad geometry (%d x %d, K=%d, %d frames)", w, h, K, n_frames);
    size_t plan[OMNI_WS_SLOTS];
    fused_ws_plan(h, w, K, ksize, n_frames, plan);
    for (int i = 0; i < OMNI_WS_SLOTS; i++)
        if (plan[i]) OMNI_TRY(omni_ws_reserve(ctx, i, plan[i]));
    // one-time objects of the fused path: constant tables, the centre-independent RGB-cell boxes
    OMNI_CUDA(fast_tables());
    OMNI_TRY(fast_rgb_boxes(ctx, ctx->stream));
    OMNI_CUDA(cudaStreamSynchronize(ctx->stream));
    return OMNI_OK;
}


// ---- stage 01 ----------------------------------------------------------------------------------------
extern "C" int omni_resize_area_u8c3(omni_ctx *ctx, const uint8_t *d_src, int sh, int sw, size_t spitch,
                                     uint8_t *d_dst, int dh, int dw, size_t dpitch, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_src && d_dst, "omni_resize_area_u8c3: NULL image pointer");
    OMNI_REQUIRE(sh > 0 && sw > 0 && dh > 0 && dw > 0 && dh <= sh && dw <= sw,
                 "omni_resize_area_u8c3: INTER_AREA shrink only, got %dx%d -> %dx%d", sw, sh, dw, dh);
    OMNI_REQUIRE(spitch >= (size_t)sw * 3 && dpitch >= (size_t)dw * 3, "omni_resize_area_u8c3: pitch smaller than a row");
    cudaStream_t st = (cudaStream_t)stream;
    double scx = (double)sw / dw, scy = (double)sh / dh;
    long isx = lrint(scx), isy = lrint(scy);
    bool fast = fabs(scx - isx) < 2.220446049250313e-16 && fabs(scy - isy) < 2.220446049250313e-16;
    if (fast) {
        if (ctx->fast && isx == 2 && isy == 2 && fast_resize_2x_ok(d_src, sw, spitch, d_dst, dw, dpitch))
            OMNI_LAUNCH(ctx, st, "resize_2x_v", fast_resize_2x(d_src, spitch, d_dst, dh, dw, dpitch, st));
        else
            OMNI_LAUNCH(ctx, st, "resize_area", g_resize_area(d_src, sh, sw, spitch, d_dst, dh, dw, dpitch, nullptr, st));
    } else {
        const ResizeTab *t = omni_get_resize_tab(ctx, sh, sw, dh, dw, st);
        if (!t) { omni_set_error("omni_resize_area_u8c3: cannot build resize tables"); return OMNI_ERR_NOMEM; }
        bool done = false;
        if (ctx->fast == 1 && ctx->pipeline == 1) {    // default family: TMA-staged separable kernel
            KScope ks(ctx, "resize_frac_tma", st);
            cudaError_t e = tma_resize_frac(d_src, sh, sw, spitch, d_dst, dh, dw, dpitch, &t->dev, st);
            if (e == cudaSuccess) done = true;
            else if (e != cudaErrorNotSupported) OMNI_CUDA(e);
            else ctx->launches--;                      // nothing was launched
        }
        if (!done && ctx->fast) {
            KScope ks(ctx, "resize_frac_v", st);
            cudaError_t e = fast_resize_frac(d_src, sh, sw, spitch, d_dst, dh, dw, dpitch, &t->dev, st);
            if (e == cudaSuccess) done = true;
            else if (e != cudaErrorNotSupported) OMNI_CUDA(e);
            else ctx->launches--;                      // nothing was launched
        }
        if (!done) OMNI_LAUNCH(ctx, st, "resize_area", g_resize_area(d_src, sh, sw, spitch, d_dst, dh, dw, dpitch, &t->dev, st));
    }
    return OMNI_OK;
}

// ---- stage 02 ----------------------------------------------------------------------------------------
static int fill_assign(AssignParams *P, const float *h_centers, const uint8_t *h_pal, int K, const uint8_t *h_lut)
{
    OMNI_REQUIRE(K >= 1 && K <= OMNI_MAX_K, "K=%d outside [1,%d]", K, OMNI_MAX_K);
    memset(P, 0, sizeof(*P));
    P->K = K;
    for (int i = 0; i < 3 * K; i++) {
        if (h_centers) P->c[i] = h_centers[i];
        if (h_pal) P->pal[i] = h_pal[i];
    }
    for (int k = 0; k < K; k++) {
        P->lut[k] = h_lut ? h_lut[k] : (u8)k;
        OMNI_REQUIRE(P->lut[k] < OMNI_MAX_K, "lut[%d]=%d out of range", k, P->lut[k]);
    }
    return OMNI_OK;
}

extern "C" int omni_assign_lab_f32(omni_ctx *ctx, const uint8_t *d_bgr, int h, int w, size_t pitch,
                                   const float *h_centers, int K, const uint8_t *h_lut,
                                   uint8_t *d_labels, size_t lpitch, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_bgr && d_labels && h_centers, "omni_assign_lab_f32: NULL pointer");
    OMNI_REQUIRE(h > 0 && w > 0 && pitch >= (size_t)w * 3 && lpitch >= (size_t)w, "omni_assign_lab_f32: bad geometry");
    AssignParams P;
    OMNI_TRY(fill_assign(&P, h_centers, nullptr, K, h_lut));
    if (ctx->fast) OMNI_LAUNCH(ctx, (cudaStream_t)stream, "assign", fast_assign(ctx, d_bgr, h, w, pitch, P, 1, d_labels, lpitch, (cudaStream_t)stream));
    else OMNI_LAUNCH(ctx, (cudaStream_t)stream, "assign", g_assign(d_bgr, h, w, pitch, P, 1, d_labels, lpitch, (cudaStream_t)stream));
    return OMNI_OK;
}

extern "C" int omni_assign_rgb_i16wrap(omni_ctx *ctx, const uint8_t *d_rgb, int h, int w, size_t pitch,
                                       const uint8_t *h_palette, int K, uint8_t *d_labels, size_t lpitch, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_rgb && d_labels && h_palette, "omni_assign_rgb_i16wrap: NULL pointer");
    OMNI_REQUIRE(h > 0 && w > 0 && pitch >= (size_t)w * 3 && lpitch >= (size_t)w, "omni_assign_rgb_i16wrap: bad geometry");
    AssignParams P;
    OMNI_TRY(fill_assign(&P, nullptr, h_palette, K, nullptr));
    if (ctx->fast) OMNI_LAUNCH(ctx, (cudaStream_t)stream, "assign", fast_assign(ctx, d_rgb, h, w, pitch, P, 0, d_labels, lpitch, (cudaStream_t)stream));
    else OMNI_LAUNCH(ctx, (cudaStream_t)stream, "assign", g_assign(d_rgb, h, w, pitch, P, 0, d_labels, lpitch, (cudaStream_t)stream));
    return OMNI_OK;
}

// generic: one-hot planes, then erode/dilate passes ping-ponging between the output and scratch
static int generic_layer_masks(omni_ctx *ctx, const uint8_t *d_labels, int h, int w, size_t lpitch, int K,
                               int open_iters, int close_iters, uint8_t *d_masks, size_t plane_stride, size_t mpitch,
                               cudaStream_t st)
{
    size_t wp = ((size_t)w + 15) & ~(size_t)15, wplane = wp * h;
    OMNI_TRY(omni_ws_reserve(ctx, 0, wplane * K));
    u8 *tmp = (u8 *)ctx->ws[0];
    OMNI_LAUNCH(ctx, st, "onehot", g_onehot(d_labels, h, w, lpitch, K, d_masks, plane_stride, mpitch, st));
    MorphSE se;
    omni_build_se(0, 3, &se);
    int oi = open_iters > 0 ? open_iters : 0, ci = close_iters > 0 ? close_iters : 0;
    // OPEN = erode^oi dilate^oi ; CLOSE = dilate^ci erode^ci
    int seq_n = 0, seq[4 * 64];
    OMNI_REQUIRE(oi <= 32 && ci <= 32, "morphology iterations too large");
    for (int i = 0; i < oi; i++) seq[seq_n++] = 0;
    for (int i = 0; i < oi; i++) seq[seq_n++] = 1;
    for (int i = 0; i < ci; i++) seq[seq_n++] = 1;
    for (int i = 0; i < ci; i++) seq[seq_n++] = 0;
    bool in_out = true;   // current data lives in d_masks
    for (int i = 0; i < seq_n; i++) {
        if (in_out) OMNI_LAUNCH(ctx, st, "morph", g_morph(d_masks, plane_stride, mpitch, tmp, wplane, wp, K, h, w, se, seq[i], st));
        else OMNI_LAUNCH(ctx, st, "morph", g_morph(tmp, wplane, wp, d_masks, plane_stride, mpitch, K, h, w, se, seq[i], st));
        in_out = !in_out;
    }
    if (!in_out) OMNI_CUDA(g_copy2d_planes(tmp, wplane, wp, d_masks, plane_stride, mpitch, K, h, w, st));
    return OMNI_OK;
}

extern "C" int omni_layer_masks(omni_ctx *ctx, const uint8_t *d_labels, int h, int w, size_t lpitch, int K,
                                int open_iters, int close_iters,
                                uint8_t *d_masks, size_t plane_stride, size_t mpitch, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_labels && d_masks, "omni_layer_masks: NULL pointer");
    OMNI_REQUIRE(K >= 1 && K <= OMNI_MAX_K, "omni_layer_masks: K=%d outside [1,%d]", K, OMNI_MAX_K);
    OMNI_REQUIRE(h > 0 && w > 0 && lpitch >= (size_t)w && mpitch >= (size_t)w && plane_stride >= mpitch * (size_t)(h - 1) + w,
                 "omni_layer_masks: bad geometry");
    cudaStream_t st = (cudaStream_t)stream;
    if (ctx->fast && fast_masks_supported(open_iters, close_iters))
        return fast_layer_masks(ctx, d_labels, h, w, lpitch, K, open_iters, close_iters, d_masks, plane_stride, mpitch, st);
    return generic_layer_masks(ctx, d_labels, h, w, lpitch, K, open_iters, close_iters, d_masks, plane_stride, mpitch, st);
}

// opt-in: the Lab centres of 02_color_extract.py:39-50 on the device (see kmeans.cu for the contract)
static int kmeans_checked(const char *fn, omni_ctx *ctx, const uint8_t *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                          const int32_t *h_sample_idx, int n_samples, int K, int attempts, int max_iter, double eps, uint64_t seed,
                          float *h_centers, double *h_compactness, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_bgr && h_centers, "%s: NULL pointer", fn);
    OMNI_REQUIRE(h > 0 && w > 0 && pitch >= (size_t)w * 3 && (long long)h * w < (1ll << 31), "%s: bad geometry", fn);
    OMNI_REQUIRE(n_frames >= 1 && (n_frames == 1 || frame_stride >= pitch * (size_t)(h - 1) + (size_t)w * 3),
                 "%s: %d frames, frame_stride %zu smaller than a frame", fn, n_frames, frame_stride);
    OMNI_REQUIRE(K >= 1 && K <= OMNI_MAX_K, "%s: K=%d outside [1,%d]", fn, K, OMNI_MAX_K);
    OMNI_REQUIRE(attempts >= 1 && attempts <= 64 && max_iter >= 1 && max_iter <= 1000 && eps >= 0.0, "%s: bad criteria", fn);
    const int n = h_sample_idx ? n_samples : h * w;
    OMNI_REQUIRE(n >= K && n <= (1 << 24), "%s: %d samples (need K <= n <= 2^24: integer accumulators)", fn, n);
    if (h_sample_idx)
        for (int i = 0; i < n; i++)
            OMNI_REQUIRE(h_sample_idx[i] >= 0 && h_sample_idx[i] < h * w, "%s: sample index %d out of range", fn, h_sample_idx[i]);
    return kmeans_lab_batch(ctx, d_bgr, n_frames, frame_stride, h, w, pitch, h_sample_idx, n, K, attempts, max_iter, (float)eps,
                            (unsigned long long)seed, h_centers, h_compactness, (cudaStream_t)stream);
}

extern "C" int omni_kmeans_lab(omni_ctx *ctx, const uint8_t *d_bgr, int h, int w, size_t pitch, const int32_t *h_sample_idx, int n_samples,
                               int K, int attempts, int max_iter, double eps, uint64_t seed, float *h_centers, double *h_compactness,
                               void *stream)
{
    return kmeans_checked("omni_kmeans_lab", ctx, d_bgr, 1, 0, h, w, pitch, h_sample_idx, n_samples, K, attempts, max_iter, eps, seed,
                          h_centers, h_compactness, stream);
}

extern "C" int omni_kmeans_lab_batch(omni_ctx *ctx, const uint8_t *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                                     const int32_t *h_sample_idx, int n_samples, int K, int attempts, int max_iter, double eps, uint64_t seed,
                                     float *h_centers, double *h_compactness, void *stream)
{
    return kmeans_checked("omni_kmeans_lab_batch", ctx, d_bgr, n_frames, frame_stride, h, w, pitch, h_sample_idx, n_samples, K, attempts,
                          max_iter, eps, seed, h_centers, h_compactness, stream);
}

// ---- stage 03 ----------------------------------------------------------------------------------------
static int check_edge_params(const omni_edge_params *p, BlurParams *bp, int *low, int *high)
{
    OMNI_REQUIRE(p != nullptr, "edge params NULL");
    OMNI_REQUIRE(p->morph_k >= 1 && p->morph_k <= OMNI_MAX_MORPH_K, "edge_morph_kernel=%d outside [1,%d]", p->morph_k, OMNI_MAX_MORPH_K);
    if (omni_gauss_weights(p->ksize, bp)) {
        omni_set_error("edge_kernel_size=%d: need an odd size in [3,%d] (apply _ensure_odd first)", p->ksize, OMNI_MAX_BLUR_K);
        return OMNI_ERR_UNSUPPORTED;
    }
    // cv2.Canny: swap if low > high, then floor both for the integer L1 magnitude (SURVEY A.5)
    double lo = p->low < p->high ? p->low : p->high, hi = p->low < p->high ? p->high : p->low;
    OMNI_REQUIRE(lo == lo && hi == hi, "Canny thresholds are NaN");
    lo = floor(lo); hi = floor(hi);
    *low = lo > 1e9 ? 1000000000 : lo < -1e9 ? -1000000000 : (int)lo;
    *high = hi > 1e9 ? 1000000000 : hi < -1e9 ? -1000000000 : (int)hi;
    return OMNI_OK;
}

// run hysteresis passes until one changes nothing (flag read back through pinned memory)
static int generic_hysteresis(omni_ctx *ctx, u8 *state, size_t plane, size_t pitch, int K, int h, int w, cudaStream_t st)
{
    int passes = 0;
    for (;;) {
        OMNI_CUDA(cudaMemsetAsync(ctx->d_flags, 0, sizeof(int), st));
        OMNI_LAUNCH(ctx, st, "hyst_pass", g_hyst_pass(state, plane, pitch, K, h, w, ctx->d_flags, st));
        OMNI_CUDA(cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, sizeof(int), cudaMemcpyDeviceToHost, st));
        OMNI_CUDA(cudaStreamSynchronize(st));
        passes++;
        if (!ctx->h_flags[0]) break;
        OMNI_REQUIRE(passes < 100000, "hysteresis did not converge");
    }
    ctx->last_hyst_passes = passes;
    OMNI_LAUNCH(ctx, st, "hyst_final", g_hyst_final(state, plane, pitch, K, h, w, st));
    return OMNI_OK;
}

// skip_morph: d_masks already holds the planes AFTER the stage-03 open/close (fast bit morphology wrote them)
static int generic_edges(omni_ctx *ctx, const uint8_t *d_masks, int K, int h, int w, size_t m_plane, size_t mpitch,
                         const omni_edge_params *prm, const BlurParams &bp, int low, int high,
                         uint8_t *d_edges, size_t e_plane, size_t epitch, cudaStream_t st, bool skip_morph = false)
{
    size_t wp = ((size_t)w + 15) & ~(size_t)15, wplane = wp * h;
    OMNI_TRY(omni_ws_reserve(ctx, 0, wplane * K));
    OMNI_TRY(omni_ws_reserve(ctx, 1, wplane * K));
    u8 *A = (u8 *)ctx->ws[0], *B = (u8 *)ctx->ws[1];
    MorphSE se;
    omni_build_se(1, prm->morph_k, &se);
    long long oi = prm->open_iters > 0 ? prm->open_iters : 0, ci = prm->close_iters > 0 ? prm->close_iters : 0;
    if (skip_morph) oi = ci = 0;
    // OPEN = erode^oi dilate^oi ; CLOSE = dilate^ci erode^ci (cv2 loops the iterations of a non-rectangular element)
    const long long n_steps = 2 * (oi + ci);
    const u8 *cur = d_masks; size_t cplane = m_plane, cpitch = mpitch;
    for (long long i = 0; i < n_steps; i++) {
        const int dilate = (i >= oi && i < 2 * oi + ci) ? 1 : 0;
        u8 *dst = (cur == A) ? B : A;
        OMNI_LAUNCH(ctx, st, "morph", g_morph(cur, cplane, cpitch, dst, wplane, wp, K, h, w, se, dilate, st));
        cur = dst; cplane = wplane; cpitch = wp;
    }
    u8 *bl = (cur == A) ? B : A;
    OMNI_LAUNCH(ctx, st, "blur", g_blur(cur, cplane, cpitch, bl, wplane, wp, K, h, w, bp, st));
    OMNI_LAUNCH(ctx, st, "canny_nms", g_canny_nms(bl, wplane, wp, d_edges, e_plane, epitch, K, h, w, low, high, st));
    return generic_hysteresis(ctx, d_edges, e_plane, epitch, K, h, w, st);
}

// masks (byte planes) -> edges with the best available kernels:
//   fast bit-plane path (edge_kernel_size 3 / 5 / 7) > fast bit morphology + generic blur/Canny (other sizes) > generic.
//   The bit morphology is fk_morph for morph_k 1 and 3 with at most one open / close, the ELLIPSE kernel of morph_ellipse.cu
//   for every other size and count; masks that are not strictly {0,255} take the generic kernels.
static int edges_dispatch(omni_ctx *ctx, const uint8_t *d_masks, int K, int h, int w, size_t m_plane, size_t mpitch,
                          const omni_edge_params *prm, const BlurParams &bp, int low, int high,
                          uint8_t *d_edges, size_t e_plane, size_t epitch, cudaStream_t st)
{
    if (ctx->fast && fast_edges_supported(prm)) {
        int rc = fast_edges(ctx, d_masks, K, h, w, m_plane, mpitch, prm, bp, low, high, d_edges, e_plane, epitch, st);
        if (rc != OMNI_ERR_UNSUPPORTED) return rc;       // non-binary masks fall through to the generic kernels
    } else if (ctx->fast && fast_morph03_supported(prm)) {
        size_t wp = ((size_t)w + 15) & ~(size_t)15, wplane = wp * h;
        OMNI_TRY(omni_ws_reserve(ctx, 0, wplane * K));
        OMNI_TRY(omni_ws_reserve(ctx, 1, wplane * K));
        u8 *m2 = (u8 *)ctx->ws[1];                       // generic_edges blurs from here into slot 0
        int rc = fast_morph03_bytes(ctx, d_masks, K, h, w, m_plane, mpitch, prm, m2, wplane, wp, st);
        if (rc == OMNI_OK)
            return generic_edges(ctx, m2, K, h, w, wplane, wp, prm, bp, low, high, d_edges, e_plane, epitch, st, true);
        if (rc != OMNI_ERR_UNSUPPORTED) return rc;
    }
    return generic_edges(ctx, d_masks, K, h, w, m_plane, mpitch, prm, bp, low, high, d_edges, e_plane, epitch, st);
}

extern "C" int omni_edges(omni_ctx *ctx, const uint8_t *d_masks, int K, int h, int w, size_t m_plane_stride, size_t mpitch,
                          const omni_edge_params *prm,
                          uint8_t *d_edges, size_t e_plane_stride, size_t epitch, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_masks && d_edges && d_masks != d_edges, "omni_edges: NULL or aliased planes");
    OMNI_REQUIRE(K >= 1 && K <= OMNI_MAX_K, "omni_edges: K=%d outside [1,%d]", K, OMNI_MAX_K);
    OMNI_REQUIRE(h > 0 && w > 0 && mpitch >= (size_t)w && epitch >= (size_t)w, "omni_edges: bad geometry");
    BlurParams bp; int low, high;
    OMNI_TRY(check_edge_params(prm, &bp, &low, &high));
    return edges_dispatch(ctx, d_masks, K, h, w, m_plane_stride, mpitch, prm, bp, low, high, d_edges, e_plane_stride, epitch,
                          (cudaStream_t)stream);
}

// ---- fused hot path -------------------------------------------------------------------------------------
extern "C" int omni_color_edge(omni_ctx *ctx, const uint8_t *d_bgr, int h, int w, size_t pitch,
                               const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                               uint8_t *d_labels, size_t lpitch,
                               uint8_t *d_masks, size_t m_plane_stride, size_t mpitch,
                               uint8_t *d_edges, size_t e_plane_stride, size_t epitch, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_bgr && d_masks && d_edges && h_centers, "omni_color_edge: NULL pointer");
    OMNI_REQUIRE(h > 0 && w > 0 && pitch >= (size_t)w * 3 && mpitch >= (size_t)w && epitch >= (size_t)w &&
                 (!d_labels || lpitch >= (size_t)w), "omni_color_edge: bad geometry");
    BlurParams bp; int low, high;
    OMNI_TRY(check_edge_params(prm, &bp, &low, &high));
    AssignParams P;
    OMNI_TRY(fill_assign(&P, h_centers, nullptr, K, h_lut));
    cudaStream_t st = (cudaStream_t)stream;
    if (ctx->fast && fast_fused_supported(prm)) {
        int rc = fast_color_edge(ctx, d_bgr, h, w, pitch, P, prm, bp, low, high, d_labels, lpitch,
                                 d_masks, m_plane_stride, mpitch, d_edges, e_plane_stride, epitch, st);
        if (rc != OMNI_ERR_UNSUPPORTED) return rc;
    }
    // composition of the unfused steps (fast kernels where they apply, e.g. edge_kernel_size != 3)
    u8 *labels = d_labels; size_t lp = lpitch;
    if (!labels) {
        lp = ((size_t)w + 15) & ~(size_t)15;
        OMNI_TRY(omni_ws_reserve(ctx, 2, lp * h));
        labels = (u8 *)ctx->ws[2];
    }
    if (ctx->fast) {
        OMNI_LAUNCH(ctx, st, "assign", fast_assign(ctx, d_bgr, h, w, pitch, P, 1, labels, lp, st));
        OMNI_TRY(fast_layer_masks(ctx, labels, h, w, lp, K, 1, 1, d_masks, m_plane_stride, mpitch, st));
    } else {
        OMNI_LAUNCH(ctx, st, "assign", g_assign(d_bgr, h, w, pitch, P, 1, labels, lp, st));
        OMNI_TRY(generic_layer_masks(ctx, labels, h, w, lp, K, 1, 1, d_masks, m_plane_stride, mpitch, st));
    }
    return edges_dispatch(ctx, d_masks, K, h, w, m_plane_stride, mpitch, prm, bp, low, high, d_edges, e_plane_stride, epitch, st);
}

extern "C" int omni_color_edge_batch(omni_ctx *ctx, const uint8_t *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                                     const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                                     uint8_t *d_masks, size_t m_plane_stride, size_t mpitch,
                                     uint8_t *d_edges, size_t e_plane_stride, size_t epitch, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_bgr && d_masks && d_edges && h_centers && n_frames >= 1, "omni_color_edge_batch: bad arguments");
    OMNI_REQUIRE(h > 0 && w > 0 && pitch >= (size_t)w * 3 && mpitch >= (size_t)w && epitch >= (size_t)w, "omni_color_edge_batch: bad geometry");
    OMNI_REQUIRE(K >= 1 && K <= OMNI_MAX_K, "K=%d outside [1,%d]", K, OMNI_MAX_K);
    BlurParams bp; int low, high;
    OMNI_TRY(check_edge_params(prm, &bp, &low, &high));
    AssignParams P;
    OMNI_TRY(fill_assign(&P, h_centers, nullptr, K, h_lut));
    cudaStream_t st = (cudaStream_t)stream;
    const int group = OMNI_MAX_K / K;                      // frames whose layers fit the plane dimension of one pass
    for (int f0 = 0; f0 < n_frames; ) {
        const int nf = (n_frames - f0) < group ? (n_frames - f0) : group;
        const uint8_t *src = d_bgr + (size_t)f0 * frame_stride;
        uint8_t *dm = d_masks + (size_t)f0 * K * m_plane_stride, *de = d_edges + (size_t)f0 * K * e_plane_stride;
        int rc = OMNI_ERR_UNSUPPORTED;
        if (ctx->fast && fast_fused_supported(prm) && nf > 1)
            rc = fast_color_edge_batch(ctx, src, nf, frame_stride, h, w, pitch, P, prm, low, high, dm, m_plane_stride, mpitch,
                                       de, e_plane_stride, epitch, st);
        if (rc == OMNI_ERR_UNSUPPORTED) {                  // outside the fast path (or a single frame): frame by frame
            for (int f = 0; f < nf; f++)
                OMNI_TRY(omni_color_edge(ctx, src + (size_t)f * frame_stride, h, w, pitch, h_centers, K, h_lut, prm, nullptr, 0,
                                         dm + (size_t)f * K * m_plane_stride, m_plane_stride, mpitch,
                                         de + (size_t)f * K * e_plane_stride, e_plane_stride, epitch, stream));
        } else if (rc != OMNI_OK) return rc;
        f0 += nf;
    }
    return OMNI_OK;
}

static inline size_t pad16(size_t v) { return (v + 15) & ~(size_t)15; }

// ---- packed (1 bit per pixel) outputs ------------------------------------------------------------------------
// Device body shared by the packed entry points: n frames at d_bgr -> packed planes (device, caller layout) + counts on the device
// (ctx->d_counts: [pixels | mask non-zeros | edge non-zeros], OMNI_MAX_K each) when want_counts.  per_frame: frame f has its own
// centres h_centers + f * K * 3 and LUT h_lut + f * K (else all frames share h_centers / h_lut).
static int packed_device(omni_ctx *ctx, const u8 *d_bgr, int nf, size_t frame_stride, int h, int w, size_t pitch, const float *h_centers,
                         int K, const uint8_t *h_lut, const omni_edge_params *prm, u8 *d_mb, size_t mb_plane, size_t mb_pitch,
                         u8 *d_eb, size_t eb_plane, size_t eb_pitch, int bit_order, bool want_counts, cudaStream_t st, bool per_frame = false)
{
    OMNI_REQUIRE(bit_order == OMNI_BITS_LSB_FIRST || bit_order == OMNI_BITS_MSB_FIRST, "bit_order must be OMNI_BITS_LSB_FIRST or OMNI_BITS_MSB_FIRST");
    OMNI_REQUIRE(nf >= 1 && nf * K <= OMNI_MAX_K, "n_frames * K = %d exceeds %d planes per call", nf * K, OMNI_MAX_K);
    const size_t rb = ((size_t)w + 7) / 8;
    OMNI_REQUIRE(mb_pitch >= rb && (!prm || eb_pitch >= rb), "packed row pitch smaller than ceil(w / 8) bytes");
    BlurParams bp; int low = 0, high = 0;
    if (prm) OMNI_TRY(check_edge_params(prm, &bp, &low, &high));
    const size_t cs = per_frame ? (size_t)3 * K : 0, ls = per_frame ? (size_t)K : 0;     // centre / LUT stride between frames
    AssignParams P, Pf[OMNI_MAX_K];
    OMNI_TRY(fill_assign(&P, h_centers, nullptr, K, h_lut));
    if (per_frame)
        for (int f = 0; f < nf; f++) OMNI_TRY(fill_assign(&Pf[f], h_centers + f * cs, nullptr, K, h_lut ? h_lut + f * ls : nullptr));
    unsigned long long *dc = want_counts ? ctx->d_counts : nullptr;
    int rc = OMNI_ERR_UNSUPPORTED;
    if (ctx->fast && ctx->pipeline == 1)
        rc = label_color_edge_packed(ctx, d_bgr, nf, frame_stride, h, w, pitch, P, prm, low, high, d_mb, mb_plane, mb_pitch, d_eb, eb_plane,
                                     eb_pitch, bit_order == OMNI_BITS_MSB_FIRST, dc, st, per_frame ? Pf : nullptr);
    if (rc != OMNI_ERR_UNSUPPORTED) return rc;
    // any other family: byte planes in workspace slot 2, then packed
    const size_t bp_pitch = ((size_t)w + 15) & ~(size_t)15, bplane = bp_pitch * h, lp = bp_pitch;
    const int KT = nf * K;
    OMNI_TRY(omni_ws_reserve(ctx, 2, lp * h + 2 * bplane * KT));
    u8 *dl = (u8 *)ctx->ws[2], *dm = dl + lp * h, *de = dm + bplane * KT;
    if (dc) OMNI_CUDA(cudaMemsetAsync(dc, 0, 3 * OMNI_MAX_K * sizeof(unsigned long long), st));
    omni_edge_params none{1, 0, 0, 3, 50.0, 150.0};          // masks only: the edge planes of a cheap dummy pass are dropped
    for (int f = 0; f < nf; f++) {
        const u8 *img = d_bgr + (size_t)f * frame_stride;
        const float *ctr = h_centers + f * cs;
        const uint8_t *lut = h_lut ? h_lut + f * ls : nullptr;
        if (prm) {
            OMNI_TRY(omni_color_edge(ctx, img, h, w, pitch, ctr, K, lut, prm, dl, lp, dm + (size_t)f * K * bplane, bplane, bp_pitch,
                                     de + (size_t)f * K * bplane, bplane, bp_pitch, st));
        } else {
            (void)none;
            OMNI_TRY(omni_assign_lab_f32(ctx, img, h, w, pitch, ctr, K, lut, dl, lp, st));
            OMNI_TRY(omni_layer_masks(ctx, dl, h, w, lp, K, 1, 1, dm + (size_t)f * K * bplane, bplane, bp_pitch, st));
        }
        if (dc) OMNI_LAUNCH(ctx, st, "count_labels", g_count_labels(dl, lp, h, w, K, dc + (size_t)f * K, st));
    }
    OMNI_LAUNCH(ctx, st, "pack_bytes", g_pack_bytes(dm, bplane, bp_pitch, KT, h, w, d_mb, mb_plane, mb_pitch, bit_order, dc ? dc + OMNI_MAX_K : nullptr, st));
    if (prm)
        OMNI_LAUNCH(ctx, st, "pack_bytes", g_pack_bytes(de, bplane, bp_pitch, KT, h, w, d_eb, eb_plane, eb_pitch, bit_order, dc ? dc + 2 * OMNI_MAX_K : nullptr, st));
    return OMNI_OK;
}

static void fetch_counts(omni_ctx *ctx, int KT, int64_t *h_counts)
{
    for (int k = 0; k < KT; k++) {
        h_counts[3 * k] = (int64_t)ctx->h_counts[k];
        h_counts[3 * k + 1] = (int64_t)ctx->h_counts[OMNI_MAX_K + k];
        h_counts[3 * k + 2] = (int64_t)ctx->h_counts[2 * OMNI_MAX_K + k];
    }
}

static int device_packed(const char *fn, omni_ctx *ctx, const uint8_t *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                         const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                         uint8_t *d_mask_bits, size_t mb_plane_stride, size_t mb_pitch,
                         uint8_t *d_edge_bits, size_t eb_plane_stride, size_t eb_pitch, int bit_order,
                         int64_t *h_counts, void *stream, bool per_frame)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_bgr && d_mask_bits && h_centers && (d_edge_bits || !prm), "%s: NULL pointer", fn);
    OMNI_REQUIRE(h > 0 && w > 0 && pitch >= (size_t)w * 3 && K >= 1 && K <= OMNI_MAX_K, "%s: bad geometry", fn);
    cudaStream_t st = (cudaStream_t)stream;
    OMNI_TRY(packed_device(ctx, d_bgr, n_frames, frame_stride, h, w, pitch, h_centers, K, h_lut, prm, d_mask_bits, mb_plane_stride, mb_pitch,
                           d_edge_bits, eb_plane_stride, eb_pitch, bit_order, h_counts != nullptr, st, per_frame));
    if (h_counts) {
        OMNI_CUDA(cudaMemcpyAsync(ctx->h_counts, ctx->d_counts, 3 * OMNI_MAX_K * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        OMNI_CUDA(cudaStreamSynchronize(st));
        fetch_counts(ctx, n_frames * K, h_counts);
    }
    return OMNI_OK;
}

extern "C" int omni_color_edge_packed(omni_ctx *ctx, const uint8_t *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                                      const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                                      uint8_t *d_mask_bits, size_t mb_plane_stride, size_t mb_pitch,
                                      uint8_t *d_edge_bits, size_t eb_plane_stride, size_t eb_pitch, int bit_order,
                                      int64_t *h_counts, void *stream)
{
    return device_packed("omni_color_edge_packed", ctx, d_bgr, n_frames, frame_stride, h, w, pitch, h_centers, K, h_lut, prm, d_mask_bits,
                         mb_plane_stride, mb_pitch, d_edge_bits, eb_plane_stride, eb_pitch, bit_order, h_counts, stream, false);
}

extern "C" int omni_color_edge_packed_frames(omni_ctx *ctx, const uint8_t *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                                             const float *h_centers, int K, const uint8_t *h_luts, const omni_edge_params *prm,
                                             uint8_t *d_mask_bits, size_t mb_plane_stride, size_t mb_pitch,
                                             uint8_t *d_edge_bits, size_t eb_plane_stride, size_t eb_pitch, int bit_order,
                                             int64_t *h_counts, void *stream)
{
    return device_packed("omni_color_edge_packed_frames", ctx, d_bgr, n_frames, frame_stride, h, w, pitch, h_centers, K, h_luts, prm,
                         d_mask_bits, mb_plane_stride, mb_pitch, d_edge_bits, eb_plane_stride, eb_pitch, bit_order, h_counts, stream, true);
}

// Host buffers, n frames sharing one centre set (or, per_frame, each with its own), H2D / kernels / D2H of consecutive frame groups
// overlapped (two staging slots on three streams).  Results are complete in the host buffers when the call returns.
static int host_packed(const char *fn, omni_ctx *ctx, const uint8_t *h_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                       const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                       uint8_t *h_mask_bits, size_t mb_plane_stride, size_t mb_pitch,
                       uint8_t *h_edge_bits, size_t eb_plane_stride, size_t eb_pitch, int bit_order,
                       int64_t *h_counts, bool per_frame)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(h_bgr && h_mask_bits && h_centers && (h_edge_bits || !prm) && n_frames >= 1, "%s: bad arguments", fn);
    OMNI_REQUIRE(h > 0 && w > 0 && pitch >= (size_t)w * 3 && K >= 1 && K <= OMNI_MAX_K, "%s: bad geometry", fn);
    const size_t rb = ((size_t)w + 7) / 8;
    OMNI_REQUIRE(mb_pitch >= rb && (!prm || eb_pitch >= rb), "packed row pitch smaller than ceil(w / 8) bytes");
    OMNI_REQUIRE(mb_plane_stride == mb_pitch * (size_t)h && (!prm || eb_plane_stride == eb_pitch * (size_t)h),
                 "%s: planes must be back to back (plane stride = pitch * h)", fn);
    if (per_frame) {                                        // every frame's LUT before any work, as fill_assign checks it
        AssignParams P;
        for (int f = 0; f < n_frames; f++)
            OMNI_TRY(fill_assign(&P, h_centers + (size_t)f * 3 * K, nullptr, K, h_lut ? h_lut + (size_t)f * K : nullptr));
    }
    const size_t cs = per_frame ? (size_t)3 * K : 0, ls = per_frame ? (size_t)K : 0;     // centre / LUT stride between frames
    const int G = OMNI_MAX_K / K;                           // frames per device pass (their G * K layers are its planes)
    const int n_groups = (n_frames + G - 1) / G;
    if (!ctx->pk_ready) {
        OMNI_CUDA(cudaStreamCreateWithFlags(&ctx->pk_in, cudaStreamNonBlocking));
        OMNI_CUDA(cudaStreamCreateWithFlags(&ctx->pk_out, cudaStreamNonBlocking));
        for (auto &e : ctx->pk_ev) OMNI_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->pk_ready = 1;
    }
    ctx->last_band_resends = -1;                            // -1: the last call was not banded
    if (n_frames == 1) {                                    // one image: row bands overlap its own copies and kernels
        BlurParams bp; int low = 0, high = 0;
        if (prm) OMNI_TRY(check_edge_params(prm, &bp, &low, &high));
        AssignParams P;
        OMNI_TRY(fill_assign(&P, h_centers, nullptr, K, h_lut));
        OMNI_REQUIRE(bit_order == OMNI_BITS_LSB_FIRST || bit_order == OMNI_BITS_MSB_FIRST, "bit_order must be OMNI_BITS_LSB_FIRST or OMNI_BITS_MSB_FIRST");
        int rc = label_host_packed_banded(ctx, h_bgr, h, w, pitch, P, prm, low, high, h_mask_bits, mb_plane_stride, mb_pitch, h_edge_bits,
                                          eb_plane_stride, eb_pitch, bit_order == OMNI_BITS_MSB_FIRST, h_counts);
        if (rc != OMNI_ERR_UNSUPPORTED) return rc;
    }
    if (h_counts && ctx->pk_counts_cap < (size_t)n_groups) {        // pinned: one block of counts per group, read after the last copy
        if (ctx->pk_counts) OMNI_CUDA(cudaFreeHost(ctx->pk_counts));
        ctx->pk_counts = nullptr; ctx->pk_counts_cap = 0;
        OMNI_CUDA(cudaHostAlloc(&ctx->pk_counts, (size_t)n_groups * 3 * OMNI_MAX_K * sizeof(unsigned long long), cudaHostAllocDefault));
        ctx->pk_counts_cap = (size_t)n_groups;
    }
    const size_t ip = pad16((size_t)w * 3), img_bytes = pad16(ip * h), dp = pad16(rb), dplane = dp * h;
    const size_t slot_in = img_bytes * G, slot_out = pad16(dplane * (size_t)G * K);
    OMNI_TRY(omni_ws_reserve(ctx, 3, 2 * slot_in + 4 * slot_out));
    u8 *base = (u8 *)ctx->ws[3];
    cudaStream_t sc = ctx->stream, si = ctx->pk_in, so = ctx->pk_out;
    // events: [0,1] H2D of slot done, [2,3] kernels of slot done (inputs free, outputs ready), [4,5] D2H of slot done
    OMNI_CUDA(cudaEventRecord(ctx->pk_ev[6], sc));          // order the side streams after earlier work of this ctx
    OMNI_CUDA(cudaStreamWaitEvent(si, ctx->pk_ev[6], 0));
    OMNI_CUDA(cudaStreamWaitEvent(so, ctx->pk_ev[6], 0));
    for (int gi = 0; gi < n_groups; gi++) {
        const int s = gi & 1, f0 = gi * G, nf = (n_frames - f0) < G ? (n_frames - f0) : G;
        u8 *d_in = base + (size_t)s * slot_in, *d_mb = base + 2 * slot_in + (size_t)(2 * s) * slot_out, *d_eb = d_mb + slot_out;
        if (gi >= 2) OMNI_CUDA(cudaStreamWaitEvent(si, ctx->pk_ev[2 + s], 0));      // the kernels of group gi-2 have read this slot
        for (int f = 0; f < nf; f++)
            OMNI_CUDA(cudaMemcpy2DAsync(d_in + (size_t)f * img_bytes, ip, h_bgr + (size_t)(f0 + f) * frame_stride, pitch, (size_t)w * 3, h,
                                        cudaMemcpyHostToDevice, si));
        OMNI_CUDA(cudaEventRecord(ctx->pk_ev[s], si));
        OMNI_CUDA(cudaStreamWaitEvent(sc, ctx->pk_ev[s], 0));
        if (gi >= 2) OMNI_CUDA(cudaStreamWaitEvent(sc, ctx->pk_ev[4 + s], 0));      // the D2H of group gi-2 has drained this slot's outputs
        OMNI_TRY(packed_device(ctx, d_in, nf, img_bytes, h, w, ip, h_centers + f0 * cs, K, h_lut ? h_lut + f0 * ls : nullptr, prm, d_mb, dplane,
                               dp, d_eb, dplane, dp, bit_order, h_counts != nullptr, sc, per_frame));
        if (h_counts)
            OMNI_CUDA(cudaMemcpyAsync(ctx->pk_counts + (size_t)gi * 3 * OMNI_MAX_K, ctx->d_counts, 3 * OMNI_MAX_K * sizeof(unsigned long long),
                                      cudaMemcpyDeviceToHost, sc));
        OMNI_CUDA(cudaEventRecord(ctx->pk_ev[2 + s], sc));
        OMNI_CUDA(cudaStreamWaitEvent(so, ctx->pk_ev[2 + s], 0));
        // the nf * K planes of the group are back to back on both sides: one strided copy of h * nf * K rows
        OMNI_CUDA(cudaMemcpy2DAsync(h_mask_bits + (size_t)f0 * K * mb_plane_stride, mb_pitch, d_mb, dp, rb, (size_t)h * nf * K,
                                    cudaMemcpyDeviceToHost, so));
        if (prm)
            OMNI_CUDA(cudaMemcpy2DAsync(h_edge_bits + (size_t)f0 * K * eb_plane_stride, eb_pitch, d_eb, dp, rb, (size_t)h * nf * K,
                                        cudaMemcpyDeviceToHost, so));
        OMNI_CUDA(cudaEventRecord(ctx->pk_ev[4 + s], so));
    }
    OMNI_CUDA(cudaStreamSynchronize(so));
    OMNI_CUDA(cudaStreamSynchronize(sc));
    if (h_counts)
        for (int gi = 0; gi < n_groups; gi++) {
            const int f0 = gi * G, nf = (n_frames - f0) < G ? (n_frames - f0) : G;
            const unsigned long long *pc = ctx->pk_counts + (size_t)gi * 3 * OMNI_MAX_K;
            for (int k = 0; k < nf * K; k++) {
                int64_t *o = h_counts + 3 * ((size_t)f0 * K + k);
                o[0] = (int64_t)pc[k]; o[1] = (int64_t)pc[OMNI_MAX_K + k]; o[2] = (int64_t)pc[2 * OMNI_MAX_K + k];
            }
        }
    return OMNI_OK;
}

extern "C" int omni_host_color_edge_packed(omni_ctx *ctx, const uint8_t *h_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                                           const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                                           uint8_t *h_mask_bits, size_t mb_plane_stride, size_t mb_pitch,
                                           uint8_t *h_edge_bits, size_t eb_plane_stride, size_t eb_pitch, int bit_order,
                                           int64_t *h_counts)
{
    return host_packed("omni_host_color_edge_packed", ctx, h_bgr, n_frames, frame_stride, h, w, pitch, h_centers, K, h_lut, prm, h_mask_bits,
                       mb_plane_stride, mb_pitch, h_edge_bits, eb_plane_stride, eb_pitch, bit_order, h_counts, false);
}

extern "C" int omni_host_color_edge_packed_frames(omni_ctx *ctx, const uint8_t *h_bgr, int n_frames, size_t frame_stride, int h, int w,
                                                  size_t pitch, const float *h_centers, int K, const uint8_t *h_luts,
                                                  const omni_edge_params *prm, uint8_t *h_mask_bits, size_t mb_plane_stride, size_t mb_pitch,
                                                  uint8_t *h_edge_bits, size_t eb_plane_stride, size_t eb_pitch, int bit_order,
                                                  int64_t *h_counts)
{
    return host_packed("omni_host_color_edge_packed_frames", ctx, h_bgr, n_frames, frame_stride, h, w, pitch, h_centers, K, h_luts, prm,
                       h_mask_bits, mb_plane_stride, mb_pitch, h_edge_bits, eb_plane_stride, eb_pitch, bit_order, h_counts, true);
}

// ---- counts / composite -----------------------------------------------------------------------------------
extern "C" int omni_count_nonzero(omni_ctx *ctx, const uint8_t *d_planes, int K, int h, int w, size_t plane_stride, size_t pitch,
                                  int64_t *h_counts, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_planes && h_counts && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0, "omni_count_nonzero: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    OMNI_CUDA(cudaMemsetAsync(ctx->d_counts, 0, K * sizeof(unsigned long long), st));
    OMNI_LAUNCH(ctx, st, "count_nonzero", g_count_nonzero(d_planes, plane_stride, pitch, K, h, w, ctx->d_counts, st));
    OMNI_CUDA(cudaMemcpyAsync(ctx->h_counts, ctx->d_counts, K * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    OMNI_CUDA(cudaStreamSynchronize(st));
    for (int k = 0; k < K; k++) h_counts[k] = (int64_t)ctx->h_counts[k];
    return OMNI_OK;
}

extern "C" int omni_edges_composite(omni_ctx *ctx, const uint8_t *d_edges, int K, int h, int w, size_t e_plane_stride, size_t epitch,
                                    const uint8_t *h_colors_bgr, uint8_t *d_canvas, size_t cpitch, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_edges && d_canvas && h_colors_bgr && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0 && cpitch >= (size_t)w * 3,
                 "omni_edges_composite: bad arguments");
    OMNI_LAUNCH(ctx, (cudaStream_t)stream, "composite", g_composite(d_edges, e_plane_stride, epitch, K, h, w, h_colors_bgr, d_canvas, cpitch, (cudaStream_t)stream));
    return OMNI_OK;
}

// host planes in, host canvas out (what 03_edge_detect.py:60-111 does with the edges.png files it has just read)
extern "C" int omni_host_edges_composite(omni_ctx *ctx, const uint8_t *h_edges, int K, int h, int w, size_t e_plane_stride, size_t epitch,
                                         const uint8_t *h_colors_bgr, uint8_t *h_canvas, size_t cpitch)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(h_edges && h_canvas && h_colors_bgr && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0 && epitch >= (size_t)w &&
                 cpitch >= (size_t)w * 3, "omni_host_edges_composite: bad arguments");
    const size_t ep = pad16((size_t)w), eplane = ep * h, cp = pad16((size_t)w * 3);
    OMNI_TRY(omni_ws_reserve(ctx, 3, eplane * K + cp * h));
    u8 *de = (u8 *)ctx->ws[3], *dc = de + eplane * K;
    for (int k = 0; k < K; k++)
        OMNI_CUDA(cudaMemcpy2DAsync(de + k * eplane, ep, h_edges + k * e_plane_stride, epitch, (size_t)w, h, cudaMemcpyHostToDevice, ctx->stream));
    OMNI_TRY(omni_edges_composite(ctx, de, K, h, w, eplane, ep, h_colors_bgr, dc, cp, ctx->stream));
    OMNI_CUDA(cudaMemcpy2DAsync(h_canvas, cpitch, dc, cp, (size_t)w * 3, h, cudaMemcpyDeviceToHost, ctx->stream));
    OMNI_CUDA(cudaStreamSynchronize(ctx->stream));
    return OMNI_OK;
}

// ---- host-buffer entry points -------------------------------------------------------------------------------
// Staging layout in workspace slot 3: [image | labels | masks | edges], rows padded to 16 bytes.

extern "C" int omni_host_resize_area_u8c3(omni_ctx *ctx, const uint8_t *h_src, int sh, int sw, size_t spitch,
                                          uint8_t *h_dst, int dh, int dw, size_t dpitch)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(h_src && h_dst && sh > 0 && sw > 0 && dh > 0 && dw > 0, "omni_host_resize_area_u8c3: bad arguments");
    size_t sp = pad16((size_t)sw * 3), dp = pad16((size_t)dw * 3);
    OMNI_TRY(omni_ws_reserve(ctx, 3, sp * sh + dp * dh));
    u8 *ds = (u8 *)ctx->ws[3], *dd = ds + sp * sh;
    OMNI_CUDA(cudaMemcpy2DAsync(ds, sp, h_src, spitch, (size_t)sw * 3, sh, cudaMemcpyHostToDevice, ctx->stream));
    OMNI_TRY(omni_resize_area_u8c3(ctx, ds, sh, sw, sp, dd, dh, dw, dp, ctx->stream));
    OMNI_CUDA(cudaMemcpy2DAsync(h_dst, dpitch, dd, dp, (size_t)dw * 3, dh, cudaMemcpyDeviceToHost, ctx->stream));
    OMNI_CUDA(cudaStreamSynchronize(ctx->stream));
    return OMNI_OK;
}

extern "C" int omni_host_assign_rgb_i16wrap(omni_ctx *ctx, const uint8_t *h_rgb, int h, int w, size_t pitch,
                                            const uint8_t *h_palette, int K, uint8_t *h_labels, size_t lpitch)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(h_rgb && h_labels && h > 0 && w > 0, "omni_host_assign_rgb_i16wrap: bad arguments");
    size_t ip = pad16((size_t)w * 3), lp = pad16((size_t)w);
    OMNI_TRY(omni_ws_reserve(ctx, 3, ip * h + lp * h));
    u8 *di = (u8 *)ctx->ws[3], *dl = di + ip * h;
    OMNI_CUDA(cudaMemcpy2DAsync(di, ip, h_rgb, pitch, (size_t)w * 3, h, cudaMemcpyHostToDevice, ctx->stream));
    OMNI_TRY(omni_assign_rgb_i16wrap(ctx, di, h, w, ip, h_palette, K, dl, lp, ctx->stream));
    OMNI_CUDA(cudaMemcpy2DAsync(h_labels, lpitch, dl, lp, (size_t)w, h, cudaMemcpyDeviceToHost, ctx->stream));
    OMNI_CUDA(cudaStreamSynchronize(ctx->stream));
    return OMNI_OK;
}

static int copy_planes_d2h(u8 *h_dst, size_t h_plane, size_t hpitch, const u8 *d_src, size_t d_plane, size_t dpitch,
                           int K, int h, int w, cudaStream_t st)
{
    // one contiguous copy only when the host rows are gap-free: with hpitch > w the bytes between the rows belong to the
    // caller (a view into a wider array) and must not be touched
    if (hpitch == (size_t)w && dpitch == hpitch && h_plane == d_plane) {
        OMNI_CUDA(cudaMemcpyAsync(h_dst, d_src, d_plane * (size_t)(K - 1) + dpitch * (size_t)(h - 1) + w, cudaMemcpyDeviceToHost, st));
        return OMNI_OK;
    }
    if (hpitch == (size_t)w && dpitch == hpitch) {      // gap-free planes, different plane strides: one 2-D copy (row = plane)
        OMNI_CUDA(cudaMemcpy2DAsync(h_dst, h_plane, d_src, d_plane, (size_t)w * h, K, cudaMemcpyDeviceToHost, st));
        return OMNI_OK;
    }
    for (int k = 0; k < K; k++)
        OMNI_CUDA(cudaMemcpy2DAsync(h_dst + k * h_plane, hpitch, d_src + k * d_plane, dpitch, (size_t)w, h, cudaMemcpyDeviceToHost, st));
    return OMNI_OK;
}

extern "C" int omni_host_edges(omni_ctx *ctx, const uint8_t *h_masks, int K, int h, int w, size_t m_plane_stride, size_t mpitch,
                               const omni_edge_params *prm,
                               uint8_t *h_edges, size_t e_plane_stride, size_t epitch)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(h_masks && h_edges && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0, "omni_host_edges: bad arguments");
    // device planes use the caller's pitch when it is 16-byte friendly so the copies are single DMA transfers
    size_t dp = (mpitch % 16 == 0) ? mpitch : pad16((size_t)w), dplane = (dp == mpitch) ? m_plane_stride : dp * h;
    size_t ep = (epitch % 16 == 0) ? epitch : pad16((size_t)w), eplane = (ep == epitch) ? e_plane_stride : ep * h;
    size_t m_bytes = pad16(dplane * K), e_bytes = pad16(eplane * K);
    OMNI_TRY(omni_ws_reserve(ctx, 3, m_bytes + e_bytes));
    u8 *dm = (u8 *)ctx->ws[3], *de = dm + m_bytes;
    if (dp == mpitch) OMNI_CUDA(cudaMemcpyAsync(dm, h_masks, m_plane_stride * (size_t)(K - 1) + mpitch * (size_t)(h - 1) + w, cudaMemcpyHostToDevice, ctx->stream));
    else for (int k = 0; k < K; k++)
        OMNI_CUDA(cudaMemcpy2DAsync(dm + k * dplane, dp, h_masks + k * m_plane_stride, mpitch, (size_t)w, h, cudaMemcpyHostToDevice, ctx->stream));
    OMNI_TRY(omni_edges(ctx, dm, K, h, w, dplane, dp, prm, de, eplane, ep, ctx->stream));
    OMNI_TRY(copy_planes_d2h(h_edges, e_plane_stride, epitch, de, eplane, ep, K, h, w, ctx->stream));
    OMNI_CUDA(cudaStreamSynchronize(ctx->stream));
    return OMNI_OK;
}

extern "C" int omni_swatch_masks(omni_ctx *ctx, const uint8_t *d_bgr, int h, int w, size_t pitch,
                                 const int32_t *h_colors, int K, int tol,
                                 uint8_t *d_masks, size_t plane_stride, size_t mpitch, int32_t *h_choice, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_bgr && d_masks && h_colors && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0, "omni_swatch_masks: bad arguments");
    OMNI_REQUIRE(pitch >= (size_t)w * 3 && mpitch >= (size_t)w, "omni_swatch_masks: pitch smaller than a row");
    OMNI_REQUIRE(tol >= 0 && tol <= 255, "omni_swatch_masks: color_tolerance %d outside [0,255]", tol);
    for (int i = 0; i < 3 * K; i++)
        OMNI_REQUIRE(h_colors[i] >= 0 && h_colors[i] <= 255, "omni_swatch_masks: swatch component %d outside [0,255]", h_colors[i]);
    return fast_swatch_masks(ctx, d_bgr, h, w, pitch, h_colors, K, tol, d_masks, plane_stride, mpitch, h_choice, (cudaStream_t)stream);
}

// ---- stage 04: thinning ------------------------------------------------------------------------------------
extern "C" int omni_thin_zhangsuen(omni_ctx *ctx, const uint8_t *d_in, int K, int h, int w, size_t in_plane_stride, size_t in_pitch,
                                   int max_iter, uint8_t *d_out, size_t out_plane_stride, size_t out_pitch,
                                   int32_t *h_removed, int32_t *h_iters, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_in && d_out && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0, "omni_thin_zhangsuen: bad arguments");
    OMNI_REQUIRE(in_pitch >= (size_t)w && out_pitch >= (size_t)w, "omni_thin_zhangsuen: pitch smaller than a row");
    OMNI_REQUIRE(max_iter >= 0 && max_iter <= 100000, "omni_thin_zhangsuen: max_iter %d out of range", max_iter);
    return fast_thin(ctx, d_in, K, h, w, in_plane_stride, in_pitch, max_iter, d_out, out_plane_stride, out_pitch, h_removed, h_iters,
                     (cudaStream_t)stream);
}

// the same on planes of 1 bit per pixel (the packed edge planes of omni_color_edge_packed): no byte planes on the way
extern "C" int omni_thin_zhangsuen_packed(omni_ctx *ctx, const uint8_t *d_bits_in, int K, int h, int w, size_t in_plane_stride, size_t in_pitch,
                                          int bit_order, int max_iter, uint8_t *d_bits_out, size_t out_plane_stride, size_t out_pitch,
                                          int32_t *h_removed, int32_t *h_iters, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_bits_in && d_bits_out && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0, "omni_thin_zhangsuen_packed: bad arguments");
    OMNI_REQUIRE(in_pitch >= (size_t)(w + 7) / 8 && out_pitch >= (size_t)(w + 7) / 8, "omni_thin_zhangsuen_packed: pitch smaller than a row");
    OMNI_REQUIRE(bit_order == OMNI_BITS_LSB_FIRST || bit_order == OMNI_BITS_MSB_FIRST, "omni_thin_zhangsuen_packed: bad bit order");
    OMNI_REQUIRE(max_iter >= 0 && max_iter <= 100000, "omni_thin_zhangsuen_packed: max_iter %d out of range", max_iter);
    return fast_thin(ctx, d_bits_in, K, h, w, in_plane_stride, in_pitch, max_iter, d_bits_out, out_plane_stride, out_pitch, h_removed, h_iters,
                     (cudaStream_t)stream, bit_order == OMNI_BITS_MSB_FIRST ? 2 : 1);
}

extern "C" int omni_host_thin_zhangsuen(omni_ctx *ctx, const uint8_t *h_in, int K, int h, int w, size_t in_plane_stride, size_t in_pitch,
                                        int max_iter, uint8_t *h_out, size_t out_plane_stride, size_t out_pitch,
                                        int32_t *h_removed, int32_t *h_iters)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(h_in && h_out && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0, "omni_host_thin_zhangsuen: bad arguments");
    size_t dp = pad16((size_t)w), dplane = dp * h, bytes = pad16(dplane * K);
    OMNI_TRY(omni_ws_reserve(ctx, 3, bytes));
    u8 *d = (u8 *)ctx->ws[3];
    for (int k = 0; k < K; k++)
        OMNI_CUDA(cudaMemcpy2DAsync(d + k * dplane, dp, h_in + k * in_plane_stride, in_pitch, (size_t)w, h, cudaMemcpyHostToDevice, ctx->stream));
    OMNI_TRY(omni_thin_zhangsuen(ctx, d, K, h, w, dplane, dp, max_iter, d, dplane, dp, h_removed, h_iters, ctx->stream));
    OMNI_TRY(copy_planes_d2h(h_out, out_plane_stride, out_pitch, d, dplane, dp, K, h, w, ctx->stream));
    OMNI_CUDA(cudaStreamSynchronize(ctx->stream));
    return OMNI_OK;
}

extern "C" int omni_skeleton_degree(omni_ctx *ctx, const uint8_t *d_skel, int K, int h, int w, size_t s_plane_stride, size_t spitch,
                                    uint8_t *d_deg, size_t d_plane_stride, size_t dpitch,
                                    uint8_t *d_nodes, size_t n_plane_stride, size_t npitch, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_skel && (d_deg || d_nodes) && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0, "omni_skeleton_degree: bad arguments");
    OMNI_REQUIRE(spitch >= (size_t)w && (!d_deg || dpitch >= (size_t)w) && (!d_nodes || npitch >= (size_t)w),
                 "omni_skeleton_degree: pitch smaller than a row");
    OMNI_LAUNCH(ctx, (cudaStream_t)stream, "skeleton_degree",
                g_skeleton_degree(d_skel, s_plane_stride, spitch, K, h, w, d_deg, d_plane_stride, dpitch, d_nodes, n_plane_stride, npitch,
                                  (cudaStream_t)stream));
    return OMNI_OK;
}

// ---- stage 04: trace_centerlines (trace.cu) ----------------------------------------------------------------
extern "C" int omni_trace_centerlines(omni_ctx *ctx, const uint8_t *d_skel, int K, int h, int w, size_t plane_stride, size_t pitch,
                                      int64_t *h_plane_info, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_skel && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0, "omni_trace_centerlines: bad arguments");
    OMNI_REQUIRE(pitch >= (size_t)w && (K == 1 || plane_stride >= pitch * (h - 1) + w), "omni_trace_centerlines: pitch smaller than a row");
    OMNI_REQUIRE((long long)((w + 1) / 2) * ((h + 1) / 2) * K < INT32_MAX, "omni_trace_centerlines: %d planes of %d x %d are too large", K, w, h);
    return trace_run(ctx, d_skel, K, h, w, plane_stride, pitch, h_plane_info, (cudaStream_t)stream);
}

extern "C" int omni_host_trace_centerlines(omni_ctx *ctx, const uint8_t *h_skel, int K, int h, int w, size_t plane_stride, size_t pitch,
                                           int64_t *h_plane_info)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(h_skel && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0 && pitch >= (size_t)w, "omni_host_trace_centerlines: bad arguments");
    size_t dp = pad16((size_t)w), dplane = dp * h;
    OMNI_TRY(omni_ws_reserve(ctx, 3, pad16(dplane * K)));
    u8 *d = (u8 *)ctx->ws[3];
    for (int k = 0; k < K; k++)
        OMNI_CUDA(cudaMemcpy2DAsync(d + k * dplane, dp, h_skel + k * plane_stride, pitch, (size_t)w, h, cudaMemcpyHostToDevice, ctx->stream));
    return omni_trace_centerlines(ctx, d, K, h, w, dplane, dp, h_plane_info, ctx->stream);
}

extern "C" int omni_trace_results(omni_ctx *ctx, int32_t *h_points, int32_t *h_path_len, int32_t *h_comp)
{
    OMNI_TRY(set_device(ctx));
    return trace_results(ctx, h_points, h_path_len, h_comp);
}

extern "C" int omni_host_color_edge(omni_ctx *ctx, const uint8_t *h_bgr, int h, int w, size_t pitch,
                                    const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                                    uint8_t *h_labels, size_t lpitch,
                                    uint8_t *h_masks, size_t m_plane_stride, size_t mpitch,
                                    uint8_t *h_edges, size_t e_plane_stride, size_t epitch,
                                    int64_t *h_counts)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(h_bgr && h_masks && h_edges && K >= 1 && K <= OMNI_MAX_K && h > 0 && w > 0, "omni_host_color_edge: bad arguments");
    size_t ip = pad16((size_t)w * 3), lp = pad16((size_t)w);
    size_t mp = (mpitch % 16 == 0) ? mpitch : pad16((size_t)w), mplane = (mp == mpitch) ? m_plane_stride : mp * h;
    size_t ep = (epitch % 16 == 0) ? epitch : pad16((size_t)w), eplane = (ep == epitch) ? e_plane_stride : ep * h;
    size_t i_bytes = pad16(ip * h), l_bytes = pad16(lp * h), m_bytes = pad16(mplane * K), e_bytes = pad16(eplane * K);
    OMNI_TRY(omni_ws_reserve(ctx, 3, i_bytes + l_bytes + m_bytes + e_bytes));
    u8 *di = (u8 *)ctx->ws[3], *dl = di + i_bytes, *dm = dl + l_bytes, *de = dm + m_bytes;
    cudaStream_t st = ctx->stream;
    int rc = OMNI_ERR_UNSUPPORTED;
    if (ctx->fast && h_centers) {
        // pipelined path: band-wise H2D / kernels / D2H on three streams
        BlurParams bp; int low, high;
        OMNI_TRY(check_edge_params(prm, &bp, &low, &high));
        AssignParams P;
        OMNI_TRY(fill_assign(&P, h_centers, nullptr, K, h_lut));
        rc = fast_host_color_edge(ctx, h_bgr, h, w, pitch, P, prm, low, high, h_labels, lpitch, h_masks, m_plane_stride, mpitch,
                                  h_edges, e_plane_stride, epitch, di, ip, dl, lp, dm, mplane, mp, de, eplane, ep,
                                  h_labels != nullptr || h_counts != nullptr);
        if (rc != OMNI_OK && rc != OMNI_ERR_UNSUPPORTED) return rc;
    }
    if (rc == OMNI_ERR_UNSUPPORTED) {
        OMNI_CUDA(cudaMemcpy2DAsync(di, ip, h_bgr, pitch, (size_t)w * 3, h, cudaMemcpyHostToDevice, st));
        OMNI_TRY(omni_color_edge(ctx, di, h, w, ip, h_centers, K, h_lut, prm, dl, lp, dm, mplane, mp, de, eplane, ep, st));
        if (h_labels) OMNI_CUDA(cudaMemcpy2DAsync(h_labels, lpitch, dl, lp, (size_t)w, h, cudaMemcpyDeviceToHost, st));
        OMNI_TRY(copy_planes_d2h(h_masks, m_plane_stride, mpitch, dm, mplane, mp, K, h, w, st));
        OMNI_TRY(copy_planes_d2h(h_edges, e_plane_stride, epitch, de, eplane, ep, K, h, w, st));
    }
    if (h_counts) {
        OMNI_CUDA(cudaMemsetAsync(ctx->d_counts, 0, 3 * OMNI_MAX_K * sizeof(unsigned long long), st));
        OMNI_LAUNCH(ctx, st, "count_labels", g_count_labels(dl, lp, h, w, K, ctx->d_counts, st));
        OMNI_LAUNCH(ctx, st, "count_nonzero", g_count_nonzero(dm, mplane, mp, K, h, w, ctx->d_counts + OMNI_MAX_K, st));
        OMNI_LAUNCH(ctx, st, "count_nonzero", g_count_nonzero(de, eplane, ep, K, h, w, ctx->d_counts + 2 * OMNI_MAX_K, st));
        OMNI_CUDA(cudaMemcpyAsync(ctx->h_counts, ctx->d_counts, 3 * OMNI_MAX_K * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    }
    OMNI_CUDA(cudaStreamSynchronize(st));
    if (h_counts)
        for (int k = 0; k < K; k++) {
            h_counts[3 * k] = (int64_t)ctx->h_counts[k];
            h_counts[3 * k + 1] = (int64_t)ctx->h_counts[OMNI_MAX_K + k];
            h_counts[3 * k + 2] = (int64_t)ctx->h_counts[2 * OMNI_MAX_K + k];
        }
    return OMNI_OK;
}

// ---- PNG files of stages 01-03 (png_encode.cu) --------------------------------------------------------------------------------
extern "C" size_t omni_png_bound(int h, int w, int format)
{
    if ((format != OMNI_PNG_GRAY1 && format != OMNI_PNG_BGR8) || h < 1 || w < 1 || h > OMNI_PNG_MAX_ROWS) return 0;
    const long long row = (format == OMNI_PNG_GRAY1 ? ((long long)w + 7) / 8 : 3LL * w) + 1;
    if (row > OMNI_PNG_MAX_SCANLINE) return 0;
    return png_file_bound(h, w, format);
}

static int png_check(const char *fn, int n, int h, int w, size_t pitch, int format, size_t out_capacity)
{
    OMNI_REQUIRE(format == OMNI_PNG_GRAY1 || format == OMNI_PNG_BGR8, "%s: unknown format %d (OMNI_PNG_GRAY1 = 0, OMNI_PNG_BGR8 = 1)",
                 fn, format);
    OMNI_REQUIRE(n >= 1, "%s: n must be at least 1 (got %d)", fn, n);
    OMNI_REQUIRE(h >= 1 && w >= 1, "%s: h and w must be at least 1 (got %d x %d)", fn, w, h);
    const long long row = format == OMNI_PNG_GRAY1 ? ((long long)w + 7) / 8 : 3LL * w;
    OMNI_REQUIRE(row + 1 <= OMNI_PNG_MAX_SCANLINE,
                 "%s: a row of %d pixels is over the encoder's limit of OMNI_PNG_MAX_SCANLINE = %d bytes per scanline (w <= %d for this format)",
                 fn, w, OMNI_PNG_MAX_SCANLINE, format == OMNI_PNG_GRAY1 ? 8 * (OMNI_PNG_MAX_SCANLINE - 1) : (OMNI_PNG_MAX_SCANLINE - 1) / 3);
    OMNI_REQUIRE(h <= OMNI_PNG_MAX_ROWS, "%s: h = %d is over the encoder's limit of OMNI_PNG_MAX_ROWS = %d rows", fn, h, OMNI_PNG_MAX_ROWS);
    OMNI_REQUIRE(pitch >= (size_t)row, "%s: pitch %zu is shorter than a row (%lld bytes)", fn, pitch, row);
    const long long nseg = ((long long)h + png_segment_rows(w, format) - 1) / png_segment_rows(w, format);
    OMNI_REQUIRE(nseg * n <= INT32_MAX, "%s: %d images of %d rows are over the encoder's limit of 2^31 - 1 segments per call", fn, n, h);
    const size_t need = (size_t)n * png_file_bound(h, w, format);
    OMNI_REQUIRE(out_capacity >= need, "%s: out_capacity %zu is below n * omni_png_bound = %zu", fn, out_capacity, need);
    return OMNI_OK;
}

extern "C" int omni_png_encode(omni_ctx *ctx, const uint8_t *d_src, int n, size_t src_stride, int h, int w, size_t pitch, int format,
                               uint8_t *d_out, size_t out_capacity, int64_t *h_sizes, void *stream)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(d_src && d_out && h_sizes, "omni_png_encode: NULL pointer argument");
    OMNI_TRY(png_check("omni_png_encode", n, h, w, pitch, format, out_capacity));
    return png_encode_run(ctx, d_src, n, src_stride, h, w, pitch, format, d_out, h_sizes, (cudaStream_t)stream);
}

extern "C" int omni_host_png_encode(omni_ctx *ctx, const uint8_t *h_src, int n, size_t src_stride, int h, int w, size_t pitch, int format,
                                    uint8_t *h_out, size_t out_capacity, int64_t *h_sizes)
{
    OMNI_TRY(set_device(ctx));
    OMNI_REQUIRE(h_src && h_out && h_sizes, "omni_host_png_encode: NULL pointer argument");
    OMNI_TRY(png_check("omni_host_png_encode", n, h, w, pitch, format, out_capacity));
    const size_t row = format == OMNI_PNG_GRAY1 ? ((size_t)w + 7) / 8 : (size_t)w * 3;
    // the span the pixels occupy goes over in one copy, with the caller's strides; the files come back in one copy of their bytes
    const size_t span = (size_t)(n - 1) * src_stride + (size_t)(h - 1) * pitch + row;
    const size_t in_bytes = pad16(span), out_bytes = (size_t)n * png_file_bound(h, w, format);
    OMNI_TRY(omni_ws_reserve(ctx, 3, in_bytes + out_bytes));
    u8 *d_in = (u8 *)ctx->ws[3], *d_out = d_in + in_bytes;
    OMNI_CUDA(cudaMemcpyAsync(d_in, h_src, span, cudaMemcpyHostToDevice, ctx->stream));
    OMNI_TRY(png_encode_run(ctx, d_in, n, src_stride, h, w, pitch, format, d_out, h_sizes, ctx->stream));
    size_t total = 0;
    for (int i = 0; i < n; i++) total += (size_t)h_sizes[i];
    OMNI_CUDA(cudaMemcpyAsync(h_out, d_out, total, cudaMemcpyDeviceToHost, ctx->stream));
    OMNI_CUDA(cudaStreamSynchronize(ctx->stream));
    return OMNI_OK;
}
