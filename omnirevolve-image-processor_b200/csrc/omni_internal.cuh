// omni_internal.cuh -- shared declarations of libomni_b200 (not part of the public ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/omni_b200.h"

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;

// ---- error plumbing --------------------------------------------------------------------------
void omni_set_error(const char *fmt, ...);
#define OMNI_CUDA(call)                                                                         \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            omni_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return OMNI_ERR_CUDA;                                                               \
        }                                                                                       \
    } while (0)
#define OMNI_REQUIRE(cond, ...)                                                                 \
    do {                                                                                        \
        if (!(cond)) { omni_set_error(__VA_ARGS__); return OMNI_ERR_ARG; }                      \
    } while (0)

// ---- small by-value parameter blocks (live in the kernel parameter bank) -----------------------
struct AssignParams {
    float c[OMNI_MAX_K * 3];   // centres (Lab, f32)
    u8 pal[OMNI_MAX_K * 3];    // palette (RGB u8) for the i16wrap variant
    u8 lut[OMNI_MAX_K];        // cluster id -> output label
    int K;
};
struct BlurParams {
    u16 w[OMNI_MAX_BLUR_K];
    int k;
};
struct MorphSE {               // structuring element as row spans, anchor (k/2, k/2), un-reflected (SURVEY A.0):
    int8_t x0[OMNI_MAX_MORPH_K];   // row i (dy = i - k/2) covers dx in [x0[i], x1[i]]; every row of RECT / ELLIPSE is non-empty
    int8_t x1[OMNI_MAX_MORPH_K];
    int k;
};
struct ResizeTabDev {          // fractional INTER_AREA tables on the device (per axis: ofs[D+1], si[], alpha[])
    const int *xofs; const int *xsi; const float *xal;
    const int *yofs; const int *ysi; const float *yal;
};

struct ResizeTab {
    void *d_blob = nullptr;
    ResizeTabDev dev{};
};

#define OMNI_WS_SLOTS 13
struct omni_ctx {
    int device = 0;
    int fast = 1;
    // grow-only device scratch
    void *ws[OMNI_WS_SLOTS] = {};          // 0-2 generic planes, 3 host staging, 4 bit-planes, 5 misc, 6 edge run lists, 7-10 trace.cu, 11 png_encode.cu, 12 thinned / byte planes of omni_centerlines_packed
    size_t ws_bytes[OMNI_WS_SLOTS] = {};
    int *d_flags = nullptr;          // 64 ints of device flags / counters
    unsigned long long *d_counts = nullptr;   // 4*OMNI_MAX_K counters
    int *h_flags = nullptr;          // pinned mirror
    unsigned long long *h_counts = nullptr;
    cudaStream_t stream = nullptr;   // own stream for the omni_host_* entry points
    std::map<std::tuple<int, int, int, int>, ResizeTab> resize_tabs;
    int last_hyst_passes = 0;
    cudaStream_t last_hyst_stream = nullptr;   // the stream the pass count in d_flags[0] is ordered on
    // launch accounting / per-kernel CUDA-event timing (omni_profile_*)
    long long launches = 0;
    int prof_on = 0;
    struct ProfRec { const char *name; cudaEvent_t a, b; };
    std::vector<ProfRec> prof;
    std::vector<cudaEvent_t> ev_pool;
    int sm_count = 0;
    int hyst_blocks = 0;
    int thin_blocks = 0;             // co-resident CTAs of the cooperative thinning kernel (0 = not queried yet)
    int e3s_per_sm = 0;              // resident CTAs per SM of the sparse edge kernel (0 = not queried yet)
    int assign_rgbcell = 1;          // 0: Lab-cell assignment kernel (the previous generation; set_fast_path mode 2)
    int edge_sparse = 1;             // 0: dense edge kernel (A/B runs, OMNI_B200_EDGE_DENSE=1)
    int assume_binary = 0;           // omni_set_assume_binary_masks: omni_edges does not wait for the "masks are {0,255}" check
    // side streams + events of the pipelined host-buffer call (fast_host_color_edge)
    int pipe_ready = 0;
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t pipe_ev[24] = {};          // 8 H2D bands, 8 morph bands, 4 pipeline joins, 2 zero-fill fork/join
    cudaEvent_t edge_join = nullptr;        // pending join of the zero-fill side stream (edge_pass_begin -> edges_from_bits)
    int occ_assign_lab = 0, occ_assign_pal = 0, occ_assign_rgb = 0, occ_assign_i16 = 0;   // resident CTAs per SM of the persistent assignment kernels
    // centres the candidate-cell table in ws[5] was built for (fast colour assignment); cleared by omni_ws_reserve when it
    // reallocates ws[5] and by omni_set_table_cache(0)
    int cells_valid = 0, cells_K = 0;
    void *cells_stream = nullptr;
    float cells_c[OMNI_MAX_K * 3];
    u8 cells_lut[OMNI_MAX_K] = {};
    // the same for the tables of the sparse generation (label_pipe.cu; tail of ws[5]), cleared in the same two places
    int cells3_valid = 0, cells3_K = 0;
    void *cells3_stream = nullptr;
    float cells3_c[OMNI_MAX_K * 3];
    u8 cells3_lut[OMNI_MAX_K] = {};
    u8 *d_rgb_boxes3 = nullptr;                // d_rgb_boxes in the cell order of fk_assign_slices
    int table_cache = 1;                       // 0: rebuild the candidate tables on every call (omni_set_table_cache)
    int tables_hold = 0;                       // inside one banded host call: the tables of its first band serve the other bands
    int occ_assign_sl = 0;
    // streams / events / pinned counts of omni_host_color_edge_packed (two staging slots)
    int pk_ready = 0;
    cudaStream_t pk_in = nullptr, pk_out = nullptr;
    cudaEvent_t pk_ev[7] = {};
    cudaEvent_t bd_ev[3 * 16 + 2] = {};        // banded single-image call: H2D of a band done, band image done, outputs of a band ready, start, edges ready
    int bd_ready = 0;
    cudaStream_t bd_tail = nullptr;            // packing / merge / hysteresis of the bands, in band order
    omni_ctx *band_helper = nullptr;           // second set of workspaces + stream: two band images in flight
    int band_overlap = 1;
    int host_bands = 2;                        // omni_set_host_bands: 0 = off, 1 = edge planes after the last band, 2 = edge rows with their band
    int last_band_resends = 0;                 // bands of the last banded call whose edge rows were sent twice (mode 2)
    unsigned long long *pk_counts = nullptr;
    size_t pk_counts_cap = 0;                  // groups of 3 * OMNI_MAX_K counts
    int pipeline = 1;                          // fused colour+edge call: 1 = sparse generation (label_pipe.cu), 0 = dense generation
    u8 *d_rgb_boxes = nullptr;                 // exact Lab box of every 4x4x4 RGB cell (centre-independent, built on first use)             // co-resident CTAs of the cooperative hysteresis kernel (0 = not queried yet)
    // result of the last omni_trace_centerlines / omni_centerlines_packed call: polylines in ws[10] (points from offset 0, path
    // lengths from trace_lens_off), sizes and per-component rows on the host
    int trace_valid = 0, trace_K = 0;
    long long trace_points = 0, trace_paths = 0;
    size_t trace_lens_off = 0;
    std::vector<long long> trace_info;         // per plane: total_fg, components, polylines, points
    std::vector<int32_t> trace_comp;           // per component: left, top, width, height, area, polylines
};

// Brackets one kernel launch: counts it and, when profiling is on, records a CUDA event pair on the
// launching stream (read back by omni_profile_summary).
struct KScope {
    omni_ctx *c; cudaStream_t st; cudaEvent_t b = nullptr;
    KScope(omni_ctx *ctx, const char *name, cudaStream_t s);
    ~KScope();
};
#define OMNI_LAUNCH(ctx, st, name, expr) do { KScope ks__(ctx, name, st); OMNI_CUDA(expr); } while (0)

int omni_ws_reserve(omni_ctx *ctx, int slot, size_t bytes);
// stage 04 trace_centerlines (trace.cu): run on K planes (synchronises st), then copy the results out
int trace_run(omni_ctx *ctx, const u8 *d_skel, int K, int h, int w, size_t plane_stride, size_t pitch, int64_t *h_info,
              cudaStream_t st);
int trace_results(omni_ctx *ctx, int32_t *points, int32_t *path_len, int32_t *comp);
// omni_centerlines_packed: planes per chunk (at least 32, more while the labels of a chunk fit 256 MiB), and the run (capi.cu
// checks the arguments; h_bits != NULL: host planes, each chunk copied in first; synchronises st)
int centerlines_chunk(int h, int w, int n_planes);
int centerlines_packed_run(omni_ctx *ctx, const u8 *d_bits, const u8 *h_bits, int n_planes, int h, int w, size_t plane_stride,
                           size_t pitch, int bit_order, int max_iter, int64_t *h_info, cudaStream_t st);
// PNG encoder (png_encode.cu): a segment holds at most PNG_SEG_MAX filtered bytes (one stored block) and PNG_SEG_ROWS rows
constexpr int PNG_SEG_MAX = 61440;
constexpr int PNG_SEG_ROWS = 256;
int png_segment_rows(int w, int fmt);
size_t png_file_bound(int h, int w, int fmt);
// n files into d_out (back to back, room for n * png_file_bound checked by the caller), sizes into h_sizes; synchronises st
int png_encode_run(omni_ctx *ctx, const u8 *d_src, int n, size_t src_stride, int h, int w, size_t pitch, int fmt, u8 *d_out,
                   int64_t *h_sizes, cudaStream_t st);
const ResizeTab *omni_get_resize_tab(omni_ctx *ctx, int sh, int sw, int dh, int dw, cudaStream_t st);
void omni_build_se(int shape_ellipse, int k, MorphSE *se);
int omni_gauss_weights(int k, BlurParams *bp);

// ---- generic kernels (generic_kernels.cu): any u8 data, any supported parameter --------------
cudaError_t g_resize_area(const u8 *src, int sh, int sw, size_t spitch, u8 *dst, int dh, int dw, size_t dpitch,
                          const ResizeTabDev *tab, cudaStream_t st);
cudaError_t g_assign(const u8 *px, int h, int w, size_t pitch, const AssignParams &P, int mode_lab,
                     u8 *labels, size_t lpitch, cudaStream_t st);
cudaError_t g_onehot(const u8 *labels, int h, int w, size_t lpitch, int K, u8 *planes, size_t plane_stride,
                     size_t pitch, cudaStream_t st);
cudaError_t g_morph(const u8 *src, size_t s_plane, size_t spitch, u8 *dst, size_t d_plane, size_t dpitch,
                    int K, int h, int w, const MorphSE &se, int is_dilate, cudaStream_t st);
cudaError_t g_blur(const u8 *src, size_t s_plane, size_t spitch, u8 *dst, size_t d_plane, size_t dpitch,
                   int K, int h, int w, const BlurParams &bp, cudaStream_t st);
cudaError_t g_canny_nms(const u8 *src, size_t s_plane, size_t spitch, u8 *state, size_t d_plane, size_t dpitch,
                        int K, int h, int w, int low, int high, cudaStream_t st);
cudaError_t g_hyst_pass(u8 *state, size_t plane, size_t pitch, int K, int h, int w, int *d_changed, cudaStream_t st);
cudaError_t g_hyst_final(u8 *state, size_t plane, size_t pitch, int K, int h, int w, cudaStream_t st);
cudaError_t g_count_nonzero(const u8 *planes, size_t plane, size_t pitch, int K, int h, int w,
                            unsigned long long *d_counts, cudaStream_t st);
cudaError_t g_count_labels(const u8 *labels, size_t pitch, int h, int w, int K, unsigned long long *d_counts,
                           cudaStream_t st);
cudaError_t g_composite(const u8 *edges, size_t plane, size_t pitch, int K, int h, int w, const u8 *colors_bgr,
                        u8 *canvas, size_t cpitch, cudaStream_t st);
cudaError_t g_skeleton_degree(const u8 *skel, size_t s_plane, size_t spitch, int K, int h, int w, u8 *deg, size_t d_plane, size_t dpitch,
                              u8 *nodes, size_t n_plane, size_t npitch, cudaStream_t st);
cudaError_t g_pack_bytes(const u8 *src, size_t s_plane, size_t spitch, int K, int h, int w, u8 *dst, size_t d_plane, size_t dpitch,
                         int msb_first, unsigned long long *counts, cudaStream_t st);
cudaError_t g_copy2d_planes(const u8 *src, size_t s_plane, size_t spitch, u8 *dst, size_t d_plane, size_t dpitch,
                            int K, int h, int w, cudaStream_t st);

// alignment class of a set of byte planes for the 32-pixel stores: 2 = base, plane stride and pitch are multiples of 32, 1 = of 16
static inline int plane_align(const void *base, size_t plane, size_t pitch)
{
    const size_t v = (size_t)(uintptr_t)base | plane | pitch;
    return base == nullptr ? 0 : (v % 32 == 0) ? 2 : (v % 16 == 0) ? 1 : 0;
}

#ifdef __CUDACC__
// bits i of a 32-bit word whose pixel (start_px + i) lies in [0, w)
__device__ __forceinline__ u32 range_mask(int start_px, int w)
{
    int lo = max(0, -start_px), hi = min(32, w - start_px);
    if (hi <= lo) return 0u;
    u32 m = hi >= 32 ? 0xffffffffu : ((1u << hi) - 1u);
    return m & ~((1u << lo) - 1u);
}

// 4 mask bits -> 4 bytes of 0x00 / 0xFF
__device__ __forceinline__ u32 expand4(u32 nib)
{
    return ((nib * 0x00204081u) & 0x01010101u) * 255u;
}

// one 32-byte store (sm_100: STG.256): a lane writes a whole sector, a warp of adjacent lanes one contiguous run
__device__ __forceinline__ void st_global_256(void *p, const uint4 a, const uint4 b)
{
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y),
                 "r"(b.z), "r"(b.w) : "memory");
}
__device__ __forceinline__ void store_32bytes(u8 *dst, const uint4 a, const uint4 b, int align)
{
#ifndef OMNI_NO_ST256
    if (align == 2) { st_global_256(dst, a, b); return; }
#endif
    uint4 *p = reinterpret_cast<uint4 *>(dst);
    p[0] = a; p[1] = b;
}

// store 32 pixels (bits of `word`) as 0/255 bytes at dst (pixel x0 = first), only pixels < w.
// align (host: plane_align()): 0 = byte stores, 1 = rows / planes 16-byte aligned, 2 = 32-byte aligned
__device__ __forceinline__ void store_word_bytes(u8 *row, int x0, int w, u32 word, int align)
{
    if (x0 + 32 <= w && align) {
        uint4 a, b;
        a.x = expand4(word & 15u);         a.y = expand4((word >> 4) & 15u);
        a.z = expand4((word >> 8) & 15u);  a.w = expand4((word >> 12) & 15u);
        b.x = expand4((word >> 16) & 15u); b.y = expand4((word >> 20) & 15u);
        b.z = expand4((word >> 24) & 15u); b.w = expand4(word >> 28);
        store_32bytes(row + x0, a, b, align);
    } else {
        int n = min(32, w - x0);
        for (int i = 0; i < n; i++) row[x0 + i] = (word >> i) & 1u ? 255 : 0;
    }
}

// same, with the bit -> byte expansion done by a 256-entry shared-memory table (8 mask bits -> 8 bytes)
__device__ __forceinline__ void expand_lut_init(uint2 *lut8, int tid, int nthreads)
{
    for (int b = tid; b < 256; b += nthreads) lut8[b] = make_uint2(expand4(b & 15u), expand4((u32)b >> 4));
}
__device__ __forceinline__ void store_word_bytes_lut(u8 *row, int x0, int w, u32 word, int align, const uint2 *lut8)
{
    if (x0 + 32 <= w && align) {
        const uint2 a = lut8[word & 255u], b = lut8[(word >> 8) & 255u], c = lut8[(word >> 16) & 255u], d = lut8[word >> 24];
        store_32bytes(row + x0, make_uint4(a.x, a.y, b.x, b.y), make_uint4(c.x, c.y, d.x, d.y), align);
    } else {
        int n = min(32, w - x0);
        for (int i = 0; i < n; i++) row[x0 + i] = (word >> i) & 1u ? 255 : 0;
    }
}

// cv2.cvtColor(u8 BGR -> Lab) integer pipeline (02_color_extract.py:35; SURVEY A.3); tables: gamma[256], cbrt[2041]
__device__ __forceinline__ int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }

__device__ __forceinline__ void bgr2lab_px(const u16 *gam, const u16 *cbrt, int B8, int G8, int R8, int &L, int &a, int &b)
{
    int B = gam[B8], G = gam[G8], R = gam[R8];
    int fX = cbrt[descale(R * 1777 + G * 1541 + B * 778, 12)];
    int fY = cbrt[descale(R * 871 + G * 2929 + B * 296, 12)];
    int fZ = cbrt[descale(R * 73 + G * 448 + B * 3575, 12)];
    L = min(255, max(0, descale(296 * fY - 1336934, 15)));
    a = min(255, max(0, descale(500 * (fX - fY) + 128 * 32768, 15)));
    b = min(255, max(0, descale(200 * (fY - fZ) + 128 * 32768, 15)));
}
#endif
