// fast_device.cuh -- device code and small host helpers shared by the bit-plane translation units (fast_kernels.cu: the
// dense generation; label_pipe.cu: the sparse generation of the fused colour+edge path).  Not part of the public ABI.
#pragma once
#include "fast_kernels.cuh"
#include <type_traits>

#define HY_WL_CAP 8192                 // words holding weak candidates (hysteresis worklist); more than this -> full sweeps

struct BitGeom {
    int h, w;
    int ww;            // words per row that hold pixels
    int ws;            // row stride in words (multiple of 4)
    size_t plane;      // words per plane
};

static inline BitGeom make_geom(int h, int w)
{
    BitGeom g;
    g.h = h; g.w = w;
    g.ww = (w + 31) >> 5;
    g.ws = (g.ww + 3) & ~3;
    g.plane = (size_t)g.ws * h;
    return g;
}


#define CELL_SHIFT 3
#define CELL_N (256 >> CELL_SHIFT)                 // 32 cells per axis
#define CELL_COUNT (CELL_N * CELL_N * CELL_N)
// RGB cells (fk_build_rgbcells): 4x4x4 colours each, 64 per axis
#define RC_SHIFT 2
#define RC_N (256 >> RC_SHIFT)
#define RC_COUNT (RC_N * RC_N * RC_N)
// workspace slot 5: [Lab candidate-cell table (u32) | hysteresis worklist | RGB cell tables: label nibbles, flags]
#define HYST_WL_OFFSET CELL_COUNT
#define RGBCELL_OFFSET (CELL_COUNT + 8192)
#define WS5_BYTES ((size_t)(CELL_COUNT + 8192) * sizeof(u32) + (size_t)RC_COUNT / 2 + (size_t)RC_COUNT / 8)


// cv2 BGR->Lab (8-bit) for one pixel, without the final saturate_cast: with OpenCV's tables L, a, b stay
// inside [0,255] for every input (L 0..255, a 42..226, b 20..223 over all 2^24 colours -- the exhaustive GPU test
// covers it), so the clamps of the generic kernel are no-ops here.
__device__ __forceinline__ void lab_noclamp(const u16 *gam, const u16 *cbrt, int B8, int G8, int R8, int &L, int &a, int &b)
{
    const int B = gam[B8], G = gam[G8], R = gam[R8];
    const int fX = cbrt[(R * 1777 + G * 1541 + B * 778 + 2048) >> 12];
    const int fY = cbrt[(R * 871 + G * 2929 + B * 296 + 2048) >> 12];
    const int fZ = cbrt[(R * 73 + G * 448 + B * 3575 + 2048) >> 12];
    L = (296 * fY - 1336934 + 16384) >> 15;
    a = (500 * (fX - fY) + 128 * 32768 + 16384) >> 15;
    b = (200 * (fY - fZ) + 128 * 32768 + 16384) >> 15;
}


#define RC_NIB_BYTES (RC_COUNT / 2)
#define RC_MB_BYTES (RC_COUNT / 8)
#define RC_MAX_K 16

// Zero fill riding on the assignment kernel: the edge pass needs its output planes cleared (dead tiles are never
// written, see edges3.cu); the assignment kernel is bound by instruction issue and leaves HBM idle, so every warp clears a
// slice of those planes with a few 16-byte stores per chunk of pixels instead of a separate memset competing with it.
struct ZeroJob { uint4 *p[2]; unsigned long long n16[2]; unsigned per[2]; };   // two regions, sizes in 16-byte units (0: nothing
                                                                                 // to do); per = units per chunk of pixels (launcher)


enum { ST_NONE = 0, ST_ER = 1, ST_DR = 2, ST_EC = 3, ST_DC = 4 };   // erode/dilate x RECT/CROSS

struct W64 { u32 lo, hi; };
__device__ __forceinline__ W64 w_shl(W64 a) { W64 r; r.lo = a.lo << 1; r.hi = __funnelshift_l(a.lo, a.hi, 1); return r; }
__device__ __forceinline__ W64 w_shr(W64 a) { W64 r; r.lo = __funnelshift_r(a.lo, a.hi, 1); r.hi = a.hi >> 1; return r; }
__device__ __forceinline__ W64 w_and3(W64 a, W64 b, W64 c) { W64 r; r.lo = a.lo & b.lo & c.lo; r.hi = a.hi & b.hi & c.hi; return r; }
__device__ __forceinline__ W64 w_or3(W64 a, W64 b, W64 c) { W64 r; r.lo = a.lo | b.lo | c.lo; r.hi = a.hi | b.hi | c.hi; return r; }

template <int OP>
__device__ __forceinline__ W64 morph_step(W64 u, W64 m, W64 d)
{
    if (OP == ST_ER) { W64 v = w_and3(u, m, d); return w_and3(v, w_shl(v), w_shr(v)); }
    if (OP == ST_DR) { W64 v = w_or3(u, m, d); return w_or3(v, w_shl(v), w_shr(v)); }
    if (OP == ST_EC) { W64 v = w_and3(m, w_shl(m), w_shr(m)); return w_and3(v, u, d); }
    if (OP == ST_DC) { W64 v = w_or3(m, w_shl(m), w_shr(m)); return w_or3(v, u, d); }
    return m;
}

__host__ __device__ constexpr int code_op(u32 code, int i) { return (int)((code >> (4 * i)) & 15u); }
__host__ __device__ constexpr int code_len(u32 code) { int n = 0; while (n < 8 && code_op(code, n) != ST_NONE) n++; return n; }
__host__ __device__ constexpr bool op_is_erode(int op) { return op == ST_ER || op == ST_EC; }

#define MORPH_TR 32          // rows per strip (default)
#define MORPH_TR_MID 48      // ... from 2048 warps on (A/B at 4096^2: 48 beats 32 and 64): TR + 16 (+4) rows are processed for TR produced
#define MORPH_TR_BIG 64      // ... from 8192 warps on (8192^2, K=16: less halo work wins once there are plenty of warps)
#define MORPH_MID_MIN_WARPS 2048
#define MORPH_BIG_MIN_WARPS 8192

// Output-of-range fix-up for a value that the step with opcode `next` will consume: columns outside the
// image and rows outside the image must read as that step's identity element.
// ROWFIX = false: every row the strip touches lies inside the image (all but the first and last strips of a plane), so only
// the columns need the fix-up -- the row tests were a third of the kernel's instructions.
// COLFIX = false: every window pixel of every lane of the warp lies inside the image (warps away from the left / right
// border), so the columns need no fix-up either.
template <int NEXT, bool ROWFIX, bool COLFIX>
__device__ __forceinline__ W64 oob_fix(W64 v, W64 colvalid, bool row_inside)
{
    if (NEXT == ST_NONE) { if (COLFIX) { v.lo &= colvalid.lo; v.hi &= colvalid.hi; } return v; }
    if (op_is_erode(NEXT)) {
        if (ROWFIX && !row_inside) { v.lo = v.hi = 0xffffffffu; return v; }
        if (COLFIX) { v.lo |= ~colvalid.lo; v.hi |= ~colvalid.hi; }
    } else {
        if (ROWFIX && !row_inside) { v.lo = v.hi = 0u; return v; }
        if (COLFIX) { v.lo &= colvalid.lo; v.hi &= colvalid.hi; }
    }
    return v;
}

template <u32 CODE, int S>
struct MorphChain {
    // applies steps S.. of CODE to `cur` (= image_S row `t - S`), updating the rolling rows
    template <int TAP, bool ROWFIX, bool COLFIX>
    static __device__ __forceinline__ void run(W64 cur, W64 (&p1)[8], W64 (&p2)[8], int t, int h, W64 colvalid, W64 &tap_out, W64 &fin)
    {
        constexpr int N = code_len(CODE);
        if (S == TAP) tap_out = cur;
        if constexpr (S < N) {
            constexpr int OP = code_op(CODE, S);
            constexpr int NEXT = (S + 1 < N) ? code_op(CODE, S + 1) : ST_NONE;
            W64 out = morph_step<OP>(p2[S], p1[S], cur);
            p2[S] = p1[S]; p1[S] = cur;
            const int r = t - S - 1;                       // row of image_{S+1} just produced
            out = oob_fix<NEXT, ROWFIX, COLFIX>(out, colvalid, !ROWFIX || (r >= 0 && r < h));
            MorphChain<CODE, S + 1>::template run<TAP, ROWFIX, COLFIX>(out, p1, p2, t, h, colvalid, tap_out, fin);
        } else {
            fin = cur;
        }
    }
};


struct MorphRuns {
    u32 *sbits, *cbits; u8 *edges; size_t estride, epitch; int aligned16;
    int *run_counts; u32 *run_items; E3RunOff off; int maxt;
    int zero_fill;                    // 1: the kernel writes the zeros of the dead tiles; 0: the planes were cleared beforehand
    int grow;                         // a tile is dead when the tile grown by `grow` pixels is uniform: 2 for blur 3 (5x5 neighbourhoods),
                                      // 3 for blur 5, 4 for blur 7 (radius of blur + Sobel); 0 is read as 2
};


constexpr u32 mk_code(int a, int b = 0, int c = 0, int d = 0, int e = 0, int f = 0, int g = 0, int hh = 0)
{
    return (u32)a | ((u32)b << 4) | ((u32)c << 8) | ((u32)d << 12) | ((u32)e << 16) | ((u32)f << 20) | ((u32)g << 24) | ((u32)hh << 28);
}
constexpr u32 CODE_R_OC = mk_code(ST_ER, ST_DR, ST_DR, ST_ER);                       // 02: RECT open, close
constexpr u32 CODE_C_O = mk_code(ST_EC, ST_DC);                                     // 03: cross open
constexpr u32 CODE_C_C = mk_code(ST_DC, ST_EC);                                     // 03: cross close
constexpr u32 CODE_C_OC = mk_code(ST_EC, ST_DC, ST_DC, ST_EC);                      // 03: cross open, close
constexpr u32 CODE_F_O = mk_code(ST_ER, ST_DR, ST_DR, ST_ER, ST_EC, ST_DC);
constexpr u32 CODE_F_C = mk_code(ST_ER, ST_DR, ST_DR, ST_ER, ST_DC, ST_EC);
constexpr u32 CODE_F_OC = mk_code(ST_ER, ST_DR, ST_DR, ST_ER, ST_EC, ST_DC, ST_DC, ST_EC);


// ---- helpers defined in fast_kernels.cu, shared with label_pipe.cu ---------------------------------------
cudaError_t fast_tables();
const u16 *fast_lab_table();                            // device address of the Lab tables (after fast_tables())
int persist_blocks(omni_ctx *ctx, int per_sm);
bool lut_below_k(const AssignParams &P);
int fast_rgb_boxes(omni_ctx *ctx, cudaStream_t st);     // ctx->d_rgb_boxes, built on first use
cudaError_t launch_build_cells(const AssignParams &P, u32 *cells, cudaStream_t st);
// flags / worklist: NULL = the ctx's own (d_flags[0..4], the list the edge kernel wrote); the banded host call passes its own
int run_hysteresis(omni_ctx *ctx, u32 *ebits, const u32 *cbits, const BitGeom &g, int K, u8 *d_edges, size_t e_plane, size_t epitch,
                   cudaStream_t st, int *flags = nullptr, const u32 *worklist = nullptr);
int run_hysteresis_wl(omni_ctx *ctx, u32 *ebits, const u32 *cbits, const BitGeom &g, int K, cudaStream_t st, const int *flags, const u32 *worklist);
int edge_pass_begin(omni_ctx *ctx, const BitGeom &g, int K, u32 *sbits, u32 *cbits, u8 *d_edges, size_t e_plane, size_t epitch,
                    cudaStream_t st, MorphRuns *R, bool *sparse, bool side_fill, ZeroJob *zjob = nullptr);
int morph03_kind(const omni_edge_params *p);
// stage-03 open/close with the ELLIPSE(morph_k) element for any size and count (morph_ellipse.cu): planes in a, b is scratch;
// *result = whichever of the two holds the end
int ellipse_morph_bits(omni_ctx *ctx, const omni_edge_params *prm, const BitGeom &g, int K, u32 *a, u32 *b, const u32 **result,
                       cudaStream_t st);

// shared-memory layout of the table-driven assignment kernels (fk_assign_rgbcell, fk_assign_slices)
#define RA_THREADS 1024
#define RA_WARPS (RA_THREADS / 32)
#define RA_OFF_MB RC_NIB_BYTES
#define RA_OFF_CBRT (RA_OFF_MB + RC_MB_BYTES)
#define RA_OFF_GAM (RA_OFF_CBRT + 2048 * 2)
#define RA_OFF_CTR (RA_OFF_GAM + 256 * 2)
#define RA_OFF_LUT (RA_OFF_CTR + OMNI_MAX_K * 16)
#define RA_OFF_WARP (RA_OFF_LUT + 64)
#define RA_WARP_BYTES (768 + 256 + 256)
#define RA_SMEM (RA_OFF_WARP + RA_WARPS * RA_WARP_BYTES)

void label_ws_bytes(int h, int w, int K, int nf, size_t out[OMNI_WS_SLOTS]);     // label_pipe.cu
// caller-layout packed planes (row pitch in bytes, LSB- / MSB-first) <-> internal bit-planes (label_pipe.cu)
cudaError_t launch_unpack_planes(const u8 *src, size_t splane, size_t spitch, int msb_first, int K, int h, int w, u32 *dst, int ws,
                                 size_t plane, int blocks, cudaStream_t st);
cudaError_t launch_pack_planes(const u32 *src, int ws, size_t plane, int K, int h, int w, u8 *dst, size_t dplane, size_t dpitch, int msb_first,
                               int blocks, cudaStream_t st);
void dense_ws_bytes(int h, int w, int K, int nf, int ksize, size_t out[OMNI_WS_SLOTS]);   // fast_kernels.cu

// opt-in device k-means of the Lab centres (kmeans.cu)
int kmeans_lab_batch(omni_ctx *ctx, const u8 *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch, const int *h_idx,
                     int n, int K, int attempts, int max_iter, float eps, unsigned long long seed, float *h_centers,
                     double *h_compactness, cudaStream_t st);

// sparse generation of the fused colour+edge call (label_pipe.cu); OMNI_ERR_UNSUPPORTED: use the dense generation
int sparse_color_edge(omni_ctx *ctx, const u8 *d_bgr, int nf, size_t frame_stride, int h, int w, size_t pitch, const AssignParams &P,
                      const omni_edge_params *prm, int low, int high, u8 *d_labels, size_t lpitch,
                      u8 *d_masks, size_t m_plane, size_t mpitch, u8 *d_edges, size_t e_plane, size_t epitch, cudaStream_t st);

