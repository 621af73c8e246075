// fast_kernels.cu -- the bit-plane fast path of libomni_b200 (the default for the parameter ranges the
// pipeline uses; everything else goes to generic_kernels.cu).
//
// Data layout.  After the colour assignment every layer is a BIT-PLANE: one u32 word holds 32
// horizontally adjacent pixels (bit i of word c of row y = pixel x = 32c + i), rows are `ws` words apart
// (ws = words per row rounded up to 4), planes `plane` words apart.  K=8 planes of a 4096^2 image are
// 16.8 MB -- they live in the 126 MB L2 between the kernels, so HBM sees only the image read (3 B/px) and
// the mask / edge byte planes written once each (2K B/px): the algorithmic N*(3+2K) bytes.
//
//   fk_assign_rgbcell image -> [labels] + raw one-hot bit-planes P0           (02:35-36,53-55,121-127,150)
//                     (RGB-cell tables in shared memory; fk_assign_bits = the Lab-cell generation, K > 16 / palette mode);
//                     its warps also clear the edge planes for the dead tiles of the edge pass (ZeroJob)
//   fk_morph<CODE>    P0 -> RECT-3 open/close -> mask BYTES (mask.png content) (02:151-154)
//                        -> ELLIPSE-3 open/close -> bit-planes M2              (03:23-30)
//                        + run lists of the live tiles for the sparse edge kernel (MorphRuns)
//   fk_edges3_simd    M2 -> blur-3 -> Sobel -> NMS -> strong/candidate bit-planes S, C + edge BYTES (edges3.cu; 03:33-34)
//   fk_hysteresis     E = S; E |= C & dilate8(E) to the global fixed point, promoted pixels patched into the edge bytes
//   also here: fractional / 2:1 resize (01), swatch mode (02:82-109), Zhang-Suen thinning (04:35-99), frame batches and
//   the band-pipelined host-buffer call
//
// Reference call sites are relative to /root/reference/image_processor/.  Arithmetic: SURVEY.md App. A.
#include "fast_kernels.cuh"
#include "omni_tables.inc"
#include "fast_device.cuh"

#include <algorithm>
#include <type_traits>
#include <cooperative_groups.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
namespace cg = cooperative_groups;

#define FK_TRY(expr) do { int rc__ = (expr); if (rc__ != OMNI_OK) return rc__; } while (0)

// ------------------------------------------------------------------------------------------------
// shared helpers
// ------------------------------------------------------------------------------------------------
__device__ u16 f_lab_tab[256 + 2048];          // gamma[256] | cbrt[2041]
static bool f_tab_ready[64] = {false};

cudaError_t fast_tables()
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 64 && f_tab_ready[dev]) return cudaSuccess;
    e = cudaMemcpyToSymbol(f_lab_tab, OMNI_LAB_GAMMA, sizeof(OMNI_LAB_GAMMA), 0);
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbol(f_lab_tab, OMNI_LAB_CBRT, sizeof(OMNI_LAB_CBRT), 256 * sizeof(u16));
    if (e != cudaSuccess) return e;
    // one-time upload from pageable memory through the legacy stream: callers launch on non-blocking streams, which the
    // legacy stream does not order against -- wait for the copy to land before anything can read the tables
    e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return e;
    if (dev < 64) f_tab_ready[dev] = true;
    return cudaSuccess;
}


// ------------------------------------------------------------------------------------------------
// stage 01: exact 2:1 INTER_AREA, vectorised (01_resize.py:20; SURVEY A.1 (i))
// Each thread produces 4 destination pixels (12 bytes) from 2 x 24 source bytes.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fk_resize_2x(const u8 *__restrict__ src, size_t spitch, u8 *__restrict__ dst, int dh, int dw,
                                                    size_t dpitch)
{
    int gx = blockIdx.x * blockDim.x + threadIdx.x;         // group of 4 destination pixels
    int y = blockIdx.y * blockDim.y + threadIdx.y;
    int x = gx * 4;
    if (x >= dw || y >= dh) return;
    const u8 *r0 = src + (size_t)(2 * y) * spitch + 6 * x, *r1 = r0 + spitch;
    u8 *o = dst + (size_t)y * dpitch + 3 * x;
    if (x + 4 <= dw) {
        // 24 source bytes per row = 3 x 8 B (8-byte aligned: 6*x with x % 4 == 0, pitches % 8 == 0 checked by the host)
        uint2 a0 = *reinterpret_cast<const uint2 *>(r0), a1 = *reinterpret_cast<const uint2 *>(r0 + 8),
              a2 = *reinterpret_cast<const uint2 *>(r0 + 16);
        uint2 b0 = *reinterpret_cast<const uint2 *>(r1), b1 = *reinterpret_cast<const uint2 *>(r1 + 8),
              b2 = *reinterpret_cast<const uint2 *>(r1 + 16);
        u32 sa[6] = {a0.x, a0.y, a1.x, a1.y, a2.x, a2.y}, sb[6] = {b0.x, b0.y, b1.x, b1.y, b2.x, b2.y};
        u8 out[12];
#pragma unroll
        for (int p = 0; p < 4; p++)
#pragma unroll
            for (int c = 0; c < 3; c++) {
                int i0 = 6 * p + c, i1 = i0 + 3;
                u32 s = ((sa[i0 >> 2] >> (8 * (i0 & 3))) & 255u) + ((sa[i1 >> 2] >> (8 * (i1 & 3))) & 255u) +
                        ((sb[i0 >> 2] >> (8 * (i0 & 3))) & 255u) + ((sb[i1 >> 2] >> (8 * (i1 & 3))) & 255u);
                out[3 * p + c] = (u8)((s + 2u) >> 2);
            }
        u32 w0 = out[0] | (out[1] << 8) | (out[2] << 16) | ((u32)out[3] << 24);
        u32 w1 = out[4] | (out[5] << 8) | (out[6] << 16) | ((u32)out[7] << 24);
        u32 w2 = out[8] | (out[9] << 8) | (out[10] << 16) | ((u32)out[11] << 24);
        u32 *po = reinterpret_cast<u32 *>(o);
        po[0] = w0; po[1] = w1; po[2] = w2;
    } else {
        for (int p = 0; x + p < dw; p++)
            for (int c = 0; c < 3; c++)
                o[3 * p + c] = (u8)((r0[6 * p + c] + r0[6 * p + c + 3] + r1[6 * p + c] + r1[6 * p + c + 3] + 2) >> 2);
    }
}

bool fast_resize_2x_ok(const u8 *src, int sw, size_t spitch, const u8 *dst, int dw, size_t dpitch)
{
    (void)sw; (void)dw;
    return ((uintptr_t)src % 8 == 0) && (spitch % 8 == 0) && ((uintptr_t)dst % 4 == 0) && (dpitch % 4 == 0);
}

cudaError_t fast_resize_2x(const u8 *src, size_t spitch, u8 *dst, int dh, int dw, size_t dpitch, cudaStream_t st)
{
    dim3 b(64, 4), g(((dw + 3) / 4 + 63) / 64, (dh + 3) / 4);
    fk_resize_2x<<<g, b, 0, st>>>(src, spitch, dst, dh, dw, dpitch);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// stage 01: fractional INTER_AREA (the default max_dimension=2000 path, e.g. 4096 -> 2000), SURVEY A.1 (iii).
// A CTA produces a tile of RF_TX x RF_TY destination pixels: the source rectangle the tile touches is staged in
// shared memory with coalesced 16-byte row segments (every source byte crosses HBM once), then each thread walks
// OpenCV's tables for its destination pixels exactly like the generic kernel (same float32 operation order:
// per source row a sequential horizontal sum, then sum = beta * buf / sum += beta * buf).
// ------------------------------------------------------------------------------------------------
#define RF_TX 128                         // destination columns per CTA (one per thread of a half)
#define RF_TY 16                          // destination rows per CTA (RF_TY / 2 per half)
#define RF_THREADS 256
#define RF_MAXTAPS 8                      // source pixels per destination pixel and axis the register path holds

// A thread owns one destination column of the tile: its horizontal taps (shared-memory byte offsets + weights) sit in
// registers for all its destination rows, and the horizontal sum of a source row is reused when the next destination
// row shares that source row (the fractional rows do).
template <int MT>                         // taps per destination pixel and axis held in registers (>= floor(scale) + 2)
__global__ void __launch_bounds__(RF_THREADS) fk_resize_frac(const u8 *__restrict__ src, int sh, int sw, size_t spitch, u8 *__restrict__ dst,
                                                             int dh, int dw, size_t dpitch, const ResizeTabDev t, int spitch_s, int vec_ok)
{
    extern __shared__ __align__(16) u8 s_src[];
    const int x0 = blockIdx.x * RF_TX, y0 = blockIdx.y * RF_TY;
    const int x1 = min(dw, x0 + RF_TX), y1 = min(dh, y0 + RF_TY);
    const int xs0 = t.xsi[t.xofs[x0]], xs1 = t.xsi[t.xofs[x1] - 1];          // source columns [xs0, xs1]
    const int ys0 = t.ysi[t.yofs[y0]], ys1 = t.ysi[t.yofs[y1] - 1];          // source rows    [ys0, ys1]
    const int b0 = (3 * xs0) & ~15;                                            // first staged byte of a row (16-aligned)
    const int nbytes = 3 * (xs1 + 1) - b0;
    const int nrows = ys1 - ys0 + 1;
    if (vec_ok) {
        // 16-byte vectors; 64 threads per source row, four rows per pass and three passes in flight (no divisions, and the
        // staging is latency-bound otherwise)
        const int nv = (nbytes + 15) >> 4;
        const int lr = threadIdx.x >> 6, v0 = threadIdx.x & 63;
        for (int vb = v0; vb < nv; vb += 64) {
            const bool vec = b0 + 16 * vb + 16 <= 3 * sw;                      // never read past the row's pixels
            for (int r0 = lr; r0 < nrows; r0 += 12) {
                uint4 val[3];
#pragma unroll
                for (int q = 0; q < 3; q++) {
                    const int r = r0 + 4 * q;
                    if (r < nrows && vec) val[q] = __ldg(reinterpret_cast<const uint4 *>(src + (size_t)(ys0 + r) * spitch + b0 + 16 * vb));
                }
#pragma unroll
                for (int q = 0; q < 3; q++) {
                    const int r = r0 + 4 * q;
                    if (r < nrows) {
                        u8 *d = s_src + (size_t)r * spitch_s + 16 * vb;
                        if (vec) *reinterpret_cast<uint4 *>(d) = val[q];
                        else {
                            const u8 *g = src + (size_t)(ys0 + r) * spitch + b0 + 16 * vb;
                            for (int e = 0; b0 + 16 * vb + e < 3 * sw; e++) d[e] = g[e];
                        }
                    }
                }
            }
        }
    } else {
        for (int r = threadIdx.x / 64; r < nrows; r += RF_THREADS / 64)
            for (int v = threadIdx.x & 63; v < nbytes; v += 64)
                s_src[(size_t)r * spitch_s + v] = src[(size_t)(ys0 + r) * spitch + b0 + v];
    }
    __syncthreads();
    const int lx = threadIdx.x & (RF_TX - 1), half = threadIdx.x / RF_TX;
    const int x = x0 + lx;
    if (x >= x1) return;
    const int xb = t.xofs[x], nt = t.xofs[x + 1] - xb;
    int off[MT];
    float wgt[MT];
#pragma unroll
    for (int q = 0; q < MT; q++) {
        off[q] = q < nt ? 3 * t.xsi[xb + q] - b0 : 0;
        wgt[q] = q < nt ? t.xal[xb + q] : 0.f;
    }
    const int ya = y0 + half * (RF_TY / 2), yb = min(y1, ya + RF_TY / 2);
    int cached = -1;
    float h0 = 0.f, h1 = 0.f, h2 = 0.f;
    for (int y = ya; y < yb; y++) {
        const int jb = t.yofs[y], je = t.yofs[y + 1];
        float s0 = 0.f, s1 = 0.f, s2 = 0.f;
        for (int j = jb; j < je; j++) {
            const int sr = t.ysi[j];
            const float beta = t.yal[j];
            if (sr != cached) {
                const u8 *r = s_src + (size_t)(sr - ys0) * spitch_s;
                h0 = h1 = h2 = 0.f;
#pragma unroll
                for (int q = 0; q < MT; q++)
                    if (q < nt) {                                              // same order as OpenCV: k ascending, 0 + p*a first
                        const u8 *p = r + off[q];
                        h0 = __fadd_rn(h0, __fmul_rn((float)p[0], wgt[q]));
                        h1 = __fadd_rn(h1, __fmul_rn((float)p[1], wgt[q]));
                        h2 = __fadd_rn(h2, __fmul_rn((float)p[2], wgt[q]));
                    }
                cached = sr;
            }
            if (j == jb) { s0 = __fmul_rn(beta, h0); s1 = __fmul_rn(beta, h1); s2 = __fmul_rn(beta, h2); }
            else {
                s0 = __fadd_rn(s0, __fmul_rn(beta, h0)); s1 = __fadd_rn(s1, __fmul_rn(beta, h1)); s2 = __fadd_rn(s2, __fmul_rn(beta, h2));
            }
        }
        u8 *o = dst + (size_t)y * dpitch + 3 * x;
        o[0] = (u8)min(255, max(0, __float2int_rn(s0)));
        o[1] = (u8)min(255, max(0, __float2int_rn(s1)));
        o[2] = (u8)min(255, max(0, __float2int_rn(s2)));
    }
}

// returns cudaErrorNotSupported when the staged rectangle would not fit (very large ratios): caller uses the generic kernel
cudaError_t fast_resize_frac(const u8 *src, int sh, int sw, size_t spitch, u8 *dst, int dh, int dw, size_t dpitch, const ResizeTabDev *tab,
                             cudaStream_t st)
{
    const double scx = (double)sw / dw, scy = (double)sh / dh;
    const int vec_ok = (((uintptr_t)src | spitch) & 15) == 0;
    // a destination pixel covers at most ceil(scale) + 1 source pixels per axis: the register path holds RF_MAXTAPS
    if ((int)ceil(scx) + 1 > RF_MAXTAPS) return cudaErrorNotSupported;
    // widest source span of a tile: RF_TX destination pixels worth of source columns, plus alignment slack
    const int span_px = (int)(scx * RF_TX) + 3;
    const int spitch_s = ((3 * span_px + 15 + 15) & ~15) + 16;
    const int rows = (int)(scy * RF_TY) + 3;
    const size_t smem = (size_t)rows * spitch_s;
    if (smem > 200 * 1024) return cudaErrorNotSupported;
    const int need = (int)floor(scx) + 2;
    dim3 grid((dw + RF_TX - 1) / RF_TX, (dh + RF_TY - 1) / RF_TY);
#define RF_LAUNCH(MT)                                                                                                             \
    do {                                                                                                                          \
        cudaError_t e = cudaFuncSetAttribute(fk_resize_frac<MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);        \
        if (e != cudaSuccess) return e;                                                                                           \
        fk_resize_frac<MT><<<grid, RF_THREADS, smem, st>>>(src, sh, sw, spitch, dst, dh, dw, dpitch, *tab, spitch_s, vec_ok);     \
    } while (0)
    if (need <= 3) RF_LAUNCH(3);
    else if (need <= 4) RF_LAUNCH(4);
    else if (need <= 6) RF_LAUNCH(6);
    else RF_LAUNCH(RF_MAXTAPS);
#undef RF_LAUNCH
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// stage 02: colour assignment -> labels and/or one-hot bit-planes
//
// Exact pruning of the centre loop.  Lab space is cut into 8x8x8 cells; fk_build_cells gives every cell the
// set of centres that can be the nearest one for SOME point of the cell: with dmin_k / dmax_k the smallest /
// largest true squared distance from centre k to the cell's box, centre k is kept iff
// dmin_k <= min_j dmax_j + 1.  A dropped centre is more than 1 farther (squared) than the true nearest centre
// of every point in the cell, and the float32 evaluation (02:53-55 order, every operation rounded) is off by
// < 0.05, so it can never win or tie the argmin.  The kept centres are evaluated with the reference's exact
// float32 sequence in ascending k with a strict '<', i.e. np.argmin's first-minimum rule.  A pixel visits ~1.3
// (K=8) .. 1.5 (K=16) centres instead of K.
//
// A warp owns 256 consecutive pixels of a row (lane l: pixels l, l+32, .., l+224).  Bit-plane words come from
// __match_any_sync on the labels of a 32-pixel group: the mask a lane gets back IS the word of its label's
// plane; the lowest lane of each label stores it (the planes are zeroed beforehand).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fk_build_cells(const __grid_constant__ AssignParams P, u32 *__restrict__ cells)
{
    // float32 is enough here: coordinates <= 255 and |centre| < 1e4 (checked), so dmin/dmax carry an absolute
    // error far below the slack of 2 used in the test (1 for the argument above + 1 for this arithmetic)
    const int ci = blockIdx.x * blockDim.x + threadIdx.x;
    if (ci >= CELL_COUNT) return;
    const int K = P.K;
    const float lo[3] = {(float)((ci >> (2 * 5)) << CELL_SHIFT), (float)(((ci >> 5) & 31) << CELL_SHIFT), (float)((ci & 31) << CELL_SHIFT)};
    const float span = (float)((1 << CELL_SHIFT) - 1);
    float U = 3.0e38f;
    bool sane = true;
    for (int k = 0; k < K; k++) {
        float dmax = 0.f;
#pragma unroll
        for (int d = 0; d < 3; d++) {
            float c = P.c[3 * k + d];
            sane = sane && (fabsf(c) < 1.0e4f);                 // also false for NaN
            float m = fmaxf(fabsf(lo[d] - c), fabsf(lo[d] + span - c));
            dmax += m * m;
        }
        U = fminf(U, dmax);
    }
    u32 mask = 0u;
    for (int k = 0; k < K; k++) {
        float dmin = 0.f;
#pragma unroll
        for (int d = 0; d < 3; d++) {
            float c = P.c[3 * k + d];
            float n = fminf(fmaxf(c, lo[d]), lo[d] + span);
            dmin += (n - c) * (n - c);
        }
        if (dmin <= U + 2.0f) mask |= 1u << k;
    }
    if (!sane || mask == 0u) mask = K >= 32 ? 0xffffffffu : ((1u << K) - 1u);
    cells[ci] = mask;
}

// ---- RGB-cell variant (the default for Lab centres) -------------------------------------------------------
// The same exact pruning, one level earlier: the RGB cube is cut into 64^3 cells of 4x4x4 colours and every cell gets
// the set of centres that can be nearest for SOME colour of the cell.  The cell's image in Lab space is bounded by the
// exact box of its 64 colours (fk_rgb_boxes: cv2's integer Lab of every colour, min / max per channel; the boxes depend
// only on the colour space, so they are computed once per context, 1.5 MB).  The box goes through
// the dmin / dmax test of fk_build_cells.  ~88 % (K=8) / ~82 % (K=16) of the pixels of the benchmark images fall
// into a cell with ONE candidate: their label is a table lookup, no Lab conversion at all.  The others (flagged
// in a second, one-bit table) are compacted over the warp (shared-memory queue) and take the Lab-cell path of
// fk_assign_bits: Lab conversion, candidate set of their Lab cell, the reference's float32 evaluation.
// The tables are 4 bits (label, K <= 16) + 1 bit (several candidates) per cell = 160 KB and live in SHARED memory: one
// 1024-thread CTA per SM copies them in once and then streams pixels (random lookups from global memory were bound
// by L1 sector traffic: the +-12 noise of neighbouring pixels scatters a warp's 32 lookups over ~20 sectors).
// exact Lab bounding box of every RGB cell: boxes[6 * cell + (0..2)] = min L, a, b; [3..5] = max (centre-independent)
__global__ void __launch_bounds__(256) fk_rgb_boxes(u8 *__restrict__ boxes)
{
    const int ci = blockIdx.x * blockDim.x + threadIdx.x;               // cell = (B >> 2, G >> 2, R >> 2), B slowest
    if (ci >= RC_COUNT) return;
    const int b0 = (ci >> (2 * 6)) << RC_SHIFT, g0 = ((ci >> 6) & (RC_N - 1)) << RC_SHIFT, r0 = (ci & (RC_N - 1)) << RC_SHIFT;
    int lo[3] = {255, 255, 255}, hi[3] = {0, 0, 0};
    for (int db = 0; db < (1 << RC_SHIFT); db++)
        for (int dg = 0; dg < (1 << RC_SHIFT); dg++)
            for (int dr = 0; dr < (1 << RC_SHIFT); dr++) {
                int v[3];
                lab_noclamp(f_lab_tab, f_lab_tab + 256, b0 + db, g0 + dg, r0 + dr, v[0], v[1], v[2]);
#pragma unroll
                for (int d = 0; d < 3; d++) { lo[d] = min(lo[d], v[d]); hi[d] = max(hi[d], v[d]); }
            }
#pragma unroll
    for (int d = 0; d < 3; d++) { boxes[6 * ci + d] = (u8)lo[d]; boxes[6 * ci + 3 + d] = (u8)hi[d]; }
}

// one thread = 8 cells consecutive in R: one u32 of label nibbles + one byte of "several candidates" flags
__global__ void __launch_bounds__(256) fk_build_rgbcells(const __grid_constant__ AssignParams P, const u8 *__restrict__ boxes,
                                                         u32 *__restrict__ nib, u8 *__restrict__ mb)
{
    const int gi = blockIdx.x * blockDim.x + threadIdx.x;               // cell index / 8
    if (gi >= RC_COUNT / 8) return;
    const int K = P.K;
    u32 nibbles = 0u, multi = 0u;
    for (int q = 0; q < 8; q++) {
        const int ci = gi * 8 + q;
        float lo[3], hi[3];
#pragma unroll
        for (int d = 0; d < 3; d++) { lo[d] = (float)boxes[6 * ci + d]; hi[d] = (float)boxes[6 * ci + 3 + d]; }
        float U = 3.0e38f;
        bool sane = true;
        for (int k = 0; k < K; k++) {
            float dmax = 0.f;
#pragma unroll
            for (int d = 0; d < 3; d++) {
                float c = P.c[3 * k + d];
                sane = sane && (fabsf(c) < 1.0e4f);                 // also false for NaN
                float m = fmaxf(fabsf(lo[d] - c), fabsf(hi[d] - c));
                dmax += m * m;
            }
            U = fminf(U, dmax);
        }
        u32 mask = 0u;
        for (int k = 0; k < K; k++) {
            float dmin = 0.f;
#pragma unroll
            for (int d = 0; d < 3; d++) {
                float c = P.c[3 * k + d];
                float n = fminf(fmaxf(c, lo[d]), hi[d]);
                dmin += (n - c) * (n - c);
            }
            if (dmin <= U + 2.0f) mask |= 1u << k;                  // slack: see fk_build_cells
        }
        const bool single = sane && mask != 0u && (mask & (mask - 1u)) == 0u;
        if (single) nibbles |= (u32)(P.lut[__ffs(mask) - 1] & 15u) << (4 * q);
        else {
            multi |= 1u << q;
            if (K < 16) nibbles |= 15u << (4 * q);               // K <= 15: the label table itself says "several candidates"
        }
    }
    nib[gi] = nibbles;
    mb[gi] = (u8)multi;
}

template <bool SEP_MULTI>                  // K == 16: the "several candidates" flag needs its own bit table; K <= 15: nibble 15
__global__ void __launch_bounds__(RA_THREADS, 1) fk_assign_rgbcell(const u8 *__restrict__ px, int h, int w, size_t pitch,
                                                                   const __grid_constant__ AssignParams P, const uint4 *__restrict__ rtab,
                                                                   const u32 *__restrict__ cells,
                                                                   u8 *__restrict__ labels, size_t lpitch,
                                                                   u32 *__restrict__ bits, int ws, size_t plane,
                                                                   int nf, size_t frame_stride /* a batch: nf frames of h rows; frame f
                                                                   writes the K planes starting at plane f * K (labels: rows f * h ..) */,
                                                                   const __grid_constant__ ZeroJob Z)
{
    extern __shared__ __align__(16) u8 smem[];
    const u32 *s_nib = reinterpret_cast<const u32 *>(smem);
    const u32 *s_mb = reinterpret_cast<const u32 *>(smem + RA_OFF_MB);
    u16 *s_cbrt = reinterpret_cast<u16 *>(smem + RA_OFF_CBRT);
    u16 *s_gam = reinterpret_cast<u16 *>(smem + RA_OFF_GAM);
    float4 *s_ctr = reinterpret_cast<float4 *>(smem + RA_OFF_CTR);
    u8 *s_lut = smem + RA_OFF_LUT;
    for (int i = threadIdx.x; i < (RC_NIB_BYTES + (SEP_MULTI ? RC_MB_BYTES : 0)) / 16; i += RA_THREADS)
        reinterpret_cast<uint4 *>(smem)[i] = __ldg(rtab + i);
    for (int i = threadIdx.x; i < 2048; i += RA_THREADS) {
        s_cbrt[i] = f_lab_tab[256 + i];
        if (i < 256) s_gam[i] = f_lab_tab[i];
    }
    if (threadIdx.x < OMNI_MAX_K) {
        s_lut[threadIdx.x] = P.lut[threadIdx.x];
        s_ctr[threadIdx.x] = make_float4(P.c[3 * threadIdx.x], P.c[3 * threadIdx.x + 1], P.c[3 * threadIdx.x + 2], 0.f);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int chunks = (w + 255) >> 8, K = P.K;
    const int total = nf * h * chunks, stride = gridDim.x * RA_WARPS;     // nf * h * chunks < 2^30 (checked by the host)
    const bool vec_ok = (((uintptr_t)px | pitch | frame_stride) & 15) == 0;
    u8 *spx = smem + RA_OFF_WARP + warp * RA_WARP_BYTES;              // per warp: the 256 pixels of the current chunk
    u8 *sq = spx + 768, *slab = sq + 256;                             //           queued pixel indices, their labels
    const u32 lt = (1u << lane) - 1u;
    uint4 pf0 = make_uint4(0, 0, 0, 0), pf1 = pf0;
    // chunk u = (row yy of the batch, chunk c of the row); the pair is advanced without divisions
    const int dyy = stride / chunks, dc = stride - dyy * chunks;
    auto prefetch = [&](int u, int yy, int c) {
        if (u < total) {
            const int f = nf > 1 ? yy / h : 0, y = yy - f * h;     // one frame: no division
            if (vec_ok && c * 256 + 256 <= w) {
                const uint4 *src = reinterpret_cast<const uint4 *>(px + (size_t)f * frame_stride + (size_t)y * pitch + (size_t)c * 768);
                pf0 = __ldg(src + lane);
                if (lane < 16) pf1 = __ldg(src + 32 + lane);
            }
        }
    };
    int u = blockIdx.x * RA_WARPS + warp;
    int yy_n = u / chunks, c_n = u - yy_n * chunks;                // the chunk the prefetch registers hold
    prefetch(u, yy_n, c_n);
    for (; u < total; u += stride) {
        const int yy = yy_n, c = c_n;
        yy_n += dyy; c_n += dc;
        if (c_n >= chunks) { c_n -= chunks; yy_n++; }
        const int f = nf > 1 ? yy / h : 0, y = yy - f * h;     // one frame: no division
        const int x0 = c * 256 + lane;
        const bool full = vec_ok && c * 256 + 256 <= w;
        __syncwarp();                                          // the previous chunk has been consumed
        if (full) {
            reinterpret_cast<uint4 *>(spx)[lane] = pf0;
            if (lane < 16) reinterpret_cast<uint4 *>(spx)[32 + lane] = pf1;
        } else {
            const u8 *row = px + (size_t)f * frame_stride + (size_t)y * pitch + (size_t)c * 768;
            const int nb = 3 * min(256, w - c * 256);
            for (int i = lane; i < nb; i += 32) spx[i] = row[i];
        }
        prefetch(u + stride, yy_n, c_n);
#pragma unroll
        for (int z = 0; z < 2; z++) {                          // this chunk's slice of the zero-fill regions (per: multiple of 32)
            if (Z.n16[z]) {
                unsigned long long idx = (unsigned long long)Z.per[z] * (unsigned)u + lane;
                uint4 *q = Z.p[z] + idx;
                for (unsigned it = Z.per[z] >> 5; it > 0; it--, idx += 32, q += 32)
                    if (idx < Z.n16[z]) *q = make_uint4(0u, 0u, 0u, 0u);
            }
        }
        __syncwarp();
        // ---- phase 1: table lookup in shared memory; pixels of cells with several candidates are queued ----
        int lab[8];
        int nq = 0;
        u32 und = 0u;
#pragma unroll
        for (int g = 0; g < 8; g++) {
            const int x = x0 + 32 * g;
            lab[g] = 255;
            bool multi = false;
            if (x < w) {
                const u8 *p = spx + 3 * lane + 96 * g;
                const u32 v0 = p[0], v1 = p[1], v2 = p[2];
                const u32 ci = ((v0 >> RC_SHIFT) << 12) | ((v1 >> RC_SHIFT) << 6) | (v2 >> RC_SHIFT);
                lab[g] = (s_nib[ci >> 3] >> ((ci & 7u) * 4u)) & 15u;
                multi = SEP_MULTI ? ((s_mb[ci >> 5] >> (ci & 31u)) & 1u) != 0u : lab[g] == 15;
            }
            const u32 bal = __ballot_sync(0xffffffffu, multi);
            if (multi) {
                sq[nq + __popc(bal & lt)] = (u8)(32 * g + lane);
                und |= 1u << g;
            }
            nq += __popc(bal);
        }
        __syncwarp();
        // ---- phase 2: Lab conversion + the reference's float32 argmin over the Lab cell's candidates, one queued pixel
        //      per lane and round ----
        for (int i = lane; i < nq; i += 32) {
            const int pi = sq[i];
            const u8 *p = spx + 3 * pi;
            int L, a, b, best = 0;
            lab_noclamp(s_gam, s_cbrt, p[0], p[1], p[2], L, a, b);
            u32 mk = __ldg(cells + (((L >> CELL_SHIFT) * CELL_N + (a >> CELL_SHIFT)) * CELL_N + (b >> CELL_SHIFT)));
            const float f0 = (float)L, f1 = (float)a, f2 = (float)b;
            float bd = 3.0e38f;
            do {
                const int k = __ffs(mk) - 1;
                mk &= mk - 1u;
                const float4 ck = s_ctr[k];
                float d0 = __fsub_rn(f0, ck.x), d1 = __fsub_rn(f1, ck.y), d2 = __fsub_rn(f2, ck.z);
                float d = __fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2, d2));
                if (d < bd) { bd = d; best = k; }
            } while (mk);
            slab[pi] = s_lut[best];
        }
        __syncwarp();
#pragma unroll
        for (int g = 0; g < 8; g++)
            if ((und >> g) & 1u) lab[g] = slab[32 * g + lane];
        // ---- phase 3: outputs ----
        if (labels) {
            u8 *lrow = labels + (size_t)yy * lpitch;
#pragma unroll
            for (int g = 0; g < 8; g++)
                if (x0 + 32 * g < w) lrow[x0 + 32 * g] = (u8)lab[g];
        }
        if (bits) {
            // 32-bit word offsets (the host checks nf * K * plane < 2^31).  A valid pixel (label < K) implies its word exists.
            u32 *brow = bits + ((u32)(f * K) * (u32)plane + (u32)y * (u32)ws + (u32)c * 8u);
            const u32 plane_bytes = (u32)plane * 4u;               // one multiply-add (32 x 32 + 64) gives the plane's row
#pragma unroll
            for (int g = 0; g < 8; g++) {
                const u32 same = __match_any_sync(0xffffffffu, lab[g]);
                if (lab[g] < K && (same & lt) == 0u)                  // the lowest lane of each label stores its word
                    reinterpret_cast<u32 *>(reinterpret_cast<char *>(brow) + (unsigned long long)(u32)lab[g] * plane_bytes)[g] = same;
            }
        }
    }
}

template <int MODE_LAB>
__global__ void __launch_bounds__(256) fk_assign_bits(const u8 *__restrict__ px, int h, int w, size_t pitch,
                                                      const __grid_constant__ AssignParams P, const u32 *__restrict__ cells,
                                                      u8 *__restrict__ labels, size_t lpitch,
                                                      u32 *__restrict__ bits, int ws, size_t plane)
{
    __shared__ u16 s_gam[256];
    __shared__ u16 s_cbrt[2048];
    __shared__ float4 s_ctr[OMNI_MAX_K];
    __shared__ u8 s_lut[OMNI_MAX_K];
    __shared__ __align__(16) u8 s_px[8][768];                 // per warp: the 256 pixels of the current chunk
    if (MODE_LAB) {
        for (int i = threadIdx.x; i < 2048; i += 256) {
            s_cbrt[i] = f_lab_tab[256 + i];
            if (i < 256) s_gam[i] = f_lab_tab[i];
        }
    }
    if (threadIdx.x < OMNI_MAX_K) {
        s_lut[threadIdx.x] = P.lut[threadIdx.x];
        s_ctr[threadIdx.x] = make_float4(P.c[3 * threadIdx.x], P.c[3 * threadIdx.x + 1], P.c[3 * threadIdx.x + 2], 0.f);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int chunks = (w + 255) >> 8, K = P.K;
    const long long total = (long long)h * chunks, stride = (long long)gridDim.x * 8;
    // rows can be moved with 16-byte loads when the image base and pitch allow it
    const bool vec_ok = (((uintptr_t)px | pitch) & 15) == 0;
    u8 *spx = s_px[warp];
    uint4 pf0 = make_uint4(0, 0, 0, 0), pf1 = pf0;
    auto chunk_full = [&](long long u) { int c = (int)(u % chunks); return vec_ok && c * 256 + 256 <= w; };
    auto prefetch = [&](long long u) {
        if (u < total && chunk_full(u)) {
            const int y = (int)(u / chunks), c = (int)(u - (long long)y * chunks);
            const uint4 *src = reinterpret_cast<const uint4 *>(px + (size_t)y * pitch + (size_t)c * 768);
            pf0 = __ldg(src + lane);
            if (lane < 16) pf1 = __ldg(src + 32 + lane);
        }
    };
    long long u = (long long)blockIdx.x * 8 + warp;
    prefetch(u);
    for (; u < total; u += stride) {
        const int y = (int)(u / chunks), c = (int)(u - (long long)y * chunks);
        const int x0 = c * 256 + lane;
        const bool full = chunk_full(u);
        __syncwarp();                                          // the previous chunk has been consumed
        if (full) {
            reinterpret_cast<uint4 *>(spx)[lane] = pf0;
            if (lane < 16) reinterpret_cast<uint4 *>(spx)[32 + lane] = pf1;
        } else {
            const u8 *row = px + (size_t)y * pitch + (size_t)c * 768;
            const int nb = 3 * min(256, w - c * 256);
            for (int i = lane; i < nb; i += 32) spx[i] = row[i];
        }
        prefetch(u + stride);
        __syncwarp();
        int lab[8];
#pragma unroll
        for (int g = 0; g < 8; g++) {
            const int x = x0 + 32 * g;
            lab[g] = 255;
            if (x < w) {
                const u8 *p = spx + 3 * lane + 96 * g;
                int v0 = p[0], v1 = p[1], v2 = p[2], best = 0;
                if (MODE_LAB) {
                    int L, a, b;
                    lab_noclamp(s_gam, s_cbrt, v0, v1, v2, L, a, b);
                    u32 mk = __ldg(cells + (((L >> CELL_SHIFT) * CELL_N + (a >> CELL_SHIFT)) * CELL_N + (b >> CELL_SHIFT)));
                    float f0 = (float)L, f1 = (float)a, f2 = (float)b, bd = 3.0e38f;
                    do {
                        const int k = __ffs(mk) - 1;
                        mk &= mk - 1u;
                        const float4 ck = s_ctr[k];
                        float d0 = __fsub_rn(f0, ck.x), d1 = __fsub_rn(f1, ck.y), d2 = __fsub_rn(f2, ck.z);
                        float d = __fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2, d2));
                        if (d < bd) { bd = d; best = k; }
                    } while (mk);
                } else {
                    int bd = 0;
                    for (int k = 0; k < K; k++) {
                        int d0 = v0 - P.pal[3 * k], d1 = v1 - P.pal[3 * k + 1], d2 = v2 - P.pal[3 * k + 2];
                        int d = (int)(short)(d0 * d0) + (int)(short)(d1 * d1) + (int)(short)(d2 * d2);
                        if (k == 0 || d < bd) { bd = d; best = k; }
                    }
                }
                lab[g] = s_lut[best];
            }
        }
        if (labels) {
            u8 *lrow = labels + (size_t)y * lpitch;
#pragma unroll
            for (int g = 0; g < 8; g++)
                if (x0 + 32 * g < w) lrow[x0 + 32 * g] = (u8)lab[g];
        }
        if (bits) {
            u32 *brow = bits + (size_t)y * ws + c * 8;
#pragma unroll
            for (int g = 0; g < 8; g++) {
                const u32 same = __match_any_sync(0xffffffffu, lab[g]);
                if (lab[g] < K && lane == __ffs(same) - 1 && c * 8 + g < ws) brow[(size_t)lab[g] * plane + g] = same;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// process_colors.assign_labels (process_colors.py:69-77) for K <= 16: argmin_k of  sum_c (i16)((v_c - p_kc)^2)  -- the products wrap to
// int16, the sum is wide.  |d| <= 255, so the wrapped square is d^2 - 65536 [ |d| >= 182 ], and
//     dist_k = sum_c v_c^2  +  sum_c p_kc^2  -  2 sum_c v_c p_kc  -  65536 n_k,      n_k = channels of centre k with |v_c - p_kc| >= 182.
// The first term is the same for every k; the dot product is one DP4A on the packed bytes; n_k comes from three table words per pixel
// (2-bit fields per k, one table per channel in shared memory: the fields add without carries, n_k <= 3).  key_k = 16 dist_k + k keeps
// np.argmin's first minimum under a plain integer min.  A lane takes 4 adjacent pixels (three 4-byte loads, one 4-byte label store).
// ------------------------------------------------------------------------------------------------
template <int KMAX>                                         // palette colours rounded up to 4, 8 or 16
__global__ void __launch_bounds__(256) fk_assign_i16wrap(const u8 *__restrict__ px, int h, int w, size_t pitch, const __grid_constant__ AssignParams P,
                                                         u8 *__restrict__ labels, size_t lpitch)
{
    __shared__ u32 s_wrap[3][256];
    __shared__ u8 s_lut[16];
    const int K = P.K;
    for (int i = threadIdx.x; i < 768; i += 256) {
        const int c = i >> 8, v = i & 255;
        u32 word = 0u;
        for (int k = 0; k < K; k++) {
            const int d = v - (int)P.pal[3 * k + c];
            word |= (u32)(d >= 182 || d <= -182) << (2 * k);
        }
        s_wrap[c][v] = word;
    }
    if (threadIdx.x < 16) s_lut[threadIdx.x] = P.lut[threadIdx.x];
    u32 pk[KMAX];
    int ck[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; k++) {
        const int p0 = P.pal[3 * k], p1 = P.pal[3 * k + 1], p2 = P.pal[3 * k + 2];
        pk[k] = k < K ? ((u32)p0 | ((u32)p1 << 8) | ((u32)p2 << 16)) : 0u;
        ck[k] = k < K ? 16 * (p0 * p0 + p1 * p1 + p2 * p2) + k : 0x7ffffff0;          // k >= K never wins
    }
    __syncthreads();
    auto label_of = [&](const u32 v) -> u32 {                // v = c0 | c1 << 8 | c2 << 16 (| anything << 24: pk has a zero there)
        const u32 cnt = s_wrap[0][v & 255u] + s_wrap[1][(v >> 8) & 255u] + s_wrap[2][(v >> 16) & 255u];
        int best = 0x7fffffff;
#pragma unroll
        for (int k = 0; k < KMAX; k++) {
            const int dot = (int)__dp4a(v, pk[k], 0u);
            const int n = (int)((cnt >> (2 * k)) & 3u);
            best = min(best, ck[k] - 32 * dot - (n << 20));
        }
        return (u32)s_lut[best & 15];
    };
    const int groups = (w + 3) >> 2;                          // 4 pixels per lane
    const bool fast_rows = (((uintptr_t)px | pitch) & 3) == 0;
    const bool fast_out = (((uintptr_t)labels | lpitch) & 3) == 0;
    const long long total = (long long)h * groups;
    for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < total; u += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(u / groups), g = (int)(u - (long long)y * groups);
        const u8 *row = px + (size_t)y * pitch + (size_t)g * 12;
        u8 *lrow = labels + (size_t)y * lpitch + (size_t)g * 4;
        if (fast_rows && g * 4 + 4 <= w) {
            const u32 a = __ldg(reinterpret_cast<const u32 *>(row)), b = __ldg(reinterpret_cast<const u32 *>(row) + 1),
                      c = __ldg(reinterpret_cast<const u32 *>(row) + 2);
            const u32 l0 = label_of(a), l1 = label_of(__byte_perm(a, b, 0x4543)), l2 = label_of(__byte_perm(b, c, 0x4432)),
                      l3 = label_of(c >> 8);
            if (fast_out) *reinterpret_cast<u32 *>(lrow) = l0 | (l1 << 8) | (l2 << 16) | (l3 << 24);
            else { lrow[0] = (u8)l0; lrow[1] = (u8)l1; lrow[2] = (u8)l2; lrow[3] = (u8)l3; }
        } else {
            for (int i = 0; i < 4 && g * 4 + i < w; i++)
                lrow[i] = (u8)label_of((u32)row[3 * i] | ((u32)row[3 * i + 1] << 8) | ((u32)row[3 * i + 2] << 16));
        }
    }
}

const u16 *fast_lab_table()
{
    void *p = nullptr;
    if (cudaGetSymbolAddress(&p, f_lab_tab) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return (const u16 *)p;
}

cudaError_t launch_build_cells(const AssignParams &P, u32 *cells, cudaStream_t st)
{
    fk_build_cells<<<CELL_COUNT / 256, 256, 0, st>>>(P, cells);
    return cudaGetLastError();
}

int fast_rgb_boxes(omni_ctx *ctx, cudaStream_t st)
{
    if (ctx->d_rgb_boxes) return OMNI_OK;              // centre-independent: once per context
    OMNI_CUDA(cudaMalloc(&ctx->d_rgb_boxes, (size_t)RC_COUNT * 6));
    KScope ks(ctx, "rgb_boxes", st);
    fk_rgb_boxes<<<RC_COUNT / 256, 256, 0, st>>>(ctx->d_rgb_boxes);
    OMNI_CUDA(cudaGetLastError());
    return OMNI_OK;
}

// labels u8 -> one-hot bit-planes (omni_layer_masks entry)
__global__ void __launch_bounds__(256) fk_labels_to_bits(const u8 *__restrict__ labels, int h, int w, size_t lpitch, int K,
                                                         u32 *__restrict__ bits, int ws, size_t plane)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int chunks = (w + 255) >> 8;
    const long long total = (long long)h * chunks;
    for (long long u = (long long)blockIdx.x * 8 + warp; u < total; u += (long long)gridDim.x * 8) {
        const int y = (int)(u / chunks), c = (int)(u - (long long)y * chunks);
        const int x0 = c * 256 + lane;
        const u8 *row = labels + (size_t)y * lpitch;
        int lab[8];
#pragma unroll
        for (int g = 0; g < 8; g++) lab[g] = (x0 + 32 * g < w) ? row[x0 + 32 * g] : 255;
        u32 mine = 0;
        for (int k = 0; k < K; k++) {
#pragma unroll
            for (int g = 0; g < 8; g++) {
                u32 b = __ballot_sync(0xffffffffu, lab[g] == k);
                if (lane == ((k & 3) * 8 + g)) mine = b;
            }
            if ((k & 3) == 3 || k == K - 1) {
                int kk = (k & ~3) + (lane >> 3), wx = c * 8 + (lane & 7);
                if (kk <= k && wx < ws) bits[(size_t)kk * plane + (size_t)y * ws + wx] = mine;
                mine = 0;
            }
        }
    }
}

// mask bytes -> bit-planes; *d_bad set when a byte is neither 0 nor 255 (caller falls back to generic).
// A warp packs 512 pixels per step: every lane reads 16 bytes with one load, turns them into 16 bits (high bit of
// "byte != 0" per byte, gathered with shifts), lane pairs are joined into words by a shuffle.  All ws words of a row
// are written (the padding words as zeros).
// CHECK = true (stage 03: masks must be {0,255}, anything else raises `bad` and the caller takes the generic kernels, so the bits only
// matter for clean masks): bit = low bit of the byte.  CHECK = false (thinning: foreground = byte > 0): bit = "byte != 0".
template <bool CHECK>
__device__ __forceinline__ u32 nz4(u32 v, u32 &bad)            // 4 bytes -> 4 bits; the partial products of the gather land on distinct bits
{
    if (CHECK) {
        const u32 t = v & 0x01010101u;
        bad |= v ^ (t * 255u);
        return (t * 0x01020408u) >> 24;
    }
    const u32 t7 = (((v & 0x7f7f7f7fu) + 0x7f7f7f7fu) | v) & 0x80808080u;      // 0x80 per non-zero byte
    return (t7 * 0x00204081u) >> 28;
}

template <bool CHECK>
__global__ void __launch_bounds__(256) fk_bytes_to_bits(const u8 *__restrict__ planes, size_t pstride, size_t pitch, int h, int w,
                                                        u32 *__restrict__ bits, int ws, size_t plane, int *d_bad)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int k = blockIdx.y;
    const int chunks = (ws + 15) >> 4;                         // 16 words = 512 pixels per warp step
    const bool vec_ok = (((uintptr_t)(planes + (size_t)k * pstride) | pitch) & 15) == 0;
    u32 bad = 0u;
    // (row, chunk) of this warp's step and the constant stride between its steps: no division inside the loop
    const int stride = (int)gridDim.x * 8, dy = stride / chunks, dch = stride - dy * chunks;
    const int u0 = (int)blockIdx.x * 8 + warp;
    int y = u0 / chunks, ch = u0 - y * chunks;
    for (; y < h; y += dy, ch += dch) {
        if (ch >= chunks) { ch -= chunks; if (++y >= h) break; }
        const int x = ch * 512 + 16 * lane;
        const u8 *row = planes + (size_t)k * pstride + (size_t)y * pitch;
        u32 m16 = 0u;
        if (vec_ok && x + 16 <= w) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(row + x));
            m16 = nz4<CHECK>(v.x, bad) | (nz4<CHECK>(v.y, bad) << 4) | (nz4<CHECK>(v.z, bad) << 8) | (nz4<CHECK>(v.w, bad) << 12);
        } else {
            for (int i = 0; i < 16 && x + i < w; i++) {
                const u32 v = row[x + i];
                bad |= (v != 0u && v != 255u);
                m16 |= (u32)(v != 0u) << i;
            }
        }
        const u32 other = __shfl_xor_sync(0xffffffffu, m16, 1);
        const int c = ch * 16 + (lane >> 1);
        if (!(lane & 1) && c < ws) bits[(size_t)k * plane + (size_t)y * ws + c] = m16 | (other << 16);
    }
    if (CHECK && __any_sync(0xffffffffu, bad != 0u) && lane == 0) atomicOr(d_bad, 1);
}

// bit-planes -> 0/255 byte planes
__global__ void __launch_bounds__(256) fk_expand_bits(const u32 *__restrict__ bits, int ws, size_t plane, int h, int w,
                                                      u8 *__restrict__ out, size_t ostride, size_t opitch, int aligned16)
{
    const int k = blockIdx.y, ww = (w + 31) >> 5;
    const long long total = (long long)h * ww;
    for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < total; u += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(u / ww), c = (int)(u - (long long)y * ww);
        u32 word = bits[(size_t)k * plane + (size_t)y * ws + c];
        store_word_bytes(out + (size_t)k * ostride + (size_t)y * opitch, c * 32, w, word, aligned16);
    }
}

// ------------------------------------------------------------------------------------------------
// binary morphology on bit-planes (02:151-154 RECT-3, 03:23-30 ELLIPSE-3 = cross); SURVEY A.0
//
// One thread owns one word column and streams down a strip of rows.  It works on a 64-bit WINDOW = its
// 32 pixels + 16 halo pixels on each side (built from the neighbouring words), so every erode/dilate step
// of the chain needs no communication: a step only invalidates one more halo bit per side.  All steps of
// the chain are software-pipelined down the rows (step s lags the input by s rows), state in registers.
// Pixels outside the image are "ignored" by OpenCV: erode sees 1s, dilate sees 0s -- applied per step.
// ------------------------------------------------------------------------------------------------
// Run lists of the sparse edge kernel, produced by the morphology kernel itself (RUNS = true): the final image rows
// pass through this lane's registers with 8 valid halo pixels per side, which is all fk_edge_runs (edges3.cu) needs
// to classify the lane's MORPH_TR / ET_R tiles -- see the comment there for the rule and the list layout.  The strip is
// extended by 2 final rows at each end for the tiles' 2-row halo.
// CODE: up to 8 steps, 4 bits each.  TAP: after this many steps the image is the stage-02 mask; it is
// written as BYTES to `masks` (TAP = -1: nothing).  The final image is written as bits to `out_bits`
// (may be NULL).
#ifndef MORPH_MINB
#define MORPH_MINB 1
#endif
template <u32 CODE, int TAP, bool RUNS, int TR>
__global__ void __launch_bounds__(128, MORPH_MINB) fk_morph(const u32 *__restrict__ in_bits, u32 *__restrict__ out_bits, int ws, size_t plane, int h,
                                                int w, u8 *__restrict__ masks, size_t mstride, size_t mpitch, int aligned16,
                                                int y_lo, int y_hi /* rows [y_lo, y_hi) are produced; input rows around them must exist */,
                                                const __grid_constant__ MorphRuns R)
{
    constexpr int N = code_len(CODE);
    const int GROW = RUNS ? (R.grow ? R.grow : 2) : 0;   // 2..4, see MorphRuns
    const int EXT = GROW;
    constexpr int TILES = TR / ET_R;
    __shared__ uint2 s_lut8[256];
    __shared__ u32 s_item[RUNS ? 4 : 1][RUNS ? TILES : 1][32];
    if (TAP >= 0) {
        expand_lut_init(s_lut8, threadIdx.x, blockDim.x);
        __syncthreads();
    }
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int ww = (w + 31) >> 5;
    const bool active = c < ww;
    if (!RUNS && !active) return;                          // with RUNS every lane stays for the warp-wide list flush
    const int k = blockIdx.z;
    const int y0 = y_lo + blockIdx.y * TR, y1 = min(y_hi, y0 + TR);
    const u32 *src = in_bits + (size_t)k * plane;
    W64 colvalid;
    colvalid.lo = range_mask(32 * c - 16, w);
    colvalid.hi = range_mask(32 * c + 16, w);
    constexpr int OP0 = N > 0 ? code_op(CODE, 0) : ST_NONE;
    W64 p1[8], p2[8];
#pragma unroll
    for (int s = 0; s < 8; s++) { p1[s].lo = p1[s].hi = p2[s].lo = p2[s].hi = 0u; }
    // the three words of the next input row are loaded one iteration ahead (the row is consumed ~250 instructions later)
    u32 nl = 0u, no = 0u, nr = 0u;
    auto fetch = [&](int t) {
        nl = no = nr = 0u;
        if (t >= 0 && t < h && active) {
            const u32 *row = src + (size_t)t * ws;
            if (c > 0) nl = __ldg(row + c - 1);
            no = __ldg(row + c);
            if (c + 1 < ww) nr = __ldg(row + c + 1);
        }
    };
    u32 live1 = 0u, live0 = 0u;                            // per tile of the strip: "has a 1" / "has a 0" in the grown tile
    auto rows = [&](auto rowfix_tag, auto colfix_tag) {
    constexpr bool ROWFIX = decltype(rowfix_tag)::value, COLFIX = decltype(colfix_tag)::value;
    fetch(y0 - N - EXT);
    for (int t = y0 - N - EXT; t < y1 + N + EXT; t++) {
        W64 cur;
        const bool inside = t >= 0 && t < h;
        cur.lo = (nl >> 16) | (no << 16);
        cur.hi = (no >> 16) | (nr << 16);
        fetch(t + 1);
        cur = oob_fix<OP0, ROWFIX, COLFIX>(cur, colvalid, !ROWFIX || inside);
        W64 tap, fin;
        tap.lo = tap.hi = fin.lo = fin.hi = 0u;
        MorphChain<CODE, 0>::template run<TAP, ROWFIX, COLFIX>(cur, p1, p2, t, h, colvalid, tap, fin);
        if (TAP >= 0) {
            const int r = t - TAP;
            if (r >= y0 && r < y1 && active) {
                u32 word = (tap.lo >> 16) | (tap.hi << 16);
                store_word_bytes_lut(masks + (size_t)k * mstride + (size_t)r * mpitch, 32 * c, w, word, aligned16, s_lut8);
            }
        }
        const int r = t - N;
        if (out_bits) {
            if (r >= y0 && r < y1 && active) {
                u32 word = ((fin.lo >> 16) | (fin.hi << 16)) & range_mask(32 * c, w);
                out_bits[(size_t)k * plane + (size_t)r * ws + c] = word;
            }
        }
        if (RUNS) {
            if (r >= y0 - GROW && r < y1 + GROW && (!ROWFIX || (r >= 0 && r < h))) {
                // window bits 16-GROW .. 47+GROW = pixels 32c-GROW .. 32c+31+GROW; fin is already 0 outside the image
                const u32 m_lo = (0xFFFFFFFFu << (16 - GROW)) & colvalid.lo, m_hi = (0xFFFFFFFFu >> (16 - GROW)) & colvalid.hi;
                const bool h1 = ((fin.lo & m_lo) | (fin.hi & m_hi)) != 0u, h0 = ((~fin.lo & m_lo) | (~fin.hi & m_hi)) != 0u;
                const int rr = r - y0, sub = rr & 7;
                u32 m = 1u << ((rr >> 3) + 1);                          // tile rr / 8 (floor), biased by one
                if (sub < GROW) m |= m >> 1;                             // also the halo rows of the tile above
                if (sub >= 8 - GROW) m |= m << 1;                        // ... of the tile below
                m = (m >> 1) & ((1u << TILES) - 1u);
                if (h1) live1 |= m;
                if (h0) live0 |= m;
            }
        }
    }
    };
    // every row of every image in the chain that this strip touches: [y0 - 2N - EXT, y1 + N + EXT)
    const bool rowfix = !(y0 - 2 * N - EXT >= 0 && y1 + N + EXT <= h);                          // uniform per CTA
    // uniform per warp (lanes right of the image have left already when there is no list flush to attend)
    const bool colfix = __any_sync(__activemask(), (colvalid.lo & colvalid.hi) != 0xffffffffu);
    if (rowfix) { if (colfix) rows(std::true_type{}, std::true_type{}); else rows(std::true_type{}, std::false_type{}); }
    else { if (colfix) rows(std::false_type{}, std::true_type{}); else rows(std::false_type{}, std::false_type{}); }
    if (RUNS) {
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        const u32 live = active ? (live1 & live0) : 0u;
        int n_items = 0, run = 0, run_j0 = 0;
        u32 lens = 0u;                                                   // 3 bits per emitted item: its run length
        auto emit = [&]() {
            lens |= (u32)run << (3 * n_items);
            s_item[wid][n_items++][lane] = ((u32)k << 27) | ((u32)run_j0 << 13) | (u32)c;
            run = 0;
        };
#pragma unroll
        for (int tl = 0; tl < TILES; tl++) {
            const int ty0 = y0 + tl * ET_R;
            if (ty0 >= y1) break;
            if ((live >> tl) & 1u) {
                if (run == 0) run_j0 = ty0 / ET_R;
                if (++run == R.maxt) emit();
            } else {
                if (run) emit();
                if (active && R.zero_fill) {
                    const int ty1 = min(y1, ty0 + ET_R);
                    for (int y = ty0; y < ty1; y++) {
                        const size_t o = (size_t)k * plane + (size_t)y * ws + c;
                        R.cbits[o] = 0u; R.sbits[o] = 0u;
                        if (R.edges) store_word_bytes(R.edges + (size_t)k * R.estride + (size_t)y * R.epitch, 32 * c, w, 0u, R.aligned16);
                    }
                }
            }
        }
        if (run) emit();
#pragma unroll
        for (int nt = 1; nt <= ET_MAXT; nt++) {
            int mine = 0;
            for (int i = 0; i < n_items; i++) mine += ((lens >> (3 * i)) & 7u) == (u32)nt;
            int x = mine;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                int y = __shfl_up_sync(0xffffffffu, x, d);
                if (lane >= d) x += y;
            }
            const int total = __shfl_sync(0xffffffffu, x, 31);
            if (total == 0) continue;
            int base = 0;
            if (lane == 31) base = atomicAdd(R.run_counts + nt - 1, total);
            base = __shfl_sync(0xffffffffu, base, 31);
            int pos = base + x - mine;
            for (int i = 0; i < n_items; i++)
                if (((lens >> (3 * i)) & 7u) == (u32)nt) R.run_items[R.off.v[nt - 1] + pos++] = s_item[wid][i][lane];
        }
    }
}

// morph03: 0 none, 1 open, 2 close, 3 open+close.  with02: prepend the RECT open/close and emit mask bytes.
// runs != NULL: also classify the tiles of the final image for the sparse edge kernel (MorphRuns).
static cudaError_t launch_morph(bool with02, int morph03, const u32 *in_bits, u32 *out_bits, const BitGeom &g, int K, u8 *masks,
                                size_t mstride, size_t mpitch, cudaStream_t st, int y_lo = 0, int y_hi = -1, const MorphRuns *runs = nullptr)
{
    if (y_hi < 0) y_hi = g.h;
    if (y_hi <= y_lo) return cudaSuccess;
    // taller strips (less halo work) once there are plenty of warps: 128-thread CTAs, 4 warps each
    auto warps_at = [&](int tr) { return (long long)((g.ww + 127) / 128) * 4 * ((y_hi - y_lo + tr - 1) / tr) * K; };
    int tr = MORPH_TR;
    if (warps_at(MORPH_TR_BIG) >= MORPH_BIG_MIN_WARPS && (y_lo % MORPH_TR_BIG) == 0) tr = MORPH_TR_BIG;
    else if (warps_at(MORPH_TR_MID) >= MORPH_MID_MIN_WARPS && (y_lo % MORPH_TR_MID) == 0) tr = MORPH_TR_MID;
    dim3 b(128), grid((g.ww + 127) / 128, (y_hi - y_lo + tr - 1) / tr, K);
    int al = plane_align(masks, mstride, mpitch);
    MorphRuns R{};
    if (runs) R = *runs;
#define LM2(CODE, TAP, RUNS, TR) fk_morph<CODE, TAP, RUNS, TR><<<grid, b, 0, st>>>(in_bits, out_bits, g.ws, g.plane, g.h, g.w, masks, mstride, mpitch, al, y_lo, y_hi, R)
#define LM3(CODE, TAP, RUNS)                                                          \
    do {                                                                               \
        if (tr == MORPH_TR_BIG) LM2(CODE, TAP, RUNS, MORPH_TR_BIG);                    \
        else if (tr == MORPH_TR_MID) LM2(CODE, TAP, RUNS, MORPH_TR_MID);               \
        else LM2(CODE, TAP, RUNS, MORPH_TR);                                           \
    } while (0)
#define LM(CODE, TAP)                                                                  \
    do {                                                                               \
        if (runs) LM3(CODE, TAP, true); else LM3(CODE, TAP, false);                    \
    } while (0)
    if (with02) {
        switch (morph03) {
        case 0: LM(CODE_R_OC, 4); break;
        case 1: LM(CODE_F_O, 4); break;
        case 2: LM(CODE_F_C, 4); break;
        default: LM(CODE_F_OC, 4); break;
        }
    } else {
        switch (morph03) {
        case 1: LM(CODE_C_O, -1); break;
        case 2: LM(CODE_C_C, -1); break;
        case 3: LM(CODE_C_OC, -1); break;
        default: return cudaErrorInvalidValue;
        }
    }
#undef LM
#undef LM3
#undef LM2
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// hysteresis on bit-planes (cv2.Canny's final stage; SURVEY A.5): E = S, then E |= C & dilate8(E) until
// nothing changes anywhere.  The edge kernel has already written the byte planes for E = S (on pipeline data
// nearly every candidate is strong), so a promoted pixel is patched to 255 the moment it is promoted.
//
// Cooperative persistent kernel; grid.sync() separates global rounds; three rotating "changed" flags let one
// barrier per round suffice.  Rounds 0..HY_WORD_ROUNDS-1 are WORD rounds: one thread per word, a word with
// promotable bits looks at its 8 neighbour words and closes the chain inside the word (pipeline data: done
// after 1-2 such rounds, each a single pass over the L2-resident bit-planes).  Longer chains escalate to TILE
// rounds: a CTA iterates a 32-row x 1024-pixel tile to its local fixed point in shared memory, so a chain
// advances by a tile, not a pixel, per round.  The result set does not depend on the propagation order.
// ------------------------------------------------------------------------------------------------
#define HB_TR 32                      // tile rows
#define HB_TW 32                      // tile words (1024 pixels)
#define HY_WORD_ROUNDS 4
#define HY_THREADS 1024                // one CTA resolves the whole worklist in the common case: make it a big one

__device__ __forceinline__ void hy_patch_bytes(u8 *row, u32 promoted)
{
    if (row == nullptr) return;                       // packed outputs: the bit-planes are the result
    while (promoted) {
        int e = __ffs(promoted) - 1;
        promoted &= promoted - 1u;
        row[e] = 255;
    }
}

// worklist mode of the hysteresis: every word that holds a weak candidate (C & ~S) is listed; on pipeline data that is a few hundred
// words, so ONE CTA resolves them.  Returns the number of rounds.
__device__ __forceinline__ int hy_worklist(u32 *__restrict__ ebits, const u32 *__restrict__ cbits, int ws, size_t plane, int h, int w, int n_weak,
                                   const u32 *__restrict__ worklist, u8 *__restrict__ edges, size_t estride, size_t epitch)
{
    const int wwl = (w + 31) >> 5;
    int rounds = 0;
    for (;;) {
        int changed = 0;
        for (int i = threadIdx.x; i < n_weak; i += HY_THREADS) {
            const u32 o = worklist[i];
            const int k = (int)(o / plane), rem = (int)(o - (size_t)k * plane);
            const int y = rem / ws, c = rem - y * ws;
            u32 *E = ebits + (size_t)k * plane + (size_t)y * ws;
            // every load of the item is issued at once (one L2 round trip instead of three dependent ones)
            const u32 cv = __ldg(cbits + o);
            u32 m3[3], l3[3], r3[3];
#pragma unroll
            for (int dy = -1; dy <= 1; dy++) {
                const bool in = y + dy >= 0 && y + dy < h;
                const u32 *Er = E + (ptrdiff_t)dy * ws;
                m3[dy + 1] = in ? __ldcg(Er + c) : 0u;
                l3[dy + 1] = (in && c > 0) ? __ldcg(Er + c - 1) : 0u;
                r3[dy + 1] = (in && c + 1 < wwl) ? __ldcg(Er + c + 1) : 0u;
            }
            const u32 ev = m3[1];
            if ((cv & ~ev) == 0u) continue;
            u32 d = 0u;
#pragma unroll
            for (int q = 0; q < 3; q++) d |= m3[q] | (m3[q] << 1) | (m3[q] >> 1) | (l3[q] >> 31) | (r3[q] << 31);
            u32 nv = ev | (cv & d);
            for (;;) {
                u32 t = nv | (cv & ((nv << 1) | (nv >> 1)));
                if (t == nv) break;
                nv = t;
            }
            if (nv != ev) {
                E[c] = nv;
                changed = 1;
                hy_patch_bytes(edges ? edges + (size_t)k * estride + (size_t)y * epitch + 32 * c : nullptr, nv & ~ev);
            }
        }
        rounds++;
        __threadfence_block();
        if (!__syncthreads_or(changed)) break;
    }
    return rounds;
}

// The same as a plain (non-cooperative) one-CTA launch: the banded host call resolves the prefix image after every band with it.  A list
// that overflowed is left alone (any subset of the final result is good enough there; the last band runs fk_hysteresis).
__global__ void __launch_bounds__(HY_THREADS) fk_hysteresis_wl(u32 *__restrict__ ebits, const u32 *__restrict__ cbits, int ws, size_t plane, int h,
                                                               int w, const int *flags, const u32 *__restrict__ worklist)
{
    const int n_weak = flags[4];
    if (n_weak > HY_WL_CAP) return;
    hy_worklist(ebits, cbits, ws, plane, h, w, n_weak, worklist, nullptr, 0, 0);
}

__global__ void __launch_bounds__(HY_THREADS) fk_hysteresis(u32 *__restrict__ ebits, const u32 *__restrict__ cbits, int ws, size_t plane, int h,
                                                     int w, int K, int *flags /* [0]=rounds, [1..3]=rotating "changed" flags, [4]=worklist count */,
                                                     const u32 *__restrict__ worklist,
                                                     u8 *__restrict__ edges, size_t estride, size_t epitch)
{
    cg::grid_group grid = cg::this_grid();
    // ---- worklist mode: the edge kernel listed every word that holds a weak candidate (C & ~S); on pipeline data
    // that is a few hundred words, so ONE CTA resolves them and the rest of the grid leaves at once ----
    const int n_weak = flags[4];
    if (n_weak <= HY_WL_CAP) {
        if (blockIdx.x != 0) return;
        const int rounds = hy_worklist(ebits, cbits, ws, plane, h, w, n_weak, worklist, edges, estride, epitch);
        if (threadIdx.x == 0) flags[0] = rounds;
        return;
    }
    __shared__ u32 s_e[(HB_TR + 2) * (HB_TW + 2)];
    __shared__ u32 s_c[HB_TR * HB_TW];
    const int ww = (w + 31) >> 5;
    const int tid = threadIdx.x;
    constexpr int SW = HB_TW + 2;
    int round = 0;
    for (;;) {
        volatile int *chg = flags + 1 + (round % 3);
        if (round < HY_WORD_ROUNDS) {
            // ---- word round: rows are walked by warps (coalesced 128-byte row segments) ----
            const long long rows = (long long)K * h;
            const int lane = tid & 31;
            const long long warp0 = ((long long)blockIdx.x * blockDim.x + tid) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
            for (long long R = warp0; R < rows; R += nwarps) {
                const int k = (int)(R / h), y = (int)(R - (long long)k * h);
                u32 *E = ebits + (size_t)k * plane + (size_t)y * ws;
                const u32 *C = cbits + (size_t)k * plane + (size_t)y * ws;
                for (int c = lane; c < ww; c += 32) {
                    const u32 cv = __ldg(C + c), ev = __ldcg(E + c);
                    if ((cv & ~ev) == 0u) continue;
                    u32 d = 0u;
#pragma unroll
                    for (int dy = -1; dy <= 1; dy++) {
                        if (y + dy < 0 || y + dy >= h) continue;
                        const u32 *Er = E + (ptrdiff_t)dy * ws;
                        u32 m = __ldcg(Er + c), l = c > 0 ? __ldcg(Er + c - 1) : 0u, r = c + 1 < ww ? __ldcg(Er + c + 1) : 0u;
                        d |= m | (m << 1) | (m >> 1) | (l >> 31) | (r << 31);
                    }
                    u32 nv = ev | (cv & d);
                    for (;;) {                                   // close the chain inside the word
                        u32 t = nv | (cv & ((nv << 1) | (nv >> 1)));
                        if (t == nv) break;
                        nv = t;
                    }
                    if (nv != ev) {
                        E[c] = nv;
                        *chg = 1;
                        hy_patch_bytes(edges ? edges + (size_t)k * estride + (size_t)y * epitch + 32 * c : nullptr, nv & ~ev);
                    }
                }
            }
        } else {
            // ---- tile round ----
            const int tx_n = (ww + HB_TW - 1) / HB_TW, ty_n = (h + HB_TR - 1) / HB_TR;
            const int tiles = tx_n * ty_n * K;
            for (int t = blockIdx.x; t < tiles; t += gridDim.x) {
                const int k = t / (tx_n * ty_n), r = t - k * (tx_n * ty_n);
                const int ty = r / tx_n, tx = r - ty * tx_n;
                const int y0 = ty * HB_TR, c0 = tx * HB_TW;
                u32 *E = ebits + (size_t)k * plane;
                const u32 *C = cbits + (size_t)k * plane;
                int pending = 0;
                for (int i = tid; i < HB_TR * HB_TW; i += HY_THREADS) {
                    int ly = i / HB_TW, lc = i - ly * HB_TW;
                    int gy = y0 + ly, gc = c0 + lc;
                    u32 cv = 0, ev = 0;
                    if (gy < h && gc < ww) { cv = __ldg(C + (size_t)gy * ws + gc); ev = __ldcg(E + (size_t)gy * ws + gc); }
                    s_c[i] = cv;
                    s_e[(ly + 1) * SW + lc + 1] = ev;
                    pending |= (cv & ~ev) != 0;
                }
                if (!__syncthreads_or(pending)) continue;
                // halo ring of E (other CTAs may be raising bits there concurrently: any snapshot is valid, bits only rise)
                for (int i = tid; i < 2 * SW + 2 * HB_TR; i += HY_THREADS) {
                    int ly, lc;
                    if (i < SW) { ly = 0; lc = i; }
                    else if (i < 2 * SW) { ly = HB_TR + 1; lc = i - SW; }
                    else { int j = i - 2 * SW; ly = 1 + (j >> 1); lc = (j & 1) ? HB_TW + 1 : 0; }
                    int gy = y0 - 1 + ly, gc = c0 - 1 + lc;
                    s_e[ly * SW + lc] = (gy >= 0 && gy < h && gc >= 0 && gc < ww) ? __ldcg(E + (size_t)gy * ws + gc) : 0u;
                }
                __syncthreads();
                int any = 0;
                for (;;) {
                    int changed = 0;
                    for (int i = tid; i < HB_TR * HB_TW; i += HY_THREADS) {
                        int ly = i / HB_TW, lc = i - ly * HB_TW;
                        u32 cv = s_c[i];
                        int o = (ly + 1) * SW + lc + 1;
                        u32 ev = s_e[o];
                        if (cv & ~ev) {
                            u32 d = 0;
#pragma unroll
                            for (int dy = -1; dy <= 1; dy++) {
                                u32 l = s_e[o + dy * SW - 1], m = s_e[o + dy * SW], rr = s_e[o + dy * SW + 1];
                                d |= m | (m << 1) | (m >> 1) | (l >> 31) | (rr << 31);
                            }
                            u32 nv = ev | (cv & d);
                            if (nv != ev) { s_e[o] = nv; changed = 1; }
                        }
                    }
                    if (!__syncthreads_or(changed)) break;
                    any = 1;
                }
                if (any) {
                    for (int i = tid; i < HB_TR * HB_TW; i += HY_THREADS) {
                        int ly = i / HB_TW, lc = i - ly * HB_TW;
                        int gy = y0 + ly, gc = c0 + lc;
                        if (gy < h && gc < ww) {
                            u32 nv = s_e[(ly + 1) * SW + lc + 1], old = __ldcg(E + (size_t)gy * ws + gc);
                            if (nv & ~old) {
                                E[(size_t)gy * ws + gc] = nv | old;
                                hy_patch_bytes(edges ? edges + (size_t)k * estride + (size_t)gy * epitch + 32 * gc : nullptr, nv & ~old);
                            }
                        }
                    }
                    if (tid == 0) *chg = 1;
                }
                __syncthreads();
            }
        }
        __threadfence();
        grid.sync();
        const int c = *chg;
        if (blockIdx.x == 0 && tid == 0) { flags[0] = round + 1; flags[1 + ((round + 2) % 3)] = 0; }
        round++;
        if (!c) break;
    }
}

// ------------------------------------------------------------------------------------------------
// host-side drivers
// ------------------------------------------------------------------------------------------------
#define HP_MAX_BANDS 8
static int pipe_init(omni_ctx *ctx);
int persist_blocks(omni_ctx *ctx, int per_sm) { return (ctx->sm_count > 0 ? ctx->sm_count : 148) * per_sm; }

// persistent grid of a kernel = SM count x the number of its CTAs that are resident per SM (queried once)
template <typename Kern>
static int resident_grid(omni_ctx *ctx, Kern kern, int block, int *cache)
{
    if (*cache == 0) {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, block, 0) != cudaSuccess || per_sm < 1) {
            cudaGetLastError();
            per_sm = 1;
        }
        *cache = per_sm;
    }
    return persist_blocks(ctx, *cache);
}

static int bit_planes(omni_ctx *ctx, const BitGeom &g, int K, int n, u32 **out /* n pointers */)
{
    size_t one = g.plane * (size_t)K * sizeof(u32);
    one = (one + 255) & ~(size_t)255;
    FK_TRY(omni_ws_reserve(ctx, 4, one * n));
    for (int i = 0; i < n; i++) out[i] = (u32 *)((u8 *)ctx->ws[4] + one * i);
    return OMNI_OK;
}

// workspace of the dense generation of the fused call (bit_planes: four plane sets in slot 4; blurred byte planes of
// edge_kernel_size 5 / 7 in slot 0; tables in slot 5; run lists in slot 6; a label plane in slot 2 when the caller passes none)
void dense_ws_bytes(int h, int w, int K, int nf, int ksize, size_t out[OMNI_WS_SLOTS])
{
    const BitGeom g = make_geom(h, w);
    const int KT = nf * K;
    size_t one = (g.plane * (size_t)KT * sizeof(u32) + 255) & ~(size_t)255;
    unsigned off[ET_MAXT];
    out[4] = std::max(out[4], one * 4);
    out[5] = std::max(out[5], WS5_BYTES);
    out[6] = std::max(out[6], edges3_run_words(h, w, KT, off) * sizeof(u32));
    out[2] = std::max(out[2], (((size_t)w + 15) & ~(size_t)15) * h);
    if (ksize != 3) out[0] = std::max(out[0], (((size_t)w + 15) & ~(size_t)15) * h * KT);
}

// the RGB-cell tables hold output labels in 4 bits (15 = "several candidates" when K <= 15): every label must be < K
bool lut_below_k(const AssignParams &P)
{
    for (int k = 0; k < P.K; k++)
        if (P.lut[k] >= P.K) return false;
    return true;
}

// candidate-cell tables for the centres of this call (workspace slot 5), built on the device
static int assign_cells(omni_ctx *ctx, const AssignParams &P, u32 **cells, u8 **rcells, cudaStream_t st)
{
    FK_TRY(omni_ws_reserve(ctx, 5, WS5_BYTES));
    const int variant = (ctx->assign_rgbcell && P.K <= RC_MAX_K && lut_below_k(P)) ? 2 : 1;
    *cells = (u32 *)ctx->ws[5];
    *rcells = (u8 *)((u32 *)ctx->ws[5] + RGBCELL_OFFSET);
    // same centres (and label map) as the previous call on this ctx (a batch of frames): the tables in the workspace are
    // still valid (calls on one ctx are serialised and go to one stream at a time, see omni_b200.h)
    if (ctx->table_cache && ctx->cells_valid == variant && ctx->cells_stream == (void *)st && ctx->cells_K == P.K &&
        memcmp(ctx->cells_c, P.c, sizeof(float) * 3 * P.K) == 0 && memcmp(ctx->cells_lut, P.lut, P.K) == 0)
        return OMNI_OK;
    memcpy(ctx->cells_c, P.c, sizeof(float) * 3 * P.K);
    memcpy(ctx->cells_lut, P.lut, P.K);
    ctx->cells_K = P.K; ctx->cells_stream = (void *)st; ctx->cells_valid = variant;
    {
        KScope ks(ctx, "build_cells", st);
        fk_build_cells<<<CELL_COUNT / 256, 256, 0, st>>>(P, *cells);
        OMNI_CUDA(cudaGetLastError());
    }
    if (variant == 2) {
        FK_TRY(fast_rgb_boxes(ctx, st));
        KScope ks(ctx, "build_rgbcells", st);
        fk_build_rgbcells<<<RC_COUNT / 8 / 256, 256, 0, st>>>(P, ctx->d_rgb_boxes, (u32 *)*rcells, *rcells + RC_NIB_BYTES);
        OMNI_CUDA(cudaGetLastError());
    }
    return OMNI_OK;
}

// will launch_assign_lab use the kernel that can carry a ZeroJob?
static bool assign_takes_zero_job(omni_ctx *ctx, const AssignParams &P, int nf, int h, int w)
{
    const unsigned long long plane = (unsigned long long)(((((w + 31) >> 5) + 3) & ~3)) * h;
    return ctx->assign_rgbcell && P.K <= RC_MAX_K && lut_below_k(P) && (long long)nf * h * ((w + 255) >> 8) < (1ll << 30) &&
           (unsigned long long)nf * P.K * plane < (1ull << 30);
}

// Lab-centre assignment of rows [0, h) at px: labels and/or one-hot bit-plane words (either may be NULL)
static int launch_assign_lab(omni_ctx *ctx, const u8 *px, int h, int w, size_t pitch, const AssignParams &P, u8 *labels, size_t lpitch,
                             u32 *bits, int ws, size_t plane, cudaStream_t st, bool scoped = true, int nf = 1, size_t frame_stride = 0,
                             const ZeroJob *zero = nullptr /* only honoured by the RGB-cell kernel: check assign_takes_zero_job() */)
{
    // the RGB-cell kernel counts chunks in 32 bits and takes a whole batch; the Lab-cell kernel takes one frame per launch
    const bool use_rgb = ctx->assign_rgbcell && P.K <= RC_MAX_K && lut_below_k(P) && (long long)nf * h * ((w + 255) >> 8) < (1ll << 30) &&
                         (unsigned long long)nf * P.K * plane < (1ull << 30);        // 32-bit word / byte offsets inside the kernel
    if (!use_rgb && nf > 1) {
        for (int f = 0; f < nf; f++)
            FK_TRY(launch_assign_lab(ctx, px + (size_t)f * frame_stride, h, w, pitch, P, labels ? labels + (size_t)f * h * lpitch : nullptr,
                                     lpitch, bits ? bits + (size_t)f * P.K * plane : nullptr, ws, plane, st, scoped, 1, 0));
        return OMNI_OK;
    }
    u32 *cells = nullptr;
    u8 *rcells = nullptr;
    FK_TRY(assign_cells(ctx, P, &cells, &rcells, st));
    KScope ks(scoped ? ctx : nullptr, "assign_bits", st);
    if (use_rgb) {
        if (!ctx->occ_assign_rgb) {
            OMNI_CUDA(cudaFuncSetAttribute(fk_assign_rgbcell<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, RA_SMEM));
            OMNI_CUDA(cudaFuncSetAttribute(fk_assign_rgbcell<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, RA_SMEM));
            ctx->occ_assign_rgb = 1;
        }
        // one CTA per SM (its tables fill most of the shared memory); no more CTAs than chunks of 32 warps
        const long long chunks = (long long)nf * h * ((w + 255) >> 8);
        const int grid = (int)std::max<long long>(1, std::min<long long>(persist_blocks(ctx, 1), (chunks + RA_WARPS - 1) / RA_WARPS));
        ZeroJob Z{};
        if (zero) Z = *zero;
        for (int z = 0; z < 2; z++)                         // units per chunk, rounded up to one store per lane
            Z.per[z] = (unsigned)(((Z.n16[z] + (unsigned long long)chunks - 1) / (unsigned long long)chunks + 31) & ~31ull);
        if (P.K >= 16)
            fk_assign_rgbcell<true><<<grid, RA_THREADS, RA_SMEM, st>>>(px, h, w, pitch, P, (const uint4 *)rcells, cells, labels, lpitch, bits, ws,
                                                                       plane, nf, frame_stride, Z);
        else
            fk_assign_rgbcell<false><<<grid, RA_THREADS, RA_SMEM, st>>>(px, h, w, pitch, P, (const uint4 *)rcells, cells, labels, lpitch, bits, ws,
                                                                        plane, nf, frame_stride, Z);
    } else {
        const int grid = resident_grid(ctx, fk_assign_bits<1>, 256, &ctx->occ_assign_lab);
        fk_assign_bits<1><<<grid, 256, 0, st>>>(px, h, w, pitch, P, cells, labels, lpitch, bits, ws, plane);
    }
    OMNI_CUDA(cudaGetLastError());
    return OMNI_OK;
}

cudaError_t fast_assign(omni_ctx *ctx, const u8 *px, int h, int w, size_t pitch, const AssignParams &P, int mode_lab,
                        u8 *labels, size_t lpitch, cudaStream_t st)
{
    cudaError_t e = fast_tables();
    if (e != cudaSuccess) return e;
    if (mode_lab) {
        if (launch_assign_lab(ctx, px, h, w, pitch, P, labels, lpitch, nullptr, 0, 0, st, false) != OMNI_OK) return cudaErrorUnknown;
    } else if (P.K <= 16) {
        const int grid = resident_grid(ctx, fk_assign_i16wrap<16>, 256, &ctx->occ_assign_i16);
        if (P.K <= 4) fk_assign_i16wrap<4><<<grid, 256, 0, st>>>(px, h, w, pitch, P, labels, lpitch);
        else if (P.K <= 8) fk_assign_i16wrap<8><<<grid, 256, 0, st>>>(px, h, w, pitch, P, labels, lpitch);
        else fk_assign_i16wrap<16><<<grid, 256, 0, st>>>(px, h, w, pitch, P, labels, lpitch);
    } else {                                                 // more than 16 palette colours: the plain K loop
        int grid = resident_grid(ctx, fk_assign_bits<0>, 256, &ctx->occ_assign_pal);
        fk_assign_bits<0><<<grid, 256, 0, st>>>(px, h, w, pitch, P, nullptr, labels, lpitch, nullptr, 0, 0);
    }
    return cudaGetLastError();
}

bool fast_masks_supported(int open_iters, int close_iters)
{
    return (open_iters == 1 && close_iters == 1) || (open_iters <= 0 && close_iters <= 0);
}

int fast_layer_masks(omni_ctx *ctx, const u8 *d_labels, int h, int w, size_t lpitch, int K, int open_iters, int close_iters,
                     u8 *d_masks, size_t plane_stride, size_t mpitch, cudaStream_t st)
{
    BitGeom g = make_geom(h, w);
    u32 *bp[1];
    FK_TRY(bit_planes(ctx, g, K, 1, bp));
    {
        KScope ks(ctx, "labels_to_bits", st);
        fk_labels_to_bits<<<persist_blocks(ctx, 8), 256, 0, st>>>(d_labels, h, w, lpitch, K, bp[0], g.ws, g.plane);
        OMNI_CUDA(cudaGetLastError());
    }
    int al = plane_align(d_masks, plane_stride, mpitch);
    if (open_iters == 1 && close_iters == 1) {
        OMNI_LAUNCH(ctx, st, "morph_bits", launch_morph(true, 0, bp[0], nullptr, g, K, d_masks, plane_stride, mpitch, st));
    } else {
        KScope ks(ctx, "expand_bits", st);
        fk_expand_bits<<<dim3(persist_blocks(ctx, 4), K), 256, 0, st>>>(bp[0], g.ws, g.plane, h, w, d_masks, plane_stride, mpitch, al);
        OMNI_CUDA(cudaGetLastError());
    }
    return OMNI_OK;
}

// which stage-03 morphology the parameters ask for: 0 none, 1 open, 2 close, 3 both; -1 = not on the fast path
int morph03_kind(const omni_edge_params *p)
{
    int oi = p->open_iters > 0 ? p->open_iters : 0, ci = p->close_iters > 0 ? p->close_iters : 0;
    if (p->morph_k == 1) return 0;                    // 1x1 element: identity
    if (p->morph_k != 3 || oi > 1 || ci > 1) return -1;
    return oi | (ci << 1);
}

// stage-03 morphology on bit-planes: fk_morph's chains (morph03_kind >= 0) or the ELLIPSE kernel of morph_ellipse.cu (every other
// element size and iteration count)
static bool morph03_bits_ok(const omni_edge_params *p) { return morph03_kind(p) >= 0 || (p->morph_k >= 2 && p->morph_k <= OMNI_MAX_MORPH_K); }

bool fast_edges_supported(const omni_edge_params *prm)
{
    return morph03_bits_ok(prm) && (prm->ksize == 3 || prm->ksize == 5 || prm->ksize == 7);
}

bool fast_fused_supported(const omni_edge_params *prm) { return morph03_kind(prm) >= 0 && prm->ksize == 3; }

bool fast_morph03_supported(const omni_edge_params *prm) { return morph03_bits_ok(prm); }

int fast_morph03_bytes(omni_ctx *ctx, const u8 *d_masks, int K, int h, int w, size_t m_plane, size_t mpitch,
                       const omni_edge_params *prm, u8 *d_out, size_t o_plane, size_t opitch, cudaStream_t st)
{
    BitGeom g = make_geom(h, w);
    u32 *bpp[2];
    FK_TRY(bit_planes(ctx, g, K, 2, bpp));
    OMNI_CUDA(cudaMemsetAsync(ctx->d_flags + 8, 0, sizeof(int), st));
    {
        KScope ks(ctx, "bytes_to_bits", st);
        fk_bytes_to_bits<true><<<dim3(persist_blocks(ctx, 2), K), 256, 0, st>>>(d_masks, m_plane, mpitch, h, w, bpp[0], g.ws, g.plane,
                                                                               ctx->d_flags + 8);
        OMNI_CUDA(cudaGetLastError());
    }
    if (!ctx->assume_binary) {                            // (omni_set_assume_binary_masks: the caller vouches, nothing to wait for)
        OMNI_CUDA(cudaMemcpyAsync(ctx->h_flags + 8, ctx->d_flags + 8, sizeof(int), cudaMemcpyDeviceToHost, st));
        OMNI_CUDA(cudaStreamSynchronize(st));
        if (ctx->h_flags[8]) return OMNI_ERR_UNSUPPORTED;     // not a {0,255} mask
    }
    const int kind = morph03_kind(prm);
    const u32 *m2 = bpp[0];
    if (kind > 0) {
        OMNI_LAUNCH(ctx, st, "morph_bits", launch_morph(false, kind, bpp[0], bpp[1], g, K, nullptr, 0, 0, st));
        m2 = bpp[1];
    } else if (kind < 0) {
        FK_TRY(ellipse_morph_bits(ctx, prm, g, K, bpp[0], bpp[1], &m2, st));
    }
    int al = plane_align(d_out, o_plane, opitch);
    KScope ks(ctx, "expand_bits", st);
    fk_expand_bits<<<dim3(persist_blocks(ctx, 4), K), 256, 0, st>>>(m2, g.ws, g.plane, h, w, d_out, o_plane, opitch, al);
    OMNI_CUDA(cudaGetLastError());
    return OMNI_OK;
}

int run_hysteresis(omni_ctx *ctx, u32 *ebits, const u32 *cbits, const BitGeom &g, int K, u8 *d_edges,
                          size_t e_plane, size_t epitch, cudaStream_t st, int *flags_in, const u32 *worklist_in)
{
    if (ctx->hyst_blocks == 0) {
        int per_sm = 0;
        OMNI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fk_hysteresis, HY_THREADS, 0));
        if (per_sm < 1) { omni_set_error("hysteresis kernel cannot be made resident"); return OMNI_ERR_CUDA; }
        ctx->hyst_blocks = per_sm * (ctx->sm_count > 0 ? ctx->sm_count : 1);
    }
    int ws = g.ws, h = g.h, w = g.w;
    size_t plane = g.plane;
    int *flags = flags_in ? flags_in : ctx->d_flags;
    const u32 *worklist = worklist_in ? worklist_in : (const u32 *)ctx->ws[5] + HYST_WL_OFFSET;
    void *args[] = {&ebits, &cbits, &ws, &plane, &h, &w, &K, &flags, &worklist, &d_edges, &e_plane, &epitch};
    OMNI_LAUNCH(ctx, st, "hysteresis_bits", cudaLaunchCooperativeKernel((const void *)fk_hysteresis, dim3(ctx->hyst_blocks), dim3(HY_THREADS),
                                                                        args, 0, st));
    if (!flags_in) {
        ctx->last_hyst_passes = -1;       // lives in d_flags[0]; fetched lazily by omni_last_hysteresis_passes
        ctx->last_hyst_stream = st;
    }
    return OMNI_OK;
}

int run_hysteresis_wl(omni_ctx *ctx, u32 *ebits, const u32 *cbits, const BitGeom &g, int K, cudaStream_t st, const int *flags, const u32 *worklist)
{
    (void)K;
    KScope ks(ctx, "hysteresis_wl", st);
    fk_hysteresis_wl<<<1, HY_THREADS, 0, st>>>(ebits, cbits, g.ws, g.plane, g.h, g.w, flags, worklist);
    OMNI_CUDA(cudaGetLastError());
    return OMNI_OK;
}

// Zeroes the device flags of an edge pass -- d_flags: [0] rounds, [1..3] changed flags, [4] weak-word count, [16..19] run
// counts per length, [20] next warp item -- and, when the sparse edge kernel will run, fills the MorphRuns block that lets
// the morphology kernel produce the run lists (returns false: dense edge kernel, nothing to prepare).
int edge_pass_begin(omni_ctx *ctx, const BitGeom &g, int K, u32 *sbits, u32 *cbits, u8 *d_edges, size_t e_plane, size_t epitch,
                           cudaStream_t st, MorphRuns *R, bool *sparse, bool side_fill, ZeroJob *zjob)
{
    FK_TRY(omni_ws_reserve(ctx, 5, WS5_BYTES));
    OMNI_CUDA(cudaMemsetAsync(ctx->d_flags, 0, 24 * sizeof(int), st));
    ctx->edge_join = nullptr;
    *sparse = ctx->edge_sparse && edges3_sparse_ok(g.h, g.w, K);
    if (!*sparse) return OMNI_OK;
    if (ctx->e3s_per_sm == 0) ctx->e3s_per_sm = edges3_sparse_blocks_per_sm();
    FK_TRY(omni_ws_reserve(ctx, 6, edges3_run_words(g.h, g.w, K, R->off.v) * sizeof(u32)));
    R->sbits = sbits; R->cbits = cbits; R->edges = d_edges; R->estride = e_plane; R->epitch = epitch;
    R->aligned16 = plane_align(d_edges, e_plane, epitch);
    R->run_counts = ctx->d_flags + 16; R->run_items = (u32 *)ctx->ws[6];
    R->maxt = edges3_pick_maxt(g.h, g.w, K, 2 * persist_blocks(ctx, ctx->e3s_per_sm));
    R->zero_fill = side_fill ? 0 : 1;
    if (side_fill && zjob && epitch == (size_t)g.w && e_plane == epitch * (size_t)g.h && (uintptr_t)d_edges % 16 == 0 &&
        (e_plane * (size_t)K) % 16 == 0 && cbits == sbits + ((g.plane * (size_t)K * sizeof(u32) + 255) & ~(size_t)255) / sizeof(u32)) {
        // contiguous planes: the assignment kernel clears them on the way (ZeroJob)
        zjob->p[0] = (uint4 *)d_edges; zjob->n16[0] = e_plane * (size_t)K / 16;
        zjob->p[1] = (uint4 *)sbits;   zjob->n16[1] = (size_t)((u8 *)cbits - (u8 *)sbits + g.plane * (size_t)K * sizeof(u32)) / 16;
        return OMNI_OK;
    }
    if (side_fill) {
        // The zeros of the dead tiles (most of the 2K bytes per pixel the edge pass writes) do not depend on anything: clear
        // the edge byte planes and the candidate / strong bit-planes on a side stream while the colour assignment and the
        // morphology (both bound by instruction issue, not by HBM) run; the edge kernel joins before it writes the live tiles.
        FK_TRY(pipe_init(ctx));
        cudaEvent_t fork = ctx->pipe_ev[2 * HP_MAX_BANDS + 4], join = ctx->pipe_ev[2 * HP_MAX_BANDS + 5];
        cudaStream_t ss = ctx->s_in;
        OMNI_CUDA(cudaEventRecord(fork, st));
        OMNI_CUDA(cudaStreamWaitEvent(ss, fork, 0));
        if (epitch == (size_t)g.w && e_plane == epitch * (size_t)g.h) OMNI_CUDA(cudaMemsetAsync(d_edges, 0, e_plane * (size_t)K, ss));
        else                                        // strided views: only the pixels of the planes may be touched
            for (int k = 0; k < K; k++) OMNI_CUDA(cudaMemset2DAsync(d_edges + (size_t)k * e_plane, epitch, 0, (size_t)g.w, g.h, ss));
        const size_t pbytes = g.plane * (size_t)K * sizeof(u32);
        OMNI_CUDA(cudaMemsetAsync(sbits, 0, pbytes, ss));
        OMNI_CUDA(cudaMemsetAsync(cbits, 0, pbytes, ss));
        OMNI_CUDA(cudaEventRecord(join, ss));
        ctx->edge_join = join;
    }
    return OMNI_OK;
}

// bit-planes M2 -> edge byte planes.  sbits doubles as the working set E of the hysteresis.  edge_pass_begin has run;
// runs_done: the morphology kernel has already produced the run lists and zero-filled the dead tiles.
static int edges_from_bits(omni_ctx *ctx, const u32 *m2, u32 *sbits, u32 *cbits, const BitGeom &g, int K, int low, int high,
                           u8 *d_edges, size_t e_plane, size_t epitch, cudaStream_t st, bool sparse, bool runs_done,
                           const u8 *blur = nullptr /* edge_kernel_size 5 / 7: the blurred planes */, size_t bstride = 0, size_t bpitch = 0)
{
    int al = plane_align(d_edges, e_plane, epitch);
    if (ctx->edge_join) {                               // the side stream has cleared the output planes
        OMNI_CUDA(cudaStreamWaitEvent(st, ctx->edge_join, 0));
        ctx->edge_join = nullptr;
    }
    if (sparse) {
        if (!runs_done)
            OMNI_LAUNCH(ctx, st, "edge_runs", launch_edge_runs(m2, g.ws, g.plane, g.h, g.w, K, sbits, cbits, d_edges, e_plane, epitch, al,
                                                               ctx->d_flags + 16, (u32 *)ctx->ws[6], 2 * persist_blocks(ctx, ctx->e3s_per_sm), st));
        OMNI_LAUNCH(ctx, st, "edges3_bits", launch_edges3_sparse(m2, g.ws, g.plane, g.h, g.w, K, low, high, persist_blocks(ctx, ctx->e3s_per_sm),
                                                                 sbits, cbits, d_edges, e_plane, epitch, al, ctx->d_flags + 4,
                                                                 (u32 *)ctx->ws[5] + HYST_WL_OFFSET, HY_WL_CAP, ctx->d_flags + 16,
                                                                 ctx->d_flags + 20, (const u32 *)ctx->ws[6], st, blur, bstride, bpitch));
    } else {
        OMNI_LAUNCH(ctx, st, "edges3_bits", launch_edges3_simd(m2, g.ws, g.plane, g.h, g.w, K, low, high, ctx->sm_count, sbits, cbits,
                                                               d_edges, e_plane, epitch, al, ctx->d_flags + 4,
                                                               (u32 *)ctx->ws[5] + HYST_WL_OFFSET, HY_WL_CAP, st, blur, bstride, bpitch));
    }
    return run_hysteresis(ctx, sbits, cbits, g, K, d_edges, e_plane, epitch, st);
}

int fast_edges(omni_ctx *ctx, const u8 *d_masks, int K, int h, int w, size_t m_plane, size_t mpitch,
               const omni_edge_params *prm, const BlurParams &bp, int low, int high,
               u8 *d_edges, size_t e_plane, size_t epitch, cudaStream_t st)
{
    (void)bp;
    if (low < 0) return OMNI_ERR_UNSUPPORTED;        // m == 0 would be a candidate: generic kernels handle it
    BitGeom g = make_geom(h, w);
    u32 *bpp[4];
    FK_TRY(bit_planes(ctx, g, K, 4, bpp));
    OMNI_CUDA(cudaMemsetAsync(ctx->d_flags + 8, 0, sizeof(int), st));
    {
        KScope ks(ctx, "bytes_to_bits", st);
        fk_bytes_to_bits<true><<<dim3(persist_blocks(ctx, 2), K), 256, 0, st>>>(d_masks, m_plane, mpitch, h, w, bpp[0], g.ws, g.plane,
                                                                               ctx->d_flags + 8);
        OMNI_CUDA(cudaGetLastError());
    }
    if (!ctx->assume_binary) {                            // (omni_set_assume_binary_masks: the caller vouches, nothing to wait for)
        OMNI_CUDA(cudaMemcpyAsync(ctx->h_flags + 8, ctx->d_flags + 8, sizeof(int), cudaMemcpyDeviceToHost, st));
        OMNI_CUDA(cudaStreamSynchronize(st));
        if (ctx->h_flags[8]) return OMNI_ERR_UNSUPPORTED;     // not a {0,255} mask
    }
    int kind = morph03_kind(prm);
    const u32 *m2 = bpp[0];
    MorphRuns R{};
    bool sparse = false;
    const int ks = prm->ksize;
    FK_TRY(edge_pass_begin(ctx, g, K, bpp[2], bpp[3], d_edges, e_plane, epitch, st, &R, &sparse, false));
    // a tile is dead when the tile grown by the radius of blur + Sobel is uniform; only fk_morph classifies with a growth other
    // than 2, so blur 5 / 7 without stage-03 morphology, or after the ELLIPSE kernel (kind < 0), takes the dense edge kernel
    R.grow = ks == 3 ? 2 : ks == 5 ? 3 : 4;
    if (ks != 3 && kind <= 0) sparse = false;
    if (kind > 0) {
        OMNI_LAUNCH(ctx, st, "morph_bits", launch_morph(false, kind, bpp[0], bpp[1], g, K, nullptr, 0, 0, st, 0, -1, sparse ? &R : nullptr));
        m2 = bpp[1];
    } else if (kind < 0) {                               // other ELLIPSE sizes / counts: the run lists come from edge_runs
        FK_TRY(ellipse_morph_bits(ctx, prm, g, K, bpp[0], bpp[1], &m2, st));
    }
    const u8 *blur = nullptr;
    size_t bp_pitch = 0, bp_plane = 0;
    if (ks != 3) {                                       // GaussianBlur 5 / 7 of the bit-planes -> u8 planes (workspace slot 0)
        bp_pitch = ((size_t)w + 15) & ~(size_t)15; bp_plane = bp_pitch * h;
        FK_TRY(omni_ws_reserve(ctx, 0, bp_plane * K));
        OMNI_LAUNCH(ctx, st, "blur_bits", launch_blur_bits(ks, m2, g.ws, g.plane, K, h, w, (u8 *)ctx->ws[0], bp_plane, bp_pitch,
                                                           persist_blocks(ctx, 16), st));
        blur = (const u8 *)ctx->ws[0];
    }
    return edges_from_bits(ctx, m2, bpp[2], bpp[3], g, K, low, high, d_edges, e_plane, epitch, st, sparse, sparse && kind > 0, blur, bp_plane,
                           bp_pitch);
}

int fast_color_edge(omni_ctx *ctx, const u8 *d_bgr, int h, int w, size_t pitch, const AssignParams &P,
                    const omni_edge_params *prm, const BlurParams &bp, int low, int high,
                    u8 *d_labels, size_t lpitch, u8 *d_masks, size_t m_plane, size_t mpitch,
                    u8 *d_edges, size_t e_plane, size_t epitch, cudaStream_t st)
{
    (void)bp;
    if (low < 0) return OMNI_ERR_UNSUPPORTED;
    if (ctx->pipeline == 1) {                          // sparse generation (label_pipe.cu) where it applies
        const int rc = sparse_color_edge(ctx, d_bgr, 1, 0, h, w, pitch, P, prm, low, high, d_labels, lpitch, d_masks, m_plane, mpitch,
                                         d_edges, e_plane, epitch, st);
        if (rc != OMNI_ERR_UNSUPPORTED) return rc;
    }
    OMNI_CUDA(fast_tables());
    BitGeom g = make_geom(h, w);
    u32 *bpp[4];
    FK_TRY(bit_planes(ctx, g, P.K, 4, bpp));
    // first of all: fork the side stream that clears the edge planes, so that it runs under the assignment kernel
    MorphRuns R{};
    bool sparse = false;
    ZeroJob Z{};
    const bool zj = assign_takes_zero_job(ctx, P, 1, h, w);
    FK_TRY(edge_pass_begin(ctx, g, P.K, bpp[2], bpp[3], d_edges, e_plane, epitch, st, &R, &sparse, true, zj ? &Z : nullptr));
    OMNI_CUDA(cudaMemsetAsync(bpp[0], 0, g.plane * (size_t)P.K * sizeof(u32), st));      // match_any stores only non-empty words
    FK_TRY(launch_assign_lab(ctx, d_bgr, h, w, pitch, P, d_labels, lpitch, bpp[0], g.ws, g.plane, st, true, 1, 0, &Z));
    int kind = morph03_kind(prm);
    OMNI_LAUNCH(ctx, st, "morph_bits", launch_morph(true, kind, bpp[0], bpp[1], g, P.K, d_masks, m_plane, mpitch, st, 0, -1, sparse ? &R : nullptr));
    return edges_from_bits(ctx, bpp[1], bpp[2], bpp[3], g, P.K, low, high, d_edges, e_plane, epitch, st, sparse, sparse);
}


// A batch of n equally sized frames that share one centre set (BASELINE config 4: video frames).  After the colour
// assignment nothing couples the K layers of a frame, so the n * K layers of the batch are simply n * K planes of one
// geometry: one morphology launch, one edge launch and one hysteresis launch serve the whole batch (a 1080p frame alone
// cannot fill the machine).  Plane f * K + k of the mask / edge tensors belongs to layer k of frame f.  n * K <= OMNI_MAX_K.
int fast_color_edge_batch(omni_ctx *ctx, const u8 *d_bgr, int n, size_t frame_stride, int h, int w, size_t pitch, const AssignParams &P,
                          const omni_edge_params *prm, int low, int high, u8 *d_masks, size_t m_plane, size_t mpitch,
                          u8 *d_edges, size_t e_plane, size_t epitch, cudaStream_t st)
{
    if (low < 0) return OMNI_ERR_UNSUPPORTED;
    const int KT = n * P.K;
    if (KT > OMNI_MAX_K) return OMNI_ERR_UNSUPPORTED;
    if (ctx->pipeline == 1) {
        const int rc = sparse_color_edge(ctx, d_bgr, n, frame_stride, h, w, pitch, P, prm, low, high, nullptr, 0, d_masks, m_plane, mpitch,
                                         d_edges, e_plane, epitch, st);
        if (rc != OMNI_ERR_UNSUPPORTED) return rc;
    }
    OMNI_CUDA(fast_tables());
    BitGeom g = make_geom(h, w);
    u32 *bpp[4];
    FK_TRY(bit_planes(ctx, g, KT, 4, bpp));
    MorphRuns R{};
    bool sparse = false;
    ZeroJob Z{};
    const bool zj = assign_takes_zero_job(ctx, P, n, h, w);
    FK_TRY(edge_pass_begin(ctx, g, KT, bpp[2], bpp[3], d_edges, e_plane, epitch, st, &R, &sparse, true, zj ? &Z : nullptr));
    OMNI_CUDA(cudaMemsetAsync(bpp[0], 0, g.plane * (size_t)KT * sizeof(u32), st));
    FK_TRY(launch_assign_lab(ctx, d_bgr, h, w, pitch, P, nullptr, 0, bpp[0], g.ws, g.plane, st, true, n, frame_stride, &Z));
    int kind = morph03_kind(prm);
    OMNI_LAUNCH(ctx, st, "morph_bits", launch_morph(true, kind, bpp[0], bpp[1], g, KT, d_masks, m_plane, mpitch, st, 0, -1, sparse ? &R : nullptr));
    return edges_from_bits(ctx, bpp[1], bpp[2], bpp[3], g, KT, low, high, d_edges, e_plane, epitch, st, sparse, sparse);
}

// ------------------------------------------------------------------------------------------------
// Host-buffer fused call, pipelined over row bands (omni_host_color_edge when the fast path applies).
// PCIe is the bound of this call (3 B/px in, 2K B/px out), so copies and kernels are overlapped:
//   copy-in stream : band b of the image                                   (H2D)
//   compute stream : assign(b) as soon as band b has landed; morph(b-1) once assign(b) is done (its 8-row halo);
//                    after the last band: edge kernel + hysteresis on the whole image
//   copy-out stream: mask planes of band b as soon as morph(b) is done; labels; edge planes at the end   (D2H)
// ------------------------------------------------------------------------------------------------
static int pipe_init(omni_ctx *ctx)
{
    if (ctx->pipe_ready) return OMNI_OK;
    OMNI_CUDA(cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
    OMNI_CUDA(cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
    for (int i = 0; i < 2 * HP_MAX_BANDS + 6; i++) OMNI_CUDA(cudaEventCreateWithFlags(&ctx->pipe_ev[i], cudaEventDisableTiming));
    ctx->pipe_ready = 1;
    return OMNI_OK;
}

void fast_ctx_release(omni_ctx *ctx)
{
    if (!ctx || !ctx->pipe_ready) return;
    cudaStreamDestroy(ctx->s_in);
    cudaStreamDestroy(ctx->s_out);
    for (int i = 0; i < 2 * HP_MAX_BANDS + 6; i++) cudaEventDestroy(ctx->pipe_ev[i]);
    ctx->pipe_ready = 0;
}

int fast_host_color_edge(omni_ctx *ctx, const u8 *h_bgr, int h, int w, size_t pitch, const AssignParams &P,
                         const omni_edge_params *prm, int low, int high,
                         u8 *h_labels, size_t lpitch, u8 *h_masks, size_t h_mplane, size_t h_mpitch,
                         u8 *h_edges, size_t h_eplane, size_t h_epitch,
                         u8 *d_img, size_t ip, u8 *d_labels, size_t lp, u8 *d_masks, size_t mplane, size_t mp,
                         u8 *d_edges, size_t eplane, size_t ep, bool want_labels)
{
    if (low < 0 || !fast_fused_supported(prm)) return OMNI_ERR_UNSUPPORTED;
    FK_TRY(pipe_init(ctx));
    OMNI_CUDA(fast_tables());
    const int K = P.K;
    BitGeom g = make_geom(h, w);
    u32 *bpp[4];
    FK_TRY(bit_planes(ctx, g, K, 4, bpp));
    cudaStream_t sc = ctx->stream, si = ctx->s_in, so = ctx->s_out;
    cudaEvent_t *evH = ctx->pipe_ev, *evM = ctx->pipe_ev + HP_MAX_BANDS, *evX = ctx->pipe_ev + 2 * HP_MAX_BANDS;
    // bands: multiples of the morphology strip height.  Tall images start with short bands (128, 128, 256, 512 rows) so that the
    // first masks leave for the host while most of the image is still arriving; the rest is split evenly.
    int ys[HP_MAX_BANDS + 1];
    int nb = 0;
    ys[0] = 0;
    if (h >= 2048) {
        const int lead[4] = {128, 128, 256, 512};
        for (int i = 0; i < 4; i++) { ys[nb + 1] = ys[nb] + lead[i]; nb++; }
    }
    {
        const int left = h - ys[nb], slots = HP_MAX_BANDS - nb;
        int n_even = slots;
        while (n_even > 1 && (left + n_even - 1) / n_even < 256) n_even--;
        const int per = ((left + n_even - 1) / n_even + MORPH_TR_BIG - 1) / MORPH_TR_BIG * MORPH_TR_BIG;
        while (ys[nb] < h) { ys[nb + 1] = min(h, ys[nb] + per); nb++; }
    }
    const int kind = morph03_kind(prm);
    // everything queued on the side streams must wait for what the caller queued before on the ctx stream -- nothing:
    // omni_host_* calls own ctx->stream; a start event orders the side streams after earlier work of this ctx
    OMNI_CUDA(cudaEventRecord(evX[0], sc));
    OMNI_CUDA(cudaStreamWaitEvent(si, evX[0], 0));
    OMNI_CUDA(cudaStreamWaitEvent(so, evX[0], 0));
    for (int b = 0; b < nb; b++) {
        int y0 = ys[b], rows = ys[b + 1] - y0;
        OMNI_CUDA(cudaMemcpy2DAsync(d_img + (size_t)y0 * ip, ip, h_bgr + (size_t)y0 * pitch, pitch, (size_t)w * 3, rows,
                                    cudaMemcpyHostToDevice, si));
        OMNI_CUDA(cudaEventRecord(evH[b], si));
    }
    OMNI_CUDA(cudaMemsetAsync(bpp[0], 0, g.plane * (size_t)K * sizeof(u32), sc));
    MorphRuns R{};
    bool sparse = false;
    FK_TRY(edge_pass_begin(ctx, g, K, bpp[2], bpp[3], d_edges, eplane, ep, sc, &R, &sparse, true));
    auto morph_band = [&](int b) -> int {
        int y0 = ys[b], y1 = ys[b + 1];
        OMNI_LAUNCH(ctx, sc, "morph_bits", launch_morph(true, kind, bpp[0], bpp[1], g, K, d_masks, mplane, mp, sc, y0, y1, sparse ? &R : nullptr));
        OMNI_CUDA(cudaEventRecord(evM[b], sc));
        OMNI_CUDA(cudaStreamWaitEvent(so, evM[b], 0));
        const bool contiguous = (h_mpitch == mp && mp == (size_t)w);      // gap-free rows on both sides only
        if (contiguous) {
            // the band of all K planes in ONE strided copy: "row" = a plane's band (contiguous rows), "pitch" = the plane stride
            OMNI_CUDA(cudaMemcpy2DAsync(h_masks + (size_t)y0 * h_mpitch, h_mplane, d_masks + (size_t)y0 * mp, mplane,
                                        (size_t)(y1 - y0 - 1) * mp + w, K, cudaMemcpyDeviceToHost, so));
        } else {
            for (int k = 0; k < K; k++)
                OMNI_CUDA(cudaMemcpy2DAsync(h_masks + (size_t)k * h_mplane + (size_t)y0 * h_mpitch, h_mpitch,
                                            d_masks + (size_t)k * mplane + (size_t)y0 * mp, mp, (size_t)w, y1 - y0, cudaMemcpyDeviceToHost, so));
        }
        return OMNI_OK;
    };
    for (int b = 0; b < nb; b++) {
        int y0 = ys[b], rows = ys[b + 1] - y0;
        OMNI_CUDA(cudaStreamWaitEvent(sc, evH[b], 0));
        FK_TRY(launch_assign_lab(ctx, d_img + (size_t)y0 * ip, rows, w, ip, P, want_labels ? d_labels + (size_t)y0 * lp : nullptr, lp,
                                 bpp[0] + (size_t)y0 * g.ws, g.ws, g.plane, sc));
        if (b > 0) FK_TRY(morph_band(b - 1));             // its halo rows (band b) are assigned now
    }
    FK_TRY(morph_band(nb - 1));
    if (want_labels && h_labels) {
        OMNI_CUDA(cudaEventRecord(evX[1], sc));
        OMNI_CUDA(cudaStreamWaitEvent(so, evX[1], 0));
        OMNI_CUDA(cudaMemcpy2DAsync(h_labels, lpitch, d_labels, lp, (size_t)w, h, cudaMemcpyDeviceToHost, so));
    }
    FK_TRY(edges_from_bits(ctx, bpp[1], bpp[2], bpp[3], g, K, low, high, d_edges, eplane, ep, sc, sparse, sparse));
    OMNI_CUDA(cudaEventRecord(evX[2], sc));
    OMNI_CUDA(cudaStreamWaitEvent(so, evX[2], 0));
    if (h_epitch == ep && ep == (size_t)w) {            // gap-free rows: a plane is one contiguous run
        OMNI_CUDA(cudaMemcpy2DAsync(h_edges, h_eplane, d_edges, eplane, (size_t)(h - 1) * ep + w, K, cudaMemcpyDeviceToHost, so));
    } else {
        for (int k = 0; k < K; k++)
            OMNI_CUDA(cudaMemcpy2DAsync(h_edges + (size_t)k * h_eplane, h_epitch, d_edges + (size_t)k * eplane, ep, (size_t)w, h,
                                        cudaMemcpyDeviceToHost, so));
    }
    // the caller continues on ctx->stream (counts) and synchronises it: make it wait for the copy-out stream
    OMNI_CUDA(cudaEventRecord(evX[3], so));
    OMNI_CUDA(cudaStreamWaitEvent(sc, evX[3], 0));
    return OMNI_OK;
}


// ------------------------------------------------------------------------------------------------
// stage 04 (SURVEY 8f rank 1): Zhang-Suen thinning of the edge planes, 04_find_contours.py:35-99.
//
// The reference runs the two sub-iterations with NumPy shifts over the bounding box of the non-zero pixels (zero
// outside -- the same as zero outside the image) until an iteration deletes nothing, at most 120 iterations.  Its
// neighbour names are rotated against the textbook:  P2 = (y+1, x)  P3 = (y+1, x-1)  P4 = (y, x-1)  P5 = (y-1, x-1)
// P6 = (y-1, x)  P7 = (y-1, x+1)  P8 = (y, x+1)  P9 = (y+1, x+1);  a pixel is deleted when  A == 1  (0 -> 1 transitions
// around P2..P9,P2),  2 <= B <= 6  (neighbour count)  and  P2 P4 P6 == 0, P4 P6 P8 == 0  (sub-step 1)  resp.
// P2 P4 P8 == 0, P2 P6 P8 == 0  (sub-step 2).
//
// Here a sub-step is ~60 bit operations per 32-pixel word: the eight neighbour planes are shifted words, B comes
// from a bit-sliced adder tree, "exactly one transition" from a one/two-or-more pair.  All K planes are thinned by ONE
// cooperative kernel: sub-step 1 reads plane set A and writes B, sub-step 2 reads B and writes A (a deletion must not
// be seen by its neighbours inside a sub-step), grid.sync() between them; three rotating "changed" flags give the
// stop test without a second barrier.  A plane that has converged stays unchanged in later iterations, so running
// all planes until the last one converges (or to max_iter) gives every plane the reference's result;
// removed[k * max_iter + i] = pixels deleted from plane k in iteration i + 1 (the number the reference logs).
// ------------------------------------------------------------------------------------------------

__device__ __forceinline__ u32 th_xor3(u32 a, u32 b, u32 c) { return a ^ b ^ c; }
__device__ __forceinline__ u32 th_maj(u32 a, u32 b, u32 c) { return (a & b) | (c & (a | b)); }

template <int STEP>
__device__ __forceinline__ u32 thin_delete_mask(u32 ul, u32 um, u32 ur, u32 ml, u32 mm, u32 mr, u32 dl, u32 dm, u32 dr)
{
    // u* = row y-1, m* = row y, d* = row y+1; *l / *m / *r = words c-1, c, c+1
    const u32 P2 = dm, P3 = __funnelshift_l(dl, dm, 1), P4 = __funnelshift_l(ml, mm, 1), P5 = __funnelshift_l(ul, um, 1);
    const u32 P6 = um, P7 = __funnelshift_r(um, ur, 1), P8 = __funnelshift_r(mm, mr, 1), P9 = __funnelshift_r(dm, dr, 1);
    // B = P2 + .. + P9, bit-sliced
    const u32 s1 = th_xor3(P2, P3, P4), c1 = th_maj(P2, P3, P4);
    const u32 s2 = th_xor3(P5, P6, P7), c2 = th_maj(P5, P6, P7);
    const u32 s3 = P8 ^ P9, c3 = P8 & P9;
    const u32 b0 = th_xor3(s1, s2, s3), c4 = th_maj(s1, s2, s3);
    const u32 t0 = th_xor3(c1, c2, c3), d1 = th_maj(c1, c2, c3);
    const u32 b1 = t0 ^ c4, d2 = t0 & c4;
    const u32 b2 = d1 ^ d2, b3 = d1 & d2;
    const u32 b_ok = (b1 | b2 | b3) & ~b3 & ~(b2 & b1 & b0);            // 2 <= B <= 6
    // A == 1: exactly one of the eight (0 -> 1) transitions
    u32 one = 0u, two = 0u, t;
    t = ~P2 & P3; two |= one & t; one |= t;
    t = ~P3 & P4; two |= one & t; one |= t;
    t = ~P4 & P5; two |= one & t; one |= t;
    t = ~P5 & P6; two |= one & t; one |= t;
    t = ~P6 & P7; two |= one & t; one |= t;
    t = ~P7 & P8; two |= one & t; one |= t;
    t = ~P8 & P9; two |= one & t; one |= t;
    t = ~P9 & P2; two |= one & t; one |= t;
    const u32 a_ok = one & ~two;
    const u32 c_ok = STEP == 1 ? (~(P2 & P4 & P6) & ~(P4 & P6 & P8)) : (~(P2 & P4 & P8) & ~(P2 & P6 & P8));
    return mm & a_ok & b_ok & c_ok;
}

// Unit skipping (exact).  Sub-steps are numbered t = 2 * iteration + (STEP - 1); every unit (16 rows x 1024 pixels) records
// in ucur whether it deleted anything in sub-step t.  What a unit sees at t differs from what it saw at t - 2 (the same kind
// of sub-step, where it deleted nothing more) only if it or one of its 8 neighbour units deleted something at t - 2 or
// t - 1 (up1 / up2): otherwise the unit is skipped.  A unit that deletes at t always runs t + 1 (its own flag), which
// rewrites the other plane set; so before every sub-step each unit's words are current in the set that is read, and a
// skipped unit holds the same words in both sets.
template <int STEP>
__device__ __forceinline__ void thin_substep(const u32 *__restrict__ src, u32 *__restrict__ dst, int ws, size_t plane, int h, int ww, int K,
                                             int *removed_it /* + k * max_iter */, int max_iter, volatile int *chg,
                                             const u8 *up1, const u8 *up2, u8 *ucur, u8 *unext, const int TH_ROWS /* rows per unit */)
{
    const int lane = threadIdx.x & 31;
    const int wcols = (ww + 31) / 32, strips = (h + TH_ROWS - 1) / TH_ROWS;
    const long long units = (long long)K * strips * wcols;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long u = warp0; u < units; u += nwarps) {
        const int wx = (int)(u % wcols);
        const long long r0 = u / wcols;
        const int strip = (int)(r0 % strips), k = (int)(r0 / strips);
        if (lane == 0) unext[u] = 0;                                        // the buffer sub-step t + 1 will set
        if (up1) {
            // lanes 0..8 / 9..17 look at the 3x3 unit neighbourhood in the flags of t - 1 / t - 2
            int f = 0;
            if (lane < 18) {
                const int q = lane % 9, sx = wx + q % 3 - 1, sy = strip + q / 3 - 1;
                if (sx >= 0 && sx < wcols && sy >= 0 && sy < strips) f = __ldcg((lane < 9 ? up1 : up2) + ((size_t)k * strips + sy) * wcols + sx);
            }
            if (!__any_sync(0xffffffffu, f != 0)) continue;
        }
        const int c = wx * 32 + lane;
        const bool active = c < ww;
        const int y0 = strip * TH_ROWS, y1 = min(h, y0 + TH_ROWS);
        const u32 *S = src + (size_t)k * plane;
        u32 *D = dst + (size_t)k * plane;
        // a row as (left, own, right) words; the neighbours' words come from the neighbouring lanes.  The loads run two
        // rows ahead of the row being decided (L2 latency), the shuffles one row ahead.
        struct Raw { u32 m, e; };                                           // own word; lanes 0 / 31: the word beyond the warp
        auto ld = [&](const int y) {
            Raw r = {0u, 0u};
            if (y >= 0 && y < h) {
                if (active) r.m = __ldcg(S + (size_t)y * ws + c);
                if (lane == 0 && c > 0 && c - 1 < ww) r.e = __ldcg(S + (size_t)y * ws + c - 1);
                if (lane == 31 && c + 1 < ww) r.e = __ldcg(S + (size_t)y * ws + c + 1);
            }
            return r;
        };
        auto mk = [&](const Raw raw, u32 &l, u32 &m, u32 &r) {
            m = raw.m;
            l = __shfl_up_sync(0xffffffffu, m, 1);
            r = __shfl_down_sync(0xffffffffu, m, 1);
            if (lane == 0) l = raw.e;
            if (lane == 31) r = raw.e;
        };
        u32 ul, um, ur, ml, mm, mr, dl, dm, dr;
        mk(ld(y0 - 1), ul, um, ur);
        mk(ld(y0), ml, mm, mr);
        Raw nxt = ld(y0 + 1);
        int cnt = 0;
        for (int y = y0; y < y1; y++) {
            const Raw nn = ld(y + 2);
            mk(nxt, dl, dm, dr);
            nxt = nn;
            u32 del = 0u;
            if (mm) del = thin_delete_mask<STEP>(ul, um, ur, ml, mm, mr, dl, dm, dr);
            if (active) D[(size_t)y * ws + c] = mm & ~del;
            cnt += __popc(del);
            ul = ml; um = mm; ur = mr; ml = dl; mm = dm; mr = dr;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
        if (lane == 0 && cnt) { atomicAdd(removed_it + (size_t)k * max_iter, cnt); *chg = 1; ucur[u] = 1; }
    }
}

__global__ void __launch_bounds__(256) fk_thin(u32 *__restrict__ A, u32 *__restrict__ B, int ws, size_t plane, int h, int w, int K, int max_iter,
                                               int *__restrict__ removed, int *flags /* [0] iterations run, [1..3] rotating changed flags */,
                                               u8 *__restrict__ unit_flags /* 4 x units, zeroed */, size_t units, int unit_rows)
{
    cg::grid_group grid = cg::this_grid();
    const int ww = (w + 31) >> 5;
    for (int it = 0; it < max_iter; it++) {
        volatile int *chg = flags + 1 + (it % 3);
        // unit flags: four buffers rotate over the sub-steps t (written at t, read at t + 1 and t + 2, cleared at t + 3)
        const int t1 = 2 * it, t2 = 2 * it + 1;
        auto ub = [&](int t) { return unit_flags + (size_t)(t & 3) * units; };
        thin_substep<1>(A, B, ws, plane, h, ww, K, removed + it, max_iter, chg, it > 0 ? ub(t1 - 1) : nullptr, ub(t1 - 2), ub(t1), ub(t1 + 1), unit_rows);
        __threadfence();
        grid.sync();
        thin_substep<2>(B, A, ws, plane, h, ww, K, removed + it, max_iter, chg, it > 0 ? ub(t2 - 1) : nullptr, ub(t2 - 2), ub(t2), ub(t2 + 1), unit_rows);
        __threadfence();
        grid.sync();
        const int c = *chg;
        if (blockIdx.x == 0 && threadIdx.x == 0) { flags[0] = it + 1; flags[1 + ((it + 2) % 3)] = 0; }
        if (!c) break;
    }
}

// planes of u8 (> 0 = foreground) -> skeleton planes {0,255}; h_removed (K * max_iter ints, may be NULL) and h_iters (K ints,
// may be NULL: iterations the reference would have run on that plane) are filled after a stream synchronisation.
// packed: 0 = byte planes in and out; 1 / 2 = planes of 1 bit per pixel in the caller's layout (LSB- / MSB-first), pitches in bytes
int fast_thin(omni_ctx *ctx, const u8 *d_in, int K, int h, int w, size_t in_plane, size_t in_pitch, int max_iter,
              u8 *d_out, size_t out_plane, size_t out_pitch, int32_t *h_removed, int32_t *h_iters, cudaStream_t st, int packed)
{
    BitGeom g = make_geom(h, w);
    u32 *bpp[2];
    FK_TRY(bit_planes(ctx, g, K, 2, bpp));
    int al = plane_align(d_out, out_plane, out_pitch);
    if (max_iter < 0) max_iter = 0;
    const size_t n_rem = (size_t)K * (max_iter > 0 ? max_iter : 1);
    if (ctx->thin_blocks == 0) {
        int per_sm = 0;
        OMNI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fk_thin, 256, 0));
        if (per_sm < 1) { omni_set_error("thinning kernel cannot be made resident"); return OMNI_ERR_CUDA; }
        ctx->thin_blocks = per_sm * (ctx->sm_count > 0 ? ctx->sm_count : 1);
    }
    // rows per unit (a warp walks a unit's rows + 2 halo rows in sequence): the height that minimises the longest chain of a
    // full sweep, ceil(units / resident warps) * (rows + 2)
    int unit_rows = 16;
    {
        const long long warps = (long long)ctx->thin_blocks * 8, cols = (g.ww + 31) / 32;
        long long best = -1;
        for (int tr = 6; tr <= 32; tr++) {
            const long long u = (long long)K * ((h + tr - 1) / tr) * cols;
            const long long cost = ((u + warps - 1) / warps) * (tr + 2);
            if (best < 0 || cost < best) { best = cost; unit_rows = tr; }
        }
    }
    size_t units = (size_t)K * ((h + unit_rows - 1) / unit_rows) * ((g.ww + 31) / 32);
    FK_TRY(omni_ws_reserve(ctx, 6, n_rem * sizeof(int) + 4 * units));
    int *d_removed = (int *)ctx->ws[6];
    u8 *d_unit = (u8 *)(d_removed + n_rem);
    OMNI_CUDA(cudaMemsetAsync(d_removed, 0, n_rem * sizeof(int) + 4 * units, st));
    // the thinning kernel has its own flag block (d_flags[32..39]): d_flags[0] keeps the pass count of the last hysteresis
    OMNI_CUDA(cudaMemsetAsync(ctx->d_flags + 32, 0, 8 * sizeof(int), st));
    OMNI_CUDA(cudaMemsetAsync(ctx->d_flags + 8, 0, sizeof(int), st));
    if (packed) {
        OMNI_LAUNCH(ctx, st, "unpack_planes", launch_unpack_planes(d_in, in_plane, in_pitch, packed == 2, K, h, w, bpp[0], g.ws, g.plane,
                                                                   persist_blocks(ctx, 8), st));
    } else {
        KScope ks(ctx, "bytes_to_bits", st);
        fk_bytes_to_bits<false><<<dim3(persist_blocks(ctx, 2), K), 256, 0, st>>>(d_in, in_plane, in_pitch, h, w, bpp[0], g.ws, g.plane, ctx->d_flags + 8);
        OMNI_CUDA(cudaGetLastError());
    }
    if (max_iter > 0) {
        // no more CTAs than warp units (8 warps per CTA): barriers get cheaper on small inputs
        int blocks = (int)std::min<long long>(ctx->thin_blocks, ((long long)units + 7) / 8);
        if (blocks < 1) blocks = 1;
        int ws = g.ws;
        size_t plane = g.plane;
        int *flags = ctx->d_flags + 32;
        void *args[] = {&bpp[0], &bpp[1], &ws, &plane, &h, &w, &K, &max_iter, &d_removed, &flags, &d_unit, &units, &unit_rows};
        OMNI_LAUNCH(ctx, st, "thin_zhangsuen", cudaLaunchCooperativeKernel((const void *)fk_thin, dim3(blocks), dim3(256), args, 0, st));
    }
    if (packed) {
        OMNI_LAUNCH(ctx, st, "pack_planes", launch_pack_planes(bpp[0], g.ws, g.plane, K, h, w, d_out, out_plane, out_pitch, packed == 2,
                                                               persist_blocks(ctx, 8), st));
    } else {
        KScope ks(ctx, "expand_bits", st);
        fk_expand_bits<<<dim3(persist_blocks(ctx, 4), K), 256, 0, st>>>(bpp[0], g.ws, g.plane, h, w, d_out, out_plane, out_pitch, al);
        OMNI_CUDA(cudaGetLastError());
    }
    if (h_removed || h_iters) {
        std::vector<int> rem(n_rem, 0);
        if (max_iter > 0) OMNI_CUDA(cudaMemcpyAsync(rem.data(), d_removed, n_rem * sizeof(int), cudaMemcpyDeviceToHost, st));
        OMNI_CUDA(cudaStreamSynchronize(st));
        for (int k = 0; k < K; k++) {
            int it = 0;
            while (it < max_iter) { it++; if (rem[(size_t)k * max_iter + it - 1] == 0) break; }   // 04:50-94: stops after the first empty iteration
            if (h_iters) h_iters[k] = it;
            if (h_removed)
                for (int i = 0; i < max_iter; i++) h_removed[(size_t)k * max_iter + i] = i < it ? rem[(size_t)k * max_iter + i] : 0;
        }
    }
    return OMNI_OK;
}


// ------------------------------------------------------------------------------------------------
// stage 02, legacy swatch mode (02_color_extract.py:82-109; SURVEY 8a row 5).  Per name the swatch is tried as RGB
// (reversed into BGR) and as-is: cv2.inRange with the clipped +-tol box, the candidate with more non-zeros wins
// (>= favours the reversed one), RECT-3 open/close.  One pass over the image fills both candidate bit-plane sets
// and their non-zero counts; the chosen planes go through the RECT open/close morphology kernel -> mask bytes.
// ------------------------------------------------------------------------------------------------
struct SwatchBoxes { u8 lo[2][OMNI_MAX_K][3], hi[2][OMNI_MAX_K][3]; int K; };

__global__ void __launch_bounds__(256) fk_inrange_bits(const u8 *__restrict__ px, int h, int w, size_t pitch, const __grid_constant__ SwatchBoxes B,
                                                       u32 *__restrict__ bits0, u32 *__restrict__ bits1, int ws, size_t plane,
                                                       unsigned long long *__restrict__ counts /* [2][OMNI_MAX_K] */)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long total = (long long)h * ws;
    unsigned long long cnt0 = 0, cnt1 = 0;                     // lane p: non-zeros of plane p of set 0 / 1
    for (long long u = (long long)blockIdx.x * 8 + warp; u < total; u += (long long)gridDim.x * 8) {
        const int y = (int)(u / ws), c = (int)(u - (long long)y * ws);
        const int x = c * 32 + lane;
        int v0 = -1, v1 = -1, v2 = -1;                         // outside the image: in no box
        if (x < w) {
            const u8 *p = px + (size_t)y * pitch + 3 * (size_t)x;
            v0 = p[0]; v1 = p[1]; v2 = p[2];
        }
        for (int k = 0; k < B.K; k++) {
#pragma unroll
            for (int s = 0; s < 2; s++) {
                const bool in = v0 >= B.lo[s][k][0] && v0 <= B.hi[s][k][0] && v1 >= B.lo[s][k][1] && v1 <= B.hi[s][k][1] &&
                                v2 >= B.lo[s][k][2] && v2 <= B.hi[s][k][2];
                const u32 word = __ballot_sync(0xffffffffu, in);
                if (lane == 0) (s ? bits1 : bits0)[(size_t)k * plane + (size_t)y * ws + c] = word;
                if (lane == k) { if (s) cnt1 += __popc(word); else cnt0 += __popc(word); }
            }
        }
    }
    if (lane < B.K) {
        if (cnt0) atomicAdd(counts + lane, cnt0);
        if (cnt1) atomicAdd(counts + OMNI_MAX_K + lane, cnt1);
    }
}

int fast_swatch_masks(omni_ctx *ctx, const u8 *d_bgr, int h, int w, size_t pitch, const int32_t *h_colors, int K, int tol,
                      u8 *d_masks, size_t plane_stride, size_t mpitch, int32_t *h_choice, cudaStream_t st)
{
    BitGeom g = make_geom(h, w);
    u32 *bpp[3];
    FK_TRY(bit_planes(ctx, g, K, 3, bpp));
    SwatchBoxes B;
    memset(&B, 0, sizeof(B));
    B.K = K;
    for (int i = 0; i < K; i++)
        for (int d = 0; d < 3; d++) {
            const int c1 = h_colors[3 * i + 2 - d], c2 = h_colors[3 * i + d];      // reversed (RGB -> BGR) / as-is
            B.lo[0][i][d] = (u8)std::max(0, c1 - tol); B.hi[0][i][d] = (u8)std::min(255, c1 + tol);
            B.lo[1][i][d] = (u8)std::max(0, c2 - tol); B.hi[1][i][d] = (u8)std::min(255, c2 + tol);
        }
    OMNI_CUDA(cudaMemsetAsync(ctx->d_counts, 0, 2 * OMNI_MAX_K * sizeof(unsigned long long), st));
    {
        KScope ks(ctx, "inrange_bits", st);
        fk_inrange_bits<<<persist_blocks(ctx, 8), 256, 0, st>>>(d_bgr, h, w, pitch, B, bpp[0], bpp[1], g.ws, g.plane, ctx->d_counts);
        OMNI_CUDA(cudaGetLastError());
    }
    OMNI_CUDA(cudaMemcpyAsync(ctx->h_counts, ctx->d_counts, 2 * OMNI_MAX_K * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    OMNI_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < K; i++) {
        const int pick = ctx->h_counts[i] >= ctx->h_counts[OMNI_MAX_K + i] ? 0 : 1;               // nz1 >= nz2 -> m1 (02:100-101)
        if (h_choice) h_choice[i] = pick;
        OMNI_CUDA(cudaMemcpyAsync(bpp[2] + (size_t)i * g.plane, bpp[pick] + (size_t)i * g.plane, g.plane * sizeof(u32),
                                  cudaMemcpyDeviceToDevice, st));
    }
    OMNI_LAUNCH(ctx, st, "morph_bits", launch_morph(true, 0, bpp[2], nullptr, g, K, d_masks, plane_stride, mpitch, st));
    return OMNI_OK;
}
