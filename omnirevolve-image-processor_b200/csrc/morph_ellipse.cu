// morph_ellipse.cu -- stage-03 ELLIPSE erode / dilate of any size on bit-planes (03_edge_detect.py:23-30): the
// edge_morph_kernel / iteration counts that fk_morph's fixed chains (fast_kernels.cu) do not cover, i.e. morph_k 2 and 4..255,
// and 3 with more than one open or close iteration.
//
// The element is a stack of rows (omni_build_se): row i, dy = i - k/2, covers dx in [x0[i], x1[i]] -- asymmetric for even k.
// cv2 does not reflect the element, so
//     erode:  out(x, y) = AND_i AND_{dx = x0[i]..x1[i]} in(x + dx, y + dy_i)
//     dilate: the same with OR, same offsets.
// The horizontal term of one row for the 32 pixels of an output word is a span of L = x1 - x0 + 1 pixels: pieces of at most
// 32 pixels, each a 64-bit window reduced by shift-and-AND doubling in ceil(log2 len) steps.  An output word costs
// sum_i ceil(L_i / 32) pieces, about k * log2(k) operations for k <= 255 (L / 32 <= 8 <= log2 L there).
//
// A CTA is one plane and EM_TW words x tr rows of output.  The input rows [y0 - k/2, y1 + (k-1) - k/2) with ceil((k/2) / 32)
// halo words on each side (two more on the right for the last window) are staged in shared memory first.  Pixels outside the
// image are staged as the identity of the operation (1 for erosion, 0 for dilation: cv2 ignores them), so the inner loop has
// no border test.  A warp is one output row: its lanes read 32 consecutive staged words (no bank conflicts) and loop over the
// same rows and pieces (no divergence).
#include "fast_kernels.cuh"
#include "fast_device.cuh"

#define EM_TW 32              // output words per CTA row (1024 pixels) = one warp
#define EM_THREADS 256
#define EM_TR 64              // output rows per CTA (the staged halo is k - 1 rows)
#define EM_SMEM_MAX (160 << 10)

// AND (erode) / OR (dilate) over the `len` pixels p + j .. p + 31 + j, j < len, of a staged row: bit b = pixel p + b.  len in [1, 32].
template <bool DILATE>
__device__ __forceinline__ u32 em_piece(const u32 *row, int p, int len)
{
    const int wi = p >> 5, b = p & 31;
    const u32 a0 = row[wi], a1 = row[wi + 1], a2 = row[wi + 2];
    u64 v = (u64)__funnelshift_r(a0, a1, b) | ((u64)__funnelshift_r(a1, a2, b) << 32);
    int m = 1;                                          // v bit j = reduction of window bits j .. j + m - 1 (valid for j + m <= 64)
    for (; 2 * m <= len; m <<= 1) v = DILATE ? (v | (v >> m)) : (v & (v >> m));
    if (m < len) v = DILATE ? (v | (v >> (len - m))) : (v & (v >> (len - m)));
    return (u32)v;
}

template <bool DILATE>
__global__ void __launch_bounds__(EM_THREADS) fk_ellipse_morph(const u32 *__restrict__ in, u32 *__restrict__ out, int ws, size_t plane,
                                                              int h, int w, int tr, int hw, const __grid_constant__ MorphSE se)
{
    extern __shared__ u32 s_rows[];
    const int k = se.k, a = k >> 1;
    const int ww = (w + 31) >> 5;
    const int c0 = blockIdx.x * EM_TW, y0 = blockIdx.y * tr, y1 = min(h, y0 + tr);
    const int sw = EM_TW + 2 * hw + 2;                  // staged words per row: staged word j = image word c0 - hw + j
    const int r0 = y0 - a, nr = (y1 - y0) + k - 1;     // staged rows [r0, r0 + nr)
    const u32 ident = DILATE ? 0u : 0xffffffffu;
    const u32 *src = in + (size_t)blockIdx.z * plane;
    for (int i = threadIdx.x; i < nr * sw; i += blockDim.x) {
        const int rr = i / sw, cc = i - rr * sw;
        const int y = r0 + rr, c = c0 - hw + cc;
        u32 v = ident;
        if (y >= 0 && y < h && c >= 0 && c < ww) {
            const u32 valid = range_mask(32 * c, w);
            v = __ldg(src + (size_t)y * ws + c);
            v = DILATE ? (v & valid) : (v | ~valid);
        }
        s_rows[i] = v;
    }
    __syncthreads();
    const int tw = min(EM_TW, ww - c0);
    u32 *dst = out + (size_t)blockIdx.z * plane;
    for (int o = threadIdx.x; o < (y1 - y0) * EM_TW; o += blockDim.x) {
        const int oy = o / EM_TW, ox = o - oy * EM_TW;
        if (ox >= tw) continue;
        u32 acc = ident;
        const int p_base = 32 * (ox + hw);
        for (int i = 0; i < k; i++) {                   // staged row oy + i = image row y0 + oy + (i - a)
            const u32 *row = s_rows + (oy + i) * sw;
            int p = p_base + se.x0[i], len = se.x1[i] - se.x0[i] + 1;
            for (; len > 32; len -= 32, p += 32) acc = DILATE ? (acc | em_piece<true>(row, p, 32)) : (acc & em_piece<false>(row, p, 32));
            acc = DILATE ? (acc | em_piece<true>(row, p, len)) : (acc & em_piece<false>(row, p, len));
        }
        const int c = c0 + ox;
        dst[(size_t)(y0 + oy) * ws + c] = acc & range_mask(32 * c, w);
    }
}

static cudaError_t launch_ellipse_step(const u32 *in, u32 *out, const BitGeom &g, int K, const MorphSE &se, bool dilate, cudaStream_t st)
{
    const int hw = ((se.k >> 1) + 31) >> 5;
    const int sw = EM_TW + 2 * hw + 2;
    int tr = EM_TR;
    while (tr > 8 && (size_t)(tr + se.k - 1) * sw * sizeof(u32) > EM_SMEM_MAX) tr >>= 1;
    const size_t smem = (size_t)(tr + se.k - 1) * sw * sizeof(u32);
    if (smem > EM_SMEM_MAX) return cudaErrorInvalidValue;
    const dim3 grid((g.ww + EM_TW - 1) / EM_TW, (g.h + tr - 1) / tr, K);
    if (smem > (48 << 10)) {                            // above the default limit: opt in (large elements only)
        cudaError_t e = cudaFuncSetAttribute(dilate ? fk_ellipse_morph<true> : fk_ellipse_morph<false>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, EM_SMEM_MAX);
        if (e != cudaSuccess) return e;
    }
    if (dilate) fk_ellipse_morph<true><<<grid, EM_THREADS, smem, st>>>(in, out, g.ws, g.plane, g.h, g.w, tr, hw, se);
    else fk_ellipse_morph<false><<<grid, EM_THREADS, smem, st>>>(in, out, g.ws, g.plane, g.h, g.w, tr, hw, se);
    return cudaGetLastError();
}

// open^oi then close^ci with the ELLIPSE(morph_k) element: erode^oi dilate^oi dilate^ci erode^ci (cv2 loops the iterations of a
// non-rectangular element).  The planes start in `a`; every step writes the other buffer.  *result: the planes holding the end.
int ellipse_morph_bits(omni_ctx *ctx, const omni_edge_params *prm, const BitGeom &g, int K, u32 *a, u32 *b, const u32 **result,
                       cudaStream_t st)
{
    MorphSE se;
    omni_build_se(1, prm->morph_k, &se);
    const long long oi = prm->open_iters > 0 ? prm->open_iters : 0, ci = prm->close_iters > 0 ? prm->close_iters : 0;
    const long long n_steps = 2 * (oi + ci);
    u32 *cur = a, *nxt = b;
    for (long long i = 0; i < n_steps; i++) {
        const bool dilate = i >= oi && i < 2 * oi + ci;
        OMNI_LAUNCH(ctx, st, "morph_ellipse_bits", launch_ellipse_step(cur, nxt, g, K, se, dilate, st));
        u32 *t = cur; cur = nxt; nxt = t;
    }
    *result = cur;
    return OMNI_OK;
}
