// generic_kernels.cu -- the GENERIC CUDA implementation of every op on the stage 01-03 path.
//
// One straightforward kernel per library call the reference makes; byte-per-pixel planes, any u8
// content, every supported parameter value (morph element up to 7x7, blur up to 31, any iteration
// counts).  The fast bit-plane kernels (fast_kernels.cu) take over for the parameter ranges the
// pipeline actually uses; these remain the path for everything else and serve as an independent
// on-device cross-check in the tests.  Arithmetic follows SURVEY.md Appendix A; reference call
// sites are cited per kernel (paths relative to /root/reference/image_processor/).
#include "omni_internal.cuh"
#include "omni_tables.inc"

__constant__ u16 c_lab_gamma[256];
__constant__ u16 c_lab_cbrt[2041];
static bool g_tables_uploaded[64] = {false};

static cudaError_t ensure_tables()
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 64 && g_tables_uploaded[dev]) return cudaSuccess;
    e = cudaMemcpyToSymbol(c_lab_gamma, OMNI_LAB_GAMMA, sizeof(OMNI_LAB_GAMMA));
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbol(c_lab_cbrt, OMNI_LAB_CBRT, sizeof(OMNI_LAB_CBRT));
    if (e != cudaSuccess) return e;
    if (dev < 64) g_tables_uploaded[dev] = true;
    return cudaSuccess;
}

int omni_gauss_weights(int k, BlurParams *bp)
{
    if (k < OMNI_GAUSS_KMIN || k > OMNI_GAUSS_KMAX || !(k & 1)) return -1;
    const unsigned short *w = OMNI_GAUSS_W + OMNI_GAUSS_OFFS[(k - 3) / 2];
    for (int i = 0; i < k; i++) bp->w[i] = w[i];
    bp->k = k;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// 01_resize.py:20  cv2.resize(..., INTER_AREA), shrink only (SURVEY A.1)
// ------------------------------------------------------------------------------------------------
__global__ void k_resize_2x(const u8 *__restrict__ src, size_t spitch, u8 *__restrict__ dst, int dh, int dw, size_t dpitch)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= dw || y >= dh) return;
    const u8 *r0 = src + (size_t)(2 * y) * spitch + 6 * x, *r1 = r0 + spitch;
    u8 *o = dst + (size_t)y * dpitch + 3 * x;
#pragma unroll
    for (int c = 0; c < 3; c++) o[c] = (u8)((r0[c] + r0[c + 3] + r1[c] + r1[c + 3] + 2) >> 2);
}

__global__ void k_resize_int(const u8 *__restrict__ src, size_t spitch, u8 *__restrict__ dst, int dh, int dw, size_t dpitch,
                             int fx, int fy, float inv_area)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= dw || y >= dh) return;
    int s0 = 0, s1 = 0, s2 = 0;
    for (int j = 0; j < fy; j++) {
        const u8 *r = src + (size_t)(y * fy + j) * spitch + 3 * (x * fx);
        for (int i = 0; i < fx; i++) { s0 += r[3 * i]; s1 += r[3 * i + 1]; s2 += r[3 * i + 2]; }
    }
    u8 *o = dst + (size_t)y * dpitch + 3 * x;
    o[0] = (u8)min(255, max(0, __float2int_rn(__fmul_rn((float)s0, inv_area))));
    o[1] = (u8)min(255, max(0, __float2int_rn(__fmul_rn((float)s1, inv_area))));
    o[2] = (u8)min(255, max(0, __float2int_rn(__fmul_rn((float)s2, inv_area))));
}

// fractional ratios: OpenCV's ResizeArea_ order -- per source row a horizontal weighted sum (f32,
// sequential), then the vertical accumulation sum = beta*buf (first row) / sum += beta*buf.
__global__ void k_resize_frac(const u8 *__restrict__ src, size_t spitch, u8 *__restrict__ dst, int dh, int dw, size_t dpitch,
                              ResizeTabDev t)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= dw || y >= dh) return;
    int xb = t.xofs[x], xe = t.xofs[x + 1], yb = t.yofs[y], ye = t.yofs[y + 1];
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    for (int j = yb; j < ye; j++) {
        const u8 *r = src + (size_t)t.ysi[j] * spitch;
        float beta = t.yal[j];
        float b0 = 0.f, b1 = 0.f, b2 = 0.f;
        for (int k = xb; k < xe; k++) {
            const u8 *p = r + 3 * t.xsi[k];
            float a = t.xal[k];
            b0 = __fadd_rn(b0, __fmul_rn((float)p[0], a));
            b1 = __fadd_rn(b1, __fmul_rn((float)p[1], a));
            b2 = __fadd_rn(b2, __fmul_rn((float)p[2], a));
        }
        if (j == yb) { s0 = __fmul_rn(beta, b0); s1 = __fmul_rn(beta, b1); s2 = __fmul_rn(beta, b2); }
        else {
            s0 = __fadd_rn(s0, __fmul_rn(beta, b0)); s1 = __fadd_rn(s1, __fmul_rn(beta, b1)); s2 = __fadd_rn(s2, __fmul_rn(beta, b2));
        }
    }
    u8 *o = dst + (size_t)y * dpitch + 3 * x;
    o[0] = (u8)min(255, max(0, __float2int_rn(s0)));
    o[1] = (u8)min(255, max(0, __float2int_rn(s1)));
    o[2] = (u8)min(255, max(0, __float2int_rn(s2)));
}

cudaError_t g_resize_area(const u8 *src, int sh, int sw, size_t spitch, u8 *dst, int dh, int dw, size_t dpitch,
                          const ResizeTabDev *tab, cudaStream_t st)
{
    dim3 b(32, 8), g((dw + 31) / 32, (dh + 7) / 8);
    if (tab) k_resize_frac<<<g, b, 0, st>>>(src, spitch, dst, dh, dw, dpitch, *tab);
    else {
        int fx = sw / dw, fy = sh / dh;
        if (fx == 2 && fy == 2) k_resize_2x<<<g, b, 0, st>>>(src, spitch, dst, dh, dw, dpitch);
        else k_resize_int<<<g, b, 0, st>>>(src, spitch, dst, dh, dw, dpitch, fx, fy, 1.f / (float)(fx * fy));
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// 02_color_extract.py:35 (BGR2LAB) + :53-55 (nearest centre, f32)  /  process_colors.py:69-77
// ------------------------------------------------------------------------------------------------
template <int MODE_LAB>
__global__ void k_assign(const u8 *__restrict__ px, int h, int w, size_t pitch, const __grid_constant__ AssignParams P,
                         u8 *__restrict__ labels, size_t lpitch)
{
    __shared__ u16 s_gam[256];
    __shared__ u16 s_cbrt[2041];
    if (MODE_LAB) {
        for (int i = threadIdx.y * blockDim.x + threadIdx.x; i < 2041; i += blockDim.x * blockDim.y) {
            s_cbrt[i] = c_lab_cbrt[i];
            if (i < 256) s_gam[i] = c_lab_gamma[i];
        }
        __syncthreads();
    }
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const u8 *p = px + (size_t)y * pitch + 3 * x;
    int v0 = p[0], v1 = p[1], v2 = p[2];
    int best = 0;
    if (MODE_LAB) {
        int L, a, b;
        bgr2lab_px(s_gam, s_cbrt, v0, v1, v2, L, a, b);
        float f0 = (float)L, f1 = (float)a, f2 = (float)b, bd = 0.f;
        for (int k = 0; k < P.K; k++) {
            float d0 = __fsub_rn(f0, P.c[3 * k]), d1 = __fsub_rn(f1, P.c[3 * k + 1]), d2 = __fsub_rn(f2, P.c[3 * k + 2]);
            float d = __fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2, d2));
            if (k == 0 || d < bd) { bd = d; best = k; }
        }
    } else {
        int bd = 0;
        for (int k = 0; k < P.K; k++) {
            int d0 = v0 - P.pal[3 * k], d1 = v1 - P.pal[3 * k + 1], d2 = v2 - P.pal[3 * k + 2];
            int d = (int)(short)(d0 * d0) + (int)(short)(d1 * d1) + (int)(short)(d2 * d2);
            if (k == 0 || d < bd) { bd = d; best = k; }
        }
    }
    labels[(size_t)y * lpitch + x] = P.lut[best];
}

cudaError_t g_assign(const u8 *px, int h, int w, size_t pitch, const AssignParams &P, int mode_lab,
                     u8 *labels, size_t lpitch, cudaStream_t st)
{
    cudaError_t e = ensure_tables();
    if (e != cudaSuccess) return e;
    dim3 b(64, 4), g((w + 63) / 64, (h + 3) / 4);
    if (mode_lab) k_assign<1><<<g, b, 0, st>>>(px, h, w, pitch, P, labels, lpitch);
    else k_assign<0><<<g, b, 0, st>>>(px, h, w, pitch, P, labels, lpitch);
    return cudaGetLastError();
}

// 02_color_extract.py:150  (labels == k) * 255
__global__ void k_onehot(const u8 *__restrict__ labels, int h, int w, size_t lpitch, int K, u8 *__restrict__ planes,
                         size_t plane_stride, size_t pitch)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    int l = labels[(size_t)y * lpitch + x];
    for (int k = 0; k < K; k++) planes[k * plane_stride + (size_t)y * pitch + x] = (l == k) ? 255 : 0;
}

cudaError_t g_onehot(const u8 *labels, int h, int w, size_t lpitch, int K, u8 *planes, size_t plane_stride,
                     size_t pitch, cudaStream_t st)
{
    dim3 b(64, 4), g((w + 63) / 64, (h + 3) / 4);
    k_onehot<<<g, b, 0, st>>>(labels, h, w, lpitch, K, planes, plane_stride, pitch);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// cv2.erode / cv2.dilate, one iteration (02:151-154, 03:24-30); outside pixels ignored (SURVEY A.0)
// ------------------------------------------------------------------------------------------------
__global__ void k_morph(const u8 *__restrict__ src, size_t s_plane, size_t spitch, u8 *__restrict__ dst, size_t d_plane,
                        size_t dpitch, int h, int w, const __grid_constant__ MorphSE se, int is_dilate)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const u8 *s = src + blockIdx.z * s_plane;
    int v = is_dilate ? 0 : 255;
    for (int i = 0; i < se.k; i++) {                       // row i of the element: dy = i - k/2, dx in [x0[i], x1[i]]
        const int yy = y + i - se.k / 2;
        if (yy < 0 || yy >= h) continue;
        const u8 *row = s + (size_t)yy * spitch;
        const int xa = max(0, x + se.x0[i]), xb = min(w - 1, x + se.x1[i]);
        for (int xx = xa; xx <= xb; xx++) {
            const int p = row[xx];
            v = is_dilate ? max(v, p) : min(v, p);
        }
    }
    dst[blockIdx.z * d_plane + (size_t)y * dpitch + x] = (u8)v;
}

cudaError_t g_morph(const u8 *src, size_t s_plane, size_t spitch, u8 *dst, size_t d_plane, size_t dpitch,
                    int K, int h, int w, const MorphSE &se, int is_dilate, cudaStream_t st)
{
    dim3 b(64, 4), g((w + 63) / 64, (h + 3) / 4, K);
    k_morph<<<g, b, 0, st>>>(src, s_plane, spitch, dst, d_plane, dpitch, h, w, se, is_dilate);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// 03_edge_detect.py:33  cv2.GaussianBlur(u8,(k,k),0): separable 8.8 fixed point, REFLECT_101 (A.2)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect101(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * (len - 1) - p;
    return p;
}

#define BL_TW 64
#define BL_TH 32
__global__ void __launch_bounds__(256) k_blur(const u8 *__restrict__ src, size_t s_plane, size_t spitch, u8 *__restrict__ dst,
                                              size_t d_plane, size_t dpitch, int h, int w, const __grid_constant__ BlurParams bp)
{
    extern __shared__ u8 smem_raw[];
    const int r = bp.k / 2, SW = BL_TW + 2 * r, SH = BL_TH + 2 * r;
    u8 *s_in = smem_raw;                                        // SH x SW
    u16 *s_h = (u16 *)(smem_raw + ((SH * SW + 15) & ~15));       // SH x BL_TW
    const u8 *s = src + blockIdx.z * s_plane;
    int x0 = blockIdx.x * BL_TW, y0 = blockIdx.y * BL_TH, tid = threadIdx.x;
    for (int i = tid; i < SH * SW; i += 256) {
        int ly = i / SW, lx = i - ly * SW;
        int gy = reflect101(min(y0 + ly - r, h - 1 + r), h), gx = reflect101(min(x0 + lx - r, w - 1 + r), w);
        s_in[i] = s[(size_t)gy * spitch + gx];
    }
    __syncthreads();
    for (int i = tid; i < SH * BL_TW; i += 256) {
        int ly = i / BL_TW, lx = i - ly * BL_TW;
        u32 acc = 0;
        for (int t = 0; t < bp.k; t++) acc += (u32)bp.w[t] * s_in[ly * SW + lx + t];
        s_h[i] = (u16)acc;
    }
    __syncthreads();
    for (int i = tid; i < BL_TH * BL_TW; i += 256) {
        int ly = i / BL_TW, lx = i - ly * BL_TW;
        int gx = x0 + lx, gy = y0 + ly;
        if (gx >= w || gy >= h) continue;
        u32 acc = 0;
        for (int t = 0; t < bp.k; t++) acc += (u32)bp.w[t] * s_h[(ly + t) * BL_TW + lx];
        dst[blockIdx.z * d_plane + (size_t)gy * dpitch + gx] = (u8)((acc + 32768u) >> 16);
    }
}

cudaError_t g_blur(const u8 *src, size_t s_plane, size_t spitch, u8 *dst, size_t d_plane, size_t dpitch,
                   int K, int h, int w, const BlurParams &bp, cudaStream_t st)
{
    int r = bp.k / 2, SW = BL_TW + 2 * r, SH = BL_TH + 2 * r;
    size_t smem = ((SH * SW + 15) & ~15) + (size_t)SH * BL_TW * 2;
    dim3 g((w + BL_TW - 1) / BL_TW, (h + BL_TH - 1) / BL_TH, K);
    k_blur<<<g, 256, smem, st>>>(src, s_plane, spitch, dst, d_plane, dpitch, h, w, bp);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// 03_edge_detect.py:34  cv2.Canny (aperture 3, L1): Sobel (REPLICATE), magnitude 0 outside, NMS (A.5)
// state out: 0 = not a candidate, 1 = weak candidate, 2 = strong
// ------------------------------------------------------------------------------------------------
#define CN_TW 64
#define CN_TH 32
__global__ void __launch_bounds__(256) k_canny_nms(const u8 *__restrict__ src, size_t s_plane, size_t spitch, u8 *__restrict__ state,
                                                   size_t d_plane, size_t dpitch, int h, int w, int low, int high)
{
    __shared__ u8 s_in[(CN_TH + 4) * (CN_TW + 4)];
    __shared__ short s_mag[(CN_TH + 2) * (CN_TW + 2)];
    __shared__ short s_dx[(CN_TH + 2) * (CN_TW + 2)];
    __shared__ short s_dy[(CN_TH + 2) * (CN_TW + 2)];
    const u8 *s = src + blockIdx.z * s_plane;
    const int SW = CN_TW + 4, MW = CN_TW + 2;
    int x0 = blockIdx.x * CN_TW, y0 = blockIdx.y * CN_TH, tid = threadIdx.x;
    for (int i = tid; i < (CN_TH + 4) * SW; i += 256) {
        int ly = i / SW, lx = i - ly * SW;
        int gy = min(max(y0 + ly - 2, 0), h - 1), gx = min(max(x0 + lx - 2, 0), w - 1);
        s_in[i] = s[(size_t)gy * spitch + gx];
    }
    __syncthreads();
    for (int i = tid; i < (CN_TH + 2) * MW; i += 256) {
        int ly = i / MW, lx = i - ly * MW;
        int gy = y0 + ly - 1, gx = x0 + lx - 1;
        const u8 *c = s_in + (ly + 1) * SW + (lx + 1);
        int dx = (c[-SW + 1] + 2 * c[1] + c[SW + 1]) - (c[-SW - 1] + 2 * c[-1] + c[SW - 1]);
        int dy = (c[SW - 1] + 2 * c[SW] + c[SW + 1]) - (c[-SW - 1] + 2 * c[-SW] + c[-SW + 1]);
        bool inside = gy >= 0 && gy < h && gx >= 0 && gx < w;
        s_dx[i] = (short)dx; s_dy[i] = (short)dy;
        s_mag[i] = inside ? (short)(abs(dx) + abs(dy)) : (short)0;
    }
    __syncthreads();
    for (int i = tid; i < CN_TH * CN_TW; i += 256) {
        int ly = i / CN_TW, lx = i - ly * CN_TW;
        int gx = x0 + lx, gy = y0 + ly;
        if (gx >= w || gy >= h) continue;
        int mi = (ly + 1) * MW + (lx + 1);
        int m = s_mag[mi], out = 0;
        if (m > low) {
            int xs = s_dx[mi], ys = s_dy[mi];
            int ax = abs(xs), ay = abs(ys) << 15, tg22 = ax * 13573;
            bool ok;
            if (ay < tg22) ok = m > s_mag[mi - 1] && m >= s_mag[mi + 1];
            else {
                int tg67 = tg22 + (ax << 16);
                if (ay > tg67) ok = m > s_mag[mi - MW] && m >= s_mag[mi + MW];
                else { int sg = (xs ^ ys) < 0 ? -1 : 1; ok = m > s_mag[mi - MW - sg] && m > s_mag[mi + MW + sg]; }
            }
            if (ok) out = m > high ? 2 : 1;
        }
        state[blockIdx.z * d_plane + (size_t)gy * dpitch + gx] = (u8)out;
    }
}

cudaError_t g_canny_nms(const u8 *src, size_t s_plane, size_t spitch, u8 *state, size_t d_plane, size_t dpitch,
                        int K, int h, int w, int low, int high, cudaStream_t st)
{
    dim3 g((w + CN_TW - 1) / CN_TW, (h + CN_TH - 1) / CN_TH, K);
    k_canny_nms<<<g, 256, 0, st>>>(src, s_plane, spitch, state, d_plane, dpitch, h, w, low, high);
    return cudaGetLastError();
}

// Hysteresis: promote weak (1) pixels that touch a strong (2) pixel, 8-connected.  Each CTA iterates
// its 64x64 tile (+1 halo) to a local fixed point in shared memory; *d_changed is set when a tile
// changed, and the host re-launches until a whole pass changes nothing.  The result set is
// order-independent (SURVEY A.5), so racing reads of neighbouring tiles are harmless: state only
// ever moves 1 -> 2 and the final, change-free pass sees a quiescent image.
#define HY_T 64
__global__ void __launch_bounds__(256) k_hyst_pass(u8 *state, size_t plane, size_t pitch, int h, int w, int *d_changed)
{
    __shared__ u8 s[(HY_T + 2) * (HY_T + 2)];
    u8 *g = state + blockIdx.z * plane;
    const int SW = HY_T + 2;
    int x0 = blockIdx.x * HY_T, y0 = blockIdx.y * HY_T, tid = threadIdx.x;
    int has_weak = 0;
    for (int i = tid; i < SW * SW; i += 256) {
        int ly = i / SW, lx = i - ly * SW;
        int gy = y0 + ly - 1, gx = x0 + lx - 1;
        u8 v = (gy >= 0 && gy < h && gx >= 0 && gx < w) ? g[(size_t)gy * pitch + gx] : 0;
        s[i] = v;
        bool interior = ly >= 1 && ly <= HY_T && lx >= 1 && lx <= HY_T;
        has_weak |= (interior && v == 1);
    }
    if (!__syncthreads_or(has_weak)) return;
    int any_change = 0;
    for (;;) {
        int changed = 0;
        for (int i = tid; i < HY_T * HY_T; i += 256) {
            int ly = i / HY_T + 1, lx = (i & (HY_T - 1)) + 1;
            int c = ly * SW + lx;
            if (s[c] == 1) {
                int m = max(max(max(s[c - SW - 1], s[c - SW]), max(s[c - SW + 1], s[c - 1])),
                            max(max(s[c + 1], s[c + SW - 1]), max(s[c + SW], s[c + SW + 1])));
                if (m == 2) { s[c] = 2; changed = 1; }
            }
        }
        if (!__syncthreads_or(changed)) break;
        any_change = 1;
    }
    if (any_change) {
        for (int i = tid; i < HY_T * HY_T; i += 256) {
            int ly = i / HY_T + 1, lx = (i & (HY_T - 1)) + 1;
            int gy = y0 + ly - 1, gx = x0 + lx - 1;
            if (gy < h && gx < w && s[ly * SW + lx] == 2) g[(size_t)gy * pitch + gx] = 2;
        }
        if (tid == 0) atomicOr(d_changed, 1);
    }
}

cudaError_t g_hyst_pass(u8 *state, size_t plane, size_t pitch, int K, int h, int w, int *d_changed, cudaStream_t st)
{
    dim3 g((w + HY_T - 1) / HY_T, (h + HY_T - 1) / HY_T, K);
    k_hyst_pass<<<g, 256, 0, st>>>(state, plane, pitch, h, w, d_changed);
    return cudaGetLastError();
}

__global__ void k_hyst_final(u8 *state, size_t plane, size_t pitch, int h, int w)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    u8 *p = state + blockIdx.z * plane + (size_t)y * pitch + x;
    *p = (*p == 2) ? 255 : 0;
}

cudaError_t g_hyst_final(u8 *state, size_t plane, size_t pitch, int K, int h, int w, cudaStream_t st)
{
    dim3 b(64, 4), g((w + 63) / 64, (h + 3) / 4, K);
    k_hyst_final<<<g, b, 0, st>>>(state, plane, pitch, h, w);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// counts (02:144,157,168 ; 03:38) and the composite paint (03:93-106)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_count_nonzero(const u8 *__restrict__ planes, size_t plane, size_t pitch, int h, int w,
                                                       unsigned long long *d_counts)
{
    const u8 *p = planes + blockIdx.z * plane;
    unsigned cnt = 0;
    for (int y = blockIdx.y; y < h; y += gridDim.y)
        for (int x = blockIdx.x * 256 + threadIdx.x; x < w; x += gridDim.x * 256) cnt += p[(size_t)y * pitch + x] != 0;
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(d_counts + blockIdx.z, (unsigned long long)cnt);
}

cudaError_t g_count_nonzero(const u8 *planes, size_t plane, size_t pitch, int K, int h, int w,
                            unsigned long long *d_counts, cudaStream_t st)
{
    dim3 g(min(8, (w + 255) / 256), min(h, 256), K);
    k_count_nonzero<<<g, 256, 0, st>>>(planes, plane, pitch, h, w, d_counts);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) k_count_labels(const u8 *__restrict__ labels, size_t pitch, int h, int w, int K,
                                                      unsigned long long *d_counts)
{
    __shared__ unsigned s_cnt[OMNI_MAX_K];
    if (threadIdx.x < OMNI_MAX_K) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    for (int y = blockIdx.y; y < h; y += gridDim.y)
        for (int x = blockIdx.x * 256 + threadIdx.x; x < w; x += gridDim.x * 256) {
            int l = labels[(size_t)y * pitch + x];
            if (l < K) atomicAdd(&s_cnt[l], 1u);
        }
    __syncthreads();
    if (threadIdx.x < K && s_cnt[threadIdx.x]) atomicAdd(d_counts + threadIdx.x, (unsigned long long)s_cnt[threadIdx.x]);
}

cudaError_t g_count_labels(const u8 *labels, size_t pitch, int h, int w, int K, unsigned long long *d_counts,
                           cudaStream_t st)
{
    dim3 g(min(8, (w + 255) / 256), min(h, 128));
    k_count_labels<<<g, 256, 0, st>>>(labels, pitch, h, w, K, d_counts);
    return cudaGetLastError();
}

struct CompositeColors { u8 c[OMNI_MAX_K * 3]; };
__global__ void k_composite(const u8 *__restrict__ edges, size_t plane, size_t pitch, int K, int h, int w,
                            const __grid_constant__ CompositeColors col, u8 *__restrict__ canvas, size_t cpitch)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    int b = 255, g = 255, r = 255;
    for (int k = 0; k < K; k++)
        if (edges[k * plane + (size_t)y * pitch + x]) { b = col.c[3 * k]; g = col.c[3 * k + 1]; r = col.c[3 * k + 2]; }
    u8 *o = canvas + (size_t)y * cpitch + 3 * x;
    o[0] = (u8)b; o[1] = (u8)g; o[2] = (u8)r;
}

cudaError_t g_composite(const u8 *edges, size_t plane, size_t pitch, int K, int h, int w, const u8 *colors_bgr,
                        u8 *canvas, size_t cpitch, cudaStream_t st)
{
    CompositeColors col;
    for (int i = 0; i < 3 * K; i++) col.c[i] = colors_bgr[i];
    dim3 b(64, 4), g((w + 63) / 64, (h + 3) / 4);
    k_composite<<<g, b, 0, st>>>(edges, plane, pitch, K, h, w, col, canvas, cpitch);
    return cudaGetLastError();
}

// 04_find_contours.py:121-130: deg = cv2.filter2D(S, CV_8U, ones(3,3) - centre, BORDER_CONSTANT) with S = (skeleton > 0):
// the number of set 8-neighbours of EVERY pixel (outside the image counts 0); nodes: 1 where an S pixel has deg == 1
// (endpoint, :124), 2 where it has deg >= 3 (junction, :125), else 0.  The reference evaluates this per connected component on the
// component's mask; a pixel's neighbours belong to its own component, so on component pixels the global map is the same.
__global__ void k_skeleton_degree(const u8 *__restrict__ skel, size_t s_plane, size_t spitch, int h, int w, u8 *__restrict__ deg,
                                  size_t d_plane, size_t dpitch, u8 *__restrict__ nodes, size_t n_plane, size_t npitch)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, k = blockIdx.z;
    if (x >= w || y >= h) return;
    const u8 *S = skel + (size_t)k * s_plane;
    int n = 0;
#pragma unroll
    for (int dy = -1; dy <= 1; dy++) {
        const int yy = y + dy;
        if (yy < 0 || yy >= h) continue;
        const u8 *row = S + (size_t)yy * spitch;
#pragma unroll
        for (int dx = -1; dx <= 1; dx++) {
            const int xx = x + dx;
            if ((dx | dy) == 0 || xx < 0 || xx >= w) continue;
            n += __ldg(row + xx) != 0;
        }
    }
    if (deg) deg[(size_t)k * d_plane + (size_t)y * dpitch + x] = (u8)n;
    if (nodes) {
        const bool on = S[(size_t)y * spitch + x] != 0;
        nodes[(size_t)k * n_plane + (size_t)y * npitch + x] = (u8)(on ? (n == 1 ? 1 : (n >= 3 ? 2 : 0)) : 0);
    }
}

cudaError_t g_skeleton_degree(const u8 *skel, size_t s_plane, size_t spitch, int K, int h, int w, u8 *deg, size_t d_plane, size_t dpitch,
                              u8 *nodes, size_t n_plane, size_t npitch, cudaStream_t st)
{
    dim3 b(64, 4), g((w + 63) / 64, (h + 3) / 4, K);
    k_skeleton_degree<<<g, b, 0, st>>>(skel, s_plane, spitch, h, w, deg, d_plane, dpitch, nodes, n_plane, npitch);
    return cudaGetLastError();
}

cudaError_t g_copy2d_planes(const u8 *src, size_t s_plane, size_t spitch, u8 *dst, size_t d_plane, size_t dpitch,
                            int K, int h, int w, cudaStream_t st)
{
    for (int k = 0; k < K; k++) {
        cudaError_t e = cudaMemcpy2DAsync(dst + k * d_plane, dpitch, src + k * s_plane, spitch, (size_t)w, (size_t)h,
                                          cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// byte planes (non-zero = set) -> packed rows in the caller's layout, with optional per-plane non-zero counts (generic family of
// the packed entry points: whatever the byte-plane kernels produced, 8 pixels per output byte)
__global__ void __launch_bounds__(256) k_pack_bytes(const u8 *__restrict__ src, size_t s_plane, size_t spitch, int K, int h, int w,
                                                    u8 *__restrict__ dst, size_t d_plane, size_t dpitch, int msb_first,
                                                    unsigned long long *__restrict__ counts)
{
    const int rb = (w + 7) >> 3;
    const long long total = (long long)K * h * rb;
    for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < total; u += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(u % rb);
        const long long r2 = u / rb;
        const int y = (int)(r2 % h), k = (int)(r2 / h);
        const u8 *row = src + (size_t)k * s_plane + (size_t)y * spitch + 8 * j;
        unsigned v = 0;
        for (int i = 0; i < 8 && 8 * j + i < w; i++)
            if (row[i]) v |= msb_first ? (0x80u >> i) : (1u << i);
        dst[(size_t)k * d_plane + (size_t)y * dpitch + j] = (u8)v;
        if (counts && v) atomicAdd(counts + k, (unsigned long long)__popc(v));
    }
}

cudaError_t g_pack_bytes(const u8 *src, size_t s_plane, size_t spitch, int K, int h, int w, u8 *dst, size_t d_plane, size_t dpitch,
                         int msb_first, unsigned long long *counts, cudaStream_t st)
{
    const long long total = (long long)K * h * ((w + 7) >> 3);
    const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
    k_pack_bytes<<<blocks > 0 ? blocks : 1, 256, 0, st>>>(src, s_plane, spitch, K, h, w, dst, d_plane, dpitch, msb_first, counts);
    return cudaGetLastError();
}
