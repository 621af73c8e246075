// trace.cu -- stage 04 `trace_centerlines` (04_find_contours.py:101-205) for K skeleton planes at once.
//
// 1. Connected components (8-connectivity on S = skel > 0), numbered the way cv2.connectedComponentsWithStats numbers them:
//    by the first 2x2 block, in block-raster order, that holds one of their pixels (block key (y>>1) * ceil(w/2) + (x>>1); the
//    foreground pixels of one 2x2 block are always 8-connected).  Block-level union-find links every tree to its minimum block,
//    so the root of a component is its minimum block; an exclusive scan over the "is root" flags gives cv2's label minus 1.
//    Then area and bounding box per component (cv2's `stats`).
// 2. The walk of the reference, one component per CTA of one warp: the warp scans for start pixels (ballots over 32 pixels),
//    lane 0 walks.  A count pass sizes the output, a write pass fills it (the walk is deterministic, so both see the same
//    polylines).  A component whose bounding box plus a one-pixel frame fits TRACE_SMEM_CAP bytes walks in a shared-memory
//    byte map (bit 0: pixel of the component, bit 1: visited); larger ones read the skeleton plane, a visited byte plane
//    (one per layer, shared by all its large components: walks never leave their component) and row-major lists of the
//    plane's foreground pixels for the start-pixel scans.
#include "omni_internal.cuh"

#include <algorithm>
#include <limits.h>
#include <numeric>

namespace {

constexpr int TRACE_SMEM_CAP = 200 * 1024;   // largest shared-memory map of one component (B200: 227 KB per block)
constexpr int CHUNK = 1024;                  // blocks per CTA of the label scan

struct TraceComp {
    int x0, y0, x1, y1;       // bounding box, inclusive
    int area, root, npaths, pad;
    long long npts, pt_base, path_base;
};

struct TraceGeom {
    const u8 *skel;
    size_t plane_stride, pitch;
    int K, h, w, bw, nb;
    const int *parent;        // [K][nb]: root block of every foreground block, -1 for empty blocks
    u8 *visited;              // [K][h][w] (large components only)
    const int *row_off;       // [K][h + 1] offsets into row_x (large components only)
    const int *row_x;         // x of every foreground pixel, row-major per plane
    long long guard_open[OMNI_MAX_K];   // 2 * total_fg of the plane (04:165)
};

__device__ __forceinline__ u8 px(const u8 *S, size_t pitch, int h, int w, int x, int y)
{
    return (x >= 0 && y >= 0 && x < w && y < h) ? S[(size_t)y * pitch + x] : 0;
}

__device__ int find_root(const int *P, int a)
{
    int p = ((const volatile int *)P)[a];
    while (p != a) { a = p; p = ((const volatile int *)P)[a]; }
    return a;
}

// union to the minimum index: the root of every tree is its smallest block
__device__ void unite(int *P, int a, int b)
{
    for (;;) {
        a = find_root(P, a);
        b = find_root(P, b);
        if (a == b) return;
        if (a < b) { const int old = atomicMin(&P[b], a); if (old == b) return; b = old; }
        else       { const int old = atomicMin(&P[a], b); if (old == a) return; a = old; }
    }
}

__global__ void k_ccl_init(TraceGeom g, int *parent)
{
    const int B = blockIdx.x * blockDim.x + threadIdx.x, k = blockIdx.y;
    if (B >= g.nb) return;
    const u8 *S = g.skel + k * g.plane_stride;
    const int x = 2 * (B % g.bw), y = 2 * (B / g.bw);
    const bool any = px(S, g.pitch, g.h, g.w, x, y) | px(S, g.pitch, g.h, g.w, x + 1, y) | px(S, g.pitch, g.h, g.w, x, y + 1) |
                     px(S, g.pitch, g.h, g.w, x + 1, y + 1);
    parent[(size_t)k * g.nb + B] = any ? B : -1;
}

// links every block to its right, down-left, down and down-right neighbour blocks where two of their pixels touch
__global__ void k_ccl_merge(TraceGeom g, int *parent)
{
    const int B = blockIdx.x * blockDim.x + threadIdx.x, k = blockIdx.y;
    if (B >= g.nb) return;
    int *P = parent + (size_t)k * g.nb;
    if (P[B] < 0) return;
    const u8 *S = g.skel + k * g.plane_stride;
    const int x = 2 * (B % g.bw), y = 2 * (B / g.bw), bx = B % g.bw;
    auto f = [&](int xx, int yy) { return px(S, g.pitch, g.h, g.w, xx, yy) != 0; };
    const bool tr = f(x + 1, y), bl = f(x, y + 1), br = f(x + 1, y + 1);
    if (bx + 1 < g.bw && (tr || br) && (f(x + 2, y) || f(x + 2, y + 1))) unite(P, B, B + 1);
    if (B + g.bw < g.nb) {
        if ((bl || br) && (f(x, y + 2) || f(x + 1, y + 2))) unite(P, B, B + g.bw);
        if (bx + 1 < g.bw && br && f(x + 2, y + 2)) unite(P, B, B + g.bw + 1);
        if (bx > 0 && bl && f(x - 1, y + 2)) unite(P, B, B + g.bw - 1);
    }
}

__global__ void k_ccl_flatten(TraceGeom g, int *parent)
{
    const int B = blockIdx.x * blockDim.x + threadIdx.x, k = blockIdx.y;
    if (B >= g.nb) return;
    int *P = parent + (size_t)k * g.nb;
    if (P[B] >= 0) P[B] = find_root(P, B);
}

// exclusive scan of v over the CTA (blockDim.x == CHUNK); returns the CTA total in *total
__device__ int block_exclusive_scan(int v, int *total)
{
    __shared__ int warp_sum[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int s = v;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += t; }
    if (lane == 31) warp_sum[wid] = s;
    __syncthreads();
    if (wid == 0) {
        int ws = lane < (int)(blockDim.x >> 5) ? warp_sum[lane] : 0;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, ws, o); if (lane >= o) ws += t; }
        warp_sum[lane] = ws;
    }
    __syncthreads();
    const int before = (wid ? warp_sum[wid - 1] : 0) + s - v;
    *total = warp_sum[(blockDim.x >> 5) - 1];
    __syncthreads();
    return before;
}

// roots per chunk of CHUNK blocks
__global__ void k_label_count(TraceGeom g, const int *parent, int nch, int *chunk)
{
    const int B = blockIdx.x * CHUNK + threadIdx.x, k = blockIdx.y;
    const int r = B < g.nb && parent[(size_t)k * g.nb + B] == B;
    const int n = __syncthreads_count(r);
    if (threadIdx.x == 0) chunk[(size_t)k * nch + blockIdx.x] = n;
}

// per plane: exclusive scan of the chunk counts (in place) and the number of components
__global__ void k_label_scan(int nch, int *chunk, int *n_comp)
{
    int *c = chunk + (size_t)blockIdx.x * nch;
    int carry = 0;
    for (int base = 0; base < nch; base += CHUNK) {
        const int i = base + threadIdx.x;
        const int v = i < nch ? c[i] : 0;
        int tot;
        const int ex = block_exclusive_scan(v, &tot);
        if (i < nch) c[i] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) n_comp[blockIdx.x] = carry;
}

// label (0-based, cv2's label - 1) of every root block
__global__ void k_label_assign(TraceGeom g, const int *parent, int nch, const int *chunk, int *rootlab)
{
    const int B = blockIdx.x * CHUNK + threadIdx.x, k = blockIdx.y;
    const int r = B < g.nb && parent[(size_t)k * g.nb + B] == B;
    int tot;
    const int ex = block_exclusive_scan(r, &tot);
    if (r) rootlab[(size_t)k * g.nb + B] = chunk[(size_t)k * nch + blockIdx.x] + ex;
}

struct CompBase { int base[OMNI_MAX_K]; };

__global__ void k_comp_init(TraceComp *c, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    TraceComp t{};
    t.x0 = t.y0 = INT_MAX; t.x1 = t.y1 = -1; t.root = -1;
    c[i] = t;
}

// area and bounding box per component, one thread per 2x2 block
__global__ void k_comp_stats(TraceGeom g, const int *rootlab, CompBase cb, TraceComp *comps)
{
    const int B = blockIdx.x * blockDim.x + threadIdx.x, k = blockIdx.y;
    if (B >= g.nb) return;
    const int r = g.parent[(size_t)k * g.nb + B];
    if (r < 0) return;
    TraceComp *c = comps + cb.base[k] + rootlab[(size_t)k * g.nb + r];
    const u8 *S = g.skel + k * g.plane_stride;
    const int x = 2 * (B % g.bw), y = 2 * (B / g.bw);
    int x0 = INT_MAX, y0 = INT_MAX, x1 = -1, y1 = -1, n = 0;
    for (int dy = 0; dy < 2; dy++)
        for (int dx = 0; dx < 2; dx++)
            if (px(S, g.pitch, g.h, g.w, x + dx, y + dy)) {
                n++; x0 = min(x0, x + dx); x1 = max(x1, x + dx); y0 = min(y0, y + dy); y1 = max(y1, y + dy);
            }
    atomicMin(&c->x0, x0); atomicMin(&c->y0, y0); atomicMax(&c->x1, x1); atomicMax(&c->y1, y1);
    atomicAdd(&c->area, n);
    if (r == B) c->root = r;
}

// ---- row-major foreground lists (start-pixel scans of the large components) --------------------------------------------
__global__ void k_row_count(TraceGeom g, int *row_cnt)
{
    const int y = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), k = blockIdx.y, lane = threadIdx.x & 31;
    if (y >= g.h) return;
    const u8 *row = g.skel + k * g.plane_stride + (size_t)y * g.pitch;
    int n = 0;
    for (int x = lane; x < g.w; x += 32) n += row[x] != 0;
    for (int o = 16; o; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if (lane == 0) row_cnt[(size_t)k * (g.h + 1) + y] = n;
}

__global__ void k_row_scan(int h, int *row_off)   // in place: counts -> exclusive offsets, [h] = total
{
    int *c = row_off + (size_t)blockIdx.x * (h + 1);
    int carry = 0;
    for (int base = 0; base < h + 1; base += CHUNK) {
        const int i = base + threadIdx.x;
        const int v = i < h ? c[i] : 0;
        int tot;
        const int ex = block_exclusive_scan(v, &tot);
        if (i < h + 1) c[i] = carry + ex;
        carry += tot;
    }
}

__global__ void k_row_fill(TraceGeom g, const int *plane_off, int *row_x)
{
    const int y = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), k = blockIdx.y, lane = threadIdx.x & 31;
    if (y >= g.h) return;
    const u8 *row = g.skel + k * g.plane_stride + (size_t)y * g.pitch;
    int o = plane_off[k] + g.row_off[(size_t)k * (g.h + 1) + y];
    for (int x0 = 0; x0 < g.w; x0 += 32) {
        const int x = x0 + lane;
        const bool f = x < g.w && row[x] != 0;
        const u32 b = __ballot_sync(0xffffffffu, f);
        if (f) row_x[o + __popc(b & ((1u << lane) - 1u))] = x;
        o += __popc(b);
    }
}

// ---- the walk (04_find_contours.py:126-200) -----------------------------------------------------------------------------
__constant__ int8_t NDX[8] = {-1, 0, 1, -1, 1, -1, 0, 1};   // NEIGH8 (04:12): the visiting order; bit i = neighbour i,
__constant__ int8_t NDY[8] = {-1, -1, -1, 0, 0, 1, 1, 1};   // neighbour 7 - i is the opposite one

// component in a shared-memory byte map with a one-pixel frame: bit 0 = pixel of the component, bit 1 = visited
struct SmemMap {
    u8 *t; int W2, x0, y0;
    __device__ int idx(int x, int y) const { return (y - y0 + 1) * W2 + (x - x0 + 1); }
    __device__ u32 nbr(int x, int y, u32 &vis) const {
        const int i = idx(x, y);
        const u8 v0 = t[i - W2 - 1], v1 = t[i - W2], v2 = t[i - W2 + 1], v3 = t[i - 1], v4 = t[i + 1], v5 = t[i + W2 - 1],
                 v6 = t[i + W2], v7 = t[i + W2 + 1];
        const u32 a = v0 | (v1 << 2) | (v2 << 4) | (v3 << 6) | (v4 << 8) | (v5 << 10) | (v6 << 12) | ((u32)v7 << 14);
        vis = even_bits(a >> 1);
        return even_bits(a);
    }
    // bits 0, 2, 4, ... 14 of a -> bits 0..7
    static __device__ __forceinline__ u32 even_bits(u32 a) {
        a &= 0x5555u;
        a = (a | (a >> 1)) & 0x3333u;
        a = (a | (a >> 2)) & 0x0f0fu;
        return (a | (a >> 4)) & 0xffu;
    }
    __device__ bool visited(int x, int y) const { return t[idx(x, y)] & 2; }
    __device__ void mark(int x, int y) const { t[idx(x, y)] = 3; }
};

// component read from the skeleton plane: a foreground 8-neighbour of a component pixel belongs to the component
struct GlobalMap {
    const u8 *S; size_t pitch; u8 *V; int h, w;
    __device__ u32 nbr(int x, int y, u32 &vis) const {
        u32 c = 0, v = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int xx = x + NDX[i], yy = y + NDY[i];
            if (xx >= 0 && yy >= 0 && xx < w && yy < h) {
                c |= (u32)(S[(size_t)yy * pitch + xx] != 0) << i;
                v |= (u32)(V[(size_t)yy * w + xx] != 0) << i;
            }
        }
        vis = v;
        return c;
    }
    __device__ bool visited(int x, int y) const { return V[(size_t)y * w + x] != 0; }
    __device__ void mark(int x, int y) const { V[(size_t)y * w + x] = 1; }
};

struct Out {                  // the polylines of one component (write pass only)
    int2 *pts; int *lens;
    long long np; int npaths;
};

// one path from (sx, sy), lane 0 only.  cycle = 0: 04:143-170, cycle = 1: 04:172-200.
template <bool WRITE, class M>
__device__ void walk(const M &m, int sx, int sy, bool cycle, long long guard, Out &o)
{
    int x = sx, y = sy, prev = -1;              // prev: neighbour index of the previous pixel as seen from (x, y)
    long long len = 1, step_guard = 0;
    m.mark(x, y);
    for (bool first = true;; first = false) {
        u32 vis;
        const u32 cm = m.nbr(x, y, vis);
        if (!cycle && !first) {                  // 04:161-165: stop at a junction or an endpoint, then the guard
            const int d = __popc(cm);
            if (d == 1 || d >= 3) break;
            if (++step_guard > guard) break;
        }
        u32 c = cm & ~vis;                       // first unvisited neighbour (the previous pixel is visited)
        if (!c && cycle) c = cm & ~(prev >= 0 ? 1u << prev : 0u);   // 04:186-192: the step onto a visited pixel
        if (!c) break;
        const int i = __ffs(c) - 1;
        if (WRITE) {
            if (len == 1) o.pts[o.np] = make_int2(sx, sy);
            o.pts[o.np + len] = make_int2(x + NDX[i], y + NDY[i]);
        }
        x += NDX[i]; y += NDY[i]; prev = 7 - i; len++;
        m.mark(x, y);
        if (cycle) {                             // 04:194-197
            if (x == sx && y == sy) break;
            if (++step_guard > guard) break;
        }
    }
    if (len < 2) return;                         // 04:168, 04:199
    if (cycle) {                                 // 04:200-203: hypot(first - last) < 1.5 closes the polyline
        const int dx = x - sx, dy = y - sy;
        if (dx * dx + dy * dy <= 2) { if (WRITE) o.pts[o.np + len] = make_int2(sx, sy); len++; }
    }
    if (WRITE) o.lens[o.npaths] = (int)len;
    o.np += len;
    o.npaths++;
}

// lane 0 walks from every start pixel of a ballot (bit i = pixel x0 + i of row y), in order
template <bool WRITE, class M>
__device__ void walk_starts(const M &m, u32 bal, const int *xs, int y, bool cycle, long long guard, Out &o)
{
    if ((threadIdx.x & 31) == 0)
        while (bal) {
            const int i = __ffs(bal) - 1;
            bal &= bal - 1;
            const int x = xs[i];
            if (!m.visited(x, y)) walk<WRITE>(m, x, y, cycle, guard, o);
        }
    __syncwarp();
}

template <bool WRITE>
__device__ void finish(TraceComp &c, const Out &o)
{
    if ((threadIdx.x & 31) == 0 && !WRITE) { c.npts = o.np; c.npaths = o.npaths; }
}

// components whose map fits in shared memory; one warp per component, order[] = biggest first
template <bool WRITE>
__global__ void __launch_bounds__(32) k_trace_walk_smem(TraceGeom g, TraceComp *comps, const int *order, const int *plane_of,
                                                          int2 *pts, int *lens)
{
    extern __shared__ __align__(16) u8 tile[];
    __shared__ int xs[32];
    const int ci = order[blockIdx.x], k = plane_of[ci], lane = threadIdx.x;
    TraceComp &c = comps[ci];
    const int x0 = c.x0, y0 = c.y0, x1 = c.x1, y1 = c.y1, W2 = x1 - x0 + 3, H2 = y1 - y0 + 3, root = c.root;
    const u8 *S = g.skel + k * g.plane_stride;
    const int *P = g.parent + (size_t)k * g.nb;
    for (int i = lane; i < W2 * H2; i += 32) {                      // the component, label-filtered, in a one-pixel frame
        const int x = x0 - 1 + i % W2, y = y0 - 1 + i / W2;
        tile[i] = (px(S, g.pitch, g.h, g.w, x, y) && P[(y >> 1) * g.bw + (x >> 1)] == root) ? 1 : 0;
    }
    __syncwarp();
    const SmemMap m{tile, W2, x0, y0};
    Out o{pts, lens, 0, 0};
    if (WRITE) { o.pts = pts + c.pt_base; o.lens = lens + c.path_base; }
    for (int cycle = 0; cycle < 2; cycle++) {
        const long long guard = cycle ? 4LL * c.area : g.guard_open[k];
        for (int y = y0; y <= y1; y++)
            for (int xb = x0; xb <= x1; xb += 32) {
                const int x = xb + lane;
                bool s = false;
                if (x <= x1 && (tile[m.idx(x, y)] & 1)) {
                    u32 vis;
                    const u32 cm = m.nbr(x, y, vis);
                    s = cycle ? !m.visited(x, y) : __popc(cm) == 1;   // endpoints (04:124) / pixels still unvisited (04:173)
                }
                const u32 bal = __ballot_sync(0xffffffffu, s);
                if (!bal) continue;
                xs[lane] = x;
                __syncwarp();
                walk_starts<WRITE>(m, bal, xs, y, cycle, guard, o);
            }
    }
    finish<WRITE>(c, o);
}

// components too large for shared memory: skeleton plane + visited plane + row-major foreground lists
template <bool WRITE>
__global__ void __launch_bounds__(32) k_trace_walk_global(TraceGeom g, TraceComp *comps, const int *order, const int *plane_of,
                                                            const int *plane_off, int2 *pts, int *lens)
{
    __shared__ int xs[32];
    const int ci = order[blockIdx.x], k = plane_of[ci], lane = threadIdx.x;
    TraceComp &c = comps[ci];
    const int x0 = c.x0, y0 = c.y0, x1 = c.x1, y1 = c.y1, root = c.root;
    const u8 *S = g.skel + k * g.plane_stride;
    const int *P = g.parent + (size_t)k * g.nb;
    const int *ro = g.row_off + (size_t)k * (g.h + 1), *rx = g.row_x + plane_off[k];
    const GlobalMap m{S, g.pitch, g.visited + (size_t)k * g.h * g.w, g.h, g.w};
    Out o{pts, lens, 0, 0};
    if (WRITE) { o.pts = pts + c.pt_base; o.lens = lens + c.path_base; }
    for (int cycle = 0; cycle < 2; cycle++) {
        const long long guard = cycle ? 4LL * c.area : g.guard_open[k];
        for (int y = y0; y <= y1; y++)
            for (int e = ro[y]; e < ro[y + 1]; e += 32) {
                const int j = e + lane;
                const int x = j < ro[y + 1] ? rx[j] : -1;
                bool s = false;
                if (x >= x0 && x <= x1 && P[(y >> 1) * g.bw + (x >> 1)] == root) {
                    u32 vis;
                    const u32 cm = m.nbr(x, y, vis);
                    s = cycle ? !m.visited(x, y) : __popc(cm) == 1;
                }
                const u32 bal = __ballot_sync(0xffffffffu, s);
                if (!bal) continue;
                xs[lane] = x;
                __syncwarp();
                walk_starts<WRITE>(m, bal, xs, y, cycle, guard, o);
            }
    }
    finish<WRITE>(c, o);
}

}   // namespace

#define TRY(expr) do { int rc__ = (expr); if (rc__ != OMNI_OK) return rc__; } while (0)

static dim3 grid_blocks(int nb, int K) { return dim3((unsigned)((nb + 255) / 256), (unsigned)K); }

template <bool WRITE>
static int launch_walks(omni_ctx *ctx, const TraceGeom &g, TraceComp *comps, const int *d_order_s, int n_s, int smem,
                        const int *d_order_g, int n_g, const int *plane_of, const int *plane_off, int2 *pts, int *lens,
                        cudaStream_t st)
{
    if (n_s) {
        OMNI_CUDA(cudaFuncSetAttribute(k_trace_walk_smem<WRITE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        OMNI_LAUNCH(ctx, st, WRITE ? "trace_walk_write" : "trace_walk_count",
                    (k_trace_walk_smem<WRITE><<<n_s, 32, smem, st>>>(g, comps, d_order_s, plane_of, pts, lens), cudaGetLastError()));
    }
    if (n_g) {
        OMNI_CUDA(cudaMemsetAsync(g.visited, 0, (size_t)g.K * g.h * g.w, st));
        OMNI_LAUNCH(ctx, st, WRITE ? "trace_walk_write_global" : "trace_walk_count_global",
                    (k_trace_walk_global<WRITE><<<n_g, 32, 0, st>>>(g, comps, d_order_g, plane_of, plane_off, pts, lens),
                     cudaGetLastError()));
    }
    return OMNI_OK;
}

// Slots: 7 = labels (parent, root labels, chunk sums, component counts), 8 = components (records, orders, plane of each,
// row-list offsets per plane), 9 = large-component planes (visited, row lists), 10 = polylines (points, lengths).
int trace_run(omni_ctx *ctx, const u8 *d_skel, int K, int h, int w, size_t plane_stride, size_t pitch, int64_t *h_info,
              cudaStream_t st)
{
    ctx->trace_valid = 0;
    const int bw = (w + 1) / 2, bh = (h + 1) / 2, nb = bw * bh, nch = (nb + CHUNK - 1) / CHUNK;
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t par_b = al((size_t)K * nb * 4), ch_b = al((size_t)K * nch * 4);
    TRY(omni_ws_reserve(ctx, 7, 2 * par_b + ch_b + 256));
    int *parent = (int *)ctx->ws[7], *rootlab = (int *)((u8 *)ctx->ws[7] + par_b), *chunk = (int *)((u8 *)ctx->ws[7] + 2 * par_b);
    int *d_ncomp = (int *)((u8 *)ctx->ws[7] + 2 * par_b + ch_b);
    TraceGeom g{};
    g.skel = d_skel; g.plane_stride = plane_stride; g.pitch = pitch; g.K = K; g.h = h; g.w = w; g.bw = bw; g.nb = nb;
    g.parent = parent;
    OMNI_LAUNCH(ctx, st, "trace_ccl_init", (k_ccl_init<<<grid_blocks(nb, K), 256, 0, st>>>(g, parent), cudaGetLastError()));
    OMNI_LAUNCH(ctx, st, "trace_ccl_merge", (k_ccl_merge<<<grid_blocks(nb, K), 256, 0, st>>>(g, parent), cudaGetLastError()));
    OMNI_LAUNCH(ctx, st, "trace_ccl_flatten", (k_ccl_flatten<<<grid_blocks(nb, K), 256, 0, st>>>(g, parent), cudaGetLastError()));
    OMNI_LAUNCH(ctx, st, "trace_label_count",
                (k_label_count<<<dim3(nch, K), CHUNK, 0, st>>>(g, parent, nch, chunk), cudaGetLastError()));
    OMNI_LAUNCH(ctx, st, "trace_label_scan", (k_label_scan<<<K, CHUNK, 0, st>>>(nch, chunk, d_ncomp), cudaGetLastError()));
    OMNI_LAUNCH(ctx, st, "trace_label_assign",
                (k_label_assign<<<dim3(nch, K), CHUNK, 0, st>>>(g, parent, nch, chunk, rootlab), cudaGetLastError()));
    OMNI_CUDA(cudaMemcpyAsync(ctx->h_flags, d_ncomp, K * sizeof(int), cudaMemcpyDeviceToHost, st));
    OMNI_CUDA(cudaStreamSynchronize(st));

    CompBase cb{};
    int n = 0;
    std::vector<int> ncomp(K), plane_of;
    for (int k = 0; k < K; k++) { ncomp[k] = ctx->h_flags[k]; cb.base[k] = n; n += ncomp[k]; }
    for (int k = 0; k < K; k++) plane_of.insert(plane_of.end(), ncomp[k], k);
    const size_t comp_b = al((size_t)n * sizeof(TraceComp) + 1), ord_b = al((size_t)n * 4 + 4);
    TRY(omni_ws_reserve(ctx, 8, comp_b + 3 * ord_b + 256));
    TraceComp *d_comps = (TraceComp *)ctx->ws[8];
    int *d_order_s = (int *)((u8 *)ctx->ws[8] + comp_b), *d_order_g = (int *)((u8 *)ctx->ws[8] + comp_b + ord_b);
    int *d_plane_of = (int *)((u8 *)ctx->ws[8] + comp_b + 2 * ord_b), *d_plane_off = (int *)((u8 *)ctx->ws[8] + comp_b + 3 * ord_b);
    std::vector<TraceComp> comps(n);
    if (n) {
        OMNI_LAUNCH(ctx, st, "trace_comp_init", (k_comp_init<<<(n + 255) / 256, 256, 0, st>>>(d_comps, n), cudaGetLastError()));
        OMNI_LAUNCH(ctx, st, "trace_comp_stats",
                    (k_comp_stats<<<grid_blocks(nb, K), 256, 0, st>>>(g, rootlab, cb, d_comps), cudaGetLastError()));
        OMNI_CUDA(cudaMemcpyAsync(comps.data(), d_comps, (size_t)n * sizeof(TraceComp), cudaMemcpyDeviceToHost, st));
        OMNI_CUDA(cudaMemcpyAsync(d_plane_of, plane_of.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
        OMNI_CUDA(cudaStreamSynchronize(st));
    }

    // per plane: total_fg (the open-phase guard), then the two classes of components, biggest first
    std::vector<long long> fg(K, 0);
    std::vector<int> plane_off(K + 1, 0), ord_s, ord_g;
    int smem = 0;
    for (int i = 0; i < n; i++) {
        const TraceComp &c = comps[i];
        fg[plane_of[i]] += c.area;
        const long long tb = (long long)(c.x1 - c.x0 + 3) * (c.y1 - c.y0 + 3);
        if (tb <= TRACE_SMEM_CAP) { ord_s.push_back(i); smem = std::max(smem, (int)tb); }
        else ord_g.push_back(i);
    }
    for (int k = 0; k < K; k++) { g.guard_open[k] = 2 * fg[k]; plane_off[k + 1] = plane_off[k] + (int)fg[k]; }
    smem = (smem + 15) & ~15;
    auto by_area = [&](int a, int b) { return comps[a].area != comps[b].area ? comps[a].area > comps[b].area : a < b; };
    std::sort(ord_s.begin(), ord_s.end(), by_area);
    std::sort(ord_g.begin(), ord_g.end(), by_area);
    if (!ord_g.empty()) {
        const size_t vis_b = al((size_t)K * h * w), ro_b = al((size_t)K * (h + 1) * 4);
        TRY(omni_ws_reserve(ctx, 9, vis_b + ro_b + al((size_t)plane_off[K] * 4 + 4)));
        g.visited = (u8 *)ctx->ws[9];
        int *row_off = (int *)((u8 *)ctx->ws[9] + vis_b), *row_x = (int *)((u8 *)ctx->ws[9] + vis_b + ro_b);
        g.row_off = row_off; g.row_x = row_x;
        const dim3 rg((unsigned)((h + 7) / 8), (unsigned)K);
        OMNI_CUDA(cudaMemcpyAsync(d_plane_off, plane_off.data(), (size_t)K * 4, cudaMemcpyHostToDevice, st));
        OMNI_LAUNCH(ctx, st, "trace_row_count", (k_row_count<<<rg, 256, 0, st>>>(g, row_off), cudaGetLastError()));
        OMNI_LAUNCH(ctx, st, "trace_row_scan", (k_row_scan<<<K, CHUNK, 0, st>>>(h, row_off), cudaGetLastError()));
        OMNI_LAUNCH(ctx, st, "trace_row_fill", (k_row_fill<<<rg, 256, 0, st>>>(g, d_plane_off, row_x), cudaGetLastError()));
    }
    if (!ord_s.empty()) OMNI_CUDA(cudaMemcpyAsync(d_order_s, ord_s.data(), ord_s.size() * 4, cudaMemcpyHostToDevice, st));
    if (!ord_g.empty()) OMNI_CUDA(cudaMemcpyAsync(d_order_g, ord_g.data(), ord_g.size() * 4, cudaMemcpyHostToDevice, st));
    TRY(launch_walks<false>(ctx, g, d_comps, d_order_s, (int)ord_s.size(), smem, d_order_g, (int)ord_g.size(), d_plane_of,
                            d_plane_off, nullptr, nullptr, st));
    if (n) {
        OMNI_CUDA(cudaMemcpyAsync(comps.data(), d_comps, (size_t)n * sizeof(TraceComp), cudaMemcpyDeviceToHost, st));
        OMNI_CUDA(cudaStreamSynchronize(st));
    }

    // output offsets: planes in order, components in label order (cv2's), polylines in walk order
    long long pts_total = 0, paths_total = 0;
    ctx->trace_info.assign((size_t)4 * K, 0);
    ctx->trace_comp.assign((size_t)6 * n, 0);
    for (int i = 0; i < n; i++) {
        TraceComp &c = comps[i];
        c.pt_base = pts_total; c.path_base = paths_total;
        pts_total += c.npts; paths_total += c.npaths;
        int32_t *r = &ctx->trace_comp[(size_t)6 * i];
        r[0] = c.x0; r[1] = c.y0; r[2] = c.x1 - c.x0 + 1; r[3] = c.y1 - c.y0 + 1; r[4] = c.area; r[5] = c.npaths;
        long long *pi = &ctx->trace_info[(size_t)4 * plane_of[i]];
        pi[2] += c.npaths; pi[3] += c.npts;
    }
    OMNI_REQUIRE(paths_total < INT_MAX, "omni_trace_centerlines: %lld polylines exceed the int32 range", paths_total);
    for (int k = 0; k < K; k++) { ctx->trace_info[(size_t)4 * k] = fg[k]; ctx->trace_info[(size_t)4 * k + 1] = ncomp[k]; }
    const size_t pts_b = al((size_t)pts_total * 8 + 8);
    TRY(omni_ws_reserve(ctx, 10, pts_b + al((size_t)paths_total * 4 + 4)));
    int2 *d_pts = (int2 *)ctx->ws[10];
    int *d_lens = (int *)((u8 *)ctx->ws[10] + pts_b);
    if (n) {
        OMNI_CUDA(cudaMemcpyAsync(d_comps, comps.data(), (size_t)n * sizeof(TraceComp), cudaMemcpyHostToDevice, st));
        // write pass, longest output first
        auto by_pts = [&](int a, int b) { return comps[a].npts != comps[b].npts ? comps[a].npts > comps[b].npts : a < b; };
        std::sort(ord_s.begin(), ord_s.end(), by_pts);
        std::sort(ord_g.begin(), ord_g.end(), by_pts);
        if (!ord_s.empty()) OMNI_CUDA(cudaMemcpyAsync(d_order_s, ord_s.data(), ord_s.size() * 4, cudaMemcpyHostToDevice, st));
        if (!ord_g.empty()) OMNI_CUDA(cudaMemcpyAsync(d_order_g, ord_g.data(), ord_g.size() * 4, cudaMemcpyHostToDevice, st));
        TRY(launch_walks<true>(ctx, g, d_comps, d_order_s, (int)ord_s.size(), smem, d_order_g, (int)ord_g.size(), d_plane_of,
                               d_plane_off, d_pts, d_lens, st));
    }
    OMNI_CUDA(cudaStreamSynchronize(st));
    ctx->trace_K = K;
    ctx->trace_points = pts_total;
    ctx->trace_paths = paths_total;
    ctx->trace_valid = 1;
    if (h_info) std::copy(ctx->trace_info.begin(), ctx->trace_info.end(), h_info);
    return OMNI_OK;
}

int trace_results(omni_ctx *ctx, int32_t *points, int32_t *path_len, int32_t *comp)
{
    OMNI_REQUIRE(ctx->trace_valid, "omni_trace_results: no omni_trace_centerlines result on this ctx");
    const size_t pts_b = (((size_t)ctx->trace_points * 8 + 8) + 255) & ~(size_t)255;
    if (points && ctx->trace_points)
        OMNI_CUDA(cudaMemcpyAsync(points, ctx->ws[10], (size_t)ctx->trace_points * 8, cudaMemcpyDefault, ctx->stream));
    if (path_len && ctx->trace_paths)
        OMNI_CUDA(cudaMemcpyAsync(path_len, (u8 *)ctx->ws[10] + pts_b, (size_t)ctx->trace_paths * 4, cudaMemcpyDefault, ctx->stream));
    OMNI_CUDA(cudaStreamSynchronize(ctx->stream));
    if (comp) std::copy(ctx->trace_comp.begin(), ctx->trace_comp.end(), comp);
    return OMNI_OK;
}
