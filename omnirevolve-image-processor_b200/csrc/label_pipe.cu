// label_pipe.cu -- the label-domain generation of the fused colour+edge call (omni_color_edge / omni_color_edge_batch).
//
// The first generation (fast_kernels.cu) writes K one-hot bit-planes and pushes every one of them through the 8-step
// morphology chain on 64-bit windows.  Here:
//
//   fk_assign_slices   image -> label BIT-SLICES (4 planes: bit b of the 4-bit label of every pixel) [+ u8 labels]
//                      (02_color_extract.py:35-36,53-55,121-127; the same exact table-driven assignment as fk_assign_rgbcell, but a
//                      lane owns 8 consecutive pixels -- three 8-byte shared-memory loads instead of 24 byte loads -- and there are
//                      no per-plane stores and no __match_any: 4 slice words per 32 pixels come out of a 4x4 byte transpose)
//   fk_open_morph      a CTA stages the label slices of one strip in shared memory (bulk copies, mbarrier completion) and computes
//                      the RECT-3 OPEN of all K one-hot planes at once, in the label domain (02:152):
//                        erode_k  = [label == k] & U        U  = "the 3x3 neighbourhood (inside the image) has one label"
//                        open_k   = [label == k] & Od       Od = dilate3(U)     (a pixel next to a uniform pixel q has q's label)
//                      so the first two steps of the chain cost ONE plane (Od, kept in shared memory) instead of K.  Then one warp
//                      per plane k: open_k = Od & [label == k], the remaining steps (02:153 RECT-3 close -> mask BYTES; 03:23-30
//                      ELLIPSE-3 open/close -> bit-plane M2) on 32-bit words: lanes are adjacent word columns, the neighbour bits
//                      of a step come from two warp shuffles (ALU pipe: 2 LOP3 + 2 SHF per step and 32 pixels instead of 4 + 4 on
//                      a 64-bit window); 30 owned columns + a halo lane on each side per warp.  Classifies its tiles for the
//                      sparse edge kernel (edges3.cu) like fk_morph does.
//   fk_edges3_simd<sparse> + fk_hysteresis as before.
//
// Reference call sites are relative to /root/reference/image_processor/.  Bit-exactness against the oracle is checked by the same
// GPU tests as the first generation (tests/test_gpu_parity.py runs every family).
#include "fast_device.cuh"

#include <algorithm>
#include <vector>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define LP_ZBUF 8192                      // zeroed shared-memory block behind the tables of fk_assign_slices (bulk-store source)
#define SP_TRY(expr) do { int rc__ = (expr); if (rc__ != OMNI_OK) return rc__; } while (0)


// ------------------------------------------------------------------------------------------------
// RGB-cell tables in the index layout of fk_assign_slices: cell = (B >> 2) | (G >> 2) << 6 | (R >> 2) << 12; the label nibble of
// cell i lives in byte (i & 0x1FFFF), high nibble when i >= 2^17; K == 16 has a separate "several candidates" bit per cell.
// The pruning rule is fk_build_rgbcells' (fast_kernels.cu): exact Lab box of the cell, dmin <= min dmax + 2.
// ------------------------------------------------------------------------------------------------
// the Lab boxes of fk_rgb_boxes (B slowest) re-ordered to this index layout, 8 bytes per cell (min L, a, b, max L, a, b, 0, 0), once
// per context: the table build then reads them with consecutive threads on consecutive cells, one 8-byte load per cell
__global__ void __launch_bounds__(256) fk_permute_boxes3(const u8 *__restrict__ boxes, uint2 *__restrict__ boxes3)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= RC_COUNT) return;
    const int ci = ((idx & 63) << 12) | (((idx >> 6) & 63) << 6) | (idx >> 12);
    const u8 *q = boxes + 6 * ci;
    boxes3[idx] = make_uint2((u32)q[0] | ((u32)q[1] << 8) | ((u32)q[2] << 16) | ((u32)q[3] << 24), (u32)q[4] | ((u32)q[5] << 8));
}

// candidate set of a box [lo, hi]^3 (fk_build_cells' rule): centres k with dmin_k <= min_j dmax_j + 2
__device__ __forceinline__ u32 lp_candidates(const AssignParams &P, const float (&lo)[3], const float (&hi)[3], bool &sane)
{
    const int K = P.K;
    float U = 3.0e38f;
    sane = true;
    for (int k = 0; k < K; k++) {
        float dmax = 0.f;
#pragma unroll
        for (int d = 0; d < 3; d++) {
            const float c = P.c[3 * k + d];
            sane = sane && (fabsf(c) < 1.0e4f);                 // also false for NaN
            const float m = fmaxf(fabsf(lo[d] - c), fabsf(hi[d] - c));
            dmax += m * m;
        }
        U = fminf(U, dmax);
    }
    u32 mask = 0u;
    for (int k = 0; k < K; k++) {
        float dmin = 0.f;
#pragma unroll
        for (int d = 0; d < 3; d++) {
            const float c = P.c[3 * k + d];
            const float n = fminf(fmaxf(c, lo[d]), hi[d]);
            dmin += (n - c) * (n - c);
        }
        if (dmin <= U + 2.0f) mask |= 1u << k;
    }
    return mask;
}

// Both candidate tables of a centre set in ONE launch: blocks [0, 512) the RGB-cell tables (a thread = the cells c and c + 2^17 that
// share a label byte), blocks [512, 640) the Lab-cell table of fk_build_cells (bit sets; same rule, same arithmetic).
#define LP_RGB_BLOCKS ((1 << 17) / 256)
#define LP_TAB_BLOCKS (LP_RGB_BLOCKS + CELL_COUNT / 256)
__global__ void __launch_bounds__(256) fk_build_tables3(const __grid_constant__ AssignParams P, const uint2 *__restrict__ boxes3,
                                                        u8 *__restrict__ nb, u32 *__restrict__ mb, u32 *__restrict__ cells)
{
    const int K = P.K;
    if (blockIdx.x >= LP_RGB_BLOCKS) {
        const int ci = (blockIdx.x - LP_RGB_BLOCKS) * 256 + threadIdx.x;
        const float lo[3] = {(float)((ci >> (2 * 5)) << CELL_SHIFT), (float)(((ci >> 5) & 31) << CELL_SHIFT), (float)((ci & 31) << CELL_SHIFT)};
        const float span = (float)((1 << CELL_SHIFT) - 1);
        const float hi[3] = {lo[0] + span, lo[1] + span, lo[2] + span};
        bool sane;
        u32 mask = lp_candidates(P, lo, hi, sane);
        if (!sane || mask == 0u) mask = K >= 32 ? 0xffffffffu : ((1u << K) - 1u);
        cells[ci] = mask;
        return;
    }
    const u32 cell = blockIdx.x * 256 + threadIdx.x;                    // < 2^17
    u32 byte = 0u;
    bool multi[2];
#pragma unroll
    for (int hs = 0; hs < 2; hs++) {
        const uint2 bx = __ldg(boxes3 + cell + ((u32)hs << 17));
        const float lo[3] = {(float)(bx.x & 255u), (float)((bx.x >> 8) & 255u), (float)((bx.x >> 16) & 255u)};
        const float hi[3] = {(float)(bx.x >> 24), (float)(bx.y & 255u), (float)((bx.y >> 8) & 255u)};
        bool sane;
        const u32 mask = lp_candidates(P, lo, hi, sane);
        const bool single = sane && mask != 0u && (mask & (mask - 1u)) == 0u;
        multi[hs] = !single;
        const u32 nib = single ? (u32)(P.lut[__ffs(mask) - 1] & 15u) : (K < 16 ? 15u : 0u);
        byte |= nib << (4 * hs);
    }
    nb[cell] = (u8)byte;
    const u32 b0 = __ballot_sync(0xffffffffu, multi[0]), b1 = __ballot_sync(0xffffffffu, multi[1]);
    if ((threadIdx.x & 31) == 0) { mb[cell >> 5] = b0; mb[(cell >> 5) + (1u << 12)] = b1; }
}

// ------------------------------------------------------------------------------------------------
// fk_assign_slices: one 1024-thread CTA per SM holds the tables in shared memory (as fk_assign_rgbcell); a warp takes 256 pixels
// of a row, a lane 8 consecutive ones (24 bytes = three 8-byte shared-memory loads).  Pixels whose RGB cell has several candidate
// centres are compacted over the warp and get the Lab conversion + the reference's float32 argmin over the Lab cell's candidates.
// Output: per 32 pixels one word in each of the 4 label bit-slices (a 4x4 byte transpose over 4 lanes), optionally u8 labels.
// ------------------------------------------------------------------------------------------------
template <bool SEP_MULTI>
__global__ void __launch_bounds__(RA_THREADS, 1) fk_assign_slices(const u8 *__restrict__ px, int h, int w, size_t pitch,
                                                                  const __grid_constant__ AssignParams P, const uint4 *__restrict__ rtab,
                                                                  const u32 *__restrict__ cells, const u16 *__restrict__ labtab,
                                                                  u8 *__restrict__ labels, size_t lpitch, u32 *__restrict__ slices,
                                                                  int ws, int nf, size_t frame_stride,
                                                                  const __grid_constant__ ZeroJob Z)
{
    extern __shared__ __align__(16) u8 smem[];
    const u8 *s_nb = smem;
    const u32 *s_mb = reinterpret_cast<const u32 *>(smem + RA_OFF_MB);
    u16 *s_cbrt = reinterpret_cast<u16 *>(smem + RA_OFF_CBRT);
    u16 *s_gam = reinterpret_cast<u16 *>(smem + RA_OFF_GAM);
    float4 *s_ctr = reinterpret_cast<float4 *>(smem + RA_OFF_CTR);
    u8 *s_lut = smem + RA_OFF_LUT;
    for (int i = threadIdx.x; i < (RC_NIB_BYTES + (SEP_MULTI ? RC_MB_BYTES : 0)) / 16; i += RA_THREADS)
        reinterpret_cast<uint4 *>(smem)[i] = __ldg(rtab + i);
    for (int i = threadIdx.x; i < 2048; i += RA_THREADS) {
        s_cbrt[i] = labtab[256 + i];
        if (i < 256) s_gam[i] = labtab[i];
    }
    if (threadIdx.x < OMNI_MAX_K) {
        s_lut[threadIdx.x] = P.lut[threadIdx.x];
        s_ctr[threadIdx.x] = make_float4(P.c[3 * threadIdx.x], P.c[3 * threadIdx.x + 1], P.c[3 * threadIdx.x + 2], 0.f);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int chunks = (w + 255) >> 8;
    const int total = nf * h * chunks, stride = gridDim.x * RA_WARPS;     // nf * h * chunks < 2^30 (checked by the host)
    const bool vec_ok = (((uintptr_t)px | pitch | frame_stride) & 15) == 0;
    const bool lab_vec = labels && ((((uintptr_t)labels | lpitch) & 7) == 0);
    u8 *spx = smem + RA_OFF_WARP + warp * RA_WARP_BYTES;              // per warp: the 256 pixels of the current chunk
    u8 *sq = spx + 768, *slab = sq + 256;                             //           queued pixel indices, their labels
    const u32 sel1 = (lane & 1) ? 0x3715u : 0x6240u, sel2 = (lane & 2) ? 0x3276u : 0x5410u;
    // zero source of the bulk stores (never written again): make the generic-proxy writes visible to the async proxy
    const u32 zsrc = (u32)__cvta_generic_to_shared(smem + RA_SMEM);
    for (int i = threadIdx.x; i < LP_ZBUF / 16; i += RA_THREADS) reinterpret_cast<uint4 *>(smem + RA_SMEM)[i] = make_uint4(0u, 0u, 0u, 0u);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    uint4 pf0 = make_uint4(0, 0, 0, 0), pf1 = pf0;
    const int dyy = stride / chunks, dc = stride - dyy * chunks;
    auto prefetch = [&](int u, int yy, int c) {
        if (u < total) {
            const int f = nf > 1 ? yy / h : 0, y = yy - f * h;
            if (vec_ok && c * 256 + 256 <= w) {
                const uint4 *src = reinterpret_cast<const uint4 *>(px + (size_t)f * frame_stride + (size_t)y * pitch + (size_t)c * 768);
                pf0 = __ldg(src + lane);
                if (lane < 16) pf1 = __ldg(src + 32 + lane);
            }
        }
    };
    int u = blockIdx.x * RA_WARPS + warp;
    int yy_n = u / chunks, c_n = u - yy_n * chunks;
    prefetch(u, yy_n, c_n);
    for (; u < total; u += stride) {
        const int yy = yy_n, c = c_n;
        yy_n += dyy; c_n += dc;
        if (c_n >= chunks) { c_n -= chunks; yy_n++; }
        const int f = nf > 1 ? yy / h : 0, y = yy - f * h;
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
        // this chunk's slice of the zero-fill regions: bulk copies (TMA engine) from the zeroed shared-memory block, issued by one
        // lane -- no LSU wavefronts, the stores drain while the warp works on its pixels
        if (lane == 0) {
#pragma unroll
            for (int z = 0; z < 2; z++) {
                if (Z.per[z]) {
                    const unsigned long long idx = (unsigned long long)Z.per[z] * (unsigned)u;
                    if (idx < Z.n16[z]) {
                        u32 left = (u32)min((unsigned long long)Z.per[z], Z.n16[z] - idx) * 16u;      // per * 16 < 2^32 (launcher)
                        char *dst = reinterpret_cast<char *>(Z.p[z] + idx);
                        do {
                            const u32 n = min(left, (u32)LP_ZBUF);
                            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(zsrc), "r"(n) : "memory");
                            dst += n; left -= n;
                        } while (left);
                    }
                }
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        __syncwarp();
        // ---- phase 1: the lane's 8 pixels: RGB-cell lookups ----
        const uint2 *q2 = reinterpret_cast<const uint2 *>(spx + 24 * lane);
        const uint2 qa = q2[0], qb = q2[1], qc = q2[2];
        const u32 wv[6] = {qa.x, qa.y, qb.x, qb.y, qc.x, qc.y};
        const int xbase = c * 256 + 8 * lane;
        u32 nibw = 0u, mm = 0u;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const int qi = (3 * j) >> 2, o = (3 * j) & 3;
            u32 v;
            if (o == 0) v = wv[qi];
            else if (o == 1) v = wv[qi] >> 8;
            else if (o == 2) v = __byte_perm(wv[qi], wv[(qi + 1) % 6], 0x4432);
            else v = __byte_perm(wv[qi], wv[(qi + 1) % 6], 0x5543);
            const u32 idx = ((v >> 2) & 0x3Fu) | ((v >> 4) & 0xFC0u) | ((v >> 6) & 0x3F000u);
            const u32 lab = ((u32)s_nb[idx & 0x1FFFFu] >> ((idx >> 15) & 4u)) & 15u;
            nibw |= lab << (4 * j);
            if (SEP_MULTI) mm |= ((s_mb[idx >> 5] >> (idx & 31u)) & 1u) << j;
        }
        if (!SEP_MULTI) {                                      // K <= 15: nibble 15 = "several candidates"; 8 nibbles -> 8 flag bits
            u32 t = nibw & (nibw >> 1) & (nibw >> 2) & (nibw >> 3) & 0x11111111u;
            t = (t | (t >> 3)) & 0x03030303u;
            mm = (t * 0x01041040u) >> 24;
        }
        if (!full) {                                           // pixels right of the image: label 0, never queued
            const int nv = max(0, min(8, w - xbase));
            const u32 keep = nv >= 8 ? 0xffffffffu : ((1u << (4 * nv)) - 1u);
            nibw &= keep;
            mm &= (1u << nv) - 1u;
        }
        // ---- the undecided pixels, compacted over the warp ----
        const int cnt = __popc(mm);
        int x = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, x, d);
            if (lane >= d) x += t;
        }
        const int nq = __shfl_sync(0xffffffffu, x, 31);
        if (nq) {
            int pos = x - cnt;
#pragma unroll
            for (int j = 0; j < 8; j++)
                if ((mm >> j) & 1u) sq[pos++] = (u8)(8 * lane + j);
            __syncwarp();
            // ---- phase 2: Lab conversion + the reference's float32 argmin over the Lab cell's candidates ----
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
            if (mm) {
                const uint2 lb = *reinterpret_cast<const uint2 *>(slab + 8 * lane);
                u32 t0 = lb.x & 0x0F0F0F0Fu, t1 = lb.y & 0x0F0F0F0Fu;            // 8 label bytes -> 8 nibbles
                t0 = (t0 | (t0 >> 4)) & 0x00FF00FFu; t0 = (t0 | (t0 >> 8)) & 0xFFFFu;
                t1 = (t1 | (t1 >> 4)) & 0x00FF00FFu; t1 = (t1 | (t1 >> 8)) & 0xFFFFu;
                const u32 fix = t0 | (t1 << 16);
                u32 m = mm;                                                       // 8 flag bits -> nibble mask
                m = (m | (m << 12)) & 0x000F000Fu; m = (m | (m << 6)) & 0x03030303u; m = (m | (m << 3)) & 0x11111111u;
                m *= 15u;
                nibw = (nibw & ~m) | (fix & m);
            }
        }
        // ---- phase 3: outputs ----
        if (labels) {
            u32 b0 = nibw & 0xFFFFu, b1 = nibw >> 16;                             // 4 nibbles -> 4 bytes
            b0 = (b0 | (b0 << 8)) & 0x00FF00FFu; b0 = (b0 | (b0 << 4)) & 0x0F0F0F0Fu;
            b1 = (b1 | (b1 << 8)) & 0x00FF00FFu; b1 = (b1 | (b1 << 4)) & 0x0F0F0F0Fu;
            u8 *lrow = labels + (size_t)yy * lpitch + xbase;
            if (lab_vec && xbase + 8 <= w) *reinterpret_cast<uint2 *>(lrow) = make_uint2(b0, b1);
            else
                for (int j = 0; j < 8 && xbase + j < w; j++) lrow[j] = (u8)((nibw >> (4 * j)) & 15u);
        }
        {
            u32 r[4];
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const u32 xb = (nibw >> b) & 0x11111111u;
                const u32 x1 = (xb | (xb >> 3)) & 0x03030303u;
                r[b] = x1 * 0x01041040u;                                           // byte 3 = bit b of the lane's 8 labels
            }
            const u32 pk = __byte_perm(__byte_perm(r[0], r[1], 0x7373), __byte_perm(r[2], r[3], 0x7373), 0x5410);
            // 4x4 byte transpose over the lanes of a quad: lane (quad q, r) ends with the 32-pixel word of slice r
            u32 t = __shfl_xor_sync(0xffffffffu, pk, 1);
            const u32 v1 = __byte_perm(pk, t, sel1);
            t = __shfl_xor_sync(0xffffffffu, v1, 2);
            const u32 word = __byte_perm(v1, t, sel2);
            // interleaved layout: the 4 slice words of a word column are adjacent (uint4 per column): the warp writes 128 B
            if (c * 8 + (lane >> 2) < ws) slices[(((size_t)f * h + y) * ws + (size_t)c * 8) * 4 + lane] = word;
        }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");     // the zero block must outlive its readers
}

// ------------------------------------------------------------------------------------------------
// fk_open_morph: the label-domain RECT-3 open and the rest of the morphology chain in one kernel.  A CTA is one frame, one strip
// of TR rows and one group of 30 word columns, with one warp per plane of a group of at most OM_PMAX planes of that frame.  The
// lanes of a warp cover the word columns c0-1 .. c0+30 and lanes 1..30 own theirs; a halo lane's word is wrong in one more outer
// bit per step, never in the bit its owned neighbour reads.
//   1. Staging: thread 0 issues one cp.async.bulk per label row (the 4 slice words of the columns c0-2 .. c0+31 are 34 adjacent
//      uint4, 544 B) for all rows [y0 - N - EXT - 2, y1 + N + EXT + 2) of the strip at once, one mbarrier per OM_CHUNK rows.
//      Columns and rows outside the image are zeros in shared memory.  The strip is fetched once per CTA, not once per plane.
//   2. Od = dilate3(U), once per CTA, the warps splitting the rows.  Per label row r:
//        dh(r) = "differs from the left or right neighbour",  dv(r) = "differs from the pixel above"      (bit-slice XORs)
//        U(r-1) = ~(dh(r-2) | dh(r-1) | dh(r) | dv(r-1) | dv(r))       (neighbours outside the image are ignored, as cv2.erode does)
//        Od(r-2) = hU(r-3) | hU(r-2) | hU(r-1),  hU = U | U << 1 | U >> 1                                  (cv2.dilate: outside = 0)
//      Lanes 0 and 31 also track U of the staged columns c0-2 / c0+31, so that Od is exact in all 32 lanes.
//   3. Per plane k: open_k = Od & [label == k] from shared memory, then the remaining steps on 32-bit words with the neighbour
//      bits from warp shuffles: 02:153 RECT-3 close -> mask bytes, 03:23-30 ELLIPSE-3 open / close -> bit-plane M2; the tiles are
//      classified and the run lists of the sparse edge kernel written as fk_morph (fast_kernels.cu) does.
// ------------------------------------------------------------------------------------------------
#define LP_COLS 30                        // owned word columns per warp
#define OM_SCOLS 34                       // staged word columns per row: c0-2 .. c0+31
#define OM_CHUNK 8                        // staged rows per mbarrier
#ifndef OM_PMAX
#define OM_PMAX 8                         // plane-warps per CTA, at most
#endif

template <int OP>
__device__ __forceinline__ u32 step32(const u32 u, const u32 m, const u32 d)
{
    if (OP == ST_ER || OP == ST_DR) {
        const u32 v = OP == ST_ER ? (u & m & d) : (u | m | d);
        const u32 l = __shfl_up_sync(0xffffffffu, v, 1), r = __shfl_down_sync(0xffffffffu, v, 1);
        const u32 sl = __funnelshift_l(l, v, 1), sr = __funnelshift_r(v, r, 1);
        return OP == ST_ER ? (v & sl & sr) : (v | sl | sr);
    }
    if (OP == ST_EC || OP == ST_DC) {
        const u32 l = __shfl_up_sync(0xffffffffu, m, 1), r = __shfl_down_sync(0xffffffffu, m, 1);
        const u32 sl = __funnelshift_l(l, m, 1), sr = __funnelshift_r(m, r, 1);
        return OP == ST_EC ? ((m & sl & sr) & u & d) : ((m | sl | sr) | u | d);
    }
    return m;
}

template <int NEXT, bool ROWFIX, bool COLFIX>
__device__ __forceinline__ u32 oob_fix32(u32 v, const u32 colvalid, const bool row_inside)
{
    if (NEXT == ST_NONE) return COLFIX ? (v & colvalid) : v;
    if (op_is_erode(NEXT)) {
        if (ROWFIX && !row_inside) return 0xffffffffu;
        return COLFIX ? (v | ~colvalid) : v;
    }
    if (ROWFIX && !row_inside) return 0u;
    return COLFIX ? (v & colvalid) : v;
}

template <u32 CODE, int S>
struct MorphChain32 {
    template <int TAP, bool ROWFIX, bool COLFIX>
    static __device__ __forceinline__ void run(u32 cur, u32 (&p1)[8], u32 (&p2)[8], int t, int h, u32 colvalid, u32 &tap_out, u32 &fin)
    {
        constexpr int N = code_len(CODE);
        if (S == TAP) tap_out = cur;
        if constexpr (S < N) {
            constexpr int OP = code_op(CODE, S);
            constexpr int NEXT = (S + 1 < N) ? code_op(CODE, S + 1) : ST_NONE;
            u32 out = step32<OP>(p2[S], p1[S], cur);
            p2[S] = p1[S]; p1[S] = cur;
            const int r = t - S - 1;
            out = oob_fix32<NEXT, ROWFIX, COLFIX>(out, colvalid, !ROWFIX || (r >= 0 && r < h));
            MorphChain32<CODE, S + 1>::template run<TAP, ROWFIX, COLFIX>(out, p1, p2, t, h, colvalid, tap_out, fin);
        } else {
            fin = cur;
        }
    }
};

// shared-memory layout of fk_open_morph: [staged slice rows RS][34] uint4 | Od rows [RO + 1][32] u32
template <u32 CODE, int TR, bool RUNS>
struct OmLayout {
    static constexpr int N = code_len(CODE), EXT = RUNS ? 2 : 0;
    static constexpr int RS = TR + 2 * (N + EXT + 2);                 // staged label rows, at most
    static constexpr int RO = TR + 2 * (N + EXT);                     // Od rows, at most (+ 1: the chain fetches one row ahead)
    static constexpr int NBAR = (RS + OM_CHUNK - 1) / OM_CHUNK;
    static constexpr int TILES = TR / ET_R;
    static constexpr size_t OFF_OD = (size_t)RS * OM_SCOLS * sizeof(uint4);
    static constexpr size_t bytes() { return OFF_OD + (size_t)(RO + 1) * 32 * sizeof(u32); }
};

__device__ __forceinline__ void om_wait(u32 bar)
{
    u32 done = 0;
    while (!done)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar) : "memory");
}

// RUNS = false: masks only (stage 02 on its own): no final bit-plane, no tile classification.  masks == NULL: no mask bytes
// (packed outputs); tap_bits != NULL: the mask as a bit-plane.  blockDim.x = 32 P; grid = column groups x planes groups x frames
// x strips, column groups fastest (the planes of a strip run together, strips top-down).
template <u32 CODE, int TAP, int TR, bool RUNS>
__global__ void __launch_bounds__(OM_PMAX * 32) fk_open_morph(const uint4 *__restrict__ slices, u32 *__restrict__ out_bits, int ws, size_t plane,
                                                             int h, int w, int K, int P, int groups, int nf, u8 *__restrict__ masks,
                                                             size_t mstride, size_t mpitch, int aligned16, u32 *__restrict__ tap_bits,
                                                             int wcols, const __grid_constant__ MorphRuns R)
{
    using L = OmLayout<CODE, TR, RUNS>;
    constexpr int N = L::N, EXT = L::EXT, TILES = L::TILES;
    extern __shared__ __align__(16) u8 smem[];
    uint4 *s_sl = reinterpret_cast<uint4 *>(smem);
    u32 *s_od = reinterpret_cast<u32 *>(smem + L::OFF_OD);
    __shared__ uint2 s_lut8[256];
    __shared__ __align__(8) unsigned long long s_bar[L::NBAR];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int wx = (int)(blockIdx.x % (unsigned)wcols);
    const int u2 = (int)(blockIdx.x / (unsigned)wcols);
    const int fg = u2 % (nf * groups), strip = u2 / (nf * groups);
    const int f = fg / groups, grp = fg - f * groups;
    const int ww = (w + 31) >> 5;
    const int c = wx * LP_COLS - 1 + lane;                     // the lane's word column = staged column lane + 1
    const int cs = c - lane - 1;                               // first staged column (c0 - 2)
    const int lo = max(0, -cs), hi = min(OM_SCOLS, ww - cs);   // staged columns inside the image
    const int y0 = strip * TR, y1 = min(h, y0 + TR);
    const int ys0 = y0 - N - EXT - 2, rs = y1 - y0 + 2 * (N + EXT + 2);    // staged rows
    const int yo0 = y0 - N - EXT, ro = y1 - y0 + 2 * (N + EXT);            // Od rows
    const u32 bar0 = (u32)__cvta_generic_to_shared(s_bar);
    // ---- 1. staging ----
    if (threadIdx.x == 0) {
        for (int j = 0; j < L::NBAR; j++) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8u * j));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint4 *src = slices + (size_t)f * plane + cs + lo;
        const u32 dst0 = (u32)__cvta_generic_to_shared(s_sl + lo), bytes = (u32)(hi - lo) * 16u;
        for (int j = 0; j * OM_CHUNK < rs; j++) {
            const int a = max(j * OM_CHUNK, -ys0), b = min(min(rs, (j + 1) * OM_CHUNK), h - ys0);     // rows inside the image
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar0 + 8u * j), "r"(b > a ? (u32)(b - a) * bytes : 0u)
                         : "memory");
            for (int r = a; r < b; r++)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(dst0 + (u32)(r * OM_SCOLS * 16)), "l"(src + (ptrdiff_t)(ys0 + r) * ws), "r"(bytes), "r"(bar0 + 8u * j)
                             : "memory");
        }
    }
    for (int i = threadIdx.x; i < rs * OM_SCOLS; i += blockDim.x) {
        const int r = i / OM_SCOLS, col = i - r * OM_SCOLS, y = ys0 + r;
        if (y < 0 || y >= h || col < lo || col >= hi) s_sl[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    expand_lut_init(s_lut8, threadIdx.x, blockDim.x);
    __syncthreads();                                           // barriers initialised, zeros and LUT written
    const bool inimg = c >= 0 && c < ww;
    const u32 colvalid = inimg ? range_mask(32 * c, w) : 0u;
    // ---- 2. Od of the rows [yo0, yo0 + ro), a segment of rows per warp ----
    {
        const int seg = (ro + P - 1) / P;
        const int ys = yo0 + wid * seg, ye = min(yo0 + ro, ys + seg);
        if (ys < ye) {
            const int ra = ys - 2 - ys0, rb = ye + 2 - ys0;    // staged rows the segment reads
            for (int j = ra / OM_CHUNK; j * OM_CHUNK < rb; j++) om_wait(bar0 + 8u * j);
            const int ce = lane == 0 ? c - 1 : c + 1;          // lanes 0 / 31: the staged column beyond the lane's
            const u32 cme = (ce >= 0 && ce < ww) ? range_mask(32 * ce, w) : 0u;
            const u32 lfix = (c == 0) ? 1u : 0u, lfixe = (ce == 0) ? 1u : 0u;                       // pixel 0 has no left neighbour
            const u32 rlast = 1u << ((w - 1) & 31);
            const u32 rfix = (c == ww - 1) ? rlast : 0u, rfixe = (ce == ww - 1) ? rlast : 0u;       // pixel w-1 has no right neighbour
            const int eidx = lane == 0 ? 0 : OM_SCOLS - 1;
            u32 sp[4] = {0u, 0u, 0u, 0u}, spe[4] = {0u, 0u, 0u, 0u};
            u32 dh1 = 0u, dh2 = 0u, dv1 = 0u, hu2 = 0u, hu3 = 0u, dhe1 = 0u, dhe2 = 0u, dve1 = 0u;
            for (int r = ys - 2; r < ye + 2; r++) {
                const uint4 *row = s_sl + (r - ys0) * OM_SCOLS;
                const uint4 v = row[lane + 1], ev = row[eidx];
                const u32 s[4] = {v.x, v.y, v.z, v.w}, e[4] = {ev.x, ev.y, ev.z, ev.w};
                const bool rin = r >= 0 && r < h;
                u32 dl = 0u, dr = 0u, dv = 0u, dle = 0u, dre = 0u, dve = 0u;
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    const u32 m = s[b], x = e[b];
                    u32 l = __shfl_up_sync(0xffffffffu, m, 1), rr = __shfl_down_sync(0xffffffffu, m, 1);
                    if (lane == 0) l = x;
                    if (lane == 31) rr = x;
                    dl |= m ^ __funnelshift_l(l, m, 1);
                    dr |= m ^ __funnelshift_r(m, rr, 1);
                    dv |= m ^ sp[b];
                    sp[b] = m;
                    // the extra column: bit 31 of lane 0's (left of m), bit 0 of lane 31's (right of m) are exact
                    dle |= x ^ (lane == 0 ? (x << 1) : __funnelshift_l(m, x, 1));
                    dre |= x ^ (lane == 0 ? __funnelshift_r(x, m, 1) : (x >> 1));
                    dve |= x ^ spe[b];
                    spe[b] = x;
                }
                dl &= ~lfix; dr &= ~rfix; dle &= ~lfixe; dre &= ~rfixe;
                const u32 dh0 = rin ? (dl | dr) : 0u, dhe0 = rin ? (dle | dre) : 0u;
                const u32 dv0 = (rin && r > 0) ? dv : 0u, dve0 = (rin && r > 0) ? dve : 0u;
                const bool yin = r - 1 >= 0 && r - 1 < h;
                const u32 U = yin ? (~(dh2 | dh1 | dh0 | dv1 | dv0) & colvalid) : 0u;
                const u32 Ue = yin ? (~(dhe2 | dhe1 | dhe0 | dve1 | dve0) & cme) : 0u;
                u32 l = __shfl_up_sync(0xffffffffu, U, 1), rr = __shfl_down_sync(0xffffffffu, U, 1);
                if (lane == 0) l = Ue;
                if (lane == 31) rr = Ue;
                const u32 hu1 = U | __funnelshift_l(l, U, 1) | __funnelshift_r(U, rr, 1);
                const int z = r - 2;
                if (z >= ys) s_od[(z - yo0) * 32 + lane] = (z >= 0 && z < h) ? ((hu3 | hu2 | hu1) & colvalid) : 0u;
                hu3 = hu2; hu2 = hu1; dh2 = dh1; dh1 = dh0; dv1 = dv0; dhe2 = dhe1; dhe1 = dhe0; dve1 = dve0;
            }
        }
    }
    __syncthreads();                                           // Od complete; no CTA-wide barrier after this point
    const int k = grp * P + wid;
    if (k >= K) return;                                        // whole warps: the list flush below is warp-wide
    // ---- 3. the chain of plane p ----
    const int p = f * K + k;
    const bool owned = inimg && lane >= 1 && lane <= LP_COLS;
    const int t_first = y0 - N - EXT;
    // running pointers of the tapped row (t - TAP) and the final row (t - N); they may point outside the planes while the row is
    // outside [0, h): never dereferenced then
    u8 *mrow = masks + (size_t)p * mstride + (ptrdiff_t)(t_first - TAP) * (ptrdiff_t)mpitch;
    u32 *trow = tap_bits + (ptrdiff_t)p * (ptrdiff_t)plane + (ptrdiff_t)(t_first - TAP) * ws + c;
    u32 *frow = out_bits + (ptrdiff_t)p * (ptrdiff_t)plane + (ptrdiff_t)(t_first - N) * ws + c;
    const u32 n0 = (k & 1) ? 0u : 0xffffffffu, n1 = (k & 2) ? 0u : 0xffffffffu, n2 = (k & 4) ? 0u : 0xffffffffu,
              n3 = (k & 8) ? 0u : 0xffffffffu;
    // pixels 32c-2, 32c-1 (top bits of the left lane's word) and 32c+32, 32c+33 (low bits of the right lane's) inside the image?
    const u32 lv = (c >= 1 && c <= ww) ? 0xC0000000u : 0u;
    const u32 rv = (c + 1 >= 0) ? (range_mask(32 * c + 32, w) & 3u) : 0u;
    constexpr int OP0 = code_op(CODE, 0);
    u32 p1[8], p2[8];
#pragma unroll
    for (int s = 0; s < 8; s++) p1[s] = p2[s] = 0u;
    // the slice words and Od of row t (zeros outside the image), read one row ahead
    const uint4 *ssl = s_sl + (t_first - ys0) * OM_SCOLS + lane + 1;
    const u32 *sod = s_od + lane;
    uint4 nsl;
    u32 nod;
    auto fetch = [&]() { nsl = *ssl; nod = *sod; ssl += OM_SCOLS; sod += 32; };
    u32 live1 = 0u, live0 = 0u;
    auto rows = [&](auto rowfix_tag, auto colfix_tag) {
        constexpr bool ROWFIX = decltype(rowfix_tag)::value, COLFIX = decltype(colfix_tag)::value;
        fetch();
        for (int t = t_first; t < y1 + N + EXT; t++) {
            u32 cur = nod & (nsl.x ^ n0) & (nsl.y ^ n1) & (nsl.z ^ n2) & (nsl.w ^ n3);          // open_k = Od & [label == k]
            const bool inside = t >= 0 && t < h;
            fetch();
            cur = oob_fix32<OP0, ROWFIX, COLFIX>(cur, colvalid, !ROWFIX || inside);
            u32 tap = 0u, fin = 0u;
            MorphChain32<CODE, 0>::template run<TAP, ROWFIX, COLFIX>(cur, p1, p2, t, h, colvalid, tap, fin);
            {
                const int r = t - TAP;
                if (r >= y0 && r < y1 && owned) {
                    if (masks) store_word_bytes_lut(mrow, 32 * c, w, tap, aligned16, s_lut8);
                    if (tap_bits) *trow = tap & colvalid;
                }
                mrow += mpitch; trow += ws;
            }
            if (!RUNS) continue;
            const int r = t - N;
            if (r >= y0 && r < y1 && owned) *frow = fin & colvalid;
            frow += ws;
            if (r >= y0 - 2 && r < y1 + 2 && (!ROWFIX || (r >= 0 && r < h))) {       // warp-uniform
                const u32 l = __shfl_up_sync(0xffffffffu, fin, 1), rr = __shfl_down_sync(0xffffffffu, fin, 1);
                const bool h1 = ((fin & colvalid) | (l & lv) | (rr & rv)) != 0u, h0 = ((~fin & colvalid) | (~l & lv) | (~rr & rv)) != 0u;
                const int q = r - y0, sub = q & 7;
                u32 m = 1u << ((q >> 3) + 1);                           // tile q / 8 (floor), biased by one
                if (sub < 2) m |= m >> 1;                                // also the 2-row halo of the tile above
                if (sub >= 6) m |= m << 1;                               // ... of the tile below
                m = (m >> 1) & ((1u << TILES) - 1u);
                if (h1) live1 |= m;
                if (h0) live0 |= m;
            }
        }
    };
    const bool rowfix = !(y0 - N - EXT >= 0 && y1 + N + EXT <= h);                                  // uniform per warp
    const bool colfix = __any_sync(0xffffffffu, colvalid != 0xffffffffu);                          // uniform per warp
    if (rowfix) { if (colfix) rows(std::true_type{}, std::true_type{}); else rows(std::true_type{}, std::false_type{}); }
    else { if (colfix) rows(std::false_type{}, std::true_type{}); else rows(std::false_type{}, std::false_type{}); }
    if (!RUNS) return;
    // ---- run lists of the sparse edge kernel (see fk_morph / fk_edge_runs for the rule and the list layout) ----
    // a run is kept in the slot of the tile where it is emitted (slot TILES: after the last tile), so that every slot index is a
    // compile-time constant and the items stay in registers
    u32 item[TILES + 1];
    const u32 live = owned ? (live1 & live0) : 0u;
    int run = 0, run_j0 = 0;
    u32 lens = 0u;                                             // 3 bits per slot: length of its run, 0 = empty
    auto emit = [&](const int slot) {
        lens |= (u32)run << (3 * slot);
        item[slot] = ((u32)p << 27) | ((u32)run_j0 << 13) | (u32)c;
        run = 0;
    };
#pragma unroll
    for (int tl = 0; tl < TILES; tl++) {
        const int ty0 = y0 + tl * ET_R;
        if (ty0 >= y1) break;
        if ((live >> tl) & 1u) {
            if (run == 0) run_j0 = ty0 / ET_R;
            if (++run == R.maxt) emit(tl);
        } else {
            if (run) emit(tl);
            if (owned && R.zero_fill) {
                const int ty1 = min(y1, ty0 + ET_R);
                for (int y = ty0; y < ty1; y++) {
                    const size_t o = (size_t)p * plane + (size_t)y * ws + c;
                    R.cbits[o] = 0u; R.sbits[o] = 0u;
                    if (R.edges) store_word_bytes(R.edges + (size_t)p * R.estride + (size_t)y * R.epitch, 32 * c, w, 0u, R.aligned16);
                }
            }
        }
    }
    if (run) emit(TILES);
#pragma unroll
    for (int nt = 1; nt <= ET_MAXT; nt++) {
        int mine = 0;
#pragma unroll
        for (int i = 0; i <= TILES; i++) mine += ((lens >> (3 * i)) & 7u) == (u32)nt;
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
#pragma unroll
        for (int i = 0; i <= TILES; i++)
            if (((lens >> (3 * i)) & 7u) == (u32)nt) R.run_items[R.off.v[nt - 1] + pos++] = item[i];
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// workspace slot 5 tail (after the tables of the first generation): [Lab cells (u32) | label nibbles | several-candidates bits]
#define WS5_LABEL_BYTES ((size_t)CELL_COUNT * sizeof(u32) + RC_NIB_BYTES + RC_MB_BYTES)

static int label_tables(omni_ctx *ctx, const AssignParams &P, u32 **cells, u8 **rtab, cudaStream_t st)
{
    SP_TRY(omni_ws_reserve(ctx, 5, WS5_BYTES + WS5_LABEL_BYTES));
    *cells = (u32 *)((u8 *)ctx->ws[5] + WS5_BYTES);
    *rtab = (u8 *)(*cells + CELL_COUNT);
    if ((ctx->table_cache || ctx->tables_hold) && ctx->cells3_valid && ctx->cells3_stream == (void *)st && ctx->cells3_K == P.K &&
        memcmp(ctx->cells3_c, P.c, sizeof(float) * 3 * P.K) == 0 && memcmp(ctx->cells3_lut, P.lut, P.K) == 0)
        return OMNI_OK;
    memcpy(ctx->cells3_c, P.c, sizeof(float) * 3 * P.K);
    memcpy(ctx->cells3_lut, P.lut, P.K);
    ctx->cells3_K = P.K; ctx->cells3_stream = (void *)st; ctx->cells3_valid = 1;
    if (!ctx->d_rgb_boxes3) {                          // centre-independent: once per context
        SP_TRY(fast_rgb_boxes(ctx, st));
        OMNI_CUDA(cudaMalloc(&ctx->d_rgb_boxes3, (size_t)RC_COUNT * sizeof(uint2)));
        KScope ks(ctx, "rgb_boxes", st);
        fk_permute_boxes3<<<RC_COUNT / 256, 256, 0, st>>>(ctx->d_rgb_boxes, (uint2 *)ctx->d_rgb_boxes3);
        OMNI_CUDA(cudaGetLastError());
    }
    KScope ks(ctx, "build_tables", st);
    fk_build_tables3<<<LP_TAB_BLOCKS, 256, 0, st>>>(P, (const uint2 *)ctx->d_rgb_boxes3, *rtab, (u32 *)(*rtab + RC_NIB_BYTES), *cells);
    OMNI_CUDA(cudaGetLastError());
    return OMNI_OK;
}

constexpr u32 CODE_L_N = mk_code(ST_DR, ST_ER);                                         // RECT close only (stage-03 morphology off)
constexpr u32 CODE_L_O = mk_code(ST_DR, ST_ER, ST_EC, ST_DC);
constexpr u32 CODE_L_C = mk_code(ST_DR, ST_ER, ST_DC, ST_EC);
constexpr u32 CODE_L_OC = mk_code(ST_DR, ST_ER, ST_EC, ST_DC, ST_DC, ST_EC);

// the dynamic shared memory of fk_open_morph may exceed the 48 KB default: raise the limit once per device and instance
template <u32 CODE, int TR, bool RUNS>
static cudaError_t open_morph_smem_attr()
{
    static unsigned done = 0;                                  // bit d: set on device d
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return cudaGetLastError();
    if (dev < 32 && ((done >> dev) & 1u)) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(fk_open_morph<CODE, 2, TR, RUNS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               (int)OmLayout<CODE, TR, RUNS>::bytes());
    if (e == cudaSuccess && dev < 32) done |= 1u << dev;
    return e;
}

static cudaError_t launch_open_morph(int kind /* -1: masks only */, const uint4 *slices, u32 *m2, const BitGeom &g, int K, int nf,
                                     u8 *masks, size_t mstride, size_t mpitch, u32 *tap_bits, const MorphRuns &R, cudaStream_t st)
{
    const int KT = nf * K;
    const int wcols = (g.ww + LP_COLS - 1) / LP_COLS;
    const int al = plane_align(masks, mstride, mpitch);
    // planes of one frame per CTA: the fewest groups of at most OM_PMAX planes, as even as possible
    const int groups = (K + OM_PMAX - 1) / OM_PMAX, P = (K + groups - 1) / groups;
    // Strip height.  A warp walks its strip row by row (+ ~20 rows of halo and pipeline): the kernel's time is about
    // waves x (rows + 20),  waves = ceil(strip-warps / resident warps).  Short strips for small grids (one wave: the shortest walk
    // wins), tall ones once there are several waves, and 56 rows where that lands the grid on a whole number of waves.
#ifdef ML_TR
    const int tr = ML_TR;
#else
    // resident warps per TR candidate (shared memory grows with TR), per CTA size
    static int resident[OM_PMAX + 1][3] = {};
    const int cands[3] = {32, 56, 64};
    if (resident[P][0] == 0) {
        int dev = 0, sms = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 1) sms = 148;
        auto occ = [&](auto kern, cudaError_t attr, size_t smem) {
            int per_sm = 0;
            if (attr != cudaSuccess || cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * P, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
            return per_sm * P * sms;
        };
        resident[P][0] = occ(fk_open_morph<CODE_L_OC, 2, 32, true>, open_morph_smem_attr<CODE_L_OC, 32, true>(), OmLayout<CODE_L_OC, 32, true>::bytes());
        resident[P][1] = occ(fk_open_morph<CODE_L_OC, 2, 56, true>, open_morph_smem_attr<CODE_L_OC, 56, true>(), OmLayout<CODE_L_OC, 56, true>::bytes());
        resident[P][2] = occ(fk_open_morph<CODE_L_OC, 2, 64, true>, open_morph_smem_attr<CODE_L_OC, 64, true>(), OmLayout<CODE_L_OC, 64, true>::bytes());
        cudaGetLastError();
    }
    int tr = 32;
    long long best = -1;
    for (int i = 0; i < 3; i++) {
        const int cand = cands[i], res = resident[P][i];
        const long long units = (long long)wcols * ((g.h + cand - 1) / cand) * KT;
        const long long cost = ((units + res - 1) / res) * (cand + 20);
        if (best < 0 || cost <= best) { best = cost; tr = cand; }
    }
#endif
    const int strips = (g.h + tr - 1) / tr;
    const dim3 grid((unsigned)((long long)wcols * groups * nf * strips)), b(32 * P);
    cudaError_t e = cudaSuccess;
#define LL2(CODE, TRV, RUNS) do { if ((e = open_morph_smem_attr<CODE, TRV, RUNS>()) != cudaSuccess) return e; \
        fk_open_morph<CODE, 2, TRV, RUNS><<<grid, b, OmLayout<CODE, TRV, RUNS>::bytes(), st>>>(slices, m2, g.ws, g.plane, g.h, g.w, K, P, groups, nf, \
                                                 masks, mstride, mpitch, al, tap_bits, wcols, R); } while (0)
#ifdef ML_TR
#define LL(CODE, RUNS) LL2(CODE, ML_TR, RUNS)
#else
#define LL(CODE, RUNS) do { if (tr == 64) LL2(CODE, 64, RUNS); else if (tr == 56) LL2(CODE, 56, RUNS); else LL2(CODE, 32, RUNS); } while (0)
#endif
    switch (kind) {
    case -1: LL(CODE_L_N, false); break;
    case 0: LL(CODE_L_N, true); break;
    case 1: LL(CODE_L_O, true); break;
    case 2: LL(CODE_L_C, true); break;
    default: LL(CODE_L_OC, true); break;
    }
#undef LL
#undef LL2
    return cudaGetLastError();
}

// Internal bit-planes of the last label-pipeline call on a ctx (valid until the next call): bit i of word c of row y = pixel 32c + i,
// rows g.ws words apart, planes g.plane words apart.
struct LabelPlanes { u32 *slices, *mask_bits, *edge_bits, *cand_bits; };

// prm == NULL: colour layers only (02_color_extract.py on its own: no stage-03 work).  d_masks / d_edges may be NULL (packed
// outputs: the bit-planes in `out` are the result).  Pf (optional): nf centre sets, frame f assigned with Pf[f] (same K as P); the
// frames then get one table build and one assignment launch each, and share every launch after the assignment.
static int label_pipeline(omni_ctx *ctx, const u8 *d_bgr, int nf, size_t frame_stride, int h, int w, size_t pitch, const AssignParams &P,
                          const omni_edge_params *prm, int low, int high, u8 *d_labels, size_t lpitch,
                          u8 *d_masks, size_t m_plane, size_t mpitch, u8 *d_edges, size_t e_plane, size_t epitch, bool want_mask_bits,
                          cudaStream_t st, LabelPlanes *out, bool skip_hysteresis = false /* bands: S and C are the result */,
                          const AssignParams *Pf = nullptr)
{
    const int K = P.K, KT = nf * K;
    const int kind = prm ? morph03_kind(prm) : -1;
    if (prm && (low < 0 || kind < 0 || prm->ksize != 3)) return OMNI_ERR_UNSUPPORTED;
    if (K > RC_MAX_K || KT > OMNI_MAX_K || !lut_below_k(P) || !edges3_sparse_ok(h, w, KT)) return OMNI_ERR_UNSUPPORTED;
    if (Pf)
        for (int f = 0; f < nf; f++)
            if (Pf[f].K != K || !lut_below_k(Pf[f])) return OMNI_ERR_UNSUPPORTED;
    const BitGeom g = make_geom(h, w);
    if ((long long)nf * h * ((w + 255) >> 8) >= (1ll << 30)) return OMNI_ERR_UNSUPPORTED;
    OMNI_CUDA(fast_tables());
    // ---- workspace (slot 4): [label slices 4 nf | M2 KT | S KT | C KT | mask bits KT]; S and C laid out as edge_pass_begin expects
    const size_t pbytes = g.plane * sizeof(u32);
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t o_sl = 0, o_m2 = al(o_sl + pbytes * 4 * nf), o_s = al(o_m2 + pbytes * KT),
                 o_c = o_s + al(pbytes * KT), o_mb = al(o_c + pbytes * KT), bits_total = al(o_mb + (want_mask_bits ? pbytes * KT : 0));
    SP_TRY(omni_ws_reserve(ctx, 4, bits_total));           // (label_ws_bytes() below states the same sizes for omni_workspace_bytes)
    u8 *b4 = (u8 *)ctx->ws[4];
    u32 *slices = (u32 *)(b4 + o_sl), *M2 = (u32 *)(b4 + o_m2), *sbits = (u32 *)(b4 + o_s), *cbits = (u32 *)(b4 + o_c);
    u32 *mbits = want_mask_bits ? (u32 *)(b4 + o_mb) : nullptr;
    if (out) { out->slices = slices; out->mask_bits = mbits; out->edge_bits = prm ? sbits : nullptr; out->cand_bits = prm ? cbits : nullptr; }
    // the zeros of the dead edge tiles: byte planes -> they ride on the assignment kernel (ZeroJob; strided planes: side stream);
    // bit-planes only -> the morphology kernel clears the candidate / strong words of its dead tiles
    MorphRuns R{};
    bool sparse = false;
    ZeroJob Z{};
    if (prm) {
        SP_TRY(edge_pass_begin(ctx, g, KT, sbits, cbits, d_edges, e_plane, epitch, st, &R, &sparse, d_edges != nullptr, d_edges ? &Z : nullptr));
        if (!sparse) return OMNI_ERR_UNSUPPORTED;
    }
    const u16 *labtab = fast_lab_table();
    if (!labtab) { omni_set_error("Lab tables not available"); return OMNI_ERR_CUDA; }
    // ---- 1. assignment -> label bit-slices: all frames in one launch, or (Pf) one table build + launch per frame ----
    if (!ctx->occ_assign_sl) {
        OMNI_CUDA(cudaFuncSetAttribute(fk_assign_slices<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, RA_SMEM + LP_ZBUF));
        OMNI_CUDA(cudaFuncSetAttribute(fk_assign_slices<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, RA_SMEM + LP_ZBUF));
        ctx->occ_assign_sl = 1;
    }
    for (int f0 = 0, n_in = Pf ? 1 : nf; f0 < nf; f0 += n_in) {
        const AssignParams &Pa = Pf ? Pf[f0] : P;
        u32 *cells = nullptr;
        u8 *rtab = nullptr;
        SP_TRY(label_tables(ctx, Pa, &cells, &rtab, st));
        const long long chunks = (long long)n_in * h * ((w + 255) >> 8);
        const int grid = (int)std::max<long long>(1, std::min<long long>(persist_blocks(ctx, 1), (chunks + RA_WARPS - 1) / RA_WARPS));
        // the zero fill rides on the first launch only, spread over that launch's chunks
        ZeroJob Za{};
        if (f0 == 0) {
            Za = Z;
            for (int z = 0; z < 2; z++)                     // units per chunk, rounded up to one store per lane
                Za.per[z] = (unsigned)(((Za.n16[z] + (unsigned long long)chunks - 1) / (unsigned long long)chunks + 31) & ~31ull);
        }
        const u8 *px = d_bgr + (size_t)f0 * frame_stride;
        u8 *lab = d_labels ? d_labels + (size_t)f0 * h * lpitch : nullptr;
        u32 *sl = slices + (size_t)f0 * 4 * g.plane;
        KScope ks(ctx, "assign_bits", st);
        if (K >= 16)
            fk_assign_slices<true><<<grid, RA_THREADS, RA_SMEM + LP_ZBUF, st>>>(px, h, w, pitch, Pa, (const uint4 *)rtab, cells, labtab, lab,
                                                                                lpitch, sl, g.ws, n_in, frame_stride, Za);
        else
            fk_assign_slices<false><<<grid, RA_THREADS, RA_SMEM + LP_ZBUF, st>>>(px, h, w, pitch, Pa, (const uint4 *)rtab, cells, labtab, lab,
                                                                                 lpitch, sl, g.ws, n_in, frame_stride, Za);
        OMNI_CUDA(cudaGetLastError());
    }
    // ---- 2. label-domain open and the rest of the morphology chain per plane, run lists for the edge kernel ----
    OMNI_LAUNCH(ctx, st, "morph_bits", launch_open_morph(kind, (const uint4 *)slices, M2, g, K, nf, d_masks, m_plane, mpitch, mbits, R, st));
    if (!prm) return OMNI_OK;
    // ---- 3. edges on the live tile runs, hysteresis ----
    if (ctx->edge_join) {                               // the side stream has cleared the output planes
        OMNI_CUDA(cudaStreamWaitEvent(st, ctx->edge_join, 0));
        ctx->edge_join = nullptr;
    }
    const int al16 = plane_align(d_edges, e_plane, epitch);
    OMNI_LAUNCH(ctx, st, "edges3_bits", launch_edges3_sparse(M2, g.ws, g.plane, h, w, KT, low, high, persist_blocks(ctx, ctx->e3s_per_sm),
                                                             sbits, cbits, d_edges, e_plane, epitch, al16, ctx->d_flags + 4,
                                                             (u32 *)ctx->ws[5] + HYST_WL_OFFSET, HY_WL_CAP, ctx->d_flags + 16,
                                                             ctx->d_flags + 20, (const u32 *)ctx->ws[6], st));
    if (skip_hysteresis) return OMNI_OK;
    return run_hysteresis(ctx, sbits, cbits, g, KT, d_edges, e_plane, epitch, st);
}

// workspace of the label pipeline for n_frames frames of h x w with K colours each (slots 4, 5, 6): omni_workspace_bytes / omni_ctx_reserve
void label_ws_bytes(int h, int w, int K, int nf, size_t out[OMNI_WS_SLOTS])
{
    const BitGeom g = make_geom(h, w);
    const int KT = nf * K;
    const size_t pbytes = g.plane * sizeof(u32);
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t o_m2 = al(pbytes * 4 * nf), o_s = al(o_m2 + pbytes * KT), o_c = o_s + al(pbytes * KT), o_mb = al(o_c + pbytes * KT);
    unsigned off[ET_MAXT];
    out[4] = std::max(out[4], al(o_mb + pbytes * KT));
    out[5] = std::max(out[5], WS5_BYTES + WS5_LABEL_BYTES);
    out[6] = std::max(out[6], edges3_run_words(h, w, KT, off) * sizeof(u32));
}

int sparse_color_edge(omni_ctx *ctx, const u8 *d_bgr, int nf, size_t frame_stride, int h, int w, size_t pitch, const AssignParams &P,
                      const omni_edge_params *prm, int low, int high, u8 *d_labels, size_t lpitch,
                      u8 *d_masks, size_t m_plane, size_t mpitch, u8 *d_edges, size_t e_plane, size_t epitch, cudaStream_t st)
{
    return label_pipeline(ctx, d_bgr, nf, frame_stride, h, w, pitch, P, prm, low, high, d_labels, lpitch, d_masks, m_plane, mpitch, d_edges,
                          e_plane, epitch, false, st, nullptr);
}

// ------------------------------------------------------------------------------------------------
// Packed outputs: the internal bit-planes re-laid for the caller (row pitch in bytes, LSB- or MSB-first bit order), per-plane
// pixel counts.  One thread per 32-pixel word.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fk_pack_planes(const u32 *__restrict__ src, int ws, size_t plane, int K, int h, int w,
                                                      u8 *__restrict__ dst, size_t dplane, size_t dpitch, int msb_first,
                                                      unsigned long long *__restrict__ counts)
{
    // grid = (row groups, planes): a warp walks rows of one plane, its lanes the words of the row (no divisions)
    const int ww = (w + 31) >> 5, rb = (w + 7) >> 3;
    const int lane = threadIdx.x & 31, k = blockIdx.y;
    const int warps = (int)gridDim.x * (int)(blockDim.x >> 5);
    if (k >= K) return;
    const u32 *sp = src + (size_t)k * plane;
    u8 *dp = dst + (size_t)k * dplane;
    const bool aligned = (((uintptr_t)dp | dpitch) & 3) == 0;
    unsigned n = 0;
    for (int y = (int)blockIdx.x * (int)(blockDim.x >> 5) + (int)(threadIdx.x >> 5); y < h; y += warps) {
        const u32 *srow = sp + (size_t)y * ws;
        u8 *row = dp + (size_t)y * dpitch;
        for (int c = lane; c < ww; c += 32) {
            const u32 word = srow[c] & range_mask(32 * c, w);
            const u32 o = msb_first ? __byte_perm(__brev(word), 0u, 0x0123) : word;
            if (aligned && 4 * c + 4 <= rb) *reinterpret_cast<u32 *>(row + 4 * c) = o;
            else
                for (int i = 0; 4 * c + i < rb && i < 4; i++) row[4 * c + i] = (u8)(o >> (8 * i));
            n += (unsigned)__popc(word);
        }
    }
    if (counts) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) n += __shfl_xor_sync(0xffffffffu, n, d);
        if (lane == 0 && n) atomicAdd(counts + k, (unsigned long long)n);
    }
}

// grid of fk_pack_planes / fk_unpack_planes: enough warps for the rows of a plane, about `blocks` CTAs in all
static inline dim3 pack_grid(int blocks, int K, int h)
{
    const int per_plane = std::max(1, std::min((h + 7) / 8, (blocks + K - 1) / K));
    return dim3((unsigned)per_plane, (unsigned)K);
}

// caller layout (pitch, bit order) -> internal bit-planes (padding words zero)
__global__ void __launch_bounds__(256) fk_unpack_planes(const u8 *__restrict__ src, size_t splane, size_t spitch, int msb_first, int K, int h, int w,
                                                        u32 *__restrict__ dst, int ws, size_t plane)
{
    const int rb = (w + 7) >> 3;
    const long long total = (long long)K * h * ws;
    for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < total; u += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(u % ws);
        const long long r2 = u / ws;
        const int y = (int)(r2 % h), k = (int)(r2 / h);
        const u8 *row = src + (size_t)k * splane + (size_t)y * spitch + 4 * c;
        u32 v = 0u;
        for (int i = 0; i < 4 && 4 * c + i < rb; i++) v |= (u32)row[i] << (8 * i);
        if (msb_first) v = __brev(__byte_perm(v, 0u, 0x0123));
        dst[(size_t)k * plane + (size_t)y * ws + c] = v & range_mask(32 * c, w);
    }
}

// launch wrappers for the other translation units (packed thinning)
cudaError_t launch_unpack_planes(const u8 *src, size_t splane, size_t spitch, int msb_first, int K, int h, int w, u32 *dst, int ws,
                                 size_t plane, int blocks, cudaStream_t st)
{
    fk_unpack_planes<<<blocks, 256, 0, st>>>(src, splane, spitch, msb_first, K, h, w, dst, ws, plane);
    return cudaGetLastError();
}
cudaError_t launch_pack_planes(const u32 *src, int ws, size_t plane, int K, int h, int w, u8 *dst, size_t dplane, size_t dpitch, int msb_first,
                               int blocks, cudaStream_t st)
{
    fk_pack_planes<<<pack_grid(blocks, K, h), 256, 0, st>>>(src, ws, plane, K, h, w, dst, dplane, dpitch, msb_first, nullptr);
    return cudaGetLastError();
}

// pixels per label from the label bit-slices (one thread per word, K ballots)
__global__ void __launch_bounds__(256) fk_count_labels_sl(const uint4 *__restrict__ slices, int ws, int h, int w, int K,
                                                          unsigned long long *__restrict__ counts)
{
    const int ww = (w + 31) >> 5;
    const long long total = (long long)h * ww;
    const int lane = threadIdx.x & 31;
    unsigned long long mine = 0;                             // lane k: pixels of label k seen by this warp
    for (long long base = ((long long)blockIdx.x * blockDim.x + threadIdx.x) - lane; base < total; base += (long long)gridDim.x * blockDim.x) {
        const long long u = base + lane;
        uint4 s = make_uint4(0u, 0u, 0u, 0u);
        u32 valid = 0u;
        if (u < total) {
            const int c = (int)(u % ww), y = (int)(u / ww);
            s = __ldg(slices + (size_t)y * ws + c);
            valid = range_mask(32 * c, w);
        }
        for (int k = 0; k < K; k++) {
            const u32 m = valid & ((k & 1) ? s.x : ~s.x) & ((k & 2) ? s.y : ~s.y) & ((k & 4) ? s.z : ~s.z) & ((k & 8) ? s.w : ~s.w);
            int n = __popc(m);
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) n += __shfl_xor_sync(0xffffffffu, n, d);
            if (lane == k) mine += (unsigned long long)n;
        }
    }
    if (lane < K && mine) atomicAdd(counts + lane, mine);
}

// Body of omni_color_edge_packed[_frames] / omni_host_color_edge_packed[_frames] (capi.cu checks the arguments): nf frames sharing
// the centre set P, or (Pf != NULL) frame f with its own set Pf[f]; plane f * K + k of the outputs is layer k of frame f.  d_* outputs are DEVICE buffers in the caller's layout; d_counts (optional,
// device, 3 * OMNI_MAX_K u64: [0..) pixels per label, [OMNI_MAX_K..) mask non-zeros, [2 OMNI_MAX_K..) edge non-zeros per plane,
// cleared here).  OMNI_ERR_UNSUPPORTED: outside the label pipeline (K > 16, edge_kernel_size != 3, ...).
int label_color_edge_packed(omni_ctx *ctx, const u8 *d_bgr, int nf, size_t frame_stride, int h, int w, size_t pitch, const AssignParams &P,
                            const omni_edge_params *prm, int low, int high, u8 *d_mask_bits, size_t mb_plane, size_t mb_pitch,
                            u8 *d_edge_bits, size_t eb_plane, size_t eb_pitch, int msb_first, unsigned long long *d_counts, cudaStream_t st,
                            const AssignParams *Pf)
{
    LabelPlanes L{};
    SP_TRY(label_pipeline(ctx, d_bgr, nf, frame_stride, h, w, pitch, P, prm, low, high, nullptr, 0, nullptr, 0, 0, nullptr, 0, 0, true, st, &L,
                          false, Pf));
    const BitGeom g = make_geom(h, w);
    const int K = P.K, KT = nf * K;
    if (d_counts) OMNI_CUDA(cudaMemsetAsync(d_counts, 0, 3 * OMNI_MAX_K * sizeof(unsigned long long), st));
    const int blocks = persist_blocks(ctx, 8);
    {
        KScope ks(ctx, "pack_planes", st);
        fk_pack_planes<<<pack_grid(blocks, KT, h), 256, 0, st>>>(L.mask_bits, g.ws, g.plane, KT, h, w, d_mask_bits, mb_plane, mb_pitch, msb_first,
                                               d_counts ? d_counts + OMNI_MAX_K : nullptr);
        OMNI_CUDA(cudaGetLastError());
    }
    if (prm) {
        KScope ks(ctx, "pack_planes", st);
        fk_pack_planes<<<pack_grid(blocks, KT, h), 256, 0, st>>>(L.edge_bits, g.ws, g.plane, KT, h, w, d_edge_bits, eb_plane, eb_pitch, msb_first,
                                               d_counts ? d_counts + 2 * OMNI_MAX_K : nullptr);
        OMNI_CUDA(cudaGetLastError());
    }
    if (d_counts)
        for (int f = 0; f < nf; f++) {
            KScope ks(ctx, "count_labels", st);
            fk_count_labels_sl<<<blocks, 256, 0, st>>>((const uint4 *)L.slices + (size_t)f * g.plane, g.ws, h, w, K, d_counts + (size_t)f * K);
            OMNI_CUDA(cudaGetLastError());
        }
    return OMNI_OK;
}

// ------------------------------------------------------------------------------------------------
// One image in HOST memory, packed outputs, row bands pipelined over three streams:
//     H2D of band b+1   |   kernels of band b   |   D2H of band b-1
// (omni_host_color_edge_packed with one frame: without bands the 50 MB in, the kernels and the 67 MB out of a 4096^2, K=16 image run
// one after the other.)
//
// A band is computed as an image of its own: rows [r0 - BD_HALO, r1 + BD_HALO) clipped to the image.  Label-domain open (2 rows),
// RECT close (2), cross open / close (4), blur 3 (1), Sobel (1) and the NMS neighbours (1) reach 11 rows, so what the band image
// gets wrong next to its artificial borders stays inside the halo; rows [r0, r1) of its mask bits and of its strong / candidate
// planes S, C are exact and are merged into full-image planes.  The hysteresis is the one global step.  Mode 1 runs it once after
// the last band and sends the edge planes then.  Mode 2 (default) runs it after every band on the prefix image [0, r1) -- a subset
// of the final result, and on pipeline data almost always equal to it -- and sends the band's edge rows at once; every word that
// holds a weak candidate is on the call's worklist (only such words can change), so after the last band one small kernel compares
// the final planes with what was sent, repairs the device copy and reports the bands that changed; those rows are sent again.
// ------------------------------------------------------------------------------------------------
#define BD_MAX_BANDS 16
#define BD_HALO 16
#define BD_FLAGS 40                   // d_flags[40..44]: flag block of the banded hysteresis ([44] = worklist length), [48] = dirty bands

__global__ void __launch_bounds__(256) fk_band_merge(const u32 *__restrict__ s_src, const u32 *__restrict__ c_src, size_t splane,
                                                     u32 *__restrict__ s_dst, u32 *__restrict__ c_dst, size_t dplane, int ws, int ww, int rows, int K,
                                                     int y0, int *wl_count, u32 *__restrict__ worklist, int wl_cap)
{
    const long long per = (long long)rows * ws, total = per * K;
    for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < total; u += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(u / per);
        const long long rem = u - (long long)k * per;
        const int c = (int)(rem % ws);
        u32 s = 0u, cd = 0u;
        if (c < ww) { s = __ldg(s_src + (size_t)k * splane + rem); cd = __ldg(c_src + (size_t)k * splane + rem); }
        const size_t o = (size_t)k * dplane + (size_t)y0 * ws + rem;
        s_dst[o] = s;
        c_dst[o] = cd;
        if (cd & ~s) {
            const int i = atomicAdd(wl_count, 1);
            if (i < wl_cap) worklist[i] = (u32)o;
        }
    }
}

struct BandRows { int n; int y[BD_MAX_BANDS + 1]; };     // band b = rows [y[b], y[b+1])

// final planes against the packed rows that were sent: repairs the device copy, dirty bit b = band b has to be sent again
__global__ void __launch_bounds__(256) fk_band_verify(const u32 *__restrict__ ebits, int ws, size_t plane, int w, const int *wl_count,
                                                      const u32 *__restrict__ worklist, int wl_cap, u8 *__restrict__ dst, size_t dplane, size_t dpitch,
                                                      int msb_first, const BandRows B, unsigned *dirty)
{
    const int n = *wl_count;
    if (n > wl_cap) {                                    // list overflowed: the caller repacks and resends everything
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(dirty, 0xffffffffu);
        return;
    }
    const int rb = (w + 7) >> 3;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const u32 o = worklist[i];
        const int k = (int)(o / plane);
        const size_t rem = o - (size_t)k * plane;
        const int y = (int)(rem / ws), c = (int)(rem - (size_t)y * ws);
        const u32 word = __ldcg(ebits + o) & range_mask(32 * c, w);
        const u32 v = msb_first ? __byte_perm(__brev(word), 0u, 0x0123) : word;
        u8 *row = dst + (size_t)k * dplane + (size_t)y * dpitch + 4 * c;
        bool diff = false;
        for (int j = 0; j < 4 && 4 * c + j < rb; j++) {
            const u8 b = (u8)(v >> (8 * j));
            if (row[j] != b) { row[j] = b; diff = true; }
        }
        if (diff) {
            int b = 0;
            while (b + 1 < B.n && y >= B.y[b + 1]) b++;
            atomicOr(dirty, 1u << b);
        }
    }
}

__global__ void __launch_bounds__(256) fk_count_bits(const u32 *__restrict__ src, int ws, size_t plane, int K, int h, int w,
                                                     unsigned long long *__restrict__ counts)
{
    const int k = blockIdx.y, ww = (w + 31) >> 5;
    const long long total = (long long)h * ww;
    unsigned long long n = 0;
    for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < total; u += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(u % ww), y = (int)(u / ww);
        n += (unsigned)__popc(__ldg(src + (size_t)k * plane + (size_t)y * ws + c) & range_mask(32 * c, w));
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) n += __shfl_xor_sync(0xffffffffu, n, d);
    if ((threadIdx.x & 31) == 0 && n) atomicAdd(counts + k, n);
    (void)K;
}

// rows [y0, y0 + rows) of K packed planes, device -> host
static cudaError_t d2h_rows(u8 *h_dst, size_t h_plane, size_t h_pitch, const u8 *d_src, size_t d_plane, size_t d_pitch, size_t rb, int y0, int rows,
                            int K, cudaStream_t st)
{
    if (h_pitch == d_pitch && d_pitch == rb)             // gap-free rows: the band of all K planes in one strided copy ("row" = a plane's band)
        return cudaMemcpy2DAsync(h_dst + (size_t)y0 * h_pitch, h_plane, d_src + (size_t)y0 * d_pitch, d_plane, (size_t)(rows - 1) * d_pitch + rb,
                                 K, cudaMemcpyDeviceToHost, st);
    for (int k = 0; k < K; k++) {
        cudaError_t e = cudaMemcpy2DAsync(h_dst + (size_t)k * h_plane + (size_t)y0 * h_pitch, h_pitch, d_src + (size_t)k * d_plane + (size_t)y0 * d_pitch,
                                          d_pitch, rb, rows, cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

struct HoldTables {                                      // the candidate tables of the first band serve the whole call
    omni_ctx *c;
    explicit HoldTables(omni_ctx *ctx) : c(ctx) {}
    ~HoldTables() { c->tables_hold = 0; }
};

static int banded_body(omni_ctx *ctx, const u8 *h_bgr, int h, int w, size_t pitch, const AssignParams &P, const omni_edge_params *prm,
                       int low, int high, u8 *h_mb, size_t mb_plane, size_t mb_pitch, u8 *h_eb, size_t eb_plane, size_t eb_pitch,
                       int msb_first, int64_t *h_counts);

int label_host_packed_banded(omni_ctx *ctx, const u8 *h_bgr, int h, int w, size_t pitch, const AssignParams &P, const omni_edge_params *prm,
                             int low, int high, u8 *h_mb, size_t mb_plane, size_t mb_pitch, u8 *h_eb, size_t eb_plane, size_t eb_pitch,
                             int msb_first, int64_t *h_counts)
{
    const int rc = banded_body(ctx, h_bgr, h, w, pitch, P, prm, low, high, h_mb, mb_plane, mb_pitch, h_eb, eb_plane, eb_pitch, msb_first, h_counts);
    // a failure in the middle leaves copies queued that read and write the caller's buffers: let them finish before the caller
    // gets the error and may free the buffers (UNSUPPORTED is decided before anything is queued)
    if (rc != OMNI_OK && rc != OMNI_ERR_UNSUPPORTED) cudaDeviceSynchronize();
    return rc;
}

static int banded_body(omni_ctx *ctx, const u8 *h_bgr, int h, int w, size_t pitch, const AssignParams &P, const omni_edge_params *prm,
                       int low, int high, u8 *h_mb, size_t mb_plane, size_t mb_pitch, u8 *h_eb, size_t eb_plane, size_t eb_pitch,
                       int msb_first, int64_t *h_counts)
{
    const int K = P.K, mode = ctx->host_bands;
    if (mode == 0 || !ctx->fast || ctx->pipeline != 1 || h < 1024 || (long long)h * w < (2ll << 20)) return OMNI_ERR_UNSUPPORTED;
    if (prm && (low < 0 || morph03_kind(prm) < 0 || prm->ksize != 3)) return OMNI_ERR_UNSUPPORTED;
    if (K > RC_MAX_K || !lut_below_k(P)) return OMNI_ERR_UNSUPPORTED;
    // ---- bands: a tall image starts with short bands (128, 256, 512 rows) so that the first results leave for the host while most
    // of the image is still arriving; the rest is split evenly (rows a multiple of 32) ----
    BandRows B{};
    {
        int y = 0;
        if (h >= 2048)
            for (int lead : {128, 256, 512}) { B.y[++B.n] = (y += lead); }
        const int left = h - y;
        int n_even = std::max(1, std::min(BD_MAX_BANDS - B.n - 1, 5));
        while (n_even > 1 && left / n_even < 256) n_even--;
        const int per = ((left + n_even - 1) / n_even + 31) & ~31;
        while (y < h) { y = std::min(h, y + per); B.y[++B.n] = y; }
    }
    const int nb = B.n;
    if (nb < 2 || nb > BD_MAX_BANDS) return OMNI_ERR_UNSUPPORTED;
    int tallest = 0;
    for (int b = 0; b < nb; b++) tallest = std::max(tallest, B.y[b + 1] - B.y[b]);
    const int hs_max = std::min(h, tallest + 2 * BD_HALO);
    if (!edges3_sparse_ok(hs_max, w, K) || !edges3_sparse_ok(h, w, K)) return OMNI_ERR_UNSUPPORTED;
    if (!ctx->bd_ready) {
        for (auto &e : ctx->bd_ev) OMNI_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        OMNI_CUDA(cudaStreamCreateWithFlags(&ctx->bd_tail, cudaStreamNonBlocking));
        ctx->bd_ready = 1;
    }
    cudaEvent_t *evH = ctx->bd_ev, *evF = ctx->bd_ev + BD_MAX_BANDS, *evB = ctx->bd_ev + 2 * BD_MAX_BANDS, evStart = ctx->bd_ev[3 * BD_MAX_BANDS],
                evEdges = ctx->bd_ev[3 * BD_MAX_BANDS + 1];
    // streams: copies in (si) and out (so); the band images (assignment .. edge kernel) alternate between this ctx and a helper ctx
    // with workspaces of its own, so that two of them are in flight (their kernels are short and latency-bound); what follows a band
    // image -- packing, the merge into the full planes, the hysteresis -- runs in band order on the tail stream tt
    omni_ctx *hx = nullptr;
    if (ctx->band_overlap && !ctx->prof_on) {
        if (!ctx->band_helper) {
            SP_TRY(omni_ctx_create(ctx->device, &ctx->band_helper));
            ctx->band_helper->edge_sparse = ctx->edge_sparse;
            ctx->band_helper->assign_rgbcell = ctx->assign_rgbcell;
        }
        hx = ctx->band_helper;
        hx->table_cache = ctx->table_cache;                  // "rebuild the tables on every call" holds for the helper's copy too
    }
    cudaStream_t sc = ctx->stream, si = ctx->pk_in, so = ctx->pk_out, tt = ctx->bd_tail;
    // ---- workspace: slot 3 = [image | packed masks | packed edges | S | C | worklist]; slots 4-6 sized for the tallest band image ----
    const BitGeom g = make_geom(h, w);
    const size_t rb = ((size_t)w + 7) / 8;
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t ip = ((size_t)w * 3 + 15) & ~(size_t)15;
    // device pitch = the host pitch when the host rows are gap-free (one strided copy per band); rows with gaps are copied row by row,
    // so that no byte outside the caller's view is written
    const size_t rb16 = (rb + 15) & ~(size_t)15;
    const size_t dpm = (mb_pitch == rb && rb % 4 == 0) ? rb : rb16, dpe = (prm && eb_pitch == rb && rb % 4 == 0) ? rb : rb16;
    const size_t pbytes = g.plane * sizeof(u32) * (size_t)K;
    const size_t o_img = 0, o_mb = al(o_img + ip * h), o_eb = al(o_mb + dpm * h * K), o_s = al(o_eb + (prm ? dpe * h * K : 0)),
                 o_c = al(o_s + (prm ? pbytes : 0)), o_wl = al(o_c + (prm ? pbytes : 0)), total = al(o_wl + HY_WL_CAP * sizeof(u32));
    SP_TRY(omni_ws_reserve(ctx, 3, total));
    {
        size_t plan[OMNI_WS_SLOTS] = {};
        label_ws_bytes(hs_max, w, K, 1, plan);
        for (int i = 4; i <= 6; i++) {
            SP_TRY(omni_ws_reserve(ctx, i, plan[i]));
            if (hx) SP_TRY(omni_ws_reserve(hx, i, plan[i]));
        }
    }
    u8 *base = (u8 *)ctx->ws[3], *d_img = base + o_img, *d_mb = base + o_mb, *d_eb = base + o_eb;
    u32 *S = (u32 *)(base + o_s), *C = (u32 *)(base + o_c), *wl = (u32 *)(base + o_wl);
    int *bflags = ctx->d_flags + BD_FLAGS;
    unsigned *d_dirty = (unsigned *)(ctx->d_flags + BD_FLAGS + 8);
    unsigned long long *dc = h_counts ? ctx->d_counts : nullptr;
    const int blocks = persist_blocks(ctx, 8);
    HoldTables hold(ctx), hold_h(hx ? hx : ctx);
    const int lag = hx ? 2 : 1;                              // the band image before this one on the same ctx
    // OMNI_B200_BAND_TRACE=1: timeline of the call on stderr (timing events: H2D done, kernels done, D2H done per band)
    static const bool trace = getenv("OMNI_B200_BAND_TRACE") != nullptr;
    std::vector<cudaEvent_t> tev;
    std::vector<int> tkind;                                  // 0 start, 1 H2D done, 2 kernels done, 3 D2H done (each in band order)
    auto tmark = [&](cudaStream_t s, int kind = 0) { if (trace) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s); tev.push_back(e); tkind.push_back(kind); } };
    // ---- start: side streams after earlier work of this ctx; all H2D bands queued at once ----
    OMNI_CUDA(cudaMemsetAsync(ctx->d_flags + BD_FLAGS, 0, 16 * sizeof(int), sc));
    if (dc) OMNI_CUDA(cudaMemsetAsync(dc, 0, 3 * OMNI_MAX_K * sizeof(unsigned long long), sc));
    tmark(sc);
    OMNI_CUDA(cudaEventRecord(evStart, sc));
    OMNI_CUDA(cudaStreamWaitEvent(si, evStart, 0));
    OMNI_CUDA(cudaStreamWaitEvent(so, evStart, 0));
    OMNI_CUDA(cudaStreamWaitEvent(tt, evStart, 0));
    if (hx) OMNI_CUDA(cudaStreamWaitEvent(hx->stream, evStart, 0));
    // the uploads are queued two bands ahead of the kernels (not all at once: the first band's kernels should not wait behind 2 nb
    // copy calls on the host); band b needs rows up to r1 + halo
    int h2d_next = 0, h2d_y = 0;
    auto queue_h2d = [&]() -> int {
        const int b = h2d_next++;
        const int ye = std::min(h, (b + 1 == nb) ? h : B.y[b + 1] + BD_HALO);
        OMNI_CUDA(cudaMemcpy2DAsync(d_img + (size_t)h2d_y * ip, ip, h_bgr + (size_t)h2d_y * pitch, pitch, (size_t)w * 3, ye - h2d_y, cudaMemcpyHostToDevice, si));
        OMNI_CUDA(cudaEventRecord(evH[b], si));
        tmark(si, 1);
        h2d_y = ye;
        return OMNI_OK;
    };
    SP_TRY(queue_h2d());
    SP_TRY(queue_h2d());
    for (int b = 0; b < nb; b++) {
        const int r0 = B.y[b], r1 = B.y[b + 1], a = std::max(0, r0 - BD_HALO), e = std::min(h, r1 + BD_HALO), hs = e - a;
        const BitGeom gs = make_geom(hs, w);
        if (h2d_next < nb) SP_TRY(queue_h2d());
        omni_ctx *cx = (hx && (b & 1)) ? hx : ctx;
        cudaStream_t sf = cx->stream;
        OMNI_CUDA(cudaStreamWaitEvent(sf, evH[b], 0));
        if (b >= lag) OMNI_CUDA(cudaStreamWaitEvent(sf, evB[b - lag], 0));      // the tail of that band has read cx's bit-planes
        LabelPlanes L{};
        int rc = label_pipeline(cx, d_img + (size_t)a * ip, 1, 0, hs, w, ip, P, prm, low, high, nullptr, 0, nullptr, 0, 0, nullptr, 0, 0, true, sf, &L, true);
        if (rc != OMNI_OK) {                                 // UNSUPPORTED can only come from the first band (same width, K, parameters)
            if (b > 0 && rc == OMNI_ERR_UNSUPPORTED) { omni_set_error("banded call: band %d outside the label pipeline", b); rc = OMNI_ERR_CUDA; }
            cudaDeviceSynchronize();
            return rc;
        }
        cx->tables_hold = 1;
        OMNI_CUDA(cudaEventRecord(evF[b], sf));
        OMNI_CUDA(cudaStreamWaitEvent(tt, evF[b], 0));
        const size_t roff = (size_t)(r0 - a) * gs.ws;
        {
            KScope ks(ctx, "pack_planes", tt);
            fk_pack_planes<<<pack_grid(blocks, K, r1 - r0), 256, 0, tt>>>(L.mask_bits + roff, gs.ws, gs.plane, K, r1 - r0, w, d_mb + (size_t)r0 * dpm, dpm * h, dpm, msb_first,
                                                   dc ? dc + OMNI_MAX_K : nullptr);
            OMNI_CUDA(cudaGetLastError());
        }
        if (dc) {
            KScope ks(ctx, "count_labels", tt);
            fk_count_labels_sl<<<blocks, 256, 0, tt>>>((const uint4 *)L.slices + roff, gs.ws, r1 - r0, w, K, dc);
            OMNI_CUDA(cudaGetLastError());
        }
        if (prm) {
            {
                KScope ks(ctx, "band_merge", tt);
                fk_band_merge<<<blocks, 256, 0, tt>>>(L.edge_bits + roff, L.cand_bits + roff, gs.plane, S, C, g.plane, g.ws, g.ww, r1 - r0, K, r0, bflags + 4,
                                                      wl, HY_WL_CAP);
                OMNI_CUDA(cudaGetLastError());
            }
            BitGeom gp = g;                                  // hysteresis of the prefix image [0, r1); the last one is the final result
            gp.h = r1;
            if (b + 1 == nb) {
                OMNI_CUDA(cudaMemsetAsync(bflags, 0, 4 * sizeof(int), tt));
                SP_TRY(run_hysteresis(ctx, S, C, gp, K, nullptr, 0, 0, tt, bflags, wl));
            } else if (mode >= 2) {
                SP_TRY(run_hysteresis_wl(ctx, S, C, gp, K, tt, bflags, wl));
            }
            if (mode >= 2) {
                KScope ks(ctx, "pack_planes", tt);
                fk_pack_planes<<<pack_grid(blocks, K, r1 - r0), 256, 0, tt>>>(S + (size_t)r0 * g.ws, g.ws, g.plane, K, r1 - r0, w, d_eb + (size_t)r0 * dpe, dpe * h, dpe, msb_first, nullptr);
                OMNI_CUDA(cudaGetLastError());
            }
        }
        OMNI_CUDA(cudaEventRecord(evB[b], tt));
        tmark(tt, 2);
        OMNI_CUDA(cudaStreamWaitEvent(so, evB[b], 0));
        OMNI_CUDA(d2h_rows(h_mb, mb_plane, mb_pitch, d_mb, dpm * h, dpm, rb, r0, r1 - r0, K, so));
        if (prm && mode >= 2) OMNI_CUDA(d2h_rows(h_eb, eb_plane, eb_pitch, d_eb, dpe * h, dpe, rb, r0, r1 - r0, K, so));
        tmark(so, 3);
    }
    // ---- after the last band ----
    if (prm) {
        if (mode >= 2) {
            KScope ks(ctx, "band_verify", tt);
            fk_band_verify<<<32, 256, 0, tt>>>(S, g.ws, g.plane, w, bflags + 4, wl, HY_WL_CAP, d_eb, dpe * h, dpe, msb_first, B, d_dirty);
            OMNI_CUDA(cudaGetLastError());
            OMNI_CUDA(cudaMemcpyAsync(ctx->h_flags + BD_FLAGS + 8, d_dirty, sizeof(unsigned), cudaMemcpyDeviceToHost, tt));
        } else {
            KScope ks(ctx, "pack_planes", tt);
            fk_pack_planes<<<pack_grid(blocks, K, h), 256, 0, tt>>>(S, g.ws, g.plane, K, h, w, d_eb, dpe * h, dpe, msb_first, nullptr);
            OMNI_CUDA(cudaGetLastError());
            OMNI_CUDA(cudaEventRecord(evEdges, tt));
            OMNI_CUDA(cudaStreamWaitEvent(so, evEdges, 0));
            OMNI_CUDA(d2h_rows(h_eb, eb_plane, eb_pitch, d_eb, dpe * h, dpe, rb, 0, h, K, so));
        }
        if (dc) {
            KScope ks(ctx, "count_bits", tt);
            fk_count_bits<<<dim3(64, K), 256, 0, tt>>>(S, g.ws, g.plane, K, h, w, dc + 2 * OMNI_MAX_K);
            OMNI_CUDA(cudaGetLastError());
        }
    }
    if (dc) OMNI_CUDA(cudaMemcpyAsync(ctx->h_counts, dc, 3 * OMNI_MAX_K * sizeof(unsigned long long), cudaMemcpyDeviceToHost, tt));
    OMNI_CUDA(cudaStreamSynchronize(tt));
    if (hx) { ctx->launches += hx->launches; hx->launches = 0; }
    ctx->last_band_resends = 0;
    if (prm && mode >= 2) {
        unsigned dirty = (unsigned)ctx->h_flags[BD_FLAGS + 8];
        if (dirty == 0xffffffffu) {                          // worklist overflow: the device copy was not repaired -- repack, send everything
            KScope ks(ctx, "pack_planes", tt);
            fk_pack_planes<<<pack_grid(blocks, K, h), 256, 0, tt>>>(S, g.ws, g.plane, K, h, w, d_eb, dpe * h, dpe, msb_first, nullptr);
            OMNI_CUDA(cudaGetLastError());
            OMNI_CUDA(cudaStreamSynchronize(tt));
            dirty = (1u << nb) - 1u;
        }
        dirty &= (1u << (nb - 1)) - 1u;                      // the last band was packed from the final planes
        for (int b = 0; b < nb; b++)
            if (dirty >> b & 1u) {
                const int r0 = B.y[b], r1 = B.y[b + 1];
                OMNI_CUDA(d2h_rows(h_eb, eb_plane, eb_pitch, d_eb, dpe * h, dpe, rb, r0, r1 - r0, K, so));
                ctx->last_band_resends++;
            }
    }
    OMNI_CUDA(cudaStreamSynchronize(so));
    if (trace) {
        float t[4][BD_MAX_BANDS] = {};
        int n[4] = {};
        for (size_t i = 1; i < tev.size(); i++) cudaEventElapsedTime(&t[tkind[i]][n[tkind[i]]++], tev[0], tev[i]);
        fprintf(stderr, "[bands] %d bands, rows:", nb);
        for (int b = 0; b < nb; b++) fprintf(stderr, " %d", B.y[b + 1] - B.y[b]);
        fprintf(stderr, "\n[bands] band: H2D done | kernels done | D2H done (ms after the start)\n");
        for (int b = 0; b < nb; b++) fprintf(stderr, "[bands] %2d: %7.3f | %7.3f | %7.3f\n", b, t[1][b], t[2][b], t[3][b]);
        for (auto e : tev) cudaEventDestroy(e);
    }
    if (h_counts)
        for (int k = 0; k < K; k++) {
            h_counts[3 * k] = (int64_t)ctx->h_counts[k];
            h_counts[3 * k + 1] = (int64_t)ctx->h_counts[OMNI_MAX_K + k];
            h_counts[3 * k + 2] = (int64_t)ctx->h_counts[2 * OMNI_MAX_K + k];
        }
    return OMNI_OK;
}
