// png_encode.cu -- the PNG files stages 01-03 write (mask.png / edges.png as 1-bit grey, resized.png and edges_composite.png as
// 8-bit RGB), encoded on the device.  n images of one geometry -> n complete PNG files, back to back.
//
// A file is cut into segments: runs of whole scanlines, at most PNG_SEG_MAX filtered bytes and PNG_SEG_ROWS rows each.  One
// CTA compresses one segment with no back-reference outside it (k_png_segments):
//   1. filter the rows into shared memory (GRAY1: filter 0; BGR8: None / Sub / Up by the smallest sum of |signed byte|, libpng's
//      heuristic, channels stored as RGB),
//   2. tokenise greedily: every maximal run of one byte value is a literal followed by matches at distance 1 (lengths 3..258);
//      runs cross scanlines, never the segment start.  A run belongs to the thread whose byte range holds its first byte, so the
//      tokens of a thread depend only on its range and the first run start after it (a block-wide suffix minimum),
//   3. histogram of the literal/length symbols, length-limited Huffman code (15 bits; code-length code 7 bits) built in place
//      (Moffat-Katajainen) and repaired to the limit on the length counts,
//   4. the smallest of the dynamic block, the fixed-Huffman block and one stored block; each thread emits its tokens at its
//      offset from a block-wide prefix sum of the bit counts,
//   5. an empty stored block (sync flush) byte-aligns the segment, and the segment is its own IDAT chunk: the CRC-32 of the
//      chunk and the Adler-32 parts of the filtered bytes are combined from per-thread partial results.
// k_png_files lays the chunks of each file out (prefix sum of the chunk sizes) and combines the per-segment Adler-32 values;
// k_png_place places the files back to back; k_png_copy moves every chunk into place and writes the signature, IHDR, the last
// IDAT (the final empty fixed block `03 00` and the Adler-32) and IEND.
// The bytes are a function of the pixels only: every choice is made from the data, and the atomics (histogram counts, bit ORs)
// commute.
#include "omni_internal.cuh"

#include <algorithm>
#include <limits.h>

namespace {

constexpr int PNG_T = 512;                  // threads of the segment kernel
constexpr u32 ADLER_MOD = 65521;
constexpr int NLL = 286;                    // literal/length symbols in use (0..285)

// x^(2^k) modulo the CRC-32 polynomial (reflected), k = 0..31: zlib's x2n_table
__constant__ u32 c_x2n[32] = {
    0x40000000u, 0x20000000u, 0x08000000u, 0x00800000u, 0x00008000u, 0xedb88320u, 0xb1e6b092u, 0xa06a2517u,
    0xed627daeu, 0x88d14467u, 0xd7bbfe6au, 0xec447f11u, 0x8e7ea170u, 0x6427800eu, 0x4d47bae0u, 0x09fe548fu,
    0x83852d0fu, 0x30362f1au, 0x7b5a9cc3u, 0x31fec169u, 0x9fec022au, 0x6c8dedc4u, 0x15d6874du, 0x5fde7a4eu,
    0xbad90e37u, 0x2e4e5eefu, 0x4eaba214u, 0xa8a472c0u, 0x429a969eu, 0x148d302au, 0xc40ba6d0u, 0xc4e22c3cu};

// deflate length codes 257..285: base length and extra bits (RFC 1951 3.2.5)
__constant__ u16 c_lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ u8 c_lextra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
// order of the code-length code lengths in a dynamic block header
__constant__ u8 c_clord[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct PngGeom {
    const u8 *src;
    size_t src_stride, pitch;
    int n, h, w, fmt;
    int rowbytes;                 // bytes of one source row that the file holds (GRAY1: ceil(w/8), BGR8: 3w)
    int L;                        // filtered scanline: filter byte + rowbytes
    int seg_rows, nseg;           // rows per segment, segments per file
    size_t slot;                  // scratch bytes of one segment's chunk
    u8 *scratch;                  // [n * nseg][slot]: the IDAT chunk of every segment
    u32 *seg_meta;                // [n * nseg][4]: chunk bytes, sum of the filtered bytes and weighted sum (both mod 65521), -
    unsigned long long *seg_off;  // [n * nseg]: offset of the chunk in its file
    unsigned long long *file_size, *file_off;   // [n]
    u32 *file_adler;              // [n]
    int64_t *sizes;               // [n]: file sizes for the host
    u8 *out;
};

// ---- CRC-32 / Adler-32 helpers --------------------------------------------------------------------------------------
__device__ __forceinline__ u32 multmodp(u32 a, u32 b)         // a * b modulo the polynomial; a != 0
{
    u32 m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = (b & 1) ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}

__device__ u32 x8nmodp(unsigned long long n)                   // x^(8n): shifts a CRC over n zero bytes
{
    u32 p = 1u << 31;
    int k = 3;
    while (n) {
        if (n & 1) p = multmodp(c_x2n[k & 31], p);
        n >>= 1;
        k++;
    }
    return p;
}

__device__ u32 crc_small(u32 crc, const u8 *p, int n)          // bitwise, for the few bytes of IHDR / the last IDAT
{
    crc = ~crc;
    for (int i = 0; i < n; i++) {
        crc ^= p[i];
        for (int k = 0; k < 8; k++) crc = (crc & 1) ? (crc >> 1) ^ 0xedb88320u : crc >> 1;
    }
    return ~crc;
}

__device__ __forceinline__ void put_be32(u8 *p, u32 v)
{
    p[0] = (u8)(v >> 24); p[1] = (u8)(v >> 16); p[2] = (u8)(v >> 8); p[3] = (u8)v;
}

// ---- block-wide scans (NT threads) ------------------------------------------------------------------------------------
// exclusive prefix sum; *total = the block's sum.  sh: NT / 32 elements.
template <int NT, typename T>
__device__ T blk_excl_sum(T v, T *total, T *sh)
{
    constexpr int NW = NT / 32;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    T s = v;
    for (int o = 1; o < 32; o <<= 1) { const T t = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += t; }
    if (lane == 31) sh[wid] = s;
    __syncthreads();
    if (wid == 0) {
        T x = lane < NW ? sh[lane] : T(0);
        for (int o = 1; o < 32; o <<= 1) { const T t = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += t; }
        if (lane < NW) sh[lane] = x;
    }
    __syncthreads();
    const T r = (wid ? sh[wid - 1] : T(0)) + s - v;
    *total = sh[NW - 1];
    __syncthreads();
    return r;
}

// minimum of x over the threads after this one (INT_MAX for the last).  sh: 2 * NT / 32 ints.
template <int NT>
__device__ int blk_excl_suffix_min(int x, int *sh)
{
    constexpr int NW = NT / 32;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int s = x;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_down_sync(0xffffffffu, s, o); if (lane + o < 32) s = min(s, t); }
    if (lane == 0) sh[wid] = s;
    __syncthreads();
    if (wid == 0) {
        int y = lane < NW ? sh[lane] : INT_MAX;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_down_sync(0xffffffffu, y, o); if (lane + o < 32) y = min(y, t); }
        if (lane < NW) sh[NW + lane] = y;
    }
    __syncthreads();
    const int nx = __shfl_down_sync(0xffffffffu, s, 1);
    int r = lane < 31 ? nx : INT_MAX;
    if (wid + 1 < NW) r = min(r, sh[NW + wid + 1]);
    __syncthreads();
    return r;
}

// ---- bit writer: LSB-first deflate bits into zeroed 32-bit words ---------------------------------------------------------
// The first and the last word of a writer's range may be shared with the neighbouring ranges and are ORed atomically; the
// words in between belong to this writer alone and are stored.
struct BitW {
    u32 *w;
    unsigned long long acc;
    int nb, word;
    bool first;
    __device__ void init(u32 *base, int bitpos) { w = base; word = bitpos >> 5; nb = bitpos & 31; acc = 0; first = true; }
    __device__ __forceinline__ void put(u32 v, int n)            // n <= 32, v < 2^n
    {
        acc |= (unsigned long long)v << nb;
        nb += n;
        if (nb >= 32) {
            if (first) atomicOr(w + word, (u32)acc);
            else w[word] = (u32)acc;
            first = false;
            word++;
            acc >>= 32;
            nb -= 32;
        }
    }
    __device__ void flush() { if (nb > 0) atomicOr(w + word, (u32)acc); }
};

__device__ __forceinline__ u32 rev_bits(u32 code, int len) { return __brev(code) >> (32 - len); }

// fixed Huffman code of literal/length symbol s (RFC 1951 3.2.6), bit-reversed for output
__device__ __forceinline__ void fixed_code(int s, u32 *code, int *len)
{
    if (s < 144)      { *len = 8; *code = rev_bits(0x30 + s, 8); }
    else if (s < 256) { *len = 9; *code = rev_bits(0x190 + s - 144, 9); }
    else if (s < 280) { *len = 7; *code = rev_bits(s - 256, 7); }
    else              { *len = 8; *code = rev_bits(0xc0 + s - 280, 8); }
}

// Code lengths of the used symbols, at most maxlen bits.  sorted[0..n): the used symbols by ascending (frequency, symbol), n >= 2;
// A: n ints and cnt: 33 ints of scratch; len: lengths out (entries of unused symbols are left alone).  Serial (one thread).
__device__ void huff_lengths(const u32 *freq, const int *sorted, int n, int maxlen, int *A, int *cnt, u8 *len)
{
    for (int i = 0; i < n; i++) A[i] = (int)freq[sorted[i]];
    // Moffat & Katajainen, in-place minimum-redundancy code: parent pointers, internal depths, leaf depths
    A[0] += A[1];
    int root = 0, leaf = 2;
    for (int next = 1; next < n - 1; next++) {
        if (leaf >= n || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = next; }
        else A[next] = A[leaf++];
        if (leaf >= n || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = next; }
        else A[next] += A[leaf++];
    }
    A[n - 2] = 0;
    for (int next = n - 3; next >= 0; next--) A[next] = A[A[next]] + 1;
    int avbl = 1, used = 0, dpth = 0;
    root = n - 2;
    int next = n - 1;
    while (avbl > 0) {
        while (root >= 0 && A[root] == dpth) { used++; root--; }
        while (avbl > used) { A[next--] = dpth; avbl--; }
        avbl = 2 * used; dpth++; used = 0;
    }
    // A[i]: depth of sorted[i] (non-increasing).  Clamp to maxlen, then repair the Kraft sum on the length counts: each step
    // lengthens one code that is shorter than maxlen and takes one code off maxlen (miniz' enforce_max_code_size)
    for (int l = 0; l <= 32; l++) cnt[l] = 0;
    for (int i = 0; i < n; i++) cnt[min(A[i], maxlen)]++;
    u32 total = 0;
    for (int l = maxlen; l > 0; l--) total += (u32)cnt[l] << (maxlen - l);
    while (total != (1u << maxlen)) {
        cnt[maxlen]--;
        for (int l = maxlen - 1; l > 0; l--)
            if (cnt[l]) { cnt[l]--; cnt[l + 1] += 2; break; }
        total--;
    }
    // the shortest codes go to the most frequent symbols
    int j = n;
    for (int l = 1; l <= maxlen; l++)
        for (int c = cnt[l]; c > 0; c--) len[sorted[--j]] = (u8)l;
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for output; cnt, next: 16 ints of scratch each
__device__ void huff_codes(const u8 *len, int nsym, int maxlen, int *cnt, int *next, u16 *code)
{
    for (int l = 0; l < 16; l++) cnt[l] = 0;
    for (int s = 0; s < nsym; s++) cnt[len[s]]++;
    cnt[0] = 0;
    int c = 0;
    for (int l = 1; l <= maxlen; l++) { c = (c + cnt[l - 1]) << 1; next[l] = c; }
    for (int s = 0; s < nsym; s++)
        if (len[s]) code[s] = (u16)rev_bits((u32)next[len[s]]++, len[s]);
}

enum { MODE_DYN = 0, MODE_FIXED = 1, MODE_STORED = 2 };

__global__ void __launch_bounds__(PNG_T, 2) k_png_segments(PngGeom g)
{
    extern __shared__ __align__(16) u8 sd[];                   // the segment's filtered bytes
    __shared__ u32 s_crc[256];
    __shared__ u32 s_hist[288];
    __shared__ u16 s_code[288];
    __shared__ u8 s_len[288];
    __shared__ u8 s_lsym[256];                                 // match length - 3 -> length code - 257
    __shared__ int s_sorted[288];
    __shared__ int s_A[288];
    __shared__ u32 s_rcost[PNG_SEG_ROWS * 3];                  // BGR8: filter costs of every row (None, Sub, Up)
    __shared__ u8 s_ftype[PNG_SEG_ROWS];
    __shared__ u8 s_rle[2 * 320];                              // code-length sequence: (symbol, extra value) pairs
    __shared__ u32 s_cfreq[19];
    __shared__ u8 s_clen[19];
    __shared__ u16 s_ccode[19];
    __shared__ int s_iscan[2 * PNG_T / 32];
    __shared__ u32 s_uscan[PNG_T / 32];
    __shared__ int s_work[33 + 16 + 16 + 19];                 // Huffman build scratch of thread 0
    __shared__ int s_par[8];                                   // mode, D, header bits, HLIT, HCLEN, rle items, body start

    const int tid = threadIdx.x;
    const int seg = blockIdx.x, img = seg / g.nseg, sidx = seg - img * g.nseg;
    const int y0 = sidx * g.seg_rows, rows = min(g.seg_rows, g.h - y0), L = g.L;
    const int N = rows * L;
    const u8 *src = g.src + (size_t)img * g.src_stride;
    u8 *chunk = g.scratch + (size_t)seg * g.slot;
    u8 *data = chunk + 8;
    u32 *wout = reinterpret_cast<u32 *>(data);

    for (int i = tid; i < 256; i += PNG_T) {
        u32 c = (u32)i;
        for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ 0xedb88320u : c >> 1;
        s_crc[i] = c;
        int li = 0;
        while (li < 28 && c_lbase[li + 1] <= i + 3) li++;
        s_lsym[i] = (u8)li;
    }
    for (int i = tid; i < 288; i += PNG_T) { s_hist[i] = 0; s_len[i] = 0; }
    for (int i = tid; i < 3 * rows; i += PNG_T) s_rcost[i] = 0;
    __syncthreads();

    // ---- 1. filter ----
    if (g.fmt == OMNI_PNG_GRAY1) {
        const u8 lastmask = (g.w & 7) ? (u8)(0xff00u >> (g.w & 7)) : (u8)0xff;   // unused bits of the last byte -> 0
        for (int i = tid; i < N; i += PNG_T) {
            const int r = i / L, j = i - r * L;
            u8 v = 0;
            if (j) {
                v = src[(size_t)(y0 + r) * g.pitch + (j - 1)];
                if (j == g.rowbytes) v &= lastmask;
            }
            sd[i] = v;
        }
    } else {
        const int rb = g.rowbytes;
        auto raw = [&](int y, int j) -> int {                  // byte j of row y in RGB order
            const int x = j / 3, c = j - 3 * x;
            return src[(size_t)y * g.pitch + 3 * x + 2 - c];
        };
        {
            int cur_r = -1;
            u32 c0 = 0, c1 = 0, c2 = 0;
            for (int i = tid; i < rows * rb; i += PNG_T) {
                const int r = i / rb, j = i - r * rb, y = y0 + r;
                if (r != cur_r) {
                    if (cur_r >= 0) { atomicAdd(&s_rcost[3 * cur_r], c0); atomicAdd(&s_rcost[3 * cur_r + 1], c1); atomicAdd(&s_rcost[3 * cur_r + 2], c2); }
                    cur_r = r; c0 = c1 = c2 = 0;
                }
                const int a = raw(y, j);
                const u8 fs = (u8)(a - (j >= 3 ? raw(y, j - 3) : 0)), fu = (u8)(a - (y > 0 ? raw(y - 1, j) : 0));
                c0 += min(a, 256 - a); c1 += min((int)fs, 256 - fs); c2 += min((int)fu, 256 - fu);
            }
            if (cur_r >= 0) { atomicAdd(&s_rcost[3 * cur_r], c0); atomicAdd(&s_rcost[3 * cur_r + 1], c1); atomicAdd(&s_rcost[3 * cur_r + 2], c2); }
        }
        __syncthreads();
        for (int r = tid; r < rows; r += PNG_T) {              // smallest sum; ties: None, then Sub, then Up
            const u32 a = s_rcost[3 * r], b = s_rcost[3 * r + 1], c = s_rcost[3 * r + 2];
            s_ftype[r] = (b < a && b <= c) ? 1 : (c < a && c < b) ? 2 : 0;
        }
        __syncthreads();
        for (int i = tid; i < N; i += PNG_T) {
            const int r = i / L, j = i - r * L, y = y0 + r, t = s_ftype[r];
            if (j == 0) { sd[i] = (u8)t; continue; }
            const int a = raw(y, j - 1);
            const int p = t == 1 ? (j - 1 >= 3 ? raw(y, j - 4) : 0) : t == 2 ? (y > 0 ? raw(y - 1, j - 1) : 0) : 0;
            sd[i] = (u8)(a - p);
        }
    }
    __syncthreads();

    // ---- 2. run starts and Adler-32 parts of this thread's byte range ----
    const int C = (N + PNG_T - 1) / PNG_T;
    const int c0 = min(N, tid * C), c1 = min(N, c0 + C);
    int first = INT_MAX;
    unsigned long long as = 0, aw = 0;
    for (int p = c0; p < c1; p++) {
        const u32 v = sd[p];
        if (first == INT_MAX && (p == 0 || sd[p - 1] != v)) first = p;
        as += v;
        aw += (unsigned long long)(c1 - p) * v;
    }
    const int nxt = min(N, blk_excl_suffix_min<PNG_T>(first, s_iscan));
    u32 tot_s, tot_w;
    blk_excl_sum<PNG_T, u32>((u32)(as % ADLER_MOD), &tot_s, s_uscan);
    blk_excl_sum<PNG_T, u32>((u32)((aw + (unsigned long long)(N - c1) * as) % ADLER_MOD), &tot_w, s_uscan);

    // every maximal run [p, e) of one byte value: a literal, then matches at distance 1 (258 at most; a remainder of 1 or 2
    // after a 258 is avoided by shortening that match) -- or up to two more literals for runs shorter than 4
    auto walk = [&](auto &&lit, auto &&match) {
        int p = first;
        while (p < c1) {
            const u8 v = sd[p];
            int q = p + 1;
            while (q < c1 && sd[q] == v) q++;
            const int e = q < c1 ? q : nxt;
            lit(v);
            int m = e - p - 1;
            if (m < 3) {
                for (; m > 0; m--) lit(v);
            } else {
                while (m > 0) {
                    int t = min(m, 258);
                    if (m - t > 0 && m - t < 3) t = m - 3;
                    match(t);
                    m -= t;
                }
            }
            p = q;
        }
    };

    // ---- 3. histogram ----
    walk([&](int v) { atomicAdd(&s_hist[v], 1u); }, [&](int t) { atomicAdd(&s_hist[257 + s_lsym[t - 3]], 1u); });
    if (tid == 0) atomicAdd(&s_hist[256], 1u);                 // end of block
    __syncthreads();

    // ---- 4. code lengths: rank the used symbols by (frequency, symbol) ----
    {
        const bool used = tid < NLL && s_hist[tid] > 0;
        if (used) {
            const u32 f = s_hist[tid];
            int rank = 0;
            for (int j = 0; j < NLL; j++) {
                const u32 fj = s_hist[j];
                rank += (fj > 0 && (fj < f || (fj == f && j < tid))) ? 1 : 0;
            }
            s_sorted[rank] = tid;
        }
    }
    const int n_used = __syncthreads_count(tid < NLL && s_hist[tid] > 0);   // >= 2: end of block and the first byte

    if (tid == 0) {
        int *cnt = s_work, *nxc = s_work + 33, *cnt2 = s_work + 49, *cs = s_work + 65;
        huff_lengths(s_hist, s_sorted, n_used, 15, s_A, cnt, s_len);
        int hlit = 257;
        for (int s = NLL - 1; s >= 257; s--) if (s_len[s]) { hlit = s + 1; break; }
        // the code-length sequence: hlit literal/length lengths, then the two distance codes (lengths 1, 1: only code 0, distance
        // 1, is used, and a complete two-code tree keeps every inflater happy), run-length coded with 16 / 17 / 18
        for (int i = 0; i < 19; i++) { s_cfreq[i] = 0; s_clen[i] = 0; }
        int nitems = 0, i = 0;
        const int total = hlit + 2;
        auto lenat = [&](int k) -> int { return k < hlit ? s_len[k] : 1; };
        while (i < total) {
            const int v = lenat(i);
            int r = 1;
            while (i + r < total && lenat(i + r) == v) r++;
            if (v == 0) {
                int left = r;
                while (left >= 11) { const int t = min(left, 138); s_rle[2 * nitems] = 18; s_rle[2 * nitems + 1] = (u8)(t - 11); nitems++; s_cfreq[18]++; left -= t; }
                if (left >= 3) { s_rle[2 * nitems] = 17; s_rle[2 * nitems + 1] = (u8)(left - 3); nitems++; s_cfreq[17]++; left = 0; }
                while (left > 0) { s_rle[2 * nitems] = 0; s_rle[2 * nitems + 1] = 0; nitems++; s_cfreq[0]++; left--; }
            } else {
                s_rle[2 * nitems] = (u8)v; s_rle[2 * nitems + 1] = 0; nitems++; s_cfreq[v]++;
                int left = r - 1;
                while (left >= 3) { const int t = min(left, 6); s_rle[2 * nitems] = 16; s_rle[2 * nitems + 1] = (u8)(t - 3); nitems++; s_cfreq[16]++; left -= t; }
                while (left > 0) { s_rle[2 * nitems] = (u8)v; s_rle[2 * nitems + 1] = 0; nitems++; s_cfreq[v]++; left--; }
            }
            i += r;
        }
        // code-length code: at least two symbols (a one-symbol code would be incomplete)
        int nc = 0;
        for (int s = 0; s < 19; s++) if (s_cfreq[s]) cs[nc++] = s;
        if (nc < 2) { const int extra = cs[0] == 0 ? 1 : 0; cs[nc++] = extra; if (cs[0] > cs[1]) { const int t = cs[0]; cs[0] = cs[1]; cs[1] = t; } }
        for (int a = 1; a < nc; a++) {                         // insertion sort by (frequency, symbol)
            const int s = cs[a];
            int b = a - 1;
            while (b >= 0 && (s_cfreq[cs[b]] > s_cfreq[s] || (s_cfreq[cs[b]] == s_cfreq[s] && cs[b] > s))) { cs[b + 1] = cs[b]; b--; }
            cs[b + 1] = s;
        }
        huff_lengths(s_cfreq, cs, nc, 7, s_A, cnt, s_clen);
        huff_codes(s_clen, 19, 7, cnt2, nxc, s_ccode);
        int hclen = 19;
        while (hclen > 4 && s_clen[c_clord[hclen - 1]] == 0) hclen--;
        long long hbits = 5 + 5 + 4 + 3 * hclen;
        for (int k = 0; k < nitems; k++) {
            const int s = s_rle[2 * k];
            hbits += s_clen[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
        }
        long long bdyn = 0, bfix = 0, nmatch = 0;
        for (int s = 0; s < NLL; s++) {
            const long long f = s_hist[s];
            if (!f) continue;
            u32 fc; int fl;
            fixed_code(s, &fc, &fl);
            bdyn += f * s_len[s];
            bfix += f * fl;
            if (s >= 257) { const int ex = c_lextra[s - 257]; bdyn += f * ex; bfix += f * ex; nmatch += f; }
        }
        bdyn += nmatch;                                        // 1-bit distance code
        bfix += 5 * nmatch;                                    // 5-bit fixed distance code
        const long long base = sidx == 0 ? 16 : 0;             // zlib header in front of the first segment
        const long long d_dyn = (base + 3 + hbits + bdyn + 3 + 7) / 8 + 4;
        const long long d_fix = (base + 3 + bfix + 3 + 7) / 8 + 4;
        const long long d_st = base / 8 + 5 + N + 5;
        int mode = MODE_DYN;
        long long D = d_dyn;
        if (d_fix < D) { mode = MODE_FIXED; D = d_fix; }
        if (d_st < D) { mode = MODE_STORED; D = d_st; }
        if (mode == MODE_DYN) {
            huff_codes(s_len, NLL, 15, cnt2, nxc, s_code);
        } else if (mode == MODE_FIXED) {
            for (int s = 0; s < NLL; s++) { u32 fc; int fl; fixed_code(s, &fc, &fl); s_code[s] = (u16)fc; s_len[s] = (u8)fl; }
        }
        s_par[0] = mode; s_par[1] = (int)D; s_par[2] = (int)hbits; s_par[3] = hlit; s_par[4] = hclen; s_par[5] = nitems;
        s_par[6] = (int)(base + 3 + (mode == MODE_DYN ? hbits : 0));
    }
    __syncthreads();
    const int mode = s_par[0], D = s_par[1];
    const int base_bytes = sidx == 0 ? 2 : 0;

    // ---- 5. emit ----
    for (int i = tid; i < (D + 3) / 4; i += PNG_T) wout[i] = 0u;
    __syncthreads();
    if (mode == MODE_STORED) {
        if (tid == 0) {
            if (sidx == 0) { data[0] = 0x78; data[1] = 0x01; }
            u8 *h = data + base_bytes;                         // BFINAL 0, BTYPE 00, padded; LEN, NLEN
            h[0] = 0; h[1] = (u8)N; h[2] = (u8)(N >> 8); h[3] = (u8)~N; h[4] = (u8)(~N >> 8);
            u8 *f = data + base_bytes + 5 + N;                 // empty stored block
            f[0] = 0; f[1] = 0; f[2] = 0; f[3] = 0xff; f[4] = 0xff;
        }
        for (int i = tid; i < N; i += PNG_T) data[base_bytes + 5 + i] = sd[i];
    } else {
        const int dbits = mode == MODE_DYN ? 1 : 5;
        int nbits = 0;
        walk([&](int v) { nbits += s_len[v]; },
             [&](int t) { const int li = s_lsym[t - 3]; nbits += s_len[257 + li] + c_lextra[li] + dbits; });
        int body_bits;
        const int off = blk_excl_sum<PNG_T, int>(nbits, &body_bits, s_iscan);
        const int body0 = s_par[6];
        BitW bw;
        bw.init(wout, body0 + off);
        walk([&](int v) { bw.put(s_code[v], s_len[v]); },
             [&](int t) {
                 const int li = s_lsym[t - 3];
                 bw.put(s_code[257 + li], s_len[257 + li]);
                 if (c_lextra[li]) bw.put((u32)(t - c_lbase[li]), c_lextra[li]);
                 bw.put(0u, dbits);
             });
        if (nbits) bw.flush();
        if (tid == 0) {
            BitW hw;
            hw.init(wout, 0);
            if (sidx == 0) { hw.put(0x78, 8); hw.put(0x01, 8); }
            hw.put(mode == MODE_DYN ? 4u : 2u, 3);             // BFINAL 0, BTYPE 10 (dynamic) / 01 (fixed)
            if (mode == MODE_DYN) {
                hw.put((u32)(s_par[3] - 257), 5);
                hw.put(1u, 5);                                 // HDIST - 1: two distance codes
                hw.put((u32)(s_par[4] - 4), 4);
                for (int k = 0; k < s_par[4]; k++) hw.put(s_clen[c_clord[k]], 3);
                for (int k = 0; k < s_par[5]; k++) {
                    const int s = s_rle[2 * k];
                    hw.put(s_ccode[s], s_clen[s]);
                    if (s >= 16) hw.put(s_rle[2 * k + 1], s == 16 ? 2 : s == 17 ? 3 : 7);
                }
            }
            hw.flush();
            BitW ew;                                           // end of block
            ew.init(wout, body0 + body_bits);
            ew.put(s_code[256], s_len[256]);
            ew.flush();
        }
        __syncthreads();
        if (tid == 0) {                                        // empty stored block: 3 zero bits, pad, 00 00 FF FF
            const int e = body0 + body_bits + s_len[256] + 3;
            u8 *f = data + (e + 7) / 8;
            f[0] = 0; f[1] = 0; f[2] = 0xff; f[3] = 0xff;
        }
    }
    __syncthreads();

    // ---- 6. CRC-32 of the chunk ("IDAT" + data) from per-thread pieces ----
    {
        const int CC = (D + PNG_T - 1) / PNG_T;
        const int b0 = min(D, tid * CC), b1 = min(D, b0 + CC);
        u32 c = 0xffffffffu;
        for (int i = b0; i < b1; i++) c = s_crc[(c ^ data[i]) & 255] ^ (c >> 8);
        c = ~c;
        u32 term = (b1 > b0) ? multmodp(x8nmodp((unsigned long long)(D - b1)), c) : 0u;
        for (int o = 16; o > 0; o >>= 1) term ^= __shfl_xor_sync(0xffffffffu, term, o);
        if ((tid & 31) == 0) s_uscan[tid >> 5] = term;
        __syncthreads();
        if (tid == 0) {
            u32 x = 0;
            for (int k = 0; k < PNG_T / 32; k++) x ^= s_uscan[k];
            const u8 tag[4] = {'I', 'D', 'A', 'T'};
            const u32 crc = multmodp(x8nmodp((unsigned long long)D), crc_small(0, tag, 4)) ^ x;
            put_be32(chunk, (u32)D);
            chunk[4] = 'I'; chunk[5] = 'D'; chunk[6] = 'A'; chunk[7] = 'T';
            put_be32(data + D, crc);
            u32 *m = g.seg_meta + 4 * (size_t)seg;
            m[0] = (u32)(D + 12); m[1] = tot_s % ADLER_MOD; m[2] = tot_w % ADLER_MOD; m[3] = (u32)mode;
        }
    }
}

// one CTA per file: chunk offsets (after signature + IHDR), file size, Adler-32 of all filtered bytes
constexpr int PNG_FT = 256;
__global__ void __launch_bounds__(PNG_FT) k_png_files(PngGeom g)
{
    __shared__ unsigned long long s_u[PNG_FT / 32];
    const int img = blockIdx.x;
    const size_t s0 = (size_t)img * g.nseg;
    unsigned long long run = 33, sum_a = 0, sum_b = 0;
    const unsigned long long n_tot = (unsigned long long)g.h * g.L;
    for (int b = 0; b < g.nseg; b += PNG_FT) {
        const int s = b + threadIdx.x;
        unsigned long long sz = 0, ta = 0, tb = 0;
        if (s < g.nseg) {
            const u32 *m = g.seg_meta + 4 * (s0 + s);
            sz = m[0];
            const unsigned long long after = (unsigned long long)(g.h - min(g.h, (s + 1) * g.seg_rows)) * g.L;
            ta = m[1];
            tb = (m[2] + (after % ADLER_MOD) * m[1]) % ADLER_MOD;
        }
        unsigned long long tot;
        const unsigned long long off = blk_excl_sum<PNG_FT, unsigned long long>(sz, &tot, s_u);
        if (s < g.nseg) g.seg_off[s0 + s] = run + off;
        run += tot;
        unsigned long long t2;
        blk_excl_sum<PNG_FT, unsigned long long>(ta, &t2, s_u);
        sum_a += t2;
        blk_excl_sum<PNG_FT, unsigned long long>(tb, &t2, s_u);
        sum_b += t2;
    }
    if (threadIdx.x == 0) {
        const u32 a = (u32)((1 + sum_a) % ADLER_MOD), bb = (u32)((n_tot % ADLER_MOD + sum_b) % ADLER_MOD);
        g.file_adler[img] = (bb << 16) | a;
        g.file_size[img] = run + 18 + 12;                      // last IDAT (6 data bytes) + IEND
    }
}

// one CTA: files back to back
constexpr int PNG_PT = 1024;
__global__ void __launch_bounds__(PNG_PT) k_png_place(PngGeom g)
{
    __shared__ unsigned long long s_u[PNG_PT / 32];
    unsigned long long run = 0;
    for (int b = 0; b < g.n; b += PNG_PT) {
        const int i = b + threadIdx.x;
        const unsigned long long sz = i < g.n ? g.file_size[i] : 0;
        unsigned long long tot;
        const unsigned long long off = blk_excl_sum<PNG_PT, unsigned long long>(sz, &tot, s_u);
        if (i < g.n) { g.file_off[i] = run + off; g.sizes[i] = (int64_t)sz; }
        run += tot;
    }
}

// one CTA per segment: its chunk into place; the first segment of a file adds signature + IHDR, the last one the final IDAT + IEND
constexpr int PNG_CT = 256;
__global__ void __launch_bounds__(PNG_CT) k_png_copy(PngGeom g)
{
    const int seg = blockIdx.x, img = seg / g.nseg, sidx = seg - img * g.nseg;
    u8 *file = g.out + g.file_off[img];
    const u8 *src = g.scratch + (size_t)seg * g.slot;
    const u32 n = g.seg_meta[4 * (size_t)seg];
    u8 *dst = file + g.seg_off[seg];
    for (u32 i = threadIdx.x; i < n; i += PNG_CT) dst[i] = src[i];
    if (threadIdx.x == 0 && sidx == 0) {
        const u8 sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
        for (int i = 0; i < 8; i++) file[i] = sig[i];
        u8 ih[17] = {'I', 'H', 'D', 'R'};
        put_be32(ih + 4, (u32)g.w);
        put_be32(ih + 8, (u32)g.h);
        ih[12] = g.fmt == OMNI_PNG_GRAY1 ? 1 : 8;              // bit depth
        ih[13] = g.fmt == OMNI_PNG_GRAY1 ? 0 : 2;              // colour type: grey / RGB
        ih[14] = ih[15] = ih[16] = 0;                          // deflate, adaptive filtering, no interlace
        put_be32(file + 8, 13);
        for (int i = 0; i < 17; i++) file[12 + i] = ih[i];
        put_be32(file + 29, crc_small(0, ih, 17));
    }
    if (threadIdx.x == 32 && sidx == g.nseg - 1) {
        u8 *t = file + g.file_size[img] - 30;
        u8 id[10] = {'I', 'D', 'A', 'T', 0x03, 0x00};          // final empty fixed-Huffman block, then the Adler-32
        put_be32(id + 6, g.file_adler[img]);
        put_be32(t, 6);
        for (int i = 0; i < 10; i++) t[4 + i] = id[i];
        put_be32(t + 14, crc_small(0, id, 10));
        const u8 iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xae, 0x42, 0x60, 0x82};
        for (int i = 0; i < 12; i++) t[18 + i] = iend[i];
    }
}

struct PngPlan {
    int rowbytes, L, seg_rows, nseg;
    size_t slot;
};

PngPlan png_plan(int h, int w, int fmt)
{
    PngPlan p;
    p.rowbytes = fmt == OMNI_PNG_GRAY1 ? (w + 7) / 8 : 3 * w;
    p.L = p.rowbytes + 1;
    p.seg_rows = png_segment_rows(w, fmt);
    p.nseg = (h + p.seg_rows - 1) / p.seg_rows;
    // chunk length + type, zlib header, stored block header, data, empty stored block, CRC, word rounding of the bit writer
    p.slot = ((size_t)8 + 2 + 5 + (size_t)p.seg_rows * p.L + 5 + 4 + 4 + 15) / 16 * 16;
    return p;
}

}  // namespace

int png_segment_rows(int w, int fmt)
{
    const int L = (fmt == OMNI_PNG_GRAY1 ? (w + 7) / 8 : 3 * w) + 1;
    return std::max(1, std::min(PNG_SEG_ROWS, PNG_SEG_MAX / L));
}

size_t png_file_bound(int h, int w, int fmt)
{
    const PngPlan p = png_plan(h, w, fmt);
    // signature + IHDR (33), zlib header (2), last IDAT (18), IEND (12); per segment a chunk (12), a stored block header (5) and
    // the empty stored block (5)
    return (size_t)65 + (size_t)22 * p.nseg + (size_t)h * p.L;
}

int png_encode_run(omni_ctx *ctx, const u8 *d_src, int n, size_t src_stride, int h, int w, size_t pitch, int fmt, u8 *d_out,
                   int64_t *h_sizes, cudaStream_t st)
{
    const PngPlan p = png_plan(h, w, fmt);
    const size_t ns = (size_t)n * p.nseg;
    auto a16 = [](size_t b) { return (b + 15) / 16 * 16; };
    const size_t b_chunks = a16(ns * p.slot), b_meta = a16(ns * 16), b_soff = a16(ns * 8), b_file = a16((size_t)n * 8);
    {
        const int rc = omni_ws_reserve(ctx, 11, b_chunks + b_meta + b_soff + 4 * b_file);
        if (rc != OMNI_OK) return rc;
    }
    u8 *ws = (u8 *)ctx->ws[11];
    PngGeom g;
    g.src = d_src; g.src_stride = src_stride; g.pitch = pitch;
    g.n = n; g.h = h; g.w = w; g.fmt = fmt;
    g.rowbytes = p.rowbytes; g.L = p.L; g.seg_rows = p.seg_rows; g.nseg = p.nseg; g.slot = p.slot;
    g.scratch = ws;
    g.seg_meta = (u32 *)(ws + b_chunks);
    g.seg_off = (unsigned long long *)(ws + b_chunks + b_meta);
    g.file_size = (unsigned long long *)(ws + b_chunks + b_meta + b_soff);
    g.file_off = g.file_size + b_file / 8;
    g.file_adler = (u32 *)(g.file_off + b_file / 8);
    g.sizes = (int64_t *)((u8 *)g.file_adler + b_file);
    g.out = d_out;
    // the segment buffer is dynamic shared memory beyond the 48 KB default (a per-device attribute: set on every call)
    OMNI_CUDA(cudaFuncSetAttribute(k_png_segments, cudaFuncAttributeMaxDynamicSharedMemorySize, PNG_SEG_MAX));
    const size_t smem = (size_t)p.seg_rows * p.L;
    OMNI_LAUNCH(ctx, st, "png_segments", (k_png_segments<<<(unsigned)ns, PNG_T, smem, st>>>(g), cudaGetLastError()));
    OMNI_LAUNCH(ctx, st, "png_files", (k_png_files<<<n, PNG_FT, 0, st>>>(g), cudaGetLastError()));
    OMNI_LAUNCH(ctx, st, "png_place", (k_png_place<<<1, PNG_PT, 0, st>>>(g), cudaGetLastError()));
    OMNI_LAUNCH(ctx, st, "png_copy", (k_png_copy<<<(unsigned)ns, PNG_CT, 0, st>>>(g), cudaGetLastError()));
    OMNI_CUDA(cudaMemcpyAsync(h_sizes, g.sizes, (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    OMNI_CUDA(cudaStreamSynchronize(st));
    return OMNI_OK;
}
