// fast_kernels.cuh -- the bit-plane fast path (fast_kernels.cu); see DESIGN.md "fast path".
#pragma once
#include "omni_internal.cuh"

void fast_ctx_release(omni_ctx *ctx);

bool fast_resize_2x_ok(const u8 *src, int sw, size_t spitch, const u8 *dst, int dw, size_t dpitch);
cudaError_t fast_resize_2x(const u8 *src, size_t spitch, u8 *dst, int dh, int dw, size_t dpitch, cudaStream_t st);
// fractional INTER_AREA with the source rectangle of each destination tile staged in shared memory;
// cudaErrorNotSupported when the ratio is too large for the staging buffer (use g_resize_area then)
cudaError_t fast_resize_frac(const u8 *src, int sh, int sw, size_t spitch, u8 *dst, int dh, int dw, size_t dpitch, const ResizeTabDev *tab,
                             cudaStream_t st);

// the same with the source rectangle staged by one TMA bulk-tensor copy and the separable two-pass form (resize_tma.cu);
// cudaErrorNotSupported when the geometry is outside it (rows not 16-byte aligned / not a whole number of words, large ratios)
cudaError_t tma_resize_frac(const u8 *src, int sh, int sw, size_t spitch, u8 *dst, int dh, int dw, size_t dpitch, const ResizeTabDev *tab,
                            cudaStream_t st);

cudaError_t fast_assign(omni_ctx *ctx, const u8 *px, int h, int w, size_t pitch, const AssignParams &P, int mode_lab,
                        u8 *labels, size_t lpitch, cudaStream_t st);

bool fast_masks_supported(int open_iters, int close_iters);
int fast_layer_masks(omni_ctx *ctx, const u8 *d_labels, int h, int w, size_t lpitch, int K, int open_iters, int close_iters,
                     u8 *d_masks, size_t plane_stride, size_t mpitch, cudaStream_t st);

bool fast_edges_supported(const omni_edge_params *prm);
// stage-03 morphology alone on the bit-plane kernels (any edge_kernel_size): masks (bytes) -> opened/closed planes (bytes).
// OMNI_ERR_UNSUPPORTED when the masks are not strictly {0,255}.
bool fast_morph03_supported(const omni_edge_params *prm);
int fast_morph03_bytes(omni_ctx *ctx, const u8 *d_masks, int K, int h, int w, size_t m_plane, size_t mpitch,
                       const omni_edge_params *prm, u8 *d_out, size_t o_plane, size_t opitch, cudaStream_t st);
// returns OMNI_ERR_UNSUPPORTED when the masks are not strictly {0,255} (caller falls back to the generic kernels)
int fast_edges(omni_ctx *ctx, const u8 *d_masks, int K, int h, int w, size_t m_plane, size_t mpitch,
               const omni_edge_params *prm, const BlurParams &bp, int low, int high,
               u8 *d_edges, size_t e_plane, size_t epitch, cudaStream_t st);
int fast_color_edge(omni_ctx *ctx, const u8 *d_bgr, int h, int w, size_t pitch, const AssignParams &P,
                    const omni_edge_params *prm, const BlurParams &bp, int low, int high,
                    u8 *d_labels, size_t lpitch, u8 *d_masks, size_t m_plane, size_t mpitch,
                    u8 *d_edges, size_t e_plane, size_t epitch, cudaStream_t st);

// edges3.cu: SIMD-in-register blur3 + Sobel + NMS on a bit-plane (strong / candidate bit-planes out).
// Dense variant: every word of every plane.  Sparse variant: fk_edge_runs lists the runs of tiles that can hold an
// edge pixel (and zero-fills the rest), the edge kernel walks only those.
#define ET_MAXT 4                         // longest run, in tiles
#define ET_R 8                            // tile rows
struct E3RunOff { unsigned v[ET_MAXT]; };  // start of the list of runs of length nt = i + 1 inside the item buffer
int edges3_pick_maxt(int h, int w, int K, int resident_warps);
size_t edges3_run_words(int h, int w, int K, unsigned off[ET_MAXT]);
bool edges3_sparse_ok(int h, int w, int K);
int edges3_sparse_blocks_per_sm();
cudaError_t launch_edge_runs(const u32 *m2, int ws, size_t plane, int h, int w, int K, u32 *sbits, u32 *cbits, u8 *edges,
                             size_t estride, size_t epitch, int aligned16, int *run_counts, u32 *run_items, int resident_warps, cudaStream_t st);
cudaError_t launch_edges3_sparse(const u32 *m2, int ws, size_t plane, int h, int w, int K, int low, int high, int grid_blocks,
                                 u32 *sbits, u32 *cbits, u8 *edges, size_t estride, size_t epitch, int aligned16, int *wl_count,
                                 u32 *worklist, int wl_cap, const int *run_counts, int *run_next, const u32 *run_items, cudaStream_t st,
                                 const u8 *blur = nullptr, size_t bstride = 0, size_t bpitch = 0);
cudaError_t launch_edges3_simd(const u32 *m2, int ws, size_t plane, int h, int w, int K, int low, int high, int sm_count,
                               u32 *sbits, u32 *cbits, u8 *edges, size_t estride, size_t epitch, int aligned16, int *wl_count, u32 *worklist, int wl_cap,
                               cudaStream_t st, const u8 *blur = nullptr, size_t bstride = 0, size_t bpitch = 0);
// GaussianBlur 5 / 7 of bit-plane masks -> u8 planes (rows 4-byte aligned, opitch >= 4 * ceil(w / 4)); edges3.cu
cudaError_t launch_blur_bits(int ksize, const u32 *m2, int ws, size_t plane, int K, int h, int w, u8 *out, size_t ostride, size_t opitch,
                             int blocks, cudaStream_t st);
bool fast_fused_supported(const omni_edge_params *prm);   // the fused colour+edge kernels: edge_kernel_size 3 only

// host-buffer fused call with H2D / kernels / D2H overlapped over row bands; OMNI_ERR_UNSUPPORTED when the parameters
// are outside the fast path.  On success all work is ordered before later work on ctx->stream.
int fast_host_color_edge(omni_ctx *ctx, const u8 *h_bgr, int h, int w, size_t pitch, const AssignParams &P,
                         const omni_edge_params *prm, int low, int high,
                         u8 *h_labels, size_t lpitch, u8 *h_masks, size_t h_mplane, size_t h_mpitch,
                         u8 *h_edges, size_t h_eplane, size_t h_epitch,
                         u8 *d_img, size_t ip, u8 *d_labels, size_t lp, u8 *d_masks, size_t mplane, size_t mp,
                         u8 *d_edges, size_t eplane, size_t ep, bool want_labels);

// stage 04 thinning (04_find_contours.py:35-99) on bit-planes; see fast_kernels.cu
int fast_thin(omni_ctx *ctx, const u8 *d_in, int K, int h, int w, size_t in_plane, size_t in_pitch, int max_iter,
              u8 *d_out, size_t out_plane, size_t out_pitch, int32_t *h_removed, int32_t *h_iters, cudaStream_t st, int packed = 0);

// stage 02 swatch mode (02_color_extract.py:82-109); h_colors: K x 3 ints as written in config.json, each in [0,255]
int fast_swatch_masks(omni_ctx *ctx, const u8 *d_bgr, int h, int w, size_t pitch, const int32_t *h_colors, int K, int tol,
                      u8 *d_masks, size_t plane_stride, size_t mpitch, int32_t *h_choice, cudaStream_t st);

// n frames sharing one centre set; their n * K layers are processed as n * K planes (n * K <= OMNI_MAX_K)
int fast_color_edge_batch(omni_ctx *ctx, const u8 *d_bgr, int n, size_t frame_stride, int h, int w, size_t pitch, const AssignParams &P,
                          const omni_edge_params *prm, int low, int high, u8 *d_masks, size_t m_plane, size_t mpitch,
                          u8 *d_edges, size_t e_plane, size_t epitch, cudaStream_t st);

// packed (1 bit per pixel) outputs of the fused call (label_pipe.cu); prm == NULL: colour layers only; Pf != NULL: frame f assigned
// with Pf[f] (nf sets, K = P.K) instead of P
int label_color_edge_packed(omni_ctx *ctx, const u8 *d_bgr, int nf, size_t frame_stride, int h, int w, size_t pitch, const AssignParams &P,
                            const omni_edge_params *prm, int low, int high, u8 *d_mask_bits, size_t mb_plane, size_t mb_pitch,
                            u8 *d_edge_bits, size_t eb_plane, size_t eb_pitch, int msb_first, unsigned long long *d_counts, cudaStream_t st,
                            const AssignParams *Pf = nullptr);
// one image in HOST memory, row bands pipelined (H2D of band b+1 | kernels of band b | D2H of band b-1); OMNI_ERR_UNSUPPORTED: not
// applicable (small image, outside the label pipeline) -- the caller takes the frame-group path
int label_host_packed_banded(omni_ctx *ctx, const u8 *h_bgr, int h, int w, size_t pitch, const AssignParams &P, const omni_edge_params *prm,
                             int low, int high, u8 *h_mask_bits, size_t mb_plane, size_t mb_pitch, u8 *h_edge_bits, size_t eb_plane,
                             size_t eb_pitch, int msb_first, int64_t *h_counts);
