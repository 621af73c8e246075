/*
 * omni_b200.h -- C ABI of libomni_b200.so: stages 01_resize / 02_color_extract / 03_edge_detect of
 * omnirevolve-image-processor as hand-written sm_100a CUDA kernels.
 *
 * The reference has NO FFI or operator interface on this path: its stages are Python scripts that
 * call OpenCV/NumPy and hand results to each other as PNG files (SURVEY.md 8b).  Each entry point
 * below therefore replaces a *library call site* inside a reference stage function, cited as
 * file:line relative to /root/reference/image_processor/.  The Python side that binds these
 * (ctypes) and keeps the reference's function signatures is omni_b200/stages.py; the binding a
 * reference maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *   - every function returns 0 (OMNI_OK) or a negative error code; omni_last_error_string() gives
 *     the detail for the calling thread.  There is no CPU fallback: without a CUDA device every
 *     compute entry point fails with OMNI_ERR_CUDA.
 *   - images are 8-bit, row-major, explicit pitches in BYTES.  "d_" pointers are device memory
 *     owned by the caller (e.g. torch.Tensor.data_ptr()); "h_" pointers are host memory.
 *     Small parameter blocks (centres, palettes, look-up tables) are always HOST pointers and are
 *     consumed before the call returns.
 *   - `stream` is a cudaStream_t passed as void*.  Device-pointer entry points only enqueue work,
 *     except omni_edges and omni_color_edge, which may synchronise the stream internally when a
 *     hysteresis chain crosses tile borders more often than the enqueued passes cover (rare; see
 *     DESIGN.md "hysteresis").  Host-pointer entry points (omni_host_*) copy in, compute, copy out
 *     and return after the results are in the host buffers.
 *   - an omni_ctx owns per-device scratch (work planes, resize tables, flags).  One ctx per host
 *     thread and device; calls on one ctx must not overlap.
 */
#ifndef OMNI_B200_H
#define OMNI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OMNI_ABI_VERSION 1
#define OMNI_MAX_K 32            /* colour layers per image (labels are u8; reference configs use 4..16) */
#define OMNI_MAX_BLUR_K 31       /* largest edge_kernel_size with a built-in 8.8 weight table */
#define OMNI_MAX_MORPH_K 255     /* largest edge_morph_kernel (element offsets are int8: +-127) */

#define OMNI_OK 0
#define OMNI_ERR_ARG (-1)
#define OMNI_ERR_CUDA (-2)
#define OMNI_ERR_UNSUPPORTED (-3)
#define OMNI_ERR_NOMEM (-4)

typedef struct omni_ctx omni_ctx;

/* 03_edge_detect.py:23-34 knobs, as read from config.json (config.py:31-36). */
typedef struct omni_edge_params {
    int32_t morph_k;      /* edge_morph_kernel: ELLIPSE structuring element size, 1..OMNI_MAX_MORPH_K */
    int32_t open_iters;   /* edge_morph_open_iters  (<= 0: skip; any positive count)              */
    int32_t close_iters;  /* edge_morph_close_iters (<= 0: skip; any positive count)              */
    int32_t ksize;        /* edge_kernel_size after _ensure_odd (03:9-11): odd, >= 3              */
    double low, high;     /* edge_low_threshold / edge_high_threshold exactly as given to Canny   */
} omni_edge_params;

/* ---- library / context ------------------------------------------------------------------- */
int omni_version(void);
const char *omni_last_error_string(void);
int omni_device_count(void);
/* Which implementation serves the calls: 0 = generic kernels only, 1 = fast bit-plane kernels where
 * the parameters allow (default: the fused colour+edge calls run the sparse generation -- label-domain
 * open, morphology and edges only where a plane has pixels), 2 = dense generation with the dense edge
 * kernel and the Lab-cell assignment, 3 = dense generation as shipped in round 1 (RGB-cell assignment,
 * morphology over every word, edge kernel over the live tile runs).  All give identical bytes.  For
 * tests and A/B measurements. */
int omni_set_fast_path(omni_ctx *ctx, int enable);
/* The candidate-centre tables of the colour assignment are rebuilt only when the centres change
 * (default, enable != 0: frames of a video share one centre set).  enable == 0 rebuilds them on every
 * call -- what a stream of single images with their own k-means centres pays. */
int omni_set_table_cache(omni_ctx *ctx, int enable);
/* omni_host_color_edge_packed with ONE frame of at least 1024 rows / 2 MP pipelines the image in row bands: the upload of band
 * b+1, the kernels of band b and the download of band b-1 overlap (a band is computed with 16 halo rows; the chain reaches 11).
 * mode 2 (default): a band's edge rows leave with the band, from the hysteresis of the rows seen so far; after the last band the
 * final planes are compared with what was sent and the bands that changed (a weak chain promoted from a later band) are sent again
 * -- omni_last_band_resends() says how many (-1: the last call was not banded).  mode 1: the edge planes leave after the last band.
 * mode 0: no bands (copy in, compute, copy out).  The bytes in the host buffers are the same in every mode. */
int omni_set_host_bands(omni_ctx *ctx, int mode);
int omni_last_band_resends(omni_ctx *ctx);
/* Workspaces.  The ctx owns its device scratch and grows it on demand (cudaFree + cudaMalloc inside the call that needs more).
 * omni_workspace_bytes: device bytes the fused device-resident calls (omni_color_edge, omni_color_edge_batch,
 * omni_color_edge_packed) allocate for n_frames frames of h x w pixels with K colours and edge_kernel_size ksize (0 for bad
 * arguments).  omni_ctx_reserve: allocates them now, builds the centre-independent tables and waits for that -- afterwards calls
 * of this geometry (or a smaller one) on this ctx only enqueue work: no allocation, no implicit synchronisation. */
size_t omni_workspace_bytes(int h, int w, int K, int ksize, int n_frames);
int omni_ctx_reserve(omni_ctx *ctx, int h, int w, int K, int ksize, int n_frames);
/* omni_edges / omni_host_edges check on the device that the masks are strictly {0,255} (hand-edited mask.png files need not be)
 * and wait for the answer before they choose the kernels.  enable = 1: the caller vouches for {0,255} masks (e.g. planes written
 * by omni_layer_masks): the check is skipped and omni_edges only enqueues; other mask values then give undefined edges. */
int omni_set_assume_binary_masks(omni_ctx *ctx, int enable);
int omni_ctx_create(int device, omni_ctx **out);
int omni_ctx_destroy(omni_ctx *ctx);
/* Pinned host memory for the omni_host_* entry points (pageable memory works, but is slower). */
int omni_host_alloc(size_t bytes, void **out);
int omni_host_free(void *p);

/* ---- stage 01: 01_resize.py:20  cv2.resize(img, (dw, dh), interpolation=cv2.INTER_AREA) ------ */
/* 3-channel u8, shrink only (dh <= sh, dw <= sw).  (dw, dh) come from the host expressions of
 * 01_resize.py:16-18 -- never recomputed here.  Exact for integer ratios; fractional ratios follow
 * OpenCV's float32 evaluation order (contract: +-1 LSB). */
int omni_resize_area_u8c3(omni_ctx *ctx, const uint8_t *d_src, int sh, int sw, size_t spitch,
                          uint8_t *d_dst, int dh, int dw, size_t dpitch, void *stream);
int omni_host_resize_area_u8c3(omni_ctx *ctx, const uint8_t *h_src, int sh, int sw, size_t spitch,
                               uint8_t *h_dst, int dh, int dw, size_t dpitch);

/* ---- stage 02: per-pixel colour assignment ------------------------------------------------- */
/* 02_color_extract.py:35-36,53-55 + relabel :121-127.
 * BGR u8 -> 8-bit Lab (cv2.cvtColor COLOR_BGR2LAB) -> argmin_k of the float32 squared distance to
 * h_centers[K][3] (evaluation order (d0^2+d1^2)+d2^2, every op rounded, first minimum) ->
 * label = h_lut ? h_lut[k] : k.  d_labels: u8 [h][lpitch]. */
int omni_assign_lab_f32(omni_ctx *ctx, const uint8_t *d_bgr, int h, int w, size_t pitch,
                        const float *h_centers, int K, const uint8_t *h_lut,
                        uint8_t *d_labels, size_t lpitch, void *stream);
/* process_colors.py:69-77 assign_labels: RGB u8 vs h_palette[K][3] u8, the int16 WRAP of diff*diff
 * reproduced (d2 = sum_c (int16)(diff_c*diff_c)), first minimum. */
int omni_assign_rgb_i16wrap(omni_ctx *ctx, const uint8_t *d_rgb, int h, int w, size_t pitch,
                            const uint8_t *h_palette, int K, uint8_t *d_labels, size_t lpitch, void *stream);
int omni_host_assign_rgb_i16wrap(omni_ctx *ctx, const uint8_t *h_rgb, int h, int w, size_t pitch,
                                 const uint8_t *h_palette, int K, uint8_t *h_labels, size_t lpitch);

/* 02_color_extract.py:136-154: for plane p in [0,K): (labels == p) * 255, then MORPH_OPEN x open_iters
 * and MORPH_CLOSE x close_iters with the 3x3 RECT element.  d_masks: K planes, plane p at
 * d_masks + p*plane_stride, rows mpitch bytes apart.  open/close_iters <= 0 skip that step
 * (process_colors.py:171-173 layers are the 0/0 case). */
int omni_layer_masks(omni_ctx *ctx, const uint8_t *d_labels, int h, int w, size_t lpitch, int K,
                     int open_iters, int close_iters,
                     uint8_t *d_masks, size_t plane_stride, size_t mpitch, void *stream);

/* 02_color_extract.py:82-109, the legacy swatch mode (`extraction_mode == "swatch"`; unreachable through
 * config.json because config.py:124-125 drops the key, kept for callers that build a Config by hand).
 * h_colors: K x 3 int32 exactly as `cfg.colors` holds them (each component in [0,255]); per name the swatch is
 * tried reversed (RGB -> BGR) and as-is with cv2.inRange(img, c - tol, c + tol) (bounds clipped to [0,255]), the
 * candidate with more non-zeros wins (ties: the reversed one), then RECT-3 open and close.  d_masks as in
 * omni_layer_masks.  h_choice (optional, K int32): 0 = reversed, 1 = as-is.  Synchronises the stream (the choice
 * needs the two counts).  Fast path only (no generic variant). */
int omni_swatch_masks(omni_ctx *ctx, const uint8_t *d_bgr, int h, int w, size_t pitch,
                      const int32_t *h_colors, int K, int tol,
                      uint8_t *d_masks, size_t plane_stride, size_t mpitch, int32_t *h_choice, void *stream);

/* OPT-IN replacement for the cv2.kmeans call of 02_color_extract.py:39-50 (0.26-0.29 s of host time per image): k-means++
 * seeding (3 trials per centre), Lloyd iterations until no centre moves by more than eps or max_iter, best of `attempts` by
 * compactness -- on the 8-bit Lab values of the pixels h_sample_idx[0 .. n_samples) (host array; pass the reference's own
 * `default_rng(42).choice(h*w, 200000, replace=False)`; NULL = every pixel, h*w <= 2^24).  cv2.kmeans draws from OpenCV's global
 * RNG, so its centres cannot be reproduced bit for bit; this call is deterministic for a given seed (integer accumulation): its
 * centres and compactness (sum of squared distances of the samples to their centre, *h_compactness if not NULL) equal bit for
 * bit those of oracle/kmeans_model.py, a NumPy restatement of the kernels (tests/test_gpu_kmeans_exact.py), and the compactness
 * is within 2 % of cv2.kmeans' on the same sample (tests/test_gpu_kmeans.py).  Synchronises the stream (centres go to the host). */
int omni_kmeans_lab(omni_ctx *ctx, const uint8_t *d_bgr, int h, int w, size_t pitch, const int32_t *h_sample_idx, int n_samples,
                    int K, int attempts, int max_iter, double eps, uint64_t seed, float *h_centers, double *h_compactness, void *stream);
/* The same for n_frames equally sized frames, frame f at d_bgr + f*frame_stride, each clustered on its own with the same sample
 * indices (the reference's subsample depends only on the pixel count; NULL = every pixel) and criteria.  h_centers: [n_frames][K][3];
 * h_compactness: [n_frames] or NULL.  Frame f's centres and compactness are bit-identical to omni_kmeans_lab on that frame: every
 * (frame, attempt) pair is an independent run of the same kernels, and the most compact attempt wins (ties: the lowest attempt).
 * All runs of a chunk of frames share each launch.  A chunk holds as many frames as fit in 256 MiB of workspace (per frame:
 * 4 * n_samples * (attempts + 1) bytes plus ~1.4 KB per attempt), at least one; the workspace is slot 6 of the ctx, which
 * omni_workspace_bytes / omni_ctx_reserve do not cover (k-means is not part of the fused calls' geometry).
 * Synchronises the stream. */
int omni_kmeans_lab_batch(omni_ctx *ctx, const uint8_t *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                          const int32_t *h_sample_idx, int n_samples, int K, int attempts, int max_iter, double eps,
                          uint64_t seed, float *h_centers, double *h_compactness, void *stream);

/* ---- stage 03: 03_edge_detect.py:23-34 per layer ------------------------------------------- */
/* K independent planes: ELLIPSE(morph_k) open/close -> GaussianBlur(ksize, sigma 0) -> Canny(low,
 * high) (aperture 3, L1, 8-connected hysteresis).  Output {0,255}.  In and out may not alias.
 * Masks may hold any u8 values (the reference reads arbitrary mask.png files). */
int omni_edges(omni_ctx *ctx, const uint8_t *d_masks, int K, int h, int w, size_t m_plane_stride, size_t mpitch,
               const omni_edge_params *prm,
               uint8_t *d_edges, size_t e_plane_stride, size_t epitch, void *stream);
int omni_host_edges(omni_ctx *ctx, const uint8_t *h_masks, int K, int h, int w, size_t m_plane_stride, size_t mpitch,
                    const omni_edge_params *prm,
                    uint8_t *h_edges, size_t e_plane_stride, size_t epitch);

/* ---- fused hot path: image -> K layer masks + K edge masks ---------------------------------- */
/* Equivalent to omni_assign_lab_f32 -> omni_layer_masks(1,1) -> omni_edges, i.e. everything
 * 02_color_extract.py:53-154 and 03_edge_detect.py:23-34 compute between the k-means centres and
 * the PNG writes.  d_labels may be NULL. */
int omni_color_edge(omni_ctx *ctx, const uint8_t *d_bgr, int h, int w, size_t pitch,
                    const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                    uint8_t *d_labels, size_t lpitch,
                    uint8_t *d_masks, size_t m_plane_stride, size_t mpitch,
                    uint8_t *d_edges, size_t e_plane_stride, size_t epitch, void *stream);
/* The same for n_frames equally sized frames that share ONE centre set (video frames; BASELINE config 4), frame f at
 * d_bgr + f*frame_stride.  Plane f*K + k of d_masks / d_edges is layer k of frame f (i.e. [n][K][H][W] when
 * contiguous).  Results are identical to n_frames calls of omni_color_edge; the layers of up to OMNI_MAX_K / K frames
 * go through each morphology / edge / hysteresis launch together, which is what fills the GPU on small frames. */
int omni_color_edge_batch(omni_ctx *ctx, const uint8_t *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                          const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                          uint8_t *d_masks, size_t m_plane_stride, size_t mpitch,
                          uint8_t *d_edges, size_t e_plane_stride, size_t epitch, void *stream);
/* Host-buffer form: H2D of the image, kernels, D2H of labels (optional), masks and edges.
 * h_counts (optional, 3*K int64): per plane [pixels labelled p, mask non-zeros, edge non-zeros] --
 * the numbers 02:168 and 03:38 print and palette_by_name.json records. */
int omni_host_color_edge(omni_ctx *ctx, const uint8_t *h_bgr, int h, int w, size_t pitch,
                         const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                         uint8_t *h_labels, size_t lpitch,
                         uint8_t *h_masks, size_t m_plane_stride, size_t mpitch,
                         uint8_t *h_edges, size_t e_plane_stride, size_t epitch,
                         int64_t *h_counts);

/* ---- packed outputs: 1 bit per pixel ------------------------------------------------------- */
/* mask.png / edges.png hold only 0 and 255, so a layer is one BIT per pixel: the planes leave the GPU 8 x smaller (PCIe is what
 * bounds the host-buffer calls), and the row format OMNI_BITS_MSB_FIRST is the scanline of a 1-bit greyscale PNG, which
 * cv2.imread(..., IMREAD_GRAYSCALE) decodes to the same {0,255} array (stages 04-13 read identical pixels).
 * Same computation as omni_color_edge[_batch]: n_frames frames sharing one centre set (n_frames * K <= OMNI_MAX_K), plane f * K + k =
 * layer k of frame f; rows are `pitch` bytes apart (>= ceil(w / 8)), unused bits of the last byte are 0.
 * prm == NULL: colour layers only (02_color_extract.py on its own; d_edge_bits unused).
 * h_counts (optional, 3 * n_frames * K int64: per plane [pixels labelled, mask non-zeros, edge non-zeros]) makes the device form
 * synchronise the stream. */
#define OMNI_BITS_LSB_FIRST 0    /* pixel x = bit (x & 7) of byte x >> 3       (numpy.packbits(..., bitorder="little")) */
#define OMNI_BITS_MSB_FIRST 1    /* pixel x = bit 7 - (x & 7) of byte x >> 3   (PNG bit depth 1, numpy.packbits default) */
int omni_color_edge_packed(omni_ctx *ctx, const uint8_t *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                           const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                           uint8_t *d_mask_bits, size_t mb_plane_stride, size_t mb_pitch,
                           uint8_t *d_edge_bits, size_t eb_plane_stride, size_t eb_pitch, int bit_order,
                           int64_t *h_counts, void *stream);
/* Host buffers (pinned for full speed); any number of frames: groups of OMNI_MAX_K / K frames go through the device with the H2D
 * of the next group and the D2H of the previous one overlapping the kernels.  Planes must be back to back (plane stride =
 * pitch * h).  Returns when all results are in the host buffers. */
int omni_host_color_edge_packed(omni_ctx *ctx, const uint8_t *h_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                                const float *h_centers, int K, const uint8_t *h_lut, const omni_edge_params *prm,
                                uint8_t *h_mask_bits, size_t mb_plane_stride, size_t mb_pitch,
                                uint8_t *h_edge_bits, size_t eb_plane_stride, size_t eb_pitch, int bit_order,
                                int64_t *h_counts);
/* Per-frame centres: as omni_color_edge_packed / omni_host_color_edge_packed, except that frame f is assigned with its own centres
 * h_centers + f*K*3 ([n_frames][K][3]) and LUT h_luts + f*K ([n_frames][K], or NULL: identity) -- photos or video shots with
 * palettes of their own (e.g. from omni_kmeans_lab_batch), still grouped n_frames * K <= OMNI_MAX_K planes per device pass.
 * Frame f's planes and counts are those of omni_color_edge_packed with that frame's centres and LUT.  Every frame's LUT is checked
 * before any work.  In the default family each frame of a group gets its own candidate-table build and assignment launch, and the
 * group shares the morphology / edge / hysteresis launches. */
int omni_color_edge_packed_frames(omni_ctx *ctx, const uint8_t *d_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                                  const float *h_centers, int K, const uint8_t *h_luts, const omni_edge_params *prm,
                                  uint8_t *d_mask_bits, size_t mb_plane_stride, size_t mb_pitch,
                                  uint8_t *d_edge_bits, size_t eb_plane_stride, size_t eb_pitch, int bit_order,
                                  int64_t *h_counts, void *stream);
int omni_host_color_edge_packed_frames(omni_ctx *ctx, const uint8_t *h_bgr, int n_frames, size_t frame_stride, int h, int w, size_t pitch,
                                       const float *h_centers, int K, const uint8_t *h_luts, const omni_edge_params *prm,
                                       uint8_t *h_mask_bits, size_t mb_plane_stride, size_t mb_pitch,
                                       uint8_t *h_edge_bits, size_t eb_plane_stride, size_t eb_pitch, int bit_order,
                                       int64_t *h_counts);

/* Non-zero count of each of K planes (02:157, 03:38 `np.count_nonzero`); h_counts: K int64.
 * Synchronises the stream. */
int omni_count_nonzero(omni_ctx *ctx, const uint8_t *d_planes, int K, int h, int w, size_t plane_stride, size_t pitch,
                       int64_t *h_counts, void *stream);

/* 03_edge_detect.py:93-106 paint: white BGR canvas, for plane p in order paint h_colors_bgr[p] where
 * edges > 0 (later planes overwrite earlier ones). */
int omni_edges_composite(omni_ctx *ctx, const uint8_t *d_edges, int K, int h, int w, size_t e_plane_stride, size_t epitch,
                         const uint8_t *h_colors_bgr, uint8_t *d_canvas, size_t cpitch, void *stream);

int omni_host_edges_composite(omni_ctx *ctx, const uint8_t *h_edges, int K, int h, int w, size_t e_plane_stride, size_t epitch,
                              const uint8_t *h_colors_bgr, uint8_t *h_canvas, size_t cpitch);

/* ---- stage 04 (first step): 04_find_contours.py:35-99  thinning_zhangsuen(bin_0_255, layer) ---- */
/* K independent planes; a pixel > 0 is foreground (`(roi > 0)`, 04:43).  Zhang-Suen thinning with the reference's
 * neighbour naming, both sub-steps per iteration, until an iteration deletes nothing or max_iter (the reference
 * uses 120) iterations have run.  Output {0,255} (04:97).  In and out may alias.
 * h_removed (optional, K*max_iter int32): pixels deleted from plane p in iteration i+1 at [p*max_iter + i] -- the
 * `removed=` number of the reference's progress lines (04:90-92); h_iters (optional, K int32): iterations the
 * reference's loop would have executed on plane p.  Either one makes the call synchronise the stream.
 * There is no generic (byte-plane) variant of this kernel: omni_set_fast_path does not affect it. */
int omni_thin_zhangsuen(omni_ctx *ctx, const uint8_t *d_in, int K, int h, int w, size_t in_plane_stride, size_t in_pitch,
                        int max_iter, uint8_t *d_out, size_t out_plane_stride, size_t out_pitch,
                        int32_t *h_removed, int32_t *h_iters, void *stream);
int omni_host_thin_zhangsuen(omni_ctx *ctx, const uint8_t *h_in, int K, int h, int w, size_t in_plane_stride, size_t in_pitch,
                             int max_iter, uint8_t *h_out, size_t out_plane_stride, size_t out_pitch,
                             int32_t *h_removed, int32_t *h_iters);
/* The same on planes of 1 bit per pixel, in and out (pitches in bytes, bit_order as for omni_color_edge_packed): the stage 03 -> 04
 * hand-off on the device without byte planes (the edge planes of omni_color_edge_packed go straight in).  In and out may alias. */
int omni_thin_zhangsuen_packed(omni_ctx *ctx, const uint8_t *d_bits_in, int K, int h, int w, size_t in_plane_stride, size_t in_pitch,
                               int bit_order, int max_iter, uint8_t *d_bits_out, size_t out_plane_stride, size_t out_pitch,
                               int32_t *h_removed, int32_t *h_iters, void *stream);

/* 04_find_contours.py:121-125 for all components at once: d_deg = cv2.filter2D(S, CV_8U, ones(3,3) minus the centre,
 * borderType=BORDER_CONSTANT) with S = (skeleton > 0), i.e. the number of set 8-neighbours of every pixel; d_nodes: 1 on
 * skeleton pixels with exactly one neighbour (`endpoints`, :124), 2 on skeleton pixels with three or more (`junctions`,
 * :125), 0 elsewhere.  The reference recomputes both per connected component on the whole image (its O(components x
 * pixels) term); a pixel's neighbours lie in its own component, so `deg[comp_mask == 1]` of the reference equals this
 * map there.  Either output may be NULL.  In and out may not alias. */
int omni_skeleton_degree(omni_ctx *ctx, const uint8_t *d_skel, int K, int h, int w, size_t s_plane_stride, size_t spitch,
                         uint8_t *d_deg, size_t d_plane_stride, size_t dpitch,
                         uint8_t *d_nodes, size_t n_plane_stride, size_t npitch, void *stream);

/* ---- stage 04: 04_find_contours.py:101-205  trace_centerlines(skel, layer) ------------------------ */
/* K skeleton planes (a pixel > 0 is foreground, `S = (skel > 0)`, 04:103), plane p at d_skel + p*plane_stride, rows pitch
 * bytes apart.  Replaces the whole function: cv2.connectedComponentsWithStats(S, connectivity=8) (04:108; same labels, same
 * stats), the per-component degree / endpoint / junction maps (04:117-125) and the walk (04:126-200: open paths from the
 * endpoints, then the cycles, same guards, same closing point), one component per CTA.  The polylines are the reference's:
 * same points in the same order.
 * The output size is found on the device, so the call SYNCHRONISES the stream.  h_plane_info (optional, 4*K int64): per plane
 * [total_fg, components, polylines, points].  The results stay in the ctx until the next omni_trace_centerlines /
 * omni_host_trace_centerlines / omni_[host_]centerlines_packed call on it; omni_trace_results copies them out. */
int omni_trace_centerlines(omni_ctx *ctx, const uint8_t *d_skel, int K, int h, int w, size_t plane_stride, size_t pitch,
                           int64_t *h_plane_info, void *stream);
/* Host-buffer form: h_skel is copied in, then as omni_trace_centerlines. */
int omni_host_trace_centerlines(omni_ctx *ctx, const uint8_t *h_skel, int K, int h, int w, size_t plane_stride, size_t pitch,
                                int64_t *h_plane_info);
/* Packed edge planes -> centrelines, any number of planes: plane p (layer p % K of frame p / K for a batch of frames) at
 * d_edge_bits + p*plane_stride, rows pitch bytes apart (>= ceil(w / 8); plane_stride >= pitch * h), bit_order as for
 * omni_color_edge_packed -- what omni_color_edge_packed / omni_host_color_edge_packed write.  Each plane's result equals
 * omni_thin_zhangsuen_packed(max_iter) on it, unpacked to {0,255} bytes, then omni_trace_centerlines on it: the same points,
 * polylines, component rows and h_plane_info row.  The planes go through in chunks -- at least 32 planes, more while the labels of a
 * chunk (8 bytes per 2x2 block and plane) fit 256 MiB -- each thinned (OMNI_MAX_K planes per launch), unpacked and traced with all
 * its components in one set of walk launches; so small frames fill the GPU that one frame's components leave idle.  The input is
 * not modified.  h_plane_info (optional, 4*n_planes int64) and the results as for omni_trace_centerlines: omni_trace_results copies
 * them out, planes in order.  Synchronises the stream.  Scratch: workspace slots 3 (host form), 7-10 and 12 of the ctx, grown on
 * demand and kept (slot 10, the polylines, grows with the output); omni_workspace_bytes / omni_ctx_reserve do not cover them. */
int omni_centerlines_packed(omni_ctx *ctx, const uint8_t *d_edge_bits, int n_planes, int h, int w, size_t plane_stride, size_t pitch,
                            int bit_order, int max_iter, int64_t *h_plane_info, void *stream);
/* Host-buffer form: each chunk's planes are copied in (on the ctx's own stream), then as omni_centerlines_packed; returns when the
 * results are in the ctx. */
int omni_host_centerlines_packed(omni_ctx *ctx, const uint8_t *h_edge_bits, int n_planes, int h, int w, size_t plane_stride,
                                 size_t pitch, int bit_order, int max_iter, int64_t *h_plane_info);
/* Copies the result of the last trace into caller buffers (host or device memory; any may be NULL) and returns when they hold it:
 * h_points: int32 [points][2] = (x, y) of every polyline, planes in order, components in label order (cv2's), polylines in the
 * reference's order; h_path_len: int32 [polylines], the number of points of each; h_comp: int32 [components][6] = cv2's stats row
 * (left, top, width, height, area) plus the number of polylines of the component.  Sizes: the totals of h_plane_info. */
int omni_trace_results(omni_ctx *ctx, int32_t *h_points, int32_t *h_path_len, int32_t *h_comp);

/* ---- PNG files of stages 01-03, encoded on the device --------------------------------------- */
/* Replaces the PNG encode of the files stages 01-03 write: cv2.imwrite of resized.png (01_resize.py:30), of mask.png
 * (02_color_extract.py:156) and edges.png (03_edge_detect.py:37), and of edges_composite.png in save_edges_composite
 * (03_edge_detect.py:60-111).  n images of one geometry, image i at src + i * src_stride, rows `pitch` bytes apart ->
 * n complete, standard PNG files, written back to back into the output buffer; h_sizes (n int64) receives each file's size.
 *   OMNI_PNG_GRAY1: packed rows in the OMNI_BITS_MSB_FIRST layout (ceil(w / 8) bytes used per row; unused bits of the last
 *                   byte are ignored) -> colour type 0, bit depth 1, filter 0 on every row (mask.png / edges.png).
 *   OMNI_PNG_BGR8:  u8 BGR, HWC as cv2 holds it -> colour type 2, bit depth 8, stored as RGB as cv2.imwrite stores it; each row
 *                   takes the filter None, Sub or Up with the smallest sum of |signed byte|.
 * Every file decodes (libpng, zlib) to exactly the source pixels, and the bytes depend on the pixels only: the same input gives
 * the same file whatever the stream, the ctx or the calls made before.  The image data is deflated in segments of whole
 * scanlines -- max(1, min(256, 61440 / (row bytes + 1))) rows, row bytes = ceil(w / 8) or 3 * w -- each compressed on its own
 * (run-length matches at distance 1, dynamic or fixed Huffman codes or a stored block, whichever is smallest) and written as
 * its own IDAT chunk.
 * Limits: a scanline of at most OMNI_PNG_MAX_SCANLINE bytes (filter byte included: GRAY1 w <= 491512, BGR8 w <= 20479) and
 * h <= OMNI_PNG_MAX_ROWS.  out_capacity must be at least n * omni_png_bound(h, w, format).  The output may not overlap the
 * input.  Scratch: workspace slot 11 of the ctx (grown on demand; not covered by omni_workspace_bytes).
 * The device form synchronises the stream (the sizes go to the host).  The host form copies the pixels in with one copy of the
 * span they occupy, encodes on the ctx's own stream and copies out only the compressed bytes; it returns when h_out holds them.
 * One call per stage (all K planes of a stage at once) keeps the GPU busy; calls on one ctx must not overlap. */
#define OMNI_PNG_GRAY1 0          /* packed MSB-first rows -> grey, bit depth 1 */
#define OMNI_PNG_BGR8 1           /* u8 BGR HWC            -> colour type 2, bit depth 8 */
#define OMNI_PNG_MAX_SCANLINE 61440
#define OMNI_PNG_MAX_ROWS (1 << 24)
/* Worst-case bytes of one file (every segment a stored block, plus chunk overhead); 0 for bad arguments. */
size_t omni_png_bound(int h, int w, int format);
int omni_png_encode(omni_ctx *ctx, const uint8_t *d_src, int n, size_t src_stride, int h, int w, size_t pitch, int format,
                    uint8_t *d_out, size_t out_capacity, int64_t *h_sizes, void *stream);
int omni_host_png_encode(omni_ctx *ctx, const uint8_t *h_src, int n, size_t src_stride, int h, int w, size_t pitch, int format,
                         uint8_t *h_out, size_t out_capacity, int64_t *h_sizes);

/* Diagnostics of the last omni_edges / omni_color_edge call on this ctx: number of global
 * hysteresis passes that were needed (>= 1). */
int omni_last_hysteresis_passes(omni_ctx *ctx);

/* ---- launch accounting and per-kernel timing (the reference has only ad-hoc perf_counter prints) -- */
/* Number of CUDA kernels this ctx has launched since it was created. */
long long omni_launch_count(omni_ctx *ctx);
/* on != 0: record a CUDA event pair around every kernel this ctx launches (on the launching stream).
 * Synchronises the device and clears earlier records. */
int omni_profile_enable(omni_ctx *ctx, int on);
/* Synchronises, then writes one line per kernel name, "name\tlaunches\ttotal_ms\n", in first-launch
 * order, NUL-terminated into buf; clears the records. */
int omni_profile_summary(omni_ctx *ctx, char *buf, size_t buflen);

#ifdef __cplusplus
}
#endif
#endif /* OMNI_B200_H */
