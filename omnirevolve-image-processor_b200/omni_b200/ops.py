"""Device- and host-level operators over libomni_b200.so.

PyTorch is used only as the owner of device memory and streams; every computation below is a
call through the C ABI (omni_b200.capi) into the hand-written CUDA kernels.  Each operator cites
the reference call site it replaces (paths relative to /root/reference/image_processor/).
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass

import sys

import numpy as np

from . import capi


class _LazyTorch:
    """`torch` is imported on first use: the host-buffer operators (what the drop-in stage scripts call) need only
    ctypes + NumPy, and a stage process should not pay the ~2 s torch import the reference's 0.5 s stages never had."""

    def __getattr__(self, name):
        import torch as _t
        globals()["torch"] = _t
        return getattr(_t, name)


torch = _LazyTorch()


@dataclass
class EdgeConfig:
    """The stage-03 knobs of config.json (config.py:31-36), defaults as in the reference."""
    low: float = 50
    high: float = 150
    ksize: int = 3
    morph_k: int = 3
    open_iters: int = 1
    close_iters: int = 1

    @staticmethod
    def ensure_odd(n) -> int:
        """03_edge_detect.py:9-11."""
        n = max(3, int(n))
        return n if n % 2 == 1 else n + 1

    @classmethod
    def from_cfg(cls, cfg) -> "EdgeConfig":
        """Reads the keys exactly as process_color does (03:23-34)."""
        return cls(low=cfg.edge_low_threshold, high=cfg.edge_high_threshold, ksize=cfg.edge_kernel_size,
                   morph_k=max(1, int(getattr(cfg, "edge_morph_kernel", 3))),
                   open_iters=int(getattr(cfg, "edge_morph_open_iters", 1)),
                   close_iters=int(getattr(cfg, "edge_morph_close_iters", 1)))

    def to_c(self) -> capi.EdgeParams:
        return capi.EdgeParams(int(self.morph_k), int(self.open_iters), int(self.close_iters),
                               self.ensure_odd(self.ksize), float(self.low), float(self.high))


@dataclass
class TraceResult:
    """trace_centerlines of one skeleton plane (04_find_contours.py:101-205)."""
    paths: list            # int32 (n,1,2) arrays of (x, y): the reference's polylines in its order
    stats: np.ndarray      # int32 [components, 5]: cv2.connectedComponentsWithStats' stats rows 1.. (left, top, width, height, area)
    polylines: np.ndarray  # int32 [components]: polylines of each component
    total_fg: int          # skeleton pixels of the plane


def _f32p(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _u8p(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8)) if a is not None else None


def _centers_luts(centers, lut, n: int):
    """centers [K,3] (one set for all n frames) or [n,K,3] (one per frame), lut [K] / [n,K] or None ->
    (ctr f32, lut u8 | None, K, per_frame)."""
    c = np.asarray(centers, dtype=np.float32)
    lut_a = None if lut is None else np.ascontiguousarray(lut, dtype=np.uint8)
    if c.ndim != 3:
        ctr = np.ascontiguousarray(c).reshape(-1, 3)
        return ctr, lut_a, ctr.shape[0], False
    if c.shape[0] != n or c.shape[2] != 3:
        raise ValueError(f"per-frame centers must be [n_frames={n}, K, 3], got {list(c.shape)}")
    K = c.shape[1]
    if lut_a is not None and lut_a.shape != (n, K):
        raise ValueError(f"per-frame lut must be [n_frames={n}, K={K}], got {list(lut_a.shape)}")
    return np.ascontiguousarray(c), lut_a, K, True


def _check_img(t: torch.Tensor, ch: int | None):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.uint8):
        raise TypeError("expected a CUDA uint8 tensor")
    if ch is not None and (t.dim() != 3 or t.shape[2] != ch or t.stride(2) != 1 or t.stride(1) != ch):
        raise ValueError(f"expected an HxWx{ch} tensor with packed pixels")
    if ch is None and (t.dim() != 2 or t.stride(1) != 1):
        raise ValueError("expected an HxW tensor with unit column stride")


def _check_planes(t: torch.Tensor):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.uint8 and t.dim() == 3 and t.stride(2) == 1):
        raise TypeError("expected a CUDA uint8 [K,H,W] tensor with unit column stride")


class Engine:
    """One omni_ctx on one device.  Not thread-safe; use one per host thread (get_engine does)."""

    def __init__(self, device: int | None = None):
        L = capi.lib()
        if L.omni_device_count() <= 0:
            raise capi.OmniError(-2, "no CUDA device visible; libomni_b200 has no CPU fallback")
        if device is None:                  # torch's current device when torch is in use, else device 0
            device = sys.modules["torch"].cuda.current_device() if "torch" in sys.modules else 0
        self.device = int(device)
        h = C.c_void_p()
        capi.check(L.omni_ctx_create(self.device, C.byref(h)))
        self._h, self._L = h, L

    def close(self):
        if getattr(self, "_h", None):
            self._L.omni_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_fast_path(self, enable):
        """False/0: generic kernels; True/1: bit-plane fast path (default: sparse generation of the fused call);
        2: dense generation with the dense edge kernel; 3: dense generation as shipped in round 1."""
        capi.check(self._L.omni_set_fast_path(self._h, int(enable)))

    def kmeans_lab(self, bgr: torch.Tensor, K: int, sample_idx=None, attempts: int = 3, max_iter: int = 40, eps: float = 0.5,
                   seed: int = 0):
        """Opt-in device k-means of the Lab centres (omni_kmeans_lab): (centers f32 [K,3], compactness).  sample_idx: the pixel
        indices to cluster (the reference's seeded 200k subsample), None = every pixel."""
        _check_img(bgr, 3)
        ctr = np.empty((K, 3), np.float32)
        comp = C.c_double(0.0)
        if sample_idx is None:
            idx_p, n = None, 0
        else:
            idx = np.ascontiguousarray(sample_idx, dtype=np.int32)
            idx_p, n = idx.ctypes.data_as(C.POINTER(C.c_int32)), idx.size
        capi.check(self._L.omni_kmeans_lab(self._h, bgr.data_ptr(), bgr.shape[0], bgr.shape[1], bgr.stride(0), idx_p, n, K, attempts,
                                           max_iter, float(eps), int(seed), _f32p(ctr), C.byref(comp), self._stream()))
        return ctr, float(comp.value)

    def kmeans_lab_batch(self, frames: torch.Tensor, K: int, sample_idx=None, attempts: int = 3, max_iter: int = 40, eps: float = 0.5,
                         seed: int = 0):
        """kmeans_lab for every frame of frames [n,H,W,3] (CUDA uint8) in shared launches (omni_kmeans_lab_batch): (centers f32
        [n,K,3], compactness f64 [n]), frame f bit-identical to kmeans_lab(frames[f], ...).  sample_idx: shared by all frames."""
        if frames.dim() != 4 or frames.shape[3] != 3 or frames.dtype != torch.uint8 or not frames.is_cuda or frames.stride(3) != 1 \
                or frames.stride(2) != 3:
            raise ValueError("frames must be a CUDA uint8 tensor [n,H,W,3] with packed pixels")
        n, h, w = frames.shape[:3]
        ctr = np.empty((n, K, 3), np.float32)
        comp = np.empty(n, np.float64)
        if sample_idx is None:
            idx_p, ns = None, 0
        else:
            idx = np.ascontiguousarray(sample_idx, dtype=np.int32)
            idx_p, ns = idx.ctypes.data_as(C.POINTER(C.c_int32)), idx.size
        capi.check(self._L.omni_kmeans_lab_batch(self._h, frames.data_ptr(), n, frames.stride(0), h, w, frames.stride(1), idx_p, ns, K,
                                                 attempts, max_iter, float(eps), int(seed), _f32p(ctr),
                                                 comp.ctypes.data_as(C.POINTER(C.c_double)), self._stream()))
        return ctr, comp

    def reserve(self, h: int, w: int, K: int, ksize: int = 3, n_frames: int = 1) -> int:
        """Allocate the workspaces of the fused calls for this geometry now (omni_ctx_reserve); returns their size in bytes."""
        capi.check(self._L.omni_ctx_reserve(self._h, h, w, K, ksize, n_frames))
        return int(self._L.omni_workspace_bytes(h, w, K, ksize, n_frames))

    def assume_binary_masks(self, enable: bool):
        """True: `edges` skips the device-side {0,255} check and its wait (the caller vouches for the masks)."""
        capi.check(self._L.omni_set_assume_binary_masks(self._h, 1 if enable else 0))

    def set_table_cache(self, enable: bool):
        """False: rebuild the candidate-centre tables on every call (single images with their own centres)."""
        capi.check(self._L.omni_set_table_cache(self._h, 1 if enable else 0))

    def set_host_bands(self, mode: int):
        """Row-band pipelining of `host_color_edge_packed` with one frame: 0 off, 1 edge planes after the last band, 2 (default)
        edge rows with their band + resend of the bands a later band changed.  Same bytes in every mode."""
        capi.check(self._L.omni_set_host_bands(self._h, int(mode)))

    def last_band_resends(self) -> int:
        """Bands of the last banded call whose edge rows went out twice (-1: the last call was not banded)."""
        return int(self._L.omni_last_band_resends(self._h))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- stage 01 ------------------------------------------------------------------------------
    def resize_area(self, src: torch.Tensor, new_w: int, new_h: int, out: torch.Tensor | None = None) -> torch.Tensor:
        """01_resize.py:20 cv2.resize(img, (new_w,new_h), INTER_AREA); HxWx3 u8, shrink only."""
        _check_img(src, 3)
        if out is None:
            out = torch.empty((new_h, new_w, 3), dtype=torch.uint8, device=src.device)
        _check_img(out, 3)
        capi.check(self._L.omni_resize_area_u8c3(self._h, src.data_ptr(), src.shape[0], src.shape[1], src.stride(0),
                                                 out.data_ptr(), new_h, new_w, out.stride(0), self._stream()))
        return out

    # ---- stage 02 ------------------------------------------------------------------------------
    def assign_lab(self, bgr: torch.Tensor, centers, lut=None, out: torch.Tensor | None = None) -> torch.Tensor:
        """02_color_extract.py:35-36,53-55 (+ relabel lut of :121-127): u8 labels [H,W]."""
        _check_img(bgr, 3)
        ctr = np.ascontiguousarray(centers, dtype=np.float32).reshape(-1, 3)
        lut_a = None if lut is None else np.ascontiguousarray(lut, dtype=np.uint8)
        if out is None:
            out = torch.empty(bgr.shape[:2], dtype=torch.uint8, device=bgr.device)
        _check_img(out, None)
        capi.check(self._L.omni_assign_lab_f32(self._h, bgr.data_ptr(), bgr.shape[0], bgr.shape[1], bgr.stride(0),
                                               _f32p(ctr), ctr.shape[0], _u8p(lut_a), out.data_ptr(), out.stride(0),
                                               self._stream()))
        return out

    def assign_rgb_i16wrap(self, rgb: torch.Tensor, palette, out: torch.Tensor | None = None) -> torch.Tensor:
        """process_colors.py:69-77 assign_labels (int16 wrap reproduced): u8 labels [H,W]."""
        _check_img(rgb, 3)
        pal = np.ascontiguousarray(palette, dtype=np.uint8).reshape(-1, 3)
        if out is None:
            out = torch.empty(rgb.shape[:2], dtype=torch.uint8, device=rgb.device)
        capi.check(self._L.omni_assign_rgb_i16wrap(self._h, rgb.data_ptr(), rgb.shape[0], rgb.shape[1], rgb.stride(0),
                                                   _u8p(pal), pal.shape[0], out.data_ptr(), out.stride(0), self._stream()))
        return out

    def layer_masks(self, labels: torch.Tensor, K: int, open_iters: int = 1, close_iters: int = 1,
                    out: torch.Tensor | None = None) -> torch.Tensor:
        """02_color_extract.py:136-154: K planes (labels==p)*255 -> RECT-3 open -> close.  [K,H,W] u8."""
        _check_img(labels, None)
        h, w = labels.shape
        if out is None:
            out = torch.empty((K, h, w), dtype=torch.uint8, device=labels.device)
        _check_planes(out)
        capi.check(self._L.omni_layer_masks(self._h, labels.data_ptr(), h, w, labels.stride(0), K, open_iters, close_iters,
                                            out.data_ptr(), out.stride(0), out.stride(1), self._stream()))
        return out

    def swatch_masks(self, bgr: torch.Tensor, colors, tol: int = 30, out: torch.Tensor | None = None, with_choice: bool = False):
        """02_color_extract.py:82-109 (swatch mode): K masks [K,H,W] u8 {0,255}; colors: K x 3 as in cfg.colors."""
        _check_img(bgr, 3)
        col = np.ascontiguousarray(np.asarray(colors, dtype=np.int32).reshape(-1, 3))
        K = col.shape[0]
        h, w = bgr.shape[:2]
        if out is None:
            out = torch.empty((K, h, w), dtype=torch.uint8, device=bgr.device)
        _check_planes(out)
        choice = np.zeros(K, np.int32)
        i32p = C.POINTER(C.c_int32)
        capi.check(self._L.omni_swatch_masks(self._h, bgr.data_ptr(), h, w, bgr.stride(0), col.ctypes.data_as(i32p), K, int(tol),
                                             out.data_ptr(), out.stride(0), out.stride(1), choice.ctypes.data_as(i32p), self._stream()))
        return (out, choice) if with_choice else out

    # ---- stage 03 ------------------------------------------------------------------------------
    def edges(self, masks: torch.Tensor, ec: EdgeConfig, out: torch.Tensor | None = None) -> torch.Tensor:
        """03_edge_detect.py:23-34 on K mask planes at once.  [K,H,W] u8 {0,255}."""
        _check_planes(masks)
        K, h, w = masks.shape
        if out is None:
            out = torch.empty((K, h, w), dtype=torch.uint8, device=masks.device)
        _check_planes(out)
        p = ec.to_c()
        capi.check(self._L.omni_edges(self._h, masks.data_ptr(), K, h, w, masks.stride(0), masks.stride(1), C.byref(p),
                                      out.data_ptr(), out.stride(0), out.stride(1), self._stream()))
        return out

    # ---- fused hot path ---------------------------------------------------------------------------
    def color_edge(self, bgr: torch.Tensor, centers, lut, ec: EdgeConfig, want_labels: bool = False,
                   masks: torch.Tensor | None = None, edges: torch.Tensor | None = None,
                   labels: torch.Tensor | None = None):
        """image -> (labels|None, masks[K,H,W], edges[K,H,W]); 02:53-154 + 03:23-34 in one call."""
        _check_img(bgr, 3)
        ctr = np.ascontiguousarray(centers, dtype=np.float32).reshape(-1, 3)
        K = ctr.shape[0]
        lut_a = None if lut is None else np.ascontiguousarray(lut, dtype=np.uint8)
        h, w = bgr.shape[:2]
        if masks is None:
            masks = torch.empty((K, h, w), dtype=torch.uint8, device=bgr.device)
        if edges is None:
            edges = torch.empty((K, h, w), dtype=torch.uint8, device=bgr.device)
        if labels is None and want_labels:
            labels = torch.empty((h, w), dtype=torch.uint8, device=bgr.device)
        p = ec.to_c()
        capi.check(self._L.omni_color_edge(
            self._h, bgr.data_ptr(), h, w, bgr.stride(0), _f32p(ctr), K, _u8p(lut_a), C.byref(p),
            labels.data_ptr() if labels is not None else None, labels.stride(0) if labels is not None else 0,
            masks.data_ptr(), masks.stride(0), masks.stride(1), edges.data_ptr(), edges.stride(0), edges.stride(1),
            self._stream()))
        return labels, masks, edges

    def color_edge_packed(self, frames: torch.Tensor, centers, lut, ec: "EdgeConfig | None", msb_first: bool = True,
                          want_counts: bool = False):
        """Packed form of color_edge / color_edge_batch: frames [H,W,3] or [n,H,W,3] (n * K <= 32) ->
        (mask_bits, edge_bits | None[, counts]) as CUDA uint8 tensors [n*K, H, ceil(W/8)], one BIT per pixel (msb_first: the
        scanline format of a 1-bit PNG = numpy.packbits default).  ec=None: colour layers only (stage 02 on its own).
        centers [K,3] / lut [K]: one set for all frames; centers [n,K,3] / lut [n,K]: frame f uses centers[f], lut[f]."""
        if frames.dim() == 3:
            frames = frames.unsqueeze(0)
        if frames.dim() != 4 or frames.shape[3] != 3 or frames.dtype != torch.uint8 or not frames.is_cuda or frames.stride(3) != 1 \
                or frames.stride(2) != 3:
            raise ValueError("frames must be a CUDA uint8 tensor [n,H,W,3] (or [H,W,3]) with packed pixels")
        n, h, w = frames.shape[:3]
        ctr, lut_a, K, per_frame = _centers_luts(centers, lut, n)
        fn = self._L.omni_color_edge_packed_frames if per_frame else self._L.omni_color_edge_packed
        rb = (w + 7) // 8
        mb = torch.empty((n * K, h, rb), dtype=torch.uint8, device=frames.device)
        eb = torch.empty((n * K, h, rb), dtype=torch.uint8, device=frames.device) if ec is not None else None
        counts = np.zeros((n * K, 3), np.int64) if want_counts else None
        p = ec.to_c() if ec is not None else None
        capi.check(fn(
            self._h, frames.data_ptr(), n, frames.stride(0), h, w, frames.stride(1), _f32p(ctr), K, _u8p(lut_a),
            C.byref(p) if p is not None else None, mb.data_ptr(), mb.stride(0), mb.stride(1),
            eb.data_ptr() if eb is not None else None, eb.stride(0) if eb is not None else 0, eb.stride(1) if eb is not None else 0,
            capi.BITS_MSB_FIRST if msb_first else capi.BITS_LSB_FIRST,
            counts.ctypes.data_as(C.POINTER(C.c_int64)) if counts is not None else None, self._stream()))
        return (mb, eb, counts) if want_counts else (mb, eb)

    def host_color_edge_packed(self, frames: np.ndarray, centers, lut, ec: "EdgeConfig | None", msb_first: bool = True,
                               mask_bits: np.ndarray | None = None, edge_bits: np.ndarray | None = None, want_counts: bool = True):
        """Host frames [n,H,W,3] (or one [H,W,3]) -> dict(mask_bits, edge_bits, counts): uint8 arrays [n*K, H, ceil(W/8)], one bit per
        pixel.  centers [K,3] / lut [K]: one centre set for all frames; centers [n,K,3] / lut [n,K]: frame f uses centers[f], lut[f].
        Any n: frame groups are pipelined through the device (H2D / kernels / D2H overlap).
        Pass pinned arrays (pinned_empty) for `frames`, `mask_bits`, `edge_bits` for full PCIe speed."""
        fr = np.asarray(frames)
        if fr.ndim == 3:
            fr = fr[None]
        if fr.dtype != np.uint8 or fr.ndim != 4 or fr.shape[3] != 3 or fr.strides[3] != 1 or fr.strides[2] != 3:
            fr = np.ascontiguousarray(fr, dtype=np.uint8)
        n, h, w = fr.shape[:3]
        ctr, lut_a, K, per_frame = _centers_luts(centers, lut, n)
        fn = self._L.omni_host_color_edge_packed_frames if per_frame else self._L.omni_host_color_edge_packed
        rb = (w + 7) // 8
        if mask_bits is None:
            mask_bits = np.empty((n * K, h, rb), np.uint8)
        if edge_bits is None and ec is not None:
            edge_bits = np.empty((n * K, h, rb), np.uint8)
        for a in (mask_bits, edge_bits):
            if a is not None and (a.shape != (n * K, h, rb) or a.dtype != np.uint8 or not a.flags.c_contiguous):
                raise ValueError("mask_bits / edge_bits must be C-contiguous uint8 [n*K, H, ceil(W/8)]")
        counts = np.zeros((n * K, 3), np.int64) if want_counts else None
        p = ec.to_c() if ec is not None else None
        capi.check(fn(
            self._h, fr.ctypes.data, n, fr.strides[0], h, w, fr.strides[1], _f32p(ctr), K, _u8p(lut_a),
            C.byref(p) if p is not None else None, mask_bits.ctypes.data, mask_bits.strides[0], mask_bits.strides[1],
            edge_bits.ctypes.data if edge_bits is not None else None, edge_bits.strides[0] if edge_bits is not None else 0,
            edge_bits.strides[1] if edge_bits is not None else 0, capi.BITS_MSB_FIRST if msb_first else capi.BITS_LSB_FIRST,
            counts.ctypes.data_as(C.POINTER(C.c_int64)) if counts is not None else None))
        return {"mask_bits": mask_bits, "edge_bits": edge_bits, "counts": counts}

    def count_nonzero(self, planes: torch.Tensor) -> np.ndarray:
        """np.count_nonzero per plane (02:157, 03:38)."""
        _check_planes(planes)
        K, h, w = planes.shape
        out = np.zeros(K, np.int64)
        capi.check(self._L.omni_count_nonzero(self._h, planes.data_ptr(), K, h, w, planes.stride(0), planes.stride(1),
                                              out.ctypes.data_as(C.POINTER(C.c_int64)), self._stream()))
        return out

    def color_edge_batch(self, frames: torch.Tensor, centers, lut, ec: EdgeConfig,
                         masks: torch.Tensor | None = None, edges: torch.Tensor | None = None):
        """n frames [n,H,W,3] sharing one centre set -> (masks[n,K,H,W], edges[n,K,H,W]); identical to n color_edge calls."""
        if frames.dim() != 4 or frames.shape[3] != 3 or frames.dtype != torch.uint8 or not frames.is_cuda or frames.stride(3) != 1 \
                or frames.stride(2) != 3:
            raise ValueError("frames must be a CUDA uint8 tensor [n,H,W,3] with packed pixels")
        ctr = np.ascontiguousarray(centers, dtype=np.float32).reshape(-1, 3)
        K = ctr.shape[0]
        lut_a = None if lut is None else np.ascontiguousarray(lut, dtype=np.uint8)
        n, h, w = frames.shape[:3]
        if masks is None:
            masks = torch.empty((n, K, h, w), dtype=torch.uint8, device=frames.device)
        if edges is None:
            edges = torch.empty((n, K, h, w), dtype=torch.uint8, device=frames.device)
        for t in (masks, edges):
            if t.shape != (n, K, h, w) or t.dtype != torch.uint8 or not t.is_cuda or t.stride(3) != 1 or t.stride(0) != K * t.stride(1):
                raise ValueError("masks/edges must be CUDA uint8 [n,K,H,W] with frame stride = K * plane stride")
        p = ec.to_c()
        capi.check(self._L.omni_color_edge_batch(
            self._h, frames.data_ptr(), n, frames.stride(0), h, w, frames.stride(1), _f32p(ctr), K, _u8p(lut_a), C.byref(p),
            masks.data_ptr(), masks.stride(1), masks.stride(2), edges.data_ptr(), edges.stride(1), edges.stride(2), self._stream()))
        return masks, edges

    def edges_composite(self, edges: torch.Tensor, colors_bgr) -> torch.Tensor:
        """03_edge_detect.py:93-106 paint on a white canvas.  HxWx3 u8."""
        _check_planes(edges)
        K, h, w = edges.shape
        col = np.ascontiguousarray(colors_bgr, dtype=np.uint8).reshape(-1, 3)[:K]
        if col.shape[0] < K:
            raise IndexError("list index out of range")        # what cfg.colors[i] raises in 03:90
        out = torch.empty((h, w, 3), dtype=torch.uint8, device=edges.device)
        capi.check(self._L.omni_edges_composite(self._h, edges.data_ptr(), K, h, w, edges.stride(0), edges.stride(1),
                                                _u8p(col), out.data_ptr(), out.stride(0), self._stream()))
        return out

    # ---- stage 04: thinning ----------------------------------------------------------------------
    def thin_zhangsuen(self, planes: torch.Tensor, max_iter: int = 120, out: torch.Tensor | None = None,
                       with_log: bool = False):
        """04_find_contours.py:35-99 on K planes at once: [K,H,W] u8 (> 0 = foreground) -> skeletons {0,255}.
        with_log: also returns (removed[K, max_iter] int32, iters[K] int32) -- what the reference prints per iteration."""
        _check_planes(planes)
        K, h, w = planes.shape
        if out is None:
            out = torch.empty((K, h, w), dtype=torch.uint8, device=planes.device)
        _check_planes(out)
        removed = np.zeros((K, max(1, max_iter)), np.int32) if with_log else None
        iters = np.zeros(K, np.int32) if with_log else None
        i32p = C.POINTER(C.c_int32)
        capi.check(self._L.omni_thin_zhangsuen(
            self._h, planes.data_ptr(), K, h, w, planes.stride(0), planes.stride(1), int(max_iter),
            out.data_ptr(), out.stride(0), out.stride(1),
            removed.ctypes.data_as(i32p) if with_log else None, iters.ctypes.data_as(i32p) if with_log else None, self._stream()))
        return (out, removed[:, :max_iter], iters) if with_log else out

    def thin_zhangsuen_packed(self, bits: torch.Tensor, w: int, max_iter: int = 120, msb_first: bool = True, out: torch.Tensor | None = None):
        """Thinning of planes given as 1 bit per pixel ([K, H, ceil(W/8)] u8, the packed edge planes of color_edge_packed): the
        skeletons in the same layout.  No byte planes are touched on the way (stage 03 -> 04 on the device)."""
        _check_planes(bits)
        K, h, rb = bits.shape
        if rb < (w + 7) // 8:
            raise ValueError("rows too short for w pixels")
        if out is None:
            out = torch.empty_like(bits)
        capi.check(self._L.omni_thin_zhangsuen_packed(
            self._h, bits.data_ptr(), K, h, w, bits.stride(0), bits.stride(1), capi.BITS_MSB_FIRST if msb_first else capi.BITS_LSB_FIRST,
            int(max_iter), out.data_ptr(), out.stride(0), out.stride(1), None, None, self._stream()))
        return out

    def skeleton_degree(self, skel: torch.Tensor):
        """04_find_contours.py:121-125 on K skeleton planes: (deg[K,H,W] = set 8-neighbours per pixel, nodes[K,H,W] with
        1 = endpoint, 2 = junction)."""
        _check_planes(skel)
        K, h, w = skel.shape
        deg = torch.empty((K, h, w), dtype=torch.uint8, device=skel.device)
        nodes = torch.empty((K, h, w), dtype=torch.uint8, device=skel.device)
        capi.check(self._L.omni_skeleton_degree(self._h, skel.data_ptr(), K, h, w, skel.stride(0), skel.stride(1),
                                                deg.data_ptr(), deg.stride(0), deg.stride(1),
                                                nodes.data_ptr(), nodes.stride(0), nodes.stride(1), self._stream()))
        return deg, nodes

    def host_thin_zhangsuen(self, planes: np.ndarray, max_iter: int = 120):
        """Host-buffer form: NumPy [K,H,W] u8 in, (skeletons, removed[K,max_iter], iters[K]) out."""
        planes = np.ascontiguousarray(planes, dtype=np.uint8)
        K, h, w = planes.shape
        out = np.empty_like(planes)
        removed = np.zeros((K, max(1, max_iter)), np.int32)
        iters = np.zeros(K, np.int32)
        i32p = C.POINTER(C.c_int32)
        capi.check(self._L.omni_host_thin_zhangsuen(
            self._h, planes.ctypes.data, K, h, w, planes.strides[0], planes.strides[1], int(max_iter),
            out.ctypes.data, out.strides[0], out.strides[1], removed.ctypes.data_as(i32p), iters.ctypes.data_as(i32p)))
        return out, removed[:, :max_iter], iters

    # ---- stage 04: trace_centerlines ----------------------------------------------------------------
    def trace_centerlines(self, skel: torch.Tensor) -> list["TraceResult"]:
        """04_find_contours.py:101-205 on K skeleton planes [K,H,W] u8 (> 0 = foreground): per plane a TraceResult (the
        reference's polylines in its order, cv2's component stats).  Synchronises the current stream."""
        _check_planes(skel)
        K, h, w = skel.shape
        info = np.zeros((K, 4), np.int64)
        capi.check(self._L.omni_trace_centerlines(self._h, skel.data_ptr(), K, h, w, skel.stride(0), skel.stride(1),
                                                  info.ctypes.data_as(C.POINTER(C.c_int64)), self._stream()))
        return self._trace_results(info)

    def host_trace_centerlines(self, skel: np.ndarray) -> list["TraceResult"]:
        """Host-buffer form of trace_centerlines: NumPy [K,H,W] or [H,W] (> 0 = foreground; ctypes + NumPy only)."""
        a = np.asarray(skel)
        if a.ndim == 2:
            a = a[None]
        if a.ndim != 3:
            raise ValueError("expected skeleton planes [K,H,W] or one [H,W]")
        if a.dtype != np.uint8:
            a = (a > 0).astype(np.uint8)
        elif a.strides[2] != 1 or a.strides[1] < a.shape[2] or a.strides[0] < 0 or a.strides[1] < 0:
            a = np.ascontiguousarray(a)
        K, h, w = a.shape
        info = np.zeros((K, 4), np.int64)
        capi.check(self._L.omni_host_trace_centerlines(self._h, a.ctypes.data, K, h, w, a.strides[0], a.strides[1],
                                                       info.ctypes.data_as(C.POINTER(C.c_int64))))
        return self._trace_results(info)

    def _trace_results(self, info: np.ndarray) -> list["TraceResult"]:
        n_comp, n_paths, n_pts = (int(v) for v in info[:, 1:].sum(axis=0))
        pts = np.empty((n_pts, 2), np.int32)
        lens = np.empty(n_paths, np.int32)
        comp = np.empty((n_comp, 6), np.int32)
        capi.check(self._L.omni_trace_results(self._h, pts.ctypes.data, lens.ctypes.data, comp.ctypes.data))
        out, c0, l0, p0 = [], 0, 0, 0
        for total_fg, nc, npath, npt in info.tolist():
            ln = lens[l0:l0 + npath]
            pl = pts[p0:p0 + npt].reshape(-1, 1, 2)
            paths = np.split(pl, np.cumsum(ln[:-1])) if npath else []
            out.append(TraceResult(paths, comp[c0:c0 + nc, :5], comp[c0:c0 + nc, 5], int(total_fg)))
            c0, l0, p0 = c0 + nc, l0 + npath, p0 + npt
        return out

    # ---- PNG files of stages 01-03 (01:30, 02:156, 03:37, 03:60-111) ------------------------------------
    def png_encode(self, images: torch.Tensor, fmt, w: int | None = None) -> list:
        """Device images -> one PNG file (bytes) each, encoded on the GPU (omni_png_encode).  fmt capi.PNG_GRAY1 ("gray1"):
        packed MSB-first rows [H, RB] or [n, H, RB] (w: pixels per row, default 8 * RB); capi.PNG_BGR8 ("bgr8"): [H, W, 3] or
        [n, H, W, 3] BGR.  Any row / image strides.  Synchronises the current stream."""
        if not (isinstance(images, torch.Tensor) and images.is_cuda and images.dtype == torch.uint8):
            raise TypeError("expected a CUDA uint8 tensor")
        fmt = _png_format(fmt)
        n, h, w, pitch, stride = _png_geometry(tuple(images.shape), tuple(images.stride()), fmt, w)
        cap = n * int(self._L.omni_png_bound(h, w, fmt))
        out = torch.empty(max(1, cap), dtype=torch.uint8, device=images.device)
        sizes = np.zeros(n, np.int64)
        capi.check(self._L.omni_png_encode(self._h, images.data_ptr(), n, stride, h, w, pitch, fmt, out.data_ptr(), cap,
                                           sizes.ctypes.data_as(C.POINTER(C.c_int64)), self._stream()))
        return _png_split(out[:int(sizes.sum())].cpu().numpy(), sizes)

    def host_png_encode(self, images: np.ndarray, fmt, w: int | None = None) -> list:
        """Host-buffer form of png_encode (NumPy in, bytes out; ctypes + NumPy only): one H2D copy of the pixels, one D2H copy
        of the compressed files."""
        a = np.asarray(images)
        if a.dtype != np.uint8:
            raise TypeError("expected a uint8 array")
        fmt = _png_format(fmt)
        if a.ndim == 0 or any(s < 0 for s in a.strides) or a.strides[-1] != 1:
            a = np.ascontiguousarray(a)
        n, h, w, pitch, stride = _png_geometry(a.shape, a.strides, fmt, w)
        cap = n * int(self._L.omni_png_bound(h, w, fmt))
        out = np.empty(max(1, cap), np.uint8)
        sizes = np.zeros(n, np.int64)
        capi.check(self._L.omni_host_png_encode(self._h, a.ctypes.data, n, stride, h, w, pitch, fmt, out.ctypes.data, cap,
                                                sizes.ctypes.data_as(C.POINTER(C.c_int64))))
        return _png_split(out, sizes)

    def last_hysteresis_passes(self) -> int:
        return int(self._L.omni_last_hysteresis_passes(self._h))

    # ---- launch accounting / per-kernel CUDA-event timing -----------------------------------------
    def launch_count(self) -> int:
        """Kernels launched by this engine so far."""
        return int(self._L.omni_launch_count(self._h))

    def profile(self, on: bool):
        capi.check(self._L.omni_profile_enable(self._h, 1 if on else 0))

    def profile_summary(self) -> dict:
        """{kernel name: (launches, total_ms)} since profile(True) / the last summary."""
        buf = C.create_string_buffer(1 << 14)
        capi.check(self._L.omni_profile_summary(self._h, buf, len(buf)))
        out = {}
        for line in buf.value.decode().splitlines():
            name, n, ms = line.split("\t")
            out[name] = (int(n), float(ms))
        return out

    # ---- host-buffer entry points (H2D + kernels + D2H inside the call) ---------------------------------
    def host_resize_area(self, img: np.ndarray, new_w: int, new_h: int) -> np.ndarray:
        img = _as_u8(img, 3)
        out = np.empty((new_h, new_w, 3), np.uint8)
        capi.check(self._L.omni_host_resize_area_u8c3(self._h, img.ctypes.data, img.shape[0], img.shape[1], img.strides[0],
                                                      out.ctypes.data, new_h, new_w, out.strides[0]))
        return out

    def host_assign_rgb_i16wrap(self, img_rgb: np.ndarray, palette) -> np.ndarray:
        img = _as_u8(img_rgb, 3)
        pal = np.ascontiguousarray(palette, dtype=np.uint8).reshape(-1, 3)
        out = np.empty(img.shape[:2], np.uint8)
        capi.check(self._L.omni_host_assign_rgb_i16wrap(self._h, img.ctypes.data, img.shape[0], img.shape[1], img.strides[0],
                                                        _u8p(pal), pal.shape[0], out.ctypes.data, out.strides[0]))
        return out

    def host_edges(self, masks: np.ndarray, ec: EdgeConfig, out: np.ndarray | None = None) -> np.ndarray:
        masks = np.ascontiguousarray(masks, dtype=np.uint8)
        K, h, w = masks.shape
        if out is None:
            out = np.empty((K, h, w), np.uint8)
        p = ec.to_c()
        capi.check(self._L.omni_host_edges(self._h, masks.ctypes.data, K, h, w, masks.strides[0], masks.strides[1],
                                           C.byref(p), out.ctypes.data, out.strides[0], out.strides[1]))
        return out

    def host_edges_composite(self, edges: np.ndarray, colors_bgr) -> np.ndarray:
        """03_edge_detect.py:93-106 on host planes [K,H,W] -> host canvas [H,W,3] (no torch needed)."""
        edges = np.ascontiguousarray(edges, dtype=np.uint8)
        K, h, w = edges.shape
        col = np.ascontiguousarray(colors_bgr, dtype=np.uint8).reshape(-1, 3)[:K]
        if col.shape[0] < K:
            raise IndexError("list index out of range")        # what cfg.colors[i] raises in 03:90
        out = np.empty((h, w, 3), np.uint8)
        capi.check(self._L.omni_host_edges_composite(self._h, edges.ctypes.data, K, h, w, edges.strides[0], edges.strides[1],
                                                     _u8p(col), out.ctypes.data, out.strides[0]))
        return out

    def host_color_edge(self, img_bgr: np.ndarray, centers, lut, ec: EdgeConfig, want_labels: bool = True,
                        masks: np.ndarray | None = None, edges: np.ndarray | None = None, want_counts: bool = True):
        """Host image -> dict(labels, masks, edges, counts) as host arrays (pass pinned arrays from
        pinned_empty() as `masks`/`edges` for full-speed copies)."""
        img = _as_u8(img_bgr, 3)
        ctr = np.ascontiguousarray(centers, dtype=np.float32).reshape(-1, 3)
        K = ctr.shape[0]
        lut_a = None if lut is None else np.ascontiguousarray(lut, dtype=np.uint8)
        h, w = img.shape[:2]
        if masks is None:
            masks = np.empty((K, h, w), np.uint8)
        if edges is None:
            edges = np.empty((K, h, w), np.uint8)
        labels = np.empty((h, w), np.uint8) if want_labels else None
        counts = np.zeros((K, 3), np.int64) if want_counts else None
        p = ec.to_c()
        capi.check(self._L.omni_host_color_edge(
            self._h, img.ctypes.data, h, w, img.strides[0], _f32p(ctr), K, _u8p(lut_a), C.byref(p),
            labels.ctypes.data if labels is not None else None, labels.strides[0] if labels is not None else 0,
            masks.ctypes.data, masks.strides[0], masks.strides[1], edges.ctypes.data, edges.strides[0], edges.strides[1],
            counts.ctypes.data_as(C.POINTER(C.c_int64)) if counts is not None else None))
        return {"labels": labels, "masks": masks, "edges": edges, "counts": counts}


def _as_u8(a: np.ndarray, ch: int) -> np.ndarray:
    a = np.asarray(a)
    if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != ch:
        raise ValueError(f"expected an HxWx{ch} uint8 array")
    if a.strides[2] != 1 or a.strides[1] != ch:
        a = np.ascontiguousarray(a)
    return a


def _png_format(fmt) -> int:
    names = {"gray1": capi.PNG_GRAY1, "bgr8": capi.PNG_BGR8}
    if isinstance(fmt, str):
        if fmt.lower() not in names:
            raise ValueError(f"unknown PNG format {fmt!r} (gray1, bgr8)")
        return names[fmt.lower()]
    return int(fmt)             # other values reach the C call, which reports them


def _png_geometry(shape, strides, fmt: int, w):
    """(n, h, w, row pitch, image stride) of one image or a stack of images for omni_png_encode (strides in bytes)."""
    batched = len(shape) == (3 if fmt == capi.PNG_GRAY1 else 4)
    if fmt == capi.PNG_BGR8:
        if len(shape) not in (3, 4) or shape[-1] != 3 or strides[-1] != 1 or strides[-2] != 3:
            raise ValueError("PNG_BGR8 expects [H, W, 3] or [n, H, W, 3] uint8 with packed pixels")
        if w is not None and int(w) != shape[-2]:
            raise ValueError(f"w={w} does not match the image width {shape[-2]}")
        h, w, pitch = shape[-3], shape[-2], strides[-3]
    else:
        if len(shape) not in (2, 3) or strides[-1] != 1:
            raise ValueError("PNG_GRAY1 expects packed rows [H, RB] or [n, H, RB] uint8 with unit column stride")
        h, rb, pitch = shape[-2], shape[-1], strides[-2]
        w = 8 * rb if w is None else int(w)
        if (w + 7) // 8 > rb:
            raise ValueError(f"w={w} needs {(w + 7) // 8} bytes per row, the rows have {rb}")
    n = shape[0] if batched else 1
    return n, h, w, pitch, (strides[0] if batched else 0)


def _png_split(buf: np.ndarray, sizes: np.ndarray) -> list:
    ends = np.cumsum(sizes)
    return [buf[e - s:e].tobytes() for s, e in zip(sizes.tolist(), ends.tolist())]


def pinned_empty(shape, dtype=np.uint8) -> np.ndarray:
    """Host array in page-locked memory (torch owns it; the numpy view keeps it alive)."""
    t = torch.empty(tuple(shape), dtype=getattr(torch, np.dtype(dtype).name), pin_memory=True)
    return t.numpy()


_engines = threading.local()


def get_engine(device: int | None = None) -> Engine:
    """Per-thread, per-device Engine cache."""
    dev = (sys.modules["torch"].cuda.current_device() if (device is None and "torch" in sys.modules
                                                           and sys.modules["torch"].cuda.is_available()) else (device or 0))
    cache = getattr(_engines, "cache", None)
    if cache is None:
        cache = _engines.cache = {}
    if dev not in cache:
        cache[dev] = Engine(dev)
    return cache[dev]
