"""Host-side mirror of the reference's stage functions for stages 01-03 (same names, arguments, files
and error behaviour), with the per-pixel arithmetic done by libomni_b200's CUDA kernels.

    reference                                   here
    01_resize.resize_if_needed(path, cfg)       resize_if_needed(path, cfg)
    02_color_extract._kmeans_lab(img, k, ..)    _kmeans_lab(img, k, ..)      (k-means itself stays on the host)
    02_color_extract.main()                     color_extract_main()
    03_edge_detect.process_color(name, cfg)     process_color(name, cfg)
    03_edge_detect.detect_all_edges(cfg)        detect_all_edges(cfg)
    03_edge_detect.save_edges_composite(cfg)    save_edges_composite(cfg)
    process_colors.assign_labels(img, pal)      assign_labels(img, pal)

Image decode/encode (cv2.imread / cv2.imwrite) and cv2.kmeans stay host-side library calls exactly as in
the reference: PNG files and k-means centres are the stage boundary / inputs, not the data-parallel path.
There is no CPU fallback for the pixel work: without a GPU every function here raises.
"""
from __future__ import annotations

import json
import os

import cv2
import numpy as np

from .ops import EdgeConfig, get_engine


# ---- 01_resize.py --------------------------------------------------------------------------------------
def resize_dims(h: int, w: int, max_dimension):
    """(new_w, new_h) or None -- the identical Python float expressions of 01_resize.py:15-18."""
    max_dim = max(h, w)
    if max_dim > max_dimension:
        scale = max_dimension / max_dim
        return int(w * scale), int(h * scale)
    return None


def resize_if_needed(image_path: str, cfg) -> np.ndarray:
    """01_resize.py:7-23."""
    img = cv2.imread(image_path)
    if img is None:
        raise ValueError(f"Failed to load image: {image_path}")
    h, w = img.shape[:2]
    dims = resize_dims(h, w, cfg.max_dimension)
    if dims is None:
        print(f"No resize required: {w}x{h}")
        return img
    new_w, new_h = dims
    print(f"Resizing: {w}x{h} -> {new_w}x{new_h}")
    return get_engine().host_resize_area(img, new_w, new_h)


def resize_main(cfg) -> str:
    """01_resize.py:25-31."""
    cfg.ensure_output_dirs()
    out = resize_if_needed(cfg.input_image, cfg)
    path = os.path.join(cfg.output_dir, "resized.png")
    cv2.imwrite(path, out)
    print(f"Saved: {path}")
    return path


# ---- 02_color_extract.py -------------------------------------------------------------------------------
def _darkness_rank(name: str) -> int:
    """02_color_extract.py:17-23."""
    s = name.lower()
    if "dark" in s:
        return 0
    if "mid" in s:
        return 1
    if "skin" in s:
        return 2
    if "light" in s:
        return 3
    return 2


def _ensure_bgr(img):
    if img.ndim == 2:
        return cv2.cvtColor(img, cv2.COLOR_GRAY2BGR)
    if img.shape[2] == 4:
        return cv2.cvtColor(img, cv2.COLOR_BGRA2BGR)
    return img


def _sample_pick(n: int, sample_limit: int):
    """02_color_extract.py:37-42: the seeded subsample (None: every pixel).  It depends on the pixel count only."""
    return np.random.default_rng(42).choice(n, size=sample_limit, replace=False) if n > sample_limit else None


def kmeans_lab_centers(img_bgr: np.ndarray, k: int, sample_limit: int = 200_000, attempts: int = 3) -> np.ndarray:
    """02_color_extract.py:35-50: centres from cv2.kmeans on the seeded <=200k-pixel Lab subsample.
    Only the sampled pixels are converted (cvtColor is per-pixel, so the values are the reference's)."""
    pick = _sample_pick(img_bgr.shape[0] * img_bgr.shape[1], sample_limit)
    if os.environ.get("OMNI_B200_KMEANS", "").lower() == "gpu":
        # opt-in (SURVEY 8f rank 2): the same subsample, clustered on the device -- cv2.kmeans' own centres cannot be reproduced
        # (global RNG); the contract is their quality (include/omni_b200.h omni_kmeans_lab, tests/test_gpu_kmeans.py)
        import torch
        centers, _comp = get_engine().kmeans_lab(torch.from_numpy(np.ascontiguousarray(img_bgr)).cuda(), k, pick, attempts=attempts)
        return centers
    return _host_kmeans(img_bgr, k, pick, attempts)


def _host_kmeans(img_bgr: np.ndarray, k: int, pick, attempts: int) -> np.ndarray:
    """The cv2.kmeans branch of kmeans_lab_centers on the subsample `pick` (None: every pixel)."""
    flat = img_bgr.reshape(-1, 3)
    if pick is not None:
        flat = flat[pick]
    lab = cv2.cvtColor(np.ascontiguousarray(flat).reshape(-1, 1, 3), cv2.COLOR_BGR2LAB)
    sample = lab.reshape(-1, 3).astype(np.float32)
    criteria = (cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_MAX_ITER, 40, 0.5)
    _compact, _labels, centers = cv2.kmeans(sample, k, None, criteria, attempts, cv2.KMEANS_PP_CENTERS)
    return centers.astype(np.float32)


def _kmeans_lab(img_bgr: np.ndarray, k: int, sample_limit: int = 200_000, attempts: int = 3):
    """02_color_extract.py:32-56 -> (centers f32[k,3], labels int32[H,W])."""
    centers = kmeans_lab_centers(img_bgr, k, sample_limit, attempts)
    import torch
    eng = get_engine()
    labels = eng.assign_lab(torch.from_numpy(np.ascontiguousarray(img_bgr)).cuda(), centers)
    return centers, labels.cpu().numpy().astype(np.int32)


def darkness_lut(centers: np.ndarray):
    """02_color_extract.py:121-127: the identical NumPy expressions (argsort is not re-implemented)."""
    order = np.argsort(centers[:, 0])
    lut = np.zeros_like(order)
    lut[order] = np.arange(len(order))
    return order, lut


def _kmeans_args(cfg):
    """02_color_extract.py:66-80 as color_extract_main reads it: (K, sample_limit, attempts)."""
    K = max(2, min(len(list(cfg.color_names)), int(getattr(cfg, "cluster_k", len(cfg.color_names)))))
    return K, int(getattr(cfg, "kmeans_sample_limit", 200_000)), int(getattr(cfg, "kmeans_attempts", 3))


def frame_centers(frames, cfg, mode: str = "host", threads: int | None = None, group: int = 64):
    """Stage 02's centres for every frame of a batch, each frame clustered on its own as a stage-02 run of that frame would:
    (centers f32 [n,K,3], luts u8 [n,K]) for Engine.host_color_edge_packed / color_edge_packed with per-frame centres.
    frames: [n,H,W,3] BGR (or a sequence of such images for mode="host").  The darkness LUT is the reference's argsort (darkness_lut).
      mode="host": exact.  Per frame cv2.setRNGSeed(0), then the cv2.kmeans expression of kmeans_lab_centers: the centres of a
        fresh-process stage-02 run on that frame (SURVEY A.7).  OpenCV's RNG is per thread, so frames run on `threads` threads
        (default: up to 8) with the same result as one after another.
      mode="gpu": opt-in, omni_kmeans_lab's quality contract (include/omni_b200.h).  Frames go to the device `group` at a time,
        one omni_kmeans_lab_batch call per group, all with the reference's subsample indices."""
    K, limit, attempts = _kmeans_args(cfg)
    n = len(frames)
    if n == 0:
        return np.empty((0, K, 3), np.float32), np.empty((0, K), np.uint8)
    if mode == "host":
        def one(img):
            img = _ensure_bgr(np.asarray(img))
            cv2.setRNGSeed(0)
            return _host_kmeans(img, K, _sample_pick(img.shape[0] * img.shape[1], limit), attempts)
        workers = max(1, min(n, threads if threads is not None else min(8, os.cpu_count() or 1)))
        if workers == 1:
            centers = [one(f) for f in frames]
        else:
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(workers) as ex:
                centers = list(ex.map(one, frames))
        centers = np.stack(centers).astype(np.float32)
    elif mode == "gpu":
        import torch
        fr = np.asarray(frames)
        if fr.ndim != 4 or fr.shape[3] != 3 or fr.dtype != np.uint8:
            raise ValueError("mode='gpu' needs frames as one uint8 array [n,H,W,3]")
        pick = _sample_pick(fr.shape[1] * fr.shape[2], limit)
        eng = get_engine()
        parts = []
        for g0 in range(0, n, group):
            d = torch.from_numpy(np.ascontiguousarray(fr[g0:g0 + group])).cuda()
            parts.append(eng.kmeans_lab_batch(d, K, pick, attempts=attempts)[0])
        centers = np.concatenate(parts)
    else:
        raise ValueError(f"mode must be 'host' or 'gpu', got {mode!r}")
    luts = np.stack([darkness_lut(c)[1] for c in centers]).astype(np.uint8)
    return centers, luts


def _lab_to_bgr(lab3) -> tuple:
    """02_color_extract.py:58-61."""
    px = np.uint8([[list(lab3)]])
    bgr = cv2.cvtColor(px, cv2.COLOR_Lab2BGR)[0, 0]
    return int(bgr[0]), int(bgr[1]), int(bgr[2])


def _write_layer_png(path: str, plane_u8=None, bits=None, w=None) -> None:
    """mask.png / edges.png: a 1-bit greyscale PNG (decodes through cv2.imread to the same {0,255} pixels; see omni_b200/png1.py)
    unless OMNI_B200_PNG_BITS=8.  Give either the u8 plane or its MSB-first packed rows."""
    from . import png1
    if png1.use_1bit():
        if bits is None:
            bits, w = np.packbits(plane_u8 > 0, axis=1), plane_u8.shape[1]
        png1.write_png1(path, bits, w)
    else:
        if plane_u8 is None:
            plane_u8 = png1.unpack_rows(bits, w)
        cv2.imwrite(path, plane_u8)


def _swatch_extract(cfg, img, names) -> None:
    """02_color_extract.py:82-109: legacy swatch mode (only reachable with a hand-built Config, config.py drops the key)."""
    tol = int(getattr(cfg, "color_tolerance", 30))
    colors = list(getattr(cfg, "colors", []))
    if not colors or len(colors) < len(names):
        raise RuntimeError("swatch mode: 'colors' must have \u2265 len(color_names) entries.")
    import torch
    cols = [[int(v) for v in colors[i]] for i in range(len(names))]
    masks = get_engine().swatch_masks(torch.from_numpy(np.ascontiguousarray(img)).cuda(), cols, tol).cpu().numpy()
    for i, name in enumerate(names):
        os.makedirs(os.path.join(cfg.output_dir, name), exist_ok=True)
        _write_layer_png(os.path.join(cfg.output_dir, name, "mask.png"), plane_u8=masks[i])
        print(f"Extracted (swatch): {name} | nz={int(np.count_nonzero(masks[i]))}")
    print("Color extraction: done.")


def color_extract_main(cfg, img=None) -> dict:
    """02_color_extract.py:66-175.  k-means mode is the only one reachable through config.json; the swatch branch
    (:82-109) is honoured when the Config object carries extraction_mode == "swatch".  Only stage 02's own work is done
    here (assignment + RECT open/close): the layers come off the GPU as packed bit rows and go straight into 1-bit PNGs."""
    os.makedirs(cfg.output_dir, exist_ok=True)
    path = os.path.join(cfg.output_dir, "resized.png")
    if img is None:                                    # (front_half_main hands the array over: the PNG is lossless, same pixels)
        img = cv2.imread(path, cv2.IMREAD_COLOR)
    if img is None:
        raise RuntimeError(f"Cannot read resized image: {path}")
    img = _ensure_bgr(img)
    names = list(cfg.color_names)
    K, sample_limit, attempts = _kmeans_args(cfg)
    if str(getattr(cfg, "extraction_mode", "kmeans")).lower() == "swatch":
        _swatch_extract(cfg, img, names)
        return {}
    centers = kmeans_lab_centers(img, K, sample_limit=sample_limit, attempts=attempts)
    order, lut = darkness_lut(centers)
    centers_sorted = centers[order]
    open_iters = int(getattr(cfg, "extract_open_iters", 1))
    close_iters = int(getattr(cfg, "extract_close_iters", 1))
    h, w = img.shape[:2]
    eng = get_engine()
    handoff_ec = None
    if open_iters == 1 and close_iters == 1:
        # One GPU pass also yields the stage-03 planes of these masks (+0.2 ms of kernels).  They are parked in hidden files
        # that 03_edge_detect.py publishes if -- and only if -- the masks and the edge keys of config.json are still the same
        # when it runs; otherwise it recomputes from mask.png as the reference does.  OMNI_B200_STAGE_HANDOFF=0: stage 02 only.
        if os.environ.get("OMNI_B200_STAGE_HANDOFF", "1") != "0":
            try:
                handoff_ec = EdgeConfig.from_cfg(cfg)
                handoff_ec.to_c()
            except Exception:
                handoff_ec = None
        try:
            r = eng.host_color_edge_packed(img, centers, lut.astype(np.uint8), handoff_ec, msb_first=True)
        except Exception:
            if handoff_ec is None:
                raise
            handoff_ec = None                           # edge keys the GPU path rejects: stage 03 will report them, not stage 02
            r = eng.host_color_edge_packed(img, centers, lut.astype(np.uint8), None, msb_first=True)
        bits, planes, counts = r["mask_bits"], None, r["counts"]
    else:                                              # other iteration counts: the unfused operators (any count, 02:151-154)
        import torch
        d_lab = eng.assign_lab(torch.from_numpy(np.ascontiguousarray(img)).cuda(), centers, lut.astype(np.uint8))
        planes = eng.layer_masks(d_lab, K, open_iters, close_iters).cpu().numpy()
        lab_h = d_lab.cpu().numpy()
        bits = None
        counts = np.array([[int((lab_h == k).sum()), int(np.count_nonzero(planes[k])), 0] for k in range(K)], np.int64)
    names_sorted = sorted(names, key=_darkness_rank)
    mapping = list(zip(names_sorted, range(K)))
    palette = {}
    for name, _k in mapping:
        os.makedirs(os.path.join(cfg.output_dir, name), exist_ok=True)
    with _io_pool(cfg, len(mapping)) as pool:                      # K PNG encodes in parallel (zlib / cv2 release the GIL)
        list(pool.map(lambda nk: _write_layer_png(os.path.join(cfg.output_dir, nk[0], "mask.png"),
                                                  plane_u8=None if planes is None else planes[nk[1]],
                                                  bits=None if bits is None else bits[nk[1]], w=w), mapping))
    for name, k in mapping:
        lab = centers_sorted[k]
        palette[name] = {
            "mode": "kmeans", "cluster_index": int(k), "cluster_lab": [int(lab[0]), int(lab[1]), int(lab[2])],
            "approx_bgr": list(_lab_to_bgr(lab.astype(np.uint8))), "pixels": int(counts[k, 0]),
            "mask_nonzero": int(counts[k, 1]),
        }
        print(f"Extracted (kmeans): {name} | cluster={k} | L*={lab[0]:.1f} | "
              f"pixels={palette[name]['pixels']} | nz={palette[name]['mask_nonzero']}")
    pal_path = os.path.join(cfg.output_dir, "palette_by_name.json")
    with open(pal_path, "w", encoding="utf-8") as fh:
        json.dump(palette, fh, ensure_ascii=False, indent=2)
    print(f"Palette saved: {pal_path}")
    print("Color extraction: done.")
    _handoff_drop(cfg)
    if handoff_ec is not None and len(mapping) == len(names):
        _handoff_write(cfg, handoff_ec, mapping, r["edge_bits"], counts, w)
    return palette


# ---- hand-off 02 -> 03 (SURVEY 8b: "script 03 just flushes cached results, but run alone it must still work from files") ----
_HANDOFF = ".omni_b200_handoff.json"
_HIDDEN_EDGES = ".edges_b200.png"
_HIDDEN_COMPOSITE = ".edges_composite_b200.png"


def _edge_keys(cfg) -> dict:
    ec = EdgeConfig.from_cfg(cfg)
    return {"low": float(ec.low), "high": float(ec.high), "ksize": int(ec.ksize), "morph_k": int(ec.morph_k),
            "open_iters": int(ec.open_iters), "close_iters": int(ec.close_iters)}


def _handoff_drop(cfg) -> None:
    for p in [os.path.join(cfg.output_dir, _HANDOFF), os.path.join(cfg.output_dir, _HIDDEN_COMPOSITE)] + \
            [os.path.join(cfg.output_dir, n, _HIDDEN_EDGES) for n in cfg.color_names]:
        try:
            os.remove(p)
        except OSError:
            pass


def _handoff_write(cfg, ec, mapping, edge_bits, counts, w) -> None:
    names = list(cfg.color_names)
    plane_of = dict(mapping)
    with _io_pool(cfg, len(names)) as pool:
        list(pool.map(lambda n: _write_layer_png(os.path.join(cfg.output_dir, n, _HIDDEN_EDGES), bits=edge_bits[plane_of[n]], w=w), names))
    note = {"edge": _edge_keys(cfg), "color_names": names, "colors": [list(map(int, c)) for c in list(cfg.colors)],
            "masks": {n: list(_stamp(os.path.join(cfg.output_dir, n, "mask.png"))) for n in names},
            "edge_nz": {n: int(counts[plane_of[n], 2]) for n in names}, "composite": False}
    if len(cfg.colors) >= len(names):                  # else 03:90 raises IndexError -- left to stage 03
        from . import png1
        stack = np.stack([png1.unpack_rows(edge_bits[plane_of[n]], w) for n in names])
        canvas = get_engine().host_edges_composite(stack, [tuple(cfg.colors[i]) for i in range(len(names))])
        cv2.imwrite(os.path.join(cfg.output_dir, _HIDDEN_COMPOSITE), canvas, [cv2.IMWRITE_PNG_COMPRESSION, 1])
        note["composite"] = True
    with open(os.path.join(cfg.output_dir, _HANDOFF), "w", encoding="utf-8") as fh:
        json.dump(note, fh)


def _handoff_publish(cfg) -> bool:
    """Stage 03 started right after this tree's stage 02 with unchanged masks and edge keys: publish the parked planes."""
    if os.environ.get("OMNI_B200_STAGE_HANDOFF", "1") == "0":
        return False
    try:
        with open(os.path.join(cfg.output_dir, _HANDOFF), "r", encoding="utf-8") as fh:
            note = json.load(fh)
        names = list(cfg.color_names)
        if note["color_names"] != names or note["edge"] != _edge_keys(cfg) or not note["composite"]:
            return False
        if note["colors"] != [list(map(int, c)) for c in list(cfg.colors)]:
            return False
        if os.path.exists(os.path.join(cfg.output_dir, "palette_by_name.json")):
            pal = json.load(open(os.path.join(cfg.output_dir, "palette_by_name.json"), "r", encoding="utf-8")) or {}
            if any(isinstance(v, dict) and "bgr" in v for v in pal.values()):
                return False                            # a palette with "bgr" keys changes the composite colours (03:86)
        for n in names:
            if list(_stamp(os.path.join(cfg.output_dir, n, "mask.png"))) != note["masks"][n]:
                return False
            if not os.path.exists(os.path.join(cfg.output_dir, n, _HIDDEN_EDGES)):
                return False
        if not os.path.exists(os.path.join(cfg.output_dir, _HIDDEN_COMPOSITE)):
            return False
    except (OSError, KeyError, ValueError, TypeError):
        return False
    for n in names:
        os.replace(os.path.join(cfg.output_dir, n, _HIDDEN_EDGES), os.path.join(cfg.output_dir, n, "edges.png"))
        print(f"Edges extracted: {n} | nz={note['edge_nz'][n]}")
    out_path = os.path.join(cfg.output_dir, "edges_composite.png")
    os.replace(os.path.join(cfg.output_dir, _HIDDEN_COMPOSITE), out_path)
    print(f"Edges composite saved: {out_path}")
    try:
        os.remove(os.path.join(cfg.output_dir, _HANDOFF))
    except OSError:
        pass
    return True


def edge_detect_main(cfg) -> None:
    """03_edge_detect.py:112-115."""
    if _handoff_publish(cfg):
        return
    detect_all_edges(cfg)
    save_edges_composite(cfg)


def front_half_main(cfg) -> None:
    """Stages 01 -> 02 -> 03 in ONE process (SURVEY 8f rank 3: in-memory hand-off): the same files and log lines as the three stage
    scripts run one after the other, but one interpreter start and one CUDA context, the resized image goes from stage 01 to
    stage 02 as an array (resized.png is written in the background, not decoded again), and stage 03 publishes the edge planes the
    fused stage-02 call has produced.  `python front_half.py` with CONFIG_PATH set, in place of steps 1-3 of pipeline.py."""
    import threading
    cfg.ensure_output_dirs()
    img = resize_if_needed(cfg.input_image, cfg)
    path = os.path.join(cfg.output_dir, "resized.png")
    writer = threading.Thread(target=cv2.imwrite, args=(path, img))       # cv2 releases the GIL while it encodes
    writer.start()
    try:
        color_extract_main(cfg, img=img)
    finally:
        writer.join()
    print(f"Saved: {path}")
    edge_detect_main(cfg)


# ---- 03_edge_detect.py ---------------------------------------------------------------------------------
def _ensure_odd(n: int) -> int:
    """03_edge_detect.py:9-11."""
    n = max(3, int(n))
    return n if n % 2 == 1 else n + 1


def _read_mask(color_name: str, cfg) -> np.ndarray:
    mask_path = os.path.join(cfg.output_dir, color_name, "mask.png")
    if not os.path.exists(mask_path):
        raise FileNotFoundError(f"Mask not found: {mask_path}")
    mask = cv2.imread(mask_path, cv2.IMREAD_GRAYSCALE)
    if mask is None:
        raise ValueError(f"Failed to load mask image: {mask_path}")
    return mask


def process_color(color_name: str, cfg):
    """03_edge_detect.py:13-40 for one layer, from <out>/<name>/mask.png."""
    mask = _read_mask(color_name, cfg)
    edges = get_engine().host_edges(mask[None], EdgeConfig.from_cfg(cfg))[0]
    out_path = os.path.join(cfg.output_dir, color_name, "edges.png")
    _write_layer_png(out_path, plane_u8=edges)
    print(f"Edges extracted: {color_name} | nz={int(np.count_nonzero(edges))}")
    return color_name, out_path


def _io_pool(cfg, n_items: int):
    from concurrent.futures import ThreadPoolExecutor
    try:
        workers = int(getattr(cfg, "n_cores", 0) or 0)
    except (TypeError, ValueError):
        workers = 0
    return ThreadPoolExecutor(max_workers=max(1, min(n_items, workers if workers > 0 else (os.cpu_count() or 1))))


def detect_all_edges(cfg) -> list:
    """03_edge_detect.py:42-48.  The reference fans layers out over a process pool; here all layers of
    equal size go through ONE batched GPU call (layers are the plane dimension of omni_edges)."""
    names = list(cfg.color_names)
    # PNG decode / encode is what is left of this stage's wall time: spread it over threads the way the reference spreads
    # layers over cfg.n_cores processes (cv2 releases the GIL); errors surface in layer order like in a serial loop
    with _io_pool(cfg, len(names)) as pool:
        masks = list(pool.map(lambda n: _read_mask(n, cfg), names))
    results = []
    shapes = {m.shape for m in masks}
    if len(shapes) == 1 and masks:
        edges = get_engine().host_edges(np.stack(masks), EdgeConfig.from_cfg(cfg))
    else:                                   # hand-edited masks of different sizes: one call per layer
        edges = [get_engine().host_edges(m[None], EdgeConfig.from_cfg(cfg))[0] for m in masks]
    paths = [os.path.join(cfg.output_dir, n, "edges.png") for n in names]
    with _io_pool(cfg, len(names)) as pool:
        list(pool.map(lambda pe: _write_layer_png(pe[0], plane_u8=pe[1]), zip(paths, edges)))
    for n, e, out_path in zip(names, edges, paths):
        print(f"Edges extracted: {n} | nz={int(np.count_nonzero(e))}")
        results.append((n, out_path))
        _JUST_WRITTEN[os.path.abspath(out_path)] = (_stamp(out_path), e)      # save_edges_composite of this process skips the decode
    return results


_JUST_WRITTEN: dict = {}       # edges.png path -> ((mtime_ns, size), plane) of files this process wrote (stage 03 paints them next)


def _stamp(path: str):
    st = os.stat(path)
    return st.st_mtime_ns, st.st_size


def _png_shape(path: str):
    """(h, w) from the IHDR chunk: 03:65 reads resized.png only for its shape (595 ms to decode 16 MP)."""
    try:
        with open(path, "rb") as fh:
            head = fh.read(24)
        if head[:8] == b"\x89PNG\r\n\x1a\n" and head[12:16] == b"IHDR":
            return int.from_bytes(head[20:24], "big"), int.from_bytes(head[16:20], "big")
    except OSError:
        pass
    return None


def save_edges_composite(cfg) -> str:
    """03_edge_detect.py:60-111.  Colours: palette_by_name.json[name]["bgr"] when present (stage 02 writes
    "approx_bgr", so in practice never), else cfg.colors[i] taken as (b, g, r) exactly as the reference
    does -- IndexError when len(colors) < len(color_names)."""
    names = list(cfg.color_names)
    rpath = os.path.join(cfg.output_dir, "resized.png")
    shape = _png_shape(rpath)
    if shape is None:                                   # not a PNG header: decode it as the reference does
        resized = cv2.imread(rpath)
        shape = None if resized is None else resized.shape[:2]
    planes = {}
    for name in names:
        p = os.path.join(cfg.output_dir, name, "edges.png")
        if os.path.exists(p):
            hit = _JUST_WRITTEN.get(os.path.abspath(p))
            e = hit[1] if hit is not None and hit[0] == _stamp(p) else cv2.imread(p, cv2.IMREAD_GRAYSCALE)
            if e is not None:
                planes[name] = e
    if shape is not None:
        h, w = shape
    elif planes:
        h, w = next(iter(planes.values())).shape[:2]
    else:
        raise FileNotFoundError("No edges found to build edges_composite.png")
    palette = {}
    pj = os.path.join(cfg.output_dir, "palette_by_name.json")
    if os.path.exists(pj):
        try:
            with open(pj, "r", encoding="utf-8") as fh:
                palette = json.load(fh) or {}
        except Exception:
            palette = {}
    name_to_bgr = {}
    for i, name in enumerate(names):
        if name in palette and "bgr" in palette[name]:
            b, g, r = palette[name]["bgr"]
        else:
            b, g, r = cfg.colors[i]
        name_to_bgr[name] = (b, g, r)
    order = [n for n in names if n in planes]
    out_path = os.path.join(cfg.output_dir, "edges_composite.png")
    if order:
        stack = np.stack([planes[n] for n in order])      # a size mismatch raises, as the reference's indexing does
        if stack.shape[1:] != (h, w):
            raise IndexError(f"edges.png size {stack.shape[1:]} does not match the canvas {(h, w)}")
        canvas = get_engine().host_edges_composite(stack, [name_to_bgr[n] for n in order])
    else:
        canvas = np.full((h, w, 3), 255, np.uint8)
    cv2.imwrite(out_path, canvas, [cv2.IMWRITE_PNG_COMPRESSION, 1])      # same pixels, a third of the encode time
    print(f"Edges composite saved: {out_path}")
    return out_path


# ---- process_colors.py ---------------------------------------------------------------------------------
def assign_labels(img_rgb: np.ndarray, palette_rgb: np.ndarray) -> np.ndarray:
    """process_colors.py:69-77 (the int16 wrap of diff*diff is reference behaviour and is reproduced)."""
    return get_engine().host_assign_rgb_i16wrap(img_rgb, palette_rgb)
