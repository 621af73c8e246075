"""Stage 04 of the reference (04_find_contours.py) on the GPU: `thinning_zhangsuen` (04:35-99) and `trace_centerlines`
(04:101-205).

The skeleton the reference computes with NumPy shifts in ~10^2 s per layer comes out of the bit-plane kernel
`omni_thin_zhangsuen` in well under a millisecond.  The walk of `trace_centerlines` is sequential within one connected
component, but the components are independent: `omni_trace_centerlines` labels them on the device (cv2's numbering and
stats) and walks every component in its own CTA, step for step as the reference does.

    thinning_zhangsuen(bin_0_255, layer)      same signature, same result, same progress lines (04:37-95)
    thin_layers(planes)                        all K edge planes in one call (what a fused stage 03 -> 04 hand-off uses)
    trace_centerlines(skel_0_255, layer)      same signature, same polylines in the same order, same progress lines
                                               (04:101-205) except the time-driven "visited n/m px" lines; one GPU call
    trace_layers(skels, names)                 all K layers in one GPU call, each layer's log lines in turn
    trace_frames(edge_bits, w, K)              packed edge planes of n frames -> thinning + polylines of every layer of every
                                               frame in one GPU call (omni_centerlines_packed); no log lines
    trace_centerlines(skel, layer, maps=...)   the host walk (a Python restatement of 04:126-200 that takes the degree /
                                               endpoint / junction maps of the whole skeleton and confines every component to
                                               its bounding box): the reference the GPU tracer is tested against
"""
from __future__ import annotations

import time

import cv2
import numpy as np

from .ops import get_engine

MAX_ITER = 120                      # 04_find_contours.py:52


def thin_layers(planes: np.ndarray, max_iter: int = MAX_ITER):
    """[K,H,W] u8 (> 0 = edge) -> (skeletons {0,255}, removed[K,max_iter], iters[K])."""
    return get_engine().host_thin_zhangsuen(planes, max_iter)


def thinning_zhangsuen(bin_0_255: np.ndarray, layer: str) -> np.ndarray:
    """Drop-in for 04_find_contours.py:35-99 (same prints; the per-iteration seconds are the kernel's share)."""
    if bin_0_255.ndim != 2:
        raise ValueError("thinning_zhangsuen expects a single-channel image")
    ys, xs = np.nonzero(bin_0_255)
    if len(xs) == 0:
        print(f"[{layer}] Thinning: empty edges.", flush=True)
        return np.zeros_like(bin_0_255)
    pad = 2                                                       # _bbox_of_nonzero, 04:24-33 (only for the log line)
    x0, x1 = max(0, xs.min() - pad), min(bin_0_255.shape[1] - 1, xs.max() + pad)
    y0, y1 = max(0, ys.min() - pad), min(bin_0_255.shape[0] - 1, ys.max() + pad)
    total0 = int(len(xs))
    print(f"[{layer}] Thinning ROI {x1 - x0 + 1}x{y1 - y0 + 1}, fg={total0} px", flush=True)
    t0 = time.perf_counter()
    src = np.ascontiguousarray(bin_0_255 if bin_0_255.dtype == np.uint8 else (bin_0_255 > 0).astype(np.uint8) * 255)
    out, removed, iters = get_engine().host_thin_zhangsuen(src[None], MAX_ITER)
    dt = time.perf_counter() - t0
    n_it = int(iters[0])
    total_removed = 0
    for it in range(1, n_it + 1):
        r = int(removed[0, it - 1])
        total_removed += r
        pct = total_removed / max(1, total0) * 100.0
        print(f"[{layer}] Thin {it:02d}: removed={r:6d} | total={total_removed:7d} ({pct:5.1f}%) | {dt / max(1, n_it):.2f}s", flush=True)
    print(f"[{layer}] Thinning done in {dt:.2f}s, fg_now={total0 - total_removed} px", flush=True)
    return out[0].astype(bin_0_255.dtype, copy=False)


def skeleton_degree(skel_0_255: np.ndarray):
    """04_find_contours.py:117-125 for ALL components at once: (deg, endpoints, junctions) of the skeleton -- what
    trace_centerlines recomputes per component with a full-image filter2D.  On the pixels of a component the maps equal the
    reference's per-component ones (a pixel's 8-neighbours belong to its own component), so inside the component loop
    `deg`, `endpoints`, `junctions` can be replaced by `deg_all`, `ep_all & (comp_mask == 1)`, `jn_all & (comp_mask == 1)`."""
    import torch
    sk = torch.from_numpy(np.ascontiguousarray(skel_0_255, dtype=np.uint8)[None]).cuda()
    deg, nodes = get_engine().skeleton_degree(sk)
    nodes = nodes[0].cpu().numpy()
    return deg[0].cpu().numpy(), nodes == 1, nodes == 2


NEIGH8 = [(-1, -1), (0, -1), (1, -1), (-1, 0), (1, 0), (-1, 1), (0, 1), (1, 1)]          # 04_find_contours.py:12 (the visiting order)


def _log_trace(r, layer: str, dt: float):
    """The log lines of 04:104-205 for one plane from the GPU result (the seconds are the call's, shared over the components)."""
    if r.total_fg == 0:
        print(f"[{layer}] Trace: empty skeleton.", flush=True)
        return []
    n = len(r.stats)
    print(f"[{layer}] Trace: fg={r.total_fg} px | components={n}", flush=True)
    done = so_far = 0
    for i, (area, npl) in enumerate(zip(r.stats[:, 4].tolist(), r.polylines.tolist()), 1):
        done += area
        so_far += npl
        print(f"[{layer}]  \u2022 Component {i}/{n}: pixels={area}", flush=True)
        print(f"[{layer}]  \u2022 Component {i} done in {dt / n:.2f}s, polylines so far: {so_far}", flush=True)
        print(f"[{layer}]  \u2022 Progress: components_fg {done}/{r.total_fg} px ({100.0 * done / r.total_fg:4.1f}%)", flush=True)
    print(f"[{layer}] Trace done: {len(r.paths)} polylines in {dt:.2f}s", flush=True)
    return r.paths


def trace_layers(skels: np.ndarray, names):
    """trace_centerlines of K skeleton planes [K,H,W] in ONE GPU call; prints each layer's log lines in turn (the seconds are the
    call's time shared over the layers) and returns the K polyline lists."""
    t0 = time.perf_counter()
    res = get_engine().host_trace_centerlines(skels)
    dt = (time.perf_counter() - t0) / max(1, len(res))
    return [_log_trace(r, name, dt) for r, name in zip(res, names)]


def trace_centerlines(skel_0_255: np.ndarray, layer: str, maps=None):
    """Drop-in for 04_find_contours.py:101-205: the reference's polylines in the reference's order, the same log lines.
    maps=None: one GPU call (omni_trace_centerlines).  maps=(deg, endpoints, junctions) of the whole skeleton: the host walk."""
    if maps is None:
        return trace_layers(np.asarray(skel_0_255)[None], [layer])[0]
    return _trace_host(skel_0_255, layer, maps)


def trace_frames(edge_bits: np.ndarray, w: int, K: int, max_iter: int = MAX_ITER):
    """Packed edge planes [n*K, H, ceil(w/8)] (MSB-first, as host_color_edge_packed / batch.process_shard_packed return them) ->
    n lists of K polyline lists: frame f, layer k = trace_centerlines(thinning_zhangsuen(plane f*K + k)), int32 (n,1,2) arrays.
    All planes go through one GPU call; a batch API, so it prints nothing."""
    a = np.asarray(edge_bits)
    if a.ndim != 3 or K < 1 or a.shape[0] % K:
        raise ValueError(f"expected packed edge planes [n*K, H, RB] with K={K} layers per frame, got {list(a.shape)}")
    res = get_engine().host_centerlines_packed(a, w, max_iter)
    return [[r.paths for r in res[f * K:(f + 1) * K]] for f in range(a.shape[0] // K)]


def _trace_host(skel_0_255: np.ndarray, layer: str, maps):
    """The host walk, kept step for step (start pixels in row-major order, NEIGH8 neighbour order, the same guards); what
    changes against the reference is where its inputs come from: `maps` = (deg, endpoints, junctions) of the whole skeleton --
    on the pixels of a component they equal the reference's per-component maps, because the 8-neighbours of a component pixel
    belong to that component -- and each component lives in its bounding box (cv2.connectedComponentsWithStats, same labels).
    The time-driven "visited n/m px" lines appear when 1.5 s have passed, as in the reference, but are only looked at every
    1024 steps."""
    t0 = time.perf_counter()
    S = (skel_0_255 > 0).astype(np.uint8)
    total_fg = int(S.sum())
    if total_fg == 0:
        print(f"[{layer}] Trace: empty skeleton.", flush=True)
        return []
    num, labels, stats, _c = cv2.connectedComponentsWithStats(S, connectivity=8)
    print(f"[{layer}] Trace: fg={total_fg} px | components={num-1}", flush=True)
    _deg_all, ep_all, jn_all = maps
    paths = []
    comp_fg_done = 0
    for comp_id in range(1, num):
        bx, by, bw, bh = (int(stats[comp_id, k]) for k in (cv2.CC_STAT_LEFT, cv2.CC_STAT_TOP, cv2.CC_STAT_WIDTH, cv2.CC_STAT_HEIGHT))
        roi = (slice(by, by + bh), slice(bx, bx + bw))
        fg_comp = int(stats[comp_id, cv2.CC_STAT_AREA])
        comp_fg_done += fg_comp
        print(f"[{layer}]  \u2022 Component {comp_id}/{num-1}: pixels={fg_comp}", flush=True)
        # the component in a frame of one background pixel, as flat byte strings: index = (y + 1) * W2 + (x + 1); the eight
        # neighbour offsets in NEIGH8 order.  (Plain Python integers: the walk below is the stage's inner loop.)
        W2 = bw + 2
        frame = np.zeros((bh + 2, W2), np.uint8)
        frame[1:-1, 1:-1] = labels[roi] == comp_id
        comp = frame.tobytes()
        inner = frame[1:-1, 1:-1].astype(bool)
        frame[1:-1, 1:-1] = inner & ep_all[roi]
        is_end = frame.tobytes()
        frame[1:-1, 1:-1] = inner & jn_all[roi]
        is_junction = frame.tobytes()
        visited = bytearray((bh + 2) * W2)
        offs = [dy * W2 + dx for dx, dy in NEIGH8]
        visited_count = 0
        t_comp = time.perf_counter()
        last_print_t = t_comp

        def emit(path, close):
            idx = np.array(path, dtype=np.int64)
            arr = np.stack([idx % W2 - 1 + bx, idx // W2 - 1 + by], axis=1).astype(np.int32).reshape(-1, 1, 2)
            if close and np.hypot(arr[0, 0, 0] - arr[-1, 0, 0], arr[0, 0, 1] - arr[-1, 0, 1]) < 1.5:
                arr = np.vstack([arr, arr[0:1]])
            paths.append(arr)

        # 1) open paths: from every endpoint to the next endpoint / junction (04:143-170)
        ys, xs = np.nonzero(inner & ep_all[roi])
        for s0 in ((ys + 1) * W2 + xs + 1).tolist():
            if visited[s0]:
                continue
            path = [s0]
            visited[s0] = 1
            visited_count += 1
            p, prev = s0, -1
            step_guard = 0
            while True:
                nxt = -1
                for o in offs:                                   # first unvisited neighbour other than the previous pixel
                    q = p + o
                    if comp[q] and q != prev and not visited[q]:
                        nxt = q
                        break
                if nxt < 0:
                    break
                path.append(nxt)
                visited[nxt] = 1
                visited_count += 1
                prev, p = p, nxt
                if is_junction[p] or is_end[p]:
                    break
                step_guard += 1
                if step_guard > total_fg * 2:
                    break
                if not step_guard & 1023 and time.perf_counter() - last_print_t > 1.5:
                    print(f"[{layer}]    visited {visited_count}/{fg_comp} px ({100.0 * visited_count / max(1, fg_comp):4.1f}%)", flush=True)
                    last_print_t = time.perf_counter()
            if len(path) >= 2:
                emit(path, False)

        # 2) what is left: cycles (04:172-200)
        left = np.frombuffer(bytes(visited), np.uint8).reshape(bh + 2, W2)[1:-1, 1:-1] == 0
        ys, xs = np.nonzero(inner & left)
        for s0 in ((ys + 1) * W2 + xs + 1).tolist():
            if visited[s0]:
                continue
            path = [s0]
            visited[s0] = 1
            visited_count += 1
            p, prev = s0, -1
            step_guard = 0
            while True:
                nxt = -1
                for o in offs:
                    q = p + o
                    if comp[q] and q != prev and not visited[q]:
                        nxt = q
                        break
                if nxt < 0:
                    for o in offs:                               # the closing step onto an already visited pixel
                        q = p + o
                        if comp[q] and q != prev:
                            nxt = q
                            break
                    if nxt < 0:
                        break
                path.append(nxt)
                if not visited[nxt]:
                    visited[nxt] = 1
                    visited_count += 1
                prev, p = p, nxt
                if p == s0:
                    break
                step_guard += 1
                if step_guard > fg_comp * 4:
                    break
                if not step_guard & 1023 and time.perf_counter() - last_print_t > 1.5:
                    print(f"[{layer}]    visited {visited_count}/{fg_comp} px ({100.0 * visited_count / max(1, fg_comp):4.1f}%)", flush=True)
                    last_print_t = time.perf_counter()
            if len(path) >= 2:
                emit(path, True)

        print(f"[{layer}]  \u2022 Component {comp_id} done in {time.perf_counter()-t_comp:.2f}s, polylines so far: {len(paths)}", flush=True)
        print(f"[{layer}]  \u2022 Progress: components_fg {comp_fg_done}/{total_fg} px ({100.0*comp_fg_done/total_fg:4.1f}%)", flush=True)
    print(f"[{layer}] Trace done: {len(paths)} polylines in {time.perf_counter()-t0:.2f}s", flush=True)
    return paths
